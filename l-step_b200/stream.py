"""Streaming PE-step API with a device-resident edge stream and PE-history ring buffer
(SURVEY §8(f) f1).

The reference's loops (train_LSTEP_link_prediction.py:205,224-230,301-306;
evaluate_model_utils.py:57-63,131-135) keep the PE history as a [V1, <=T+1, d] tensor that they
trim (full clone), slice, and re-concatenate every batch — 3 GB of copies per batch at Reddit
size — and hand every batch to the model as host numpy arrays. `PEStream` is an additional,
numerically identical way to run the same per-batch sequence

    a3  fft = fourier_transform_pe(ids, hist[:, -T:], batch_idx)
        cur = clone(hist[:, -1]); cur[ids] = fft
    a6  C x compute_neighborhood_pe(cur, q_ids, times)
    a7/a8 update_pe(cur, ids, ..., current_time = max(times))
        hist = cat(hist, cur)

with the whole edge stream uploaded once and the history held in a ring of T slots, so a step
moves only the bytes the algorithm needs. `export_history()` materialises the reference layout
[V1, Th, d] (chronological, oldest first) for torch.save / parity checks, `import_history()`
adopts one (utils/EarlyStopping.py:79-82,100-104).
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib
from .changelog import ChangeLogOwner, RingHistory
from .hostfeed import HostFed
from .model import LSTEP
from .peer import batch_plan

C_void_p = ctypes.c_void_p
C_byref = ctypes.byref
_I64 = np.dtype(np.int64)


class PEStream(HostFed):
    def __init__(self, model: LSTEP, src_node_ids: np.ndarray, dst_node_ids: np.ndarray, node_interact_times: np.ndarray,
                 batch_size: int, num_neighbors: int = 20, initial_pe: torch.Tensor = None, history: torch.Tensor = None,
                 start: int = 0, stop: int = None, row_capacity: int = None, new_node_pe=None, max_nodes: int = None):
        """row_capacity: rows to allocate for the table and the history (default: the initial V1), so that add_nodes /
        grow=True add nodes without reallocating until it runs out (then it doubles). new_node_pe: the row [d] a node added
        by a count or by grow=True starts with (default zeros). max_nodes: optional limit on the node count."""
        self.model = model
        self.K = int(num_neighbors)
        self.B = int(batch_size)
        self.T = model.num_fft_batches
        self.d = model.pe_dim
        dev = self.dev = model._dev()
        if dev.type != "cuda":
            raise _lib.LstepError("PEStream needs the model on a CUDA device (no CPU path)")
        stop = len(src_node_ids) if stop is None else stop
        self.start, self.stop = int(start), int(stop)
        self.src_np = np.ascontiguousarray(src_node_ids, dtype=np.int64)
        self.dst_np = np.ascontiguousarray(dst_node_ids, dtype=np.int64)
        self.t_np = np.ascontiguousarray(node_interact_times, dtype=np.float64)
        # whole stream resident in HBM (24 B/edge)
        self.src = torch.from_numpy(self.src_np).to(dev)
        self.dst = torch.from_numpy(self.dst_np).to(dev)
        self.t = torch.from_numpy(self.t_np).to(dev)
        # per-batch sorted unique node ids (the loops compute them on the host with torch.unique:
        # evaluate_model_utils.py:54-55); done once for the whole stream here
        self._adopt_plan(batch_plan(self.src_np, self.dst_np, self.t_np, self.start, self.stop, self.B))
        self._host_init()
        self._growth_init(new_node_pe, max_nodes)
        self._row_cap_arg = row_capacity
        self.V1 = None
        self.batch_idx = 0
        if history is not None:
            self.import_history(history)
        elif initial_pe is not None:
            self.import_history(initial_pe.unsqueeze(1))

    # ---- history ring -----------------------------------------------------------------------
    def import_history(self, history: torch.Tensor):
        """Adopt a reference-layout history [V1, Th, d] (chronological; its last T steps are kept)."""
        history = history.to(self.dev, torch.float32)[:, -self.T:]
        assert history.shape[2] == self.d
        self._check_stream_ids(history.shape[0])
        self._new_state(RingHistory(history.shape[0], self.T, self.d, self.dev, self._row_cap_arg))
        self.head, self.len = self.history.load(history, self.cur)
        self.steps_done, self.edges_done = 0, self.start

    @property
    def ring(self) -> torch.Tensor:
        """The dense history [row_cap, T, d], node-major (None on a change-log history)."""
        return self.history.ring

    # ---- one batch --------------------------------------------------------------------------
    def batch_arrays(self, b: int):
        lo = int(self.batch_lo[b])
        return lo, lo + int(self.n_edges[b]), int(self.ids_off[b]), int(self.ids_off[b + 1])

    @property
    def _desc_ref(self):
        return C_byref(self.desc)

    def step(self, b: int, queries, out: torch.Tensor = None, batch_idx: int = None):
        """Run batch b of the resident stream. `queries`: list of device int64 tensors [B_b] of node ids
        for the compute_neighborhood_pe calls (positive sources / destinations, negatives), all queried
        at the batch's edge times. Returns a [C, B_b, d] tensor of neighbourhood PEs; the updated
        table is self.cur and has been appended to the ring."""
        return self._step(b, queries, out, 7, batch_idx)

    def _step_call(self, b, lo, n, ids, n_ids, tmax, G, qptrs, C, q_off, q_rows, out, ws, phases) -> int:
        m = self.model
        slot = (self.head + self.len) % self.T  # (the slot changelog.advance writes: the next free one, then the oldest)
        return self.lib.lstep_pe_step(self._desc_ref, m.neighbor_sampler.csr_ref, lo, n, ids, n_ids, tmax, self.head, self.len, slot,
                                      _lib.ptr(G), qptrs, C, _lib.ptr(out), self.K, m._mlp_ref("nbr"), m._mlp_ref("update"), _lib.ptr(ws),
                                      ws.numel(), _lib.ptr(m.neighbor_sampler._err), _lib.stream_ptr())

    def run(self, b0: int, n_steps: int, queries, out: torch.Tensor = None, check: bool = False) -> torch.Tensor:
        """Batches b0 .. b0+n_steps-1 of the resident stream in ONE native call (lstep_pe_steps): the per-batch loop
        runs in C, so the host pays six kernel launches per step and nothing else. `queries`: list of device int64
        tensors holding, for every query set, the node ids of ALL edges of those batches back to back (entry e belongs
        to edge lo(b0) + e). Returns the neighbourhood PEs of the LAST step [C, n_last, d] (or fills and returns `out`
        [n_steps, C, B, d] with every step's). While the history is still filling, and on a history without a native
        multi-step call (ChangeLogStream), it calls step() per batch.
        check=True: read the device error flag afterwards (synchronises; IndexError for a query id unknown to the sampler)."""
        if n_steps <= 0:
            return None
        if self.len == self.T and self._run_call is not None:
            last = self._run_call(b0, n_steps, queries, out)
        else:
            lo0 = int(self.batch_lo[b0])
            for i in range(n_steps):
                lo, hi, _, _ = self.batch_arrays(b0 + i)
                last = self.step(b0 + i, [q[lo - lo0:hi - lo0] for q in queries], None if out is None else out[i])
        if check:
            self.check_errors()
        return out if out is not None else last

    def _run_call(self, b0: int, n_steps: int, queries, out: torch.Tensor = None) -> torch.Tensor:
        """run() on a full history: one lstep_pe_steps call. Returns the last step's neighbourhood PEs."""
        lib, m = self.lib, self.model
        B, d, C = self.B, self.d, len(queries)
        los, ne, tmax = (a[b0:b0 + n_steps] for a in (self.batch_lo, self.n_edges, self.batch_tmax))
        ids_off = self.ids_off[b0:b0 + n_steps + 1]
        q_off = los - los[0]
        with torch.cuda.device(self.dev), torch.no_grad():
            G = m._collapsed_filter(self.T, False)
            ws = self._workspace(int(np.diff(ids_off).max()), int(ne.max()), C)
            if out is None:
                buf = torch.empty((max(C, 1), B, d), dtype=torch.float32, device=self.dev)
                stride = 0
            else:
                buf = out
                stride = max(C, 1) * B * d
                if ne.min() != B:
                    raise ValueError("run(out=...) needs full batches (a ragged last batch changes the [C, n, d] layout)")
            qptrs = (C_void_p * max(C, 1))(*[q.data_ptr() for q in queries])
            head, ln = ctypes.c_int(self.head), ctypes.c_int(self.len)
            rc = lib.lstep_pe_steps(self._desc_ref, m.neighbor_sampler.csr_ref, n_steps, los.ctypes.data, ne.ctypes.data,
                                    self.ids.data_ptr(), ids_off.ctypes.data, tmax.ctypes.data, C_byref(head), C_byref(ln), G.data_ptr(),
                                    qptrs, q_off.ctypes.data, C, buf.data_ptr(), stride, self.K, m._mlp_ref("nbr"), m._mlp_ref("update"),
                                    ws.data_ptr(), ws.numel(), m.neighbor_sampler._err.data_ptr(),
                                    torch.cuda.current_stream().cuda_stream)
            done = (head.value - self.head) % self.T if rc != 0 else n_steps
            self._advance(done, int(ne[:done].sum()))
            if rc != 0:
                _lib.check(rc, "lstep_pe_steps")
        n_last = int(ne[-1])
        return buf.view(-1)[:max(C, 1) * n_last * d].view(max(C, 1), n_last, d)

    # ---- host-fed steps: step_host_async / step_host / run_host and result are hostfeed.HostFed's, which validates, stages,
    # arms the ingest, moves the window and keeps the tickets around the native calls of csrc/host_step.cu below. A layout
    # supplies its own checks of a batch and these two native calls; ChangeLogStream replaces the checks and
    # the calls. Each call returns the native status.
    def _host_sampler(self):
        return self.model.neighbor_sampler

    def _check_host(self, src, dst, times, qs, ids, V1: int, n_max: int):
        """None beyond the shared checks: the native stager rejects ids outside the table and the sampler's rows."""
        return None if ids is None else np.ascontiguousarray(ids, dtype=_I64)

    def _host_step_call(self, h, n, src, dst, times, ids, G, qptrs, C, out, ws, phases, ticket) -> int:
        m, samp = self.model, self.model.neighbor_sampler
        return self.lib.lstep_pe_step_host(h, self._desc_ref, samp.csr_ref, n, src.ctypes.data, dst.ctypes.data, times.ctypes.data,
                                           ids.ctypes.data if ids is not None else None, len(ids) if ids is not None else 0, self.head,
                                           self.len, (self.head + self.len) % self.T, G.data_ptr(), qptrs, C,
                                           out.data_ptr() if out is not None else None, self.K, m._mlp_ref("nbr"), m._mlp_ref("update"),
                                           ws.data_ptr(), ws.numel(), samp._err.data_ptr(), torch.cuda.current_stream().cuda_stream,
                                           C_byref(ticket))

    def _host_run_call(self, h, n, src, dst, times, qptrs, C, G, ws, res, done) -> int:
        m, samp = self.model, self.model.neighbor_sampler
        head, ln = ctypes.c_int(self.head), ctypes.c_int(self.len)  # (the window is moved by HostFed._advance from done)
        return self.lib.lstep_pe_steps_host(h, self._desc_ref, samp.csr_ref, n, self.B, src.ctypes.data, dst.ctypes.data,
                                            times.ctypes.data, qptrs, C, C_byref(head), C_byref(ln), G.data_ptr(), self.K,
                                            m._mlp_ref("nbr"), m._mlp_ref("update"), ws.data_ptr(), ws.numel(), samp._err.data_ptr(),
                                            torch.cuda.current_stream().cuda_stream, res.ctypes.data, C_byref(done))


class ChangeLogStream(ChangeLogOwner, PEStream):
    """PEStream on a CHANGE-LOG history (csrc/changelog.cu) instead of the dense ring: base rows + the rows every step
    changed, V1 + T * (rows changed per step) rows instead of V1 * T — 7.8 GB instead of 688 GB for the 10 M-node graph at
    T = 100, and ~9 MB written per step instead of 13.8 GB (the dense ring's append copies one row per node per step).
    Same API (step, the host-fed step_host_async / step_host / run_host with ingest=, cur, export_history / import_history); the DFT filter sums (events in window + 1) rows per node with
    span sums of G as weights. `event_capacity`: events one step may record (default: every row a batch can touch,
    2B + 2BK + 2, capped at V1); importing a dense history needs capacity for the rows that differ between consecutive
    snapshots. `row_mul` / `row_add`: node-id sharded groups keep only the nodes v % row_mul == row_add.

    `checkpoint`: resume from a checkpoint directory that save_checkpoint or a PeerRank group of any world size wrote (or
    the checkpoint.History that checkpoint.read returned), instead of initial_pe / history; head, len, batch_idx and
    steps_done continue from it. `batch_idx` overrides the batch index the next step masks the filter with while the
    history is shorter than T (the reference's evaluate loop restarts it at 0: Q5)."""

    def __init__(self, model: LSTEP, src_node_ids: np.ndarray, dst_node_ids: np.ndarray, node_interact_times: np.ndarray,
                 batch_size: int, num_neighbors: int = 20, initial_pe: torch.Tensor = None, history: torch.Tensor = None,
                 start: int = 0, stop: int = None, row_capacity: int = None, new_node_pe=None, max_nodes: int = None, *,
                 event_capacity: int = None, checkpoint=None, batch_idx: int = None):
        if checkpoint is not None and (initial_pe is not None or history is not None):
            raise ValueError("ChangeLogStream: give one of initial_pe, history and checkpoint")
        self._cap_arg = event_capacity
        super().__init__(model, src_node_ids, dst_node_ids, node_interact_times, batch_size, num_neighbors, None, None, start, stop,
                         row_capacity, new_node_pe, max_nodes)
        self._start(initial_pe, history, checkpoint, batch_idx)

    def import_history(self, history: torch.Tensor):
        self._start(None, history, None, None)

    def _default_event_cap(self, V1: int) -> int:
        return min(V1, 2 * self.B * (self.K + 1) + 2)  # every row a batch can touch, at most every node

    def _step_call(self, b, lo, n, ids, n_ids, tmax, G, qptrs, C, q_off, q_rows, out, ws, phases) -> int:
        m = self.model
        return self.lib.lstep_pe_step_changelog(self._desc_ref, self.changelog.ref, m.neighbor_sampler.csr_ref, lo, n, ids, n_ids, tmax,
                                                self.head, self.len, _lib.ptr(G), qptrs, C, q_off, q_rows, _lib.ptr(out), self.K,
                                                m._mlp_ref("nbr"), m._mlp_ref("update"), _lib.ptr(ws), ws.numel(),
                                                _lib.ptr(m.neighbor_sampler._err), _lib.stream_ptr(), 0)

    _run_call = None  # (no native multi-step call for this history: run() calls step() per batch)

    # ---- host-fed steps: HostFed's driver, with the change-log step as the native call ---------------------------------
    def _check_host(self, src, dst, times, qs, ids, V1: int, n_max: int):
        """A step records its events in the log: event_capacity, sized from batch_size by default, bounds them, so a batch
        longer than batch_size is rejected before anything is enqueued."""
        if len(src) > n_max:
            raise ValueError(f"ChangeLogStream: a host batch of {len(src)} edges is longer than batch_size ({self.B}), which sizes the "
                             f"change log's event_capacity ({self.cap}); split the batch or build the stream with a larger batch_size")
        return super()._check_host(src, dst, times, qs, ids, V1, n_max)

    def _host_step_call(self, h, n, src, dst, times, ids, G, qptrs, C, out, ws, phases, ticket) -> int:
        m, samp = self.model, self.model.neighbor_sampler
        return self.lib.lstep_pe_step_changelog_host(h, self._desc_ref, self.changelog.ref, samp.csr_ref, n, src.ctypes.data,
                                                     dst.ctypes.data, times.ctypes.data, ids.ctypes.data if ids is not None else None,
                                                     len(ids) if ids is not None else 0, self.head, self.len, G.data_ptr(), qptrs, C,
                                                     out.data_ptr() if out is not None else None, self.K, m._mlp_ref("nbr"),
                                                     m._mlp_ref("update"), ws.data_ptr(), ws.numel(), samp._err.data_ptr(),
                                                     torch.cuda.current_stream().cuda_stream, C_byref(ticket))

    def _host_run_call(self, h, n, src, dst, times, qptrs, C, G, ws, res, done) -> int:
        m, samp = self.model, self.model.neighbor_sampler
        head, ln = ctypes.c_int(self.head), ctypes.c_int(self.len)
        return self.lib.lstep_pe_steps_changelog_host(h, self._desc_ref, self.changelog.ref, samp.csr_ref, n, self.B, src.ctypes.data,
                                                      dst.ctypes.data, times.ctypes.data, qptrs, C, C_byref(head), C_byref(ln), G.data_ptr(),
                                                      self.K, m._mlp_ref("nbr"), m._mlp_ref("update"), ws.data_ptr(), ws.numel(),
                                                      samp._err.data_ptr(), torch.cuda.current_stream().cuda_stream, res.ctypes.data,
                                                      C_byref(done))
