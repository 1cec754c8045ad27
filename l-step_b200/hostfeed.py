"""Host-fed steps: the Python side every history layout shares (PEStream, ChangeLogStream, PeerRank).

A host-fed step hands one batch of HOST (numpy) arrays to a native stepper (csrc/host_step.cu), which packs it into a pinned
slot, copies it in, runs the step and copies the per-query row sums back, and returns a ticket. `HostFed` owns that stepper and
what surrounds the native call: the normalisation of the host arrays, the validation and room-making of a batch that is ingested
into a growable sampler (ingest=True), the arming of the stepper for it, the ticket bookkeeping and `result`, and the resync of
the sampler after a failed call. A class that mixes it in provides `dev`, `B`, `d` and `_host_sampler()`, the sampler whose CSR
its steps read.

It also owns the growth of the node set (add_nodes, and grow=True on the host-fed steps): new node ids continue after the
last live one, and a new node starts with its initial row r0 in the table, in every history slot and as its change-log base
row, which is exactly the state a node no edge has touched has in a stream built with those rows from the start. So a grown
stream computes the bits of the pre-sized one. The class provides `V1`, `row_cap`, `_grow_capacity(row_cap)`, which
reallocates its tables for more rows (every new buffer allocated before any is swapped in), `_init_rows(v0, v1, rows,
stride)`, which enqueues lstep_pe_rows_init, and `_set_live(V1)`."""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib
from .sampler import NODE_ID_MAX, check_edges, new_row_need

C_void_p = ctypes.c_void_p
C_byref = ctypes.byref
_I64, _F64 = np.dtype(np.int64), np.dtype(np.float64)


def host_arrays(src, dst, times, query_ids, what: str):
    """(src, dst, times, query sets) as contiguous int64 / float64 arrays (no copy when they already are). ValueError when
    the lengths differ."""
    n = len(src)
    if src.dtype != _I64 or not src.flags.c_contiguous:
        src = np.ascontiguousarray(src, dtype=_I64)
    if dst.dtype != _I64 or not dst.flags.c_contiguous:
        dst = np.ascontiguousarray(dst, dtype=_I64)
    if times.dtype != _F64 or not times.flags.c_contiguous:
        times = np.ascontiguousarray(times, dtype=_F64)
    qs = [q if (q.dtype == _I64 and q.flags.c_contiguous) else np.ascontiguousarray(q, dtype=_I64) for q in query_ids]
    if len(dst) != n or len(times) != n or any(len(q) != n for q in qs):
        raise ValueError(f"{what}: src, dst, times and every query set must have the same length")
    return src, dst, times, qs


class HostFed:
    HOST_SLOTS = 4  # steps that may be in flight before step_host_async blocks on the oldest

    def _host_init(self):
        self._host_stepper = None
        self._armed = None  # (stepper, sampler, sampler version) the stepper was armed to ingest into, see _arm_ingest
        self._ticket_shape = {}
        self._drained = {}  # public ticket -> result read out before its stepper was replaced
        self._epoch = 0
        self._libc = _lib.load()

    def _host_sampler(self):
        raise NotImplementedError

    def _stepper(self, n_edges: int, C: int):
        lib = _lib.load()
        st = self._host_stepper
        if st is None or st[1] < n_edges or st[2] < C:
            if st is not None:
                # a larger batch / more query sets than the stepper was sized for: results of tickets still outstanding
                # are read out first (the native ticket numbering restarts with the new stepper; public tickets carry the
                # stepper's epoch so an old one can never alias a new one)
                for tk in sorted(self._ticket_shape):
                    try:
                        self._drained[tk] = self._result_now(tk)
                    except ValueError:  # result slot already reused by later steps (e.g. a run_host call): nothing to keep
                        pass
                self._ticket_shape.clear()
                lib.lstep_host_stepper_destroy(st[0])
                self._epoch += 1
                self._armed = None
            h = C_void_p()
            cap_e, cap_c = max(self.B, n_edges), max(C, 4)
            with torch.cuda.device(self.dev):
                _lib.check(lib.lstep_host_stepper_create(self.HOST_SLOTS, cap_e, cap_c, self.d, C_byref(h)), "lstep_host_stepper_create")
            self._host_stepper = st = (h, cap_e, cap_c)
        return st[0]

    def _host_stepper_for(self, n_edges: int, C: int):
        st = self._host_stepper
        if st is None or st[1] < n_edges or st[2] < C:
            return self._stepper(n_edges, C)
        return st[0]

    def __del__(self):
        st = getattr(self, "_host_stepper", None)
        if st is not None:
            try:
                _lib.load(False).lstep_host_stepper_destroy(st[0])
            except Exception:
                pass
            self._host_stepper = None

    # ---- node growth --------------------------------------------------------------------------------------------------
    def _growth_init(self, new_node_pe=None, max_nodes: int = None):
        """new_node_pe: the row [d] a node added without explicit rows starts with (default zeros, what RandomWalkPE gives an
        isolated node); max_nodes: optional limit on the node count (ids >= max_nodes raise IndexError)."""
        r0 = np.zeros(self.d, np.float32) if new_node_pe is None else self._rows_array(new_node_pe, 1)
        self._r0 = torch.from_numpy(r0).to(self.dev)
        self.max_nodes = None if max_nodes is None else int(max_nodes)

    def _rows_array(self, rows, ndim: int) -> np.ndarray:
        """rows as a contiguous float32 host array of shape [d] (ndim 1) or [n, d] (ndim 2); ValueError otherwise."""
        if isinstance(rows, torch.Tensor):
            rows = rows.detach().cpu()
        try:
            a = np.ascontiguousarray(np.asarray(rows, dtype=np.float32))
        except (TypeError, ValueError) as e:
            raise ValueError(f"new node rows must convert to float32: {e}") from None
        if a.ndim != ndim or a.shape[-1] != self.d:
            raise ValueError(f"new node rows must have shape {'[d]' if ndim == 1 else '[n, d]'} with d = {self.d} (got {a.shape})")
        if not np.isfinite(a).all():
            raise ValueError("new node rows must be finite")
        return a

    def _check_new_ids(self, hi: int):
        """IndexError when node id `hi` may not be added (int32 limit of the change log's node ids, max_nodes)."""
        if hi > NODE_ID_MAX:
            raise IndexError(f"node id {hi} exceeds the int32 node id limit ({NODE_ID_MAX})")
        if self.max_nodes is not None and hi >= self.max_nodes:
            raise IndexError(f"node id {hi} is outside max_nodes ({self.max_nodes})")

    def _check_event_capacity(self, V1: int):
        """Change-log histories: ValueError when a step on V1 nodes could change more rows than the log records per step."""

    def _new_nodes_for(self, arrays) -> int:
        """grow=True: validate the ids of a batch (or a run) and return how many nodes it adds (ids up to its maximum).
        Nothing is written."""
        lo = min(int(a.min()) for a in arrays if len(a))
        hi = max(int(a.max()) for a in arrays if len(a))
        if lo < 0:
            raise IndexError(f"list index out of range: node id {lo}")
        n_new = max(0, hi + 1 - self.V1)
        if n_new:
            self._check_new_ids(hi)
            self._growable_sampler()
        return n_new

    def add_nodes(self, rows_or_count, _edges=None) -> int:
        """Add nodes with the next ids and return the first of them. rows_or_count: a count n (each new node starts with
        the stream's new_node_pe row) or per-node rows [n, d] (float32-convertible, finite). The table, the history and
        the model's growable sampler grow together; everything is validated before any device write, and the rows are
        written on the current stream, behind the steps already enqueued (which touch only rows below the old V1). When
        the row capacity runs out it doubles: new buffers are allocated first, then the live rows are copied."""
        if isinstance(rows_or_count, (int, np.integer)):
            n, rows, stride = int(rows_or_count), self._r0, 0
            if n < 0:
                raise ValueError("add_nodes: the count must be >= 0")
        else:
            a = self._rows_array(rows_or_count, 2)
            n, rows, stride = a.shape[0], a, self.d
        v0 = self.V1
        if n == 0:
            return v0
        self._check_new_ids(v0 + n - 1)
        self._check_event_capacity(v0 + n)
        samp = self._growable_sampler()
        if isinstance(rows, np.ndarray):
            rows = torch.from_numpy(rows).pin_memory().to(self.dev, non_blocking=True)
        v1 = v0 + n
        if v1 > self.row_cap:
            self._grow_capacity(max(2 * self.row_cap, v1))
        if v1 > samp.num_rows:
            k = v1 - samp.num_rows
            samp.add_rows(k, None if _edges is None else new_row_need(_edges[0], _edges[1], samp.num_rows, k))
        with torch.cuda.device(self.dev):
            self._init_rows(v0, v1, rows, stride)
        self._set_live(v1)
        return v0

    # ---- ingest -------------------------------------------------------------------------------------------------------
    def _growable_sampler(self):
        samp = self._host_sampler()
        if samp is None or not samp.is_growable:
            raise ValueError("ingest=True needs a growable neighbor sampler: model.set_neighbor_sampler(NeighborSampler.growable(...))")
        return samp

    def _check_ingest(self, src, dst, times, edge_id_start, n_new: int = 0):
        """Validate a host batch for ingestion (its ids against the rows it will have after n_new nodes are added), add
        those nodes and make room for it; returns its first edge id. Nothing is written to the device before the batch is
        validated."""
        samp = self._growable_sampler()
        eid0 = samp.next_edge_id if edge_id_start is None else int(edge_id_start)
        check_edges(src, dst, eid0, times, max(samp.num_rows, self.V1 + n_new) if n_new else samp.num_rows, samp.last_time)
        if n_new:
            self.add_nodes(n_new, _edges=(src, dst))
        samp.reserve(src, dst)
        return eid0

    def _arm_ingest(self, h, eid0: int):
        """Arm the stepper to append each batch to the sampler's CSR before its step (lstep_host_stepper_set_ingest). Re-armed
        only when the stepper, the sampler or its arrays changed, or edge ids do not continue: arming makes the next append
        wait for the compute stream, which costs the copy-in its overlap with the previous step."""
        samp = self._host_sampler()
        key = (h.value, id(samp), samp._version)
        if self._armed != key or eid0 != samp.next_edge_id:
            _lib.check(self._libc.lstep_host_stepper_set_ingest(h, _lib.ptr(samp.fill), eid0, samp.last_time),
                       "lstep_host_stepper_set_ingest")
            self._armed = key

    def _disarm_ingest(self, h):
        if self._armed is not None:
            _lib.check(self._libc.lstep_host_stepper_set_ingest(h, None, 0, 0.0), "lstep_host_stepper_set_ingest")
            self._armed = None

    def _set_ingest(self, h, ingest: bool, eid0):
        if ingest:
            self._arm_ingest(h, eid0)
        elif self._armed is not None:
            self._disarm_ingest(h)

    def _host_failed(self, rc: int, what: str, ingest: bool, samp, src, dst, eid0, times):
        """A native host-fed call returned rc != 0: the append of (a prefix of) the batches may have been enqueued before it
        failed, so the sampler takes its state from the device; then raise."""
        if ingest:
            samp._resync(src, dst, eid0, times)
        _lib.check(rc, what)

    # ---- tickets ------------------------------------------------------------------------------------------------------
    def _new_ticket(self, native: int, C: int, n: int) -> int:
        tk = (self._epoch << 32) | native
        self._ticket_shape[tk] = (C, n)
        self._ticket_shape.pop(tk - self.HOST_SLOTS, None)
        self._drained.pop(tk - 2 * self.HOST_SLOTS, None)
        return tk

    def result(self, ticket: int) -> np.ndarray:
        """Per-query row sums [C, n] of step `ticket` (waits for that step's device-to-host copy)."""
        r = self._drained.pop(ticket, None)
        if r is not None:
            return r
        if ticket >> 32 != self._epoch or ticket not in self._ticket_shape:
            raise KeyError(f"result: ticket {ticket} is not outstanding (already read, or overwritten: the last {self.HOST_SLOTS} are kept)")
        return self._result_now(ticket)

    def _result_now(self, ticket: int) -> np.ndarray:
        p = ctypes.POINTER(ctypes.c_float)()
        nf = ctypes.c_int64(0)
        rc = self._libc.lstep_host_step_result(self._host_stepper[0], ticket & 0xFFFFFFFF, C_byref(p), C_byref(nf))
        if rc != 0:
            _lib.check(rc, "lstep_host_step_result")
        C, n = self._ticket_shape[ticket]
        if nf.value == 0:
            return np.zeros((C, n), np.float32)
        return np.ctypeslib.as_array(p, shape=(C, n)).copy()
