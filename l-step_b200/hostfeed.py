"""Host-fed and resident steps: the Python side every history layout shares (PEStream, ChangeLogStream, PeerRank).

A host-fed step hands one batch of HOST (numpy) arrays to a native stepper (csrc/host_step.cu), which packs it into a pinned
slot, copies it in, runs the step and copies the per-query row sums back, and returns a ticket. `HostFed` owns the driver:
step_host_async, step_host, run_host and `result`. A step has two halves: `_host_prepare` validates a batch (or a whole run),
adds the nodes of grow=True and reserves room for ingest=True, writing nothing before all of it has passed; `_host_phase`
issues phases of the step on the prepared batch (all at once, 7, except PeerLocalGroup's 1, 2 and 4 per rank) and moves the
window and the counters (`_advance`). `_step` is the same for a batch of the resident stream, the one uploaded at
construction, whose per-batch plan (peer.batch_plan) a layout adopts with `_adopt_plan`.

It owns the state those steps act on, too: `_new_state` adopts a history (changelog.RingHistory or ChangeLogHistory, which
the layout builds from its own inputs and loads) with a new table `cur`, the step descriptor and the step workspace;
check_errors, history_bytes and export_history read it. And it owns the growth of the node set (add_nodes, and grow=True on
the host-fed steps): new node ids continue after the last live one, and a new node starts with its initial row r0 in the
table, in every history slot and as its change-log base row, which is exactly the state a node no edge has touched has in
a stream built with those rows from the start. So a grown stream computes the bits of the pre-sized one.

A class that mixes it in provides `dev`, `B`, `K`, `d`, `T`, `model`, `start` and the resident stream `src` / `dst` / `t` on
the device, and what differs between layouts: `_host_sampler()`, the sampler its steps read; `_check_host(...)`, its own
checks of a batch; `_host_step_call`, `_host_run_call` and `_step_call`, the native host-fed per-step and multi-batch calls
and the resident per-step call; `share_of(n)`, its share of a batch's queries (all of them on a single GPU)."""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib
from .changelog import advance, filter_len
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
    if len(dst) != n or len(times) != n or [q for q in qs if len(q) != n]:  # (no generator: this runs once per host-fed step)
        raise ValueError(f"{what}: src, dst, times and every query set must have the same length")
    return src, dst, times, qs


class HostFed:
    HOST_SLOTS = 4  # steps that may be in flight before step_host_async blocks on the oldest

    def _host_init(self):
        self.lib = _lib.load()
        self._host_stepper = None
        self._armed = None  # (stepper, sampler, sampler version) the stepper was armed to ingest into, see _set_ingest
        self._ticket_shape = {}
        self._drained = {}  # public ticket -> result read out before its stepper was replaced
        self._epoch = 0

    def _host_sampler(self):
        raise NotImplementedError

    def _stepper(self, n_edges: int, C: int):
        lib = self.lib
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

    def __del__(self):
        st = getattr(self, "_host_stepper", None)
        if st is not None:
            try:
                _lib.load(False).lstep_host_stepper_destroy(st[0])
            except Exception:
                pass
            self._host_stepper = None

    # ---- the state: table, history, step descriptor, workspace --------------------------------------------------------
    def _new_state(self, history):
        """Adopt `history` (history.V1 live rows of history.row_cap) with a new table cur [row_cap, d] for its loader to fill,
        the step descriptor over the resident stream and no workspace yet."""
        self.history, self.V1, self.row_cap = history, history.V1, history.row_cap
        self.cur = torch.empty((self.row_cap, self.d), dtype=torch.float32, device=self.dev)
        self.desc = _lib.PEStreamDesc(self.src.data_ptr(), self.dst.data_ptr(), self.t.data_ptr(), _lib.ptr(history.ring), self.cur.data_ptr(),
                                      self.V1, self.T, self.d, self.row_cap)
        self._ws, self._ws_cap = None, (0, 0, 0)

    def _workspace(self, n_ids: int, n_edges: int, C: int) -> torch.Tensor:
        """The step workspace for n_ids batch nodes, n_edges edges and C query sets: reallocated only when a step needs more
        than it holds, then sized for at least 2B ids, B edges and 4 query sets."""
        cap = self._ws_cap
        if self._ws is not None and n_ids <= cap[0] and n_edges <= cap[1] and C <= cap[2]:
            return self._ws
        need = self.lib.lstep_pe_step_workspace_bytes(n_ids, n_edges, C, self.K, self.d, self.model.time_feat_dim, self.row_cap)
        if self._ws is None or self._ws.numel() < need:
            self._ws_cap = (max(2 * self.B, n_ids), max(self.B, n_edges), max(C, 4))  # (ids, edges, query sets) it is sized for
            self._ws = self._new_workspace(self.row_cap)
        return self._ws

    def _new_workspace(self, row_cap: int) -> torch.Tensor:
        """A zeroed workspace for _ws_cap whose per-node maps cover row_cap rows."""
        n = self.lib.lstep_pe_step_workspace_bytes(*self._ws_cap, self.K, self.d, self.model.time_feat_dim, row_cap) + 4096
        ws = torch.empty(n, dtype=torch.uint8, device=self.dev)
        _lib.check(self.lib.lstep_update_pe_workspace_init(_lib.ptr(ws), n, row_cap, _lib.stream_ptr()), "workspace_init")
        return ws

    def check_errors(self):
        """Synchronising read of the device error flag the step's lookups raise for query ids outside the sampler's
        rows (such a query yields an empty neighbourhood and reads table row 0; nothing is written by query ids).
        Raises IndexError like the reference's lookup (utils/utils.py:140, Q8); LstepError when a step changed more rows
        than a change log's event capacity. Called by export_history(), save_checkpoint() and run(check=True); the
        host-fed calls validate ids on the host before anything is enqueued. Call it yourself after a loop of step()."""
        samp = self._host_sampler()
        self.history.check_full(samp._err, int(samp._err.item()))
        samp.check_errors()

    def history_bytes(self) -> int:
        """Bytes the history occupies: the dense ring, or the change log's base and event rows and index structures."""
        return self.history.nbytes()

    def export_history(self) -> torch.Tensor:
        """The history in the reference's layout [V1, len, d], oldest first (for save_pe / torch.cat; a change log is replayed,
        which needs V1 * len * d * 4 bytes). On a PeerRank, export_history_rows: the owned rows, row l = node l * world + rank."""
        self.check_errors()
        return self.history.replay(self.head, self.len)

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
        """Change-log histories (changelog.ChangeLogOwner): ValueError when a step on V1 nodes could change more rows than the
        log records per step."""

    def _grow_capacity(self, row_cap: int):
        """Reallocate the table, the history and the workspace (if there is one yet) for row_cap rows. Every new buffer is
        allocated before any is swapped in, so that an out-of-memory error leaves the old state whole; the live rows are
        copied on the current stream, behind the steps already enqueued."""
        with torch.cuda.device(self.dev):
            cur = torch.empty((row_cap, self.d), dtype=torch.float32, device=self.dev)
            ws = None if self._ws is None else self._new_workspace(row_cap)
            self.history.grow_capacity(row_cap)
            cur[:self.V1].copy_(self.cur[:self.V1])
        self.cur, self._ws, self.row_cap = cur, ws, int(row_cap)
        self.desc.cur, self.desc.ring, self.desc.row_cap = cur.data_ptr(), _lib.ptr(self.history.ring), self.row_cap

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
            self.history.init_rows(self.cur, v0, v1, rows, stride)
        self.history.add_rows(v1)
        self.V1 = self.desc.V1 = v1
        return v0

    # ---- ingest -------------------------------------------------------------------------------------------------------
    def _growable_sampler(self):
        samp = self._host_sampler()
        if samp is None or not samp.is_growable:
            raise ValueError("ingest=True needs a growable neighbor sampler: model.set_neighbor_sampler(NeighborSampler.growable(...))")
        return samp

    def _set_ingest(self, h, eid0):
        """Arm the stepper to append each batch to the sampler's CSR before its step, with edge ids from eid0 on
        (lstep_host_stepper_set_ingest), or disarm it (eid0 None). Re-armed only when the stepper, the sampler or its arrays
        changed, or edge ids do not continue: arming makes the next append wait for the compute stream, which costs the
        copy-in its overlap with the previous step."""
        if eid0 is None:
            if self._armed is not None:
                _lib.check(self.lib.lstep_host_stepper_set_ingest(h, None, 0, 0.0), "lstep_host_stepper_set_ingest")
                self._armed = None
            return
        samp = self._host_sampler()
        key = (h.value, id(samp), samp._version)
        if self._armed != key or eid0 != samp.next_edge_id:
            _lib.check(self.lib.lstep_host_stepper_set_ingest(h, _lib.ptr(samp.fill), eid0, samp.last_time),
                       "lstep_host_stepper_set_ingest")
            self._armed = key

    # ---- the host-fed step --------------------------------------------------------------------------------------------
    def step_host_async(self, src: np.ndarray, dst: np.ndarray, times: np.ndarray, query_ids, batch_idx: int = None,
                        ids: np.ndarray = None, out: torch.Tensor = None, ingest: bool = False, edge_id_start: int = None,
                        grow: bool = False) -> int:
        """One step fed from HOST arrays (what a loop holding numpy batches calls): the batch's endpoints, times and the query
        id sets are packed into a pinned slot and uploaded by one async copy inside the native call, the step's kernels are
        enqueued behind it, and the per-query row sums of the neighbourhood PEs are copied back to a pinned result slot.
        Returns a ticket at once (nothing synchronises); `result(ticket)` waits for that step only, so a loop can read results
        one step behind. The result is [C, n], or on a PeerRank this rank's share [C, q_rows] (share_of(n)), every rank of the
        group calling it with the same batch. `ids` (sorted unique batch nodes) is computed natively when omitted; `out`
        [C, rows, d] keeps the full neighbourhood PEs on the device. This is the per-batch host path: it avoids every
        avoidable Python call (≈ 25 µs of interpreter time per step).
        A batch is validated before anything is enqueued; on a change-log history (ChangeLogStream, PeerRank) a batch longer
        than batch_size is rejected, since batch_size sizes the log's event capacity.
        ingest=True: the batch's edges are not in the sampler yet. The sampler must be growable (NeighborSampler.growable; a
        PeerRank's own one); room is reserved, and the native call appends the batch to the CSR (edge ids edge_id_start + i,
        default: the sampler's next_edge_id) before the step's lookups run.
        grow=True: ids above the last live one (in the batch or the query sets) are new nodes, added first (add_nodes, with
        the new_node_pe row); without it such an id raises IndexError, as an unknown node does in the reference.
        head / len, batch_idx, steps_done and edges_done (and a PeerRank's epoch) advance as in a resident step."""
        return self._host_phase(self._host_prepare(src, dst, times, query_ids, ids, ingest, edge_id_start, grow), 7, batch_idx, out)

    def step_host(self, src: np.ndarray, dst: np.ndarray, times: np.ndarray, query_ids, batch_idx: int = None, ids: np.ndarray = None,
                  ingest: bool = False, edge_id_start: int = None, grow: bool = False) -> np.ndarray:
        """Synchronous form of step_host_async: the step's per-query row sums [len(query_ids), rows]."""
        return self.result(self.step_host_async(src, dst, times, query_ids, batch_idx, ids, ingest=ingest, edge_id_start=edge_id_start,
                                                grow=grow))

    def run_host(self, src: np.ndarray, dst: np.ndarray, times: np.ndarray, query_ids, ingest: bool = False,
                 edge_id_start: int = None, grow: bool = False) -> np.ndarray:
        """A run of consecutive batches fed from HOST arrays (an evaluation split): batch b is edges [b*B, (b+1)*B) of the given
        arrays; every step copies its own inputs in and its own per-query row sums out. Returns [n_batches, C, B] float32: row
        [b, c, :rows] holds batch b's row sums (a PeerRank's share of them), the rest is zero. While the history is still
        filling (the filter changes with every step) the batches are stepped one by one; the rest goes in ONE native call,
        which reads the results one step behind. The whole run is validated first, as step_host_async validates a batch;
        ingest=True reserves room for all of it first, so the native loop never regrows (on a peer group: no rank synchronises
        while its peers wait at a barrier), and grow=True adds the nodes up to the run's largest id before its first step,
        which changes nothing (they are the rows of a node no edge has touched). A batch the native call rejects raises after
        the batches before it were applied; the host state and the sampler follow the device."""
        n_total, B, C = len(src), self.B, len(query_ids)
        res = np.zeros(((n_total + B - 1) // B, C, B), dtype=np.float32)
        if n_total == 0:
            host_arrays(src, dst, times, query_ids, "run_host")
            return res
        src, dst, times, qs, _, eid0 = self._host_prepare(src, dst, times, query_ids, None, ingest, edge_id_start, grow, n_total)
        lo, pend = 0, []
        while lo < n_total and self.len < self.T:  # the history fills: per-step calls (validated above), results one behind
            hi = min(lo + B, n_total)
            part = (src[lo:hi], dst[lo:hi], times[lo:hi], [q[lo:hi] for q in qs], None, None if eid0 is None else eid0 + lo)
            pend.append((lo // B, self._host_phase(part)))
            if len(pend) > 1:
                b, tk = pend.pop(0)
                r = self.result(tk)
                res[b, :, :r.shape[1]] = r
            lo = hi
        for b, tk in pend:
            r = self.result(tk)
            res[b, :, :r.shape[1]] = r
        if lo == n_total:
            return res
        if torch.cuda.current_device() != self.dev.index:
            torch.cuda.set_device(self.dev)
        h = self._stepper(B, C)
        eid0 = None if eid0 is None else eid0 + lo
        self._set_ingest(h, eid0)
        G = self.model._collapsed_filter(self.T, False)
        qptrs = (C_void_p * max(C, 1))(*[q[lo:].ctypes.data for q in qs])
        done = ctypes.c_int64(0)
        src, dst, times = src[lo:], dst[lo:], times[lo:]
        rc = self._host_run_call(h, n_total - lo, src, dst, times, qptrs, C, G, self._workspace(2 * B, B, C), res[lo // B:], done)
        n_app = min(done.value * B, n_total - lo)  # batches applied before an error stay applied
        self._advance(done.value, n_app, C)
        if rc != 0:  # (the failed batch's append may have been enqueued although its step was not applied)
            self._host_failed(rc, "run_host", src, dst, times, eid0)
        if eid0 is not None and n_app:
            self._host_sampler()._note_ingested(src[:n_app], dst[:n_app], eid0 + n_app - 1, times[n_app - 1])
        return res

    def _host_prepare(self, src, dst, times, query_ids, ids=None, ingest=False, edge_id_start=None, grow=False, n_max=None):
        """First half of a host-fed step: normalise and validate a batch (or a whole run of n_max edges), then, with grow, add
        the nodes up to its largest id and, with ingest, reserve room for its edges in the sampler. Nothing is written before
        all of it has passed. Returns the batch for _host_phase: (src, dst, times, query sets, ids, eid0), eid0 its first edge
        id with ingest, else None."""
        src, dst, times, qs = host_arrays(src, dst, times, query_ids, "step_host" if n_max is None else "run_host")
        n_new = self._new_nodes_for([src, dst] + qs) if grow and len(src) else 0
        samp = self._growable_sampler() if ingest else None
        ids = self._check_host(src, dst, times, qs, ids, self.V1 + n_new, self.B if n_max is None else n_max)
        eid0 = None
        if ingest:
            eid0 = samp.next_edge_id if edge_id_start is None else int(edge_id_start)
            check_edges(src, dst, eid0, times, max(samp.num_rows, self.V1 + n_new) if n_new else samp.num_rows, samp.last_time)
        if n_new:
            self.add_nodes(n_new, _edges=(src, dst) if ingest else None)
        if ingest:
            samp.reserve(src, dst)
        return src, dst, times, qs, ids, eid0

    def _host_phase(self, batch: tuple, phases: int = 7, batch_idx: int = None, out: torch.Tensor = None):
        """Second half: issue `phases` of the step on the prepared batch. The call with bit 0 stages the batch (and appends it
        to the sampler with ingest); the one with bit 2 finishes the step, advances the state and returns the ticket."""
        src, dst, times, qs, ids, eid0 = batch
        n, C = len(src), len(qs)
        if torch.cuda.current_device() != self.dev.index:
            torch.cuda.set_device(self.dev)
        if phases & 1:
            bi = self.batch_idx if batch_idx is None else int(batch_idx)
            h = self._stepper(n, C)
            self._set_ingest(h, eid0)
            G = self.model._collapsed_filter(filter_len(bi, self.len, self.T), False)
            qptrs = (C_void_p * max(C, 1))(*[q.ctypes.data for q in qs])
            ws = self._workspace(2 * n if ids is None else len(ids), n, C)
            if not phases & 4:  # (the later phases reuse them: like the stepper, a rank stages one batch at a time)
                self._staged = (bi, h, G, qptrs, ws, out)
        else:
            bi, h, G, qptrs, ws, out = self._staged
        ticket = ctypes.c_int64(-1)
        rc = self._host_step_call(h, n, src, dst, times, ids, G, qptrs, C, out, ws, phases, ticket)
        if rc != 0:  # (the append may have been enqueued before the step failed)
            self._host_failed(rc, "step_host", src, dst, times, eid0)
        if eid0 is not None and phases & 1:  # the append is enqueued with the staging
            self._host_sampler()._note_ingested(src, dst, eid0 + n - 1, times[-1])
        if not phases & 4:
            return None
        self.batch_idx = bi
        self._advance(1, n, C)
        return self._new_ticket(ticket.value, C, self.share_of(n)[1])

    def _host_failed(self, rc: int, what: str, src, dst, times, eid0):
        """A native host-fed call returned rc != 0: with ingest the append of (a prefix of) the batches may have been enqueued
        before it failed, so the sampler takes its state from the device; then raise."""
        if eid0 is not None:
            self._host_sampler()._resync(src, dst, eid0, times)
        _lib.check(rc, f"{type(self).__name__}.{what}")

    # ---- the resident step: batch b of the edge stream uploaded at construction ----------------------------------------
    def _adopt_plan(self, plan: dict):
        """The per-batch plan of the resident stream (peer.batch_plan) as the attributes the resident step reads; the
        batch node lists are uploaded once."""
        self.num_batches = plan["num_batches"]
        self.batch_lo, self.n_edges, self.batch_tmax, self.ids_off = plan["lo"], plan["n_edges"], plan["tmax"], plan["ids_off"]
        self.ids_np = plan["ids"]
        self.ids = torch.from_numpy(self.ids_np).to(self.dev)

    def _check_stream_ids(self, V1: int):
        """IndexError when the resident stream's batch nodes fall outside the table's V1 rows or the sampler's rows, or the
        sampler knows more rows than the table. Made once, before a layout allocates its state: the resident step reads and
        WRITES table rows by these ids, and the reference raises IndexError for an unknown node at its first lookup (Q8)."""
        ids = self.ids_np
        if not len(ids):
            return
        lo_id, hi_id = int(ids.min()), int(ids.max())
        if lo_id < 0 or hi_id >= V1:
            raise IndexError(f"edge stream holds node id {hi_id if hi_id >= V1 else lo_id} but the PE table has {V1} rows")
        samp = self._host_sampler()
        if samp is not None and hi_id >= samp.num_rows:
            raise IndexError(f"list index out of range: node id {hi_id} is unknown to the neighbor sampler ({samp.num_rows} rows)")
        if samp is not None and samp.num_rows > V1:
            raise IndexError(f"pe has {V1} rows but the sampler knows node ids up to {samp.num_rows - 1}")

    def share_of(self, n: int):
        """(q_off, q_rows): the edges of a batch of n whose a6 queries (and step_host row sums) this layout computes."""
        return 0, n

    def _step(self, b: int, queries, out: torch.Tensor = None, phases: int = 7, batch_idx: int = None) -> torch.Tensor:
        """Issue `phases` of the step on batch b of the resident stream. queries: device int64 tensors with the ids of ALL
        edges of the batch, of which this layout reads its share (share_of). out: a caller buffer, of which a prefix is viewed
        as the result [C, q_rows, d], or None for a new one. The call with bit 2 advances the state, as in _host_phase."""
        lo, n = int(self.batch_lo[b]), int(self.n_edges[b])
        q_off, q_rows = self.share_of(n)
        C = len(queries)
        if out is None:
            out = torch.empty((max(C, 1), q_rows, self.d), dtype=torch.float32, device=self.dev)
        else:
            out = out.view(-1)[:max(C, 1) * q_rows * self.d].view(max(C, 1), q_rows, self.d)
        bi = self.batch_idx if batch_idx is None else batch_idx
        i0, i1 = int(self.ids_off[b]), int(self.ids_off[b + 1])
        with torch.cuda.device(self.dev), torch.no_grad():
            G = self.model._collapsed_filter(filter_len(bi, self.len, self.T), False)
            ws = self._workspace(i1 - i0, n, C)
            qptrs = (C_void_p * max(C, 1))(*[q.data_ptr() + 8 * q_off for q in queries])
            rc = self._step_call(b, lo, n, self.ids.data_ptr() + 8 * i0, i1 - i0, float(self.batch_tmax[b]), G, qptrs, C, q_off, q_rows,
                                 out, ws, phases)
        if rc != 0:
            _lib.check(rc, f"{type(self).__name__}.step")
        if phases & 4:
            self.batch_idx = bi
            self._advance(1, n)
        return out

    def _advance(self, steps: int, edges: int, C: int = None):
        """Move the window (changelog.advance), batch_idx and the step and edge counters by `steps` steps of `edges` edges.
        C: host-fed steps with C query sets, which also count what the stepper copied in (src, dst, t, <= 2n batch ids, C
        query sets)."""
        _, self.head, self.len = advance(self.head, self.len, self.T, steps)
        self.batch_idx += steps
        self.steps_done += steps
        self.edges_done += edges
        if C is not None:
            self.model.h2d_bytes += 8 * edges * (5 + C)

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
        rc = self.lib.lstep_host_step_result(self._host_stepper[0], ticket & 0xFFFFFFFF, C_byref(p), C_byref(nf))
        if rc != 0:
            _lib.check(rc, "lstep_host_step_result")
        C, n = self._ticket_shape[ticket]
        if nf.value == 0:
            return np.zeros((C, n), np.float32)
        return np.ctypeslib.as_array(p, shape=(C, n)).copy()
