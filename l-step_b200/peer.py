"""Peer group: the scale-out PE step over NVLink peer memory (BASELINE config 5: 10 M nodes on 2 / 4 / 8 B200s; SURVEY §8(e)).

One process per GPU. Every rank keeps a replica of the current PE table and of the temporal CSR and OWNS the nodes v with
v % world == rank: their PE history (change log) and every piece of the step whose result is a row of an owned node —
1 / world of the DFT filter, of the a6 query rows, of update_pe's phase A and phase B. Owners copy the rows they change, as
contiguous blocks, into small fixed inbox regions of the other ranks through peer pointers (CUDA IPC over NVLink / NVSwitch);
every rank scatters its inbox into its replica right after the first of the two flag barriers of a step (also in peer memory).
No NCCL call, no host synchronisation and no data-dependent message size is on the step's path. The protocol and the argument why two barriers suffice are in csrc/peer.cu; the C entry points
are lstep_pe_step_peer / lstep_pe_steps_peer (include/lstep_b200.h), and lstep_pe_step_peer_host / lstep_pe_steps_peer_host for
batches fed from host arrays (PeerRank.step_host / run_host, with ingest=True into every rank's own CSR replica).

    PeerRank         this rank's state: table replica, change log of the owned nodes, per-batch plan, peer-shared buffers
    PeerLocalGroup   all ranks of a group in ONE process on one device (tests): peer pointers are plain device pointers and the
                     step is issued phase by phase for every rank
    connect_ipc      one process per GPU (torchrun): exchanges the CUDA IPC handles through torch.distributed and opens them
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib
from .changelog import ChangeLogOwner
from .hostfeed import HostFed, host_arrays
from .model import LSTEP
from .sampler import NeighborSampler, check_edges


class _DevMem:
    """A cudaMalloc'ed block (lstep_ipc_alloc) viewed as a torch tensor through __cuda_array_interface__."""

    def __init__(self, lib, nbytes: int):
        p = ctypes.c_void_p()
        _lib.check(lib.lstep_ipc_alloc(int(nbytes), ctypes.byref(p)), "ipc_alloc")
        self.lib, self.ptr, self.nbytes = lib, int(p.value), int(nbytes)

    def tensor(self, shape, dtype, device):
        typestr = {torch.float32: "<f4", torch.int32: "<i4", torch.uint8: "|u1"}[dtype]

        class _View:
            pass

        v = _View()
        v.__cuda_array_interface__ = {"shape": tuple(int(x) for x in shape), "typestr": typestr, "data": (self.ptr, False), "version": 2,
                                      "strides": None}
        v._keep = self
        return torch.as_tensor(v, device=device)

    def handle(self) -> bytes:
        h = (ctypes.c_ubyte * 64)()
        _lib.check(self.lib.lstep_ipc_export(ctypes.c_void_p(self.ptr), h), "ipc_export")
        return bytes(h)

    def free(self):
        if self.ptr:
            self.lib.lstep_ipc_free(ctypes.c_void_p(self.ptr))
            self.ptr = 0


def batch_plan(src: np.ndarray, dst: np.ndarray, t: np.ndarray, start: int, stop: int, B: int, world: int = 1, rank: int = 0) -> dict:
    """Host-side plan of the resident edge stream: edges [start, stop) of (src, dst, t) in batches of B, for rank `rank` of a
    peer group of `world` (a single GPU is the group of one). Pure numpy: CPU-testable. Per batch b: `lo` its first edge,
    `n_edges`, `tmax` its largest time, `share` the edges [q_off, q_off + q_rows) of it whose a6 queries this rank computes
    (share_of); `ids` the sorted unique batch nodes (replicated on every rank), `mine` the ones this rank owns (v % world ==
    rank), `pos` their positions in the batch's ids (where the owner stores a node's row in the peers' buffers). The lists are
    concatenated, batch b's ids at ids[ids_off[b]:ids_off[b + 1]], its owned ones at mine_off[b]. The owners' lists
    partition each batch's ids, the shares partition the batch."""
    lo = np.arange(start, stop, B, dtype=np.int64)
    n_edges = np.minimum(lo + B, stop) - lo
    ids_l, tmax = [], np.empty(len(lo), np.float64)
    for b, (a, z) in enumerate(zip(lo.tolist(), (lo + n_edges).tolist())):
        ids_l.append(np.unique(np.concatenate([src[a:z], dst[a:z]])))
        tmax[b] = t[a:z].max()
    nb = len(lo)
    ids = np.concatenate(ids_l).astype(np.int64, copy=False) if nb else np.zeros(0, np.int64)
    ids_off = np.concatenate([[0], np.cumsum([len(x) for x in ids_l], dtype=np.int64)])
    own = np.nonzero(ids % world == rank)[0]
    of_batch = np.repeat(np.arange(nb), np.diff(ids_off))[own]
    mine_off = np.concatenate([[0], np.cumsum(np.bincount(of_batch, minlength=nb), dtype=np.int64)])
    return dict(num_batches=nb, lo=lo, n_edges=n_edges, tmax=tmax, share=[share_of(int(n), world, rank) for n in n_edges], ids=ids,
                ids_off=ids_off, mine=ids[own], pos=own - ids_off[of_batch], mine_off=mine_off)


def peer_batch_plan(src: np.ndarray, dst: np.ndarray, batch_size: int, world: int, rank: int) -> dict:
    """batch_plan of the whole of (src, dst) in batches of batch_size for rank `rank` of `world`, where only the node lists
    and the shares are wanted: the times are taken as zero."""
    return batch_plan(src, dst, np.zeros(len(src)), 0, len(src), batch_size, world, rank)


def share_of(n: int, world: int, rank: int):
    """(q_off, q_rows): rank's share of a batch of n edges for the a6 queries; the shares of the ranks partition the batch."""
    return rank * n // world, (rank + 1) * n // world - rank * n // world


def check_host_batch(src, dst, times, query_ids, V1: int, batch_size: int, ids=None, ingest=None):
    """Validation of a host batch for PeerRank.step_host_async, pure numpy (nothing is read from or written to a device). Every
    rank of a group makes it on the same batch, so every rank accepts it or every rank rejects it, before any rank enqueues
    anything. Raises ValueError for an empty batch, unequal lengths, more than 8 query sets, a batch longer than `batch_size`
    (the change log's event capacity and the peer buffers are sized from it) and ids that are not sorted and unique; IndexError
    for a node id outside [0, V1). ingest = (num_rows, last_time, first edge id): the conditions of sampler.check_edges (finite,
    non-decreasing times from last_time on, ids inside the sampler's rows, edge ids inside [0, 2^31)). Returns the arrays as
    host_arrays does, and ids."""
    src, dst, times, qs = host_arrays(src, dst, times, query_ids, "step_host")
    n = len(src)
    if n == 0:
        raise ValueError("step_host: empty batch")
    if n > batch_size:
        raise ValueError(f"PeerRank: a host batch of {n} edges is longer than batch_size ({batch_size}), which sizes the change log's "
                         f"event_capacity and the peer buffers; split the batch or build the ranks with a larger batch_size")
    if len(qs) > 8:
        raise ValueError("step_host: at most 8 query sets")
    for a in [src, dst] + qs:
        lo, hi = int(a.min()), int(a.max())
        if lo < 0 or hi >= V1:
            raise IndexError(f"list index out of range: node id {lo if lo < 0 else hi} is outside the PE table's {V1} rows")
    if ids is not None:
        ids = np.ascontiguousarray(ids, dtype=np.int64)
        if len(ids) > 2 * n or (len(ids) and (int(ids[0]) < 0 or int(ids[-1]) >= V1)) or (len(ids) > 1 and not (np.diff(ids) > 0).all()):
            raise ValueError("step_host: ids must be the sorted unique batch nodes")
    if ingest is not None:
        num_rows, last_time, eid0 = ingest
        check_edges(src, dst, int(eid0), times, num_rows, last_time)
    return src, dst, times, qs, ids


class PeerRank(ChangeLogOwner, HostFed):
    """Rank `rank` of `world` (see the module docstring). src / dst / t: the whole edge stream (replicated, device or host
    arrays); the per-batch plan (sorted unique batch nodes, the owned ones and their positions) of the resident stream
    [start, stop) is computed and its ids are checked once, like PEStream's. src = dst = t = None: no resident stream; the rank then serves host-fed
    steps (step_host_async / step_host / run_host), online with ingest=True into its own growable `sampler`
    (NeighborSampler.growable; every rank holds its own CSR replica, so each rank needs a sampler of its own).

    The PE state comes from exactly one of `initial_pe` (the table [V1, d]), `history` (a dense history [V1, Th, d],
    oldest first, as ChangeLogStream.import_history takes it) and `checkpoint` (a directory that save_checkpoint wrote at
    any world size, or ChangeLogStream.save_checkpoint; or the checkpoint.History that checkpoint.read returned: head, len,
    batch_idx and steps_done continue from it). `batch_idx` overrides the batch index the next step masks the filter with
    while the history is shorter than T (the reference's evaluate loop restarts it at 0: Q5)."""

    def __init__(self, model: LSTEP, rank: int, world: int, src, dst, t, num_nodes: int, batch_size: int, num_neighbors: int,
                 initial_pe: torch.Tensor = None, start: int = 0, stop: int = None, device=None, sampler: NeighborSampler = None,
                 event_capacity: int = None, timeout_ms: int = 4000, history: torch.Tensor = None, checkpoint=None, batch_idx: int = None,
                 row_capacity: int = None, new_node_pe=None, max_nodes: int = None):
        assert 1 <= world <= 16 and 0 <= rank < world
        if (initial_pe is None) + (history is None) + (checkpoint is None) != 2:
            raise ValueError("PeerRank: give exactly one of initial_pe, history and checkpoint")
        self._host_init()
        self.model, self.rank, self.G = model, int(rank), int(world)
        self.dev = dev = torch.device(device) if device is not None else model._dev()
        self.B, self.K, self.T, self.d = int(batch_size), int(num_neighbors), model.num_fft_batches, model.pe_dim
        self.V1 = int(num_nodes) + 1
        self.timeout_ms = int(timeout_ms)
        self._cap_arg, self._row_cap_arg = event_capacity, row_capacity
        self._growth_init(new_node_pe, max_nodes)
        lib = self.lib
        as_dev = lambda a, dt: (torch.zeros(0, dtype=dt, device=dev) if a is None else a.to(dev, dt) if isinstance(a, torch.Tensor) else
                                torch.from_numpy(np.ascontiguousarray(a)).to(dev, dt))
        G, B, d = self.G, self.B, self.d
        with torch.cuda.device(dev):
            self.src, self.dst, self.t = as_dev(src, torch.int64), as_dev(dst, torch.int64), as_dev(t, torch.float64)
            E = int(self.src.shape[0])
            stop = E if stop is None else int(stop)
            self.start, self.stop = int(start), stop
            if sampler is None:
                eid = torch.arange(1, E + 1, dtype=torch.int64, device=dev)
                sampler = NeighborSampler.from_edges(self.src, self.dst, eid, self.t, "recent", device=dev, num_rows=self.V1)
                del eid
            self.sampler = model.neighbor_sampler = sampler
            # ---- per-batch plan of the resident stream: one pass on the host (over [start, stop) only), uploaded once
            part = lambda a: a[self.start:stop].cpu().numpy()
            plan = batch_plan(part(self.src), part(self.dst), part(self.t), 0, stop - self.start, B, G, self.rank)
            plan["lo"] += self.start
            self._adopt_plan(plan)
            self.ids_mine, self.pos_mine = torch.from_numpy(plan["mine"]).to(dev), torch.from_numpy(plan["pos"]).to(dev)
            self.mine_off = plan["mine_off"]
        # ---- the table replica and the change log of the owned nodes; its capacity is the same on every rank: the inbox blocks
        # are laid out by it
        self.batch_idx = 0
        self._start(initial_pe, history, checkpoint, batch_idx, G, self.rank, self.V1)
        with torch.cuda.device(dev):
            # ---- memory the other ranks WRITE (cudaMalloc + CUDA IPC; small fixed regions): phase-A row buffer, filtered-row buffer,
            # inbox (one block per source rank for the rows it changed in a step), barrier flags
            self._mem_rows = _DevMem(lib, 2 * B * d * 4)
            self._mem_filt = _DevMem(lib, 2 * B * d * 4)
            self._mem_inbox = _DevMem(lib, max(int(lib.lstep_peer_inbox_bytes(G, self.cap, d)), 256))
            self._mem_flags = _DevMem(lib, 16 * 4)
            self.new_rows = self._mem_rows.tensor((2 * B, d), torch.float32, dev)
            # the step workspace, sized here (and by growth) for the most check_host_batch lets through, so that no step
            # allocates: a rank must not allocate while its peers wait at a barrier
            self._workspace(2 * B, B, 8)
        self.epoch = ctypes.c_uint32(0)  # (a fresh rank: the flag blocks are zeroed by lstep_ipc_alloc)
        self.grp = None
        self._opened = []

    # ---- node growth (add_nodes and grow=True: hostfeed.HostFed). Every rank of a group calls add_nodes with the same argument
    # and grows its own replica, the change-log rows it owns and its own sampler: no peer holds a pointer into a rank's table or
    # change log (the group shares only the four batch-sized regions of _SHARED), so nothing is exchanged.
    def _grow_capacity(self, row_cap: int):
        super()._grow_capacity(row_cap)
        if self.grp is not None:
            self.grp.table[self.rank] = self.cur.data_ptr()

    def _default_event_cap(self, V1: int) -> int:
        G = self.G
        return min((V1 + G - 1) // G, 2 * (2 * self.B * (self.K + 1) + 2) // G + 1024)

    # ---- group wiring ---------------------------------------------------------------------------------------------------
    _SHARED = ("_mem_rows", "_mem_filt", "_mem_inbox", "_mem_flags")

    def set_group(self, rows, filts, inboxes, flags):
        """Device pointers (ints) of every rank's new_rows buffer / filt buffer / inbox / flag block, indexed by rank."""
        g = _lib.PeerGroup()
        g.rank, g.world, g.cap = self.rank, self.G, self.cap
        for i in range(self.G):
            g.new_rows[i], g.filt[i], g.inbox[i], g.flags[i] = rows[i], filts[i], inboxes[i], flags[i]
        g.table[self.rank] = self.cur.data_ptr()
        self.grp = g

    def local_ptrs(self):
        return tuple(getattr(self, m).ptr for m in self._SHARED)

    def connect_ipc(self, group=None):
        """One process per GPU: exchange the CUDA IPC handles of the four peer-written blocks through torch.distributed and open
        the other ranks' (cudaIpcOpenMemHandle enables peer access over NVLink)."""
        import torch.distributed as dist
        mine = (self.rank,) + tuple(getattr(self, m).handle() for m in self._SHARED)
        allh = [None] * self.G
        if self.G > 1:
            dist.all_gather_object(allh, mine, group=group)
        else:
            allh = [mine]
        ptrs = [[0] * self.G for _ in range(len(self._SHARED))]
        for r, *hs in allh:
            for k, h in enumerate(hs):
                if r == self.rank:
                    ptrs[k][r] = self.local_ptrs()[k]
                else:
                    p = ctypes.c_void_p()
                    buf = (ctypes.c_ubyte * 64).from_buffer_copy(h)
                    with torch.cuda.device(self.dev):
                        _lib.check(self.lib.lstep_ipc_open(buf, ctypes.byref(p)), "ipc_open")
                    self._opened.append(int(p.value))
                    ptrs[k][r] = int(p.value)
        self.set_group(*ptrs)
        if self.G > 1:
            dist.barrier(group=group)

    def close(self):
        torch.cuda.synchronize(self.dev)
        for p in self._opened:
            self.lib.lstep_ipc_close(ctypes.c_void_p(p))
        self._opened = []

    # ---- the step -------------------------------------------------------------------------------------------------------
    def batch(self, b: int):
        lo = int(self.batch_lo[b])
        return lo, lo + int(self.n_edges[b])

    def share(self, b: int):
        """(q_off, q_rows): this rank's share of the batch's edges for the a6 queries."""
        return self.share_of(int(self.n_edges[b]))

    def step(self, b: int, queries, out: torch.Tensor = None, phases: int = 7) -> torch.Tensor:
        """One step on batch b. queries: device int64 tensors with the ids of ALL edges of the batch (this rank reads its
        share). Returns [C, q_rows, d]. phases: see lstep_pe_step_peer (7 = whole step; the state advances with bit 2)."""
        assert self.grp is not None, "set_group / connect_ipc first"
        return self._step(b, queries, out, phases)

    def _step_call(self, b, lo, n, ids, n_ids, tmax, G, qptrs, C, q_off, q_rows, out, ws, phases) -> int:
        m, m0, m1 = self.model, int(self.mine_off[b]), int(self.mine_off[b + 1])
        return self.lib.lstep_pe_step_peer(ctypes.byref(self.desc), self.changelog.ref, self.sampler.csr_ref, ctypes.byref(self.grp), lo, n, ids,
                                           n_ids, self.ids_mine.data_ptr() + 8 * m0, self.pos_mine.data_ptr() + 8 * m0, m1 - m0, tmax, self.head,
                                           self.len, _lib.ptr(G), qptrs, C, q_off, q_rows, _lib.ptr(out), self.K, m._mlp_ref("nbr"),
                                           m._mlp_ref("update"), _lib.ptr(ws), ws.numel(), _lib.ptr(self.sampler._err), self.epoch.value,
                                           self.timeout_ms, phases, _lib.stream_ptr())

    def _advance(self, steps: int, edges: int, C: int = None):
        """HostFed._advance, and the epoch of the step barriers: two per step."""
        super()._advance(steps, edges, C)
        self.epoch = ctypes.c_uint32((self.epoch.value + 2 * steps) & 0xffffffff)

    def run(self, b0: int, n_steps: int, query_arrays, out: torch.Tensor = None, out_step_stride: int = 0):
        """n_steps consecutive steady-state steps (full history) starting at batch b0 in ONE native call (lstep_pe_steps_peer).
        query_arrays: device int64 tensors indexed by GLOBAL edge position (query set c of a step = query_arrays[c][lo:lo+n]).
        out: [C, max q_rows, d] (every step overwrites it) or, with out_step_stride, one block per step."""
        assert self.grp is not None and self.len == self.T and b0 + n_steps <= self.num_batches
        lib, m, d = self.lib, self.model, self.d
        C = len(query_arrays)
        if out is None:
            out = torch.empty((max(C, 1), self.B // self.G + 1, d), dtype=torch.float32, device=self.dev)
        qptrs = (ctypes.c_void_p * max(C, 1))(*[q.data_ptr() for q in query_arrays])
        ap = lambda a: a[b0:].ctypes.data_as(ctypes.c_void_p)
        head, epoch = ctypes.c_int(self.head), ctypes.c_uint32(self.epoch.value)
        with torch.cuda.device(self.dev), torch.no_grad():
            Gt = m._collapsed_filter(self.T, False)
            rc = lib.lstep_pe_steps_peer(ctypes.byref(self.desc), self.changelog.ref, self.sampler.csr_ref, ctypes.byref(self.grp), n_steps,
                                         ap(self.batch_lo), ap(self.n_edges), ap(self.batch_tmax), _lib.ptr(self.ids), ap(self.ids_off),
                                         _lib.ptr(self.ids_mine), _lib.ptr(self.pos_mine), ap(self.mine_off), ctypes.byref(head), _lib.ptr(Gt), qptrs,
                                         ap(self.batch_lo), C, _lib.ptr(out), int(out_step_stride), self.K, m._mlp_ref("nbr"),
                                         m._mlp_ref("update"), _lib.ptr(self._ws), self._ws.numel(), _lib.ptr(self.sampler._err),
                                         ctypes.byref(epoch), self.timeout_ms, _lib.stream_ptr())
        done = ((epoch.value - self.epoch.value) & 0xffffffff) // 2  # (two barrier epochs per applied step)
        self._advance(done, int(self.n_edges[b0:b0 + done].sum()))
        _lib.check(rc, "lstep_pe_steps_peer")
        return out

    # ---- host-fed steps: HostFed's driver (step_host_async / step_host / run_host) around the peer calls of csrc/host_step.cu ---
    def _host_sampler(self):
        return self.sampler  # (this rank's own CSR replica: in a single-process group the ranks share the model)

    def share_of(self, n: int):
        """(q_off, q_rows): this rank's share of a batch of n edges for the a6 queries (and of step_host's row sums)."""
        return share_of(n, self.G, self.rank)

    def _check_host(self, src, dst, times, qs, ids, V1: int, n_max: int):
        """check_host_batch: every rank of a group makes the same checks on the same batch, so either every rank accepts it or
        every rank rejects it, before any rank enqueues anything (a run is validated whole: n_max is its length)."""
        assert self.grp is not None, "set_group / connect_ipc first"
        return check_host_batch(src, dst, times, qs, V1, n_max, ids)[4]

    def _host_step_call(self, h, n, src, dst, times, ids, G, qptrs, C, out, ws, phases, ticket) -> int:
        m, samp = self.model, self.sampler
        return self.lib.lstep_pe_step_peer_host(
            h, ctypes.byref(self.desc), self.changelog.ref, samp.csr_ref, ctypes.byref(self.grp), n, src.ctypes.data, dst.ctypes.data,
            times.ctypes.data, ids.ctypes.data if ids is not None else None, len(ids) if ids is not None else 0, self.head, self.len,
            _lib.ptr(G), qptrs, C, _lib.ptr(out), self.K, m._mlp_ref("nbr"), m._mlp_ref("update"), _lib.ptr(ws), ws.numel(),
            _lib.ptr(samp._err), self.epoch.value, self.timeout_ms, phases, _lib.stream_ptr(), ctypes.byref(ticket))

    def _host_run_call(self, h, n, src, dst, times, qptrs, C, G, ws, res, done) -> int:
        m, samp = self.model, self.sampler
        head, ln, epoch = ctypes.c_int(self.head), ctypes.c_int(self.len), ctypes.c_uint32(self.epoch.value)  # (moved by _advance)
        return self.lib.lstep_pe_steps_peer_host(
            h, ctypes.byref(self.desc), self.changelog.ref, samp.csr_ref, ctypes.byref(self.grp), n, self.B, src.ctypes.data,
            dst.ctypes.data, times.ctypes.data, qptrs, C, ctypes.byref(head), ctypes.byref(ln), _lib.ptr(G), self.K, m._mlp_ref("nbr"),
            m._mlp_ref("update"), _lib.ptr(ws), ws.numel(), _lib.ptr(samp._err), ctypes.byref(epoch), self.timeout_ms, _lib.stream_ptr(),
            res.ctypes.data, ctypes.byref(done))

    def barrier(self):
        """Barrier + application of the inbox: once the kernels this enqueues have run, this replica holds the rows every rank changed
        in the last step."""
        e = (self.epoch.value + 1) & 0xffffffff
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.lstep_peer_sync_tables(ctypes.byref(self.grp), e, self.timeout_ms, _lib.ptr(self.sampler._err), self.d, self.V1,
                                                       _lib.stream_ptr()), "peer_sync_tables")
        self.epoch = ctypes.c_uint32((self.epoch.value + 2) & 0xffffffff)

    def check_errors(self):
        if int(self.sampler._err.item()) & _lib.FLAG_PEER_TIMEOUT:
            self.sampler._err.zero_()
            raise _lib.LstepError("a peer GPU did not reach a step barrier in time (peer group step)")
        super().check_errors()

    export_history_rows = HostFed.export_history  # [rows, len, d], oldest first: row l = node l * G + rank


class PeerLocalGroup:
    """All ranks of a group in one process on one device (tests): the peer pointers are the rank states' own device pointers
    and every phase of a step is issued for all ranks before the next one (the barriers are then already satisfied)."""

    def __init__(self, ranks):
        self.ranks, self.G = ranks, len(ranks)
        assert len({rk.cap for rk in ranks}) == 1
        ptrs = [[rk.local_ptrs()[k] for rk in ranks] for k in range(len(PeerRank._SHARED))]
        for rk in ranks:
            rk.set_group(*ptrs)

    def step_host(self, src, dst, times, queries, ingest: bool = False, edge_id_start: int = None, batch_idx: int = None,
                  grow: bool = False) -> np.ndarray:
        """PeerRank.step_host for every rank on the same host batch: validated for all ranks before any rank stages anything,
        then phases 1, 2 and 4 issued for every rank. Returns the shares concatenated, [C, n]: the single-GPU result. grow=True:
        every rank adds the nodes up to the batch's largest id first."""
        hbs = [rk._host_prepare(src, dst, times, queries, None, ingest, edge_id_start, grow) for rk in self.ranks]
        tks = [None] * self.G
        for ph in (1, 2, 4):
            for i, rk in enumerate(self.ranks):
                tks[i] = rk._host_phase(hbs[i], ph, batch_idx)
        return np.concatenate([rk.result(tk) for rk, tk in zip(self.ranks, tks)], axis=1)

    def step(self, b: int, queries):
        outs = [None] * self.G
        for ph in (1, 2, 4):
            for i, rk in enumerate(self.ranks):
                o = rk.step(b, queries, out=outs[i], phases=ph)
                outs[i] = o
        return outs

    def barrier(self):
        for rk in self.ranks:
            e = (rk.epoch.value + 1) & 0xffffffff
            _lib.check(rk.lib.lstep_peer_signal(ctypes.byref(rk.grp), e, _lib.stream_ptr()), "peer_signal")
        for rk in self.ranks:
            rk.barrier()
