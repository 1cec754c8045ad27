"""Node-id sharded PE state for graphs beyond one GPU's working set (BASELINE config 5: 10 M nodes,
SURVEY §8(e)). One process per GPU; rank r of G owns the nodes v with v % G == r:

    sharded   PE history ring   float32[V1/G][T][d]   (the 688 GB object at T=100, d=172)
    sharded   temporal CSR      rows of owned nodes, neighbour ids stay global
    cached    current table     float32[V1][d] on every rank (6.9 GB at 10 M nodes): owned rows are
                                authoritative, other rows are refreshed on demand

The batch is replicated; compute is owner-local and the single-GPU kernels run unchanged on global
ids. A step has two row exchanges (NCCL all-to-all over NVLink):

    p1  DFT filter of owned batch nodes -> table; neighbour lookup for owned query rows
    X1  request / response of the table rows this rank will read but does not own
        (sampled neighbours of its query rows, other endpoints of its batch nodes' edges)
    p2  neighbourhood PE of owned query rows; update phase A of owned batch nodes (in place);
        update phase B aggregation for the (node, time) pairs it owns -> partial rows per destination
    X2  partial aggregate rows -> owners of the destinations
    p3  fixed-order sum of the partials per destination, MLP, in-place write of owned rows; ring append

`LocalGroup` runs all ranks of a group inside one process on one device (lock-step, exchanges are
tensor copies) — that is how the sharded algorithm is tested on a single GPU; `DistGroup` is the
torch.distributed implementation (NCCL on GPUs; gloo in the CPU tests of the exchange layer).
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib
from . import checkpoint as ckpt
from .changelog import ChangeLogHistory, advance, filter_len
from .model import LSTEP
from .peer import batch_plan
from .sampler import NeighborSampler


# ---------------------------------------------------------------------------------------------
# host-side partition plan (pure numpy: CPU-testable)
# ---------------------------------------------------------------------------------------------
def owner_of(ids, world: int):
    return ids % world


def plan_batch(ids: np.ndarray, src: np.ndarray, dst: np.ndarray, world: int, rank: int) -> dict:
    """What rank `rank` does for a batch whose sorted unique nodes are `ids`:
    pos      positions i (into ids) of the nodes it owns — phase-B pairs (ids[i], times[i]) need i (Q1b)
    mine     those node ids (global), local = mine // world
    n_valid  how many of them have i < min(len(ids), len(src))  (zip truncation, Q1)
    others   other endpoints of the batch edges incident to its nodes that it does not own (phase-A reads)
    """
    pos = np.nonzero(owner_of(ids, world) == rank)[0].astype(np.int64)
    mine = ids[pos]
    n_valid = int(np.count_nonzero(pos < min(len(ids), len(src))))
    s_m, d_m = owner_of(src, world) == rank, owner_of(dst, world) == rank
    others = np.unique(np.concatenate([dst[s_m], src[d_m]]))
    others = others[owner_of(others, world) != rank]
    return dict(pos=pos, mine=mine, local=mine // world, n_valid=n_valid, others=others.astype(np.int64))


def plan_queries(queries, world: int, rank: int):
    """Rows (set c, position i) of the C query sets whose node this rank owns: flat row index c*B+i."""
    flat = np.concatenate(queries) if len(queries) else np.zeros(0, np.int64)
    rows = np.nonzero(owner_of(flat, world) == rank)[0].astype(np.int64)
    return rows, flat[rows]


def group_by_owner(ids: torch.Tensor, world: int):
    """Stable grouping of ids by owner: (ids sorted by owner, counts[world] on the host)."""
    own = ids % world
    order = torch.sort(own, stable=True).indices
    counts = torch.bincount(own, minlength=world).cpu().tolist()
    return ids[order], order, counts


# ---------------------------------------------------------------------------------------------
# exchange layer
# ---------------------------------------------------------------------------------------------
class DistGroup:
    """all-to-all-v over torch.distributed (one process per rank)."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist, self.group = dist, group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)

    def alltoallv(self, send: torch.Tensor, counts, recv_counts=None):
        """send: rows grouped by destination rank (counts[r] rows for rank r). Returns (recv rows grouped by
        source rank, recv counts). When the receive counts are already known (the reply of a request, a
        second payload with the same split) the count exchange and its host sync are skipped."""
        dist = self.dist
        dev = send.device
        if recv_counts is None:
            c_out = torch.tensor(counts, dtype=torch.int64, device=dev)
            c_in = torch.empty_like(c_out)
            dist.all_to_all_single(c_in, c_out, group=self.group)
            rc = c_in.cpu().tolist()
        else:
            rc = list(recv_counts)
        recv = torch.empty((sum(rc),) + tuple(send.shape[1:]), dtype=send.dtype, device=dev)
        dist.all_to_all_single(recv, send.contiguous(), output_split_sizes=rc, input_split_sizes=list(counts), group=self.group)
        return recv, rc

    def allreduce_sum(self, x: torch.Tensor):
        self.dist.all_reduce(x, group=self.group)
        return x


def fetch_rows(comm, table: torch.Tensor, need_sorted: torch.Tensor, counts, world: int):
    """Request/response: ask the owners for rows `need_sorted` (grouped by owner) of their table and store
    them into this rank's copy. Every rank of the group must call it (collective)."""
    req, rc = comm.alltoallv(need_sorted, counts)      # ids other ranks ask me for
    rows = table.index_select(0, req)                  # my authoritative rows
    got, _ = comm.alltoallv(rows, rc, recv_counts=counts)  # rows I asked for, in the order I asked
    if need_sorted.numel():
        table.index_copy_(0, need_sorted, got)
    return int(need_sorted.numel()), int(req.numel())


# ---------------------------------------------------------------------------------------------
class ShardRank:
    """State and per-phase compute of one rank."""

    def __init__(self, model: LSTEP, rank: int, world: int, src_np, dst_np, t_np, eid_np, num_nodes: int, batch_size: int,
                 num_neighbors: int, initial_pe: torch.Tensor, start: int = 0, stop: int = None, device=None, T: int = None):
        self.m, self.rank, self.G = model, rank, world
        self.dev = dev = torch.device(device) if device is not None else model._dev()
        self.B, self.K = int(batch_size), int(num_neighbors)
        self.T = model.num_fft_batches if T is None else int(T)
        assert self.T == model.num_fft_batches
        self.d, self.t = model.pe_dim, model.time_feat_dim
        self.V1 = int(num_nodes) + 1
        stop = len(src_np) if stop is None else stop
        self.start, self.stop = int(start), int(stop)
        self.src_np = np.ascontiguousarray(src_np, dtype=np.int64)
        self.dst_np = np.ascontiguousarray(dst_np, dtype=np.int64)
        self.t_np = np.ascontiguousarray(t_np, dtype=np.float64)
        lib = self.lib = _lib.load()
        with torch.cuda.device(dev):
            self.src = torch.from_numpy(self.src_np).to(dev)
            self.dst = torch.from_numpy(self.dst_np).to(dev)
            self.tt = torch.from_numpy(self.t_np).to(dev)
            eid = torch.from_numpy(np.ascontiguousarray(eid_np, dtype=np.int64)).to(dev)
            # adjacency entries of owned nodes, in the reference's insertion order (utils/utils.py:297-299)
            owner = torch.stack([self.src, self.dst], 1).reshape(-1)
            keep = (owner % world) == rank
            nbr = torch.stack([self.dst, self.src], 1).reshape(-1)[keep]
            e2 = eid.repeat_interleave(2)[keep]
            t2 = self.tt.repeat_interleave(2)[keep]
            owner_local = owner[keep] // world
            self.rows_local = (self.V1 - rank + world - 1) // world  # owned node ids: rank, rank+G, ...
            self.sampler = NeighborSampler.__new__(NeighborSampler)
            NeighborSampler.__init__(self.sampler, None, "recent", 0.0, None, dev, _csr_tensors=())
            self.sampler._build("lstep_csr_build_from_entries", (owner_local, nbr, e2, t2), int(owner_local.numel()),
                                int(owner_local.numel()), max(self.rows_local, 1))
            del owner, keep, nbr, e2, t2, owner_local, eid
            self.cur = initial_pe.to(dev, torch.float32).clone().contiguous()
            assert tuple(self.cur.shape) == (self.V1, self.d)
            self.ring = torch.zeros((max(self.rows_local, 1), self.T, self.d), dtype=torch.float32, device=dev)
            self.head, self.len = 0, 1
            _lib.check(lib.lstep_ring_copy_rows(_lib.ptr(self.ring), _lib.ptr(self.cur), self.rows_local, self.T, self.d, 0, world, rank,
                                                1, _lib.stream_ptr()), "ring init")
            need = lib.lstep_update_pe_workspace_bytes(2 * self.B, self.B, self.K, self.d, self.t, self.V1)
            self.ws = torch.empty(need + 4096, dtype=torch.uint8, device=dev)
            _lib.check(lib.lstep_update_pe_workspace_init(_lib.ptr(self.ws), self.ws.numel(), self.V1, _lib.stream_ptr()), "ws init")
        self.err = torch.zeros(1, dtype=torch.int32, device=dev)
        self.batch_idx = 0
        pk = model._packed_mlp("update")
        self._noself = _lib.PEMLP(pk.w1, pk.b1, pk.w2, pk.b2, None, None, pk.tw, pk.d, pk.t, pk.w1_tc, pk.w2_tc, None)  # phase B: no self term (Q3)
        self.bytes_x1 = self.bytes_x2 = 0

    # ---- helpers ------------------------------------------------------------------------------
    def _up(self, arrays):
        return self.m._upload(arrays) if self.m._dev() == self.dev else [torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(self.dev)
                                                                         for a, dt in arrays]

    def batch(self, b: int):
        lo = self.start + b * self.B
        hi = min(lo + self.B, self.stop)
        return lo, hi

    # ---- p1 -------------------------------------------------------------------------------------
    def p1(self, b: int, queries):
        lib, G, r, K, d = self.lib, self.G, self.rank, self.K, self.d
        lo, hi = self.batch(b)
        src, dst, tt = self.src_np[lo:hi], self.dst_np[lo:hi], self.t_np[lo:hi]
        ids = np.unique(np.concatenate([src, dst]))
        pl = plan_batch(ids, src, dst, G, r)
        q_rows, q_ids = plan_queries(queries, G, r)
        nB = hi - lo
        q_tpos = q_rows % nB
        I64, F64 = np.dtype(np.int64), np.dtype(np.float64)
        # times paired with owned phase-B sources: times[pos] (clamped; rows >= n_valid are never looked up)
        tpos = np.minimum(pl["pos"], nB - 1)
        up = self._up([(pl["mine"], I64), (pl["local"], I64), (pl["others"], I64), (q_ids, I64), (q_ids // G, I64), (tt[q_tpos], F64),
                       (tt[tpos], F64), (q_rows, I64)])
        st = dict(b=b, lo=lo, hi=hi, nB=nB, n_ids_all=len(ids), tmax=float(tt.max()), pl=pl)
        (st["mine"], st["local"], st["others"], st["q_ids"], st["q_local"], st["q_t"], st["src_t"], st["q_rows"]) = up
        T = self.T
        bmask = min(max(self.batch_idx, 0), T) if self.len < T else T
        with torch.cuda.device(self.dev), torch.no_grad():
            n_mine = st["mine"].shape[0]
            if n_mine:
                Gt = self.m._collapsed_filter(bmask, False)
                _lib.check(lib.lstep_dft_filter_scatter(_lib.ptr(self.ring), T * d, d, self.head, T, self.len, d, _lib.ptr(st["local"]),
                                                        _lib.ptr(st["mine"]), n_mine, _lib.ptr(Gt), _lib.ptr(self.cur), d,
                                                        _lib.stream_ptr()), "dft_filter_scatter")
            nq = st["q_ids"].shape[0]
            if nq:
                st["nbr"], st["nt"] = self.sampler.sample_device(st["q_local"], st["q_t"], nq, nq, K)
                nb = st["nbr"].reshape(-1).to(torch.int64)
                need = torch.cat([nb[(nb % G) != r], st["others"]])
            else:
                need = st["others"]
            need = torch.unique(need)
            st["need"], _, st["need_counts"] = group_by_owner(need, G)
        return st

    # ---- p2 -------------------------------------------------------------------------------------
    def p2(self, st, out_full: torch.Tensor):
        """out_full: zero-initialised [C*B_b, d]; this rank writes the rows it owns."""
        lib, G, r, K, d, t = self.lib, self.G, self.rank, self.K, self.d, self.t
        m = self.m
        with torch.cuda.device(self.dev), torch.no_grad():
            nq = st["q_ids"].shape[0]
            if nq:
                o = torch.empty((nq, d), dtype=torch.float32, device=self.dev)
                ws = torch.empty(nq * (d + t + 3), dtype=torch.float32, device=self.dev)
                _lib.check(lib.lstep_neighborhood_pe(_lib.ptr(self.cur), self.V1, _lib.ptr(st["q_ids"]), _lib.ptr(st["q_t"]),
                                                     _lib.ptr(st["nbr"]), _lib.ptr(st["nt"]), nq, K, m._mlp_ref("nbr"), _lib.ptr(o),
                                                     _lib.ptr(ws), ws.numel() * 4, _lib.stream_ptr()), "lstep_neighborhood_pe")
                out_full.index_copy_(0, st["q_rows"], o)
            n_mine = st["mine"].shape[0]
            lo, hi = st["lo"], st["hi"]
            st["send_u"], st["send_rows"], st["send_counts"] = (torch.zeros(0, dtype=torch.int64, device=self.dev),
                                                                torch.zeros((0, d + t), dtype=torch.float32, device=self.dev), [0] * G)
            if n_mine == 0:
                return st
            _lib.check(lib.lstep_update_pe_phase_a(_lib.ptr(self.cur), self.V1, _lib.ptr(st["mine"]), n_mine, _lib.ptr(self.src[lo:hi]),
                                                   _lib.ptr(self.dst[lo:hi]), _lib.ptr(self.tt[lo:hi]), st["nB"], st["tmax"], K,
                                                   m._mlp_ref("update"), _lib.ptr(self.ws), self.ws.numel(), _lib.stream_ptr()),
                       "phase_a")
            _lib.check(lib.lstep_update_pe_phase_b_partial(_lib.ptr(self.cur), self.V1, self.sampler.csr_ref, _lib.ptr(st["local"]),
                                                           _lib.ptr(st["mine"]), n_mine, _lib.ptr(st["src_t"]), st["pl"]["n_valid"],
                                                           st["nB"], st["tmax"], K, m._mlp_ref("update"), _lib.ptr(self.ws),
                                                           self.ws.numel(), _lib.ptr(self.err), _lib.stream_ptr()), "phase_b_partial")
            offs = (ctypes.c_int64 * 4)()
            _lib.check(lib.lstep_update_pe_workspace_layout(n_mine, st["nB"], K, d, t, self.V1, offs), "layout")
            counters = self.ws[offs[0]:offs[0] + 32].view(torch.int32)
            M, hz = counters[:2].cpu().tolist()
            n = M + (1 if hz else 0)
            lda = int(offs[3])
            U = self.ws[offs[1]:offs[1] + 8 * n].view(torch.int64)
            A = self.ws[offs[2]:offs[2] + 4 * n * lda].view(torch.float32).view(n, lda)[:, :d + t]
            u_sorted, order, counts = group_by_owner(U, G)
            st["send_u"], st["send_rows"], st["send_counts"] = u_sorted, A.index_select(0, order).contiguous(), counts
        return st

    # ---- p3 -------------------------------------------------------------------------------------
    def p3(self, st, recv_u: torch.Tensor, recv_rows: torch.Tensor):
        lib, G, r, d, t = self.lib, self.G, self.rank, self.d, self.t
        with torch.cuda.device(self.dev), torch.no_grad():
            if r == 0:
                self.cur[0].zero_()  # pe[0] = 0 before the phase-B write-back (LSTEP.py:317)
            if recv_u.numel():
                srt = torch.sort(recv_u, stable=True)  # partials of one destination stay in source-rank order
                uniq, cnt = torch.unique_consecutive(srt.values, return_counts=True)
                seg = torch.zeros(uniq.numel() + 1, dtype=torch.int64, device=self.dev)
                seg[1:] = torch.cumsum(cnt, 0)
                rows = recv_rows.index_select(0, srt.indices).contiguous()
                n_u = uniq.numel()
                A = torch.empty((n_u, d + t), dtype=torch.float32, device=self.dev)
                _lib.check(lib.lstep_segment_sum_rows(_lib.ptr(rows), d + t, _lib.ptr(seg), n_u, d + t, _lib.ptr(A), d + t,
                                                      _lib.stream_ptr()), "segment_sum_rows")
                _lib.check(lib.lstep_pe_mlp_apply(_lib.ptr(A), _lib.ptr(self.cur), _lib.ptr(uniq), n_u, ctypes.byref(self._noself), None, d,
                                                  _lib.ptr(self.cur), _lib.stream_ptr()), "phase_b apply")
            T = self.T
            if self.len < T:
                slot, self.len = (self.head + self.len) % T, self.len + 1
            else:
                slot, self.head = self.head, (self.head + 1) % T
            _lib.check(lib.lstep_ring_copy_rows(_lib.ptr(self.ring), _lib.ptr(self.cur), self.rows_local, T, d, slot, G, r, 1,
                                                _lib.stream_ptr()), "ring append")
        self.batch_idx += 1

    def owned_table(self) -> torch.Tensor:
        """Authoritative rows of this rank, [rows_local, d], row l = node l*G + rank."""
        return self.cur[self.rank::self.G]


# ---------------------------------------------------------------------------------------------
class LocalGroup:
    """All G ranks in one process on one device, in lock step (tests; exchanges are tensor copies)."""

    def __init__(self, ranks):
        self.ranks = ranks
        self.G = len(ranks)

    @staticmethod
    def _a2a(send, counts):
        """send[r]: rows of rank r grouped by destination, counts[r][dest]. Returns recv[dest] grouped by source
        and the receive counts."""
        G = len(send)
        offs = [np.concatenate([[0], np.cumsum(c)]) for c in counts]
        recv, rc = [], []
        for dest in range(G):
            parts = [send[r][offs[r][dest]:offs[r][dest + 1]] for r in range(G)]
            recv.append(torch.cat(parts) if parts else send[0][:0])
            rc.append([int(p.shape[0]) for p in parts])
        return recv, rc

    def step(self, b: int, queries):
        R, G = self.ranks, self.G
        sts = [rk.p1(b, queries) for rk in R]
        # X1: request / response
        req, rc = self._a2a([s["need"] for s in sts], [s["need_counts"] for s in sts])
        rows = [R[r].cur.index_select(0, req[r]) for r in range(G)]
        got, _ = self._a2a(rows, rc)
        for r in range(G):
            if sts[r]["need"].numel():
                R[r].cur.index_copy_(0, sts[r]["need"], got[r])
        nB = sts[0]["nB"]
        outs = [torch.zeros((len(queries) * nB, R[0].d), dtype=torch.float32, device=R[0].dev) for _ in range(G)]
        sts = [R[r].p2(sts[r], outs[r]) for r in range(G)]
        out = outs[0]
        for o in outs[1:]:
            out += o
        ru, _ = self._a2a([s["send_u"] for s in sts], [s["send_counts"] for s in sts])
        rr, _ = self._a2a([s["send_rows"] for s in sts], [s["send_counts"] for s in sts])
        for r in range(G):
            R[r].p3(sts[r], ru[r], rr[r])
        return out.view(len(queries), nB, R[0].d)

    def gather_table(self) -> torch.Tensor:
        """The full current table assembled from the owners' rows."""
        R = self.ranks
        full = torch.empty_like(R[0].cur)
        for rk in R:
            full[rk.rank::rk.G] = rk.cur[rk.rank::rk.G]
        return full


class ShardedPEStream:
    """One process per GPU (torchrun): this rank's shard + the torch.distributed exchanges."""

    def __init__(self, rank_state: ShardRank, comm: DistGroup):
        self.rk, self.comm = rank_state, comm

    def step(self, b: int, queries):
        rk, comm = self.rk, self.comm
        st = rk.p1(b, queries)
        n_req, n_served = fetch_rows(comm, rk.cur, st["need"], st["need_counts"], rk.G)
        rk.bytes_x1 += (n_req + n_served) * (rk.d * 4 + 8)
        out = torch.zeros((len(queries) * st["nB"], rk.d), dtype=torch.float32, device=rk.dev)
        st = rk.p2(st, out)
        comm.allreduce_sum(out)  # every row is non-zero on exactly one rank: an exact, order-free combine
        ru, rc = comm.alltoallv(st["send_u"], st["send_counts"])
        rr, _ = comm.alltoallv(st["send_rows"], st["send_counts"], recv_counts=rc)
        rk.bytes_x2 += int(st["send_rows"].numel() * 4 + rr.numel() * 4)
        rk.p3(st, ru, rr)
        return out.view(len(queries), st["nB"], rk.d)


# =============================================================================================
# Replicated table, sharded history (the default scale-out layout of bench.py --workload scaleout)
# =============================================================================================
class ReplicatedTableRank:
    """Rank r of G for graphs whose PE HISTORY does not fit one GPU (BASELINE config 5: 10 M nodes; the history ring is
    V1 x T x d x 4 B = 688 GB at T = 100, the current table 6.9 GB, the temporal CSR of 5e8 edges 16 GB):

        sharded      history ring   float32[V1/G][T][d]      rows of the nodes v with v % G == r (spreads hubs)
        replicated   current table  float32[V1][d], temporal CSR, resident edge stream

    Per step the only data one rank needs from another is the DFT-filtered row of the batch nodes whose history it does
    not hold, so a step is
        p1   DFT filter (a3) of the OWNED batch nodes off the local ring                      1/G of the filter's HBM traffic
        X    one NCCL all-gather of the filtered rows (N x d x 4 B = 1.7 MB at B = 2000), scattered into every replica
        p2   lstep_pe_step_sharded: a6 for this rank's 1/G share of the query rows; update_pe (a7 / a8) in full on every
             rank — identical inputs and deterministic kernels keep the table replicas bit-identical with no exchange;
             ring append of the owned rows
    with NO host synchronisation and no data-dependent message sizes: which rank owns which batch node follows from the
    (replicated) batch, so every split size is known on the host of every rank, and the per-batch plan (sorted unique
    ids, owned ids, scatter order) is computed once for the whole resident stream like PEStream's. Compared with the
    owner-computes / all-to-all layout above (table sharded too; kept as ShardRank for reference and tested against this
    one) it trades 1/G of the update's arithmetic for the removal of two data-dependent all-to-all exchanges whose
    host-side planning cost 10x the step's kernels."""

    def __init__(self, model: LSTEP, rank: int, world: int, src, dst, t, num_nodes: int, batch_size: int, num_neighbors: int,
                 initial_pe: torch.Tensor, start: int = 0, stop: int = None, device=None, sampler: NeighborSampler = None,
                 history: str = "ring", event_capacity: int = None):
        """history: "ring" = dense ring of the owned nodes' snapshots (V1/G x T rows); "changelog" = change-log history of the
        owned nodes (csrc/changelog.cu: V1/G base rows + the owned rows every step changed), which holds T = 100 for the
        10 M-node graph on ONE GPU and writes ~9 MB per step instead of one row per owned node."""
        assert history in ("ring", "changelog")
        self.history = history
        self.m, self.rank, self.G = model, int(rank), int(world)
        self.dev = dev = torch.device(device) if device is not None else model._dev()
        self.B, self.K, self.T = int(batch_size), int(num_neighbors), model.num_fft_batches
        self.d, self.t_dim = model.pe_dim, model.time_feat_dim
        self.V1 = int(num_nodes) + 1
        lib = self.lib = _lib.load()
        as_dev = lambda a, dt: (a.to(dev, dt) if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a)).to(dev, dt))
        with torch.cuda.device(dev):
            self.src, self.dst, self.tt = as_dev(src, torch.int64), as_dev(dst, torch.int64), as_dev(t, torch.float64)
            E = int(self.src.shape[0])
            stop = E if stop is None else int(stop)
            self.start, self.stop = int(start), stop
            if sampler is None:
                eid = torch.arange(1, E + 1, dtype=torch.int64, device=dev)
                sampler = NeighborSampler.from_edges(self.src, self.dst, eid, self.tt, "recent", device=dev, num_rows=self.V1)
                del eid
            self.sampler = model.neighbor_sampler = sampler
            # table with one spare row: padded slots of the all-gather are scattered there
            self._cur_full = torch.empty((self.V1 + 1, self.d), dtype=torch.float32, device=dev)
            self._cur_full[:self.V1] = initial_pe.to(dev, torch.float32)
            self._cur_full[self.V1].zero_()
            self.cur = self._cur_full[:self.V1]
            self.rows_local = ckpt.rows_of(self.V1, self.G, self.rank)  # owned node ids: rank, rank + G, ...
            self.head, self.len = 0, 1
            if history == "ring":
                self.ring = torch.zeros((max(self.rows_local, 1), self.T, self.d), dtype=torch.float32, device=dev)
                _lib.check(lib.lstep_ring_copy_rows(_lib.ptr(self.ring), _lib.ptr(self.cur), self.rows_local, self.T, self.d, 0, self.G, self.rank, 1,
                                                    _lib.stream_ptr()), "ring init")
                ring_ptr = self.ring.data_ptr()
            else:
                cap = event_capacity if event_capacity is not None else min(self.rows_local, 2 * (2 * int(batch_size) * (self.K + 1) + 2) // self.G + 1024)
                self.changelog = ChangeLogHistory(self.V1, self.T, self.d, cap, self.G, self.rank, dev)
                self.cap = self.changelog.cap
                self.changelog.reset(self.cur)
                self.ring = None
                ring_ptr = None
            self.desc = _lib.PEStreamDesc(self.src.data_ptr(), self.dst.data_ptr(), self.tt.data_ptr(), ring_ptr, self.cur.data_ptr(),
                                          self.V1, self.T, self.d)
            # ---- per-batch plan of the resident stream [start, stop) (batch_plan) and the scatter lists of the all-gather:
            # one pass on the host, uploaded once
            B, G = self.B, self.G
            part = lambda a: a[self.start:stop].cpu().numpy()
            plan = batch_plan(part(self.src), part(self.dst), part(self.tt), 0, stop - self.start, B, G, self.rank)
            self.num_batches, self.ids_off, self.mine_off, self.tmax = plan["num_batches"], plan["ids_off"], plan["mine_off"], plan["tmax"]
            scat_l, self.scat_off, self.max_n = [], [0], []
            for b in range(self.num_batches):
                ids = plan["ids"][self.ids_off[b]:self.ids_off[b + 1]]
                own = ids % G
                counts = np.bincount(own, minlength=G)
                mx = max(int(counts.max()), 1)
                scat = np.full((G, mx), self.V1, dtype=np.int64)  # padded slots -> the spare row
                for g in range(G):
                    scat[g, :counts[g]] = ids[own == g]
                scat_l.append(scat.reshape(-1))
                self.scat_off.append(self.scat_off[-1] + scat.size)
                self.max_n.append(mx)
            up = lambda a: torch.from_numpy(a).to(dev)
            mine = plan["mine"] // G if history == "ring" else plan["mine"]  # ring rows / global ids
            self.ids, self.mine_local = up(plan["ids"]), up(mine)
            self.scat = up(np.concatenate(scat_l) if scat_l else np.zeros(0, np.int64))
            if len(plan["ids"]) and int(plan["ids"].max()) >= self.V1:
                raise IndexError("edge stream holds a node id outside the PE table")
            need = lib.lstep_pe_step_workspace_bytes(2 * B, B, 8, self.K, self.d, self.t_dim, self.V1)
            self.ws = torch.empty(need + 4096, dtype=torch.uint8, device=dev)
            _lib.check(lib.lstep_update_pe_workspace_init(_lib.ptr(self.ws), self.ws.numel(), self.V1, _lib.stream_ptr()), "ws init")
            self._gbuf = torch.empty((G * 2 * B, self.d), dtype=torch.float32, device=dev)  # all-gather buffer (>= G * max_n rows)
            self._mine = torch.empty((2 * B, self.d), dtype=torch.float32, device=dev)
        self.batch_idx = 0
        self.bytes_allgather = 0

    def batch(self, b: int):
        lo = self.start + b * self.B
        return lo, min(lo + self.B, self.stop)

    def share(self, b: int):
        """(q_off, q_rows): this rank's share of the batch's edges for the a6 queries."""
        lo, hi = self.batch(b)
        n = hi - lo
        return self.rank * n // self.G, (self.rank + 1) * n // self.G - self.rank * n // self.G

    # ---- p1: filter the owned batch nodes off the local ring into a padded send block -----------------------------------
    def p1(self, b: int) -> torch.Tensor:
        lib, T, d = self.lib, self.T, self.d
        n_mine = self.mine_off[b + 1] - self.mine_off[b]
        mx = self.max_n[b]
        send = self._mine[:mx]
        with torch.cuda.device(self.dev), torch.no_grad():
            if n_mine:
                Gt = self.m._collapsed_filter(filter_len(self.batch_idx, self.len, T), False)
                loc = self.mine_local[self.mine_off[b]:self.mine_off[b + 1]]
                if self.history == "ring":
                    _lib.check(lib.lstep_dft_filter(_lib.ptr(self.ring), T * d, d, self.head, T, self.len, d, _lib.ptr(loc), n_mine, _lib.ptr(Gt),
                                                    _lib.ptr(send), d, _lib.stream_ptr()), "dft_filter")
                else:
                    _lib.check(lib.lstep_changelog_filter(self.changelog.ref, self.head, self.len, _lib.ptr(loc), n_mine, _lib.ptr(Gt), _lib.ptr(send),
                                                          d, None, _lib.stream_ptr()), "changelog_filter")
        return send

    # ---- p2: scatter the gathered rows, run this rank's share of the step, append the owned rows ---------------------------
    def p2(self, b: int, gathered: torch.Tensor, queries, out: torch.Tensor = None) -> torch.Tensor:
        """gathered: [G * max_n, d] = every rank's padded block in rank order. queries: device int64 tensors with the ids of
        ALL edges of the batch (this rank reads its share). Returns [C, q_rows, d]."""
        lib, T, d, G = self.lib, self.T, self.d, self.G
        lo, hi = self.batch(b)
        n = hi - lo
        q_off, q_rows = self.share(b)
        C = len(queries)
        with torch.cuda.device(self.dev), torch.no_grad():
            self._cur_full.index_copy_(0, self.scat[self.scat_off[b]:self.scat_off[b + 1]], gathered)
            if out is None:
                out = torch.empty((max(C, 1), q_rows, d), dtype=torch.float32, device=self.dev)
            ids = self.ids[self.ids_off[b]:self.ids_off[b + 1]]
            qptrs = (ctypes.c_void_p * max(C, 1))(*[q.data_ptr() + 8 * q_off for q in queries])
            if self.history == "changelog":  # step + retire / append of the owned rows' events (phase 2: the filter is done)
                _lib.check(lib.lstep_pe_step_changelog(ctypes.byref(self.desc), self.changelog.ref, self.sampler.csr_ref, lo, n, _lib.ptr(ids),
                                                       ids.shape[0], self.tmax[b], self.head, self.len, None, qptrs, C, q_off, q_rows, _lib.ptr(out),
                                                       self.K, self.m._mlp_ref("nbr"), self.m._mlp_ref("update"), _lib.ptr(self.ws), self.ws.numel(),
                                                       _lib.ptr(self.sampler._err), _lib.stream_ptr(), 2), "lstep_pe_step_changelog")
                _, self.head, self.len = advance(self.head, self.len, T)
                self.batch_idx += 1
                return out
            _lib.check(lib.lstep_pe_step_sharded(ctypes.byref(self.desc), self.sampler.csr_ref, lo, n, _lib.ptr(ids), ids.shape[0], self.tmax[b],
                                                 qptrs, C, q_off, q_rows, _lib.ptr(out), self.K, self.m._mlp_ref("nbr"), self.m._mlp_ref("update"),
                                                 _lib.ptr(self.ws), self.ws.numel(), _lib.ptr(self.sampler._err), _lib.stream_ptr()),
                       "lstep_pe_step_sharded")
            slot, self.head, self.len = advance(self.head, self.len, T)
            _lib.check(lib.lstep_ring_copy_rows(_lib.ptr(self.ring), _lib.ptr(self.cur), self.rows_local, T, d, slot, G, self.rank, 1,
                                                _lib.stream_ptr()), "ring append")
        self.batch_idx += 1
        return out

    def check_errors(self):
        if self.history == "changelog":
            self.changelog.check_full(self.sampler._err, int(self.sampler._err.item()))
        self.sampler.check_errors()

    def history_bytes(self) -> int:
        if self.history == "changelog":
            return self.changelog.nbytes()
        return self.ring.numel() * self.ring.element_size()

    def export_history_rows(self) -> torch.Tensor:
        """[rows_local, len, d], oldest first: row l = node l * G + rank."""
        if self.history == "changelog":
            return self.changelog.replay(self.head, self.len)
        idx = (self.head + torch.arange(self.len, device=self.dev)) % self.T
        return self.ring.index_select(1, idx)[:self.rows_local]


class ReplicatedLocalGroup:
    """All G ranks in one process on one device, in lock step (tests): the all-gather is a concatenation."""

    def __init__(self, ranks):
        self.ranks, self.G = ranks, len(ranks)

    def step(self, b: int, queries):
        blocks = [rk.p1(b).clone() for rk in self.ranks]
        gathered = torch.cat(blocks)
        return [rk.p2(b, gathered, queries) for rk in self.ranks]


class ReplicatedTableStream:
    """One process per GPU (torchrun): this rank's state + the NCCL all-gather."""

    def __init__(self, rank_state: ReplicatedTableRank, group=None):
        import torch.distributed as dist
        self.rk, self.dist, self.group = rank_state, dist, group

    def step(self, b: int, queries, out: torch.Tensor = None) -> torch.Tensor:
        rk = self.rk
        send = rk.p1(b)
        mx = rk.max_n[b]
        gathered = rk._gbuf[:rk.G * mx]
        if rk.G > 1:
            self.dist.all_gather_into_tensor(gathered, send, group=self.group)
            rk.bytes_allgather += gathered.numel() * 4
        else:
            gathered = send
        return rk.p2(b, gathered, queries, out)
