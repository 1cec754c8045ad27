"""Drop-in for the reference's temporal neighbour sampler (utils/utils.py:70-301), backed by a
time-sorted CSR in HBM and the warp-cooperative lookup kernel (csrc/sampler.cu).

Same names, argument meaning and error behaviour as the reference:

    get_neighbor_sampler(data, sample_neighbor_strategy, time_scaling_factor, seed)
    NeighborSampler(adj_list, sample_neighbor_strategy, time_scaling_factor, seed)
        .get_historical_neighbors(node_ids, node_interact_times, num_neighbors=20)
            -> (int64[n,K], int64[n,K], float32[n,K]) numpy arrays
        .find_neighbors_before / .get_multi_hop_neighbors / .get_all_first_hop_neighbors
        .reset_random_state(), .sample_neighbor_strategy, .seed

Only the 'recent' strategy — the one LSTEP's defaults and best-configs use
(utils/load_configs.py:22,81-96) — runs on the device; 'uniform' / 'time_interval_aware' draw from
numpy's RandomState on the host in the reference and are outside the hot path (SURVEY §2 #1):
asking for them raises NotImplementedError instead of silently computing on the CPU.

A GROWABLE sampler (NeighborSampler.growable, csrc/csr_grow.cu) serves an edge stream that is still arriving: its
rows end in padding, `ingest` appends a batch on the device, and every lookup returns what the exact sampler of the
edges ingested so far returns. Capacity is planned on the host (check_edges, overflow_rows, plan_capacity below:
numpy only), so deciding to regrow never synchronises.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib

_STRATEGIES = ("uniform", "recent", "time_interval_aware")

# Smallest spare room a regrow gives a row. Every row gets need + max(MIN_SLACK, need), so rows can double before the
# next regrow; the floor keeps rows that are still small from forcing one regrow after another while a stream starts
# from empty. The floor is also room on every row, untouched ones included. Measured on a B200 (profiles/r03_csr_grow.json):
#   Reddit shape (11 k rows, 1.3 M entries, B=200): floor 1 / 4 / 16 / 64 -> 253 / 52 / 19 / 12 regrows, 38 / 9.5 / 3.7 /
#   2.1 ms of regrows in all, CSR 39 / 39 / 43 / 34 MB at the end;
#   2 M rows, 4 M entries (B=2000): floor 4 / 16 / 64 -> 56 / 19 / 11 regrows, 530 / 179 / 167 ms, CSR 0.25 / 0.62 / 2.1 GB.
# 64 saves a few regrows on the small graph but makes a graph with many rows and few entries per row 3.4x larger than 16,
# for 12 ms less regrowing; 4 regrows three times as often. Hence 16.
MIN_SLACK = 16
_EID_MAX = 0x7FFFFFFF
NODE_ID_MAX = 0x7FFFFFFE  # largest node id a growing stream accepts: the change log records node ids as int32


def check_edges(src, dst, edge_ids, times, num_rows: int, last_time: float = -np.inf):
    """Validate a batch for ingestion into a growable CSR and return it as contiguous (int64, int64, int64, float64)
    arrays. Raises ValueError for unequal lengths, non-finite or decreasing times, a first time before `last_time` (the
    last time ingested) and edge ids outside [0, 2^31); IndexError for a node id outside [0, num_rows), as the
    reference's adjacency lookup does (SURVEY Q8). edge_ids may be an int: the first of n consecutive ids, returned as
    the array of all n."""
    src = np.ascontiguousarray(src, dtype=np.int64)
    dst = np.ascontiguousarray(dst, dtype=np.int64)
    t = np.ascontiguousarray(times, dtype=np.float64)
    n = len(src)
    if isinstance(edge_ids, (int, np.integer)):
        eid = np.arange(int(edge_ids), int(edge_ids) + n, dtype=np.int64)
        n_eid = n
    else:
        eid = np.ascontiguousarray(edge_ids, dtype=np.int64)
        n_eid = len(eid)
    if len(dst) != n or n_eid != n or len(t) != n:
        raise ValueError(f"ingest: src, dst, edge_ids and times must have the same length ({n}, {len(dst)}, {n_eid}, {len(t)})")
    if n == 0:
        return src, dst, eid, t
    lo, hi = min(int(src.min()), int(dst.min())), max(int(src.max()), int(dst.max()))
    if lo < 0 or hi >= num_rows:
        raise IndexError(f"list index out of range: node id {lo if lo < 0 else hi} is outside the sampler's {num_rows} rows")
    if not np.isfinite(t).all():
        raise ValueError("ingest: times must be finite")
    if n > 1 and not (np.diff(t) >= 0).all():
        raise ValueError("ingest: times must be non-decreasing within a batch")
    if t[0] < last_time:
        raise ValueError(f"ingest: the batch starts at time {t[0]!r}, before the last time ingested ({last_time!r})")
    if int(eid.min()) < 0 or int(eid.max()) > _EID_MAX:
        raise ValueError("ingest: edge ids must lie in [0, 2^31)")
    return src, dst, eid, t


def row_counts(src: np.ndarray, dst: np.ndarray):
    """(rows, counts): the rows a batch appends to and how many entries each gets (one per endpoint: a self-loop
    counts twice)."""
    return np.unique(np.concatenate([src, dst]), return_counts=True)


def overflow_rows(fill: np.ndarray, cap: np.ndarray, src: np.ndarray, dst: np.ndarray) -> np.ndarray:
    """Rows the batch (src, dst) touches that have no room for its entries. O(batch): only touched rows are looked at."""
    rows, cnt = row_counts(src, dst)
    return rows[fill[rows] + cnt > cap[rows]]


def plan_capacity(need: np.ndarray, min_slack: int = MIN_SLACK) -> np.ndarray:
    """Row capacities of a regrow: need + max(min_slack, need) for every row."""
    need = np.asarray(need, dtype=np.int64)
    return need + np.maximum(int(min_slack), need)


def tail_entries(spare_rows: int, min_slack: int = MIN_SLACK) -> int:
    """Entries of padding a regrow leaves past the live rows for rows added later: 2 * min_slack per spare row of capacity
    (a new row takes need + max(min_slack, need) of them, so this covers spare rows that arrive with up to min_slack
    entries each)."""
    return int(spare_rows) * 2 * int(min_slack)


def plan_layout(need: np.ndarray, row_cap: int, min_slack: int = MIN_SLACK):
    """(indptr [row_cap + 1], total) of a regrow with len(need) live rows: row capacities plan_capacity(need), every row
    at or above the live ones empty at the end of the live rows, and total = that end + tail_entries(spare rows)."""
    need = np.asarray(need, dtype=np.int64)
    rows = len(need)
    indptr = np.zeros(int(row_cap) + 1, dtype=np.int64)
    np.cumsum(plan_capacity(need, min_slack), out=indptr[1:rows + 1])
    indptr[rows + 1:] = indptr[rows]
    return indptr, int(indptr[rows]) + tail_entries(int(row_cap) - rows, min_slack)


def rows_fit(num_rows: int, row_cap: int, tail0: int, total: int, new_cap: np.ndarray) -> bool:
    """Whether len(new_cap) rows with those capacities can be added without a regrow: within the row capacity and inside
    the tail [tail0, total)."""
    return num_rows + len(new_cap) <= row_cap and tail0 + int(np.sum(new_cap)) <= total


def new_row_need(src: np.ndarray, dst: np.ndarray, num_rows: int, new_rows: int) -> np.ndarray:
    """Entries the edges (src, dst) give each of the rows [num_rows, num_rows + new_rows)."""
    ends = np.concatenate([src, dst])
    ends = ends[ends >= num_rows] - num_rows
    return np.bincount(ends, minlength=new_rows)[:new_rows].astype(np.int64)


def _dev(device=None) -> torch.device:
    if device is None:
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device(device)


class NeighborSampler:
    def __init__(self, adj_list: list = None, sample_neighbor_strategy: str = "uniform", time_scaling_factor: float = 0.0,
                 seed: int = None, device=None, _csr_tensors=None):
        """adj_list: list (index = node id) of lists of (neighbor_id, edge_id, timestamp) tuples, as in the
        reference (utils/utils.py:72-80). Each list is stably sorted by timestamp on the device."""
        self.sample_neighbor_strategy = sample_neighbor_strategy
        self.time_scaling_factor = time_scaling_factor
        self.seed = seed
        if self.seed is not None:
            self.random_state = np.random.RandomState(self.seed)
        self._lib = _lib.load()
        self.device = _dev(device)
        self._err = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.fill = None  # growable samplers only: device int32 [num_rows], see growable()
        if _csr_tensors is not None:
            self._set_csr(*_csr_tensors)
            return
        owner = np.fromiter((i for i, lst in enumerate(adj_list) for _ in lst), dtype=np.int64)
        n = owner.shape[0]
        flat = [x for lst in adj_list for x in lst]
        nbr = np.fromiter((x[0] for x in flat), dtype=np.int64, count=n)
        eid = np.fromiter((x[1] for x in flat), dtype=np.int64, count=n)
        t = np.fromiter((x[2] for x in flat), dtype=np.float64, count=n)
        self._build("lstep_csr_build_from_entries", (owner, nbr, eid, t), n, n, len(adj_list))

    # ---- construction -----------------------------------------------------------------------
    @classmethod
    def from_edges(cls, src_node_ids, dst_node_ids, edge_ids, node_interact_times, sample_neighbor_strategy="recent",
                   time_scaling_factor=0.0, seed=None, device=None, num_rows=None):
        """Build straight from an edge stream (what get_neighbor_sampler does, utils/utils.py:292-299)
        without materialising python adjacency lists. Arrays may be numpy or CUDA tensors."""
        self = cls.__new__(cls)
        NeighborSampler.__init__(self, None, sample_neighbor_strategy, time_scaling_factor, seed, device,
                                 _csr_tensors=())  # placeholder, replaced below
        E = int(len(src_node_ids))
        if num_rows is None:
            mx = max(int(src_node_ids.max()), int(dst_node_ids.max())) if E else 0
            num_rows = mx + 1
        self._build("lstep_csr_build_from_edges", (src_node_ids, dst_node_ids, edge_ids, node_interact_times), E, 2 * E,
                    int(num_rows))
        return self

    @classmethod
    def growable(cls, num_rows: int, src=(), dst=(), edge_ids=(), times=(), sample_neighbor_strategy="recent",
                 time_scaling_factor=0.0, seed=None, device=None, min_slack: int = MIN_SLACK, row_capacity: int = None):
        """A sampler that grows batch by batch (`ingest`), for a stream whose edges are not known in advance. The optional
        prefix (src, dst, edge_ids, times; times non-decreasing) is built with the exact builder and then laid out with
        room to grow. Node ids must lie in [0, num_rows). Lookups equal those of from_edges on the edges ingested so far.
        `row_capacity` (default num_rows): rows allocated, so that add_rows can make up to row_capacity - num_rows more
        rows live without a regrow (each spare row reserves tail_entries(1, min_slack) entries)."""
        num_rows = int(num_rows)
        if num_rows <= 0:
            raise ValueError("growable: num_rows must be positive")
        row_cap = num_rows if row_capacity is None else int(row_capacity)
        if row_cap < num_rows or row_cap > NODE_ID_MAX + 1:
            raise ValueError(f"growable: row_capacity must lie in [num_rows, 2^31 - 1] (got {row_cap})")
        src, dst, eid, t = check_edges(src, dst, edge_ids, times, num_rows)
        self = cls.from_edges(src, dst, eid, t, sample_neighbor_strategy, time_scaling_factor, seed, device, num_rows=num_rows)
        self.min_slack = int(min_slack)
        self._version = 0
        fill = np.bincount(src, minlength=num_rows) + np.bincount(dst, minlength=num_rows)
        self._fill_h = fill.astype(np.int64)
        self._n_entries = int(2 * len(src))
        self._last_t = float(t[-1]) if len(t) else -np.inf
        self._next_eid = int(eid[-1]) + 1 if len(eid) else 1
        self.regrows = 0
        self.row_cap = row_cap
        self._regrow(self._fill_h)
        self.regrows = 0  # regrows after construction
        return self

    @property
    def is_growable(self) -> bool:
        return self.fill is not None

    @property
    def num_entries(self) -> int:
        """Real (ingested) adjacency entries; `nnz` is the length of the arrays, padding included."""
        return self._n_entries if self.is_growable else self.nnz

    @property
    def last_time(self) -> float:
        """Time of the last edge ingested (-inf before the first); the next batch may not start earlier."""
        return self._last_t

    @property
    def next_edge_id(self) -> int:
        """Edge id after the last one ingested (1 before the first: the reference's edge ids start at 1, 0 is padding)."""
        return self._next_eid

    def _require_growable(self):
        if not self.is_growable:
            raise ValueError("this NeighborSampler holds an exact CSR; build one with NeighborSampler.growable(...) to ingest edges")

    def _regrow(self, need: np.ndarray):
        """Lay the CSR out again with capacity plan_capacity(need) per row for len(need) >= num_rows live rows (the rows
        above num_rows become live, empty), and a padded tail for the rest of the row capacity, which doubles when the
        rows outgrow it. Synchronises the device once (appends may still be in flight on other streams, and the old arrays
        are released afterwards). Every new array is allocated before any state changes."""
        new_rows = len(need)
        row_cap = self.row_cap if new_rows <= self.row_cap else max(2 * self.row_cap, new_rows)
        indptr_h, total = plan_layout(need, row_cap, self.min_slack)
        if total > _EID_MAX:  # the kernels index entries with int64 but the builder's limit is kept for the whole CSR
            raise _lib.LstepError(f"growable CSR: {total} entries of capacity exceed 2^31")
        dev = self.device
        torch.cuda.synchronize(dev)
        indptr = torch.from_numpy(indptr_h).to(dev)
        nbr = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
        eid = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
        t = torch.empty(max(total, 1), dtype=torch.float64, device=dev)
        fill = torch.empty(row_cap, dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            rc = self._lib.lstep_csr_relayout_rows(self.csr_ref, _lib.ptr(self.fill), new_rows, row_cap, _lib.ptr(indptr), total,
                                                   _lib.ptr(nbr), _lib.ptr(eid), _lib.ptr(t), _lib.ptr(fill), _lib.ptr(self._err),
                                                   _lib.stream_ptr())
        _lib.check(rc, "lstep_csr_relayout_rows")
        self._set_csr(indptr, nbr[:total], eid[:total], t[:total], num_rows=new_rows)
        self.fill = fill
        self.row_cap = row_cap
        # host mirrors of fill and the row capacities, allocated for row_cap rows so that add_rows only writes the new rows
        self._fill_buf = np.zeros(row_cap, np.int64)
        self._fill_buf[:len(self._fill_h)] = self._fill_h
        self._cap_buf = np.zeros(row_cap, np.int64)
        self._cap_buf[:new_rows] = plan_capacity(need, self.min_slack)
        self._fill_h, self._cap_h = self._fill_buf[:new_rows], self._cap_buf[:new_rows]
        self._tail0 = int(indptr_h[new_rows])
        self.regrows += 1
        self._version += 1

    def add_rows(self, n: int, need=None) -> int:
        """Make n more rows (node ids num_rows .. num_rows + n - 1) live, empty, and return the first new id. `need`: entries
        each new row is about to receive (e.g. from the batch that introduces it), so that row gets need + max(min_slack,
        need) entries of room. Within the row capacity and the padded tail this moves no entry and enqueues one small
        kernel on the current stream (lstep_csr_add_rows: the new rows' indptr and fill), ordered after lookups already
        enqueued, which never read these rows (a host-fed stream's next append waits for it); otherwise it regrows (one device synchronisation) with the row capacity
        doubled. Raises ValueError on an exact sampler."""
        self._require_growable()
        n = int(n)
        r0 = self.num_rows
        if n < 0:
            raise ValueError("add_rows: n must be >= 0")
        if r0 + n > NODE_ID_MAX + 1:
            raise IndexError(f"add_rows: node ids up to {r0 + n - 1} exceed the int32 node id limit ({NODE_ID_MAX})")
        need = np.zeros(n, np.int64) if need is None else np.ascontiguousarray(need, dtype=np.int64)
        if len(need) != n or (n and int(need.min()) < 0):
            raise ValueError("add_rows: need must hold one count >= 0 per new row")
        if n == 0:
            return r0
        cap = plan_capacity(need, self.min_slack)
        if not rows_fit(r0, self.row_cap, self._tail0, self.nnz, cap):
            self._regrow(np.concatenate([self._fill_h, need]))
            return r0
        dev = self.device
        cap_d = torch.from_numpy(cap).pin_memory().to(dev, non_blocking=True)
        with torch.cuda.device(dev):
            rc = self._lib.lstep_csr_add_rows(self.csr_ref, _lib.ptr(self.fill), n, _lib.ptr(cap_d), _lib.stream_ptr())
        _lib.check(rc, "lstep_csr_add_rows")
        self.num_rows = int(self.csr.num_rows)
        self._cap_buf[r0:r0 + n] = cap
        self._fill_buf[r0:r0 + n] = 0
        self._fill_h, self._cap_h = self._fill_buf[:r0 + n], self._cap_buf[:r0 + n]
        self._tail0 += int(cap.sum())
        self._version += 1  # a host-fed stepper re-arms, so its next append (on its copy-in stream) waits for these rows
        return r0

    def reserve(self, src, dst):
        """Make room for the entries the edges (src, dst) will add (known future endpoints, e.g. a whole split). Regrows
        (one device synchronisation) only when a touched row lacks room; every row then gets need + max(min_slack, need)."""
        self._require_growable()
        src = np.ascontiguousarray(src, dtype=np.int64)
        dst = np.ascontiguousarray(dst, dtype=np.int64)
        if len(src) == 0:
            return
        rows, cnt = row_counts(src, dst)
        if int(rows[0]) < 0 or int(rows[-1]) >= self.num_rows:
            raise IndexError(f"list index out of range: node id outside the sampler's {self.num_rows} rows")
        if (self._fill_h[rows] + cnt > self._cap_h[rows]).any():
            need = self._fill_h.copy()
            need[rows] += cnt
            self._regrow(need)

    def _note_ingested(self, src, dst, last_eid: int, last_t: float):
        """Host mirror of an append enqueued on the device (here or by a host-fed stream step)."""
        rows, cnt = row_counts(src, dst)
        self._fill_h[rows] += cnt
        self._n_entries += 2 * len(src)
        self._next_eid = int(last_eid) + 1
        self._last_t = float(last_t)

    def _resync(self, src, dst, eid0: int, times):
        """After a failed call that may have enqueued the appends of a prefix of the edges (src[i], dst[i], eid0 + i,
        times[i]) before failing: synchronise, take fill from the device, and count the edges that landed (appends are
        whole batches, in order). The version bump makes a host-fed stream re-arm its stepper from this state."""
        torch.cuda.synchronize(self.device)
        fill = self.fill[:self.num_rows].cpu().numpy().astype(np.int64)
        landed = int(fill.sum() - self._n_entries) // 2
        if landed > 0:
            self._note_ingested(src[:landed], dst[:landed], eid0 + landed - 1, times[landed - 1])
        self._fill_h[:] = fill
        self._version += 1

    def ingest(self, src, dst, edge_ids, times):
        """Append a batch of edges (the reference's get_neighbor_sampler order: source side, then destination side, in
        edge order). edge_ids may be an int: the first of len(src) consecutive ids. The batch is validated on the host
        before any device write (check_edges), copied to the device (a synchronous copy from pageable memory), and the
        append is enqueued on the current stream."""
        self._require_growable()
        src, dst, eid, t = check_edges(src, dst, edge_ids, times, self.num_rows, self._last_t)
        n = len(src)
        if n == 0:
            return
        self.reserve(src, dst)
        dev = self.device
        a = [torch.from_numpy(x).to(dev, non_blocking=False) for x in (src, dst, eid, t)]
        with torch.cuda.device(dev):
            rc = self._lib.lstep_csr_ingest(self.csr_ref, _lib.ptr(self.fill), _lib.ptr(a[0]), _lib.ptr(a[1]), _lib.ptr(a[2]), 0,
                                            _lib.ptr(a[3]), n, _lib.ptr(self._err), _lib.stream_ptr())
        _lib.check(rc, "lstep_csr_ingest")
        self._note_ingested(src, dst, int(eid[-1]), float(t[-1]))
        self._version += 1

    @classmethod
    def from_reference(cls, ref_sampler, device=None):
        """Adopt an instance of the reference's own NeighborSampler (already-sorted per-node arrays)."""
        adj = [list(zip(np.asarray(a).tolist(), np.asarray(b).tolist(), np.asarray(c).tolist()))
               for a, b, c in zip(ref_sampler.nodes_neighbor_ids, ref_sampler.nodes_edge_ids, ref_sampler.nodes_neighbor_times)]
        return cls(adj, ref_sampler.sample_neighbor_strategy, getattr(ref_sampler, "time_scaling_factor", 0.0),
                   ref_sampler.seed, device)

    def _to_dev(self, a, dtype):
        if isinstance(a, torch.Tensor):
            return a.to(device=self.device, dtype=dtype).contiguous()
        return torch.from_numpy(np.ascontiguousarray(a, dtype={torch.int64: np.int64, torch.float64: np.float64}[dtype])).to(self.device)

    def _build(self, fn_name, arrays, n_in, n_entries, num_rows):
        lib, dev = self._lib, self.device
        a0, a1, a2 = (self._to_dev(a, torch.int64) for a in arrays[:3])
        a3 = self._to_dev(arrays[3], torch.float64)
        indptr = torch.empty(num_rows + 1, dtype=torch.int64, device=dev)
        nbr = torch.empty(max(n_entries, 1), dtype=torch.int32, device=dev)
        eid = torch.empty(max(n_entries, 1), dtype=torch.int32, device=dev)
        t = torch.empty(max(n_entries, 1), dtype=torch.float64, device=dev)
        ws_bytes = lib.lstep_csr_build_workspace_bytes(n_entries, num_rows)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        self._err.zero_()
        with torch.cuda.device(dev):
            rc = getattr(lib, fn_name)(_lib.ptr(a0), _lib.ptr(a1), _lib.ptr(a2), _lib.ptr(a3), n_in, num_rows,
                                       _lib.ptr(indptr), _lib.ptr(nbr), _lib.ptr(eid), _lib.ptr(t), _lib.ptr(ws), ws_bytes,
                                       _lib.ptr(self._err), _lib.stream_ptr())
        _lib.check(rc, fn_name)
        if int(self._err.item()) & _lib.FLAG_NODE_OUT_OF_RANGE:
            raise IndexError("node / edge id out of range while building the temporal adjacency")
        del ws
        self._set_csr(indptr, nbr[:n_entries], eid[:n_entries], t[:n_entries])

    def _set_csr(self, *tensors, num_rows: int = None):
        """Adopt CSR arrays; num_rows: live rows when indptr holds more (a growable CSR's row capacity)."""
        if not tensors:
            return
        self.indptr, self.nbr, self.eid, self.t = tensors
        self.num_rows = int(self.indptr.shape[0] - 1) if num_rows is None else int(num_rows)
        self.nnz = int(self.nbr.shape[0])
        self.csr = _lib.CSR(self.indptr.data_ptr(), self.nbr.data_ptr(), self.eid.data_ptr(), self.t.data_ptr(), self.num_rows,
                            self.nnz)
        self.csr_ref = C.byref(self.csr)

    # ---- reference API ----------------------------------------------------------------------
    def reset_random_state(self):
        self.random_state = np.random.RandomState(self.seed)

    def _require_recent(self):
        if self.sample_neighbor_strategy == "recent":
            return
        if self.sample_neighbor_strategy in _STRATEGIES:
            raise NotImplementedError(f"sample_neighbor_strategy '{self.sample_neighbor_strategy}' draws from a host RNG in the "
                                      "reference and is outside the B200 hot path; use 'recent'")
        raise ValueError(f"Not implemented error for sample_neighbor_strategy {self.sample_neighbor_strategy}!")

    def sample_device(self, node_ids_dev: torch.Tensor, times_dev: torch.Tensor, n_rows: int, n_valid: int, num_neighbors: int):
        """Device-resident lookup for the kernels downstream: (int32[n,K] ids, float32[n,K] times).
        Errors (out-of-range ids) accumulate in a device flag; see check_errors()."""
        K = int(num_neighbors)
        out_n = torch.empty((n_rows, K), dtype=torch.int32, device=self.device)
        out_t = torch.empty((n_rows, K), dtype=torch.float32, device=self.device)
        rc = self._lib.lstep_sample_recent_compact(self.csr_ref, _lib.ptr(node_ids_dev), _lib.ptr(times_dev), n_rows, n_valid, K,
                                                   _lib.ptr(out_n), _lib.ptr(out_t), _lib.ptr(self._err), _lib.stream_ptr())
        _lib.check(rc, "lstep_sample_recent_compact")
        return out_n, out_t

    def check_errors(self):
        """Synchronising check of the device error flag; raises what the reference would."""
        flag = int(self._err.item())
        if flag:
            self._err.zero_()
        if flag & _lib.FLAG_NODE_OUT_OF_RANGE:
            raise IndexError("list index out of range")  # utils/utils.py:140 on an unknown node id (SURVEY Q8)
        if flag & _lib.FLAG_CSR_FULL:
            raise _lib.LstepError("an append to the growable CSR found a row without room (reserve before appending)")
        if flag & _lib.FLAG_UNSORTED_STREAM:
            raise ValueError("an append to the growable CSR was earlier than the row's last entry")
        if flag & _lib.FLAG_FIXED_POINT_RANGE:
            raise FloatingPointError("update_pe phase B met a PE value that is non-finite or at least 2^31 / (n_ids*K + 1) in "
                                     "magnitude (the limit of its 32.32 fixed-point sums); the updated rows are not valid")

    def get_historical_neighbors(self, node_ids: np.ndarray, node_interact_times: np.ndarray, num_neighbors: int = 20):
        assert num_neighbors > 0, 'Number of sampled neighbors for each node should be greater than 0!'
        self._require_recent()
        K = int(num_neighbors)
        n_rows = len(node_ids)
        n_valid = min(n_rows, len(node_interact_times))  # zip() truncation (utils/utils.py:169)
        dev = self.device
        if n_rows == 0:
            return (np.zeros((0, K), np.int64), np.zeros((0, K), np.int64), np.zeros((0, K), np.float32))
        q_n = torch.from_numpy(np.ascontiguousarray(node_ids, dtype=np.int64)).to(dev, non_blocking=True)
        q_t = torch.from_numpy(np.ascontiguousarray(node_interact_times, dtype=np.float64)).to(dev, non_blocking=True)
        out_n = torch.empty((n_rows, K), dtype=torch.int64, device=dev)
        out_e = torch.empty((n_rows, K), dtype=torch.int64, device=dev)
        out_t = torch.empty((n_rows, K), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            rc = self._lib.lstep_sample_recent(self.csr_ref, _lib.ptr(q_n), _lib.ptr(q_t), n_rows, n_valid, K, _lib.ptr(out_n),
                                               _lib.ptr(out_e), _lib.ptr(out_t), _lib.ptr(self._err), _lib.stream_ptr())
        _lib.check(rc, "lstep_sample_recent")
        res = (out_n.cpu().numpy(), out_e.cpu().numpy(), out_t.cpu().numpy())
        self.check_errors()
        return res

    def find_neighbors_before(self, node_id: int, interact_time: float, return_sampled_probabilities: bool = False):
        """All interactions of node_id strictly before interact_time, sorted by time (utils/utils.py:129-146)."""
        if return_sampled_probabilities:
            raise NotImplementedError("sampled probabilities belong to the 'time_interval_aware' strategy")
        node_id = int(node_id)
        if node_id >= self.num_rows or node_id < -self.num_rows:
            raise IndexError("list index out of range")
        node_id %= self.num_rows
        lo, hi = (int(x) for x in self.indptr[node_id:node_id + 2].tolist())
        if self.is_growable:
            hi = lo + int(self._fill_h[node_id])  # the rest of the row is padding
        t = self.t[lo:hi].cpu().numpy()
        i = int(np.searchsorted(t, interact_time))
        return (self.nbr[lo:lo + i].cpu().numpy().astype(np.int64), self.eid[lo:lo + i].cpu().numpy().astype(np.int64), t[:i], None)

    def get_multi_hop_neighbors(self, num_hops: int, node_ids: np.ndarray, node_interact_times: np.ndarray, num_neighbors: int = 20):
        assert num_hops > 0, 'Number of sampled hops should be greater than 0!'
        n = len(node_ids)
        ids, eids, times = self.get_historical_neighbors(node_ids, node_interact_times, num_neighbors)
        out = ([ids], [eids], [times])
        for _ in range(1, num_hops):
            ids, eids, times = self.get_historical_neighbors(out[0][-1].flatten(), out[2][-1].flatten(), num_neighbors)
            for lst, a in zip(out, (ids, eids, times)):
                lst.append(a.reshape(n, -1))
        return out

    def get_all_first_hop_neighbors(self, node_ids: np.ndarray, node_interact_times: np.ndarray):
        res = ([], [], [])
        for node_id, tq in zip(node_ids, node_interact_times):
            a, b, c, _ = self.find_neighbors_before(node_id, tq)
            res[0].append(a), res[1].append(b), res[2].append(c)
        return res


def get_neighbor_sampler(data, sample_neighbor_strategy: str = "uniform", time_scaling_factor: float = 0.0, seed: int = None,
                         device=None) -> NeighborSampler:
    """Same contract as utils/utils.py:282-301: `data` has src_node_ids, dst_node_ids, edge_ids,
    node_interact_times; the adjacency is undirected and each node's list is sorted by time."""
    return NeighborSampler.from_edges(data.src_node_ids, data.dst_node_ids, data.edge_ids, data.node_interact_times,
                                      sample_neighbor_strategy, time_scaling_factor, seed, device)
