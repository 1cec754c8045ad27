"""The PE histories on the host side. The change log (csrc/changelog.cu on the device; layout in include/lstep_b200.h,
`struct lstep_changelog`): one rank's log, the descriptor the kernels take, loading a logical history (checkpoint.History)
into it, saving it as a checkpoint shard and replaying it into dense rows. ChangeLogStream (world 1),
ReplicatedTableRank(history="changelog") and PeerRank each own one; `ChangeLogOwner` is what ChangeLogStream and PeerRank
share about it. `RingHistory` is PEStream's dense ring, with the methods of the change log that hostfeed.HostFed calls. The
owners keep the window position (head, len) and move it with `advance`, the rule the native multi-step calls follow too.
`filter_len` is the window the DFT filter is masked to."""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib
from . import checkpoint as ckpt


def filter_len(batch_idx: int, length: int, T: int) -> int:
    """Window length the next step's DFT filter is masked to: keyed on batch_idx while the history is shorter than T (Q5)."""
    return min(max(batch_idx, 0), T) if length < T else T


def advance(head: int, length: int, T: int, steps: int = 1):
    """(slot, head, len) of `steps` steps on a window of T slots: the slot the first of them writes, and the window after
    them. The window fills, then each step overwrites its oldest slot."""
    fill = steps if steps < T - length else T - length
    return (head + length) % T, (head + steps - fill) % T, length + fill


def _to_dev(a, dev, dtype):
    """A tensor, or a host numpy array (memory-mapped ones included: copied first), on `dev`."""
    if isinstance(a, torch.Tensor):
        return a.to(dev, dtype)
    return torch.from_numpy(np.array(a, dtype={torch.float32: np.float32, torch.int64: np.int64}[dtype])).to(dev)


class RingHistory:
    """The dense PE history: T window slots per node, node-major `ring` [row_cap, T, d] (68.8 KB a node at T = 100,
    d = 172), of which the first V1 rows are live. Rows above V1 are written by `init_rows` before they go live."""

    def __init__(self, V1: int, T: int, d: int, device, row_cap: int = None):
        self.V1, self.T, self.d, self.dev = int(V1), int(T), int(d), device
        self.row_cap = max(self.V1, int(row_cap or 0))
        self.ring = torch.zeros((self.row_cap, T, d), dtype=torch.float32, device=device)

    def load(self, history: torch.Tensor, cur: torch.Tensor):
        """Load a dense history [V1, Th, d] (oldest first, Th <= T, on the device) into the ring and its newest step into the
        table `cur` (lstep_ring_load). Returns the window (head, len)."""
        Th = history.shape[1]
        self.ring[:self.V1, :Th] = history
        with torch.cuda.device(self.dev):
            _lib.check(_lib.load().lstep_ring_load(_lib.ptr(self.ring), _lib.ptr(cur), self.V1, self.T, self.d, (Th - 1) % self.T,
                                                   _lib.stream_ptr()), "lstep_ring_load")
        return 0, Th

    def grow_capacity(self, row_cap: int):
        """Reallocate the ring for `row_cap` nodes and copy the live rows over (on the current stream)."""
        ring = torch.zeros((row_cap, self.T, self.d), dtype=torch.float32, device=self.dev)
        ring[:self.V1].copy_(self.ring[:self.V1])
        self.ring, self.row_cap = ring, int(row_cap)

    def add_rows(self, V1: int):
        """Make nodes [self.V1, V1) live (V1 <= row_cap); init_rows must have written their slots."""
        assert self.V1 <= V1 <= self.row_cap
        self.V1 = int(V1)

    def init_rows(self, table: torch.Tensor, v0: int, v1: int, rows: torch.Tensor, stride: int):
        """Write the initial rows of nodes [v0, v1) to the table and to all T ring slots (lstep_pe_rows_init): `rows` is one
        row [d] for all of them (stride 0) or one per node (stride d)."""
        _lib.check(_lib.load().lstep_pe_rows_init(_lib.ptr(table), _lib.ptr(self.ring), self.T, self.d, None, 1, 0, v0, v1, _lib.ptr(rows),
                                                  stride, _lib.stream_ptr()), "lstep_pe_rows_init")

    def replay(self, head: int, length: int) -> torch.Tensor:
        """The window (head, length) as dense rows [V1, length, d], oldest first."""
        idx = (head + torch.arange(length, device=self.dev)) % self.T
        return self.ring[:self.V1].index_select(1, idx).contiguous()

    def nbytes(self) -> int:
        return self.ring.numel() * self.ring.element_size()

    def check_full(self, err: torch.Tensor, flag: int):
        """Nothing: every step writes one slot of every node, so the ring cannot overflow."""


class ChangeLogHistory:
    """The change log of rank `rank` of a world-`world` group over V1 nodes: the nodes v with v % world == rank, node v at
    row (v - rank) / world, `rows` of them (checkpoint.rows_of). `cap` events per window slot (at least 1). `ref` is the
    lstep_changelog descriptor to pass to the native calls. The base rows of a new log are unset: `reset` or `load` fills
    them. `row_cap` (>= V1, default V1): nodes base / ev_mask are allocated for, so that `add_rows` can grow V1 in place;
    the descriptor carries the live row count."""

    ring = None  # (no dense ring: the step descriptor's ring pointer is null)

    def __init__(self, V1: int, T: int, d: int, cap: int, world: int, rank: int, device, row_cap: int = None):
        if T > 128:
            raise _lib.LstepError("the change-log history supports T <= 128 window steps")
        self.V1, self.T, self.d, self.world, self.rank, self.dev = int(V1), int(T), int(d), int(world), int(rank), device
        self.rows = ckpt.rows_of(self.V1, self.world, self.rank)
        self.row_cap = max(self.V1, int(row_cap or 0))
        rows_cap = ckpt.rows_of(self.row_cap, self.world, self.rank)
        self.cap = cap = int(max(cap, 1))
        H = 1
        while H < 2 * cap:
            H *= 2
        self.base = torch.empty((rows_cap, d), dtype=torch.float32, device=device)
        self.ev_node = torch.zeros((T, cap), dtype=torch.int32, device=device)
        self.ev_row = torch.empty((T, cap, d), dtype=torch.float32, device=device)
        self.ev_cnt = torch.zeros(T, dtype=torch.int32, device=device)
        self.ev_hash = torch.full((T, H), -1, dtype=torch.int64, device=device)
        self.ev_mask = torch.zeros((max(rows_cap, 1), 4), dtype=torch.int32, device=device)
        self.desc = _lib.ChangeLog(self.base.data_ptr(), self.ev_node.data_ptr(), self.ev_row.data_ptr(), self.ev_cnt.data_ptr(),
                                   self.ev_hash.data_ptr(), self.ev_mask.data_ptr(), max(self.rows, 1), T, cap, H, d, self.world,
                                   self.rank)
        self.ref = ctypes.byref(self.desc)

    def grow_capacity(self, row_cap: int):
        """Reallocate base and ev_mask for `row_cap` nodes and copy the live rows over (on the current stream, behind the steps
        already enqueued). Both new tensors are allocated before either is swapped in."""
        rows_cap = ckpt.rows_of(int(row_cap), self.world, self.rank)
        base = torch.empty((rows_cap, self.d), dtype=torch.float32, device=self.dev)
        mask = torch.zeros((max(rows_cap, 1), 4), dtype=torch.int32, device=self.dev)
        base[:self.rows].copy_(self.base[:self.rows])
        mask[:self.rows].copy_(self.ev_mask[:self.rows])
        self.base, self.ev_mask, self.row_cap = base, mask, int(row_cap)
        self.desc.base, self.desc.ev_mask = base.data_ptr(), mask.data_ptr()

    def add_rows(self, V1: int):
        """Make nodes [self.V1, V1) live (V1 <= row_cap). Their base rows must be written (lstep_pe_rows_init) before a step
        reads them; their event masks are zero, as allocated."""
        assert self.V1 <= V1 <= self.row_cap
        self.V1 = int(V1)
        self.rows = ckpt.rows_of(self.V1, self.world, self.rank)
        self.desc.rows = max(self.rows, 1)

    def init_rows(self, table: torch.Tensor, v0: int, v1: int, rows: torch.Tensor, stride: int):
        """Write the initial rows of nodes [v0, v1) to the table and, for the owned ones, to their base rows
        (lstep_pe_rows_init): `rows` is one row [d] for all of them (stride 0) or one per node (stride d)."""
        _lib.check(_lib.load().lstep_pe_rows_init(_lib.ptr(table), None, self.T, self.d, _lib.ptr(self.base), self.world, self.rank, v0, v1,
                                                  _lib.ptr(rows), stride, _lib.stream_ptr()), "lstep_pe_rows_init")

    def reset(self, cur: torch.Tensor):
        """A one-step history: base = the owned rows of the table `cur` [V1, d], no events. Returns the window (head, len)."""
        self.base[:self.rows].copy_(cur[:self.V1][self.rank::self.world])
        self.ev_cnt.zero_()
        self.ev_hash.fill_(-1)
        self.ev_mask.zero_()
        return 0, 1

    def load(self, hist: "ckpt.History", cur: torch.Tensor):
        """Load a logical history (any world size) into this log and the table `cur` [V1, d]. cur = every node's base row;
        then, for every window position f in order, cur[nodes of f] = their rows and lstep_changelog_append records the rows
        of the owned nodes as the events of slot f, exactly as a live step records them. After the last position cur is the
        current table. The event count of every position is checked against the capacity before any device write. Returns
        the window (head, len)."""
        world, rank, dev = self.world, self.rank, self.dev
        cnt = hist.counts(world)[:, rank]
        if len(cnt) and int(cnt.max()) > self.cap:
            f = int(cnt.argmax())
            raise _lib.LstepError(f"window position {f} of the history holds {int(cnt[f])} events of rank {rank} of {world} but "
                                  f"event_capacity is {self.cap}: pass a larger event_capacity")
        lib = _lib.load()
        chunk = max(1, (256 << 20) // (4 * hist.d))
        with torch.cuda.device(dev), torch.no_grad():
            for g, sh in enumerate(hist.shards):
                dst = cur[:self.V1][g::hist.world]
                for a in range(0, dst.shape[0], chunk):
                    dst[a:a + chunk].copy_(_to_dev(sh["base"][a:a + chunk], dev, torch.float32))
            self.reset(cur)
            err = torch.zeros(1, dtype=torch.int32, device=dev)
            for f in range(hist.len):
                nodes, rows = hist.events(f)
                ids = _to_dev(nodes, dev, torch.int64) if len(nodes) else None
                if ids is not None:
                    cur[ids] = _to_dev(rows, dev, torch.float32)
                _lib.check(lib.lstep_changelog_append(self.ref, f, 0, _lib.ptr(cur), None, None, 0, _lib.ptr(ids), len(nodes), None, 0, 0,
                                                      _lib.ptr(err), _lib.stream_ptr()), "lstep_changelog_append")
            if int(err.item()):
                raise _lib.LstepError(f"loading the history overflowed the change log (flag {int(err.item())})")
        return 0, hist.len

    def save(self, path: str, head: int, length: int, meta: dict):
        """Write the window (head, length) of this log as shard `rank` of a checkpoint in directory `path`: the base rows and
        the events of every window position in logical order (sorted by node within a position, so that one state always
        gives the same files). `meta`: batch_idx, steps_done and edges_done. Call the owner's check_errors() first."""
        torch.cuda.synchronize(self.dev)
        cnt = self.ev_cnt.cpu().numpy()
        slots = [(head + f) % self.T for f in range(length)]
        off = np.cumsum([0] + [int(cnt[s]) for s in slots]).astype(np.int64)
        ev_node = np.empty(int(off[-1]), np.int64)
        ev_row = np.empty((int(off[-1]), self.d), np.float32)
        for f, s in enumerate(slots):
            n = int(cnt[s])
            if n:
                nodes = self.ev_node[s, :n].cpu().numpy()
                order = np.argsort(nodes, kind="stable")
                ev_node[off[f]:off[f + 1]] = nodes[order]
                ev_row[off[f]:off[f + 1]] = self.ev_row[s, :n].cpu().numpy()[order]
        meta = dict(meta, world=self.world, rank=self.rank, V1=self.V1, d=self.d, T=self.T, len=length)
        ckpt.write_shard(path, meta, self.base[:self.rows].cpu().numpy(), off, ev_node, ev_row)

    def replay(self, head: int, length: int) -> torch.Tensor:
        """The window (head, length) as dense rows [rows, length, d], oldest first (needs rows * length * d * 4 bytes)."""
        snap = self.base[:self.rows].clone()
        out = torch.empty((self.rows, length, self.d), dtype=torch.float32, device=self.dev)
        cnt = self.ev_cnt.cpu().tolist()
        for f in range(length):
            s = (head + f) % self.T
            if cnt[s]:
                snap[(self.ev_node[s, :cnt[s]].long() - self.rank) // self.world] = self.ev_row[s, :cnt[s]]
            out[:, f, :] = snap
        return out

    def nbytes(self) -> int:
        """Bytes the log occupies (base + event rows + index structures)."""
        return sum(t.numel() * t.element_size() for t in (self.base, self.ev_node, self.ev_row, self.ev_cnt, self.ev_hash, self.ev_mask))

    def check_full(self, err: torch.Tensor, flag: int):
        """LstepError if `flag`, the value read from the device error flag `err`, says a step recorded more events than the
        capacity (FLAG_CHANGELOG_FULL); the flag is cleared first."""
        if flag & _lib.FLAG_CHANGELOG_FULL:
            err.zero_()
            raise _lib.LstepError(f"a step changed more rows than the change-log history's event capacity ({self.cap})")


class ChangeLogOwner:
    """What the owners of a change-log history, ChangeLogStream and PeerRank, share on top of hostfeed.HostFed: the state
    they start from, save_checkpoint and the event-capacity check of growth. An owner sets `_cap_arg` and `_row_cap_arg`
    (its event_capacity and row_capacity) and provides `_default_event_cap(V1)`, the events per step its log records by
    default. `changelog` is its history."""

    changelog = property(lambda self: self.history)
    cap = property(lambda self: self.history.cap)

    def _start(self, initial_pe, history, checkpoint, batch_idx, world: int = 1, rank: int = 0, V1: int = None):
        """Load the state of the nodes v % world == rank from `checkpoint` (a directory that save_checkpoint wrote at any
        world size, or the checkpoint.History that checkpoint.read returned), else from the dense `history` [V1, Th, d]
        (oldest first), else from the table `initial_pe` [V1, d]; none of them: no state. V1: the node count the owner was
        built for (None: the history's). head, len, batch_idx, steps_done and edges_done continue from a checkpoint; a dense
        history restarts steps_done and edges_done (at start). `batch_idx` then overrides the batch index the next step masks
        the filter with while the history is shorter than T (the reference's evaluate loop restarts it at 0: Q5)."""
        hist = None
        if checkpoint is not None:
            hist = checkpoint if isinstance(checkpoint, ckpt.History) else ckpt.read(checkpoint)
        elif history is not None or initial_pe is not None:
            dense = history if history is not None else initial_pe.unsqueeze(1)
            with torch.cuda.device(self.dev):
                hist = ckpt.from_dense(dense.to(self.dev, torch.float32), self.T)
        if hist is not None:
            hist.check(V1=V1, d=self.d, T=self.T)
            self._check_stream_ids(hist.V1)
            cap = self._cap_arg if self._cap_arg is not None else self._default_event_cap(max(hist.V1, int(self._row_cap_arg or 0),
                                                                                              self.max_nodes or 0))
            self._new_state(ChangeLogHistory(hist.V1, self.T, self.d, cap, world, rank, self.dev, self._row_cap_arg))
            self.head, self.len = self.history.load(hist, self.cur)
            self.steps_done, self.edges_done = 0, self.start
            if checkpoint is not None:
                self.batch_idx, self.steps_done, self.edges_done = (int(hist.meta[k]) for k in ("batch_idx", "steps_done", "edges_done"))
        if batch_idx is not None:
            self.batch_idx = int(batch_idx)

    def save_checkpoint(self, path: str):
        """Write this owner's shard of a checkpoint into directory `path` (l-step_b200/checkpoint.py): the base rows and the
        events of every window position of the nodes it owns (about V1 + T * (rows changed per step) rows over all shards;
        not the table, the CSR or the model parameters). A ChangeLogStream writes a world-1 checkpoint; every rank of a peer
        group calls it after the same step, with no barrier (an owner's history is always current on its own rank).
        ChangeLogStream(..., checkpoint=path) and PeerRank(..., checkpoint=path) at any world size resume from it with the
        bits of the uninterrupted run."""
        self.check_errors()
        self.history.save(path, self.head, self.len, dict(batch_idx=self.batch_idx, steps_done=self.steps_done, edges_done=self.edges_done))

    def _check_event_capacity(self, V1: int):
        """The default event capacity is sized for the nodes the owner may hold (max_nodes, else its row capacity): growing
        beyond what it covers raises ValueError before any write (a step could change more rows than the log records). On a
        peer group it is the same on every rank and cannot grow: the inbox blocks are laid out by it."""
        if self._cap_arg is None and self.cap < self._default_event_cap(V1):
            raise ValueError(f"{type(self).__name__}: {V1} nodes need an event capacity of {self._default_event_cap(V1)} rows per step, "
                             f"the log was sized for {self.cap}; build it with max_nodes (or event_capacity) covering its growth")
