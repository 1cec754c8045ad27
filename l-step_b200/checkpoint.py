"""Checkpoints of the change-log PE history (csrc/changelog.cu) in a compact format that does not depend on the world size
(pure numpy + JSON: CPU-testable, like peer.peer_batch_plan).

A checkpoint is a directory. A peer group of world N writes one shard per rank, a ChangeLogStream one shard with N = 1.
Shard g consists of

    rank{g}.meta.json    format, world, rank, V1, d, T, len, batch_idx, steps_done, edges_done (the global edge offset of
                         the next batch; recorded for information only)
    rank{g}.base.npy     float32 [rows_g, d]  base rows of the owned nodes v = g (mod N), node v at row (v - g) / N
    rank{g}.ev_off.npy   int64 [len + 1]      the events of window position f (f = 0 .. len-1, oldest first) are
    rank{g}.ev_node.npy  int64 [n_ev]         [ev_off[f], ev_off[f + 1]) of ev_node / ev_row
    rank{g}.ev_row.npy   float32 [n_ev, d]

History value x[v, f] = the row of v's latest event at a window position <= f, else base[v]; the current table is
x[:, len - 1]. The ring slots of the change log are normalised away and ownership is a function of the node id, so a
checkpoint loads into a change log of any world size (changelog.ChangeLogHistory.load). The table, the CSR and the model
parameters are not stored: the table is the newest window position, the CSR is rebuilt from the edge stream and the
parameters are the caller's state_dict.

Files are written under a temporary name and renamed into place, the meta file last, so an interrupted save never leaves a
shard that looks valid. They are read with mmap and allow_pickle=False and validated completely before anything uses
them (`read`): a checkpoint is input from outside the program."""
from __future__ import annotations

import json
import os

import numpy as np

FORMAT = 1
META_KEYS = ("format", "world", "rank", "V1", "d", "T", "len", "batch_idx", "steps_done", "edges_done")
_AGREE = ("format", "world", "V1", "d", "T", "len", "batch_idx", "steps_done")  # every shard of a checkpoint holds the same
_ARRAYS = ("base", "ev_off", "ev_node", "ev_row")


def rows_of(V1: int, world: int, rank: int) -> int:
    """Number of nodes v in [0, V1) with v % world == rank."""
    return (V1 - rank + world - 1) // world


def _name(rank: int, what: str) -> str:
    return f"rank{rank}.{what}.json" if what == "meta" else f"rank{rank}.{what}.npy"


def _replace(path: str, name: str, write):
    tmp = os.path.join(path, f".{name}.tmp{os.getpid()}")
    try:
        with open(tmp, "wb") as f:
            write(f)
            f.flush()
            os.fsync(f.fileno())
        os.replace(tmp, os.path.join(path, name))
    except BaseException:
        if os.path.exists(tmp):
            os.remove(tmp)
        raise


def write_shard(path: str, meta: dict, base: np.ndarray, ev_off: np.ndarray, ev_node: np.ndarray, ev_row: np.ndarray):
    """Write shard meta["rank"] of a checkpoint into directory `path` (created if needed). `meta`: every key of META_KEYS
    but "format". A meta file this rank left earlier is removed first, and the new one is written after the arrays."""
    meta = {k: int(meta[k]) for k in META_KEYS if k != "format"}
    meta = {"format": FORMAT, **meta}
    g, n_ev = meta["rank"], int(ev_off[-1])
    arrays = {"base": np.ascontiguousarray(base, np.float32), "ev_off": np.ascontiguousarray(ev_off, np.int64),
              "ev_node": np.ascontiguousarray(ev_node, np.int64), "ev_row": np.ascontiguousarray(ev_row, np.float32)}
    assert arrays["base"].shape == (rows_of(meta["V1"], meta["world"], g), meta["d"]) and arrays["ev_off"].shape == (meta["len"] + 1,)
    assert arrays["ev_node"].shape == (n_ev,) and arrays["ev_row"].shape == (n_ev, meta["d"])
    os.makedirs(path, exist_ok=True)
    old = os.path.join(path, _name(g, "meta"))
    if os.path.exists(old):
        os.remove(old)
    for k in _ARRAYS:
        _replace(path, _name(g, k), lambda f, a=arrays[k]: np.save(f, a, allow_pickle=False))
    _replace(path, _name(g, "meta"), lambda f: f.write(json.dumps(meta).encode()))
    fd = os.open(path, os.O_RDONLY)
    try:
        os.fsync(fd)
    finally:
        os.close(fd)


class History:
    """The logical form of a change-log history: `meta` (V1, d, T, len, batch_idx, steps_done, edges_done) and the shards of
    a world-N group (shards[g]: dict of base / ev_off / ev_node / ev_row as in the module docstring). `read` returns one from
    a checkpoint directory, `from_dense` from a dense history; ev_node / ev_off are always host numpy arrays."""

    def __init__(self, meta: dict, shards: list):
        self.meta, self.shards, self.world = dict(meta), list(shards), len(shards)
        self.V1, self.d, self.T, self.len = (int(self.meta[k]) for k in ("V1", "d", "T", "len"))

    def check(self, V1: int = None, d: int = None, T: int = None):
        """ValueError unless the history has these dimensions (None: any)."""
        for k, want in (("V1", V1), ("d", d), ("T", T)):
            if want is not None and getattr(self, k) != int(want):
                raise ValueError(f"checkpoint has {k} = {getattr(self, k)} but the model and stream need {k} = {int(want)}")

    def events(self, f: int):
        """(nodes, rows) of window position f over all shards."""
        parts = [(sh["ev_node"][sh["ev_off"][f]:sh["ev_off"][f + 1]], sh["ev_row"][sh["ev_off"][f]:sh["ev_off"][f + 1]]) for sh in self.shards]
        if len(parts) == 1:
            return parts[0]
        return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])

    def counts(self, world: int) -> np.ndarray:
        """int64 [len, world]: events per window position that rank r of a world-`world` group owns."""
        c = np.zeros(self.len * world, np.int64)
        for sh in self.shards:
            pos = np.repeat(np.arange(self.len, dtype=np.int64), np.diff(sh["ev_off"]))
            c += np.bincount(pos * world + np.asarray(sh["ev_node"]) % world, minlength=self.len * world)
        return c.reshape(self.len, world)

    def shard(self, world: int, rank: int) -> dict:
        """The shard rank `rank` of a world-`world` group holding this history writes (numpy arrays in memory)."""
        N = self.world
        base = np.empty((rows_of(self.V1, world, rank), self.d), np.float32)
        v = np.arange(rank, self.V1, world, dtype=np.int64)
        for g, sh in enumerate(self.shards):
            sel = np.nonzero(v % N == g)[0]
            base[sel] = np.asarray(sh["base"])[(v[sel] - g) // N]
        nodes, rows, off = [], [], [0]
        for f in range(self.len):
            n, r = self.events(f)
            keep = np.asarray(n) % world == rank
            nodes.append(np.asarray(n)[keep])
            rows.append(np.asarray(r)[keep])
            off.append(off[-1] + int(keep.sum()))
        return dict(base=base, ev_off=np.asarray(off, np.int64), ev_node=np.concatenate(nodes).astype(np.int64),
                    ev_row=np.concatenate(rows).reshape(-1, self.d).astype(np.float32))

    def replay(self) -> np.ndarray:
        """The dense history [V1, len, d] (oldest first): the base rows, then the events of every position in order."""
        cur = np.empty((self.V1, self.d), np.float32)
        for g, sh in enumerate(self.shards):
            cur[g::self.world] = sh["base"]
        out = np.empty((self.V1, self.len, self.d), np.float32)
        for f in range(self.len):
            n, r = self.events(f)
            cur[np.asarray(n)] = r
            out[:, f] = cur
        return out

    def in_memory(self) -> "History":
        """The same history with every array read into host memory."""
        return History(self.meta, [{k: np.array(a) for k, a in sh.items()} for sh in self.shards])


def from_dense(history, T: int) -> History:
    """Logical form (world 1) of a dense history [V1, Th, d] (chronological; numpy array or torch tensor, device included):
    the last min(Th, T) snapshots, the first of them as the base rows, and as the events of position s the rows of snapshot s
    that differ from snapshot s - 1 (elementwise `!=`: a row holding a NaN always counts as changed). base / ev_row are
    views or gathers of `history` of its own type; batch_idx / steps_done / edges_done are 0."""
    V1, Th, d = (int(x) for x in history.shape)
    if Th > T:
        history = history[:, Th - T:]
        Th = T
    nodes = [np.zeros(0, np.int64)]
    for s in range(1, Th):
        m = (history[:, s] != history[:, s - 1]).any(1)
        nodes.append(np.flatnonzero(m if isinstance(m, np.ndarray) else m.cpu().numpy()).astype(np.int64))
    off = np.cumsum([0] + [len(n) for n in nodes]).astype(np.int64)
    ev_node = np.concatenate(nodes)
    ev_row = history[ev_node, np.repeat(np.arange(Th, dtype=np.int64), np.diff(off))]
    meta = dict(format=FORMAT, world=1, rank=0, V1=V1, d=d, T=int(T), len=Th, batch_idx=0, steps_done=0, edges_done=0)
    return History(meta, [dict(base=history[:, 0], ev_off=off, ev_node=ev_node, ev_row=ev_row)])


# ---- reading: every check before anything uses the data --------------------------------------------------------------------
def _bad(path: str, msg: str):
    return ValueError(f"checkpoint {path}: {msg}")


def _read_meta(path: str, g: int, world: int) -> dict:
    fn = os.path.join(path, _name(g, "meta"))
    if not os.path.isfile(fn):
        raise _bad(path, f"shard {g} of {world} is missing ({_name(g, 'meta')} not found)" if world else f"no shard 0 ({_name(0, 'meta')} not found)")
    try:
        with open(fn, "rb") as f:
            m = json.loads(f.read(1 << 16).decode())
    except (OSError, UnicodeDecodeError, json.JSONDecodeError) as e:
        raise _bad(path, f"{_name(g, 'meta')} is not a meta file ({e})") from None
    if not isinstance(m, dict) or sorted(m) != sorted(META_KEYS) or any(type(m[k]) is not int for k in META_KEYS):
        raise _bad(path, f"{_name(g, 'meta')} must hold exactly the integer fields {', '.join(META_KEYS)}")
    return m


def _check_meta(path: str, m: dict):
    if m["format"] != FORMAT:
        raise _bad(path, f"format version {m['format']}, this build reads version {FORMAT}")
    ok = (m["world"] >= 1 and 1 <= m["V1"] < 2 ** 31 and m["d"] >= 1 and 1 <= m["T"] <= 128 and 1 <= m["len"] <= m["T"]
          and min(m["batch_idx"], m["steps_done"], m["edges_done"]) >= 0)
    if not ok:
        raise _bad(path, f"meta out of range: {m}")


def _load_array(path: str, g: int, what: str, dtype, shape) -> np.ndarray:
    fn = os.path.join(path, _name(g, what))
    if not os.path.isfile(fn):
        raise _bad(path, f"shard {g} is incomplete ({_name(g, what)} not found)")
    try:
        a = np.load(fn, mmap_mode="r", allow_pickle=False)
    except (ValueError, OSError, EOFError) as e:
        raise _bad(path, f"{_name(g, what)} is not a plain .npy array ({e})") from None
    if not isinstance(a, np.ndarray) or a.dtype != np.dtype(dtype) or a.shape != shape:
        raise _bad(path, f"{_name(g, what)} holds {getattr(a, 'dtype', type(a))} {getattr(a, 'shape', '')}, expected {np.dtype(dtype)} {shape}")
    return a


def read(path: str) -> History:
    """Open and validate the checkpoint in directory `path` (ValueError on any defect): every shard present, the meta
    files agree, arrays of the right dtype and shape, ev_off monotone within the arrays, every node id in [0, V1) and owned
    by the shard that holds it, no node twice in one window position. Arrays stay memory-mapped."""
    path = os.fspath(path)
    m0 = _read_meta(path, 0, 0)
    _check_meta(path, m0)
    N = m0["world"]
    metas = [m0] + [_read_meta(path, g, N) for g in range(1, N)]
    for g, m in enumerate(metas):
        if m["rank"] != g:
            raise _bad(path, f"{_name(g, 'meta')} says rank {m['rank']}")
        diff = [k for k in _AGREE if m[k] != m0[k]]
        if diff:
            raise _bad(path, f"shard {g} disagrees with shard 0 on {', '.join(diff)} (every rank must save after the same step)")
    V1, d, L = m0["V1"], m0["d"], m0["len"]
    shards = []
    for g in range(N):
        ev_off = _load_array(path, g, "ev_off", np.int64, (L + 1,))
        ev_off = np.array(ev_off)
        if ev_off[0] != 0 or np.any(np.diff(ev_off) < 0):
            raise _bad(path, f"{_name(g, 'ev_off')} is not a monotone offset list from 0")
        n_ev = int(ev_off[-1])
        base = _load_array(path, g, "base", np.float32, (rows_of(V1, N, g), d))
        ev_node = _load_array(path, g, "ev_node", np.int64, (n_ev,))
        ev_row = _load_array(path, g, "ev_row", np.float32, (n_ev, d))
        nodes = np.array(ev_node)
        if n_ev:
            if nodes.min() < 0 or nodes.max() >= V1:
                raise _bad(path, f"{_name(g, 'ev_node')} holds a node id outside [0, {V1})")
            if np.any(nodes % N != g):
                raise _bad(path, f"{_name(g, 'ev_node')} holds a node that shard {g} of {N} does not own")
            key = np.sort(np.repeat(np.arange(L, dtype=np.int64), np.diff(ev_off)) * V1 + nodes)
            if np.any(key[1:] == key[:-1]):
                f = int(key[1:][key[1:] == key[:-1]][0] // V1)
                raise _bad(path, f"{_name(g, 'ev_node')} holds a node twice in window position {f}")
        shards.append(dict(base=base, ev_off=ev_off, ev_node=nodes, ev_row=ev_row))
    return History(m0, shards)
