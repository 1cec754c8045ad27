"""The change-log checkpoint format (l-step_b200/checkpoint.py) on the CPU: write / read round trip, resharding a world-N
checkpoint to world M, the replay of the logical form against the dense history, the dense -> logical diff, and every
rejection of a malformed checkpoint."""
import json
import os

import numpy as np
import pytest

from lstep_b200 import checkpoint as ckpt

V1, D, T = 37, 8, 6


def dense_history(seed=0, V1=V1, Th=5, d=D, p=0.3):
    """[V1, Th, d]: every snapshot changes a random ~p of the rows of the previous one."""
    rng = np.random.default_rng(seed)
    h = np.empty((V1, Th, d), np.float32)
    h[:, 0] = rng.standard_normal((V1, d))
    for s in range(1, Th):
        h[:, s] = h[:, s - 1]
        ch = rng.random(V1) < p
        h[ch, s] = rng.standard_normal((int(ch.sum()), d))
    return h


def steady_history(seed=1):
    """A logical history as a full window has it: events at every position, position 0 included."""
    rng = np.random.default_rng(seed)
    off, nodes = [0], []
    for f in range(T):
        n = rng.choice(V1, size=int(rng.integers(0, V1 // 2)), replace=False).astype(np.int64)
        nodes.append(n)
        off.append(off[-1] + len(n))
    ev_node = np.concatenate(nodes)
    meta = dict(format=ckpt.FORMAT, world=1, rank=0, V1=V1, d=D, T=T, len=T, batch_idx=250, steps_done=240, edges_done=12345)
    return ckpt.History(meta, [dict(base=rng.standard_normal((V1, D)).astype(np.float32), ev_off=np.asarray(off, np.int64),
                                    ev_node=ev_node, ev_row=rng.standard_normal((len(ev_node), D)).astype(np.float32))])


def write(path, hist, world):
    for g in range(world):
        meta = dict(hist.meta, world=world, rank=g)
        ckpt.write_shard(str(path), meta, **hist.shard(world, g))


def events_of(hist, f):
    n, r = hist.events(f)
    n, r = np.asarray(n), np.asarray(r)
    o = np.argsort(n)
    return n[o], r[o]


def test_write_read_round_trip(tmp_path):
    h = steady_history()
    write(tmp_path, h, 3)
    assert sorted(os.listdir(tmp_path)) == sorted(f"rank{g}.{k}" for g in range(3) for k in
                                                  ("meta.json", "base.npy", "ev_off.npy", "ev_node.npy", "ev_row.npy"))
    r = ckpt.read(tmp_path)
    assert r.world == 3 and {k: r.meta[k] for k in ("V1", "d", "T", "len", "batch_idx", "steps_done", "edges_done")} == \
        {k: h.meta[k] for k in ("V1", "d", "T", "len", "batch_idx", "steps_done", "edges_done")}
    for g in range(3):
        want = h.shard(3, g)
        for k in ("base", "ev_off", "ev_node", "ev_row"):
            assert np.array_equal(r.shards[g][k], want[k]), (g, k)
    assert np.array_equal(r.replay(), h.replay())
    assert np.array_equal(r.in_memory().replay(), h.replay())
    r.check(V1=V1, d=D, T=T)


@pytest.mark.parametrize("N,M", [(1, 3), (2, 3), (3, 2), (8, 1), (2, 8), (4, 4), (3, 5)])
def test_reshard(tmp_path, N, M):
    h = steady_history(seed=N * 10 + M)
    write(tmp_path, h, N)
    r = ckpt.read(tmp_path)
    new = [r.shard(M, k) for k in range(M)]
    cnt = r.counts(M)
    for f in range(T):
        n0, r0 = events_of(h, f)
        got_n, got_r = [], []
        for k, sh in enumerate(new):
            a, b = sh["ev_off"][f], sh["ev_off"][f + 1]
            assert np.all(sh["ev_node"][a:b] % M == k)  # each event on its owner
            assert cnt[f, k] == b - a
            got_n.append(sh["ev_node"][a:b])
            got_r.append(sh["ev_row"][a:b])
        got_n, got_r = np.concatenate(got_n), np.concatenate(got_r)
        o = np.argsort(got_n)
        assert np.array_equal(got_n[o], n0) and np.array_equal(got_r[o], r0), f  # every event exactly once, rows unchanged
    base = h.shards[0]["base"]
    for k, sh in enumerate(new):
        assert sh["base"].shape == (ckpt.rows_of(V1, M, k), D)
        for loc in range(sh["base"].shape[0]):
            assert np.array_equal(sh["base"][loc], base[loc * M + k])
    # and through the files again at world M
    write(tmp_path / "m", r, M)
    assert np.array_equal(ckpt.read(tmp_path / "m").replay(), h.replay())


def test_replay_equals_dense_replay():
    h = steady_history(seed=7)
    cur = h.shards[0]["base"].copy()
    want = np.empty((V1, T, D), np.float32)
    for f in range(T):
        a, b = h.shards[0]["ev_off"][f], h.shards[0]["ev_off"][f + 1]
        for i in range(a, b):
            cur[h.shards[0]["ev_node"][i]] = h.shards[0]["ev_row"][i]
        want[:, f] = cur
    assert np.array_equal(h.replay(), want)


def test_dense_diff_round_trip():
    torch = pytest.importorskip("torch")
    h = dense_history(Th=5)
    h[3, 2, 1] = np.nan  # a NaN row differs from itself: an event at every later snapshot
    h[3, 3:, 1] = np.nan
    lg = ckpt.from_dense(h, T)
    assert lg.len == 5 and lg.shards[0]["ev_off"][1] == 0
    assert all(3 in events_of(lg, f)[0] for f in range(2, 5))
    assert np.array_equal(lg.replay(), h, equal_nan=True)
    for f in range(1, 5):
        n, _ = events_of(lg, f)
        assert np.array_equal(n, np.flatnonzero((h[:, f] != h[:, f - 1]).any(1)))
    # longer than T: the last T snapshots
    hl = dense_history(seed=3, Th=T + 3)
    lg = ckpt.from_dense(hl, T)
    assert lg.len == T and np.array_equal(lg.replay(), hl[:, 3:])
    # a torch tensor gives the same logical form
    lt = ckpt.from_dense(torch.from_numpy(hl), T)
    assert np.array_equal(lt.shards[0]["ev_node"], lg.shards[0]["ev_node"])
    assert np.array_equal(lt.shards[0]["ev_row"].numpy(), lg.shards[0]["ev_row"])
    # one snapshot: base only
    lg = ckpt.from_dense(h[:, :1], T)
    assert lg.len == 1 and len(lg.shards[0]["ev_node"]) == 0 and np.array_equal(lg.replay(), h[:, :1])


def test_counts():
    h = steady_history(seed=9)
    for M in (1, 2, 5):
        c = h.counts(M)
        for f in range(T):
            n, _ = h.events(f)
            assert np.array_equal(c[f], np.bincount(np.asarray(n) % M, minlength=M))


# ---- rejections -------------------------------------------------------------------------------------------------------------
@pytest.fixture
def good(tmp_path):
    write(tmp_path, steady_history(seed=5), 2)
    return tmp_path


def _meta(path, g, **kw):
    fn = os.path.join(path, f"rank{g}.meta.json")
    with open(fn) as f:
        m = json.load(f)
    m.update(kw)
    with open(fn, "w") as f:
        json.dump(m, f)


def _arr(path, g, what):
    return np.load(os.path.join(path, f"rank{g}.{what}.npy"))


def _put(path, g, what, a, **kw):
    np.save(os.path.join(path, f"rank{g}.{what}.npy"), a, **kw)


def test_good_fixture_reads(good):
    ckpt.read(good)


def test_rejects_missing_shard(good):
    os.remove(good / "rank1.meta.json")
    with pytest.raises(ValueError, match="shard 1 of 2 is missing"):
        ckpt.read(good)


def test_rejects_shard_without_meta(good):
    os.remove(good / "rank0.meta.json")
    with pytest.raises(ValueError, match="no shard 0"):
        ckpt.read(good)


def test_rejects_missing_array(good):
    os.remove(good / "rank1.ev_row.npy")
    with pytest.raises(ValueError, match="incomplete"):
        ckpt.read(good)


def test_interrupted_save_never_looks_valid(good, monkeypatch):
    """A save that dies after its arrays leaves no meta file of that rank (the old one is removed first)."""
    h = ckpt.read(good).in_memory()
    calls = []

    def boom(*a, **k):
        calls.append(1)
        if len(calls) == 5:  # the meta file
            raise OSError("disk full")
        return real(*a, **k)
    real = ckpt._replace
    monkeypatch.setattr(ckpt, "_replace", boom)
    with pytest.raises(OSError):
        ckpt.write_shard(str(good), dict(h.meta, world=2, rank=1, steps_done=999), **h.shard(2, 1))
    monkeypatch.undo()
    assert not (good / "rank1.meta.json").exists()
    assert not [f for f in os.listdir(good) if ".tmp" in f]
    with pytest.raises(ValueError, match="missing"):
        ckpt.read(good)


@pytest.mark.parametrize("field", ["world", "V1", "d", "T", "len", "batch_idx", "steps_done", "format"])
def test_rejects_disagreeing_meta(good, field):
    m = json.loads((good / "rank1.meta.json").read_text())
    _meta(good, 1, **{field: m[field] + 1})
    with pytest.raises(ValueError):
        ckpt.read(good)


def test_rejects_wrong_rank_and_bad_meta(good):
    _meta(good, 1, rank=0)
    with pytest.raises(ValueError, match="says rank 0"):
        ckpt.read(good)
    _meta(good, 1, rank=1, steps_done="7")
    with pytest.raises(ValueError, match="integer fields"):
        ckpt.read(good)
    (good / "rank1.meta.json").write_text("{not json")
    with pytest.raises(ValueError, match="not a meta file"):
        ckpt.read(good)


@pytest.mark.parametrize("field,value", [("format", 2), ("len", T + 1), ("T", 129), ("V1", 2 ** 31), ("world", 0)])
def test_rejects_meta_out_of_range(tmp_path, field, value):
    write(tmp_path, steady_history(seed=5), 1)
    _meta(tmp_path, 0, **{field: value})
    with pytest.raises(ValueError):
        ckpt.read(tmp_path)


def test_rejects_model_mismatch(good):
    h = ckpt.read(good)
    h.check(V1=V1, d=D, T=T)
    for kw in (dict(V1=V1 + 1), dict(d=D + 4), dict(T=T + 1)):
        with pytest.raises(ValueError, match=list(kw)[0]):
            h.check(**kw)


@pytest.mark.parametrize("what,mk", [
    ("ev_row", lambda a: a.astype(np.float64)),
    ("base", lambda a: a[:-1]),
    ("base", lambda a: a.astype(">f4")),
    ("ev_node", lambda a: a.astype(np.int32)),
    ("ev_off", lambda a: a[:-1]),
    ("ev_row", lambda a: a[:, :-1]),
])
def test_rejects_dtype_and_shape(good, what, mk):
    _put(good, 1, what, mk(_arr(good, 1, what)))
    with pytest.raises(ValueError):
        ckpt.read(good)


def test_rejects_pickled_object_array(good):
    _put(good, 0, "ev_node", np.array([1, "x", None], dtype=object), allow_pickle=True)
    with pytest.raises(ValueError, match="not a plain .npy"):
        ckpt.read(good)
    with open(good / "rank0.ev_node.npy", "wb") as f:
        import pickle
        pickle.dump({"a": 1}, f)
    with pytest.raises(ValueError, match="not a plain .npy"):
        ckpt.read(good)


def test_rejects_bad_offsets(good):
    off = _arr(good, 1, "ev_off")
    bad = off.copy()
    bad[2], bad[3] = bad[3], bad[2] - 1  # not monotone
    _put(good, 1, "ev_off", bad)
    with pytest.raises(ValueError, match="monotone"):
        ckpt.read(good)
    bad = off.copy()
    bad[-1] += 1  # past the arrays
    _put(good, 1, "ev_off", bad)
    with pytest.raises(ValueError):
        ckpt.read(good)
    bad = off.copy()
    bad[0] = 1
    _put(good, 1, "ev_off", bad)
    with pytest.raises(ValueError, match="monotone"):
        ckpt.read(good)


@pytest.mark.parametrize("value,msg", [(V1 + 1, "outside"), (-1, "outside"), (2, "does not own")])
def test_rejects_bad_node(good, value, msg):
    n = _arr(good, 1, "ev_node")
    n[0] = value
    _put(good, 1, "ev_node", n)
    with pytest.raises(ValueError, match=msg):
        ckpt.read(good)


def test_rejects_node_twice_in_a_position(good):
    off, n = _arr(good, 1, "ev_off"), _arr(good, 1, "ev_node")
    f = int(np.nonzero(np.diff(off) >= 2)[0][0])
    n[off[f] + 1] = n[off[f]]
    _put(good, 1, "ev_node", n)
    with pytest.raises(ValueError, match=f"twice in window position {f}"):
        ckpt.read(good)
