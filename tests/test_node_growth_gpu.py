"""A node set that grows batch by batch (NeighborSampler.add_rows, PEStream / ChangeLogStream / PeerRank .add_nodes and
grow=True on the host-fed steps). New node ids continue after the last live one. The reference of every case is the same
stream built pre-sized to the final V1, the rows above the initially known nodes holding the initial row r0: a grown stream
must compute the same bits (torch.equal / np.array_equal), whatever row capacity it started with."""
import numpy as np
import pytest

from common import seeded_normal
from lstep_b200 import synth

pytestmark = pytest.mark.gpu

T, K, D = 100, 20, 172


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    from lstep_b200 import _lib
    assert _lib.load().lstep_device_ok() == 1, "not a compute-capability 10.x device"
    return torch


def _dense_graph(name: str, n_edges: int, seed: int, **kw):
    """A synthetic stream whose node ids are renumbered by first appearance (1, 2, ...), as the ids of an online stream
    arrive: a prefix of the stream knows a prefix of the ids. Returns (graph, V1 of the whole stream)."""
    g = synth.make_graph(name, seed=seed, num_edges=n_edges, **kw)
    ends = np.stack([g.src_node_ids, g.dst_node_ids], 1).ravel()
    uniq, first = np.unique(ends, return_index=True)
    order = uniq[np.argsort(first)]
    lab = np.zeros(int(ends.max()) + 1, np.int64)
    lab[order] = np.arange(1, len(order) + 1)
    g.src_node_ids, g.dst_node_ids = lab[g.src_node_ids], lab[g.dst_node_ids]
    return g, len(order) + 1


def _known(g, n_edges: int) -> int:
    """V1 of the nodes the first n_edges edges know."""
    return int(max(g.src_node_ids[:n_edges].max(), g.dst_node_ids[:n_edges].max())) + 1


def _model(g, samp, tag="full"):
    from harness import build_dropin
    return build_dropin(tag, g, samp, 172, D, 100, T, K)[0].eval()


def _init(V1, V1_0, seed=21):
    """Initial rows: seeded for the nodes known at the start, r0 = 0 for the rest (the pre-sized stream's late rows)."""
    import torch
    init = seeded_normal(seed, (V1, D), 0.3)
    init[0] = 0
    init[V1_0:] = 0
    return torch.from_numpy(init).cuda()


def _negatives(g, seed=3):
    """One negative destination per edge among the ids known up to that edge."""
    cm = np.maximum.accumulate(np.maximum(g.src_node_ids, g.dst_node_ids))
    return (np.random.default_rng(seed).random(len(cm)) * cm).astype(np.int64) + 1


def _stream(cls, model, B, **kw):
    e = np.zeros(0, np.int64)
    return cls(model, e, e, np.zeros(0), B, K, **kw)


def _pair(cls, g, V1, V1_0, B, cap_extra, init=None, **kw):
    """(pre-sized stream, growing stream), each on its own model and growable sampler."""
    from lstep_b200 import NeighborSampler
    init = _init(V1, V1_0) if init is None else init
    sa = NeighborSampler.growable(V1)
    a = _stream(cls, _model(g, sa), B, initial_pe=init.clone(), **kw)
    sb = NeighborSampler.growable(V1_0, row_capacity=V1_0 + cap_extra)
    b = _stream(cls, _model(g, sb), B, initial_pe=init[:V1_0].clone(), row_capacity=V1_0 + cap_extra, **kw)
    return a, b


def _same(torch, a, b, head=True):
    """Same table, history and window; head=False: a resumed stream, whose window starts at slot 0 of its log."""
    assert a.V1 == b.V1
    assert torch.equal(a.cur[:a.V1], b.cur[:b.V1])
    assert torch.equal(a.export_history(), b.export_history())
    assert (a.len, a.batch_idx, a.steps_done) == (b.len, b.batch_idx, b.steps_done)
    assert not head or a.head == b.head


def _batch(g, neg, lo, hi):
    s, d = g.src_node_ids[lo:hi], g.dst_node_ids[lo:hi]
    return s, d, g.node_interact_times[lo:hi], [s, d, neg[lo:hi]]


# ---- 1. sampler ------------------------------------------------------------------------------------------------------
def test_sampler_add_rows_matches_exact(torch_cuda):
    """add_rows + ingest batch by batch, crossing the padded tail and the row capacity several times, against from_edges
    on the same edges with num_rows = the live rows; an id at or above the live rows still raises IndexError."""
    torch = torch_cuda
    from lstep_b200 import NeighborSampler
    from lstep_b200.sampler import new_row_need
    B = 200
    g, V1 = _dense_graph("reddit", 60 * B, seed=7)
    src, dst, t = g.src_node_ids, g.dst_node_ids, g.node_interact_times
    V1_0 = _known(g, B)
    samp = NeighborSampler.growable(V1_0, row_capacity=V1_0 + 10, min_slack=2)
    caps = {samp.row_cap}
    for b in range(60):
        lo, hi = b * B, (b + 1) * B
        k = _known(g, hi) - samp.num_rows
        if k > 0:
            assert samp.add_rows(k, new_row_need(src[lo:hi], dst[lo:hi], samp.num_rows, k)) == _known(g, hi) - k
        samp.ingest(src[lo:hi], dst[lo:hi], lo + 1, t[lo:hi])
        caps.add(samp.row_cap)
        if b % 6 == 5 or b == 59:
            ex = NeighborSampler.from_edges(src[:hi], dst[:hi], np.arange(1, hi + 1), t[:hi], "recent", num_rows=samp.num_rows)
            ids = np.arange(samp.num_rows, dtype=np.int64)
            for tq in (t[hi - 1] + 1.0, t[lo]):
                qt = np.full(len(ids), tq)
                for x, y in zip(samp.get_historical_neighbors(ids, qt, K), ex.get_historical_neighbors(ids, qt, K)):
                    assert np.array_equal(x, y), b
                qd, qtd = torch.from_numpy(ids).cuda(), torch.from_numpy(qt).cuda()
                for x, y in zip(samp.sample_device(qd, qtd, len(ids), len(ids), K), ex.sample_device(qd, qtd, len(ids), len(ids), K)):
                    assert torch.equal(x, y), b
    assert samp.num_rows == _known(g, 60 * B)
    assert len(caps) >= 3 and samp.regrows >= 2  # the row capacity doubled at least twice; tail regrows as well
    with pytest.raises(IndexError):
        samp.get_historical_neighbors(np.array([samp.num_rows], np.int64), np.array([1e12]), K)
    samp.get_historical_neighbors(np.array([samp.num_rows - 1], np.int64), np.array([1e12]), K)


# ---- 2. / 3. PEStream and ChangeLogStream online ----------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["step_host", "run_host"])
@pytest.mark.parametrize("shape,B", [("reddit", 200), ("flights", 2000)])
@pytest.mark.parametrize("kind", ["PEStream", "ChangeLogStream"])
def test_online_growth_matches_presized(torch_cuda, kind, shape, B, mode):
    """Start knowing the nodes of the first batches; every later batch adds its new nodes (grow=True) and ingests its edges.
    A small initial row capacity makes the table, the history and the sampler reallocate mid-run. Every step's row sums, the
    full neighbourhood PEs (step_host), the final table and the exported history equal the pre-sized stream's."""
    torch = torch_cuda
    import lstep_b200
    cls = getattr(lstep_b200, kind)
    nb = T + 11
    g, V1 = _dense_graph(shape, nb * B - 37, seed=5)
    E = g.num_edges
    V1_0 = _known(g, 3 * B)
    neg = _negatives(g)
    a, b = _pair(cls, g, V1, V1_0, B, cap_extra=64, max_nodes=V1)
    cap0 = b.row_cap
    if mode == "step_host":
        for i in range(nb):
            lo, hi = i * B, min((i + 1) * B, E)
            s, d, t, qs = _batch(g, neg, lo, hi)
            oa = torch.empty((3, hi - lo, D), device="cuda")
            ob = torch.empty((3, hi - lo, D), device="cuda")
            ra = a.result(a.step_host_async(s, d, t, qs, out=oa, ingest=True))
            rb = b.result(b.step_host_async(s, d, t, qs, out=ob, ingest=True, grow=True))
            assert np.array_equal(ra, rb), i
            assert torch.equal(oa, ob), i
            assert b.V1 == max(V1_0, _known(g, hi)), i  # (negatives are known ids)
    else:
        cuts = [0, 2 * B, (T // 2) * B, (T + 4) * B, E]  # the ring fills in the first calls; growth inside every call
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            s, d, t, qs = _batch(g, neg, lo, hi)
            ra = a.run_host(s, d, t, qs, ingest=True)
            rb = b.run_host(s, d, t, qs, ingest=True, grow=True)
            assert np.array_equal(ra, rb), lo
    assert b.V1 == V1 and b.row_cap > cap0  # reallocated
    _same(torch, a, b)
    a.check_errors()
    b.check_errors()


def test_changelog_checkpoint_after_growth(torch_cuda, tmp_path):
    """A ChangeLogStream grown online, saved mid-run, resumed (with a sampler of the edges so far) and grown further computes
    the bits of the uninterrupted pre-sized run; the checkpoint records the grown V1."""
    torch = torch_cuda
    from lstep_b200 import ChangeLogStream, NeighborSampler, checkpoint as ckpt
    B = 200
    nb = T + 11
    g, V1 = _dense_graph("reddit", nb * B, seed=9)
    V1_0 = _known(g, 2 * B)
    neg = _negatives(g)
    a, b = _pair(ChangeLogStream, g, V1, V1_0, B, cap_extra=32, max_nodes=V1)
    mid = (T + 3) * B
    s, d, t, qs = _batch(g, neg, 0, mid)
    assert np.array_equal(a.run_host(s, d, t, qs, ingest=True), b.run_host(s, d, t, qs, ingest=True, grow=True))
    b.save_checkpoint(str(tmp_path / "ck"))
    V1_mid = b.V1
    assert ckpt.read(str(tmp_path / "ck")).V1 == V1_mid < V1
    s, d, t = g.src_node_ids, g.dst_node_ids, g.node_interact_times
    sc = NeighborSampler.growable(V1_mid, s[:mid], d[:mid], np.arange(1, mid + 1), t[:mid])
    c = ChangeLogStream(_model(g, sc), np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros(0), B, K, checkpoint=str(tmp_path / "ck"),
                        max_nodes=V1)
    for lo in range(mid, nb * B, B):
        sb, db, tb, qs = _batch(g, neg, lo, lo + B)
        assert np.array_equal(a.step_host(sb, db, tb, qs, ingest=True), c.step_host(sb, db, tb, qs, ingest=True, grow=True)), lo
    _same(torch, a, c, head=False)


# ---- 4. explicit rows ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["PEStream", "ChangeLogStream"])
def test_add_nodes_explicit_rows(torch_cuda, kind):
    """add_nodes([n, d] rows) with non-zero per-node rows (in two calls, the second reallocating) against a pre-sized stream
    holding those rows; then online steps."""
    torch = torch_cuda
    import lstep_b200
    cls = getattr(lstep_b200, kind)
    B = 200
    nb = T + 6
    g, V1 = _dense_graph("reddit", nb * B, seed=11)
    V1_0 = _known(g, 2 * B)
    init = torch.from_numpy(seeded_normal(4, (V1, D), 0.3)).cuda()
    init[0] = 0
    a, b = _pair(cls, g, V1, V1_0, B, cap_extra=10, init=init, max_nodes=V1)
    late = init[V1_0:].cpu().numpy()
    assert b.add_nodes(late[:7]) == V1_0
    assert b.add_nodes(late[7:]) == V1_0 + 7
    assert b.V1 == V1 and b.model.neighbor_sampler.num_rows == V1
    _same(torch, a, b)
    neg = _negatives(g)
    for lo in range(0, nb * B, B):
        s, d, t, qs = _batch(g, neg, lo, lo + B)
        assert np.array_equal(a.step_host(s, d, t, qs, ingest=True), b.step_host(s, d, t, qs, ingest=True)), lo
    _same(torch, a, b)


# ---- 5. peer group ---------------------------------------------------------------------------------------------------
PB = 48


def _peer_graph(n_edges, seed=4):
    g, V1 = _dense_graph("tiny_bip", n_edges, seed=seed, num_nodes=300)
    t = g.node_interact_times
    q = (t[-1] - t[0]) / (n_edges / 100.0)
    g.node_interact_times = np.floor(t / q) * q
    return g, V1


def _group(g, world, V1_0, init, cap_extra, checkpoint=None, prefix=0, max_nodes=None):
    from lstep_b200 import NeighborSampler, PeerLocalGroup, PeerRank
    s, d, t = g.src_node_ids, g.dst_node_ids, g.node_interact_times
    samps = [NeighborSampler.growable(V1_0, s[:prefix], d[:prefix], np.arange(1, prefix + 1), t[:prefix], row_capacity=V1_0 + cap_extra)
             for _ in range(world)]
    m = _model(g, samps[0], "fullu")
    kw = dict(checkpoint=checkpoint) if checkpoint is not None else dict(initial_pe=init[:V1_0].clone())
    ranks = [PeerRank(m, r, world, None, None, None, V1_0 - 1, PB, K, sampler=samps[r], row_capacity=V1_0 + cap_extra, max_nodes=max_nodes,
                      **kw)
             for r in range(world)]
    return ranks, PeerLocalGroup(ranks)


def _single_presized(g, V1, init):
    from lstep_b200 import ChangeLogStream, NeighborSampler
    sa = NeighborSampler.growable(V1)
    return _stream(ChangeLogStream, _model(g, sa, "fullu"), PB, initial_pe=init.clone())


def _same_group(torch, single, ranks):
    hist = single.export_history()
    for rk in ranks:
        assert rk.V1 == single.V1
        assert torch.equal(rk.cur[:rk.V1], single.cur), rk.rank
        assert torch.equal(rk.export_history_rows(), hist[rk.rank::rk.G]), rk.rank


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_peer_group_growth(torch_cuda, world):
    """A host-fed peer group (one process) growing its nodes inside the run, a reallocation included: every step's result,
    every rank's replica and its owned history equal the single-GPU pre-sized stream's."""
    torch = torch_cuda
    nb = T + 12
    g, V1 = _peer_graph(nb * PB)
    V1_0 = _known(g, 2 * PB)
    init = _init(V1, V1_0, seed=17)
    neg = _negatives(g)
    single = _single_presized(g, V1, init)
    ranks, grp = _group(g, world, V1_0, init, cap_extra=16, max_nodes=V1)
    cap0 = ranks[0].row_cap
    for lo in range(0, nb * PB, PB):
        s, d, t, qs = _batch(g, neg, lo, lo + PB)
        want = single.step_host(s, d, t, qs, ingest=True)
        got = grp.step_host(s, d, t, qs, ingest=True, grow=True)
        assert np.array_equal(want, got), lo
    grp.barrier()
    assert ranks[0].row_cap > cap0
    _same_group(torch, single, ranks)
    for rk in ranks:
        rk.check_errors()


def test_peer_checkpoint_world2_to_world3_after_growth(torch_cuda, tmp_path):
    """Save at world 2 after growth, resume at world 3, keep growing: the bits of the uninterrupted single-GPU run."""
    torch = torch_cuda
    nb = T + 12
    g, V1 = _peer_graph(nb * PB, seed=6)
    V1_0 = _known(g, 2 * PB)
    init = _init(V1, V1_0, seed=19)
    neg = _negatives(g)
    single = _single_presized(g, V1, init)
    ranks, grp = _group(g, 2, V1_0, init, cap_extra=8, max_nodes=V1)
    mid = 6 * PB  # (the 300-node graph knows all its nodes after a few dozen batches)
    for lo in range(0, mid, PB):
        s, d, t, qs = _batch(g, neg, lo, lo + PB)
        assert np.array_equal(single.step_host(s, d, t, qs, ingest=True), grp.step_host(s, d, t, qs, ingest=True, grow=True)), lo
    grp.barrier()
    for rk in ranks:
        rk.save_checkpoint(str(tmp_path / "ck"))
    V1_mid = ranks[0].V1
    assert V1_mid < V1
    ranks3, grp3 = _group(g, 3, V1_mid, None, cap_extra=4, checkpoint=str(tmp_path / "ck"), prefix=mid, max_nodes=V1)
    for lo in range(mid, nb * PB, PB):
        s, d, t, qs = _batch(g, neg, lo, lo + PB)
        assert np.array_equal(single.step_host(s, d, t, qs, ingest=True), grp3.step_host(s, d, t, qs, ingest=True, grow=True)), lo
    grp3.barrier()
    _same_group(torch, single, ranks3)


# ---- 6. rejections ---------------------------------------------------------------------------------------------------
def test_rejections_leave_state_unchanged(torch_cuda):
    """Each bad call raises before any device write: the stream, its sampler and the rest of the run are those of a run that
    never saw it."""
    torch = torch_cuda
    from lstep_b200 import ChangeLogStream, NeighborSampler
    B = 200
    nb = T + 4
    g, V1 = _dense_graph("reddit", nb * B, seed=13)
    V1_0 = _known(g, 2 * B)
    neg = _negatives(g)
    a, b = _pair(ChangeLogStream, g, V1, V1_0, B, cap_extra=16, max_nodes=V1 + 5)
    a.max_nodes = None
    samp = b.model.neighbor_sampler
    half = (nb // 2) * B
    for lo in range(0, half, B):
        s, d, t, qs = _batch(g, neg, lo, lo + B)
        assert np.array_equal(a.step_host(s, d, t, qs, ingest=True), b.step_host(s, d, t, qs, ingest=True, grow=True))
    snap = (b.V1, b.row_cap, samp.num_rows, samp.row_cap, samp.nnz, samp.regrows, samp.next_edge_id, b.cur[:b.V1].clone())
    s, d, t, qs = _batch(g, neg, half, half + B)
    hi_new = b.V1 + 3
    bad_d = d.copy()
    bad_d[5] = hi_new
    with pytest.raises(IndexError):  # grow=False: an unknown id, as today
        b.step_host(s, bad_d, t, qs, ingest=True)
    with pytest.raises(ValueError):
        b.add_nodes(np.zeros((3, D + 1), np.float32))
    with pytest.raises(ValueError):
        b.add_nodes(np.full((2, D), np.nan, np.float32))
    with pytest.raises(ValueError):
        b.add_nodes([["x"] * D])
    over = d.copy()
    over[0] = V1 + 5  # max_nodes
    with pytest.raises(IndexError):
        b.step_host(s, over, t, qs, ingest=True, grow=True)
    over[0] = 2 ** 31  # int32 node ids
    with pytest.raises(IndexError):
        b.step_host(s, over, t, qs, ingest=True, grow=True)
    with pytest.raises(IndexError):
        b.add_nodes(V1 + 5 - b.V1 + 1)
    bad_t = t.copy()
    bad_t[3] = np.nan  # a batch the ingest rejects must not grow the node set either
    big = d.copy()
    big[1] = b.V1 + 2
    with pytest.raises(ValueError):
        b.step_host(s, big, bad_t, [s, big, qs[2]], ingest=True, grow=True)
    assert (b.V1, b.row_cap, samp.num_rows, samp.row_cap, samp.nnz, samp.regrows, samp.next_edge_id) == snap[:7]
    assert torch.equal(b.cur[:b.V1], snap[7])
    exact = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V1)
    with pytest.raises(ValueError):
        exact.add_rows(1)
    sc = NeighborSampler.growable(V1_0)
    c = _stream(ChangeLogStream, _model(g, sc), B, initial_pe=_init(V1, V1_0)[:V1_0])  # event log sized for V1_0 nodes
    with pytest.raises(ValueError):
        c.add_nodes(V1 - V1_0)
    assert c.V1 == V1_0 and sc.num_rows == V1_0
    for lo in range(half, nb * B, B):
        s, d, t, qs = _batch(g, neg, lo, lo + B)
        assert np.array_equal(a.step_host(s, d, t, qs, ingest=True), b.step_host(s, d, t, qs, ingest=True, grow=True))
    _same(torch, a, b)


def test_group_rejects_alike(torch_cuda):
    """On a group every rank rejects a bad growth alike, and the group goes on with the bits of the single-GPU run."""
    torch = torch_cuda
    nb = T + 3
    g, V1 = _peer_graph(nb * PB, seed=8)
    V1_0 = _known(g, 2 * PB)
    init = _init(V1, V1_0, seed=23)
    neg = _negatives(g)
    single = _single_presized(g, V1, init)
    ranks, grp = _group(g, 3, V1_0, init, cap_extra=8, max_nodes=V1)
    for lo in range(0, nb * PB, PB):
        s, d, t, qs = _batch(g, neg, lo, lo + PB)
        if lo == 10 * PB:
            state = [(rk.V1, rk.row_cap, rk.sampler.num_rows, rk.sampler.nnz) for rk in ranks]
            over = d.copy()
            over[2] = V1
            with pytest.raises(IndexError):
                grp.step_host(s, over, t, [s, over, qs[2]], ingest=True, grow=True)
            bad = d.copy()
            bad[2] = ranks[0].V1 + 1
            with pytest.raises(IndexError):
                grp.step_host(s, bad, t, [s, bad, qs[2]], ingest=True)
            assert state == [(rk.V1, rk.row_cap, rk.sampler.num_rows, rk.sampler.nnz) for rk in ranks]
        assert np.array_equal(single.step_host(s, d, t, qs, ingest=True), grp.step_host(s, d, t, qs, ingest=True, grow=True)), lo
    grp.barrier()
    _same_group(torch, single, ranks)


def test_peer_growth_over_ipc(torch_cuda):
    """Two REAL ranks (one process per GPU under torchrun, CUDA IPC peer pointers) growing their node set online, step by step
    and through run_host, against the pre-sized ChangeLogStream on every rank (tests/run_peer_growth_ipc_check.py). Needs 2
    GPUs."""
    import os
    import subprocess
    import sys
    torch = torch_cuda
    world = 2
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, this box has {torch.cuda.device_count()}")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    port = 29700 + os.getpid() % 90
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(root, "tests", "run_peer_growth_ipc_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    assert res.stdout.count("growing peer group == pre-sized single GPU") == world, res.stdout[-2000:]
