"""Host-fed and online steps on the peer group (PeerRank.step_host_async / step_host / run_host, PeerLocalGroup.step_host;
lstep_pe_step_peer_host / lstep_pe_steps_peer_host in csrc/host_step.cu). Every comparison is BIT-identical: the group's
concatenated shares of the per-query row sums against the single-GPU ChangeLogStream's host-fed steps, every replica's table
after a barrier, the owners' replayed history, and with ingest=True every rank's own growable CSR replica."""
import numpy as np
import pytest

from common import seeded_normal
from lstep_b200 import synth

pytestmark = pytest.mark.gpu

T, K, D, B = 100, 20, 172, 48


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    from lstep_b200 import _lib
    assert _lib.load().lstep_device_ok() == 1, "not a compute-capability 10.x device"
    return torch


def _graph(n_edges: int, seed: int = 4, self_loops: bool = False):
    """The peer-group test graph; coarse times, so that runs of equal times straddle batch boundaries; optionally self-loops."""
    g = synth.make_graph("tiny_bip", seed=seed, num_nodes=300, num_edges=n_edges)
    t = g.node_interact_times
    q = (t[-1] - t[0]) / (n_edges / 100.0)
    g.node_interact_times = np.floor(t / q) * q
    if self_loops:
        g.dst_node_ids = g.dst_node_ids.copy()
        g.dst_node_ids[::97] = g.src_node_ids[::97]
    return g


def _model(g, samp):
    from harness import build_dropin
    return build_dropin("fullu", g, samp, 172, D, 100, T, K)[0].eval()


def _init(V1, seed=17):
    import torch
    init = torch.from_numpy(seeded_normal(seed, (V1, D), 0.3)).cuda()
    init[0] = 0
    return init


def _exact(g):
    from lstep_b200 import NeighborSampler
    return NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=g.num_nodes + 1)


def _grow(g, p: int):
    from lstep_b200 import NeighborSampler
    return NeighborSampler.growable(g.num_nodes + 1, g.src_node_ids[:p], g.dst_node_ids[:p], g.edge_ids[:p], g.node_interact_times[:p],
                                    min_slack=1)


def _single(g, samp, init=None, **kw):
    from lstep_b200 import ChangeLogStream
    e = np.zeros(0, np.int64)
    if init is not None:
        kw["initial_pe"] = init.clone()
    return ChangeLogStream(_model(g, samp), e, e, np.zeros(0), B, K, **kw)


def _host_group(g, world, samplers, init=None, **kw):
    """A host-fed group (no resident stream): one model shared by the ranks, each rank with its sampler."""
    from lstep_b200 import PeerLocalGroup, PeerRank
    m = _model(g, samplers[0])
    if init is not None:
        kw["initial_pe"] = init.clone()
    ranks = [PeerRank(m, r, world, None, None, None, g.num_nodes, B, K, sampler=samplers[r], **kw) for r in range(world)]
    return ranks, PeerLocalGroup(ranks)


def _queries(g, lo, hi, neg):
    return [g.src_node_ids[lo:hi], g.dst_node_ids[lo:hi], g.src_node_ids[lo:hi], neg[lo:hi]]


def _batch(g, lo, hi):
    return g.src_node_ids[lo:hi], g.dst_node_ids[lo:hi], g.node_interact_times[lo:hi]


def _same_state(torch, grp, ranks, single):
    grp.barrier()
    for rk in ranks:
        assert torch.equal(rk.cur, single.cur), rk.rank
        assert (rk.head, rk.len, rk.batch_idx, rk.steps_done, rk.edges_done) == \
            (ranks[0].head, ranks[0].len, single.batch_idx, single.steps_done, single.edges_done), rk.rank


def _same_history(torch, ranks, single):
    h = single.export_history()
    for rk in ranks:
        rk.check_errors()
        assert torch.equal(rk.export_history_rows(), h[rk.rank::rk.G]), rk.rank


def _csr_content(s):
    """(fill, nbr, eid, t) of the real entries of a growable CSR, row by row: independent of the row capacities, which depend
    on when room was reserved."""
    indptr, fill = s.indptr.cpu().numpy(), s.fill.cpu().numpy().astype(np.int64)
    idx = np.repeat(indptr[:-1], fill) + np.arange(int(fill.sum())) - np.repeat(np.cumsum(fill) - fill, fill)
    return fill, s.nbr.cpu().numpy()[idx], s.eid.cpu().numpy()[idx], s.t.cpu().numpy()[idx]


def _same_replicas(torch, samplers):
    a = samplers[0]
    for s in samplers[1:]:
        assert torch.equal(s.fill, a.fill) and torch.equal(s.indptr, a.indptr) and torch.equal(s.nbr, a.nbr)
        assert torch.equal(s.eid, a.eid) and torch.equal(s.t, a.t)
    for s in samplers:
        s.check_errors()
        assert np.array_equal(s.fill.cpu().numpy(), s._fill_h)


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_host_fed_group_matches_single_gpu_and_resident_group(torch_cuda, world):
    """Exact CSR: PeerLocalGroup.step_host against ChangeLogStream.step_host and the resident PeerLocalGroup.step on the same
    batches, through the filling and the steady regime, a ragged last batch, a query set passed twice, and (world 8) ranks
    that own no batch node of some batches."""
    torch = torch_cuda
    from lstep_b200 import PeerLocalGroup, PeerRank
    nb = T + 15
    g = _graph(9000)
    V1, E = g.num_nodes + 1, g.num_edges
    e0 = E - (nb - 1) * B - 7
    exact = _exact(g)
    init = _init(V1)
    single = _single(g, exact, init)
    ranks, grp = _host_group(g, world, [exact] * world, init)
    mr = _model(g, exact)
    res_ranks = [PeerRank(mr, r, world, g.src_node_ids, g.dst_node_ids, g.node_interact_times, g.num_nodes, B, K, init.clone(), start=e0,
                          sampler=exact) for r in range(world)]
    res_grp = PeerLocalGroup(res_ranks)
    assert res_ranks[0].num_batches == nb
    neg = np.random.default_rng(3).integers(1, V1, E).astype(np.int64)
    negd = torch.from_numpy(neg).cuda()
    src_d, dst_d = res_ranks[0].src, res_ranks[0].dst
    for i in range(nb):
        lo, hi = e0 + i * B, min(e0 + (i + 1) * B, E)
        want = single.step_host(*_batch(g, lo, hi), _queries(g, lo, hi, neg))
        got = grp.step_host(*_batch(g, lo, hi), _queries(g, lo, hi, neg))
        assert got.shape == want.shape and np.array_equal(got, want), i
        res_grp.step(i, [src_d[lo:hi], dst_d[lo:hi], src_d[lo:hi], negd[lo:hi]])
        if i % 25 == 0 or i == nb - 1:
            _same_state(torch, grp, ranks, single)
            res_grp.barrier()
            for a, b in zip(ranks, res_ranks):
                assert torch.equal(a.cur, b.cur) and (a.head, a.len, a.epoch.value) == (b.head, b.len, b.epoch.value), (i, a.rank)
    _same_history(torch, ranks, single)
    _same_history(torch, res_ranks, single)


@pytest.mark.parametrize("start", ["empty", "prefix"])
@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_online_group_matches_exact_csr(torch_cuda, world, start):
    """ingest=True, every rank with its own growable sampler (small slack: regrows during the run), from empty or from a
    prefix of the stream, with ties across batches and self-loops: the same row sums as the exact-CSR single-GPU run, the
    same tables and history, and every rank's CSR replica equal to every other's."""
    torch = torch_cuda
    nb = T + 12
    p = 0 if start == "empty" else 1500
    g = _graph(p + nb * B - 7, seed=6, self_loops=True)
    V1, E = g.num_nodes + 1, g.num_edges
    init = _init(V1, seed=5)
    single = _single(g, _exact(g), init)
    samplers = [_grow(g, p) for _ in range(world)]
    ranks, grp = _host_group(g, world, samplers, init)
    neg = np.random.default_rng(4).integers(1, V1, E).astype(np.int64)
    for i in range(nb):
        lo, hi = p + i * B, min(p + (i + 1) * B, E)
        want = single.step_host(*_batch(g, lo, hi), _queries(g, lo, hi, neg))
        got = grp.step_host(*_batch(g, lo, hi), _queries(g, lo, hi, neg), ingest=True)
        assert np.array_equal(got, want), i
    assert samplers[0].regrows >= 1
    assert all(s.num_entries == 2 * E and s.next_edge_id == E + 1 for s in samplers)
    _same_state(torch, grp, ranks, single)
    _same_history(torch, ranks, single)
    _same_replicas(torch, samplers)


def test_world1_run_host_matches_step_host(torch_cuda):
    """World 1, where the whole step runs in one call: PeerRank.run_host (the native multi-batch call once the log is full)
    against per-step step_host calls, on the exact CSR and online from a prefix."""
    torch = torch_cuda
    nb = T + 14
    p = 900
    g = _graph(p + nb * B - 5, seed=8, self_loops=True)
    V1, E = g.num_nodes + 1, g.num_edges
    init = _init(V1, seed=9)
    neg = np.random.default_rng(5).integers(1, V1, E).astype(np.int64)
    cuts = [p, p + 60 * B, p + 104 * B, E]  # filling, across the switch to the steady regime, steady + ragged
    for ingest in (False, True):
        mk = (lambda: _grow(g, p)) if ingest else (lambda: _exact(g))
        sa, sb = mk(), mk()
        (a,), _ = _host_group(g, 1, [sa], init)
        (b,), _ = _host_group(g, 1, [sb], init)
        for lo0, hi0 in zip(cuts[:-1], cuts[1:]):
            ra = a.run_host(*_batch(g, lo0, hi0), _queries(g, lo0, hi0, neg), ingest=ingest)
            for j, lo in enumerate(range(lo0, hi0, B)):
                hi = min(lo + B, hi0)
                rb = b.step_host(*_batch(g, lo, hi), _queries(g, lo, hi, neg), ingest=ingest)
                assert np.array_equal(ra[j, :, :hi - lo], rb), (ingest, lo)
            assert not ra[-1, :, hi0 - lo0 - (len(ra) - 1) * B:].any()
        assert torch.equal(a.cur, b.cur) and torch.equal(a.export_history_rows(), b.export_history_rows())
        assert (a.head, a.len, a.batch_idx, a.steps_done, a.edges_done, a.epoch.value) == \
            (b.head, b.len, b.batch_idx, b.steps_done, b.edges_done, b.epoch.value) == \
            (a.head, T, nb, nb, E - p, (2 * nb) & 0xffffffff)
        if ingest:  # (run_host reserves room for a whole call at once, step_host batch by batch: the layouts may differ)
            for x, y in zip(_csr_content(sa), _csr_content(sb)):
                assert np.array_equal(x, y)
            sa.check_errors()
            sb.check_errors()


@pytest.mark.parametrize("n_from,n_to,s0", [(2, 3, 60), (3, 2, 104), (1, 8, 104)])
def test_online_resume_at_another_world_size(torch_cuda, tmp_path, n_from, n_to, s0):
    """An online group of n_from ranks saves a checkpoint after s0 steps; a group of n_to ranks resumes it with growable
    samplers rebuilt from the first edges_done edges and continues online: every later result, the tables and the history
    equal the uninterrupted run's."""
    torch = torch_cuda
    from lstep_b200 import checkpoint
    nb = T + 10
    g = _graph(nb * B - 11, seed=12, self_loops=True)
    V1, E = g.num_nodes + 1, g.num_edges
    init = _init(V1, seed=8)
    neg = np.random.default_rng(6).integers(1, V1, E).astype(np.int64)
    ranks, grp = _host_group(g, n_from, [_grow(g, 0) for _ in range(n_from)], init)
    path = str(tmp_path / "ck")
    want = []
    for i in range(nb):
        if i == s0:
            for rk in ranks:
                rk.save_checkpoint(path)
        lo, hi = i * B, min((i + 1) * B, E)
        want.append(grp.step_host(*_batch(g, lo, hi), _queries(g, lo, hi, neg), ingest=True))
    e = int(checkpoint.read(path).meta["edges_done"])
    assert e == s0 * B
    samplers = [_grow(g, e) for _ in range(n_to)]
    ranks2, grp2 = _host_group(g, n_to, samplers, checkpoint=path)
    assert (ranks2[0].len, ranks2[0].batch_idx, ranks2[0].steps_done, ranks2[0].edges_done) == (min(s0 + 1, T), s0, s0, e)
    for i in range(s0, nb):
        lo, hi = i * B, min((i + 1) * B, E)
        got = grp2.step_host(*_batch(g, lo, hi), _queries(g, lo, hi, neg), ingest=True)
        assert np.array_equal(got, want[i]), (n_from, n_to, i)
    grp.barrier()
    grp2.barrier()
    for rk in ranks2:
        assert torch.equal(rk.cur, ranks[0].cur), rk.rank
        assert rk.edges_done == E and rk.steps_done == nb
    single = _single(g, _exact(g), init)  # the owners' histories: against the single-GPU run of the same batches
    for i in range(nb):
        lo, hi = i * B, min((i + 1) * B, E)
        single.step_host(*_batch(g, lo, hi), _queries(g, lo, hi, neg))
    _same_history(torch, ranks2, single)
    _same_replicas(torch, samplers)


def test_rejected_batches_change_nothing(torch_cuda):
    """A host batch every rank rejects (bad id, bad times, longer than batch_size, edge ids past int32, a sampler that cannot
    grow) leaves head, len, epoch, fill and the next result unchanged on every rank; then a valid batch steps normally."""
    torch = torch_cuda
    world = 3
    nb = 8
    p = 600
    g = _graph(p + nb * B, seed=17)
    V1, E = g.num_nodes + 1, g.num_edges
    init = _init(V1, seed=9)
    single = _single(g, _exact(g), init)
    samplers = [_grow(g, p) for _ in range(world)]
    ranks, grp = _host_group(g, world, samplers, init)
    neg = np.random.default_rng(7).integers(1, V1, E).astype(np.int64)

    def step(i, **kw):
        lo, hi = p + i * B, p + (i + 1) * B
        want = single.step_host(*_batch(g, lo, hi), _queries(g, lo, hi, neg))
        assert np.array_equal(grp.step_host(*_batch(g, lo, hi), _queries(g, lo, hi, neg), ingest=True, **kw), want), i

    for i in range(3):
        step(i)
    snap = lambda: [((rk.head, rk.len, rk.epoch.value, rk.batch_idx, rk.steps_done, rk.edges_done), rk.cur.clone(), s.fill.clone(),
                     s._fill_h.copy(), s.num_entries, s.next_edge_id, s.last_time) for rk, s in zip(ranks, samplers)]

    def unchanged(s0):
        for a, b in zip(snap(), s0):
            assert a[0] == b[0] and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2]) and np.array_equal(a[3], b[3]) and a[4:] == b[4:]

    s0 = snap()
    lo, hi = p + 3 * B, p + 4 * B
    src, dst, t = _batch(g, lo, hi)
    qs = _queries(g, lo, hi, neg)
    bad = [x.copy() for x in qs]
    bad[3][17] = V1
    cases = [(IndexError, (src, dst, t, bad), {}),
             (IndexError, (np.where(np.arange(B) == 5, V1 + 40, src), dst, t, qs), {}),
             (ValueError, (src, dst, np.where(np.arange(B) == 40, t[39] - 1.0, t), qs), {}),
             (ValueError, (src, dst, np.where(np.arange(B) == 3, np.nan, t), qs), {}),
             (ValueError, (*_batch(g, lo, hi + 1), _queries(g, lo, hi + 1, neg)), {}),
             (ValueError, (src, dst, t, qs), {"edge_id_start": 2 ** 31 - 10})]
    for exc, args, kw in cases:
        with pytest.raises(exc):
            grp.step_host(*args, ingest=True, **kw)
        unchanged(s0)
    step(3)
    for i in range(4, nb):
        step(i)
    _same_state(torch, grp, ranks, single)
    _same_replicas(torch, samplers)


def test_peer_host_over_ipc(torch_cuda):
    """Two REAL ranks (one process per GPU under torchrun, CUDA IPC peer pointers): online steps with ingest, step by step and
    through run_host, against ChangeLogStream on every rank (tests/run_peer_host_ipc_check.py). Needs 2 GPUs."""
    import os
    import subprocess
    import sys
    torch = torch_cuda
    world = 2
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, this box has {torch.cuda.device_count()}")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    port = 29800 + os.getpid() % 90
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(root, "tests", "run_peer_host_ipc_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    assert res.stdout.count("host-fed peer group == single GPU") == world, res.stdout[-2000:]
