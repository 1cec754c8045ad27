"""Host-fed and online steps on the change-log history (ChangeLogStream.step_host_async / step_host / run_host;
lstep_pe_step_changelog_host / lstep_pe_steps_changelog_host in csrc/host_step.cu). Wherever the same kernels see the same
inputs the results must be BIT-identical: host-fed against resident steps, online (growable CSR, ingest=True) against the
exact CSR of the whole stream, and a run resumed from a checkpoint against the uninterrupted run."""
import numpy as np
import pytest

from common import pe_close, seeded_normal
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


def _model(g, samp, tag="full"):
    from harness import build_dropin
    return build_dropin(tag, g, samp, 172, D, 100, T, K)[0].eval()


def _init(V1, seed=21):
    import torch
    init = seeded_normal(seed, (V1, D), 0.3)
    init[0] = 0
    return torch.from_numpy(init).cuda()


def _empty_stream(model, B, **kw):
    from lstep_b200 import ChangeLogStream
    e = np.zeros(0, np.int64)
    return ChangeLogStream(model, e, e, np.zeros(0), B, K, **kw)


def _state(st):
    return st.head, st.len, st.batch_idx, st.steps_done, st.edges_done


def _online_graph(kind: str, n_edges: int, seed: int):
    """Reddit-shaped or hub (zipf 1.2) stream with coarse times, so that runs of equal times straddle batch boundaries."""
    g = synth.make_graph("reddit", seed=seed, num_edges=n_edges, zipf_s=1.2 if kind == "hub" else 0.8)
    g.node_interact_times = np.floor(g.node_interact_times / 400.0) * 400.0
    return g


def _same_history(torch, a, b):
    assert torch.equal(a.cur, b.cur)
    assert torch.equal(a.export_history(), b.export_history())
    assert _state(a) == _state(b)


@pytest.mark.parametrize("mode", ["step_host", "run_host"])
@pytest.mark.parametrize("B", [200, 2000])
def test_host_fed_matches_resident(torch_cuda, B, mode):
    """Host-fed steps on a ChangeLogStream over an EMPTY edge stream against resident ChangeLogStream.step on the same
    edges and the same exact sampler: the filling (masked) regime, then the steady regime with retiring events, a ragged
    last batch, and the source set passed twice (the query dedup path). B = 200 and B = 2000 run both MLP kernels."""
    torch = torch_cuda
    from lstep_b200 import ChangeLogStream, NeighborSampler
    nb = T + 21
    g = synth.make_graph("reddit", seed=8, num_edges=nb * B - 37)
    V1, E = g.num_nodes + 1, g.num_edges
    src, dst, t = g.src_node_ids, g.dst_node_ids, g.node_interact_times
    exact = NeighborSampler.from_edges(src, dst, g.edge_ids, t, "recent", num_rows=V1)
    m = _model(g, exact)
    init = _init(V1)
    a = ChangeLogStream(m, src, dst, t, B, K, initial_pe=init.clone())
    b = _empty_stream(m, B, initial_pe=init.clone())
    assert b.num_batches == 0 and a.num_batches == nb
    neg = np.random.default_rng(3).integers(1, V1, E).astype(np.int64)
    negd = torch.from_numpy(neg).cuda()
    qs = [src, dst, src, neg]
    if mode == "step_host":
        for i in range(nb):
            lo, hi = i * B, min((i + 1) * B, E)
            oa = a.step(i, [a.src[lo:hi], a.dst[lo:hi], a.src[lo:hi], negd[lo:hi]])
            ob = torch.empty((4, hi - lo, D), device="cuda")
            b.result(b.step_host_async(src[lo:hi], dst[lo:hi], t[lo:hi], [x[lo:hi] for x in qs], out=ob))
            assert torch.equal(oa, ob), i
            assert torch.equal(a.cur, b.cur), i
            assert _state(a) == _state(b), i
    else:
        c = _empty_stream(m, B, initial_pe=init.clone())  # per-step host-fed calls: the same row-sum kernel as run_host
        for i in range(nb):
            lo, hi = i * B, min((i + 1) * B, E)
            a.step(i, [a.src[lo:hi], a.dst[lo:hi], a.src[lo:hi], negd[lo:hi]])
        rb = b.run_host(src, dst, t, qs)
        assert rb.shape == (nb, 4, B)
        for i in range(nb):
            lo, hi = i * B, min((i + 1) * B, E)
            rc = c.step_host(src[lo:hi], dst[lo:hi], t[lo:hi], [x[lo:hi] for x in qs])
            assert np.array_equal(rb[i, :, :hi - lo], rc), i
        assert not rb[-1, :, E - (nb - 1) * B:].any()
        _same_history(torch, b, c)
    _same_history(torch, a, b)
    assert (b.head, b.len, b.edges_done) == ((nb - (T - 1)) % T, T, E)  # (initial_pe: the log starts with one position)
    b.check_errors()


@pytest.mark.parametrize("mode", ["step_host", "run_host"])
@pytest.mark.parametrize("kind", ["reddit", "hub"])
def test_online_matches_exact_sampler(torch_cuda, kind, mode):
    """Online: a ChangeLogStream over an empty edge stream with a growable sampler, every batch ingested by its own host-fed
    step, against the same host-fed calls on the exact sampler of the whole stream. The small slack makes the CSR regrow
    during the run (run_host: in several calls, each of which reserves room for its batches first)."""
    torch = torch_cuda
    from lstep_b200 import NeighborSampler
    B = 200
    nb = T + 21
    g = _online_graph(kind, nb * B - 37, seed=12)
    V1, E = g.num_nodes + 1, g.num_edges
    src, dst, t = g.src_node_ids, g.dst_node_ids, g.node_interact_times
    exact = NeighborSampler.from_edges(src, dst, g.edge_ids, t, "recent", num_rows=V1)
    grow = NeighborSampler.growable(V1, min_slack=1)
    init = _init(V1, seed=5)
    a = _empty_stream(_model(g, exact), B, initial_pe=init.clone())
    b = _empty_stream(_model(g, grow), B, initial_pe=init.clone())
    neg = np.random.default_rng(4).integers(1, V1, E).astype(np.int64)
    qs = [src, dst, neg]
    if mode == "step_host":
        for i in range(nb):
            lo, hi = i * B, min((i + 1) * B, E)
            q = [x[lo:hi] for x in qs]
            ra = a.step_host(src[lo:hi], dst[lo:hi], t[lo:hi], q)
            rb = b.step_host(src[lo:hi], dst[lo:hi], t[lo:hi], q, ingest=True)
            assert np.array_equal(ra, rb), i
    else:
        cuts = [0, 60 * B, 104 * B, 112 * B, E]  # masked, across the switch to the steady regime, steady, steady + ragged
        regrows = []
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            ra = a.run_host(src[lo:hi], dst[lo:hi], t[lo:hi], [x[lo:hi] for x in qs])
            rb = b.run_host(src[lo:hi], dst[lo:hi], t[lo:hi], [x[lo:hi] for x in qs], ingest=True)
            assert np.array_equal(ra, rb), lo
            regrows.append(grow.regrows)
        assert regrows[-1] > regrows[0], regrows  # a later call of the run had to regrow
    assert grow.regrows >= 1
    _same_history(torch, a, b)
    assert b.edges_done == E
    grow.check_errors()
    assert grow.num_entries == 2 * E and grow.next_edge_id == E + 1
    assert np.array_equal(grow.fill.cpu().numpy(), grow._fill_h)


def test_online_resume_from_checkpoint(torch_cuda, tmp_path):
    """An online run saved once while the log fills and once in the steady regime; each is resumed with a growable sampler
    rebuilt from the first edges_done edges and continued online: every later output, the table and the history equal the
    uninterrupted run's."""
    torch = torch_cuda
    from lstep_b200 import NeighborSampler, checkpoint
    B = 200
    nb = T + 21
    g = _online_graph("reddit", nb * B - 37, seed=15)
    V1, E = g.num_nodes + 1, g.num_edges
    src, dst, eid, t = g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times
    neg = np.random.default_rng(6).integers(1, V1, E).astype(np.int64)
    qs = [src, dst, src, neg]
    init = _init(V1, seed=8)
    full = _empty_stream(_model(g, NeighborSampler.growable(V1, min_slack=2)), B, initial_pe=init.clone())
    saves = (37, 108)
    want = []
    for i in range(nb):
        if i in saves:
            assert (i < T) == (full.len < T) and full.edges_done == i * B
            full.save_checkpoint(str(tmp_path / str(i)))
        lo, hi = i * B, min((i + 1) * B, E)
        want.append(full.step_host(src[lo:hi], dst[lo:hi], t[lo:hi], [x[lo:hi] for x in qs], ingest=True))
    for s0 in saves:
        path = str(tmp_path / str(s0))
        e = int(checkpoint.read(path).meta["edges_done"])  # the edges the caller has to give back to the sampler
        assert e == s0 * B
        samp = NeighborSampler.growable(V1, src[:e], dst[:e], eid[:e], t[:e], min_slack=2)
        r = _empty_stream(_model(g, samp), B, checkpoint=path)
        assert (r.len, r.batch_idx, r.steps_done, r.edges_done) == (min(s0 + 1, T), s0, s0, e)
        for i in range(s0, nb):
            lo, hi = i * B, min((i + 1) * B, E)
            if i == s0 + 3:  # the rest of the run in one call
                got = r.run_host(src[lo:], dst[lo:], t[lo:], [x[lo:] for x in qs], ingest=True)
                for j in range(i, nb):
                    n = min(B, E - j * B)
                    assert np.array_equal(got[j - i, :, :n], want[j]), (s0, j)
                break
            assert np.array_equal(r.step_host(src[lo:hi], dst[lo:hi], t[lo:hi], [x[lo:hi] for x in qs], ingest=True), want[i]), (s0, i)
        assert torch.equal(r.cur, full.cur)
        assert torch.equal(r.export_history(), full.export_history())
        assert _state(r)[1:] == _state(full)[1:]  # (loading normalises the ring head away)


def test_rejections(torch_cuda):
    """Bad input is rejected on the host before anything is enqueued: stream position, counters, table and CSR stay as they
    were. A bad query id in batch k of run_host leaves batches [0, k) applied, with the host state following the device,
    and the next call continues as a resident run of the same batches does."""
    torch = torch_cuda
    from lstep_b200 import ChangeLogStream, NeighborSampler
    B = 200
    nb = T + 12
    g = _online_graph("reddit", nb * B, seed=17)
    V1, E = g.num_nodes + 1, g.num_edges
    src, dst, eid, t = g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times
    exact = NeighborSampler.from_edges(src, dst, eid, t, "recent", num_rows=V1)
    grow = NeighborSampler.growable(V1, min_slack=2)
    init = _init(V1, seed=9)
    a = ChangeLogStream(_model(g, exact), src, dst, t, B, K, initial_pe=init.clone())
    mb = _model(g, grow)
    b = _empty_stream(mb, B, initial_pe=init.clone())
    neg = np.random.default_rng(7).integers(1, V1, E).astype(np.int64)
    qs = [src, dst, neg]
    for i in range(3):
        lo, hi = i * B, (i + 1) * B
        a.step(i, [a.src[lo:hi], a.dst[lo:hi], torch.from_numpy(neg[lo:hi]).cuda()])
        b.step_host(src[lo:hi], dst[lo:hi], t[lo:hi], [x[lo:hi] for x in qs], ingest=True)

    snap = lambda: (_state(b), b.cur.clone(), grow.num_entries, grow.next_edge_id, grow.last_time, grow._fill_h.copy(), grow.fill.clone())

    def unchanged(s0):
        s1 = snap()
        assert s1[0] == s0[0] and torch.equal(s1[1], s0[1]) and s1[2:5] == s0[2:5]
        assert np.array_equal(s1[5], s0[5]) and torch.equal(s1[6], s0[6])

    lo, hi = 3 * B, 4 * B
    s0 = snap()
    q = [x[lo:hi].copy() for x in qs]
    q[2][17] = V1  # a query id outside the table
    with pytest.raises(IndexError):
        b.step_host(src[lo:hi], dst[lo:hi], t[lo:hi], q, ingest=True)
    unchanged(s0)
    for bad_src in (V1, V1 + 40):  # an endpoint id outside the table (and the sampler's rows)
        sb = src[lo:hi].copy()
        sb[5] = bad_src
        with pytest.raises(IndexError):
            b.step_host(sb, dst[lo:hi], t[lo:hi], [x[lo:hi] for x in qs], ingest=True)
        unchanged(s0)
    tb = t[lo:hi].copy()
    tb[40] = tb[39] - 1.0  # decreasing times
    with pytest.raises(ValueError):
        b.step_host(src[lo:hi], dst[lo:hi], tb, [x[lo:hi] for x in qs], ingest=True)
    unchanged(s0)
    with pytest.raises(ValueError, match="batch_size.*event_capacity"):
        b.step_host(src[lo:hi + 1], dst[lo:hi + 1], t[lo:hi + 1], [x[lo:hi + 1] for x in qs], ingest=True)
    unchanged(s0)
    mb.set_neighbor_sampler(exact)
    with pytest.raises(ValueError, match="growable"):
        b.step_host(src[lo:hi], dst[lo:hi], t[lo:hi], [x[lo:hi] for x in qs], ingest=True)
    mb.set_neighbor_sampler(grow)
    unchanged(s0)

    # run_host: masked batches 3 .. T-1, then a steady-state call whose batch k = 4 holds a bad query id
    b.run_host(src[lo:T * B], dst[lo:T * B], t[lo:T * B], [x[lo:T * B] for x in qs], ingest=True)
    assert b.len == T
    lo, hi = T * B, (T + 8) * B
    q = [x[lo:hi].copy() for x in qs]
    q[0][4 * B + 11] = V1 + 2
    head0 = b.head
    with pytest.raises(IndexError):
        b.run_host(src[lo:hi], dst[lo:hi], t[lo:hi], q, ingest=True)
    assert (b.head, b.len, b.batch_idx, b.steps_done, b.edges_done) == ((head0 + 4) % T, T, T + 4, T + 4, (T + 4) * B)
    assert grow.num_entries == 2 * (T + 4) * B and grow.next_edge_id == int(eid[(T + 4) * B - 1]) + 1
    assert np.array_equal(grow.fill.cpu().numpy(), grow._fill_h)
    lo = (T + 4) * B
    b.run_host(src[lo:], dst[lo:], t[lo:], [x[lo:] for x in qs], ingest=True)
    for i in range(3, nb):
        lo, hi = i * B, (i + 1) * B
        a.step(i, [a.src[lo:hi], a.dst[lo:hi], torch.from_numpy(neg[lo:hi]).cuda()])
    _same_history(torch, a, b)
    grow.check_errors()


def test_event_capacity_overflow_raises_at_check_errors(torch_cuda):
    """An explicitly small event_capacity keeps the change log's device-side guard: the overflowing host-fed step sets
    FLAG_CHANGELOG_FULL, which check_errors() raises."""
    from lstep_b200 import NeighborSampler, _lib
    B = 200
    g = synth.make_graph("reddit", seed=3, num_edges=4 * B)
    V1 = g.num_nodes + 1
    src, dst, t = g.src_node_ids, g.dst_node_ids, g.node_interact_times
    st = _empty_stream(_model(g, NeighborSampler.growable(V1, min_slack=2)), B, initial_pe=_init(V1), event_capacity=16)
    st.step_host(src[:B], dst[:B], t[:B], [src[:B]], ingest=True)
    with pytest.raises(_lib.LstepError, match="event capacity"):
        st.check_errors()


def test_online_close_to_dense_ring(torch_cuda):
    """The configuration of test_changelog_history_matches_dense_ring (replay_fullu, a one-snapshot history), fed online:
    PEStream and ChangeLogStream, both host-fed with ingest=True from growable samplers that hold the edges before e0. The
    change-log filter groups its sums differently (span sums of G), so the two agree to that test's bar, not bit for bit."""
    torch = torch_cuda
    from common import golden_path
    from harness import build_dropin
    from lstep_b200 import ChangeLogStream, NeighborSampler, PEStream
    z = np.load(golden_path("replay_fullu.npz"))
    d, Tz, Kz, t_dim, F, B = (int(z[k]) for k in ("pe_dim", "T", "K", "time_dim", "feat_dim", "B"))
    V, E, e0 = int(z["V"]), int(z["E"]), int(z["e0"])
    g = synth.make_graph("tiny", seed=int(z["graph_seed"]), num_nodes=V, num_edges=E)
    src, dst, eid, t = g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times
    hist0 = seeded_normal(int(z["hist0_seed"]), (V + 1, 1, d), 0.3)
    hist0[0] = 0
    e = np.zeros(0, np.int64)

    def mk(cls, **kw):
        samp = NeighborSampler.growable(V + 1, src[:e0], dst[:e0], eid[:e0], t[:e0], min_slack=2)
        m = build_dropin("fullu", g, samp, F, d, t_dim, Tz, Kz)[0].eval()
        return cls(m, e, e, np.zeros(0), B, Kz, history=torch.from_numpy(hist0).cuda(), **kw)

    a, b = mk(PEStream), mk(ChangeLogStream, event_capacity=V + 1)
    neg = z["neg_dst"].astype(np.int64)
    n_steps = min((E - e0 + B - 1) // B, Tz + 30)
    assert n_steps > Tz
    for i in range(n_steps):
        lo, hi = e0 + i * B, min(e0 + (i + 1) * B, E)
        q = [src[lo:hi], dst[lo:hi], neg[i][:hi - lo]]
        oa, ob = torch.empty((3, hi - lo, d), device="cuda"), torch.empty((3, hi - lo, d), device="cuda")
        a.result(a.step_host_async(src[lo:hi], dst[lo:hi], t[lo:hi], q, out=oa, ingest=True))
        b.result(b.step_host_async(src[lo:hi], dst[lo:hi], t[lo:hi], q, out=ob, ingest=True))
        ok, w = pe_close(ob.cpu().numpy(), oa.cpu().numpy(), 1e-5)
        assert ok, (i, "outputs", w)
        ok, w = pe_close(b.cur.cpu().numpy(), a.cur.cpu().numpy(), 1e-5)
        assert ok, (i, "table", w)
        assert (a.head, a.len, a.batch_idx) == (b.head, b.len, b.batch_idx)
    ok, w = pe_close(b.export_history().cpu().numpy(), a.export_history().cpu().numpy(), 1e-5)
    assert ok, ("history", w)
