"""Growable CSR (csrc/csr_grow.cu, NeighborSampler.growable / ingest, PEStream host-fed steps with ingest=True) against
the exact CSR of the same edges: every lookup, the real entries, and whole streaming runs must be BIT-identical, since
the same kernels read the same entries in the same order."""
import numpy as np
import pytest

from common import seeded_normal
from lstep_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    from lstep_b200 import _lib
    assert _lib.load().lstep_device_ok() == 1, "not a compute-capability 10.x device"
    return torch


def real_entries(s):
    """(indptr, nbr, eid, t) of the real entries of a growable sampler, in the exact CSR's layout; also checks that the
    rest of every row is padding and that the host mirror of fill equals the device's."""
    ip = s.indptr.cpu().numpy()
    f = s.fill.cpu().numpy().astype(np.int64)
    assert np.array_equal(f, s._fill_h)
    assert (f <= np.diff(ip)).all()
    off = np.concatenate([[0], np.cumsum(f)])
    idx = np.repeat(ip[:-1], f) + (np.arange(off[-1]) - np.repeat(off[:-1], f))
    nbr, eid, t = s.nbr.cpu().numpy(), s.eid.cpu().numpy(), s.t.cpu().numpy()
    pad = np.ones(len(t), bool)
    pad[idx] = False
    assert (nbr[pad] == 0).all() and (eid[pad] == 0).all() and np.isposinf(t[pad]).all()
    return off, nbr[idx], eid[idx], t[idx]


def exact_arrays(s):
    return s.indptr.cpu().numpy(), s.nbr.cpu().numpy(), s.eid.cpu().numpy(), s.t.cpu().numpy()


def stream(kind: str, n_edges: int, seed: int):
    """Reddit- or Flights-shaped stream, or a hub stream (zipf 1.2), with self-loops; the Reddit-shaped ones get coarse
    times so that ties straddle batch boundaries too."""
    if kind == "flights":
        g = synth.make_graph("flights", seed=seed, num_edges=n_edges)
    else:
        g = synth.make_graph("reddit", seed=seed, num_edges=n_edges, zipf_s=1.2 if kind == "hub" else 0.8)
        g.node_interact_times = np.floor(g.node_interact_times / 400.0) * 400.0
    rng = np.random.default_rng(seed)
    loops = rng.random(n_edges) < 0.01
    g.dst_node_ids = np.where(loops, g.src_node_ids, g.dst_node_ids)
    return g


def ragged_bounds(n: int, rng, hi: int = 900):
    b = [0]
    while b[-1] < n:
        b.append(min(n, b[-1] + int(rng.integers(1, hi))))
    return b


@pytest.mark.parametrize("kind", ["reddit", "flights", "hub"])
def test_ingest_from_empty_matches_exact_after_every_batch(torch_cuda, kind):
    torch = torch_cuda
    from lstep_b200 import NeighborSampler
    g = stream(kind, 24_000, seed=11)
    V1 = g.num_nodes + 1
    src, dst, eid, t = g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times
    s = NeighborSampler.growable(V1, min_slack=1)
    rng = np.random.default_rng(2)
    bounds = ragged_bounds(len(src), rng)
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        s.ingest(src[lo:hi], dst[lo:hi], eid[lo:hi], t[lo:hi])
        ex = NeighborSampler.from_edges(src[:hi], dst[:hi], eid[:hi], t[:hi], num_rows=V1)
        q = np.concatenate([src[lo:hi], dst[lo:hi]])
        qt = np.concatenate([t[lo:hi], t[lo:hi]])
        for K in (1, 20):
            got, want = s.get_historical_neighbors(q, qt, K), ex.get_historical_neighbors(q, qt, K)
            for a, b in zip(got, want):
                assert np.array_equal(a, b), (kind, lo, K)
        # just after the batch: every entry of the batch is visible
        qa = qt + 1.0
        for a, b in zip(s.get_historical_neighbors(q, qa, 20), ex.get_historical_neighbors(q, qa, 20)):
            assert np.array_equal(a, b), (kind, lo)
        qd = torch.from_numpy(q).cuda()
        td = torch.from_numpy(qt).cuda()
        a, b = s.sample_device(qd, td, len(q), len(q), 20), ex.sample_device(qd, td, len(q), len(q), 20)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
        for v, tv in ((int(src[hi - 1]), float(t[hi - 1])), (int(dst[lo]), float(t[lo]) + 0.5), (int(src[lo]), np.inf)):
            for x, y in zip(s.find_neighbors_before(v, tv)[:3], ex.find_neighbors_before(v, tv)[:3]):
                assert np.array_equal(x, y), (kind, lo, v)
    s.check_errors()
    assert s.regrows >= 3, s.regrows  # the tiny slack forces several regrows along the way
    assert s.num_entries == 2 * len(src) and s.next_edge_id == int(eid[-1]) + 1 and s.last_time == float(t[-1])
    got = real_entries(s)
    want = exact_arrays(NeighborSampler.from_edges(src, dst, eid, t, num_rows=V1))
    for a, b in zip(got, want):
        assert np.array_equal(a, b), kind


def test_growable_prefix_then_ingest_equals_from_edges(torch_cuda):
    from lstep_b200 import NeighborSampler
    g = stream("flights", 20_000, seed=4)
    V1 = g.num_nodes + 1
    src, dst, eid, t = g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times
    p = 12_345  # inside a run of equal times
    s = NeighborSampler.growable(V1, src[:p], dst[:p], eid[:p], t[:p], min_slack=2)
    assert s.num_entries == 2 * p and s.next_edge_id == int(eid[p - 1]) + 1
    for a, b in zip(real_entries(s), exact_arrays(NeighborSampler.from_edges(src[:p], dst[:p], eid[:p], t[:p], num_rows=V1))):
        assert np.array_equal(a, b)
    for lo in range(p, len(src), 1500):
        s.ingest(src[lo:lo + 1500], dst[lo:lo + 1500], eid[lo:lo + 1500], t[lo:lo + 1500])
    s.check_errors()
    for a, b in zip(real_entries(s), exact_arrays(NeighborSampler.from_edges(src, dst, eid, t, num_rows=V1))):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("mode", ["step_host", "run_host"])
@pytest.mark.parametrize("B", [200, 2000])
def test_online_pestream_matches_exact_sampler(torch_cuda, B, mode):
    """A PEStream over an EMPTY edge stream with a growable sampler, every batch ingested by its own host-fed step, against
    host-fed steps on the exact sampler of the whole stream: masked (ring filling) and steady regime, B = 200 and B = 2000
    (the tcgen05 MLP)."""
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import NeighborSampler, PEStream
    T, K, d = 100, 20, 172
    nb = T + 21
    g = synth.make_graph("reddit", seed=8, num_edges=nb * B - 37)  # the last batch is ragged
    V1, E = g.num_nodes + 1, g.num_edges
    src, dst, t = g.src_node_ids, g.dst_node_ids, g.node_interact_times
    exact = NeighborSampler.from_edges(src, dst, g.edge_ids, t, "recent", num_rows=V1)
    grow = NeighborSampler.growable(V1, min_slack=4)
    ma = build_dropin("full", g, exact, 172, d, 100, T, K)[0].eval()
    mb = build_dropin("full", g, grow, 172, d, 100, T, K)[0].eval()
    init = seeded_normal(21, (V1, d), 0.3)
    init[0] = 0
    a = PEStream(ma, src, dst, t, B, K, initial_pe=torch.from_numpy(init).cuda())
    empty = np.zeros(0, np.int64)
    b = PEStream(mb, empty, empty, np.zeros(0), B, K, initial_pe=torch.from_numpy(init).cuda())
    assert b.num_batches == 0
    neg = np.random.default_rng(3).integers(1, V1, E).astype(np.int64)
    qs = [src, dst, neg]
    if mode == "step_host":
        for i in range(nb):
            lo, hi = i * B, min((i + 1) * B, E)
            q = [x[lo:hi] for x in qs]
            if i in (2, T + 5, nb - 1):  # full [C, n, d] outputs of a few steps
                oa = torch.empty((3, hi - lo, d), device="cuda")
                ob = torch.empty((3, hi - lo, d), device="cuda")
                ra = a.result(a.step_host_async(src[lo:hi], dst[lo:hi], t[lo:hi], q, out=oa))
                rb = b.result(b.step_host_async(src[lo:hi], dst[lo:hi], t[lo:hi], q, out=ob, ingest=True))
                assert torch.equal(oa, ob), i
            else:
                ra = a.step_host(src[lo:hi], dst[lo:hi], t[lo:hi], q)
                rb = b.step_host(src[lo:hi], dst[lo:hi], t[lo:hi], q, ingest=True, edge_id_start=int(g.edge_ids[lo]))
            assert np.array_equal(ra, rb), i
    else:
        ra = a.run_host(src, dst, t, qs)
        rb = b.run_host(src, dst, t, qs, ingest=True)
        assert np.array_equal(ra, rb)
    assert torch.equal(a.cur, b.cur)
    assert torch.equal(a.export_history(), b.export_history())
    assert (a.head, a.len, a.batch_idx) == (b.head, b.len, b.batch_idx)
    grow.check_errors()
    assert grow.num_entries == 2 * E and grow.next_edge_id == E + 1
    for x, y in zip(real_entries(grow), exact_arrays(exact)):
        assert np.array_equal(x, y)
    if mode == "run_host":
        assert grow.regrows == 1  # room for the whole run was reserved up front


def test_dropin_methods_on_growable_sampler(torch_cuda):
    """LSTEP.aggregated_node_embeddings (the feature branch reads edge features by eid) and compute_neighborhood_pe on the
    growable sampler equal the exact sampler's."""
    torch = torch_cuda
    from lstep_b200 import LSTEP, NeighborSampler
    g = stream("reddit", 16_000, seed=5)
    V1, E = g.num_nodes + 1, g.num_edges
    src, dst, eid, t = g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times
    exact = NeighborSampler.from_edges(src, dst, eid, t, num_rows=V1)
    grow = NeighborSampler.growable(V1, min_slack=2)
    for lo in range(0, E, 777):
        grow.ingest(src[lo:lo + 777], dst[lo:lo + 777], eid[lo:lo + 777], t[lo:lo + 777])
    rng = np.random.default_rng(1)
    nf = rng.standard_normal((V1, 172)).astype(np.float32)
    ef = rng.standard_normal((E + 1, 172)).astype(np.float32)
    torch.manual_seed(0)
    m = LSTEP(nf, ef, exact, exact, pe_dim=172, num_neighbors=20, time_feat_dim=100, num_fft_batches=100, device="cuda").to("cuda").eval()
    pe = torch.from_numpy(seeded_normal(9, (V1, 172), 0.3)).cuda()
    q = rng.integers(1, V1, 600)
    qt = np.sort(rng.random(600) * (t[-1] + 10.0))
    with torch.no_grad():
        want = (m.aggregated_node_embeddings(q, qt, 20, time_gap=64), m.compute_neighborhood_pe(pe, q, qt, 20))
        m.set_neighbor_sampler(grow)
        got = (m.aggregated_node_embeddings(q, qt, 20, time_gap=64), m.compute_neighborhood_pe(pe, q, qt, 20))
    for a, b in zip(got, want):
        assert torch.equal(a, b)


def test_rejections_leave_csr_and_fill_unchanged(torch_cuda):
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import NeighborSampler, PEStream
    g = synth.make_graph("tiny", seed=2)
    V1 = g.num_nodes + 1
    src, dst, eid, t = g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times
    s = NeighborSampler.growable(V1, src[:700], dst[:700], eid[:700], t[:700], min_slack=2)
    snap = lambda: [x.clone() for x in (s.indptr, s.nbr, s.eid, s.t, s.fill)]
    state = lambda: (s.num_entries, s.regrows, s.next_edge_id, s.last_time, s._fill_h.copy())
    before, st0 = snap(), state()
    lo, hi = 700, 760
    b = [src[lo:hi].copy(), dst[lo:hi].copy(), eid[lo:hi].copy(), t[lo:hi].copy()]

    def bad(i, pos, val):
        x = [y.copy() for y in b]
        x[i][pos] = val
        return x

    cases = [(bad(3, 5, t[lo + 40]), ValueError),   # times decrease inside the batch
             (bad(3, 0, t[10]), ValueError),        # the batch starts before the last time ingested
             (bad(0, 7, V1), IndexError),           # id >= num_rows
             (bad(1, 7, -1), IndexError),
             (bad(3, 9, np.nan), ValueError),       # non-finite time
             (bad(3, 59, np.inf), ValueError),
             (bad(2, 3, 2 ** 31), ValueError)]      # edge id outside int32
    for x, err in cases:
        with pytest.raises(err):
            s.ingest(*x)
        after = snap()
        assert all(torch.equal(p, q) for p, q in zip(before, after))
        s1 = state()
        assert s1[:4] == st0[:4] and np.array_equal(s1[4], st0[4])
    ex = NeighborSampler.from_edges(src, dst, eid, t, num_rows=V1)
    with pytest.raises(ValueError, match="growable"):
        ex.ingest(*b)
    s.ingest(*b)  # the good batch still goes in
    s.check_errors()
    for p, q in zip(real_entries(s), exact_arrays(NeighborSampler.from_edges(src[:hi], dst[:hi], eid[:hi], t[:hi], num_rows=V1))):
        assert np.array_equal(p, q)
    # the host-fed step rejects before anything is enqueued: ring position and CSR stay as they were
    m = build_dropin("full", g, s, 172, 172, 100, 100, 20)[0].eval()
    init = torch.from_numpy(seeded_normal(3, (V1, 172), 0.3)).cuda()
    e = np.zeros(0, np.int64)
    st = PEStream(m, e, e, np.zeros(0), 32, 20, initial_pe=init)
    lo2 = hi
    st.step_host(src[lo2:lo2 + 32], dst[lo2:lo2 + 32], t[lo2:lo2 + 32], [src[lo2:lo2 + 32]], ingest=True, edge_id_start=int(eid[lo2]))
    before, st0, pos = snap(), state(), (st.head, st.len, st.batch_idx)
    lo3 = lo2 + 32
    tb = t[lo3:lo3 + 32].copy()
    tb[3] = t[0]
    with pytest.raises(ValueError):
        st.step_host(src[lo3:lo3 + 32], dst[lo3:lo3 + 32], tb, [src[lo3:lo3 + 32]], ingest=True)
    sb = src[lo3:lo3 + 32].copy()
    sb[1] = V1 + 3
    with pytest.raises(IndexError):
        st.step_host(sb, dst[lo3:lo3 + 32], t[lo3:lo3 + 32], [src[lo3:lo3 + 32]], ingest=True)
    assert (st.head, st.len, st.batch_idx) == pos
    assert all(torch.equal(p, q) for p, q in zip(before, snap()))
    assert state()[:4] == st0[:4]
    m.set_neighbor_sampler(ex)
    with pytest.raises(ValueError, match="growable"):
        st.step_host(src[lo3:lo3 + 32], dst[lo3:lo3 + 32], t[lo3:lo3 + 32], [src[lo3:lo3 + 32]], ingest=True)
    s.check_errors()


def test_device_guards_of_the_append_kernel(torch_cuda):
    """lstep_csr_ingest called directly (the C ABI, bypassing the host checks): a row without room gets nothing and raises
    LSTEP_FLAG_CSR_FULL; an entry earlier than its row's last one raises LSTEP_FLAG_UNSORTED_STREAM."""
    torch = torch_cuda
    from lstep_b200 import NeighborSampler, _lib
    lib = _lib.load()
    V1 = 8
    s = NeighborSampler.growable(V1, [1, 2], [2, 3], [1, 2], [1.0, 2.0], min_slack=0)  # capacity: row 1: 2, 2: 4, 3: 2, others 0
    cap = np.diff(s.indptr.cpu().numpy())
    assert cap.tolist() == [0, 2, 4, 2, 0, 0, 0, 0]

    def append(a, b, tt):
        x = [torch.tensor(v, dtype=dt, device="cuda") for v, dt in ((a, torch.int64), (b, torch.int64), (tt, torch.float64))]
        _lib.check(lib.lstep_csr_ingest(s.csr_ref, _lib.ptr(s.fill), _lib.ptr(x[0]), _lib.ptr(x[1]), None, 50, _lib.ptr(x[2]), len(a),
                                        _lib.ptr(s._err), _lib.stream_ptr()), "lstep_csr_ingest")
        torch.cuda.synchronize()

    t_before = s.t.clone()
    append([2], [5], [3.0])  # row 2 has room, row 5 has none
    assert s.fill.cpu().tolist() == [0, 1, 3, 1, 0, 0, 0, 0]
    assert s.t[s.indptr[2] + 2].item() == 3.0 and s.eid[s.indptr[2] + 2].item() == 50
    assert torch.equal(s.t[:int(s.indptr[2])], t_before[:int(s.indptr[2])])
    with pytest.raises(_lib.LstepError):
        s.check_errors()
    append([3], [1], [0.5])  # earlier than the last entries of rows 3 and 1
    with pytest.raises(ValueError):
        s.check_errors()


def test_int_edge_ids_equal_explicit_ones(torch_cuda):
    """edge_ids given as an int (the first of consecutive ids), to growable() and to ingest(): the same CSR as from_edges
    with the explicit ids."""
    from lstep_b200 import NeighborSampler
    g = stream("reddit", 9_000, seed=6)
    V1 = g.num_nodes + 1
    src, dst, t = g.src_node_ids, g.dst_node_ids, g.node_interact_times
    eid = np.arange(40, 40 + len(src), dtype=np.int64)
    p = 3_001
    s = NeighborSampler.growable(V1, src[:p], dst[:p], 40, t[:p], min_slack=2)
    for lo in range(p, len(src), 997):
        hi = min(lo + 997, len(src))
        s.ingest(src[lo:hi], dst[lo:hi], 40 + lo, t[lo:hi])
    s.check_errors()
    assert s.next_edge_id == 40 + len(src)
    for a, b in zip(real_entries(s), exact_arrays(NeighborSampler.from_edges(src, dst, eid, t, num_rows=V1))):
        assert np.array_equal(a, b)


def test_failed_step_after_its_append_keeps_the_host_mirror(torch_cuda):
    """A host-fed step that fails after its append was enqueued (here the step's own argument check rejects the ring
    length): the append stays, the sampler's host mirror follows the device, and the next ingesting step continues from
    there."""
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import NeighborSampler, PEStream
    g = synth.make_graph("tiny", seed=3)
    V1 = g.num_nodes + 1
    src, dst, eid, t = g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times
    grow = NeighborSampler.growable(V1, min_slack=2)
    m = build_dropin("full", g, grow, 172, 172, 100, 100, 20)[0].eval()
    e = np.zeros(0, np.int64)
    st = PEStream(m, e, e, np.zeros(0), 50, 20, initial_pe=torch.from_numpy(seeded_normal(4, (V1, 172), 0.3)).cuda())
    for lo in range(0, 150, 50):
        st.step_host(src[lo:lo + 50], dst[lo:lo + 50], t[lo:lo + 50], [src[lo:lo + 50]], ingest=True)
    pos = (st.head, st.len, st.batch_idx)
    st.len = st.T + 1  # lstep_pe_step_host appends the batch, then its step rejects the ring length
    with pytest.raises(ValueError):
        st.step_host(src[150:200], dst[150:200], t[150:200], [src[150:200]], ingest=True)
    st.len = pos[1]
    assert (st.head, st.len, st.batch_idx) == pos
    assert grow.num_entries == 400 and grow.next_edge_id == int(eid[199]) + 1 and grow.last_time == float(t[199])
    for a, b in zip(real_entries(grow), exact_arrays(NeighborSampler.from_edges(src[:200], dst[:200], eid[:200], t[:200], num_rows=V1))):
        assert np.array_equal(a, b)
    st.step_host(src[200:250], dst[200:250], t[200:250], [src[200:250]], ingest=True)
    grow.check_errors()
    for a, b in zip(real_entries(grow), exact_arrays(NeighborSampler.from_edges(src[:250], dst[:250], eid[:250], t[:250], num_rows=V1))):
        assert np.array_equal(a, b)
