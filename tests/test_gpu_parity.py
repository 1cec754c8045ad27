"""Parity of the CUDA path (through the C ABI and the drop-in Python API) against
 (a) golden vectors produced by the unmodified reference, and
 (b) the CPU oracle on seeded inputs at sizes the oracle finishes in seconds.
Bars: indices / CSR bit-exact; fp32 PE values |a-b| <= 1e-5 * max(|b|, rms(b)), every element, for the time encoder,
the DFT filter, the neighbourhood aggregate and the tables after update_pe; the single exception (rows on which
the fp32 reference itself is further than 1e-5 from a float64 evaluation: row 0, hub rows, twice-updated rows) is
stated in tests/golden/common.py::check_updated_table and the rows are named per case in
profiles/r02_parity_errors.json (written from the `parity_log` fixture). Two weight regimes: `full` = PE-MLP weights
x2 (stress), `fullu` = the torch initialisation as it is (realistic). AP / AUC: equal unless the reference's own
positive / negative scores tie within the fp32 noise (tests/harness.py::check_rank_metrics)."""
import numpy as np
import pytest

from common import check_updated_table, checksum, golden_path, pe_close, seeded_edge_feats, seeded_normal, update_error_report
from lstep_b200 import synth
from oracle import lstep_oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    from lstep_b200 import _lib
    lib = _lib.load()
    assert lib.lstep_device_ok() == 1, "not a compute-capability 10.x device"
    return torch


# ------------------------------------------------------------------------------------------ a1/a2
@pytest.mark.parametrize("gname", ["tiny", "tiny_bip", "tiny_ties"])
def test_csr_and_sampler_vs_reference_golden(torch_cuda, gname):
    from lstep_b200 import NeighborSampler
    z = np.load(golden_path(f"sampler_{gname}.npz"))
    s = NeighborSampler.from_edges(z["src"], z["dst"], z["eid"], z["t"], "recent")
    assert np.array_equal(s.indptr.cpu().numpy(), z["csr_indptr"])
    assert np.array_equal(s.nbr.cpu().numpy().astype(np.int64), z["csr_nbr"])
    assert np.array_equal(s.eid.cpu().numpy().astype(np.int64), z["csr_eid"])
    assert np.array_equal(s.t.cpu().numpy(), z["csr_t"])
    for ci in range(int(z["num_cases"])):
        for K in (1, 5, 20, 70):
            a, b, c = s.get_historical_neighbors(z[f"q{ci}_ids"], z[f"q{ci}_t"], K)
            assert a.dtype == np.int64 and b.dtype == np.int64 and c.dtype == np.float32
            assert a.shape == z[f"q{ci}_K{K}_nbr"].shape
            assert np.array_equal(a, z[f"q{ci}_K{K}_nbr"]), (ci, K)
            assert np.array_equal(b, z[f"q{ci}_K{K}_eid"]), (ci, K)
            assert np.array_equal(c, z[f"q{ci}_K{K}_t"]), (ci, K)


def test_adj_list_constructor_matches_edge_builder(torch_cuda):
    """NeighborSampler(adj_list=...) — the reference's constructor form, lists given unsorted."""
    from lstep_b200 import NeighborSampler
    z = np.load(golden_path("sampler_tiny_ties.npz"))
    n_rows = int(max(z["src"].max(), z["dst"].max())) + 1
    adj = [[] for _ in range(n_rows)]
    for s_, d_, e_, t_ in zip(z["src"].tolist(), z["dst"].tolist(), z["eid"].tolist(), z["t"].tolist()):
        adj[s_].append((d_, e_, t_))
        adj[d_].append((s_, e_, t_))
    rng = np.random.default_rng(0)
    # shuffle inside equal-time groups would change the stable order, so only reverse-time-shuffle whole lists
    # by moving a late block to the front: the device sort must restore time order and keep tie order.
    s = NeighborSampler(adj, "recent", seed=3)
    assert np.array_equal(s.nbr.cpu().numpy().astype(np.int64), z["csr_nbr"])
    assert np.array_equal(s.eid.cpu().numpy().astype(np.int64), z["csr_eid"])
    assert s.seed == 3 and s.sample_neighbor_strategy == "recent"
    # unsorted input: rotate every list by a random offset; stable sort by time of the rotated list
    adj2 = []
    for lst in adj:
        k = int(rng.integers(0, len(lst))) if lst else 0
        adj2.append(lst[k:] + lst[:k])
    s2 = NeighborSampler(adj2, "recent")
    want = [sorted(l, key=lambda x: x[2]) for l in adj2]
    assert np.array_equal(s2.nbr.cpu().numpy(), np.array([x[0] for l in want for x in l], dtype=np.int32))
    assert np.array_equal(s2.eid.cpu().numpy(), np.array([x[1] for l in want for x in l], dtype=np.int32))


def test_sampler_errors(torch_cuda):
    from lstep_b200 import NeighborSampler
    z = np.load(golden_path("sampler_tiny.npz"))
    s = NeighborSampler.from_edges(z["src"], z["dst"], z["eid"], z["t"], "recent")
    with pytest.raises(AssertionError):
        s.get_historical_neighbors(np.array([1]), np.array([1.0]), 0)
    with pytest.raises(IndexError):  # Q8
        s.get_historical_neighbors(np.array([1, 10 ** 6]), np.array([1.0, 2.0]), 3)
    # the flag is cleared: the next call works
    a, _, _ = s.get_historical_neighbors(np.array([1]), np.array([1e9]), 3)
    assert a.shape == (1, 3)
    s.sample_neighbor_strategy = "bogus"
    with pytest.raises(ValueError):
        s.get_historical_neighbors(np.array([1]), np.array([1.0]), 3)
    s.sample_neighbor_strategy = "uniform"
    with pytest.raises(NotImplementedError):
        s.get_historical_neighbors(np.array([1]), np.array([1.0]), 3)


@pytest.mark.parametrize("gname,n_edges", [("enron", None), ("reddit", 200_000), ("flights", 300_000)])
def test_sampler_vs_oracle_dataset_shapes(torch_cuda, gname, n_edges):
    """Dataset-shaped graphs (hubs with 10^4+ entries, heavy timestamp ties on the Flights shape)."""
    from lstep_b200 import NeighborSampler
    g = synth.make_graph(gname, seed=0, num_edges=n_edges)
    adj = orc.build_adjacency(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times)
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent")
    indptr, nbr, eid, t = adj.to_csr()
    assert np.array_equal(s.indptr.cpu().numpy(), indptr)
    assert np.array_equal(s.nbr.cpu().numpy().astype(np.int64), nbr)
    assert np.array_equal(s.eid.cpu().numpy().astype(np.int64), eid)
    assert np.array_equal(s.t.cpu().numpy(), t)
    rng = np.random.default_rng(1)
    E = g.num_edges
    lo = E - 400
    q_ids = np.concatenate([g.src_node_ids[lo:], g.dst_node_ids[lo:], rng.integers(0, int(max(g.src_node_ids.max(), g.dst_node_ids.max())) + 1, 200)])
    q_t = np.concatenate([g.node_interact_times[lo:], g.node_interact_times[lo:],
                          g.node_interact_times[rng.integers(0, E, 200)]])
    for K in (20, 2000):
        got = s.get_historical_neighbors(q_ids, q_t, K)
        want = orc.sample_recent(adj, q_ids, q_t, K)
        for a, b in zip(got, want):
            assert a.dtype == b.dtype and np.array_equal(a, b), (gname, K)


# ------------------------------------------------------------------------------------------ a5
def test_time_encoder_all_cosine_branches(torch_cuda, parity_log):
    """TimeEncoder.forward (models/modules.py:27-39) on its own: cos(fp32(dt) * w_j), through lstep_time_features, against
    the oracle's float64 cosine of the same fp32 product. Covers the three argument ranges of accurate_cos (|x| < 2^14,
    2^14 <= |x| < 2^32, |x| >= 2^32 incl. the e >= 214 cosf fallback), negative arguments, zero, denormals and the
    products a timestamp difference actually yields. Bar: 1.2e-7 absolute (one fp32 ulp of values near 1)."""
    torch = torch_cuda
    from lstep_b200 import _lib
    lib = _lib.load()
    w = orc.time_encoder_weights(100)
    rng = np.random.default_rng(0)
    mags = np.concatenate([
        rng.random(4000) * 16384.0,                       # Cody-Waite branch
        2.0 ** (14 + 18 * rng.random(6000)),              # fixed-point Payne-Hanek branch (2^14 .. 2^32)
        2.0 ** (32 + 60 * rng.random(3000)),              # general window (2^32 .. 2^92)
        2.0 ** (92 + 35 * rng.random(500)),               # up to 2^127: e >= 214 takes cosf
        np.array([0.0, 1e-42, 16383.999, 16384.0, 16384.001, 4294967040.0, 4294967296.0, 4294967808.0, 1.1e8, 2.68e6, 3.0e38]),
        np.abs(rng.standard_normal(2000)) * 1e6,          # typical dt in seconds
    ]).astype(np.float32)
    dt = np.concatenate([mags, -mags[::3]]).astype(np.float32)
    dt_d = torch.from_numpy(dt).cuda()
    w_d = torch.from_numpy(w).cuda()
    out = torch.empty((len(dt), len(w)), dtype=torch.float32, device="cuda")
    _lib.check(lib.lstep_time_features(_lib.ptr(dt_d), len(dt), _lib.ptr(w_d), len(w), _lib.ptr(out), _lib.stream_ptr()), "time_features")
    got = out.cpu().numpy()
    want = orc.time_encode(dt, w)  # float64 cosine of the fp32 product, rounded to fp32
    arg = np.abs(dt[:, None] * w[None, :])
    err = np.abs(got.astype(np.float64) - want.astype(np.float64))
    rep = {}
    for name, lo, hi in (("lt_2^14", 0.0, 16384.0), ("2^14..2^32", 16384.0, 4294967296.0), ("ge_2^32", 4294967296.0, np.inf)):
        m = (arg >= lo) & (arg < hi)
        assert m.sum() > 1000, name
        rep[name] = {"n": int(m.sum()), "max_abs_err": float(err[m].max())}
        assert err[m].max() <= 1.2e-7, (name, float(err[m].max()))
    parity_log["a5/time_encoder"] = rep
    # with w = 1 (j = 0) directly on the branch boundaries: every element of dt is its own argument
    one = torch.ones(1, device="cuda")
    out1 = torch.empty((len(dt), 1), dtype=torch.float32, device="cuda")
    _lib.check(lib.lstep_time_features(_lib.ptr(dt_d), len(dt), _lib.ptr(one), 1, _lib.ptr(out1), _lib.stream_ptr()), "time_features")
    e1 = np.abs(out1.cpu().numpy()[:, 0].astype(np.float64) - np.cos(dt.astype(np.float64)))
    assert e1.max() <= 1.2e-7, float(e1.max())
    assert (np.abs(dt) >= 2.0 ** 92).sum() > 100  # the cosf fallback was reached


# ------------------------------------------------------------------------------------------ a3
@pytest.mark.parametrize("tag", ["small", "full"])
def test_dft_filter_vs_reference_golden(torch_cuda, tag):
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import NeighborSampler
    z = np.load(golden_path(f"module_{tag}.npz"))
    d, T, K, t_dim, F = (int(z[k]) for k in ("pe_dim", "T", "K", "time_dim", "feat_dim"))
    g = synth.make_graph(str(z["gname"]), seed=0)
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent")
    lstep = build_dropin(tag, g, s, F, d, t_dim, T, K)[0].eval()
    V1 = g.num_nodes + 1
    with torch.no_grad():
        for ci, (Th, bidx) in enumerate(z["dft_cases"]):
            hist = torch.from_numpy(seeded_normal(100 + ci, (V1, int(Th), d), 0.5)).cuda()
            y = lstep.fourier_transform_pe(z["dft_ids"], hist, int(bidx))
            ok, worst = pe_close(y.cpu().numpy(), z[f"dft{ci}_out"])
            assert ok, (ci, Th, bidx, worst)
        hist = torch.from_numpy(seeded_normal(99, (V1, T, d), 0.5)).cuda()
        y = lstep.fourier_transform_pe(z["dft_ids"][:1], hist, 3)
        assert tuple(y.shape) == (d,)
        assert pe_close(y.cpu().numpy(), z["dft_single_out"])[0]
        # a non-contiguous history view (the loops pass slices of a longer tensor before cloning)
        big = torch.from_numpy(seeded_normal(100 + 7, (V1, T, d), 0.5)).cuda()
        padded = torch.zeros((V1, T + 3, d), device="cuda")
        padded[:, 3:, :] = big
        y = lstep.fourier_transform_pe(z["dft_ids"], padded[:, 3:, :], int(z["dft_cases"][7][1]))
        assert pe_close(y.cpu().numpy(), z["dft7_out"])[0]
        with pytest.raises(RuntimeError):
            lstep.fourier_transform_pe(z["dft_ids"], torch.zeros((V1, T + 1, d), device="cuda"), 0)
        with pytest.raises(IndexError):
            lstep.fourier_transform_pe(np.array([V1 + 5]), hist, 0)
        with pytest.raises(RuntimeError):
            lstep.fourier_transform_pe(z["dft_ids"], hist.cpu(), 0)  # no CPU path


def test_dft_filter_linearity_full_size(torch_cuda):
    """Size-independent property at the Reddit shape (V1=10 985, T=100, d=172, N=300): the filter is
    linear in the history, and equals the oracle on a sample of nodes."""
    torch = torch_cuda
    from harness import build_dropin, lstep_params_np
    from lstep_b200 import NeighborSampler
    g = synth.make_graph("tiny_bip", seed=0)
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent")
    lstep = build_dropin("full", g, s, 172, 172, 100, 100, 20)[0].eval()
    V1, T, d = 10_985, 100, 172
    gen = torch.Generator(device="cuda").manual_seed(0)
    h1 = torch.randn((V1, T, d), device="cuda", generator=gen) * 0.5
    h2 = torch.randn((V1, T, d), device="cuda", generator=gen) * 0.5
    ids = np.sort(np.random.default_rng(0).choice(np.arange(1, V1), 300, replace=False))
    with torch.no_grad():
        y1 = lstep.fourier_transform_pe(ids, h1, 500)
        y2 = lstep.fourier_transform_pe(ids, h2, 500)
        y12 = lstep.fourier_transform_pe(ids, 2.0 * h1 - 0.5 * h2, 500)
    lin = (2.0 * y1 - 0.5 * y2).cpu().numpy()
    ok, worst = pe_close(y12.cpu().numpy(), lin, 2e-5)
    assert ok, worst
    p = lstep_params_np("full")
    sub = ids[:12]
    want = orc.fourier_transform_pe(p, np.arange(len(sub)), h1[torch.from_numpy(sub).cuda()].cpu().numpy(), 500, T)
    ok, worst = pe_close(y1[:12].cpu().numpy(), want)
    assert ok, worst


# ------------------------------------------------------------------------------------------ a6/a7/a8
@pytest.mark.parametrize("tag", ["small", "full", "fullu"])
def test_neighborhood_and_update_vs_reference_golden(torch_cuda, tag, parity_log):
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import NeighborSampler
    z = np.load(golden_path(f"module_{tag}.npz"))
    d, T, K, t_dim, F = (int(z[k]) for k in ("pe_dim", "T", "K", "time_dim", "feat_dim"))
    g = synth.make_graph(str(z["gname"]), seed=0)
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent")
    lstep = build_dropin(tag, g, s, F, d, t_dim, T, K)[0].eval()
    V1 = g.num_nodes + 1
    from harness import lstep_params_np
    p_np = lstep_params_np(tag)
    adj = orc.build_adjacency(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times)
    pe = torch.from_numpy(seeded_normal(5, (V1, d), 0.3)).cuda()
    with torch.no_grad():
        for KK in (K, 3):
            y = lstep.compute_neighborhood_pe(pe, z["nbr_q_ids"], z["nbr_q_t"], num_neighbors=KK)
            ok, worst = pe_close(y.cpu().numpy(), z[f"nbr_out_K{KK}"])
            parity_log[f"golden/{tag}/nbr_K{KK}"] = {"max": worst}
            assert ok, (KK, worst)
        for ci, (st, B) in enumerate(z["upd_cases"]):
            st, B = int(st), int(B)
            src, dst = g.src_node_ids[st:st + B], g.dst_node_ids[st:st + B]
            tt, ee = g.node_interact_times[st:st + B], g.edge_ids[st:st + B]
            ids = synth.unique_batch_nodes(src, dst)
            pe_t = torch.from_numpy(seeded_normal(40 + ci, (V1, d), 0.3)).cuda()
            ret = lstep.update_pe(pe_t, ids, ee, src, dst, tt, tt.max(), num_neighbors=K)
            assert ret is pe_t  # Q7
            with orc.high_precision():
                truth = orc.update_pe(p_np, adj, seeded_normal(40 + ci, (V1, d), 0.3).astype(np.float64), ids, src, dst, tt,
                                      tt.max(), K)
            check_updated_table(pe_t.cpu().numpy(), z[f"upd{ci}_out"], f"golden/{tag}/upd{ci}", truth, log=parity_log)
        st, B = [int(x) for x in z["upd_cases"][0]]
        src, dst = g.src_node_ids[st:st + B], g.dst_node_ids[st:st + B]
        tt, ee = g.node_interact_times[st:st + B], g.edge_ids[st:st + B]
        pe_t = torch.from_numpy(seeded_normal(49, (V1, d), 0.3)).cuda()
        lstep.update_pe(pe_t, z["upd_subset_ids"], ee, src, dst, tt, tt.max(), num_neighbors=K)
        with orc.high_precision():
            truth = orc.update_pe(p_np, adj, seeded_normal(49, (V1, d), 0.3).astype(np.float64), z["upd_subset_ids"], src, dst, tt,
                                  tt.max(), K)
        check_updated_table(pe_t.cpu().numpy(), z["upd_subset_out"], f"golden/{tag}/upd_subset", truth, log=parity_log)
        # running the same update twice from the same input gives the same bits (workspace invariants hold)
        a = torch.from_numpy(seeded_normal(40, (V1, d), 0.3)).cuda()
        b = a.clone()
        st, B = [int(x) for x in z["upd_cases"][2]]
        args = (synth.unique_batch_nodes(g.src_node_ids[st:st + B], g.dst_node_ids[st:st + B]), g.edge_ids[st:st + B],
                g.src_node_ids[st:st + B], g.dst_node_ids[st:st + B], g.node_interact_times[st:st + B],
                g.node_interact_times[st:st + B].max())
        lstep.update_pe(a, *args, num_neighbors=K)
        lstep.update_pe(b, *args, num_neighbors=K)
        assert torch.equal(a, b)
        with pytest.raises(IndexError):
            lstep.update_pe(a, np.array([V1 + 1]), ee, src, dst, tt, tt.max(), num_neighbors=K)


@pytest.mark.parametrize("gname,B,K", [("enron", 200, 20), ("wikipedia", 200, 20), ("reddit", 200, 20), ("flights", 2000, 20)])
def test_pe_step_vs_oracle_dataset_shapes(torch_cuda, gname, B, K, parity_log):
    """One teacher-forced module-boundary step (a3 + 4 x a6 + a7/a8) on every BASELINE dataset shape at its FULL edge
    count and a full history (T = 100 steps per node), against the oracle, in both weight regimes."""
    torch = torch_cuda
    from harness import build_dropin, lstep_params_np
    from lstep_b200 import NeighborSampler
    g = synth.make_graph(gname, seed=0)
    assert g.num_edges == synth.SHAPES[gname]["num_edges"]
    d, T, t_dim = 172, 100, 100
    adj = orc.build_adjacency_fast(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, num_rows=g.num_nodes + 1)
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent",
                                   num_rows=g.num_nodes + 1)
    V1 = g.num_nodes + 1
    lo = g.num_edges - B
    src, dst, tt, ee = (a[lo:lo + B] for a in (g.src_node_ids, g.dst_node_ids, g.node_interact_times, g.edge_ids))
    ids = synth.unique_batch_nodes(src, dst)
    rng = np.random.default_rng(5)
    neg = rng.choice(g.dst_node_ids, B)
    queries = [(src, tt), (dst, tt), (src, tt), (neg, tt)]
    # the oracle only reads the history rows of the batch nodes: keep the host copy to those (the device gets all V1 rows)
    gen = torch.Generator(device="cuda").manual_seed(3)
    pe_h = torch.randn((V1, T, d), device="cuda", generator=gen) * 0.3
    hist_ids = pe_h[torch.from_numpy(ids).cuda()].cpu().numpy()
    last = pe_h[:, -1, :].cpu().numpy()
    for tag in ("fullu", "full"):
        lstep = build_dropin(tag, g, s, 172, d, t_dim, T, K)[0].eval()
        p = lstep_params_np(tag)

        def oracle_step():
            fft = orc.fourier_transform_pe(p, np.arange(len(ids)), hist_ids, 50, T)
            cur = last.astype(fft.dtype)
            cur[ids] = fft
            outs = [orc.compute_neighborhood_pe(p, adj, cur, qi, qt, K) for qi, qt in queries]
            return fft, outs, orc.update_pe(p, adj, cur, ids, src, dst, tt, tt.max(), K)

        fft_o, outs_o, cur_o = oracle_step()
        with orc.high_precision():
            _, outs_truth, cur_truth = oracle_step()
        with torch.no_grad():
            fft = lstep.fourier_transform_pe(ids, pe_h, 50)
            ok, worst = pe_close(fft.cpu().numpy(), fft_o)
            parity_log[f"shape/{gname}/{tag}/dft"] = {"max": worst, "N": int(len(ids))}
            assert ok, (gname, tag, "dft", worst)
            cur = pe_h[:, -1, :].clone()
            cur[torch.from_numpy(ids).cuda()] = fft
            for c, ((qi, qt), want, truth) in enumerate(zip(queries, outs_o, outs_truth)):
                got = lstep.compute_neighborhood_pe(cur, qi, qt, num_neighbors=K)
                check_updated_table(got.cpu().numpy(), want, f"shape/{gname}/{tag}/nbr{c}", truth, log=parity_log)
            lstep.update_pe(cur, ids, ee, src, dst, tt, tt.max(), num_neighbors=K)
        check_updated_table(cur.cpu().numpy(), cur_o, f"shape/{gname}/{tag}/update", cur_truth, log=parity_log)
    del pe_h
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------ training
@pytest.mark.parametrize("tag", ["small", "full"])
def test_training_step_gradients_vs_reference_golden(torch_cuda, tag):
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import NeighborSampler
    z = np.load(golden_path(f"module_{tag}.npz"))
    d, T, K, t_dim, F = (int(z[k]) for k in ("pe_dim", "T", "K", "time_dim", "feat_dim"))
    g = synth.make_graph(str(z["gname"]), seed=0)
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent")
    model = build_dropin(tag, g, s, F, d, t_dim, T, K)
    lstep = model[0]
    model.train()
    V1 = g.num_nodes + 1
    lo = g.num_edges // 2
    hist = torch.from_numpy(seeded_normal(77, (V1, T, d), 0.5)).cuda()
    src, dst, tt = g.src_node_ids[lo:lo + 16], g.dst_node_ids[lo:lo + 16], g.node_interact_times[lo:lo + 16]
    ids = synth.unique_batch_nodes(src, dst)
    fft_pe = lstep.fourier_transform_pe(ids, hist, 2 * T)
    cur = torch.clone(hist[:, -1, :])
    cur[torch.from_numpy(ids).cuda()] = fft_pe
    a = lstep.compute_neighborhood_pe(cur, src, tt, num_neighbors=K)
    b = lstep.compute_neighborhood_pe(cur, dst, tt, num_neighbors=K)
    sd, dd = torch.from_numpy(src).cuda(), torch.from_numpy(dst).cuda()
    loss = (a * b).sum() + (cur[sd] - cur[dd]).pow(2).mean()
    loss.backward()
    assert abs(loss.item() - float(z["train_loss"])) <= 2e-5 * max(1.0, abs(float(z["train_loss"])))
    named = dict(lstep.named_parameters())
    for name in ["fft_filter.weight", "fft_agg.weight", "pe_neighbor_mlp_1.weight", "pe_neighbor_mlp_1.bias",
                 "pe_neighbor_mlp_2.weight", "self_update_neighbor_pe.weight"]:
        want = z["grad_" + name]
        got = named[name].grad.cpu().numpy()
        if np.iscomplexobj(want):
            got, want = np.stack([got.real, got.imag]), np.stack([want.real, want.imag])
        ok, worst = pe_close(got, want, 1e-4)
        assert ok, (name, worst)
    # update_pe stays forward-only and returns the caller's tensor even while autograd records
    ret = lstep.update_pe(cur.detach().clone(), ids, g.edge_ids[lo:lo + 16], src, dst, tt, tt.max(), num_neighbors=K)
    assert ret.grad_fn is None
    for name in ["self_update_pe.weight", "pe_mlp_1.weight", "pe_mlp_2.weight"]:
        assert named[name].grad is None


# ------------------------------------------------------------------------------------------ replay
@pytest.mark.parametrize("tag", ["small", "full", "fullu"])
def test_free_running_replay_ap_auc(torch_cuda, tag, parity_log):
    """>= 200-step free-running eval replay (evaluate_model_utils.py:38-142) against the reference's
    per-batch PE checksums, link probabilities, AP, AUC and final table."""
    torch = torch_cuda
    from harness import build_dropin, check_rank_metrics, oracle_replay_f64, replay_eval
    from lstep_b200 import NeighborSampler
    z = np.load(golden_path(f"replay_{tag}.npz"))
    d, T, K, t_dim, F, tg, B = (int(z[k]) for k in ("pe_dim", "T", "K", "time_dim", "feat_dim", "time_gap", "B"))
    V, E, e0 = int(z["V"]), int(z["E"]), int(z["e0"])
    g = synth.make_graph("tiny", seed=int(z["graph_seed"]), num_nodes=V, num_edges=E)
    assert np.allclose(checksum(g.node_interact_times), z["graph_ck"], rtol=0, atol=1e-6)
    ef = seeded_edge_feats(E, F)
    assert np.allclose(checksum(ef), z["edge_feats_ck"], rtol=0, atol=1e-6)
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent")
    model = build_dropin(tag, g, s, F, d, t_dim, T, K, edge_feats=ef)
    hist0 = seeded_normal(int(z["hist0_seed"]), (V + 1, 1, d), 0.3)
    hist0[0] = 0
    cks = []
    aps, aucs, losses, cur = replay_eval(model, hist0, g, e0, B, z["neg_dst"], T, K, tg,
                                         on_batch=lambda b, c: cks.append(checksum(c.cpu().numpy())))
    cks = np.stack(cks)
    rel = np.abs(cks[:, 1] - z["pe_ck"][:, 1]) / z["pe_ck"][:, 1]
    assert rel.max() < 1e-5, rel.max()
    # final table after the whole free-running recurrence (errors of every step compound): factor 2 of the rule
    check_updated_table(cur.cpu().numpy(), z["last_pe"], f"replay/{tag}/final_table", oracle_replay_f64(tag), factor=2.0, log=parity_log)
    assert len(aps) == len(z["ap"]) >= (200 if tag != "small" else 50)
    rep = check_rank_metrics(replay_eval.last_predicts, z["predicts"], B, aps, aucs, z["ap"], z["auc"], f"replay/{tag}/ap_auc", parity_log)
    assert rep["mean_ap_diff"] < 2e-5 and rep["mean_auc_diff"] < 2e-5, rep
    assert np.abs(losses - z["losses"]).max() < 1e-4


# ------------------------------------------------------------------------------------------ f1 streaming API
@pytest.mark.parametrize("tag", ["small", "full", "fullu"])
def test_stream_api_matches_reference_replay(torch_cuda, tag, parity_log):
    """PEStream (device-resident edge stream + history ring, one C call per batch) against the
    reference's free-running replay: per-batch PE checksums, final table, exported history layout,
    and the neighbourhood outputs against the drop-in method on the same table."""
    torch = torch_cuda
    from harness import build_dropin, oracle_replay_f64
    from lstep_b200 import NeighborSampler, PEStream
    z = np.load(golden_path(f"replay_{tag}.npz"))
    d, T, K, t_dim, F, B = (int(z[k]) for k in ("pe_dim", "T", "K", "time_dim", "feat_dim", "B"))
    V, E, e0 = int(z["V"]), int(z["E"]), int(z["e0"])
    g = synth.make_graph("tiny", seed=int(z["graph_seed"]), num_nodes=V, num_edges=E)
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent",
                                   num_rows=V + 1)
    lstep = build_dropin(tag, g, s, F, d, t_dim, T, K)[0].eval()
    hist0 = seeded_normal(int(z["hist0_seed"]), (V + 1, 1, d), 0.3)
    hist0[0] = 0
    st = PEStream(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, history=torch.from_numpy(hist0).cuda(),
                  start=e0)
    assert st.num_batches == len(z["ap"])
    neg = torch.from_numpy(z["neg_dst"].astype(np.int64)).cuda()
    worst = 0.0
    for b in range(st.num_batches):
        lo, hi, _, _ = st.batch_arrays(b)
        qs = [st.src[lo:hi], st.dst[lo:hi], neg[b][:hi - lo].contiguous()]
        if b in (3, st.num_batches // 2, st.num_batches - 1):
            # the a6 outputs are computed on the table *before* the update: reproduce with the drop-in method
            with torch.no_grad():  # eval path (under autograd the MLP runs as torch Linear layers)
                table = st.cur.clone()
                fft = lstep.fourier_transform_pe(st.ids_np[st.ids_off[b]:st.ids_off[b + 1]], st.export_history(), b)
                table[st.ids[st.ids_off[b]:st.ids_off[b + 1]]] = fft
                want = [lstep.compute_neighborhood_pe(table, q.cpu().numpy(), g.node_interact_times[lo:hi], num_neighbors=K)
                        for q in qs]
            out = st.step(b, qs)
            for c, w in enumerate(want):
                assert torch.equal(out[c], w), (b, c)  # same kernels, same inputs: bit-identical
        else:
            st.step(b, qs)
        ck = checksum(st.cur.cpu().numpy())
        worst = max(worst, abs(ck[1] - z["pe_ck"][b][1]) / z["pe_ck"][b][1])
    assert worst < 1e-5, worst
    check_updated_table(st.cur.cpu().numpy(), z["last_pe"], f"stream/{tag}/final_table", oracle_replay_f64(tag), factor=2.0, log=parity_log)
    h = st.export_history()
    assert tuple(h.shape) == (V + 1, min(T, st.num_batches + 1), d)
    assert torch.equal(h[:, -1, :], st.cur)
    # export -> import round trip keeps stepping consistent (checkpoint interop, EarlyStopping.py:79-104)
    st2 = PEStream(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, history=h, start=e0)
    assert torch.equal(st2.cur, st.cur) and torch.equal(st2.export_history(), h)


def test_host_fed_step_matches_device_resident_step(torch_cuda):
    """PEStream.step_host_async (native stager: pinned slot -> one H2D copy -> step -> row sums -> pinned D2H,
    results read one step behind) against PEStream.step on a twin stream: tables bit-identical after every
    step, row sums equal to the row sums of the device-resident outputs, ids computed natively == np.unique."""
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import NeighborSampler, PEStream
    g = synth.make_graph("tiny_bip", seed=5)
    V, d, T, K, B = g.num_nodes, 172, 100, 20, 64
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V + 1)
    lstep = build_dropin("full", g, s, 172, d, 100, T, K)[0].eval()
    init = seeded_normal(11, (V + 1, d), 0.3)
    init[0] = 0
    e0 = g.num_edges - 12 * B - 17  # last batch is ragged
    a = PEStream(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, initial_pe=torch.from_numpy(init).cuda(), start=e0)
    b = PEStream(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, initial_pe=torch.from_numpy(init).cuda(), start=e0)
    rng = np.random.default_rng(0)
    pending, want_prev = None, None
    for i in range(a.num_batches):
        lo, hi, io, ie = a.batch_arrays(i)
        neg = rng.integers(1, V + 1, hi - lo).astype(np.int64)
        q_np = [g.src_node_ids[lo:hi], g.dst_node_ids[lo:hi], neg]
        out = a.step(i, [torch.from_numpy(np.ascontiguousarray(q)).cuda() for q in q_np])
        want = out.sum(dim=2).cpu().numpy()
        # odd steps pass precomputed ids, even steps let the native side sort + unique
        ids = a.ids_np[io:ie] if i % 2 else None
        tk = b.step_host_async(g.src_node_ids[lo:hi], g.dst_node_ids[lo:hi], g.node_interact_times[lo:hi], q_np, ids=ids)
        if pending is not None:
            got = b.result(pending)
            assert got.shape == want_prev.shape
            np.testing.assert_allclose(got, want_prev, rtol=1e-5, atol=1e-5)
        pending, want_prev = tk, want
        assert torch.equal(a.cur, b.cur), i
    np.testing.assert_allclose(b.result(pending), want_prev, rtol=1e-5, atol=1e-5)
    assert torch.equal(a.export_history(), b.export_history())
    with pytest.raises(ValueError):
        b.step_host_async(g.src_node_ids[:4], g.dst_node_ids[:3], g.node_interact_times[:4], [])
    # ids outside the table are rejected on the host side of the native call, before anything is enqueued
    head, ln, bidx = b.head, b.len, b.batch_idx
    bad = g.src_node_ids[:4].copy()
    bad[2] = V + 7
    with pytest.raises(IndexError):
        b.step_host_async(bad, g.dst_node_ids[:4], g.node_interact_times[:4], [g.dst_node_ids[:4]])
    with pytest.raises(IndexError):
        b.step_host_async(g.src_node_ids[:4], g.dst_node_ids[:4], g.node_interact_times[:4], [bad])
    assert (b.head, b.len, b.batch_idx) == (head, ln, bidx)
    assert torch.equal(a.cur, b.cur)
    s.check_errors()


def test_run_host_matches_device_resident_steps(torch_cuda):
    """PEStream.run_host (a whole run of batches in one native call, both while the ring is filling — per-step calls —
    and in the steady state — lstep_pe_steps_host) against PEStream.step on a twin stream."""
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import NeighborSampler, PEStream
    g = synth.make_graph("tiny_bip", seed=6)
    V, d, T, K, B = g.num_nodes, 172, 100, 20, 16
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V + 1)
    lstep = build_dropin("full", g, s, 172, d, 100, T, K)[0].eval()
    init = seeded_normal(13, (V + 1, d), 0.3)
    init[0] = 0
    e0 = g.num_edges - 118 * B - 5  # 119 batches, the last one ragged: the ring (T = 100) fills after 99 of them
    a = PEStream(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, initial_pe=torch.from_numpy(init).cuda(), start=e0)
    b = PEStream(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, initial_pe=torch.from_numpy(init).cuda(), start=e0)
    rng = np.random.default_rng(0)
    neg = rng.integers(1, V + 1, g.num_edges - e0).astype(np.int64)
    want = np.zeros((a.num_batches, 3, B), np.float32)
    for i in range(a.num_batches):
        lo, hi, _, _ = a.batch_arrays(i)
        out = a.step(i, [a.src[lo:hi], a.dst[lo:hi], torch.from_numpy(neg[lo - e0:hi - e0]).cuda()])
        want[i, :, :hi - lo] = out.sum(dim=2).cpu().numpy()
    got = b.run_host(g.src_node_ids[e0:], g.dst_node_ids[e0:], g.node_interact_times[e0:],
                     [g.src_node_ids[e0:], g.dst_node_ids[e0:], neg])
    assert got.shape == want.shape
    np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-5)
    assert torch.equal(a.cur, b.cur) and torch.equal(a.export_history(), b.export_history())
    assert (b.head, b.len, b.batch_idx) == (a.head, a.len, a.batch_idx)
    s.check_errors()


def test_run_host_error_midway_keeps_host_state_in_step_with_the_ring(torch_cuda):
    """A bad id in batch k of a run_host call: IndexError (like the reference's lookup), batches [0, k) stay applied, and
    the Python-side ring position / batch counter describe exactly that state (a twin stream stepped k times is
    bit-identical, and both continue identically). Also: a larger batch re-creates the native stepper — tickets issued
    before that stay readable and cannot alias new ones."""
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import NeighborSampler, PEStream
    g = synth.make_graph("tiny_bip", seed=8)
    V, d, T, K, B = g.num_nodes, 172, 100, 20, 16
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V + 1)
    lstep = build_dropin("full", g, s, 172, d, 100, T, K)[0].eval()
    init = seeded_normal(17, (V + 1, d), 0.3)
    init[0] = 0
    e0 = g.num_edges - 122 * B
    NF = 104  # good batches first: the ring (T = 100) is full after 99 of them
    mk = lambda: PEStream(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, initial_pe=torch.from_numpy(init).cuda(), start=e0)
    a, b = mk(), mk()
    src, dst, tt = g.src_node_ids[e0:].copy(), g.dst_node_ids[e0:].copy(), g.node_interact_times[e0:]
    fill = NF * B
    b.run_host(src[:fill], dst[:fill], tt[:fill], [src[:fill]])
    k_bad = 5
    bad = src.copy()
    bad[fill + k_bad * B + 3] = V + 11
    with pytest.raises(IndexError):
        b.run_host(bad[fill:fill + 10 * B], dst[fill:fill + 10 * B], tt[fill:fill + 10 * B], [src[fill:fill + 10 * B]])
    for i in range(NF + k_bad):
        lo, hi, _, _ = a.batch_arrays(i)
        a.step(i, [a.src[lo:hi]])
    assert (b.head, b.len, b.batch_idx, b.steps_done) == (a.head, a.len, a.batch_idx, a.steps_done)
    assert torch.equal(a.cur, b.cur) and torch.equal(a.export_history(), b.export_history())
    # both continue from there
    lo = fill + k_bad * B
    got = b.run_host(src[lo:lo + 3 * B], dst[lo:lo + 3 * B], tt[lo:lo + 3 * B], [src[lo:lo + 3 * B]])
    for i in range(NF + k_bad, NF + k_bad + 3):
        l2, h2, _, _ = a.batch_arrays(i)
        out = a.step(i, [a.src[l2:h2]])
    np.testing.assert_allclose(got[-1, 0], out[0].sum(dim=1).cpu().numpy(), rtol=1e-5, atol=1e-5)
    assert torch.equal(a.cur, b.cur)
    # stepper re-creation with a ticket outstanding
    lo = lo + 3 * B
    tk_small = b.step_host_async(src[lo:lo + B], dst[lo:lo + B], tt[lo:lo + B], [src[lo:lo + B]])
    lo += B
    tk_big = b.step_host_async(src[lo:lo + 3 * B], dst[lo:lo + 3 * B], tt[lo:lo + 3 * B], [src[lo:lo + 3 * B]])  # > stepper capacity
    assert tk_big != tk_small and tk_big >> 32 == (tk_small >> 32) + 1
    r_small, r_big = b.result(tk_small), b.result(tk_big)
    assert r_small.shape == (1, B) and r_big.shape == (1, 3 * B)
    with pytest.raises(KeyError):
        b.result(tk_small)  # read once after its stepper is gone
    s.check_errors()


def test_lookup_fused_aggregate_matches_sampler_plus_aggregate(torch_cuda):
    """lstep_nbr_lookup_aggregate (lookup inside the gather kernel) == lstep_sample_recent_compact + lstep_nbr_aggregate,
    bit for bit, including ties, empty histories and K larger than a warp."""
    torch = torch_cuda
    from lstep_b200 import NeighborSampler, _lib
    lib = _lib.load()
    g = synth.make_graph("tiny_ties", seed=3)
    V1, d, t = g.num_nodes + 1, 172, 100
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V1)
    rng = np.random.default_rng(1)
    pe = torch.from_numpy(seeded_normal(8, (V1, d), 0.3)).cuda()
    tw = torch.from_numpy((1.0 / 10 ** np.linspace(0, 9, t, dtype=np.float32)).astype(np.float32)).cuda()
    n = 333
    q = torch.from_numpy(rng.integers(0, V1, n).astype(np.int64)).cuda()  # includes the padding node 0
    qt = torch.from_numpy(rng.choice(g.node_interact_times, n).astype(np.float64) + rng.integers(0, 2, n)).cuda()
    for K in (1, 20, 70):
        nbr = torch.empty((n, K), dtype=torch.int32, device="cuda")
        nt = torch.empty((n, K), dtype=torch.float32, device="cuda")
        S0 = torch.empty((n, d + t), dtype=torch.float32, device="cuda")
        S1 = torch.empty_like(S0)
        _lib.check(lib.lstep_sample_recent_compact(s.csr_ref, _lib.ptr(q), _lib.ptr(qt), n, n, K, _lib.ptr(nbr), _lib.ptr(nt),
                                                   _lib.ptr(s._err), _lib.stream_ptr()), "k1")
        _lib.check(lib.lstep_nbr_aggregate(_lib.ptr(pe), V1, _lib.ptr(qt), _lib.ptr(nbr), _lib.ptr(nt), n, K, _lib.ptr(tw), d, t,
                                           _lib.ptr(S0), _lib.stream_ptr()), "agg")
        _lib.check(lib.lstep_nbr_lookup_aggregate(s.csr_ref, _lib.ptr(q), _lib.ptr(qt), n, K, _lib.ptr(pe), V1, _lib.ptr(tw), d, t,
                                                  _lib.ptr(S1), _lib.ptr(s._err), _lib.stream_ptr()), "fused")
        assert torch.equal(S0, S1), K
    s.check_errors()


def test_stream_is_bit_reproducible(torch_cuda):
    """Two streams fed the same batches end with bit-identical tables and histories: the programmatic-dependent-launch
    chain (kernels resident before their predecessors finish, work done before the dependency wait) and the atomic
    fixed-point accumulation leave no run-to-run freedom."""
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import NeighborSampler, PEStream
    g = synth.make_graph("tiny_bip", seed=9)
    V, d, T, K, B = g.num_nodes, 172, 100, 20, 40
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V + 1)
    lstep = build_dropin("full", g, s, 172, d, 100, T, K)[0].eval()
    init = seeded_normal(12, (V + 1, d), 0.3)
    init[0] = 0
    e0 = g.num_edges - 30 * B
    rng = np.random.default_rng(4)
    negs = [torch.from_numpy(rng.integers(1, V + 1, B).astype(np.int64)).cuda() for _ in range(30)]
    tables = []
    for rep in range(2):
        st = PEStream(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, initial_pe=torch.from_numpy(init).cuda(), start=e0)
        outs = []
        for b in range(st.num_batches):
            lo, hi, _, _ = st.batch_arrays(b)
            outs.append(st.step(b, [st.src[lo:hi], st.dst[lo:hi], negs[b][:hi - lo]]).clone())
        tables.append((st.cur.clone(), st.export_history(), torch.cat([o.reshape(-1) for o in outs])))
    for a, b in zip(tables[0], tables[1]):
        assert torch.equal(a, b)
    s.check_errors()


# ------------------------------------------------------------------------------------------ (e) sharded table
@pytest.mark.parametrize("world", [2, 3])
def test_sharded_ranks_match_single_gpu_stream(torch_cuda, world, parity_log):
    """The node-id sharded algorithm (owner-computes, two row exchanges per step) with all ranks of the
    group emulated in one process on one GPU (LocalGroup) against the single-GPU PEStream and the
    reference's replay checksums: neighbourhood outputs bit-identical (same kernels per row), tables within
    the update bar (phase-B partial sums are combined per rank, so the add order differs)."""
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import LocalGroup, NeighborSampler, PEStream, ShardRank
    tag = "small" if world == 3 else "full"
    z = np.load(golden_path(f"replay_{tag}.npz"))
    d, T, K, t_dim, F, B = (int(z[k]) for k in ("pe_dim", "T", "K", "time_dim", "feat_dim", "B"))
    V, E, e0 = int(z["V"]), int(z["E"]), int(z["e0"])
    g = synth.make_graph("tiny", seed=int(z["graph_seed"]), num_nodes=V, num_edges=E)
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent",
                                   num_rows=V + 1)
    lstep = build_dropin(tag, g, s, F, d, t_dim, T, K)[0].eval()
    hist0 = seeded_normal(int(z["hist0_seed"]), (V + 1, 1, d), 0.3)
    hist0[0] = 0
    init = torch.from_numpy(hist0[:, 0, :]).cuda()
    st = PEStream(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, initial_pe=init, start=e0)
    ranks = [ShardRank(lstep, r, world, g.src_node_ids, g.dst_node_ids, g.node_interact_times, g.edge_ids, V, B, K, init, start=e0)
             for r in range(world)]
    grp = LocalGroup(ranks)
    n_steps = min(st.num_batches, 120)
    worst = 0.0
    for b in range(n_steps):
        lo, hi, _, _ = st.batch_arrays(b)
        nd = z["neg_dst"][b][:hi - lo].astype(np.int64)
        q_np = [g.src_node_ids[lo:hi], g.dst_node_ids[lo:hi], nd]
        want = st.step(b, [st.src[lo:hi], st.dst[lo:hi], torch.from_numpy(nd).cuda()])
        got = grp.step(b, q_np)
        if b < 4 or b % 10 == 0:
            # the padding row pe[0] (a sum of thousands of contributions, reduced in a different grouping when
            # it is split over ranks) enters every padded neighbour slot, so the outputs agree to a few 1e-5
            ok, w = pe_close(got.cpu().numpy(), want.cpu().numpy(), 1e-4)
            assert ok, (b, w)
            q = float(np.quantile(np.abs(got.cpu().numpy() - want.cpu().numpy()) / np.maximum(np.abs(want.cpu().numpy()), 1e-3), 0.99))
            assert q < 1e-4, (b, q)  # 99th percentile; same bar as the element-wise check above (measured 4e-5 .. 5.5e-5)
        ck = checksum(grp.gather_table().cpu().numpy())
        worst = max(worst, abs(ck[1] - z["pe_ck"][b][1]) / z["pe_ck"][b][1])
    assert worst < 1e-5, worst
    from harness import oracle_replay_f64
    truth = oracle_replay_f64(tag) if n_steps == len(z["ap"]) else None
    rep = update_error_report(grp.gather_table().cpu().numpy(), st.cur.cpu().numpy(), truth)
    parity_log[f"sharded/G{world}/table_vs_single_gpu"] = rep
    # float partial rows are summed per rank and then in rank order: same terms, other grouping than the single-GPU
    # exact fixed-point sum -> a few 1e-5 on row 0 / hub rows over 120 free-running steps
    assert rep["max"] <= 1e-4, rep
    # the sharded rings hold exactly the owners' rows of the single-GPU ring
    h = st.export_history()
    for rk in ranks:
        idx = (rk.head + torch.arange(rk.len, device="cuda")) % rk.T
        mine = rk.ring.index_select(1, idx)[:rk.rows_local]
        r2 = update_error_report(mine.cpu().numpy(), h[rk.rank::world].cpu().numpy())
        assert r2["max"] <= 1e-4, (rk.rank, r2)


@pytest.mark.parametrize("world", [2])
def test_sharded_ranks_over_nccl(torch_cuda, world):
    """The same comparison with REAL ranks: one process per GPU under torchrun, NCCL all-to-all row exchanges
    (tests/run_sharded_nccl_check.py: every rank's owned rows and the neighbourhood outputs against the single-GPU
    stream). Needs `world` GPUs on the box; skipped otherwise (the emulated-ranks test above always runs)."""
    import os
    import subprocess
    import sys
    torch = torch_cuda
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, this box has {torch.cuda.device_count()}")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    port = 29600 + os.getpid() % 300
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(root, "tests", "run_sharded_nccl_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    assert res.stdout.count("sharded == single GPU") == world, res.stdout[-2000:]


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_peer_group_emulated_is_bit_identical_to_single_gpu(torch_cuda, world):
    """The peer-group step (owner-computes filter / phase A / phase B, replicas kept equal by the owners' stores, two flag
    barriers per step; l-step_b200/peer.py, csrc/peer.cu) with all ranks emulated in one process — peer pointers are plain
    device pointers, each phase issued for every rank before the next: every replica's table at every step, each rank's
    share of the a6 outputs and the owners' replayed history must be BIT-identical to the single-GPU ChangeLogStream
    through the filling and the steady regime (ragged last batch; ranks that own no batch node at world = 8)."""
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import ChangeLogStream, NeighborSampler, PeerLocalGroup, PeerRank
    g = synth.make_graph("tiny_bip", seed=4, num_nodes=300, num_edges=9000)
    V, d, K, B = g.num_nodes, 172, 20, 48
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V + 1)
    lstep = build_dropin("fullu", g, s, 172, d, 100, 100, K)[0].eval()
    init = torch.from_numpy(seeded_normal(17, (V + 1, d), 0.3)).cuda()
    init[0] = 0
    e0 = g.num_edges - 115 * B - 7
    st = ChangeLogStream(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, initial_pe=init.clone(), start=e0)
    ranks = [PeerRank(lstep, r, world, g.src_node_ids, g.dst_node_ids, g.node_interact_times, V, B, K, init.clone(), start=e0, sampler=s)
             for r in range(world)]
    grp = PeerLocalGroup(ranks)
    neg = torch.from_numpy(np.random.default_rng(3).integers(1, V + 1, g.num_edges - e0).astype(np.int64)).cuda()
    for b in range(st.num_batches):
        lo, hi, _, _ = st.batch_arrays(b)
        qs = [st.src[lo:hi], st.dst[lo:hi], st.src[lo:hi], neg[lo - e0:hi - e0].contiguous()]
        want = st.step(b, qs)
        got = torch.cat(grp.step(b, qs), dim=1)
        assert got.shape == want.shape and torch.equal(got, want), b
        if b % 10 == 0 or b == st.num_batches - 1:
            # a replica holds the other owners' rows of a step once it has pulled them (normally at the next step's
            # barrier 1; here by an extra synchronisation, which later steps must tolerate)
            grp.barrier()
            for rk in ranks:
                assert torch.equal(rk.cur, st.cur), (b, rk.rank)
    grp.barrier()
    for rk in ranks:
        rk.check_errors()
    h = st.export_history()
    for rk in ranks:
        assert torch.equal(rk.export_history_rows(), h[rk.rank::world]), rk.rank


@pytest.mark.parametrize("world", [2])
def test_peer_group_over_ipc(torch_cuda, world):
    """The same comparison with REAL ranks: one process per GPU under torchrun, CUDA IPC peer pointers, NVLink peer stores and
    flag barriers (tests/run_peer_ipc_check.py), step by step and through the native multi-step call. Needs `world` GPUs."""
    import os
    import subprocess
    import sys
    torch = torch_cuda
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, this box has {torch.cuda.device_count()}")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    port = 29900 + os.getpid() % 90
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(root, "tests", "run_peer_ipc_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    assert res.stdout.count("peer group == single GPU") == world, res.stdout[-2000:]


def test_device_resident_stream_rejects_out_of_range_ids(torch_cuda):
    """ADVICE r1 (medium): the device-resident path must not read or write beyond the table. The stream's own ids are
    checked against the table / sampler when the history is adopted (IndexError, like the reference's first lookup, Q8);
    a query id the sampler does not know raises the device error flag (IndexError at check_errors()), yields an empty
    neighbourhood, reads table row 0 as its own row and leaves the update untouched."""
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import NeighborSampler, PEStream
    g = synth.make_graph("tiny_bip", seed=5)
    V, d, T, K, B = g.num_nodes, 172, 100, 20, 32
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V + 1)
    lstep = build_dropin("full", g, s, 172, d, 100, T, K)[0].eval()
    init = torch.from_numpy(seeded_normal(11, (V + 1, d), 0.3)).cuda()
    e0 = g.num_edges - 6 * B
    with pytest.raises(IndexError):  # table smaller than the ids of the stream
        PEStream(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, initial_pe=init[:V - 3], start=e0)
    bad_src = g.src_node_ids.copy()
    bad_src[-1] = V + 9
    with pytest.raises(IndexError):
        PEStream(lstep, bad_src, g.dst_node_ids, g.node_interact_times, B, K, initial_pe=init, start=e0)
    a = PEStream(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, initial_pe=init.clone(), start=e0)
    b = PEStream(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, initial_pe=init.clone(), start=e0)
    lo, hi, _, _ = a.batch_arrays(0)
    good = a.dst[lo:hi].clone()
    bad = good.clone()
    bad[3] = V + 1000  # far outside the table
    bad[7] = -5
    oa = a.step(0, [a.src[lo:hi], good]).clone()
    a.check_errors()  # (the error flag lives in the sampler both streams share)
    ob = b.step(0, [b.src[lo:hi], bad]).clone()
    with pytest.raises(IndexError):
        b.check_errors()
    b.check_errors()  # the flag is cleared by the read
    assert torch.equal(a.cur, b.cur) and torch.equal(a.export_history(), b.export_history())
    keep = torch.ones(hi - lo, dtype=torch.bool, device="cuda")
    keep[3] = keep[7] = False
    assert torch.equal(oa[0], ob[0]) and torch.equal(oa[1][keep], ob[1][keep])
    assert torch.isfinite(ob).all()


def test_every_layout_checks_the_resident_ids_alike(torch_cuda):
    """PEStream, ChangeLogStream and PeerRank make the same check of their resident stream's ids when they adopt their state,
    with the same messages: a negative id and an id past the sampler's rows (inside the table) raise IndexError at
    construction, before a step could index the table with them."""
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import ChangeLogStream, NeighborSampler, PEStream, PeerRank
    g = synth.make_graph("tiny_bip", seed=5)
    V, d, T, K, B = g.num_nodes, 172, 100, 20, 32
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V + 1)
    lstep = build_dropin("full", g, s, 172, d, 100, T, K)[0].eval()
    init = torch.from_numpy(seeded_normal(11, (V + 2, d), 0.3)).cuda()  # one row more than the sampler knows
    e0 = g.num_edges - 6 * B
    for bad, V1, msg in ((-4, V + 1, "edge stream holds node id -4 but the PE table has"),
                         (V + 1, V + 2, f"node id {V + 1} is unknown to the neighbor sampler")):
        src = g.src_node_ids.copy()
        src[-1] = bad
        for cls in (PEStream, ChangeLogStream):
            with pytest.raises(IndexError, match=msg):
                cls(lstep, src, g.dst_node_ids, g.node_interact_times, B, K, initial_pe=init[:V1].clone(), start=e0)
        with pytest.raises(IndexError, match=msg):
            PeerRank(lstep, 0, 1, src, g.dst_node_ids, g.node_interact_times, V1 - 1, B, K, init[:V1].clone(), start=e0, sampler=s)


@pytest.mark.parametrize("layout", ["PEStream", "ChangeLogStream"])
def test_run_check_reads_the_error_flag_while_the_history_fills(torch_cuda, layout):
    """run(check=True) reads the device error flag on every path: also from a history shorter than T, where run() steps
    batch by batch, a query id the sampler does not know raises IndexError."""
    torch = torch_cuda
    import lstep_b200
    from harness import build_dropin
    from lstep_b200 import NeighborSampler
    g = synth.make_graph("tiny_bip", seed=5)
    V, d, T, K, B = g.num_nodes, 172, 100, 20, 32
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V + 1)
    lstep = build_dropin("full", g, s, 172, d, 100, T, K)[0].eval()
    init = torch.from_numpy(seeded_normal(11, (V + 1, d), 0.3)).cuda()
    e0 = g.num_edges - 6 * B
    st = getattr(lstep_b200, layout)(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, initial_pe=init, start=e0)
    assert st.len < st.T
    bad = st.dst[e0:].clone()
    bad[B + 3] = V + 1000
    with pytest.raises(IndexError):
        st.run(0, 3, [st.src[e0:], bad], check=True)
    assert st.steps_done == 3
    st.check_errors()  # (the read cleared the flag)


def test_native_multi_step_run_and_profile_are_bit_identical_to_single_steps(torch_cuda):
    """PEStream.run (lstep_pe_steps: the per-batch loop in C) against PEStream.step, and the same steps with the per-kernel
    event profile switched on (events between the kernels serialise the chain): tables, histories and outputs are
    bit-identical; the profile returns one positive duration per kernel of the step."""
    torch = torch_cuda
    import ctypes
    from harness import build_dropin
    from lstep_b200 import NeighborSampler, PEStream, _lib
    lib = _lib.load()
    g = synth.make_graph("tiny_bip", seed=8)
    V, d, T, K, B = g.num_nodes, 172, 100, 20, 16
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V + 1)
    lstep = build_dropin("full", g, s, 172, d, 100, T, K)[0].eval()
    hist = torch.from_numpy(seeded_normal(21, (V + 1, T, d), 0.3)).cuda()  # full ring: steady state from the first step
    e0 = g.num_edges - 24 * B
    mk = lambda: PEStream(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, history=hist.clone(), start=e0)
    a, b, c = mk(), mk(), mk()
    neg = torch.from_numpy(np.random.default_rng(1).integers(1, V + 1, g.num_edges - e0).astype(np.int64)).cuda()
    n = a.num_batches
    outs_a = torch.empty((n, 3, B, d), device="cuda")
    for i in range(n):
        lo, hi, _, _ = a.batch_arrays(i)
        outs_a[i] = a.step(i, [a.src[lo:hi], a.dst[lo:hi], neg[lo - e0:hi - e0]])
    outs_b = torch.empty((n, 3, B, d), device="cuda")
    half = n // 2
    b.run(0, half, [b.src[e0:], b.dst[e0:], neg], out=outs_b[:half])
    lo_h = b.batch_lo[half]
    b.run(half, n - half, [b.src[lo_h:], b.dst[lo_h:], neg[lo_h - e0:]], out=outs_b[half:], check=True)
    assert torch.equal(outs_a, outs_b)
    assert torch.equal(a.cur, b.cur) and torch.equal(a.export_history(), b.export_history())
    assert (a.head, a.len, a.batch_idx) == (b.head, b.len, b.batch_idx)
    _lib.check(lib.lstep_step_profile(1), "profile on")
    try:
        ms = (ctypes.c_float * 6)()
        for i in range(n):
            lo, hi, _, _ = c.batch_arrays(i)
            o = c.step(i, [c.src[lo:hi], c.dst[lo:hi], neg[lo - e0:hi - e0]])
            _lib.check(lib.lstep_step_profile_read(ms), "profile read")
            assert all(0.0 < ms[k] < 5.0 for k in range(6)), list(ms)
            assert torch.equal(o, outs_a[i])
    finally:
        lib.lstep_step_profile(0)
    assert torch.equal(a.cur, c.cur) and torch.equal(a.export_history(), c.export_history())
    v = ctypes.c_int(-1)
    assert lib.lstep_get_option(b"pdl", ctypes.byref(v)) == 0 and v.value == 1
    assert lib.lstep_set_option(b"no_such_option", 1) != 0
    # switches that were removed must be rejected, not silently ignored
    for name in (b"cos_spread", b"gather_narrow", b"dft_early_trigger", b"host_memcpy", b"dft_ctas_per_sm", b"dft_generic",
                 b"mlp_ring", b"gather_fuse", b"mlp_pair", b"early_append", b"dft_prefetch", b"query_dedup"):
        assert lib.lstep_set_option(name, 1) != 0, name
        assert lib.lstep_get_option(name, ctypes.byref(v)) != 0, name


@pytest.mark.parametrize("tag", ["small", "full"])
def test_tensor_core_mlp_matches_simt_mlp_and_float64(torch_cuda, tag, parity_log):
    """The tcgen05 BF16x3 PE-MLP kernel (csrc/mlp_umma.cu; taken by launches of >= 1536 rows) against the fp32 SIMT cluster
    kernel and a float64 evaluation of the same function, through lstep_pe_mlp_apply with the kernel forced either way:
    row counts around the 64-row tile, one wave and several waves of tiles, with and without the self term's weights.
    Bar: both kernels within 4e-6 * max(|y|, rms) of float64 — the tensor-core path must be as accurate as the SIMT one."""
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import NeighborSampler, _lib
    lib = _lib.load()
    g = synth.make_graph("tiny_bip" if tag == "full" else "tiny", seed=0)
    F, d, t, T, K = dict(full=(172, 172, 100, 100, 20), small=(12, 12, 10, 8, 4))[tag]
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent")
    lstep = build_dropin(tag, g, s, F, d, t, T, K)[0].eval()
    V1 = 3000
    gen = torch.Generator(device="cuda").manual_seed(0)
    pe = torch.randn((V1, d), device="cuda", generator=gen) * 0.3
    worst = {"simt": 0.0, "umma": 0.0}
    try:
        for which, pre, selfn in (("nbr", "pe_neighbor_mlp", "self_update_neighbor_pe"), ("update", "pe_mlp", "self_update_pe")):
            p = {k: v.double() for k, v in lstep.state_dict().items() if not k.startswith("fft")}
            for n in (1, 63, 64, 65, 800, 9600, 20000):
                A = torch.randn((n, d + t), device="cuda", generator=gen) * 2.0
                ids = torch.randint(0, V1, (n,), device="cuda", generator=gen)
                a64, b64 = A.double(), pe[ids].double()
                h = torch.relu(a64 @ p[pre + "_1.weight"].T + p[pre + "_1.bias"])
                z = h @ p[pre + "_2.weight"].T + p[pre + "_2.bias"] + b64 @ p[selfn + ".weight"].T + p[selfn + ".bias"]
                want = b64 + torch.tanh(z)
                scale = torch.maximum(want.abs(), want.pow(2).mean().sqrt())
                for name, on in (("simt", 0), ("umma", 1)):
                    _lib.check(lib.lstep_set_option(b"mlp_umma", on), "opt")
                    _lib.check(lib.lstep_set_option(b"mlp_umma_min_rows", 0), "opt")
                    out = torch.full((n, d), float("nan"), device="cuda")
                    _lib.check(lib.lstep_pe_mlp_apply(_lib.ptr(A), _lib.ptr(pe), _lib.ptr(ids), n, lstep._mlp_ref(which), _lib.ptr(out), d, None,
                                                      _lib.stream_ptr()), "mlp")
                    e = float(((out.double() - want).abs() / scale).max())
                    worst[name] = max(worst[name], e)
                    assert e <= 4e-6, (tag, which, n, name, e)
    finally:
        lib.lstep_set_option(b"mlp_umma", 1)
        lib.lstep_set_option(b"mlp_umma_min_rows", 1536)
    parity_log[f"mlp_kernels/{tag}"] = worst


@pytest.mark.parametrize("zipf_s", [0.8, 1.2], ids=["zipf0.8", "hubs-zipf1.2"])
def test_stress_2000_steps_pdl_vs_plain_launches_bit_identical(torch_cuda, zipf_s):
    """VERDICT r1 #7: the step depends on work done BEFORE the dependency wait under programmatic dependent launch, on L2-coherent
    loads of predecessor data and on inter-CTA claims in the push kernel. 2000 consecutive steps at the Reddit shape
    (full graph, B = 200, T = 100) with the PDL chain and the same 2000 steps with plain stream launches (kernel
    boundaries between all kernels) must leave bit-identical tables, histories and outputs. zipf 1.2 (SURVEY §8(d)'s skew): a
    batch collapses onto ~160 nodes, so the push kernel's claims, its same-destination fixed-point reductions and the padding-row
    partial sums are contended several times harder than in the bench's stream."""
    torch = torch_cuda
    from lstep_b200 import NeighborSampler, PEStream, _lib
    import bench
    lib = _lib.load()
    g = synth.make_graph("reddit", seed=0, zipf_s=zipf_s)
    V1, B, K = g.num_nodes + 1, 200, 20
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V1)
    model = bench.make_params_model(g, s, torch.device("cuda"))
    gen = torch.Generator(device="cuda").manual_seed(5)
    hist = torch.randn((V1, 100, 172), device="cuda", generator=gen) * 0.1
    hist[0] = 0
    n_steps = 2000
    e0 = g.num_edges - n_steps * B
    neg = torch.from_numpy(np.random.default_rng(2).choice(np.unique(g.dst_node_ids), size=n_steps * B).astype(np.int64)).cuda()
    res = []
    try:
        for pdl in (1, 0):
            _lib.check(lib.lstep_set_option(b"pdl", pdl), "opt")
            st = PEStream(model, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, history=hist, start=e0)
            assert st.num_batches == n_steps and st.len == 100
            outs = torch.empty((n_steps // 10, 4, B, 172), device="cuda")
            for c in range(10):  # 10 native calls of 200 steps; the outputs of every 10th call's steps are kept
                b0 = c * (n_steps // 10)
                lo0 = st.batch_lo[b0]
                st.run(b0, n_steps // 10, [st.src[lo0:], st.dst[lo0:], st.src[lo0:], neg[lo0 - e0:]], out=outs)
            st.check_errors()
            res.append((st.cur.clone(), st.export_history(), outs.clone()))
            del st
    finally:
        lib.lstep_set_option(b"pdl", 1)
    for a, b in zip(res[0], res[1]):
        assert torch.equal(a, b)
    assert torch.isfinite(res[0][0]).all()


def test_identical_query_sets_computed_once_match_equal_copies(torch_cuda):
    """The eval loop passes the batch's sources twice (positive source, negative source under random negative sampling:
    evaluate_model_utils.py:51-52). The step recognises identical sets (same device pointer / same host array), computes
    them once and fans the rows out in the MLP epilogue: outputs, tables and histories must be bit-identical to the step
    given an equal copy of the set instead (a distinct pointer / array: computed separately), for the device-resident and the
    host-fed step, B = 200 (SIMT MLP) and B = 2000 (tcgen05 MLP)."""
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import NeighborSampler, PEStream
    for B in (200, 2000):
        g = synth.make_graph("reddit", seed=1, num_edges=40_000)
        V, d, T, K = g.num_nodes, 172, 100, 20
        s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V + 1)
        lstep = build_dropin("full", g, s, 172, d, 100, T, K)[0].eval()
        gen = torch.Generator(device="cuda").manual_seed(3)
        hist = torch.randn((V + 1, T, d), device="cuda", generator=gen) * 0.2
        e0 = g.num_edges - 4 * B
        neg_np = np.random.default_rng(0).integers(1, V + 1, g.num_edges - e0).astype(np.int64)
        neg = torch.from_numpy(neg_np).cuda()
        res = []
        for dedup in (1, 0):
            st = PEStream(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, history=hist, start=e0)
            outs = []
            for b in range(2):
                lo, hi, _, _ = st.batch_arrays(b)
                src_view = st.src[lo:hi]
                outs.append(st.step(b, [src_view, st.dst[lo:hi], src_view if dedup else src_view.clone(), neg[lo - e0:hi - e0]]).clone())
            for b in range(2, 4):  # host-fed: the same numpy array object twice
                lo, hi, _, _ = st.batch_arrays(b)
                src_np = g.src_node_ids[lo:hi]
                outs.append(torch.from_numpy(st.step_host(src_np, g.dst_node_ids[lo:hi], g.node_interact_times[lo:hi],
                                                          [src_np, g.dst_node_ids[lo:hi], src_np if dedup else src_np.copy(),
                                                           neg_np[lo - e0:hi - e0]])))
            st.check_errors()
            res.append((outs, st.cur.clone(), st.export_history()))
        for a, b_ in zip(res[0][0], res[1][0]):
            assert torch.equal(a, b_)
        assert torch.equal(res[0][0][0][0], res[0][0][0][2])  # the two source sets' outputs are the same rows
        assert torch.equal(res[0][1], res[1][1]) and torch.equal(res[0][2], res[1][2])


@pytest.mark.parametrize("B", [200, 2000])
def test_gather_pipe_and_query_dedup_variants_are_bit_identical(torch_cuda, B):
    """The variants of the step's fused gather must not change a bit of the outputs, tables and histories: gather_pipe — at
    B = 2000 (more query rows than the launch has CTAs) the CTAs walk several rows each with an extra warp looking one row ahead
    (nbr_aggregate_rows_piped) — on and off, each with the identical source query sets passed as one pointer (computed once)
    and as an equal copy (computed separately). Ragged last batch."""
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import NeighborSampler, PEStream, _lib
    lib = _lib.load()
    g = synth.make_graph("flights", seed=2, num_edges=60_000)
    V, d, T, K = g.num_nodes, 172, 100, 20
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V + 1)
    lstep = build_dropin("fullu", g, s, 172, d, 100, T, K)[0].eval()
    gen = torch.Generator(device="cuda").manual_seed(5)
    hist = torch.randn((V + 1, T, d), device="cuda", generator=gen) * 0.2
    e0 = g.num_edges - 3 * B - 11  # ragged last batch
    neg = torch.from_numpy(np.random.default_rng(1).integers(1, V + 1, g.num_edges - e0).astype(np.int64)).cuda()
    res = {}
    try:
        for dedup, pipe in ((1, 0), (1, 1), (0, 1), (0, 0)):
            _lib.check(lib.lstep_set_option(b"gather_pipe", pipe), "opt")
            st = PEStream(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, history=hist, start=e0)
            outs = []
            for b in range(st.num_batches):
                lo, hi, _, _ = st.batch_arrays(b)
                sv = st.src[lo:hi]
                outs.append(st.step(b, [sv, st.dst[lo:hi], sv if dedup else sv.clone(), neg[lo - e0:hi - e0]]).clone())
            st.check_errors()
            res[(dedup, pipe)] = (outs, st.cur.clone(), st.export_history())
    finally:
        lib.lstep_set_option(b"gather_pipe", 1)
    ref = res[(1, 0)]
    for key, got in res.items():
        for a, b_ in zip(ref[0], got[0]):
            assert torch.equal(a, b_), key
        assert torch.equal(ref[1], got[1]) and torch.equal(ref[2], got[2]), key


@pytest.mark.parametrize("world", [1, 3])
def test_replicated_table_sharded_changelog_matches_single_gpu_changelog(torch_cuda, world):
    """Same layout with the owners' history kept as a change log: every replica's table, each rank's share of the outputs and
    the owners' replayed history rows are BIT-identical to the single-GPU ChangeLogStream (same kernels, same inputs; the
    owner-local filter maps global ids to local rows)."""
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import ChangeLogStream, NeighborSampler, ReplicatedLocalGroup, ReplicatedTableRank
    g = synth.make_graph("tiny_bip", seed=4, num_nodes=300, num_edges=9000)
    V, d, K, B = g.num_nodes, 172, 20, 48
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V + 1)
    lstep = build_dropin("fullu", g, s, 172, d, 100, 100, K)[0].eval()
    init = torch.from_numpy(seeded_normal(17, (V + 1, d), 0.3)).cuda()
    init[0] = 0
    e0 = g.num_edges - 115 * B - 7
    st = ChangeLogStream(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, initial_pe=init.clone(), start=e0)
    ranks = [ReplicatedTableRank(lstep, r, world, g.src_node_ids, g.dst_node_ids, g.node_interact_times, V, B, K, init.clone(), start=e0, sampler=s,
                                 history="changelog") for r in range(world)]
    grp = ReplicatedLocalGroup(ranks)
    neg = torch.from_numpy(np.random.default_rng(3).integers(1, V + 1, g.num_edges - e0).astype(np.int64)).cuda()
    for b in range(st.num_batches):
        lo, hi, _, _ = st.batch_arrays(b)
        qs = [st.src[lo:hi], st.dst[lo:hi], st.src[lo:hi], neg[lo - e0:hi - e0].contiguous()]
        want = st.step(b, qs)
        got = torch.cat(grp.step(b, qs), dim=1)
        assert torch.equal(got, want), b
    for rk in ranks:
        assert torch.equal(rk.cur, st.cur), rk.rank
        rk.check_errors()
    h = st.export_history()
    for rk in ranks:
        assert torch.equal(rk.export_history_rows(), h[rk.rank::world]), rk.rank
    assert sum(rk.history_bytes() for rk in ranks) < 1.3 * st.history_bytes() + 4e6


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_replicated_table_sharded_history_is_bit_identical_to_single_gpu(torch_cuda, world):
    """The scale-out layout (history ring sharded by node id, table and CSR replicated, one all-gather of the filtered rows
    per step; l-step_b200/shard.py::ReplicatedTableRank) with all ranks emulated in one process: every replica's table,
    the owners' history rows and each rank's share of the a6 outputs must be BIT-identical to the single-GPU stream — the
    same kernels see the same inputs — through the masked (ring filling) and the steady regime."""
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import NeighborSampler, PEStream, ReplicatedLocalGroup, ReplicatedTableRank
    g = synth.make_graph("tiny_bip", seed=4, num_nodes=300, num_edges=9000)
    V, d, K, B = g.num_nodes, 172, 20, 48
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V + 1)
    model = build_dropin("full", g, s, 172, d, 100, 100, K)
    lstep = model[0].eval()
    init = torch.from_numpy(seeded_normal(17, (V + 1, d), 0.3)).cuda()
    init[0] = 0
    e0 = g.num_edges - 115 * B - 7  # 116 batches (ragged tail): the ring (T = 100) fills after 99 of them
    st = PEStream(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, initial_pe=init.clone(), start=e0)
    ranks = [ReplicatedTableRank(lstep, r, world, g.src_node_ids, g.dst_node_ids, g.node_interact_times, V, B, K, init.clone(), start=e0, sampler=s)
             for r in range(world)]
    grp = ReplicatedLocalGroup(ranks)
    assert ranks[0].num_batches == st.num_batches
    neg = torch.from_numpy(np.random.default_rng(3).integers(1, V + 1, g.num_edges - e0).astype(np.int64)).cuda()
    for b in range(st.num_batches):
        lo, hi, _, _ = st.batch_arrays(b)
        qs = [st.src[lo:hi], st.dst[lo:hi], st.src[lo:hi], neg[lo - e0:hi - e0].contiguous()]
        want = st.step(b, qs)
        outs = grp.step(b, qs)
        got = torch.cat(outs, dim=1)
        assert got.shape == want.shape and torch.equal(got, want), b
        if b % 20 == 0 or b == st.num_batches - 1:
            for rk in ranks:
                assert torch.equal(rk.cur, st.cur), (b, rk.rank)
    h = st.export_history()
    for rk in ranks:
        assert torch.equal(rk.export_history_rows(), h[rk.rank::world]), rk.rank
    s.check_errors()


@pytest.mark.parametrize("tag,Th0,bar", [("small", 1, 1e-5), ("fullu", 1, 1e-5), ("fullu", 100, 1e-5), ("full", 1, 3e-4)])
def test_changelog_history_matches_dense_ring(torch_cuda, tag, Th0, bar, parity_log):
    """ChangeLogStream (history = base rows + the rows every step changed; csrc/changelog.cu) against the dense-ring PEStream
    on the same stream: through the filling (masked) regime and the steady regime with retiring events, from an initial
    table (Th0 = 1) and from an imported dense history in which every row differs between snapshots (Th0 = T). The filter
    sums the same products in another grouping (span sums of G), so values agree to fp32 rounding, not bit for bit:
    two FREE-RUNNING recurrences are compared, so the bar is 1e-5 (every element of outputs, tables and replayed
    history) for the small model and the realistic weights, and 3e-4 for the stress weights (x2), where update_pe is
    ill-conditioned on row 0 / hub rows (profiles/r02_parity_errors.json: the fp32 reference itself is up to 4.7e-5
    from float64 after ONE step there) and any 1e-7 difference in the filter is amplified step after step."""
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import ChangeLogStream, NeighborSampler, PEStream
    z = np.load(golden_path(f"replay_{tag}.npz"))
    d, T, K, t_dim, F, B = (int(z[k]) for k in ("pe_dim", "T", "K", "time_dim", "feat_dim", "B"))
    V, E, e0 = int(z["V"]), int(z["E"]), int(z["e0"])
    g = synth.make_graph("tiny", seed=int(z["graph_seed"]), num_nodes=V, num_edges=E)
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V + 1)
    lstep = build_dropin(tag, g, s, F, d, t_dim, T, K)[0].eval()
    Th = min(Th0, T)
    hist0 = seeded_normal(int(z["hist0_seed"]), (V + 1, Th, d), 0.3)
    hist0[0] = 0
    mk = lambda cls, **kw: cls(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, history=torch.from_numpy(hist0).cuda(),
                               start=e0, **kw)
    a, b = mk(PEStream), mk(ChangeLogStream, event_capacity=V + 1)
    assert torch.equal(b.export_history(), a.export_history()) and torch.equal(a.cur, b.cur)
    neg = torch.from_numpy(z["neg_dst"].astype(np.int64)).cuda()
    n_steps = min(a.num_batches, T + 30)
    worst_out = worst_tab = 0.0
    for i in range(n_steps):
        lo, hi, _, _ = a.batch_arrays(i)
        qs = [a.src[lo:hi], a.dst[lo:hi], neg[i][:hi - lo].contiguous()]
        oa, ob = a.step(i, qs), b.step(i, qs)
        ok, w = pe_close(ob.cpu().numpy(), oa.cpu().numpy(), bar)
        worst_out = max(worst_out, w)
        assert ok, (i, "outputs", w)
        ok, w = pe_close(b.cur.cpu().numpy(), a.cur.cpu().numpy(), bar)
        worst_tab = max(worst_tab, w)
        assert ok, (i, "table", w)
        assert (a.head, a.len) == (b.head, b.len)
    b.check_errors()
    ha, hb = a.export_history(), b.export_history()
    assert ha.shape == hb.shape
    ok, w = pe_close(hb.cpu().numpy(), ha.cpu().numpy(), bar)
    assert ok, ("history", w)
    assert torch.equal(hb[:, -1, :], b.cur)
    parity_log[f"changelog/{tag}/Th0={Th0}"] = {"steps": n_steps, "worst_output": worst_out, "worst_table": worst_tab, "history": w,
                                               "log_bytes": b.history_bytes(), "dense_bytes": int(a.ring.numel() * 4)}
    # capacity overflow is reported, not silently dropped
    c = mk(ChangeLogStream, event_capacity=8) if Th0 == 1 else None
    if c is not None:
        lo, hi, _, _ = c.batch_arrays(0)
        c.step(0, [c.src[lo:hi]])
        with pytest.raises(Exception):
            c.check_errors()
