"""Phase B of update_pe adds its contributions in 32.32 fixed point with 64-bit integer atomics (push kernel, the pull
form's lists of more than 4 slots). The sums are exact only while every column sum fits in int64, so the kernels raise
LSTEP_FLAG_FIXED_POINT_RANGE (FloatingPointError at check_errors) for a contribution that is non-finite or at least
fixed_point_bound(n_ids, K) = 2^31 / (n_ids*K + 1) in magnitude (csrc/common.cuh).

Every case runs through both phase-B forms and both phase-B MLP kernels against the oracle (fp32 = the reference's
own error, float64 = the exact value) and must do exactly what the bound predicts, worked out on the host from the
oracle's phase-A rows and lookup before the kernel runs:
  (a) no flag, and the table within the parity bar (non-finite positions equal to the reference's), or
  (b) the flag.
The push form flags when any batch row's phase-A value fails |x| < bound; the pull form when such a row reaches a
destination with more than 4 slots (shorter lists and the padding row are fp32 sums there, as in the reference)."""
import numpy as np
import pytest

from common import check_updated_table, seeded_normal
from lstep_b200 import synth
from oracle import lstep_oracle as orc

pytestmark = pytest.mark.gpu

HUB_LEN = 4  # kHubLen in csrc/update.cu: longer lists are summed in fixed point by the pull form
COMBOS = [(push, umma) for push in (1, 0) for umma in (0, 1)]  # (phaseb_push, tcgen05 MLP for every launch)


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    from lstep_b200 import _lib
    assert _lib.load().lstep_device_ok() == 1, "not a compute-capability 10.x device"
    return torch


# ------------------------------------------------------------------------------------------------ inputs
def _graph(n_b, K, hubs=(4, 5, 40), deg=(1, 30), short="some", pool=400, ties=False, seed=0):
    """Deterministic batch of n_b batch nodes 1..n_b (ring edges v -> v % n_b + 1, all at the batch time, so no batch edge
    is sampled). Batch node v's history is a list of neighbours among `pool` filler nodes, deg[0]..deg[1] long, and hub
    j (node n_b + 1 + j) is the MOST RECENT neighbour of exactly hubs[j] batch nodes, so it receives exactly hubs[j]
    slots. short: "some" keeps the drawn lengths (row 0 is reached by every node with fewer than K entries), "one" gives
    every node but node 1 at least K entries, "all" gives every node fewer than K. ties: history times repeat."""
    rng = np.random.default_rng(seed)
    H0, F0 = n_b + 1, n_b + 1 + len(hubs)
    lo, hi = deg
    if short == "one":
        lo, hi = K + 1, max(hi, K + 1)
    elif short == "all":  # (hubs append up to len(hubs) more)
        lo, hi = 0, max(0, K - 1 - len(hubs))
    lists = [list(F0 + rng.integers(0, pool, int(rng.integers(lo, hi + 1)))) for _ in range(n_b)]
    if short == "one":
        lists[0] = lists[0][:max(0, K - 2)]
    for j, c in enumerate(hubs):
        for v in rng.choice(n_b, c, replace=False):
            lists[v].append(H0 + j)
    src, dst, t = [], [], []
    for p in range(max(len(x) for x in lists) if lists else 0):
        for v in range(n_b):
            if p < len(lists[v]):
                src.append(v + 1)
                dst.append(lists[v][p])
                t.append(float(p if ties else len(t)) + 1.0)
    tb = float(max(t, default=0.0) + 1.0)
    bsrc = np.arange(1, n_b + 1, dtype=np.int64)
    bdst = bsrc % n_b + 1
    src = np.concatenate([np.asarray(src, np.int64), bsrc])
    dst = np.concatenate([np.asarray(dst, np.int64), bdst])
    tt = np.concatenate([np.asarray(t, np.float64), np.full(n_b, tb)])
    return dict(src=src, dst=dst, t=tt, V1=F0 + pool, lo=len(src) - n_b)


def _synth(gname, n_edges, B):
    g = synth.make_graph(gname, seed=0, num_edges=n_edges)
    return dict(src=g.src_node_ids, dst=g.dst_node_ids, t=g.node_interact_times, V1=g.num_nodes + 1, lo=g.num_edges - B)


class _Case:
    """A model (oracle parameters of shape d, t), the sampler over the graph, and the batch [lo, end)."""

    def __init__(self, torch, gr, d, t, K, seed=0):
        from lstep_b200 import LSTEP, NeighborSampler
        self.torch, self.K, self.d, self.V1 = torch, K, d, gr["V1"]
        self.s = NeighborSampler.from_edges(gr["src"], gr["dst"], np.arange(1, len(gr["src"]) + 1), gr["t"], "recent",
                                            num_rows=self.V1)
        self.p = orc.init_params(pe_dim=d, time_dim=t, T=8, seed=seed)
        m = LSTEP(np.zeros((self.V1, 4), np.float32), np.zeros((len(gr["src"]) + 1, 4), np.float32), self.s, self.s, pe_dim=d,
                  num_neighbors=K, time_feat_dim=t, num_fft_batches=8, device="cuda")
        sd = {k: torch.from_numpy(v) for k, v in self.p.items() if not k.startswith("fft")}
        missing = set(sd) - set(m.state_dict())
        assert not missing, missing
        m.load_state_dict(sd, strict=False)
        self.m = m.cuda().eval()
        self.adj = orc.build_adjacency_fast(gr["src"], gr["dst"], np.arange(1, len(gr["src"]) + 1), gr["t"], num_rows=self.V1)
        lo = gr["lo"]
        self.src, self.dst, self.tt = gr["src"][lo:], gr["dst"][lo:], gr["t"][lo:]
        self.ids = synth.unique_batch_nodes(self.src, self.dst)
        self.tc = float(self.tt.max())
        self.nbr = orc.sample_recent(self.adj, self.ids, self.tt, K)[0]

    def expect(self, pe0):
        """The outcomes the bound allows for the push form and for the pull form ({True}, {False}, or both when a phase-A
        value lies within rounding of the bound: the kernel's and the oracle's phase A round differently near a saturated
        tanh), the max column sum of |contribution| over the destinations, and the slot count of every node — from the
        oracle's phase-A rows and lookup."""
        from lstep_b200 import _lib
        with np.errstate(invalid="ignore", over="ignore"):  # (non-finite inputs)
            pa = orc.update_pe_phase_a(self.p, pe0.copy(), self.ids, self.src, self.dst, self.tt, self.tc)
        x = pa[self.ids].astype(np.float64)
        x[self.ids == 0] = 0.0
        bound = _lib.fixed_point_bound(len(self.ids), self.K)
        margin = 4.0 + 1e-5 * bound
        with np.errstate(invalid="ignore"):
            surely_bad = ~(np.abs(x) < bound + margin).all(axis=1)  # (NaN compares false: a NaN row is bad)
            maybe_bad = ~(np.abs(x) < bound - margin).all(axis=1)
        cnt = np.bincount(self.nbr[self.nbr > 0].reshape(-1), minlength=self.V1)
        reaches_long = np.array([(cnt[r[r > 0]] > HUB_LEN).any() for r in self.nbr])
        allowed = lambda rows: {bool((surely_bad & rows).any()), bool((maybe_bad & rows).any())}
        # Σ|contribution| per destination column (row 0 takes z_i copies of row i)
        dest = np.where(self.nbr > 0, self.nbr, 0)
        colsum = np.zeros((self.V1, x.shape[1]))
        np.add.at(colsum, dest.reshape(-1), np.repeat(np.abs(np.nan_to_num(x, nan=np.inf)), self.K, axis=0))
        return allowed(np.ones(len(x), bool)), allowed(reaches_long), float(colsum.max()), cnt

    def run(self, pe0, push, umma):
        """The drop-in update_pe on a copy of pe0 with the phase-B form and MLP kernel forced; (table, flag raised)."""
        torch = self.torch
        from lstep_b200 import _lib
        lib = _lib.load()
        _lib.check(lib.lstep_set_option(b"phaseb_push", push), "opt")
        _lib.check(lib.lstep_set_option(b"mlp_umma", umma), "opt")
        _lib.check(lib.lstep_set_option(b"mlp_umma_min_rows", 0 if umma else 1536), "opt")
        self.s.check_errors()
        pe = torch.from_numpy(pe0).cuda()
        self.m.update_pe(pe, self.ids, np.arange(len(self.src)), self.src, self.dst, self.tt, self.tc, num_neighbors=self.K)
        try:
            self.s.check_errors()
            flagged = False
        except FloatingPointError:
            flagged = True
        return pe.cpu().numpy(), flagged

    def check(self, pe0, what, log=None):
        """Every form x MLP kernel on pe0: exactly (a) or (b) as predicted. Returns the predicted push-form flag."""
        from lstep_b200 import _lib
        flag_push, flag_pull, colmax, _ = self.expect(pe0)
        bound = _lib.fixed_point_bound(len(self.ids), self.K)
        if True not in flag_push:  # the bound's promise, on these data: every column sum fits the 32.32 format
            assert colmax < 2.0 ** 31, (what, colmax, bound)
        with np.errstate(invalid="ignore", over="ignore"), orc.high_precision():
            truth = orc.update_pe(self.p, self.adj, pe0.astype(np.float64), self.ids, self.src, self.dst, self.tt, self.tc, self.K)
        with np.errstate(invalid="ignore", over="ignore"):
            want = orc.update_pe(self.p, self.adj, pe0.copy(), self.ids, self.src, self.dst, self.tt, self.tc, self.K)
        lib = _lib.load()
        try:
            for push, umma in COMBOS:
                got, flagged = self.run(pe0, push, umma)
                expect = flag_push if push else flag_pull
                tag = f"{what}/push{push}/umma{umma}"
                assert flagged in expect, (tag, "range flag", flagged, "allowed", expect, "bound", bound)
                if flagged:
                    continue
                fin = np.isfinite(want)
                assert np.array_equal(np.isfinite(got), fin), (tag, "non-finite positions", np.argwhere(np.isfinite(got) != fin)[:8])
                assert np.array_equal(got[~fin], want[~fin], equal_nan=True), (tag, "non-finite values")
                z = lambda a: np.where(fin, a, 0)
                check_updated_table(z(got), z(want), tag, z(truth), log=log)
        finally:
            lib.lstep_set_option(b"phaseb_push", 1)
            lib.lstep_set_option(b"mlp_umma", 1)
            lib.lstep_set_option(b"mlp_umma_min_rows", 1536)
        return True in flag_push


def _table(V1, d, S, same_sign, seed):
    a = seeded_normal(seed, (V1, d), 1.0).astype(np.float64)
    if same_sign:
        a = np.abs(a)
    a = (a * S).astype(np.float32)
    a[0] = 0
    return a


# ------------------------------------------------------------------------------------------------ magnitudes
MAGS = [2.0 ** e for e in range(-20, 25, 4)]


@pytest.mark.parametrize("same_sign", [False, True], ids=["signed", "same-sign"])
def test_magnitude_sweep_is_exact_or_flagged(torch_cuda, same_sign, parity_log):
    """S·N(0,1) and S·|N(0,1)| tables, S = 2^-20 .. 2^24, on a batch with hubs of 4, 5 and 40 slots and padded slots:
    within the bound the kernel is within the parity bar (small S: the 2^-32 quantum is no worse than the fp32 reference's
    own error), at or beyond it the flag is raised — never a silent mismatch. Both outcomes must occur in the sweep."""
    c = _Case(torch_cuda, _graph(200, 20, seed=1), 172, 100, 20)
    seen = set()
    for i, S in enumerate(MAGS):
        seen.add(c.check(_table(c.V1, 172, S, same_sign, 100 + i), f"fx/sweep/{'abs' if same_sign else 'sgn'}/S{S:g}", parity_log))
    assert seen == {False, True}, seen


@pytest.mark.parametrize("gname,n_edges,B", [("reddit", 100_000, 200), ("flights", 300_000, 2000)])
def test_dataset_shaped_batches_are_exact_or_flagged(torch_cuda, gname, n_edges, B, parity_log):
    """The same rule on the last batch of a Reddit-shaped (B = 200) and a Flights-shaped (B = 2000, ties) synth stream."""
    c = _Case(torch_cuda, _synth(gname, n_edges, B), 172, 100, 20)
    flags = [c.check(_table(c.V1, 172, S, ss, 7), f"fx/{gname}/S{S:g}/{ss}", parity_log)
             for S, ss in ((2.0 ** -20, False), (1.0, False), (2.0 ** 10, True), (2.0 ** 24, False))]
    assert flags == [False, False, False, True], flags


# ------------------------------------------------------------------------------------------------ non-finite values
@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf], ids=["nan", "+inf", "-inf"])
def test_non_finite_values(torch_cuda, bad, parity_log):
    """A non-finite value in a batch node's row is flagged (the node reaches the 40-slot hub, so both forms add it in fixed
    point); in a row that is only a phase-B destination (node_pe2) it is not a contribution: no flag, and the output's
    non-finite positions are the reference's."""
    c = _Case(torch_cuda, _graph(120, 20, seed=2), 172, 100, 20)
    hub = 120 + 1 + 2
    v = int(next(i for i, r in zip(c.ids, c.nbr) if (r == hub).any()))
    pe0 = _table(c.V1, 172, 0.3, False, 3)
    pe0[v, 17] = bad
    assert c.expect(pe0)[:2] == ({True}, {True})
    c.check(pe0, f"fx/nonfinite/batch/{bad}", parity_log)
    pe0 = _table(c.V1, 172, 0.3, False, 3)
    pe0[hub, 5] = bad
    pe0[hub + 1 + 7, 9] = bad  # a filler destination
    assert c.expect(pe0)[:2] == ({False}, {False})
    c.check(pe0, f"fx/nonfinite/dest/{bad}", parity_log)


# ------------------------------------------------------------------------------------------------ shapes
SHAPES = ([dict(n_b=n, K=20, d=172, t=100) for n in (1184, 1185, 2368, 2369)]  # push split 4 / 2 / 1 CTAs per node
          + [dict(n_b=200, K=K, d=172, t=100) for K in (1, 3, 5, 33, 64)]  # uneven slot split; K > 32: two claim passes
          + [dict(n_b=200, K=20, d=12, t=10), dict(n_b=200, K=20, d=256, t=128)]  # <6,4> and <8,8> push templates
          + [dict(n_b=200, K=20, d=172, t=100, short="one"), dict(n_b=200, K=20, d=172, t=100, short="all"),
             dict(n_b=64, K=20, d=172, t=100, ties=True)])


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "-".join(f"{k}{v}" for k, v in s.items()))
def test_shapes_in_and_out_of_range(torch_cuda, shape, parity_log):
    """Every launch shape the phase-B kernels switch on, with destinations of exactly 4 and 5 slots (the pull form's
    fp32 / fixed-point switch) and row 0 reached by one batch node or by all: S = 1 is within the parity bar without a
    flag, S = 2^24 raises the flag."""
    sh = dict(shape)
    n_b, K, d, t = sh.pop("n_b"), sh.pop("K"), sh.pop("d"), sh.pop("t")
    hubs = (4, 5, 40) if K > 1 else (4, 5)
    c = _Case(torch_cuda, _graph(n_b, K, hubs=hubs, seed=n_b + K + d, **sh), d, t, K)
    cnt = c.expect(_table(c.V1, d, 1.0, False, 0))[3]
    assert (cnt == 4).any() and (cnt == 5).any()
    z = (c.nbr == 0).sum(axis=1)
    if sh.get("short") == "one":
        assert (z > 0).sum() == 1
    if sh.get("short") == "all":
        assert (z > 0).all()
    assert c.check(_table(c.V1, d, 1.0, False, 1), f"fx/shape/{shape}/S1", parity_log) is False
    assert c.check(_table(c.V1, d, 2.0 ** 24, True, 2), f"fx/shape/{shape}/S2^24", parity_log) is True


# ------------------------------------------------------------------------------------------------ entry points
def test_every_entry_point_raises_the_flag(torch_cuda):
    """PEStream.step, a ChangeLogStream step and the emulated peer group at world 3 from a full history (no DFT mask):
    at S = 1 no flag and the group's outputs equal the change-log stream's bits; at S = 2^30 every one raises the flag.
    (The drop-in update_pe is covered by the tests above.)"""
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import ChangeLogStream, NeighborSampler, PEStream, PeerLocalGroup, PeerRank
    g = synth.make_graph("tiny_bip", seed=4, num_nodes=300, num_edges=9000)
    V, d, K, B, T = g.num_nodes, 172, 20, 48, 100
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V + 1)
    lstep = build_dropin("fullu", g, s, 172, d, 100, T, K)[0].eval()
    e0 = g.num_edges - 3 * B
    neg = torch.from_numpy(np.random.default_rng(3).integers(1, V + 1, g.num_edges - e0).astype(np.int64)).cuda()
    for S, flagged in ((1.0, False), (2.0 ** 30, True)):
        hist = torch.from_numpy(seeded_normal(23, (V + 1, T, d), 1.0)).cuda() * S
        hist[0] = 0
        args = (g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K)
        pes = PEStream(lstep, *args, history=hist.clone(), start=e0)
        cls = ChangeLogStream(lstep, *args, history=hist.clone(), start=e0, event_capacity=V + 1)
        ranks = [PeerRank(lstep, r, 3, g.src_node_ids, g.dst_node_ids, g.node_interact_times, V, B, K, history=hist.clone(), start=e0,
                          sampler=s, event_capacity=V + 1) for r in range(3)]
        grp = PeerLocalGroup(ranks)
        lo, hi, _, _ = pes.batch_arrays(0)
        qs = [pes.src[lo:hi], pes.dst[lo:hi], neg[lo - e0:hi - e0].contiguous()]
        for name, stepper, check in (("PEStream", lambda: pes.step(0, qs), pes.check_errors),
                                     ("ChangeLogStream", lambda: cls.step(0, qs), cls.check_errors),
                                     ("peer group", lambda: (grp.step(0, qs), grp.barrier()), ranks[0].check_errors)):
            s.check_errors()
            out = stepper()
            torch.cuda.synchronize()
            if flagged:
                with pytest.raises(FloatingPointError, match="2\\^31"):
                    check()
            else:
                check()
            if name == "ChangeLogStream":
                want = out.clone()
            if name == "peer group" and not flagged:
                assert torch.equal(torch.cat(out[0], dim=1), want)
                for rk in ranks:
                    assert torch.equal(rk.cur, cls.cur), rk.rank
        del pes, cls, ranks, grp, hist
        torch.cuda.empty_cache()
