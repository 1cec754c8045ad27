"""CPU oracle for the L-STEP positional-encoding hot path — TEST INFRASTRUCTURE ONLY.

This is a numpy restatement of the reference's algorithm for the path SURVEY.md §8 scopes
(temporal neighbour lookup, DFT filter over the PE history, neighbourhood PE aggregate, PE
update). It is a checker: only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
`--impl reference` legs may import it. The product (lstep_b200) never does and has no CPU path.

Parity pin: the reference ships no tests or golden vectors (SURVEY §4), so this oracle is pinned
against outputs of the *unmodified* reference run in the build container through import shims
(tests/golden/make_golden.py writes tests/golden/*.npz; tests/test_oracle_vs_golden.py checks
every function below against them). Integer outputs must be bit-identical; fp32 outputs agree
with the reference's torch CPU kernels to a few ulp (BLAS summation order and the cos / tanh
implementations differ between numpy and torch), which the tests state as tolerances.

Every function follows the reference literally — FFT / mask / filter / iFFT, V1-sized scatter
buffers, python row loops — rather than the restructured form the CUDA kernels use, so that the
restructuring itself is what the parity tests check. Citations are relative to /root/reference.
"""
from __future__ import annotations

import contextlib

import numpy as np
import scipy.fft as _sfft

F32 = np.float32   # fixed-precision casts that are part of the reference's contract (fp32 time deltas, fp32 tables)
ACC = np.float32   # arithmetic precision of sums / matmuls / cos / tanh; float64 under `high_precision()`


@contextlib.contextmanager
def high_precision():
    """Evaluate the same functions with float64 arithmetic (inputs still quantised exactly as the
    reference quantises them). Used by tests as the 'exact' answer against which the fp32 error of the
    reference-style evaluation and of the CUDA kernels are both measured."""
    global ACC
    old, ACC = ACC, np.float64
    try:
        yield
    finally:
        ACC = old


# --------------------------------------------------------------------------------------------
# a1 — temporal adjacency (utils/utils.py:282-301 builds adj lists, :95-102 sorts them)
# --------------------------------------------------------------------------------------------
class Adjacency:
    """Per-node neighbour / edge-id / time arrays, each sorted by time with a stable sort."""

    def __init__(self, nbr, eid, t):
        self.nbr, self.eid, self.t = nbr, eid, t  # lists of np arrays, index = node id

    @property
    def num_rows(self):
        return len(self.nbr)

    def to_csr(self):
        deg = np.array([len(x) for x in self.nbr], dtype=np.int64)
        indptr = np.zeros(len(deg) + 1, dtype=np.int64)
        np.cumsum(deg, out=indptr[1:])
        cat = lambda xs, dt: (np.concatenate(xs).astype(dt) if indptr[-1] else np.zeros(0, dt))
        return indptr, cat(self.nbr, np.int64), cat(self.eid, np.int64), cat(self.t, np.float64)


def build_adjacency(src, dst, eid, t) -> Adjacency:
    """get_neighbor_sampler (utils/utils.py:292-299): for every edge, in data order, append
    (dst,eid,t) to adj[src] then (src,eid,t) to adj[dst]; NeighborSampler.__init__ (:95-102)
    sorts each list by time with python's stable `sorted`."""
    max_id = int(max(src.max(), dst.max()))
    adj = [[] for _ in range(max_id + 1)]
    for s, d, e, tt in zip(src.tolist(), dst.tolist(), eid.tolist(), t.tolist()):
        adj[s].append((d, e, tt))
        adj[d].append((s, e, tt))
    nbr, eids, times = [], [], []
    for lst in adj:
        lst = sorted(lst, key=lambda x: x[2])
        nbr.append(np.array([x[0] for x in lst]))
        eids.append(np.array([x[1] for x in lst]))
        times.append(np.array([x[2] for x in lst]))
    return Adjacency(nbr, eids, times)


def build_adjacency_fast(src, dst, eid, t, num_rows=None) -> Adjacency:
    """Same result as build_adjacency for graphs too large for python lists (full-size dataset shapes): the 2E
    entries in insertion order (edge i: entry 2i under src, entry 2i+1 under dst) sorted by (node, time) with a stable
    sort == per-node stable `sorted` by time. tests/test_oracle_vs_golden.py checks it against build_adjacency."""
    E = len(src)
    owner = np.empty(2 * E, np.int64)
    owner[0::2], owner[1::2] = src, dst
    other = np.empty(2 * E, np.int64)
    other[0::2], other[1::2] = dst, src
    ee = np.repeat(np.asarray(eid, np.int64), 2)
    tt = np.repeat(np.asarray(t, np.float64), 2)
    order = np.lexsort((tt, owner))  # stable: ties keep insertion order
    n = int(owner.max()) + 1 if num_rows is None else int(num_rows)
    cuts = np.cumsum(np.bincount(owner, minlength=n))[:-1]
    return Adjacency(np.split(other[order], cuts), np.split(ee[order], cuts), np.split(tt[order], cuts))


# --------------------------------------------------------------------------------------------
# a2 — most-recent-K lookup (utils/utils.py:129-146, 148-213, 'recent' branch :199-208)
# --------------------------------------------------------------------------------------------
def sample_recent(adj: Adjacency, node_ids, node_interact_times, num_neighbors: int = 20):
    assert num_neighbors > 0, 'Number of sampled neighbors for each node should be greater than 0!'  # :156
    n = len(node_ids)
    out_n = np.zeros((n, num_neighbors)).astype(np.longlong)  # :160
    out_e = np.zeros((n, num_neighbors)).astype(np.longlong)  # :163
    out_t = np.zeros((n, num_neighbors)).astype(np.float32)  # :166
    # `zip` stops at the shorter input (:169) — rows beyond len(times) stay zero (SURVEY Q1)
    for idx, (node, tq) in enumerate(zip(node_ids, node_interact_times)):
        i = np.searchsorted(adj.t[node], tq)  # side='left' -> strictly earlier (:140); IndexError if node too large (Q8)
        nn, ee, tt = adj.nbr[node][:i], adj.eid[node][:i], adj.t[node][:i]
        if len(nn) > 0:
            nn, ee, tt = nn[-num_neighbors:], ee[-num_neighbors:], tt[-num_neighbors:]  # :201-203
            out_n[idx, num_neighbors - len(nn):] = nn  # right aligned (:206-208)
            out_e[idx, num_neighbors - len(ee):] = ee
            out_t[idx, num_neighbors - len(tt):] = tt  # f64 -> f32 RN on store
    return out_n, out_e, out_t


# --------------------------------------------------------------------------------------------
# a5 — TimeEncoder (models/modules.py:20,27-39): cos(fp32(dt) * w_j + 0)
# --------------------------------------------------------------------------------------------
def time_encoder_weights(time_dim: int) -> np.ndarray:
    return (1 / 10 ** np.linspace(0, 9, time_dim, dtype=np.float32)).astype(F32)  # modules.py:20


def time_encode(dt_f32: np.ndarray, w: np.ndarray) -> np.ndarray:
    dt_f32 = np.asarray(dt_f32, dtype=F32)
    arg = dt_f32[..., None] * w.astype(F32)  # fp32 product, as Linear(1->t) with zero bias computes it
    # cos evaluated in float64 and rounded: the correctly rounded value every fp32 cosf approximates to <= 1 ulp
    # (numpy's own float32 cos drops to scalar libm for |x| > 7e4, 25x slower on these arguments)
    return np.cos(arg.astype(np.float64)).astype(ACC)


# --------------------------------------------------------------------------------------------
# parameters — names are the reference's state_dict keys (SURVEY §8(b))
# --------------------------------------------------------------------------------------------
def _linear(x, p, name):
    return x.astype(ACC) @ p[name + ".weight"].T.astype(ACC) + p[name + ".bias"].astype(ACC)


def init_params(pe_dim=172, time_dim=100, T=100, seed=0) -> dict:
    """Random parameters with the reference's shapes (models/LSTEP.py:50-70) — used where a
    test does not take them from a golden file. Not the torch initialiser; any values do."""
    rng = np.random.default_rng(seed)
    u = lambda *s, k=1.0: ((rng.random(s) * 2 - 1) * k).astype(F32)
    d, t = pe_dim, time_dim
    p = {"time_encoder.w.weight": time_encoder_weights(t).reshape(t, 1),
         "time_encoder.w.bias": np.zeros(t, F32),
         "fft_filter.weight": (u(T, d, k=d ** -0.5) + 1j * u(T, d, k=d ** -0.5)).astype(np.complex64),
         "fft_agg.weight": u(1, T, k=T ** -0.5)}
    for name, (o, i) in {"self_update_pe": (d, d), "pe_mlp_1": (d, d + t), "pe_mlp_2": (d, d),
                         "self_update_neighbor_pe": (d, d), "pe_neighbor_mlp_1": (d, d + t),
                         "pe_neighbor_mlp_2": (d, d)}.items():
        p[name + ".weight"] = u(o, i, k=i ** -0.5)
        p[name + ".bias"] = u(o, k=i ** -0.5)
    return p


# --------------------------------------------------------------------------------------------
# a3 — LSTEP.fourier_transform_pe (models/LSTEP.py:104-137)
# --------------------------------------------------------------------------------------------
def fourier_transform_pe(p: dict, node_ids, pe_hist: np.ndarray, batch_idx: int, num_fft_batches: int):
    x = pe_hist[node_ids].astype(F32)  # [N, Th, d]  (:105)
    cdt = np.complex64 if ACC is np.float32 else np.complex128
    mask = None
    T = num_fft_batches
    if x.shape[1] < T:  # :108-113 — zero-pad to T; mask is keyed on batch_idx (Q5)
        x = np.concatenate([x, np.zeros((x.shape[0], T - x.shape[1], x.shape[2]), F32)], axis=1)
        mask = np.zeros(x.shape, F32)
        mask[:, :batch_idx, :] += 1
    X = _sfft.fft(x.astype(cdt), axis=1, workers=-1).astype(cdt)  # :116-117
    if mask is not None:
        X = X * mask
    X = p["fft_filter.weight"][None].astype(cdt) * X  # [T,d] table, elementwise (:121)
    if mask is not None:
        X = X * mask
    y = _sfft.ifft(X, axis=1, workers=-1).astype(cdt)  # :125
    if mask is not None:
        y = y * mask
    y = y.real.astype(ACC)  # complex -> float32 keeps the real part (:129)
    out = y.transpose(0, 2, 1) @ p["fft_agg.weight"].astype(ACC).T  # Linear(T->1), no bias (:135)
    return np.squeeze(out[..., 0]) if out.shape[0] == 1 else out[..., 0]  # .squeeze()


# --------------------------------------------------------------------------------------------
# a6 — LSTEP.compute_neighborhood_pe (models/LSTEP.py:222-249)
# --------------------------------------------------------------------------------------------
def compute_neighborhood_pe(p: dict, adj: Adjacency, pe: np.ndarray, node_ids, node_interact_times,
                            num_neighbors: int = 30):
    nbr, _, nt = sample_recent(adj, node_ids, node_interact_times, num_neighbors)  # :223
    w = p["time_encoder.w.weight"].reshape(-1)
    dt = (np.asarray(node_interact_times)[:, None] - nt).astype(F32)  # f64 - f32 -> f64 -> .float() (:228-230)
    tf = time_encode(dt, w)  # [B,K,t]
    tf[nbr == 0] = 0.0  # :231
    nbr_pe = pe[nbr]  # [B,K,d]; padded slots read pe[0] (nonzero after an update — Q2) (:233)
    node_pe = pe[node_ids]  # :235
    s = np.concatenate([nbr_pe.astype(ACC), tf], axis=-1).sum(axis=1, dtype=ACC)  # :238
    h = _linear(s, p, "pe_neighbor_mlp_1")
    h = np.maximum(h, 0)
    h = _linear(h, p, "pe_neighbor_mlp_2")
    h = _linear(node_pe, p, "self_update_neighbor_pe") + h  # :244
    return (node_pe + np.tanh(h, dtype=ACC)).astype(ACC)  # :245-247


# --------------------------------------------------------------------------------------------
# a9 — torch_scatter.scatter(src, index, dim=0, out=out, reduce='sum') == out.scatter_add_
# (third-party, un-vendored and unpinned in the reference; call sites models/LSTEP.py:283-290,
#  320-322). CPU semantics: serial adds in index order.
# --------------------------------------------------------------------------------------------
def scatter_sum_rows(src: np.ndarray, index: np.ndarray, out: np.ndarray):
    np.add.at(out, index, src)  # unbuffered, in order of `index`
    return out


# --------------------------------------------------------------------------------------------
# a7 + a8 — LSTEP.update_pe (models/LSTEP.py:268-341); mutates and returns `pe`
# --------------------------------------------------------------------------------------------
def update_pe_phase_a(p: dict, pe: np.ndarray, node_ids, batch_src_node_ids, batch_dst_node_ids, node_interact_times,
                      current_time):
    """Phase A of update_pe (models/LSTEP.py:273-303) on its own; mutates and returns `pe`. Phase B adds these rows."""
    w = p["time_encoder.w.weight"].reshape(-1)
    d = pe.shape[1]
    tc = np.float32(current_time)  # torch.Tensor([current_time]) is fp32 (Q4)
    node_pe = pe[node_ids].copy()  # :273
    dt = (np.float64(tc) - np.asarray(node_interact_times, dtype=np.float64)).astype(F32)  # f32 - f64 -> f64 -> float
    tf = time_encode(dt, w)  # [E,t]
    agg = np.zeros((pe.shape[0], d + tf.shape[1]), ACC)  # :282
    scatter_sum_rows(np.concatenate([pe[batch_dst_node_ids].astype(ACC), tf], axis=-1), batch_src_node_ids, agg)  # :283-286
    scatter_sum_rows(np.concatenate([pe[batch_src_node_ids].astype(ACC), tf], axis=-1), batch_dst_node_ids, agg)  # :287-290
    a = agg[node_ids]  # :292
    h = _linear(np.maximum(_linear(a, p, "pe_mlp_1"), 0), p, "pe_mlp_2")  # :294-297
    upd = node_pe + np.tanh(_linear(node_pe, p, "self_update_pe") + h, dtype=ACC)  # :299-301
    pe[node_ids] = upd  # :303
    return pe


def update_pe(p: dict, adj: Adjacency, pe: np.ndarray, node_ids, batch_src_node_ids, batch_dst_node_ids,
              node_interact_times, current_time, num_neighbors: int = 30):
    w = p["time_encoder.w.weight"].reshape(-1)
    d = pe.shape[1]
    tc = np.float32(current_time)  # torch.Tensor([current_time]) is fp32 (Q4)
    # ---- phase A (:277-303)
    update_pe_phase_a(p, pe, node_ids, batch_src_node_ids, batch_dst_node_ids, node_interact_times, current_time)
    # ---- phase B (:306-339)
    nbr, _, nt = sample_recent(adj, node_ids, node_interact_times, num_neighbors)  # N ids zipped with B times (Q1/Q1b)
    src_flat = np.broadcast_to(np.asarray(node_ids)[:, None], nbr.shape).reshape(-1)  # :310
    nbr_flat = nbr.reshape(-1)
    nt_flat = nt.reshape(-1)
    dt2 = (tc - nt_flat).astype(F32)  # f32 - f32 (:314)
    tf2 = time_encode(dt2, w)
    tf2[nbr_flat == 0] = 0.0  # :316
    pe[0] = 0.0  # :317
    agg2 = np.zeros((pe.shape[0], d + tf2.shape[1]), ACC)  # :319
    scatter_sum_rows(np.concatenate([pe[src_flat].astype(ACC), tf2], axis=-1), nbr_flat, agg2)  # :320-322, phase-A-updated pe
    uniq = np.unique(nbr_flat)  # sorted; contains 0 when any slot is padding (:324)
    a2 = agg2[uniq]
    node_pe2 = pe[uniq]  # :325
    h2 = _linear(np.maximum(_linear(a2, p, "pe_mlp_1"), 0), p, "pe_mlp_2")  # :329-332
    # :334-335 — the self_update_pe term is computed and then overwritten: tanh(h2) only (Q3)
    pe[uniq] = node_pe2 + np.tanh(h2, dtype=ACC)  # :336-339 (row 0 becomes nonzero — Q2)
    return pe  # same object (Q7)


# --------------------------------------------------------------------------------------------
# the per-batch module-boundary path in the order the eval loop calls it
# (evaluate_model_utils.py:54-135): a3, caller's clone + index_put, C x a6, a7+a8, caller's append
# --------------------------------------------------------------------------------------------
def pe_step(p: dict, adj: Adjacency, hist: np.ndarray, batch_idx: int, src, dst, times, query_sets,
            num_fft_batches: int = 100, num_neighbors: int = 20):
    """One batch. `hist` is [V1, Th, d]; `query_sets` is a list of (node_ids, times) for the
    compute_neighborhood_pe calls (pos_src, pos_dst, neg_src, neg_dst). Returns
    (new_hist, neighbourhood outputs, current PE table)."""
    ids = np.unique(np.concatenate([src, dst]))
    if hist.shape[1] > num_fft_batches:
        hist = hist[:, -num_fft_batches:, :].copy()  # evaluate_model_utils.py:57-58
    fft_pe = fourier_transform_pe(p, ids, hist, batch_idx, num_fft_batches)
    cur = hist[:, -1, :].copy()  # :62
    cur[ids] = fft_pe  # :63
    outs = [compute_neighborhood_pe(p, adj, cur, q_ids, q_t, num_neighbors) for q_ids, q_t in query_sets]
    cur = update_pe(p, adj, cur, ids, src, dst, times, times.max(), num_neighbors)  # :120-129
    hist = np.concatenate([hist, cur[:, None, :]], axis=1)  # :135
    return hist, outs, cur
