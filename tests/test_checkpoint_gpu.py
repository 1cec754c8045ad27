"""Checkpoint and resume of the change-log PE history (l-step_b200/checkpoint.py; ChangeLogStream / PeerRank save_checkpoint
and checkpoint=): a resumed run, at the same or any other world size, computes the bits of the uninterrupted single-GPU
run. The filter orders a node's versions by logical window position, not by ring slot, so its sums depend only on the
events of every position, which the checkpoint keeps."""
import hashlib
import os

import numpy as np
import pytest

from common import pe_close, seeded_normal
from lstep_b200 import synth

pytestmark = pytest.mark.gpu

B, K, D = 48, 20, 172


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    from lstep_b200 import _lib
    lib = _lib.load()
    assert lib.lstep_device_ok() == 1, "not a compute-capability 10.x device"
    return torch


@pytest.fixture(scope="module")
def setup(torch_cuda):
    """The small graph of the peer-group tests: T = 100, about 115 batches after e0 (filling and steady regime)."""
    torch = torch_cuda
    from harness import build_dropin
    from lstep_b200 import NeighborSampler
    g = synth.make_graph("tiny_bip", seed=4, num_nodes=300, num_edges=9000)
    V = g.num_nodes
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V + 1)
    lstep = build_dropin("fullu", g, s, 172, D, 100, 100, K)[0].eval()
    init = torch.from_numpy(seeded_normal(17, (V + 1, D), 0.3)).cuda()
    init[0] = 0
    e0 = g.num_edges - 115 * B - 7
    neg = torch.from_numpy(np.random.default_rng(3).integers(1, V + 1, g.num_edges).astype(np.int64)).cuda()
    return dict(g=g, V=V, s=s, lstep=lstep, init=init, e0=e0, neg=neg)


def _stream(S, **kw):
    from lstep_b200 import ChangeLogStream
    g = S["g"]
    kw.setdefault("start", S["e0"])
    return ChangeLogStream(S["lstep"], g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, **kw)


def _ranks(S, world, **kw):
    from lstep_b200 import PeerLocalGroup, PeerRank
    g = S["g"]
    ranks = [PeerRank(S["lstep"], r, world, g.src_node_ids, g.dst_node_ids, g.node_interact_times, S["V"], B, K, start=S["e0"], sampler=S["s"], **kw)
             for r in range(world)]
    return ranks, PeerLocalGroup(ranks)


def _queries(st, S, b):
    lo, hi, _, _ = st.batch_arrays(b)
    return [st.src[lo:hi], st.dst[lo:hi], st.src[lo:hi], S["neg"][lo:hi].contiguous()]


def _files(path):
    return {f: hashlib.sha256(open(os.path.join(path, f), "rb").read()).hexdigest() for f in sorted(os.listdir(path))}


def test_changelog_stream_resume_is_bit_identical(setup, tmp_path):
    """Saved once while the history fills (len < T) and once in the steady regime (head != 0): the resumed streams give
    torch.equal outputs and tables at every later step, and the same history at the end."""
    torch, S = __import__("torch"), setup
    st = _stream(S, initial_pe=S["init"].clone())
    saves = {37: None, 108: None}
    for b in range(st.num_batches):
        if b in saves:
            assert (b < 100) == (st.len < st.T) and (b < 100 or st.head != 0)
            st.save_checkpoint(str(tmp_path / str(b)))
            r = _stream(S, checkpoint=str(tmp_path / str(b)))
            assert (r.head, r.len, r.batch_idx, r.steps_done) == (0, st.len, st.batch_idx, st.steps_done)
            assert torch.equal(r.cur, st.cur)
            saves[b] = r
        qs = _queries(st, S, b)
        want = st.step(b, qs)
        for r in saves.values():
            if r is not None:
                assert torch.equal(r.step(b, qs), want), b
                assert torch.equal(r.cur, st.cur), b
    h = st.export_history()
    for b, r in saves.items():
        assert torch.equal(r.export_history(), h), b


@pytest.mark.parametrize("N,M,save_at", [(1, 3, 50), (2, 3, 104), (3, 2, 104), (8, 1, 104), (2, 8, 60)])
def test_peer_group_resharded_resume_is_bit_identical(setup, tmp_path, N, M, save_at):
    """Saved by an emulated group of world N, resumed by one of world M: every step's shares, every replica after a barrier
    and the owners' history rows are bit-identical to the uninterrupted single-GPU ChangeLogStream."""
    torch, S = __import__("torch"), setup
    st = _stream(S, initial_pe=S["init"].clone())
    ranks, grp = _ranks(S, N, initial_pe=S["init"].clone())
    for b in range(save_at):
        qs = _queries(st, S, b)
        st.step(b, qs)
        grp.step(b, qs)
    for rk in ranks:
        rk.check_errors()
        rk.save_checkpoint(str(tmp_path))
    del ranks, grp
    ranks, grp = _ranks(S, M, checkpoint=str(tmp_path))
    for rk in ranks:
        assert (rk.head, rk.len, rk.batch_idx, rk.steps_done) == (0, st.len, st.batch_idx, st.steps_done)
        assert torch.equal(rk.cur, st.cur), rk.rank
    for b in range(save_at, st.num_batches):
        qs = _queries(st, S, b)
        want = st.step(b, qs)
        got = torch.cat(grp.step(b, qs), dim=1)
        assert got.shape == want.shape and torch.equal(got, want), b
        grp.barrier()
        for rk in ranks:
            assert torch.equal(rk.cur, st.cur), (b, rk.rank)
    for rk in ranks:
        rk.check_errors()
    h = st.export_history()
    for rk in ranks:
        assert torch.equal(rk.export_history_rows(), h[rk.rank::M]), rk.rank


def test_two_evaluations_from_one_checkpoint(setup, tmp_path):
    """The reference's train-then-evaluate-twice bracket: two streams loaded from one checkpoint (saved while len < T) run
    on two different splits with batch_idx restarted at 0; the files stay as they were and each stream matches a dense
    PEStream built from the history exported at the save point, within the change-log-vs-ring bar."""
    torch, S = __import__("torch"), setup
    from lstep_b200 import PEStream
    g, e0 = S["g"], S["e0"]
    st = _stream(S, initial_pe=S["init"].clone())
    save_at = 45
    for b in range(save_at):
        st.step(b, _queries(st, S, b))
    st.save_checkpoint(str(tmp_path))
    h = st.export_history()
    files = _files(tmp_path)
    split_lo = [e0 + save_at * B, g.num_edges - 30 * B]
    for lo in split_lo:
        stop = lo + 30 * B
        r = _stream(S, checkpoint=str(tmp_path), batch_idx=0, start=lo, stop=stop)
        a = PEStream(S["lstep"], g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, history=h.clone(), start=lo, stop=stop)
        assert torch.equal(r.export_history(), a.export_history()) and torch.equal(r.cur, a.cur)
        for b in range(r.num_batches):
            qs = _queries(a, S, b)
            oa, orr = a.step(b, qs), r.step(b, qs)
            ok, w = pe_close(orr.cpu().numpy(), oa.cpu().numpy(), 1e-5)
            assert ok, (lo, b, "outputs", w)
            ok, w = pe_close(r.cur.cpu().numpy(), a.cur.cpu().numpy(), 1e-5)
            assert ok, (lo, b, "table", w)
        ok, w = pe_close(r.export_history().cpu().numpy(), a.export_history().cpu().numpy(), 1e-5)
        assert ok, (lo, "history", w)
    assert _files(tmp_path) == files


def test_peer_rank_dense_history_equals_changelog_stream(setup):
    """PeerRank(history=dense) and ChangeLogStream(history=dense) go through the same loader: bit-identical state and steps."""
    torch, S = __import__("torch"), setup
    st = _stream(S, initial_pe=S["init"].clone())
    for b in range(30):
        st.step(b, _queries(st, S, b))
    h = st.export_history()
    c = _stream(S, history=h.clone())
    ranks, grp = _ranks(S, 2, history=h.clone())
    hc = c.export_history()
    assert torch.equal(hc, h)
    for rk in ranks:
        assert torch.equal(rk.cur, c.cur) and torch.equal(rk.export_history_rows(), hc[rk.rank::2]), rk.rank
    for b in range(10):
        qs = _queries(c, S, b)
        want = c.step(b, qs)
        assert torch.equal(torch.cat(grp.step(b, qs), dim=1), want), b
    grp.barrier()
    for rk in ranks:
        assert torch.equal(rk.cur, c.cur)


def test_resume_rejects_before_any_device_write(setup, tmp_path):
    """A checkpoint of another model shape or one that needs more event capacity than the new rank has is refused."""
    S = setup
    from lstep_b200 import _lib
    st = _stream(S, initial_pe=S["init"].clone())
    for b in range(5):
        st.step(b, _queries(st, S, b))
    st.save_checkpoint(str(tmp_path))
    with pytest.raises(_lib.LstepError, match="event_capacity"):
        _stream(S, checkpoint=str(tmp_path), event_capacity=4)
    with pytest.raises(_lib.LstepError, match="event_capacity"):
        _ranks(S, 2, checkpoint=str(tmp_path), event_capacity=4)
    g = S["g"]
    from lstep_b200 import PeerRank
    with pytest.raises(ValueError, match="V1"):
        PeerRank(S["lstep"], 0, 1, g.src_node_ids, g.dst_node_ids, g.node_interact_times, S["V"] + 5, B, K, start=S["e0"], sampler=S["s"],
                 checkpoint=str(tmp_path))
    with pytest.raises(ValueError, match="exactly one"):
        PeerRank(S["lstep"], 0, 1, g.src_node_ids, g.dst_node_ids, g.node_interact_times, S["V"], B, K, S["init"], start=S["e0"], sampler=S["s"],
                 checkpoint=str(tmp_path))


@pytest.mark.parametrize("world", [2])
def test_peer_checkpoint_over_ipc(torch_cuda, world):
    """Real ranks (tests/run_peer_checkpoint_check.py under torchrun): save, build fresh ranks from the checkpoint, connect
    them over CUDA IPC and continue step by step and through the native multi-step call. Needs `world` GPUs."""
    import subprocess
    import sys
    torch = torch_cuda
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, this box has {torch.cuda.device_count()}")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    port = 29400 + os.getpid() % 90
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(root, "tests", "run_peer_checkpoint_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    assert res.stdout.count("resumed peer group == single GPU") == world, res.stdout[-2000:]
