"""Multi-GPU check of a peer group whose node set grows during the run (PeerRank.step_host / run_host with ingest=True and
grow=True) with REAL ranks: one process per GPU under torchrun, CUDA IPC peer pointers, flag barriers in peer memory:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29514 \
        tests/run_peer_growth_ipc_check.py

The node ids of the stream are renumbered by first appearance, and every rank starts knowing only the nodes of the first
batches, with a small row capacity, so that each rank reallocates its table replica, its owned change-log rows and its CSR
replica mid-run (no IPC handle changes: the group shares only the batch-sized regions). Every rank also runs the single-GPU
ChangeLogStream built pre-sized to the final node count and compares, BIT for bit, its share of every step's per-query row
sums, its table replica and its owned history rows. Prints one line per rank and exits non-zero on a mismatch."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "golden")]
from common import seeded_normal  # noqa: E402
from harness import build_dropin  # noqa: E402
from lstep_b200 import ChangeLogStream, NeighborSampler, PeerRank, synth  # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    T, K, d, B = 100, 20, 172, 48
    nb = T + 20
    g = synth.make_graph("tiny_bip", seed=6, num_nodes=300, num_edges=nb * B - 7)
    t = g.node_interact_times
    q = (t[-1] - t[0]) / (g.num_edges / 100.0)
    g.node_interact_times = np.floor(t / q) * q  # runs of equal times across batch boundaries
    ends = np.stack([g.src_node_ids, g.dst_node_ids], 1).ravel()
    uniq, first = np.unique(ends, return_index=True)
    lab = np.zeros(int(ends.max()) + 1, np.int64)
    lab[uniq[np.argsort(first)]] = np.arange(1, len(uniq) + 1)  # ids by first appearance, as an online stream's arrive
    src, dst, tt = lab[g.src_node_ids], lab[g.dst_node_ids], g.node_interact_times
    E, V1 = len(src), len(uniq) + 1
    V1_0 = int(max(src[:2 * B].max(), dst[:2 * B].max())) + 1
    init = torch.from_numpy(seeded_normal(17, (V1, d), 0.3)).cuda()
    init[0] = 0
    init[V1_0:] = 0  # the initial row of a new node
    e = np.zeros(0, np.int64)
    pre = NeighborSampler.growable(V1)
    single = ChangeLogStream(build_dropin("fullu", g, pre, 172, d, 100, T, K)[0].eval(), e, e, np.zeros(0), B, K, initial_pe=init.clone())
    grow = NeighborSampler.growable(V1_0, row_capacity=V1_0 + 8)
    rk = PeerRank(build_dropin("fullu", g, grow, 172, d, 100, T, K)[0].eval(), rank, world, None, None, None, V1_0 - 1, B, K,
                  init[:V1_0].clone(), sampler=grow, row_capacity=V1_0 + 8, max_nodes=V1)
    rk.connect_ipc()
    cm = np.maximum.accumulate(np.maximum(src, dst))
    neg = (np.random.default_rng(3).random(E) * cm).astype(np.int64) + 1
    qs = [src, dst, src, neg]
    n_step = T + 4  # the log is full after T - 1 steps
    for b in range(n_step):
        lo, hi = b * B, min((b + 1) * B, E)
        want = single.step_host(src[lo:hi], dst[lo:hi], tt[lo:hi], [x[lo:hi] for x in qs], ingest=True)
        got = rk.step_host(src[lo:hi], dst[lo:hi], tt[lo:hi], [x[lo:hi] for x in qs], ingest=True, grow=True)
        q_off, q_rows = rk.share_of(hi - lo)
        assert np.array_equal(got, want[:, q_off:q_off + q_rows]), (rank, b)
    lo = n_step * B
    got = rk.run_host(src[lo:], dst[lo:], tt[lo:], [x[lo:] for x in qs], ingest=True, grow=True)
    for i, b in enumerate(range(n_step, nb)):
        lo, hi = b * B, min((b + 1) * B, E)
        want = single.step_host(src[lo:hi], dst[lo:hi], tt[lo:hi], [x[lo:hi] for x in qs], ingest=True)
        q_off, q_rows = rk.share_of(hi - lo)
        assert np.array_equal(got[i, :, :q_rows], want[:, q_off:q_off + q_rows]), (rank, b, "run_host")
    rk.barrier()
    torch.cuda.synchronize()
    rk.check_errors()
    assert rk.V1 == V1 and rk.row_cap > V1_0 + 8, (rank, rk.V1, rk.row_cap)
    assert torch.equal(rk.cur[:V1], single.cur), (rank, "table replica")
    h = single.export_history()
    assert torch.equal(rk.export_history_rows(), h[rank::world]), (rank, "history")
    print(f"rank {rank}/{world}: growing peer group == pre-sized single GPU (bit-identical shares of {nb} online steps, {V1_0} -> {V1} "
          f"nodes, table, owned history)", flush=True)
    dist.barrier()
    rk.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
