"""Multi-GPU check of the host-fed, online peer step (PeerRank.step_host / run_host with ingest=True; csrc/host_step.cu
lstep_pe_step_peer_host / lstep_pe_steps_peer_host) with REAL ranks: one process per GPU under torchrun, CUDA IPC peer
pointers, flag barriers in peer memory:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29512 \
        tests/run_peer_host_ipc_check.py

Every rank holds no resident stream and a growable sampler of its own, receives the same host batches, ingests them and steps;
it also runs the single-GPU ChangeLogStream host-fed on the exact CSR of the whole stream and compares, BIT for bit, its share
of the per-query row sums of every step, its CSR replica against the other ranks' (gathered), its table replica and the owned
history rows. The log fills step by step; the steady part goes through run_host (the native multi-batch call). Prints one line
per rank and exits non-zero on a mismatch."""
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
    g.dst_node_ids = g.dst_node_ids.copy()
    g.dst_node_ids[::97] = g.src_node_ids[::97]  # self-loops
    V, E = g.num_nodes, g.num_edges
    src, dst, eid, tt = g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times
    exact = NeighborSampler.from_edges(src, dst, eid, tt, "recent", num_rows=V + 1)
    grow = NeighborSampler.growable(V + 1, min_slack=1)
    init = torch.from_numpy(seeded_normal(17, (V + 1, d), 0.3)).cuda()
    init[0] = 0
    e = np.zeros(0, np.int64)
    single = ChangeLogStream(build_dropin("fullu", g, exact, 172, d, 100, T, K)[0].eval(), e, e, np.zeros(0), B, K, initial_pe=init.clone())
    rk = PeerRank(build_dropin("fullu", g, grow, 172, d, 100, T, K)[0].eval(), rank, world, None, None, None, V, B, K, init.clone(), sampler=grow)
    rk.connect_ipc()
    neg = np.random.default_rng(3).integers(1, V + 1, E).astype(np.int64)
    qs = [src, dst, src, neg]
    n_step = T + 4  # the log is full after T - 1 steps
    for b in range(n_step):
        lo, hi = b * B, min((b + 1) * B, E)
        want = single.step_host(src[lo:hi], dst[lo:hi], tt[lo:hi], [x[lo:hi] for x in qs])
        got = rk.step_host(src[lo:hi], dst[lo:hi], tt[lo:hi], [x[lo:hi] for x in qs], ingest=True)
        q_off, q_rows = rk.share_of(hi - lo)
        assert np.array_equal(got, want[:, q_off:q_off + q_rows]), (rank, b)
    lo = n_step * B
    got = rk.run_host(src[lo:], dst[lo:], tt[lo:], [x[lo:] for x in qs], ingest=True)
    for i, b in enumerate(range(n_step, nb)):
        lo, hi = b * B, min((b + 1) * B, E)
        want = single.step_host(src[lo:hi], dst[lo:hi], tt[lo:hi], [x[lo:hi] for x in qs])
        q_off, q_rows = rk.share_of(hi - lo)
        assert np.array_equal(got[i, :, :q_rows], want[:, q_off:q_off + q_rows]), (rank, b, "run_host")
    rk.barrier()
    torch.cuda.synchronize()
    rk.check_errors()
    grow.check_errors()
    assert grow.num_entries == 2 * E and grow.regrows >= 1, (rank, grow.num_entries, grow.regrows)
    assert torch.equal(rk.cur, single.cur), (rank, "table replica")
    h = single.export_history()
    assert torch.equal(rk.export_history_rows(), h[rank::world]), (rank, "history")
    for a in (grow.fill, grow.indptr, grow.nbr, grow.eid, grow.t):  # every rank's CSR replica equals rank 0's
        ref = a.clone()
        dist.broadcast(ref, 0)
        assert torch.equal(a, ref), (rank, "CSR replica")
    print(f"rank {rank}/{world}: host-fed peer group == single GPU (bit-identical shares of {nb} online steps, CSR, table, owned history)",
          flush=True)
    dist.barrier()
    rk.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
