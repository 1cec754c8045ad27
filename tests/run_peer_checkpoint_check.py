"""Multi-GPU check of checkpoint and resume for the peer group (l-step_b200/peer.py, l-step_b200/checkpoint.py) with REAL
ranks: one process per GPU under torchrun.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29411 \
        tests/run_peer_checkpoint_check.py

Every rank runs the single-GPU ChangeLogStream on a small graph as the reference. The group steps while its history fills,
every rank saves its shard, and FRESH ranks are built from the checkpoint and connected over CUDA IPC. They continue step
by step (lstep_pe_step_peer) to a full window, then in one native call (lstep_pe_steps_peer). Their shares of every step's
outputs, the table replicas and the owned history rows must equal the reference BIT for bit. Prints one line per rank and
exits non-zero on a mismatch."""
import os
import shutil
import sys
import tempfile

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
    g = synth.make_graph("tiny_bip", seed=4, num_nodes=300, num_edges=9000)
    V, d, K, B = g.num_nodes, 172, 20, 48
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V + 1)
    lstep = build_dropin("fullu", g, s, 172, d, 100, 100, K)[0].eval()
    init = torch.from_numpy(seeded_normal(17, (V + 1, d), 0.3)).cuda()
    init[0] = 0
    e0 = g.num_edges - 135 * B - 7
    single = ChangeLogStream(lstep, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, initial_pe=init.clone(), start=e0)
    old = PeerRank(lstep, rank, world, g.src_node_ids, g.dst_node_ids, g.node_interact_times, V, B, K, init.clone(), start=e0, sampler=s)
    old.connect_ipc()
    neg = torch.from_numpy(np.random.default_rng(3).integers(1, V + 1, g.num_edges).astype(np.int64)).cuda()
    nb = single.num_batches

    def queries(b):
        lo, hi, _, _ = single.batch_arrays(b)
        return [single.src[lo:hi], single.dst[lo:hi], single.src[lo:hi], neg[lo:hi].contiguous()]

    save_at, n_single = 60, 104  # saved while the history fills (T = 100); full after 99 steps
    for b in range(save_at):
        single.step(b, queries(b))
        old.step(b, queries(b))
    path = [tempfile.mkdtemp(prefix="lstep_ckpt_") if rank == 0 else None]
    dist.broadcast_object_list(path, src=0)
    old.save_checkpoint(path[0])
    dist.barrier()
    rk = PeerRank(lstep, rank, world, g.src_node_ids, g.dst_node_ids, g.node_interact_times, V, B, K, start=e0, sampler=s, checkpoint=path[0])
    rk.connect_ipc()
    assert (rk.len, rk.batch_idx, rk.steps_done) == (single.len, single.batch_idx, single.steps_done), rank
    assert torch.equal(rk.cur, single.cur), (rank, "loaded table")
    for b in range(save_at, n_single):
        want = single.step(b, queries(b))
        got = rk.step(b, queries(b))
        q_off, q_rows = rk.share(b)
        assert torch.equal(got, want[:, q_off:q_off + q_rows]), (rank, b)
    n_run = nb - n_single
    stride = 4 * (B // world + 1) * d
    out = torch.zeros((n_run, 4, B // world + 1, d), dtype=torch.float32, device="cuda")
    rk.run(n_single, n_run, [rk.src, rk.dst, rk.src, neg], out=out, out_step_stride=stride)
    for i in range(n_run):
        b = n_single + i
        want = single.step(b, queries(b))
        q_off, q_rows = rk.share(b)
        got = out[i].reshape(-1)[:4 * q_rows * d].view(4, q_rows, d)
        assert torch.equal(got, want[:, q_off:q_off + q_rows]), (rank, b, "native run")
    rk.barrier()
    torch.cuda.synchronize()
    rk.check_errors()
    assert torch.equal(rk.cur, single.cur), (rank, "table replica")
    h = single.export_history()
    assert torch.equal(rk.export_history_rows(), h[rank::world]), (rank, "history")
    print(f"rank {rank}/{world}: resumed peer group == single GPU (checkpoint after {save_at} steps; bit-identical outputs of "
          f"{nb - save_at} later steps, table replica, owned history)", flush=True)
    dist.barrier()
    rk.close()
    old.close()
    if rank == 0:
        shutil.rmtree(path[0], ignore_errors=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
