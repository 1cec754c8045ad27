"""CPU tests of the multi-GPU (node-id sharded) path's host logic: the per-rank partition plan and the
all-to-all-v row exchange, the latter under torch.distributed with the gloo backend, world size 2."""
import os

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from lstep_b200 import shard, synth


@pytest.mark.parametrize("world", [2, 3, 8])
def test_partition_plan_covers_batch_exactly_once(world):
    g = synth.make_graph("tiny_bip", seed=0)
    lo, B = 900, 64
    src, dst = g.src_node_ids[lo:lo + B], g.dst_node_ids[lo:lo + B]
    ids = np.unique(np.concatenate([src, dst]))
    seen = []
    n_valid_total = 0
    for r in range(world):
        pl = shard.plan_batch(ids, src, dst, world, r)
        assert np.all(pl["mine"] % world == r) and np.array_equal(ids[pl["pos"]], pl["mine"])
        assert np.array_equal(pl["local"] * world + r, pl["mine"])
        assert np.all(pl["others"] % world != r)
        # every other endpoint of an owned node's edge is either owned or requested
        for s_, d_ in zip(src, dst):
            if s_ % world == r:
                assert d_ % world == r or d_ in pl["others"]
            if d_ % world == r:
                assert s_ % world == r or s_ in pl["others"]
        seen.append(pl["mine"])
        n_valid_total += pl["n_valid"]
    assert np.array_equal(np.sort(np.concatenate(seen)), ids)
    assert n_valid_total == min(len(ids), B)
    queries = [src, dst, src]
    rows = [shard.plan_queries(queries, world, r)[0] for r in range(world)]
    assert np.array_equal(np.sort(np.concatenate(rows)), np.arange(3 * B))


def _exchange_worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        comm = shard.DistGroup()
        V1, d = 41, 6
        # every rank's copy: owned rows authoritative (value = 1000*owner + row), other rows garbage
        table = torch.full((V1, d), -1.0)
        own = torch.arange(rank, V1, world)
        table[own] = (1000.0 * rank + own.float())[:, None].expand(-1, d)
        gen = torch.Generator().manual_seed(rank)
        need = torch.unique(torch.randint(0, V1, (17,), generator=gen))
        need = need[need % world != rank]
        need_sorted, _, counts = shard.group_by_owner(need, world)
        shard.fetch_rows(comm, table, need_sorted, counts, world)
        want = (1000.0 * (need % world).float() + need.float())[:, None].expand(-1, d)
        ok = bool(torch.equal(table[need], want)) and bool(torch.equal(table[own], (1000.0 * rank + own.float())[:, None].expand(-1, d)))
        # all-to-all-v of ragged rows keeps per-source order
        send = torch.arange(5 * world, dtype=torch.float32).reshape(-1, 1) + 100 * rank
        cnt = [5] * world
        recv, rc = comm.alltoallv(send, cnt)
        ok = ok and rc == [5] * world and bool(torch.equal(recv[:5, 0], torch.arange(5 * rank, 5 * rank + 5, dtype=torch.float32)))
        x = torch.ones(3) * (rank + 1)
        comm.allreduce_sum(x)
        ok = ok and float(x[0]) == sum(range(1, world + 1))
        ret[rank] = ok
    finally:
        dist.destroy_process_group()


def test_row_exchange_gloo_world2():
    world = 2
    port = 29500 + (os.getpid() % 2000)
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_exchange_worker, args=(world, port, ret), nprocs=world, join=True)
    assert dict(ret) == {0: True, 1: True}


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_peer_group_plan_partitions_every_batch(world):
    """Host plan of the peer group (l-step_b200/peer.py::peer_batch_plan): over the ranks, the owned-node lists partition every
    batch's sorted unique id list, `pos` are the owners' positions in it (where a row goes in the peers' new_rows / filt
    buffers), and the a6 shares partition the batch's edges — ragged last batch and ranks without any node included."""
    from lstep_b200.peer import peer_batch_plan
    g = synth.make_graph("tiny_bip", seed=1)
    src, dst = g.src_node_ids[:1000 + 37], g.dst_node_ids[:1000 + 37]
    B = 48
    plans = [peer_batch_plan(src, dst, B, world, r) for r in range(world)]
    nb = plans[0]["num_batches"]
    assert nb == (len(src) + B - 1) // B
    for b in range(nb):
        lo, hi = b * B, min((b + 1) * B, len(src))
        ids = np.unique(np.concatenate([src[lo:hi], dst[lo:hi]]))
        covered = np.zeros(len(ids), dtype=int)
        edges = np.zeros(hi - lo, dtype=int)
        for r, pl in enumerate(plans):
            assert np.array_equal(pl["ids"][pl["ids_off"][b]:pl["ids_off"][b + 1]], ids)
            mine = pl["mine"][pl["mine_off"][b]:pl["mine_off"][b + 1]]
            pos = pl["pos"][pl["mine_off"][b]:pl["mine_off"][b + 1]]
            assert np.all(mine % world == r) and np.array_equal(ids[pos], mine) and np.all(np.diff(pos) > 0)
            covered[pos] += 1
            q_off, q_rows = pl["share"][b]
            edges[q_off:q_off + q_rows] += 1
        assert np.all(covered == 1) and np.all(edges == 1)


@pytest.mark.parametrize("start,stop,B", [(0, None, 48), (213, 1037, 48), (5, 9, 200), (40, 40, 16)])
def test_single_gpu_plan_equals_the_per_batch_loop(start, stop, B):
    """The plan of a single-GPU stream (world 1: PEStream / ChangeLogStream) equals the per-batch loop it replaced, restated in
    numpy: batches of B edges from `start` (the last one ragged), each with its first edge, edge count, largest time and
    sorted unique nodes, concatenated with offsets."""
    from lstep_b200.peer import batch_plan
    g = synth.make_graph("tiny_bip", seed=3)
    src, dst, t = g.src_node_ids, g.dst_node_ids, g.node_interact_times
    stop = len(src) if stop is None else stop
    pl = batch_plan(src, dst, t, start, stop, B)
    batch_lo = list(range(start, stop, B))
    ids, off, n_edges, tmax = [], [0], [], []
    for lo in batch_lo:
        hi = min(lo + B, stop)
        u = np.unique(np.concatenate([src[lo:hi], dst[lo:hi]]))
        ids.append(u)
        off.append(off[-1] + len(u))
        n_edges.append(hi - lo)
        tmax.append(float(t[lo:hi].max()))
    assert pl["num_batches"] == len(batch_lo)
    assert pl["lo"].tolist() == batch_lo and pl["n_edges"].tolist() == n_edges and pl["tmax"].tolist() == tmax
    assert pl["ids_off"].tolist() == off
    assert np.array_equal(pl["ids"], np.concatenate(ids) if ids else np.zeros(0, np.int64))
    for a in ("lo", "n_edges", "ids", "ids_off"):
        assert pl[a].dtype == np.int64, a
