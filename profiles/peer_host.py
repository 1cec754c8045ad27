"""Host-fed and online steps on the peer group (PeerRank.run_host, csrc/host_step.cu lstep_pe_steps_peer_host) at BASELINE
config 5 (10 M nodes, B = 2000, T = 100, d = 172, four query sets), against the resident stream:

    python profiles/peer_host.py [--out FILE]                                  # N = 1
    python -m torch.distributed.run --nproc-per-node N profiles/peer_host.py   # N ranks, one GPU each

Three arms of PeerRank on the same batches of a synth.make_graph("scaleout") stream, each rank with its own table replica,
change log and CSR replica:
    resident     PeerRank.run on the stream uploaded at construction (the per-batch plan computed on the host up front)
    host_exact   PeerRank.run_host on the exact CSR of the whole stream, no resident stream (plan derived on the device)
    host_ingest  PeerRank.run_host(ingest=True) from a growable sampler holding the edges before the online part
The log fills over T batches and a few more steady batches warm every arm up; then the rest is cut into --reps chunks, each run
on every arm in turn (alternating), host clock around calls that end synchronised (max over ranks). Reports ms per step, the
ratio to resident, the host-side part of host_ingest's time, and whether host_exact and host_ingest give bit-identical results
and tables. Prints one JSON line (rank 0) with the card name and power limit read in the same run; exits 1 when the two host
arms differ."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from lstep_b200 import LSTEP, NeighborSampler, PeerRank, _lib, synth  # noqa: E402
from lstep_b200.peer import check_host_batch  # noqa: E402
from lstep_b200.sampler import row_counts  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = (x.strip() for x in q.split(",", 1))
        return name, power
    except Exception as e:  # the name from the runtime, the power limit unknown
        return torch.cuda.get_device_name(), f"unknown ({e})"


def model(T, dev):
    torch.manual_seed(0)
    return LSTEP(np.zeros((2, 172), np.float32), np.zeros((1, 172), np.float32), None, None, pe_dim=172, num_neighbors=20,
                 time_feat_dim=100, num_fft_batches=T, device=dev).to(dev).eval()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=10_000_000)
    ap.add_argument("--edges", type=int, default=20_000_000, help="edges of the scale-out stream (prefix + online part)")
    ap.add_argument("--batch", type=int, default=2000)
    ap.add_argument("--chunk", type=int, default=60, help="batches per timed chunk")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file (rank 0)")
    a = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    assert _lib.load().lstep_device_ok() == 1, "not a compute-capability 10.x device"
    V, B, T, K = a.nodes, a.batch, 100, 20
    g = synth.make_graph("scaleout", seed=0, num_edges=a.edges, num_nodes=V)
    V1, E = g.num_nodes + 1, g.num_edges
    src, dst, eid, t = g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times
    warm = T + 5
    n_online = warm + a.reps * a.chunk
    e0 = E - n_online * B
    assert e0 > 0, "--edges too small for the online part"
    neg = np.random.default_rng(4).integers(1, V1, E).astype(np.int64)
    negd = torch.from_numpy(neg).to(dev)
    init = torch.randn((V1, 172), device=dev, generator=torch.Generator(device=dev).manual_seed(3)) * 0.1
    init[0] = 0
    res = PeerRank(model(T, dev), rank, world, src, dst, t, V, B, K, init, start=e0)
    exact = res.sampler
    grow = NeighborSampler.growable(V1, src[:e0], dst[:e0], eid[:e0], t[:e0])
    arms = {"resident": res,
            "host_exact": PeerRank(model(T, dev), rank, world, None, None, None, V, B, K, init, sampler=exact),
            "host_ingest": PeerRank(model(T, dev), rank, world, None, None, None, V, B, K, init, sampler=grow)}
    del init
    for rk in arms.values():
        rk.connect_ipc()
    q = lambda lo, hi: [src[lo:hi], dst[lo:hi], src[lo:hi], neg[lo:hi]]

    def run(arm, b0, nbat):
        rk = arms[arm]
        lo, hi = e0 + b0 * B, e0 + (b0 + nbat) * B
        if arm == "resident":
            if rk.len < T:
                for b in range(b0, b0 + nbat):
                    l2, h2 = rk.batch(b)
                    rk.step(b, [rk.src[l2:h2], rk.dst[l2:h2], rk.src[l2:h2], negd[l2:h2]])
            else:
                rk.run(b0, nbat, [rk.src, rk.dst, rk.src, negd])
            return None
        return rk.run_host(src[lo:hi], dst[lo:hi], t[lo:hi], q(lo, hi), ingest=arm == "host_ingest")

    out = {arm: run(arm, 0, warm) for arm in arms}
    same = bool(np.array_equal(out["host_exact"], out["host_ingest"]))
    ms = {arm: [] for arm in arms}
    host_ms = []
    for r in range(a.reps):
        b0 = warm + r * a.chunk
        for arm in arms:
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            out[arm] = run(arm, b0, a.chunk)
            torch.cuda.synchronize()
            dt = torch.tensor([(time.perf_counter() - t0) * 1e3 / a.chunk], device=dev)
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            ms[arm].append(round(float(dt.item()), 4))
        same &= bool(np.array_equal(out["host_exact"], out["host_ingest"]))
        # the host-side work of host_ingest's call alone, on the same chunk: validation, and the two row counts of the sampler's
        # host mirror (reserve before the native call, the fill update after it)
        lo, hi = e0 + b0 * B, e0 + (b0 + a.chunk) * B
        t0 = time.perf_counter()
        check_host_batch(src[lo:hi], dst[lo:hi], t[lo:hi], q(lo, hi), V1, hi - lo, None, (V1, float(t[lo]), 1))
        row_counts(src[lo:hi], dst[lo:hi])
        row_counts(src[lo:hi], dst[lo:hi])
        host_ms.append(round((time.perf_counter() - t0) * 1e3 / a.chunk, 4))
    for rk in arms.values():
        rk.barrier()
    torch.cuda.synchronize()
    for rk in arms.values():
        rk.check_errors()
    same &= bool(torch.equal(arms["host_exact"].cur, arms["host_ingest"].cur))
    tables_equal_resident = bool(torch.equal(arms["resident"].cur, arms["host_exact"].cur))
    flags = torch.tensor([int(same), int(tables_equal_resident)], device=dev)
    if world > 1:
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    med = {arm: float(np.median(v)) for arm, v in ms.items()}
    line = {"metric": "peer_host", "world": world, "nodes": V, "B": B, "T": T, "queries": 4, "stream_edges": E, "prefix_edges": e0,
            "warmup_batches": warm, "batches_per_chunk": a.chunk, "ms_per_step": ms,
            "median_ratio_over_resident": {arm: round(med[arm] / med["resident"], 4) for arm in ms},
            "host_ingest_host_side_ms_per_step": host_ms,
            "host_arms_bit_identical": bool(flags[0].item()), "resident_table_equals_host": bool(flags[1].item()),
            "regrows": grow.regrows}
    name, power = card()
    line.update(gpu=name, power_limit=power,
                notes="ms per step = host clock around one call that ends synchronised over a chunk of batches, divided by the chunk's "
                      "batches, max over ranks; chunks alternated between the arms; resident = PeerRank.run (lstep_pe_steps_peer), "
                      "host_exact / host_ingest = PeerRank.run_host (lstep_pe_steps_peer_host) on the exact CSR of the whole stream / "
                      "with ingest=True from a growable sampler holding the prefix (its time includes validating the chunk and "
                      "reserving its room); host_ingest_host_side_ms_per_step = the host-side part of that arm alone, timed on the same chunk: "
                      "check_host_batch and the two row counts of the sampler's host mirror (reserve, fill update); every arm steps the "
                      "same batches; the host arms also copy every batch in and the row sums "
                      "out, which the resident arm does not")
    if rank == 0:
        s = json.dumps(line)
        print(s, flush=True)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                f.write(s + "\n")
    for rk in arms.values():
        rk.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if not line["host_arms_bit_identical"]:
        sys.exit(1)


if __name__ == "__main__":
    main()
