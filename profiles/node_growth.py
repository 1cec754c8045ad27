"""Cost of growing the node set online (add_nodes via run_host(ingest=True, grow=True)) on one GPU:

    python profiles/node_growth.py [--out FILE] [--reps 4] [--large-edges 20000000] [--large-batches 500]

The node ids of each synthetic stream are renumbered by first appearance (as an online stream's ids arrive), and the stream
is cut after the prefix that knows half of its nodes. Two arms start from that prefix (a growable sampler built from it):
  presized  the stream built for all V1 nodes up front, run_host(ingest=True);
  grown     the stream built for the known half only (row capacity = that half), run_host(ingest=True, grow=True): every
            call first adds the nodes up to its largest id, reallocating (capacity doubling) when the rows run out.
After T + 5 warm-up batches (the history fills), the rest is cut into --reps chunks of whole batches, each run on both arms,
alternating, host clock around calls that end synchronised. Reported per shape: edges/s of both arms, the rate ratio
grown / presized, the reallocations of the grown arm's table and history in the timed chunks and their time (device
synchronised around each, measured inside the timed calls), the sampler regrows, and whether both arms' row sums and final
tables are bit-identical. Shapes: Reddit (B = 200) and Flights (B = 2000) on PEStream (dense ring), and config 5 (10 M
nodes, B = 2000) on ChangeLogStream. Prints one JSON line with the card name and power limit read in the same run; exits 1
when the arms differ."""
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
from lstep_b200 import LSTEP, ChangeLogStream, NeighborSampler, PEStream, _lib, synth  # noqa: E402

EMPTY = np.zeros(0, np.int64)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = (x.strip() for x in q.split(",", 1))
        return name, power
    except Exception as e:  # the name from the runtime, the power limit unknown
        return torch.cuda.get_device_name(), f"unknown ({e})"


def model(sampler, T):
    torch.manual_seed(0)
    return LSTEP(np.zeros((2, 172), np.float32), np.zeros((1, 172), np.float32), sampler, sampler, pe_dim=172, num_neighbors=20,
                 time_feat_dim=100, num_fft_batches=T, device="cuda").to("cuda").eval()


def dense_ids(src, dst):
    """Ids renumbered by first appearance (1, 2, ...); returns (src, dst, V1)."""
    ends = np.stack([src, dst], 1).ravel()
    uniq, first = np.unique(ends, return_index=True)
    lab = np.zeros(int(ends.max()) + 1, np.int64)
    lab[uniq[np.argsort(first)]] = np.arange(1, len(uniq) + 1)
    return lab[src], lab[dst], len(uniq) + 1


def shape_run(cls, g, B, reps, n_batches=None, T=100, K=20):
    src, dst, V1 = dense_ids(g.src_node_ids, g.dst_node_ids)
    t = g.node_interact_times
    cm = np.maximum.accumulate(np.maximum(src, dst))
    p = int(np.searchsorted(cm, V1 // 2))  # the prefix knows half of the nodes
    E = len(src) if n_batches is None else min(len(src), p + n_batches * B)
    V1_0 = int(cm[p - 1]) + 1
    neg = (np.random.default_rng(1).random(E) * cm[:E]).astype(np.int64) + 1
    eid = np.arange(1, p + 1)
    init = torch.randn((V1, 172), device="cuda", generator=torch.Generator(device="cuda").manual_seed(2)) * 0.1
    init[0] = 0
    init[V1_0:] = 0
    sa = NeighborSampler.growable(V1, src[:p], dst[:p], eid, t[:p])
    a = cls(model(sa, T), EMPTY, EMPTY, np.zeros(0), B, K, initial_pe=init)
    sb = NeighborSampler.growable(V1_0, src[:p], dst[:p], eid, t[:p])
    b = cls(model(sb, T), EMPTY, EMPTY, np.zeros(0), B, K, initial_pe=init[:V1_0], max_nodes=V1)
    del init
    reallocs = []
    grow_capacity = b._grow_capacity

    def timed_grow(row_cap):  # (synchronised on both sides: a reallocation's own time)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        grow_capacity(row_cap)
        torch.cuda.synchronize()
        reallocs.append((int(row_cap), time.perf_counter() - t0))

    b._grow_capacity = timed_grow
    q = lambda lo, hi: [src[lo:hi], dst[lo:hi], neg[lo:hi]]
    run = {"presized": lambda lo, hi: a.run_host(src[lo:hi], dst[lo:hi], t[lo:hi], q(lo, hi), ingest=True),
           "grown": lambda lo, hi: b.run_host(src[lo:hi], dst[lo:hi], t[lo:hi], q(lo, hi), ingest=True, grow=True)}
    warm = p + (T + 5) * B
    res = {arm: f(p, warm) for arm, f in run.items()}
    same = bool(np.array_equal(res["presized"], res["grown"]))
    n_warm_realloc, regrows0 = len(reallocs), sb.regrows
    chunk = (E - warm) // reps // B * B
    ts = {arm: [] for arm in run}
    for r in range(reps):
        lo, hi = warm + r * chunk, warm + (r + 1) * chunk
        order = list(run) if r % 2 == 0 else list(run)[::-1]
        for arm in order:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res[arm] = run[arm](lo, hi)
            torch.cuda.synchronize()
            ts[arm].append(time.perf_counter() - t0)
        same &= bool(np.array_equal(res["presized"], res["grown"]))
    a.check_errors()
    b.check_errors()
    same &= bool(torch.equal(a.cur[:b.V1], b.cur[:b.V1]))
    eps = {arm: [round(chunk / x) for x in v] for arm, v in ts.items()}
    med = {arm: float(np.median(v)) for arm, v in eps.items()}
    timed = reallocs[n_warm_realloc:]
    return {"stream": cls.__name__, "B": B, "T": T, "queries": 3, "V1": V1, "V1_known_at_start": V1_0, "prefix_edges": p,
            "V1_grown_at_end": b.V1, "edges_per_chunk": chunk, "chunks": reps, "edges_per_s": eps,
            "rate_ratio_grown_over_presized": round(med["grown"] / med["presized"], 4),
            "reallocations_warmup": n_warm_realloc, "reallocations_timed": len(timed),
            "realloc_ms": [round(1e3 * x, 3) for _, x in reallocs], "realloc_row_caps": [c for c, _ in reallocs],
            "sampler_regrows_timed": sb.regrows - regrows0, "bit_identical": same}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=4)
    ap.add_argument("--large-edges", type=int, default=20_000_000, help="edges generated for the config-5 stream")
    ap.add_argument("--large-batches", type=int, default=500, help="online batches of B = 2000 after the half-known prefix")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    assert _lib.load().lstep_device_ok() == 1, "not a compute-capability 10.x device"
    line = {"metric": "node_growth"}
    line["shapes"] = [shape_run(PEStream, synth.make_graph("reddit", seed=0), 200, a.reps),
                      shape_run(PEStream, synth.make_graph("flights", seed=0), 2000, a.reps)]
    torch.cuda.empty_cache()
    g = synth.make_graph("scaleout", seed=0, num_edges=a.large_edges, num_nodes=10_000_000)
    line["shapes"].append(shape_run(ChangeLogStream, g, 2000, a.reps, n_batches=a.large_batches))
    name, power = card()
    line.update(gpu=name, power_limit=power,
                notes="edges/s: host clock around run_host calls that end synchronised, chunks alternated between the arms; the grown "
                      "arm's time includes its growth (add_nodes before each call) and its reallocations, each of which is also "
                      "timed on its own between device synchronisations (realloc_ms, all reallocations of the run in order)")
    s = json.dumps(line)
    print(s, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    if not all(r["bit_identical"] for r in line["shapes"]):
        sys.exit(1)


if __name__ == "__main__":
    main()
