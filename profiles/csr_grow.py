"""Cost of serving an edge stream that is still arriving (growable CSR, csrc/csr_grow.cu) on one GPU:

    python profiles/csr_grow.py [--out FILE] [--reps 3]

1. PEStream.run_host edges/s at the Reddit shape (B = 200) and the Flights shape (B = 2000), T = 100, d = 172, three query
   sets: on the exact CSR of the whole stream, and from EMPTY with ingest=True (every batch appended by its own step).
   After T + 5 warm-up batches the rest of the stream is cut into --reps chunks; each chunk runs on both arms, alternating,
   host clock around calls that end synchronised (run_host returns after its last result is read). The ingest arm's
   time includes its own capacity reservation. The two arms' results are compared bit for bit.
2. The append kernel alone (lstep_csr_ingest) by CUDA events over 400 launches at B = 200 and B = 2000.
3. The whole Reddit-shaped stream appended batch by batch (B = 200) from empty through NeighborSampler.ingest, for several
   min_slack values: regrows, their total time (each one synchronises before and, here, after), the total time, and
   capacity over entries at the end. The same for a graph with many rows and few entries per row (2 M nodes, 2 M edges,
   B = 2000), where min_slack decides most of the capacity: also the bytes of the CSR arrays at the end.
Prints one JSON line with the card name and power limit read in the same run."""
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
from lstep_b200 import LSTEP, NeighborSampler, PEStream, _lib, synth  # noqa: E402
from lstep_b200.sampler import MIN_SLACK  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = (x.strip() for x in q.split(",", 1))
        return name, power
    except Exception as e:  # the name from the runtime, the power limit unknown
        return torch.cuda.get_device_name(), f"unknown ({e})"


def model(sampler, V1, E, T):
    torch.manual_seed(0)
    return LSTEP(np.zeros((V1, 172), np.float32), np.zeros((E + 1, 172), np.float32), sampler, sampler, pe_dim=172, num_neighbors=20,
                 time_feat_dim=100, num_fft_batches=T, device="cuda").to("cuda").eval()


def run_host_arms(shape, B, reps, T=100, K=20):
    g = synth.make_graph(shape, seed=0)
    V1, E = g.num_nodes + 1, g.num_edges
    src, dst, t = g.src_node_ids, g.dst_node_ids, g.node_interact_times
    neg = np.random.default_rng(1).integers(1, V1, E).astype(np.int64)
    exact = NeighborSampler.from_edges(src, dst, g.edge_ids, t, num_rows=V1)
    grow = NeighborSampler.growable(V1)
    init = torch.randn((V1, 172), device="cuda", generator=torch.Generator(device="cuda").manual_seed(2)) * 0.1
    init[0] = 0
    a = PEStream(model(exact, V1, E, T), src, dst, t, B, K, initial_pe=init.clone())
    e = np.zeros(0, np.int64)
    b = PEStream(model(grow, V1, E, T), e, e, np.zeros(0), B, K, initial_pe=init.clone())
    warm = (T + 5) * B
    chunk = (E - warm) // reps // B * B
    same = True
    q = lambda lo, hi: [src[lo:hi], dst[lo:hi], neg[lo:hi]]
    ra = a.run_host(src[:warm], dst[:warm], t[:warm], q(0, warm))
    rb = b.run_host(src[:warm], dst[:warm], t[:warm], q(0, warm), ingest=True)
    same &= bool(np.array_equal(ra, rb))
    ts = {"exact": [], "ingest": []}
    for r in range(reps):
        lo, hi = warm + r * chunk, warm + (r + 1) * chunk
        for arm, st in (("exact", a), ("ingest", b)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = st.run_host(src[lo:hi], dst[lo:hi], t[lo:hi], q(lo, hi), ingest=arm == "ingest")
            torch.cuda.synchronize()
            ts[arm].append(time.perf_counter() - t0)
            if arm == "exact":
                ra = res
            else:
                same &= bool(np.array_equal(ra, res))
    a.check_errors()
    b.check_errors()
    same &= bool(torch.equal(a.cur, b.cur))
    eps = {arm: [round(chunk / x) for x in v] for arm, v in ts.items()}
    return {"shape": shape, "B": B, "T": T, "queries": 3, "edges_per_chunk": chunk, "warmup_edges": warm,
            "edges_per_s": eps, "median_ratio_ingest_over_exact": round(float(np.median(eps["ingest"]) / np.median(eps["exact"])), 4),
            "regrows": grow.regrows, "capacity_over_entries": round(grow.nnz / grow.num_entries, 3), "bit_identical": same}


def ingest_kernel_us(B, n_launch=400):
    lib = _lib.load()
    g = synth.make_graph("reddit", seed=3, num_edges=B * n_launch)
    V1 = g.num_nodes + 1
    s = NeighborSampler.growable(V1)
    s.reserve(g.src_node_ids, g.dst_node_ids)
    d = [torch.from_numpy(x).cuda() for x in (g.src_node_ids, g.dst_node_ids, g.node_interact_times)]
    stream = _lib.stream_ptr()

    def launch(i):
        lo = i * B
        _lib.check(lib.lstep_csr_ingest(s.csr_ref, _lib.ptr(s.fill), _lib.ptr(d[0][lo:]), _lib.ptr(d[1][lo:]), None, lo + 1,
                                        _lib.ptr(d[2][lo:]), B, _lib.ptr(s._err), stream), "lstep_csr_ingest")

    for i in range(20):  # warm-up: the first launches load the module
        launch(i)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(20, n_launch):
        launch(i)
    ev1.record()
    torch.cuda.synchronize()
    s.check_errors()
    return round(ev0.elapsed_time(ev1) * 1000.0 / (n_launch - 20), 2)


def from_empty(min_slack, B=200, **shape):
    g = synth.make_graph("reddit", seed=0, **shape)
    V1, E = g.num_nodes + 1, g.num_edges
    s = NeighborSampler.growable(V1, min_slack=min_slack)
    regrow_s = []
    inner = s._regrow

    def timed(need):
        t0 = time.perf_counter()
        inner(need)
        torch.cuda.synchronize()
        regrow_s.append(time.perf_counter() - t0)

    s._regrow = timed
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for lo in range(0, E, B):
        s.ingest(g.src_node_ids[lo:lo + B], g.dst_node_ids[lo:lo + B], g.edge_ids[lo:lo + B], g.node_interact_times[lo:lo + B])
    torch.cuda.synchronize()
    total = time.perf_counter() - t0
    s.check_errors()
    return {"min_slack": min_slack, "batches": (E + B - 1) // B, "regrows": s.regrows, "regrow_total_ms": round(1000 * sum(regrow_s), 2),
            "ingest_total_ms": round(1000 * total, 1), "entries": s.num_entries, "capacity": s.nnz,
            "capacity_over_entries": round(s.nnz / s.num_entries, 3),
            "csr_bytes": int(sum(x.numel() * x.element_size() for x in (s.indptr, s.nbr, s.eid, s.t, s.fill)))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    assert _lib.load().lstep_device_ok() == 1, "not a compute-capability 10.x device"
    line = {"metric": "csr_grow", "default_min_slack": MIN_SLACK}
    line["run_host"] = [run_host_arms("reddit", 200, a.reps), run_host_arms("flights", 2000, a.reps)]
    line["ingest_kernel_us"] = {"B200": ingest_kernel_us(200), "B2000": ingest_kernel_us(2000)}
    line["reddit_from_empty_B200"] = [from_empty(ms) for ms in (1, 4, 16, 64)]
    line["sparse_2M_nodes_2M_edges_from_empty_B2000"] = [from_empty(ms, B=2000, num_nodes=2_000_000, num_edges=2_000_000)
                                                         for ms in (4, 16, 64)]
    name, power = card()
    line.update(gpu=name, power_limit=power,
                notes="run_host: host clock around calls that end synchronised, chunks alternated between the arms; ingest arm "
                      "from an empty sampler and an empty PEStream, its time includes its capacity reservation (one regrow per "
                      "chunk at most); ingest_kernel_us: CUDA events around 380 back-to-back launches on one stream (not "
                      "overlapped with a step); from_empty: NeighborSampler.ingest per batch on the current stream")
    s = json.dumps(line)
    print(s, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    if not all(r["bit_identical"] for r in line["run_host"]):
        sys.exit(1)


if __name__ == "__main__":
    main()
