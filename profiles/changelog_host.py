"""Host-fed and online steps on the change-log history (ChangeLogStream.run_host, csrc/host_step.cu) on one GPU:

    python profiles/changelog_host.py [--out FILE] [--reps 3] [--large-edges 20000000]

1. Edges/s at the Reddit shape (B = 200) and the Flights shape (B = 2000), T = 100, d = 172, three query sets, four arms:
   ChangeLogStream.run (resident stream, one C call per step), ChangeLogStream.run_host on the exact CSR of the whole
   stream, ChangeLogStream.run_host(ingest=True) from an empty sampler, and PEStream.run_host (dense ring) for reference.
   After T + 5 warm-up batches the rest of the stream is cut into --reps chunks; each chunk runs on every arm, alternating,
   host clock around calls that end synchronised. The two ChangeLogStream.run_host arms' results and tables are compared
   bit for bit.
2. One large shape: 10 M nodes, B = 2000, a growable sampler built from the first --large-edges minus --large-batches * B
   edges of a synth.make_graph("scaleout") stream, then --large-batches online batches through run_host(ingest=True): the
   log fills over T batches, the rest (steady regime) is timed. Reports edges/s, history_bytes(), the CSR's bytes and the
   peak device memory of the run.
Prints one JSON line with the card name and power limit read in the same run; exits 1 when the run_host arms differ."""
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


def csr_bytes(s):
    return int(sum(x.numel() * x.element_size() for x in (s.indptr, s.nbr, s.eid, s.t) + ((s.fill,) if s.is_growable else ())))


def arms(shape, B, reps, T=100, K=20):
    g = synth.make_graph(shape, seed=0)
    V1, E = g.num_nodes + 1, g.num_edges
    src, dst, t = g.src_node_ids, g.dst_node_ids, g.node_interact_times
    neg = np.random.default_rng(1).integers(1, V1, E).astype(np.int64)
    exact = NeighborSampler.from_edges(src, dst, g.edge_ids, t, num_rows=V1)
    grow = NeighborSampler.growable(V1)
    init = torch.randn((V1, 172), device="cuda", generator=torch.Generator(device="cuda").manual_seed(2)) * 0.1
    init[0] = 0
    st = {"resident": ChangeLogStream(model(exact, T), src, dst, t, B, K, initial_pe=init.clone()),
          "host_exact": ChangeLogStream(model(exact, T), EMPTY, EMPTY, np.zeros(0), B, K, initial_pe=init.clone()),
          "host_ingest": ChangeLogStream(model(grow, T), EMPTY, EMPTY, np.zeros(0), B, K, initial_pe=init.clone()),
          "pestream_host": PEStream(model(exact, T), EMPTY, EMPTY, np.zeros(0), B, K, initial_pe=init.clone())}
    negd = torch.from_numpy(neg).cuda()
    q = lambda lo, hi: [src[lo:hi], dst[lo:hi], neg[lo:hi]]

    def run(arm, lo, hi):
        s = st[arm]
        if arm == "resident":
            s.run(lo // B, (hi - lo) // B, [s.src[lo:hi], s.dst[lo:hi], negd[lo:hi]])
            return None
        return s.run_host(src[lo:hi], dst[lo:hi], t[lo:hi], q(lo, hi), ingest=arm == "host_ingest")

    warm = (T + 5) * B
    chunk = (E - warm) // reps // B * B
    same = True
    res = {arm: run(arm, 0, warm) for arm in st}
    same &= bool(np.array_equal(res["host_exact"], res["host_ingest"]))
    ts = {arm: [] for arm in st}
    for r in range(reps):
        lo, hi = warm + r * chunk, warm + (r + 1) * chunk
        for arm in st:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res[arm] = run(arm, lo, hi)
            torch.cuda.synchronize()
            ts[arm].append(time.perf_counter() - t0)
        same &= bool(np.array_equal(res["host_exact"], res["host_ingest"]))
    for s in st.values():
        s.check_errors()
    same &= bool(torch.equal(st["host_exact"].cur, st["host_ingest"].cur))
    eps = {arm: [round(chunk / x) for x in v] for arm, v in ts.items()}
    med = {arm: float(np.median(v)) for arm, v in eps.items()}
    return {"shape": shape, "B": B, "T": T, "queries": 3, "edges_per_chunk": chunk, "warmup_edges": warm, "edges_per_s": eps,
            "median_ratio_over_resident": {arm: round(med[arm] / med["resident"], 4) for arm in eps},
            "run_host_bit_identical": same, "resident_table_equals_host": bool(torch.equal(st["resident"].cur, st["host_exact"].cur)),
            "regrows": grow.regrows}


def large(n_edges, n_online, B=2000, T=100, K=20, V=10_000_000):
    g = synth.make_graph("scaleout", seed=0, num_edges=n_edges, num_nodes=V)
    V1, E = g.num_nodes + 1, g.num_edges
    src, dst, eid, t = g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times
    p = E - n_online * B
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    grow = NeighborSampler.growable(V1, src[:p], dst[:p], eid[:p], t[:p])
    init = torch.randn((V1, 172), device="cuda", generator=torch.Generator(device="cuda").manual_seed(3)) * 0.1
    init[0] = 0
    st = ChangeLogStream(model(grow, T), EMPTY, EMPTY, np.zeros(0), B, K, initial_pe=init)
    del init
    neg = np.random.default_rng(4).integers(1, V1, E).astype(np.int64)
    q = lambda lo, hi: [src[lo:hi], dst[lo:hi], neg[lo:hi]]
    fill_hi = p + T * B  # the filling (masked) regime, one step at a time inside run_host
    st.run_host(src[p:fill_hi], dst[p:fill_hi], t[p:fill_hi], q(p, fill_hi), ingest=True)
    grow.reserve(src[fill_hi:], dst[fill_hi:])  # the timed call then needs no regrow
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    st.run_host(src[fill_hi:], dst[fill_hi:], t[fill_hi:], q(fill_hi, E), ingest=True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    st.check_errors()
    return {"nodes": V, "B": B, "T": T, "queries": 3, "stream_edges": E, "prefix_edges": p, "online_batches": n_online,
            "timed_edges": E - fill_hi, "edges_per_s": round((E - fill_hi) / dt), "history_bytes": st.history_bytes(),
            "dense_ring_bytes": V1 * T * 172 * 4, "csr_bytes": csr_bytes(grow), "csr_entries": grow.num_entries,
            "regrows": grow.regrows, "peak_device_bytes": int(torch.cuda.max_memory_allocated()), "edges_done": st.edges_done}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--large-edges", type=int, default=20_000_000, help="edges of the scale-out stream (prefix + online)")
    ap.add_argument("--large-batches", type=int, default=400, help="online batches of B = 2000 at the scale-out shape")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    assert _lib.load().lstep_device_ok() == 1, "not a compute-capability 10.x device"
    line = {"metric": "changelog_host"}
    line["arms"] = [arms("reddit", 200, a.reps), arms("flights", 2000, a.reps)]
    torch.cuda.empty_cache()
    line["scaleout_online"] = large(a.large_edges, a.large_batches)
    name, power = card()
    line.update(gpu=name, power_limit=power,
                notes="arms: host clock around calls that end synchronised, chunks alternated between the arms; resident = "
                      "ChangeLogStream.run (one C call per step), host_exact / host_ingest = ChangeLogStream.run_host on the "
                      "exact CSR / from an empty growable sampler with ingest=True (its time includes its capacity reservation), "
                      "pestream_host = PEStream.run_host (dense ring); scaleout_online: growable sampler from the stream's prefix, "
                      "the log filled over T online batches, then the remaining online batches timed in one run_host(ingest=True) "
                      "call after their room was reserved; peak_device_bytes = torch.cuda.max_memory_allocated over the whole "
                      "scale-out run (sampler, table, log, workspaces)")
    s = json.dumps(line)
    print(s, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    if not all(r["run_host_bit_identical"] for r in line["arms"]):
        sys.exit(1)


if __name__ == "__main__":
    main()
