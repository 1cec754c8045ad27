"""How large |pe| gets over a full stream, against the range of phase B's 32.32 fixed-point sums:

    python profiles/pe_magnitude.py [--out FILE] [--every 100]

Runs the full Reddit-shaped (B = 200) and Flights-shaped (B = 2000) synth streams once each through PEStream.run (T = 100,
d = 172, K = 20, torch-initialised weights, initial table N(0, 0.1^2) with row 0 zero, three query sets). Every --every
steps it records max |pe| over the table, and the guard's quantity for the next batch: the largest |value| of that batch's
node rows in the current table against fixed_point_bound(n_ids, K) = 2^31 / (n_ids*K + 1) (the contributions phase B adds
are those rows after the DFT filter and phase A, which move a row by the filter's gain and by less than 1). It then reads
the device error flag (FloatingPointError if a step raised the range flag). Prints one JSON line with the card's name and
power limit read in the same run; --out also writes the full result with the trace."""
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


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = (x.strip() for x in q.split(",", 1))
        return name, power
    except Exception as e:  # the name from the runtime, the power limit unknown
        return torch.cuda.get_device_name(), f"unknown ({e})"


def stream(shape, B, every, T=100, K=20):
    g = synth.make_graph(shape, seed=0)
    V1, E = g.num_nodes + 1, g.num_edges
    s = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, num_rows=V1)
    torch.manual_seed(0)
    m = LSTEP(np.zeros((2, 172), np.float32), np.zeros((1, 172), np.float32), s, s, pe_dim=172, num_neighbors=K, time_feat_dim=100,
              num_fft_batches=T, device="cuda").to("cuda").eval()
    init = torch.randn((V1, 172), device="cuda", generator=torch.Generator(device="cuda").manual_seed(2)) * 0.1
    init[0] = 0
    st = PEStream(m, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, initial_pe=init)
    neg = torch.from_numpy(np.random.default_rng(1).integers(1, V1, E).astype(np.int64)).cuda()
    rows = []
    t0 = time.perf_counter()
    b = 0
    while b < st.num_batches:
        n = min(every, st.num_batches - b)
        lo, hi = st.batch_lo[b], E if b + n >= st.num_batches else st.batch_lo[b + n]
        st.run(b, n, [st.src[lo:hi], st.dst[lo:hi], neg[lo:hi]])
        b += n
        cur = st.cur
        rec = {"steps": b, "max_abs_pe": float(cur.abs().max()), "rms_pe": float(cur.pow(2).mean().sqrt())}
        if b < st.num_batches:
            ids = st.ids[st.ids_off[b]:st.ids_off[b + 1]]
            bound = _lib.fixed_point_bound(len(ids), K)
            x = float(cur[ids].abs().max())
            rec.update({"next_n_ids": int(len(ids)), "next_max_abs_contribution": x, "bound": bound, "ratio": x / bound})
        rows.append(rec)
    torch.cuda.synchronize()
    st.check_errors()
    ratios = [r["ratio"] for r in rows if "ratio" in r]
    return {"shape": shape, "B": B, "K": K, "edges": E, "steps": st.num_batches, "seconds": time.perf_counter() - t0,
            "final_max_abs_pe": rows[-1]["max_abs_pe"], "max_ratio": max(ratios), "min_bound": min(r["bound"] for r in rows if "bound" in r),
            "every": every, "trace": rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the full result (with the per-100-step trace) to this file")
    ap.add_argument("--every", type=int, default=100)
    a = ap.parse_args()
    name, power = card()
    res = {"card": name, "power_limit": power, "runs": [stream("reddit", 200, a.every), stream("flights", 2000, a.every)]}
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f)
    print(json.dumps({k: v for k, v in res.items() if k != "runs"} | {"runs": [{k: v for k, v in r.items() if k != "trace"} for r in res["runs"]]}))


if __name__ == "__main__":
    main()
