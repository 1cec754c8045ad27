"""Size and speed of a change-log checkpoint at the scale-out shape (BASELINE config 5 on one GPU: 10 M nodes, E = 100 M,
B = 2000, T = 100, d = 172, a world-1 PeerRank), and the bit-identity of the resumed run:

    python profiles/checkpoint_io.py [--out FILE]

1. fill the window (T + 1 steps, so that the ring head has moved), 2. save, 3. load into a fresh rank, 4. run 10 more
steps on the original and on the resumed rank and compare outputs and tables bit for bit. Prints one JSON line: the shard
bytes; save and load time (host clock around work that ends in a device synchronise); the load split into reading and
validating the files, reading them into host memory, and the device part (upload + one append per window position) on the
in-memory history; the bit-identity; the card name and power limit read in the same run. The checkpoint goes to a
temporary directory (--dir: its parent) and is deleted on exit. The files were just written, so the reads are served
from the page cache."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from lstep_b200 import LSTEP, PeerRank, _lib, checkpoint, synth  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = (x.strip() for x in q.split(",", 1))
        return name, power
    except Exception as e:  # the name from the runtime, the power limit unknown
        return torch.cuda.get_device_name(), f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=10_000_000)
    ap.add_argument("--edges", type=int, default=100_000_000)
    ap.add_argument("--batch", type=int, default=2000)
    ap.add_argument("--T", type=int, default=100)
    ap.add_argument("--more", type=int, default=10, help="steps after the resume")
    ap.add_argument("--dir", default=None, help="parent of the temporary checkpoint directory")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    dev = torch.device("cuda", torch.cuda.current_device())
    assert _lib.load().lstep_device_ok() == 1, "not a compute-capability 10.x device"
    V, E, B, T, K, D = a.nodes, a.edges, a.batch, a.T, 20, 172
    src, dst, tt = synth.make_scaleout_device(V, E, dev, seed=0)
    torch.manual_seed(0)
    m = LSTEP(np.zeros((2, 172), dtype=np.float32), np.zeros((1, 172), dtype=np.float32), None, None, pe_dim=D, num_neighbors=K,
              time_feat_dim=100, num_fft_batches=T, device=dev).to(dev).eval()
    init = torch.randn((V + 1, D), device=dev, generator=torch.Generator(device=dev).manual_seed(1)) * 0.1
    init[0] = 0
    fill = T + 1
    e0 = int(E * 0.7) // B * B
    stop = min(E, e0 + (fill + a.more) * B)
    rk = PeerRank(m, 0, 1, src, dst, tt, V, B, K, init, start=e0, stop=stop)
    del init
    rk.connect_ipc()
    neg = torch.randint(1, V + 1, (stop,), device=dev, generator=torch.Generator(device=dev).manual_seed(2))

    def queries(r, b):
        lo, hi = r.batch(b)
        return [r.src[lo:hi], r.dst[lo:hi], r.src[lo:hi], neg[lo:hi]]

    for b in range(fill):
        rk.step(b, queries(rk, b))
    torch.cuda.synchronize()
    rk.check_errors()
    tmp = tempfile.mkdtemp(prefix="lstep_ckpt_", dir=a.dir)
    try:
        t0 = time.perf_counter()
        rk.save_checkpoint(tmp)
        t_save = time.perf_counter() - t0
        nbytes = sum(os.path.getsize(os.path.join(tmp, f)) for f in os.listdir(tmp))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rk2 = PeerRank(m, 0, 1, src, dst, tt, V, B, K, start=e0, stop=stop, sampler=rk.sampler, checkpoint=tmp)
        torch.cuda.synchronize()
        t_load = time.perf_counter() - t0
        t0 = time.perf_counter()
        hist = checkpoint.read(tmp)
        t_read = time.perf_counter() - t0
        t0 = time.perf_counter()
        hist = hist.in_memory()
        t_mem = time.perf_counter() - t0
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rk2.head, rk2.len = rk2.changelog.load(hist, rk2.cur)  # the same state again, from host memory: the device part alone
        torch.cuda.synchronize()
        t_dev = time.perf_counter() - t0
        n_ev = int(sum(int(sh["ev_off"][-1]) for sh in hist.shards))
        del hist
        rk2.connect_ipc()
        same = bool(torch.equal(rk2.cur, rk.cur)) and (rk2.len, rk2.batch_idx, rk2.steps_done) == (rk.len, rk.batch_idx, rk.steps_done)
        for b in range(fill, fill + a.more):
            o1 = rk.step(b, queries(rk, b))
            o2 = rk2.step(b, queries(rk2, b))
            same = same and bool(torch.equal(o1, o2))
        torch.cuda.synchronize()
        rk.check_errors()
        rk2.check_errors()
        same = same and bool(torch.equal(rk.cur, rk2.cur))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    name, power = card()
    line = {"metric": "changelog_checkpoint_io", "nodes": V, "edges": E, "batch": B, "T": T, "d": D, "world": 1,
            "saved_after_steps": fill, "len": rk2.len, "events": n_ev, "shard_bytes": nbytes, "save_s": round(t_save, 3),
            "load_s": round(t_load, 3), "load_read_validate_s": round(t_read, 3), "load_files_to_host_memory_s": round(t_mem, 3),
            "load_device_s": round(t_dev, 3), "resumed_steps": a.more, "bit_identical": same, "gpu": name, "power_limit": power,
            "notes": "save_s: device->host copies + .npy writes with fsync; load_s: PeerRank(checkpoint=dir) with the sampler reused, "
                     "ending in a device synchronise; load_device_s: the same load from a history already in host memory; reads "
                     "come from the page cache (the files were just written)"}
    s = json.dumps(line)
    print(s, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    rk.close()
    rk2.close()
    if not same:
        sys.exit(1)


if __name__ == "__main__":
    main()
