#!/usr/bin/env python
"""bench.py — temporal edges/s through the L-STEP positional-encoding hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload reddit|wikipedia|enron|flights]
    python bench.py --impl reference ...        # the CPU oracle port of the reference path
    python bench.py --dump-outputs DIR ...      # also write the last timed step's outputs to DIR/*.npy (see dump_outputs)

A step is one pass of the module-boundary PE path over one batch of the synthetic edge stream
(SURVEY §8(d)): DFT filter on the batch nodes (a3), C=4 neighbourhood aggregates (a6: pos src,
pos dst, neg src, neg dst — the eval loop's four calls), update_pe (a7+a8), plus the history
bookkeeping the streaming API does instead of the loops' clone/cat (one table copy in, one out).

    value   edges/s with the edge stream, negatives and PE history resident in HBM: the K timed steps are ONE native call
            (PEStream.run -> lstep_pe_steps) queued behind a short spin kernel, so the region is device-bound at any K
    e2e     edges/s through PEStream.run_host(): numpy batches in (pinned H2D), per-query row sums out (D2H)
    roofline  the step's dominant kernel (largest median duration of its six launches, CUDA events around each kernel of the
              real step on live data): algorithmic bytes (or flops) / duration vs the measured peak
    cpu_baseline  the UNMODIFIED reference (oracle/_ref, torch CPU) on this box's host cores, bounded sample of the same
              workload with the same weights; the numpy oracle port when oracle/_ref is absent

One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from lstep_b200 import synth  # noqa: E402

WORKLOADS = {  # name -> (batch size, K)  (BASELINE.json configs; K=20 is the reference default)
    "enron": (200, 20), "wikipedia": (200, 20), "reddit": (200, 20), "flights": (2000, 20), "tiny_bip": (50, 20),
}
D, T_DIM, T_HIST, C_CALLS = 172, 100, 100, 4
ZIPF_S = 0.8  # endpoint skew of the synthetic stream (--zipf; DESIGN §10: SURVEY §8(d) names 1.2, the hub-heavy regime)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def clk_ghz(clk):
    try:
        return float(clk["sm_mhz"]) * 1e-3
    except Exception:
        return 1.965


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# algorithmic bytes (SURVEY §8(d)); N, M measured per batch
def bytes_model(B, N, M, K, d=D, t=T_DIM, T=T_HIST, C=C_CALLS, V1=0):
    F = 4 * d * (N * T + T + N)
    S = (C * B + N) * (16 + 16 * K)
    P = C * B * 4 * d * (K + 2)
    UA = 4 * d * (2 * B + 2 * N) + 24 * B
    UB = 4 * d * (N + 2 * M) + 8 * (d + t) * M + 12 * N * K
    W = 4 * (2 * (d + t) * d + 4 * d * d + 6 * d)
    H = 4 * d * 2 * V1
    return dict(F=F, S=S, P=P, UA=UA, UB=UB, W=W, bytes_path=F + S + P + UA + UB + W, H=H)


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index=0, period=0.05):
        super().__init__(daemon=True)
        self.period, self.index = period, index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            self.nv = None
            log("nvml unavailable:", e)

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
def make_params_model(graph, sampler, device):
    """LSTEP drop-in with random-init weights of the reference architecture (no checkpoints offline)."""
    import torch
    from lstep_b200 import LSTEP
    torch.manual_seed(0)
    node_feats = np.zeros((graph.num_nodes + 1, 172), dtype=np.float32)
    edge_feats = np.zeros((1, 172), dtype=np.float32)  # the feature branch is not on the PE path
    m = LSTEP(node_feats, edge_feats, sampler, sampler, pe_dim=D, num_neighbors=20, time_feat_dim=T_DIM, num_fft_batches=T_HIST,
              device=device)
    return m.to(device).eval()


def workload_config(workload, g, B, K, world=1):
    """The `config` both arms print (same string for the CUDA arm and the reference arm: the driver compares them)."""
    skew = "" if ZIPF_S == 0.8 else f", endpoint skew zipf s={ZIPF_S}"
    return {"workload": f"{workload}-shaped synthetic temporal graph, V={g.num_nodes}, E={g.num_edges}, B={B}, K={K}, "
                        f"T={T_HIST}, d={D}, t={T_DIM}, C={C_CALLS} neighbourhood calls/batch (eval loop){skew}",
            "parallelism": "single GPU" if world == 1 else f"{world} independent replicas (path does not shard at this size)",
            "l2_policy": f"inputs larger than L2: PE history {(g.num_nodes + 1) * T_HIST * D * 4 / 1e6:.0f} MB, a different node set is read each step"}


def headline_setup(workload, seed, dev):
    """The state the headline workload starts from: the seeded synthetic stream of `workload`, the device sampler over it,
    the drop-in with seeded weights, a PEStream over the evaluation split (the last 30 % of the stream, like val+test; nb
    full batches, wrapped around when more steps are asked for) and the negatives. `queries(b)`: the four query sets of
    batch b (the eval loop's calls: positive source, positive destination, negative source, negative destination)."""
    import types
    import torch
    from lstep_b200 import NeighborSampler, PEStream
    B, K = WORKLOADS[workload]
    g = synth.make_graph(workload, seed=seed, zipf_s=ZIPF_S)
    V1 = g.num_nodes + 1
    t0 = time.time()
    sampler = NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent", num_rows=V1)
    torch.cuda.synchronize()
    t_csr = time.time() - t0
    model = make_params_model(g, sampler, dev)
    init = torch.from_numpy(synth.make_initial_pe(g.num_nodes, D, seed=1)).to(dev)
    e0 = int(g.num_edges * 0.7) // B * B
    stream = PEStream(model, g.src_node_ids, g.dst_node_ids, g.node_interact_times, B, K, initial_pe=init, start=e0)
    nb = stream.num_batches
    if stream.batch_lo[-1] + B > g.num_edges:
        nb -= 1  # full batches only (a ragged tail would change the per-step work)
    rng = np.random.default_rng(2)
    neg_all = rng.choice(np.unique(g.dst_node_ids), size=g.num_edges - e0).astype(np.int64)
    neg_dev = torch.from_numpy(neg_all).to(dev)

    def queries(b):
        lo, hi, _, _ = stream.batch_arrays(b)
        return [stream.src[lo:hi], stream.dst[lo:hi], stream.src[lo:hi], neg_dev[lo - e0:hi - e0]]

    return types.SimpleNamespace(g=g, sampler=sampler, model=model, stream=stream, nb=nb, e0=e0, neg_all=neg_all, neg_dev=neg_dev,
                                 queries=queries, t_csr=t_csr)


def run_ours(args, rank, world, own_pg=True):
    """The headline workload on every rank (N > 1: independent replicas, weak scaling — the path does not shard at
    this size). Returns the result line on rank 0; emits it when it owns the process group."""
    import torch
    import torch.distributed as dist
    from lstep_b200 import _lib

    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 and own_pg:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    assert lib.lstep_device_ok() == 1
    B, K = WORKLOADS[args.workload]
    h = headline_setup(args.workload, rank, dev)  # replicas: each rank its own stream of the same shape
    g, sampler, model, stream, nb, e0, neg_all, neg_dev, queries = (h.g, h.sampler, h.model, h.stream, h.nb, h.e0, h.neg_all,
                                                                    h.neg_dev, h.queries)
    V1 = g.num_nodes + 1

    def run_steps(first, n):
        """n consecutive steps starting at step number `first` (wrapping over the evaluation split): one native call per
        contiguous run of batches. Returns the neighbourhood PEs of the last step [C, B, d]."""
        done, last = 0, None
        while done < n:
            b0 = (first + done) % nb
            cnt = min(n - done, nb - b0)
            lo0 = stream.batch_lo[b0]
            del last  # free the previous call's output before the next call allocates its own
            last = stream.run(b0, cnt, [stream.src[lo0:], stream.dst[lo0:], stream.src[lo0:], neg_dev[lo0 - e0:]])
            done += cnt
        return last

    outs = torch.empty((C_CALLS, B, D), dtype=torch.float32, device=dev)
    W, Ksteps = args.warmup, args.steps
    W = max(W, 3)
    step_no = 0
    # the measured regime is the steady state with a FULL history (T steps per node: the DFT filter reads all of
    # them); if fewer warm-up steps were asked for, the ring is filled first (untimed, reported in config)
    fill = max(0, T_HIST + 10 - W)
    for _ in range(min(fill + W, T_HIST + 2)):  # per-step calls while the ring fills (the filter changes every step)
        stream.step(step_no % nb, queries(step_no % nb), outs)
        step_no += 1
    rest = fill + W - step_no
    if rest > 0:
        run_steps(step_no, rest)
        step_no += rest
    torch.cuda.synchronize()
    sampler.check_errors()
    if world > 1:
        dist.barrier()
    clocks = ClockSampler(local)
    clocks.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    Ns, edges = [], 0
    for i in range(Ksteps):
        lo, hi, io, ie = stream.batch_arrays((step_no + i) % nb)
        edges += hi - lo
        Ns.append(ie - io)
    torch.cuda.synchronize()
    # a short spin keeps the GPU busy while the host enqueues the first steps: the clock starts when the spin ends, with
    # launches already queued behind it, so the timed region is the device's own chain of kernels at any K
    torch.cuda._sleep(int(1.0e6))
    ev0.record()
    last_out = run_steps(step_no, Ksteps)
    ev1.record()
    torch.cuda.synchronize()
    step_no += Ksteps
    ms_total = ev0.elapsed_time(ev1)
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, stream, last_out)
    t_max = torch.tensor([ms_total], device=dev)
    edges_t = torch.tensor([float(edges)], device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(t_max, op=dist.ReduceOp.MAX)
        dist.all_reduce(edges_t, op=dist.ReduceOp.SUM)
    ms_total_max = float(t_max.item())
    value = float(edges_t.item()) / (ms_total_max * 1e-3)
    # the same steps through one Python call per step (what a loop calling PEStream.step pays), for reference
    n_py = min(Ksteps, 200)
    torch.cuda.synchronize()
    t_py = time.perf_counter()
    for _ in range(n_py):
        stream.step(step_no % nb, queries(step_no % nb), outs)
        step_no += 1
    torch.cuda.synchronize()
    py_ms = (time.perf_counter() - t_py) * 1e3 / n_py

    # ---- per-kernel durations of the step's OWN six launches (CUDA events around every kernel of the real step)
    n_prof = max(20, min(Ksteps, 100))
    kern, M_meas = profile_pass(stream, sampler, queries, step_no, nb, n_prof, K, lib, outs)
    step_no += n_prof
    N_mean = float(np.mean(Ns))
    M_mean = float(np.mean(M_meas)) if M_meas else 0.0
    bm = bytes_model(B, N_mean, M_mean, K, V1=V1)
    hbm_peak, peak_src = peaks()
    roof_all = kernel_rooflines(kern, bm, B, N_mean, M_mean, K, V1, hbm_peak, clk)
    dom = max(roof_all, key=lambda k: roof_all[k]["ms_per_launch"])
    roof = dict(kernel=dom, peak_source=peak_src, **roof_all[dom])
    serial_ms = sum(v["ms_per_launch"] for v in roof_all.values())
    path_gbs = bm["bytes_path"] / (ms_total_max / Ksteps * 1e-3) / 1e9

    # ---- end to end through the host-facing API (numpy in, result out), same stream / model
    e2e = None
    if rank == 0 or world > 1:
        e2e = e2e_pass(stream, g, e0, neg_all, step_no, nb, min(max(Ksteps, 100), 300), B, world, dev)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:  # reported at N = 1 only
        cpu = cpu_baseline(args.workload, B, K, args.cpu_batches)

    if rank == 0:
        cfg = workload_config(args.workload, g, B, K, world)
        info = {"timed_region": "K steps in one native call (PEStream.run -> lstep_pe_steps) queued behind a spin kernel; CUDA events on the launch stream",
                "N_mean": N_mean, "M_mean": M_mean, "csr_build_s": h.t_csr, "history_fill_steps_before_warmup": fill}
        out = {
            "metric": "temporal edges/sec through PE update+aggregation; % HBM roofline", "value": value, "unit": "edges/s",
            "n_gpus": world, "steps": Ksteps, "warmup": W, "ms_per_step": ms_total_max / Ksteps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg,
            "run_info": info,
            "clocks": clk,
            "e2e": e2e,
            "gpu_launches": int(6 * Ksteps),
            "roofline": roof,
            "roofline_kernels": roof_all,
            "path_roofline": {"bytes_path_per_step": bm["bytes_path"], "bytes_breakdown": {k: bm[k] for k in ("F", "S", "P", "UA", "UB", "W", "H")},
                              "achieved_GBps": path_gbs, "peak_GBps": hbm_peak, "frac": path_gbs / hbm_peak, "peak_source": peak_src,
                              "with_H": {"bytes_step": bm["bytes_path"] + bm["H"],
                                         "frac": (bm["bytes_path"] + bm["H"]) / (ms_total_max / Ksteps * 1e-3) / 1e9 / hbm_peak}},
            "step_ms": {"device_chain": ms_total_max / Ksteps, "python_call_per_step": py_ms, "sum_of_serialised_kernels": serial_ms,
                        "note": "device_chain < sum_of_serialised_kernels: programmatic dependent launch overlaps each kernel's "
                                "pre-wait work with its predecessor"},
            "cpu_baseline": cpu,
        }
        if own_pg:
            emit(out)
    else:
        out = None
    if world > 1 and own_pg:
        dist.destroy_process_group()
    del stream, model, sampler
    torch.cuda.empty_cache()
    return out


DUMP_HISTORY_ROWS = 256  # node rows of the PE history in the dump: all T steps of each (the whole history is 756 MB at Reddit size)
DUMP_MAX_BYTES = 64_000_000


def dump_outputs(path, stream, nbr_pe):
    """Writes what the timed path computed in its last step, as a caller of PEStream.run receives it, to path/<name>.npy
    (float32): the step's neighbourhood PEs [C, B, d] (run's return value), the updated PE table [V1, d], and the PE history
    [rows, T, d] (oldest step first) of a fixed sample of node rows (seed 0). The inputs are seeded, so two builds run with
    the same arguments can be compared output for output."""
    import torch
    rows = np.sort(np.random.default_rng(0).choice(stream.V1, size=min(DUMP_HISTORY_ROWS, stream.V1), replace=False))
    arrays = {"neighborhood_pe": nbr_pe, "pe_table": stream.cur,
              "pe_history_sample": stream.export_history()[torch.from_numpy(rows).to(stream.dev)]}
    arrays = {k: v.float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES} byte budget")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a)
    log(f"dumped {', '.join(f'{k} {list(a.shape)}' for k, a in arrays.items())} ({total / 1e6:.1f} MB) -> {path}")


def run_sharded(args, rank, world, own_pg=True):
    """BASELINE config 5: the scale-out graph (10 M nodes) on a PEER GROUP (l-step_b200/peer.py, csrc/peer.cu): every rank keeps a
    replica of the current table and of the temporal CSR and owns the nodes v % N == rank — their PE history (change log: base
    rows + the rows every step changed, 13 GB instead of 688 GB at T = 100) and 1/N of every phase of the step (DFT filter, a6
    query rows, update_pe phase A and phase B). Owners store the rows they change into the other replicas through NVLink peer
    pointers (CUDA IPC); two flag barriers per step in peer memory; no NCCL call and no host synchronisation on the step's
    path. The batch is replicated, so the work per rank shrinks with N ("scaling": "strong"). The timed region is ONE native
    call for all K steps (lstep_pe_steps_peer) queued behind a spin kernel."""
    import torch
    import torch.distributed as dist
    from lstep_b200 import LSTEP, PeerRank, _lib

    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if own_pg and world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    assert lib.lstep_device_ok() == 1
    B, K = args.scaleout_batch, 20
    T = args.scaleout_T if args.scaleout_T else T_HIST
    V, E = args.scaleout_nodes, args.scaleout_edges
    t0 = time.time()
    src, dst, tt = synth.make_scaleout_device(V, E, dev, seed=0)
    torch.cuda.synchronize()
    t_gen = time.time() - t0
    if world > 1:  # every rank must hold the same stream
        # exact integer checksums (a floating-point sum of 1e8 doubles may be reduced in another order on another device)
        ck = torch.stack([src.sum(), dst.sum(), tt.view(torch.int64).sum(), src[::1009].sum() ^ dst[::1013].sum()])
        lo_, hi_ = ck.clone(), ck.clone()
        dist.all_reduce(lo_, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi_, op=dist.ReduceOp.MAX)
        assert torch.equal(lo_, hi_), "ranks generated different edge streams"
    torch.manual_seed(0)
    m = LSTEP(np.zeros((2, 172), dtype=np.float32), np.zeros((1, 172), dtype=np.float32), None, None, pe_dim=D, num_neighbors=20,
              time_feat_dim=T_DIM, num_fft_batches=T, device=dev).to(dev).eval()
    gen = torch.Generator(device=dev).manual_seed(1)
    init = torch.randn((V + 1, D), device=dev, generator=gen) * 0.1
    init[0] = 0
    W, Ksteps = max(args.warmup, 3), args.steps
    if not own_pg:  # riding along with the headline run: a bounded sample
        W, Ksteps = min(W, 10), min(Ksteps, 100)
    W = max(W, T + 5)  # full history before the clock starts
    n_e2e = min(Ksteps, 50)
    e0 = int(E * 0.7) // B * B
    stop = min(E, e0 + (W + Ksteps + n_e2e + 12) * B)
    t0 = time.time()
    rk = PeerRank(m, rank, world, src, dst, tt, V, B, K, init, start=e0, stop=stop)
    del init
    rk.connect_ipc()
    torch.cuda.synchronize()
    t_setup = time.time() - t0
    nb = rk.num_batches
    # negative destinations, indexed by global edge position (only [e0, stop) is read)
    neg_all = torch.zeros(stop, dtype=torch.int64, device=dev)
    neg_all[e0:] = torch.randint(1, V + 1, (stop - e0,), device=dev, generator=torch.Generator(device=dev).manual_seed(2))
    q_arrays = [rk.src, rk.dst, rk.src, neg_all]

    def queries(b):
        lo, hi = rk.batch(b)
        return [rk.src[lo:hi], rk.dst[lo:hi], rk.src[lo:hi], neg_all[lo:hi]]

    step_no = 0
    out = torch.empty((C_CALLS, B // world + 1, D), dtype=torch.float32, device=dev)
    for _ in range(T + 2):  # the history fills step by step (the filter changes with its length)
        rk.step(step_no, queries(step_no))
        step_no += 1
    rk.run(step_no, W - (T + 2), q_arrays, out=out)  # the rest of the warm-up through the native multi-step call
    step_no += W - (T + 2)
    torch.cuda.synchronize()
    rk.check_errors()
    if world > 1:
        dist.barrier()
    clocks = ClockSampler(local)
    clocks.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(int(2.0e6))  # the host queues the first steps behind a spin: the region is device-bound
    ev0.record()
    rk.run(step_no, Ksteps, q_arrays, out=out)
    ev1.record()
    torch.cuda.synchronize()
    edges = int(rk.n_edges[step_no:step_no + Ksteps].sum())
    step_no += Ksteps
    ms = ev0.elapsed_time(ev1)
    clk = clocks.stop()
    rk.check_errors()
    tm = torch.tensor([ms], device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    ms_max = float(tm.item())
    value = edges / (ms_max * 1e-3)  # the batch is replicated: edges of the job, not per rank
    # end to end: the negatives of every step come from host memory and this rank's per-query row sums go back to it
    neg_host = neg_all[e0:].cpu().numpy()
    d2h = h2d = 0
    e_edges = 0
    if world > 1:
        dist.barrier()
    t_wall = time.perf_counter()
    ev0.record()
    for _ in range(n_e2e):
        b = step_no
        lo, hi = rk.batch(b)
        negs = torch.from_numpy(neg_host[lo - e0:hi - e0]).to(dev, non_blocking=True)
        h2d += negs.numel() * 8
        o = rk.step(b, [rk.src[lo:hi], rk.dst[lo:hi], rk.src[lo:hi], negs])
        r = o.sum(dim=2).cpu()
        d2h += r.numel() * 4
        e_edges += hi - lo
        step_no += 1
    ev1.record()
    torch.cuda.synchronize()
    rk.check_errors()
    tm = torch.tensor([max(ev0.elapsed_time(ev1), (time.perf_counter() - t_wall) * 1e3)], device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    e2e = {"value": e_edges / (float(tm.item()) * 1e-3), "unit": "edges/s", "h2d_bytes_per_step": h2d / n_e2e, "d2h_bytes_per_step": d2h / n_e2e,
           "steps": n_e2e, "api": "PeerRank.step per rank (one call per batch): the step's negative ids from host memory, this rank's "
                                  "per-query row sums back to the host (a synchronising read every step)"}
    # per-kernel times of this rank's share (events between kernels; medians over 8 steps), waits = time lost to the other ranks
    import ctypes
    names = ["filter+signal1", "wait1", "gather_ab", "mlp_pair", "bcast+signal2", "wait2", "push", "mlp_B", "append"]
    _lib.check(lib.lstep_step_profile(1), "profile on")
    rows_ms = []
    try:
        for _ in range(8):
            b = step_no
            rk.step(b, queries(b))
            step_no += 1
            ms9 = (ctypes.c_float * 9)()
            _lib.check(lib.lstep_step_profile_read_all(ms9, 9), "profile read")
            rows_ms.append(list(ms9))
    finally:
        lib.lstep_step_profile(0)
    med = np.median(np.asarray(rows_ms), axis=0)
    per_kernel = {n: float(v) for n, v in zip(names, med)}
    all_pk = [per_kernel]
    if world > 1:
        all_pk = [None] * world
        dist.all_gather_object(all_pk, per_kernel)
    # replica check: every rank's table must equal rank 0's (checksums of a strided sample + of the rows the last step changed)
    rk.barrier()
    torch.cuda.synchronize()
    ck = torch.stack([rk.cur[::997].double().sum(), rk.cur[::997].double().abs().sum(), rk.cur[rk.ids[-4000:]].double().sum()])
    lo_, hi_ = ck.clone(), ck.clone()
    if world > 1:
        dist.all_reduce(lo_, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi_, op=dist.ReduceOp.MAX)
    replicas_equal = bool(torch.equal(lo_, hi_))
    # rows a step changes (peer stores): owned filtered rows + owned final rows go to N-1 replicas, phase-A rows to N buffers
    n_ids_mean = float(np.diff(rk.ids_off).mean())
    free_b, total_b = torch.cuda.mem_get_info(dev)
    if rank == 0:
        out_d = {
            "metric": "temporal edges/sec through PE update+aggregation; % HBM roofline", "value": value, "unit": "edges/s",
            "n_gpus": world, "steps": Ksteps, "warmup": W, "ms_per_step": ms_max / Ksteps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"scale-out synthetic temporal graph, V={V}, E={E} (Zipf 0.8 endpoints, generated on the device), B={B}, K={K}, "
                                   f"T={T}, d={D}, t={T_DIM}, C={C_CALLS}",
                       "parallelism": f"peer group of {world} GPU(s): node v is owned by rank v mod N (its PE history as a change log, 1/N of the DFT "
                                      "filter, of the a6 query rows, of update_pe phase A and phase B); current table + temporal CSR replicated, "
                                      "owners store changed rows into the other replicas over NVLink peer pointers (CUDA IPC), two flag barriers "
                                      "per step in peer memory; no NCCL call on the step's path",
                       "l2_policy": f"inputs larger than L2: history {rk.history_bytes() / 1e9:.1f} GB per rank (dense [V1, T, d] would be "
                                    f"{(V + 1) * T * D * 4 / 1e9:.0f} GB in total), table {(V + 1) * D * 4 / 1e9:.1f} GB, CSR {2 * E * 16 / 1e9:.1f} GB"},
            "run_info": {"graph_gen_s": t_gen, "setup_s": t_setup, "hbm_used_GB": (total_b - free_b) / 1e9, "history": "changelog", "T": T,
                         "timed_region": "K steps in one native call (PeerRank.run -> lstep_pe_steps_peer) queued behind a spin kernel; CUDA events, max over ranks",
                         "batch_nodes_mean": n_ids_mean, "replicas_equal_after_run": replicas_equal,
                         "per_kernel_ms_median_by_rank": all_pk},
            "clocks": clk, "e2e": e2e,
            "gpu_launches": int(Ksteps * 10 * world),
            "roofline": None, "cpu_baseline": None,
        }
        if own_pg:
            emit(out_d)
    else:
        out_d = None
    rk.close()
    if own_pg and world > 1:
        dist.destroy_process_group()
    del rk, src, dst, tt, neg_all
    torch.cuda.empty_cache()
    return out_d


KERNELS = ["dft_filter", "gather_ab (a6 lookup+aggregate || a7 edge aggregate)", "pe_mlp pair (neighbourhood MLP || phase-A MLP)",
           "phaseB_push", "pe_mlp (phase B)", "ring_append"]


def profile_pass(stream, sampler, queries, step_no, nb, n, K, lib, outs):
    """Durations of the six kernels of the REAL step on live data: lstep_step_profile(1) makes the step record a CUDA
    event on its launch stream before its first kernel and after each kernel (csrc/step.cu); an event between two
    kernels also removes their programmatic overlap, so these are the kernels run back to back. Medians over n steps
    after 3 warm steps. Also measures M (distinct sampled neighbours per batch) for the byte model."""
    import ctypes
    import torch
    from lstep_b200 import _lib
    ms = (ctypes.c_float * 6)()
    rows = []
    _lib.check(lib.lstep_step_profile(1), "profile on")
    try:
        for i in range(n + 3):
            b = (step_no + i) % nb
            stream.step(b, queries(b), outs)
            _lib.check(lib.lstep_step_profile_read(ms), "profile read")
            if i >= 3:
                rows.append([float(x) for x in ms])
    finally:
        lib.lstep_step_profile(0)
    arr = np.array(rows)
    kern = {name: {"ms": float(np.median(arr[:, k])), "ms_min": float(arr[:, k].min()), "ms_p90": float(np.quantile(arr[:, k], 0.9)),
                   "launches_per_step": 1} for k, name in enumerate(KERNELS)}
    M_meas = []
    for i in range(min(n, 20)):
        b = (step_no + i) % nb
        lo, hi, io, ie = stream.batch_arrays(b)
        nv = min(ie - io, hi - lo)
        nbr, _ = sampler.sample_device(stream.ids[io:ie], stream.t[lo:hi], ie - io, nv, K)
        M_meas.append(int(torch.unique(nbr).numel()))
    return kern, M_meas


def kernel_rooflines(kern, bm, B, N, M, K, V1, hbm_peak, clk, d=D, t=T_DIM, C=C_CALLS):
    """Algorithmic bytes / flops of each of the step's six launches (SURVEY §8(d) terms split by kernel; every distinct
    tensor a kernel touches counted once) against its measured duration. Memory kernels: bound 'hbm' vs the measured copy
    peak. The two MLP launches are fp32 FMA work (1e-5 parity rules out single-pass TF32 / BF16): bound 'fp32_fma' vs
    148 SMs x 128 FMA/clk x SM clock."""
    CB, W = C * B, bm["W"]
    try:
        with open(os.path.join(ROOT, "profiles", "r02_ncu_full_kernels.json")) as f:
            ncu_full = {e["kernel"]: e for e in json.load(f) if "kernel" in e}
    except Exception:
        ncu_full = {}
    alg = {
        KERNELS[0]: bm["F"],
        KERNELS[1]: CB * (16 + 16 * K) + CB * 4 * d * K + CB * 4 * (d + t) + 4 * d * 2 * B + 24 * B + 4 * (d + t) * N,
        KERNELS[2]: (CB + N) * (4 * (d + t) + 8 * d) + W,
        KERNELS[3]: N * (16 + 16 * K) + 8 * d * N + 8 * (d + t) * M + 12 * N * K,
        KERNELS[4]: M * (8 * (d + t) + 12 * d) + W / 2,
        KERNELS[5]: bm["H"],
    }
    flops = {KERNELS[2]: 2.0 * (CB + N) * ((d + t) * d + 2 * d * d), KERNELS[4]: 2.0 * M * ((d + t) * d + d * d)}
    fma_peak = 148 * 128 * 2 * clk_ghz(clk)  # GFLOP/s * 1e-3 = TFLOP/s
    out = {}
    for name in KERNELS:
        ms = kern[name]["ms"]
        gbs = alg[name] / (ms * 1e-3) / 1e9
        e = {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
             "traffic": (ncu_full.get(name) or {}).get("dram_bytes_per_launch"), "algorithmic_bytes_per_launch": alg[name],
             "ms_per_launch": ms, "ms_min": kern[name]["ms_min"], "ms_p90": kern[name]["ms_p90"]}
        if name in flops:
            tf = flops[name] / (ms * 1e-3) / 1e12
            e.update({"bound": "fp32_fma", "achieved": tf, "peak": fma_peak * 1e-3, "unit": "TFLOP/s", "frac": tf / (fma_peak * 1e-3),
                      "flops_per_launch": flops[name], "hbm_GBps": gbs, "hbm_frac": gbs / hbm_peak})
        out[name] = e
    return out


def e2e_pass(stream, g, e0, neg_all, step_no, nb, n, B, world, dev):
    """End to end through the host-facing API: every step hands numpy arrays (the batch's endpoints and times,
    the four query id sets) to PEStream.step_host_async — pinned staging + one H2D copy + the step's kernels +
    the D2H copy of the per-query row sums, all inside the timed region — and reads the PREVIOUS step's result
    (double-buffered: the read never waits on the step just enqueued; the last result is read before the clock stops)."""
    import torch
    import torch.distributed as dist
    m = stream.model

    def batch(i):
        b = (step_no + i) % nb
        lo, hi, _, _ = stream.batch_arrays(b)
        return (g.src_node_ids[lo:hi], g.dst_node_ids[lo:hi], g.node_interact_times[lo:hi],
                [g.src_node_ids[lo:hi], g.dst_node_ids[lo:hi], g.src_node_ids[lo:hi], neg_all[lo - e0:hi - e0]]), hi - lo

    for i in range(3):  # warm the staging path
        a, _ = batch(i)
        stream.step_host(*a)
    step_no += 3
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    h0 = m.h2d_bytes
    d2h = 0
    edges = 0
    pending = None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall = time.perf_counter()
    ev0.record()
    for i in range(n):
        a, ne = batch(i)
        tk = stream.step_host_async(*a)
        if pending is not None:
            d2h += stream.result(pending).nbytes
        pending = tk
        edges += ne
    d2h += stream.result(pending).nbytes
    ev1.record()
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t_wall) * 1e3
    ms = max(ev0.elapsed_time(ev1), wall_ms)  # device clock and host clock agree when the pipeline is full; take the slower
    h2d = m.h2d_bytes - h0
    per_step_ms = ms / n
    # the same workload through ONE call for the whole run of batches (PEStream.run_host -> lstep_pe_steps_host: the
    # per-batch loop, every step's copy-in and result read included, runs natively): this is the e2e headline
    n = min(n, nb)  # (a short evaluation split: one pass over it)
    b0 = (step_no + n) % nb
    if b0 + n > nb:
        b0 = 0
    lo0 = stream.batch_arrays(b0)[0]
    hi0 = stream.batch_arrays(b0 + n - 1)[1]
    sl = slice(lo0, hi0)
    qs_run = [g.src_node_ids[sl], g.dst_node_ids[sl], g.src_node_ids[sl], neg_all[lo0 - e0:hi0 - e0]]
    stream.run_host(g.src_node_ids[lo0:lo0 + 3 * B], g.dst_node_ids[lo0:lo0 + 3 * B], g.node_interact_times[lo0:lo0 + 3 * B],
                    [q[:3 * B] for q in qs_run])  # warm
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    h1 = m.h2d_bytes
    t_run = time.perf_counter()
    ev0.record()
    res = stream.run_host(g.src_node_ids[sl], g.dst_node_ids[sl], g.node_interact_times[sl], qs_run)
    ev1.record()
    torch.cuda.synchronize()
    ms = max(ev0.elapsed_time(ev1), (time.perf_counter() - t_run) * 1e3)
    edges = hi0 - lo0
    h2d = m.h2d_bytes - h1
    d2h = res.nbytes
    # every result read right after its own step (no overlap of host and device), for reference
    n_sync = min(n, 100)
    t_sync = time.perf_counter()
    for i in range(n_sync):
        a, ne = batch(n + i)
        stream.step_host(*a)
    sync_ms = (time.perf_counter() - t_sync) * 1e3 / n_sync
    tm = torch.tensor([ms], device=dev)
    et = torch.tensor([float(edges)], device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(et, op=dist.ReduceOp.SUM)
    return {"value": float(et.item()) / (float(tm.item()) * 1e-3), "unit": "edges/s", "h2d_bytes_per_step": h2d / n,
            "d2h_bytes_per_step": d2h / n, "steps": n, "ms_per_step": float(tm.item()) / n,
            "per_step_call_ms_per_step": per_step_ms, "per_step_call_value": B / (per_step_ms * 1e-3),
            "unpipelined_ms_per_step": sync_ms, "unpipelined_value": B / (sync_ms * 1e-3),
            "api": "PEStream.run_host: one native call for the run of batches; per batch: numpy slices -> pinned slot -> copy-in kernel "
                   "reading the pinned slot (side stream) -> the step's 6 kernels -> per-query row sums written to the pinned result "
                   "slot -> read into the caller's array one step behind. per_step_call_* = the same through one Python call per "
                   "batch (step_host_async + result)"}


# ------------------------------------------------------------------------------------------------
def oracle_setup(workload, B, K, n_batches, seed=0):
    """(fallback when oracle/_ref is absent) bounded sample of the workload for the numpy port: the first
    max(40 000, 4 x the edges of n_batches + 4 batches) edges of the stream, the whole stream at most, build the adjacency
    (its python loops dominate the set-up); the timed batches come from the sample's tail (oracle_batch_starts)."""
    from oracle import lstep_oracle as orc
    full = synth.SHAPES[workload]["num_edges"]
    n_edges = min(full, max(40_000, (n_batches + 4) * B * 4))
    g = synth.make_graph(workload, seed=seed, num_edges=n_edges, zipf_s=ZIPF_S)
    adj = orc.build_adjacency(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times)
    p = orc.init_params(D, T_DIM, T_HIST, seed=0)
    V1 = g.num_nodes + 1
    rng = np.random.default_rng(1)
    hist = (rng.standard_normal((V1, T_HIST, D)) * 0.1).astype(np.float32)
    return orc, g, adj, p, hist, n_edges


def oracle_batch_starts(n_edges, B, n):
    """Start offsets of the n batches the port times: consecutive full batches that end at the end of the sample, wrapping
    over its last 30 % when more batches are asked for than that holds."""
    k = min(n, (n_edges - int(n_edges * 0.7)) // B)
    return [n_edges - k * B + (i % k) * B for i in range(n)]


def oracle_batch(orc, g, adj, p, hist, lo, B, K, neg):
    """Module-boundary functions only (fourier_transform_pe, C x compute_neighborhood_pe, update_pe),
    timed; the loops' own clone of the current table is outside the timer."""
    src, dst, tt = g.src_node_ids[lo:lo + B], g.dst_node_ids[lo:lo + B], g.node_interact_times[lo:lo + B]
    ids = np.unique(np.concatenate([src, dst]))
    t0 = time.perf_counter()
    fft = orc.fourier_transform_pe(p, ids, hist, 10 ** 6, T_HIST)
    t1 = time.perf_counter()
    cur = hist[:, -1, :].copy()
    cur[ids] = fft
    t2 = time.perf_counter()
    for q in (src, dst, src, neg):
        orc.compute_neighborhood_pe(p, adj, cur, q, tt, K)
    orc.update_pe(p, adj, cur, ids, src, dst, tt, tt.max(), K)
    t3 = time.perf_counter()
    return (t1 - t0) + (t3 - t2)


class ReferenceArm:
    """The UNMODIFIED reference's own CPU implementation of the path (oracle/_ref: models/LSTEP.py + utils/utils.py as they
    lie in /root/reference, imported through oracle/refload.py) on the SAME workload as the CUDA arm: the full synthetic
    graph, the reference's own NeighborSampler built over all its edges, the same weights (the drop-in's constructor under
    torch.manual_seed(0) — identical state_dict keys — loaded into the reference module), T = 100 history steps per node,
    torch CPU kernels on all host threads. A step = the module-boundary functions of one batch: fourier_transform_pe,
    C x compute_neighborhood_pe, update_pe (the loop's own clone / index_put between them is outside the timer)."""

    def __init__(self, workload, B, K):
        import torch
        from oracle import refload
        self.ref = refload.load()
        if self.ref is None:
            raise RuntimeError("oracle/_ref not materialised")
        ref = self.ref
        torch.set_num_threads(os.cpu_count())
        self.torch, self.B, self.K = torch, B, K
        self.g = g = synth.make_graph(workload, seed=0, zipf_s=ZIPF_S)
        V1 = g.num_nodes + 1
        t0 = time.time()
        self.sampler = ref.get_neighbor_sampler(ref.Data(g.src_node_ids, g.dst_node_ids, g.node_interact_times, g.edge_ids, g.labels),
                                                "recent", seed=1)
        self.t_sampler = time.time() - t0
        node_feats = np.zeros((V1, 172), dtype=np.float32)
        edge_feats = np.zeros((1, 172), dtype=np.float32)
        from lstep_b200 import LSTEP as DropIn
        torch.manual_seed(0)  # make_params_model(): the CUDA arm's weights
        ours = DropIn(node_feats, edge_feats, None, None, pe_dim=D, num_neighbors=20, time_feat_dim=T_DIM, num_fft_batches=T_HIST, device="cpu")
        self.model = ref.LSTEP(node_feats, edge_feats, self.sampler, self.sampler, pe_dim=D, num_neighbors=20, time_feat_dim=T_DIM,
                               num_fft_batches=T_HIST, device="cpu")
        self.model.load_state_dict(ours.state_dict())
        self.model.eval()
        gen = torch.Generator().manual_seed(1)
        self.hist = torch.randn((V1, T_HIST, D), generator=gen) * 0.1
        self.e0 = int(g.num_edges * 0.7) // B * B
        self.rng = np.random.default_rng(3)
        self.dst_pool = np.unique(g.dst_node_ids)

    def batch(self, i):
        """Batch i of the evaluation split; returns seconds spent in the module-boundary functions."""
        torch, g, B, K, m = self.torch, self.g, self.B, self.K, self.model
        lo = self.e0 + (i * B) % ((g.num_edges - self.e0) // B * B)
        src, dst, tt, ee = (a[lo:lo + B] for a in (g.src_node_ids, g.dst_node_ids, g.node_interact_times, g.edge_ids))
        neg = self.rng.choice(self.dst_pool, len(src))
        ids = torch.from_numpy(np.array(src.tolist() + dst.tolist())).unique().numpy()  # evaluate_model_utils.py:54-55
        with torch.no_grad():
            t0 = time.perf_counter()
            fft = m.fourier_transform_pe(ids, self.hist, 10 ** 6)
            t1 = time.perf_counter()
            cur = torch.clone(self.hist[:, -1, :])
            cur[torch.from_numpy(ids)] = fft
            t2 = time.perf_counter()
            for q in (src, dst, src, neg):
                m.compute_neighborhood_pe(cur, q, tt, num_neighbors=K)
            m.update_pe(cur, ids, ee, src, dst, tt, tt.max(), num_neighbors=K)
            t3 = time.perf_counter()
        return (t1 - t0) + (t3 - t2), len(src)


def cpu_baseline(workload, B, K, n_batches):
    """Reported beside the CUDA number as a baseline only. kind 'reference': the unmodified reference (oracle/_ref);
    kind 'port': the numpy oracle, when oracle/_ref is absent."""
    try:
        arm = ReferenceArm(workload, B, K)
    except Exception as e:  # oracle/_ref absent
        log("reference unavailable (", repr(e)[:120], "): timing the numpy oracle port instead")
        arm = None
    times = []
    if arm is not None:
        budget = time.time() + 25.0
        for i in range(n_batches + 3):
            dt, _ = arm.batch(i)
            if i >= 3:
                times.append(dt)
            if time.time() > budget and len(times) >= 5:
                break
        med = float(np.median(times))
        return {"value": B / med, "unit": "edges/s", "cores": os.cpu_count(), "kind": "reference", "ms_per_batch": med * 1e3,
                "sample": f"{len(times)} batches of {B} edges after 3 warm-up, median; the unmodified reference (oracle/_ref: models/LSTEP.py, "
                          f"utils/utils.py) on torch CPU, {os.cpu_count()} threads, full {workload}-shaped graph (E={arm.g.num_edges}), same weights, "
                          f"T={T_HIST}; module-boundary functions only (fourier_transform_pe, {C_CALLS} x compute_neighborhood_pe, update_pe); "
                          f"reference sampler build {arm.t_sampler:.1f} s (untimed)"}
    orc, g, adj, p, hist, n_edges = oracle_setup(workload, B, K, n_batches)
    rng = np.random.default_rng(3)
    for i, lo in enumerate(oracle_batch_starts(n_edges, B, n_batches + 3)):
        neg = rng.choice(g.dst_node_ids, B)
        dt = oracle_batch(orc, g, adj, p, hist, lo, B, K, neg)
        if i >= 3:
            times.append(dt)
    med = float(np.median(times))
    return {"value": B / med, "unit": "edges/s", "cores": os.cpu_count(), "kind": "port",
            "sample": f"{n_batches} batches of {B} edges after 3 warm-up, median; oracle/lstep_oracle.py (numpy port of the reference path) on the "
                      f"first {n_edges} edges of the same synthetic stream; module-boundary functions only", "ms_per_batch": med * 1e3}


def run_reference(args, rank, world):
    """`--impl reference`: the reference's own CPU implementation of the path (ReferenceArm) on this box's host cores, on the
    CUDA arm's config / metric / unit; each step is one batch. Rank 0 alone runs it (N > 1: the other ranks exit)."""
    if rank != 0:
        return
    global T_HIST
    workload = args.workload
    if workload == "scaleout":
        # the sharded arm's config: batch shape of the Flights config (B=2000, K=20), T = --scaleout-T
        workload, T_HIST = "flights", (args.scaleout_T or T_HIST)
    B, K = WORKLOADS[workload]
    steps, warm = args.steps, max(args.warmup, 1)
    warm = min(warm, 5)
    kind = "reference"
    try:
        arm = ReferenceArm(workload, B, K)
    except Exception as e:
        log("reference unavailable (", repr(e)[:120], "): timing the numpy oracle port instead")
        arm, kind = None, "port"
    tot, edges = 0.0, 0
    if arm is not None:
        for i in range(steps + warm):
            dt, ne = arm.batch(i)
            if i >= warm:
                tot += dt
                edges += ne
        g = arm.g
        sample = (f"{steps} batches of {B} edges: the unmodified reference (oracle/_ref) on torch CPU, {os.cpu_count()} threads, full "
                  f"{workload}-shaped graph, same weights as the CUDA arm, T={T_HIST}; module-boundary functions only")
    else:
        orc, g, adj, p, hist, n_edges = oracle_setup(workload, B, K, steps + warm)
        rng = np.random.default_rng(3)
        for i, lo in enumerate(oracle_batch_starts(n_edges, B, steps + warm)):
            neg = rng.choice(g.dst_node_ids, B)
            dt = oracle_batch(orc, g, adj, p, hist, lo, B, K, neg)
            if i >= warm:
                tot += dt
                edges += B
        g = synth.make_graph(workload, seed=0, num_edges=1000, zipf_s=ZIPF_S)
        g_full = synth.SHAPES[workload]
        sample = f"{steps} batches of {B} edges on the first {n_edges} edges of the synthetic stream (oracle port, numpy + BLAS threads)"
    value = edges / tot
    cfg = workload_config(workload, arm.g if arm is not None else synth.make_graph(workload, seed=0, zipf_s=ZIPF_S), B, K, 1)
    out = {"impl": "reference", "metric": "temporal edges/sec through PE update+aggregation; % HBM roofline", "value": value,
           "unit": "edges/s", "n_gpus": world, "steps": steps, "warmup": warm, "ms_per_step": tot / steps * 1e3, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": cfg,
           "cpu_baseline": {"value": value, "unit": "edges/s", "cores": os.cpu_count(), "kind": kind, "sample": sample},
           "e2e": {"value": value, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(out)


_REAL_STDOUT = None


def quiet_stdout():
    """Libraries (NCCL prints its version banner) write to fd 1; the driver wants exactly one JSON line there.
    Route fd 1 to stderr for the duration of the run; emit() restores it for the result line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(obj), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="reddit", choices=sorted(WORKLOADS) + ["scaleout"])
    ap.add_argument("--replicas", action="store_true", help="N > 1: only the replicas of the single-GPU workload (skip the sharded scale-out sample)")
    ap.add_argument("--scaleout-batch", type=int, default=2000, help="edges per step of the scale-out arm (BASELINE config 5 is quoted at 2000)")
    ap.add_argument("--scaleout-nodes", type=int, default=10_000_000)
    ap.add_argument("--scaleout-edges", type=int, default=100_000_000)
    ap.add_argument("--scaleout-T", type=int, default=0, help="history steps per node of the scale-out arm (default: 100 with the change-log "
                    "history; 12 with the dense ring, whose N = 1 point must fit one GPU — T = 100 needs 8 GPUs there)")
    ap.add_argument("--scaleout-history", default="changelog", choices=["changelog", "ring"],
                    help="scale-out arm's history: change-log (base + changed rows; N = 1 holds T = 100) or the dense ring sharded by node id")
    ap.add_argument("--no-scaleout", action="store_true", help="N = 1: skip the scale-out sample that rides along with the headline run")
    ap.add_argument("--scaleout-timeout", type=float, default=420.0, help="seconds the scale-out sample may take at N > 1")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--zipf", type=float, default=0.8, help="endpoint skew of the synthetic stream (0.8: the headline workload; 1.2: hub-heavy)")
    ap.add_argument("--cpu-batches", type=int, default=40)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed steps computed in the last one to DIR/<name>.npy (headline workload, rank 0)")
    args = ap.parse_args()
    global ZIPF_S
    ZIPF_S = float(args.zipf)
    if args.steps is None:  # (the reference arm runs its steps on the host CPU: a shorter default)
        args.steps = 1000 if args.workload != "scaleout" and args.impl != "reference" else 100
    if args.warmup is None:
        args.warmup = 120 if args.workload != "scaleout" else 30
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload == "scaleout"):
        ap.error("--dump-outputs writes the outputs of the CUDA path's headline workload (not --impl reference, not --workload scaleout)")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    quiet_stdout()
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif args.workload == "scaleout":
        run_sharded(args, rank, world)
    else:
        # The headline workload does not shard at this size (7 MB table, strictly sequential 200-edge batches): at N > 1 the main
        # line is N independent replicas of it (weak scaling, comparable with the N = 1 line). The scale-out graph of BASELINE
        # config 5 (history ring sharded by node id, NCCL all-gather per step) is measured in the same run — at EVERY N,
        # N = 1 included, so that the record holds its whole 1 -> 8 curve — and reported under "scaleout" (strong scaling).
        import torch
        if world > 1:
            import torch.distributed as dist
            local = int(os.environ.get("LOCAL_RANK", 0))
            torch.cuda.set_device(local)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        out = run_ours(args, rank, world, own_pg=False)
        extra = None
        if not (args.replicas or args.no_scaleout):
            # the main line must survive the extra arm: an exception is caught, and a hang (a collective that never
            # completes) is cut by a watchdog that prints the main line and leaves
            def bail():
                log(f"scale-out arm exceeded {args.scaleout_timeout:.0f} s: reporting the main line only")
                if rank == 0:
                    out["scaleout"] = {"error": f"timed out after {args.scaleout_timeout:.0f} s"}
                    emit(out)
                os._exit(0)
            dog = threading.Timer(args.scaleout_timeout, bail)
            dog.daemon = True
            dog.start()
            try:
                extra = run_sharded(args, rank, world, own_pg=False)
            except Exception as e:
                log("scale-out arm failed:", repr(e))
                extra = {"error": repr(e)[:300]}
            dog.cancel()
        if rank == 0:
            if extra is not None:
                out["scaleout"] = {k: extra[k] for k in ("value", "unit", "ms_per_step", "steps", "warmup", "scaling", "config", "run_info", "e2e",
                                                         "error") if k in extra}
            emit(out)
        if world > 1:
            try:
                dist.destroy_process_group()
            except Exception:
                pass


if __name__ == "__main__":
    main()
