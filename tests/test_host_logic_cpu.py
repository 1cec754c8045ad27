"""CPU-side checks of the host logic around the CUDA path: the byte model bench.py's roofline uses, the synthetic
workloads of BASELINE.json's configs, the rule that the product path never touches the oracle, and that it fails loudly
(no CPU fallback) when no CUDA device is present."""
import ast
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "l-step_b200")


@pytest.mark.parametrize("B,N,M,V,want_mb,want_h_mb", [
    (200, 105, 178, 184, 21.8, 0.25),        # Enron-shaped
    (200, 300, 2000, 9227, 42.3, 12.7),      # Wikipedia-shaped
    (200, 300, 2300, 10984, 43.4, 15.1),     # Reddit-shaped (the headline workload)
    (2000, 2500, 9000, 13169, 340.0, 18.1),  # Flights-shaped
])
def test_byte_model_reproduces_the_survey_figures(B, N, M, V, want_mb, want_h_mb):
    """SURVEY §8(d) 'Algorithmic bytes per batch': bench.py's bytes_model (the numerator of `roofline.achieved` and of
    `path_roofline`) gives the survey's illustrative values for the survey's N and M."""
    import bench
    b = bench.bytes_model(B, N, M, 20, V1=V + 1)
    assert b["bytes_path"] == b["F"] + b["S"] + b["P"] + b["UA"] + b["UB"] + b["W"]
    assert abs(b["bytes_path"] / 1e6 - want_mb) < 0.06 * max(1.0, want_mb / 40)
    assert abs(b["H"] / 1e6 - want_h_mb) < 0.06
    assert abs(b["W"] / 1e6 - 0.85) < 0.01  # six weight matrices once


@pytest.mark.parametrize("name", ["enron", "wikipedia", "reddit", "flights"])
def test_synthetic_workloads_have_the_baseline_shapes(name):
    """SURVEY §8(d) 'Synthetic inputs': ids 1..V (row 0 is the padding node), timestamps ascending float64, bipartite
    offset for Wikipedia / Reddit, integer day stamps with heavy ties for Flights; the stream is a pure function of
    the seed."""
    from lstep_b200 import synth
    spec = synth.SHAPES[name]
    E = min(spec["num_edges"], 200_000)  # a prefix-sized sample keeps the CPU suite short; the generator is O(E)
    g = synth.make_graph(name, seed=0, num_edges=E)
    assert g.num_nodes == spec["num_nodes"] and g.num_edges == E
    for a in (g.src_node_ids, g.dst_node_ids, g.edge_ids):
        assert a.dtype == np.int64 and a.shape == (E,)
    assert g.node_interact_times.dtype == np.float64
    assert g.src_node_ids.min() >= 1 and g.dst_node_ids.min() >= 1
    assert max(g.src_node_ids.max(), g.dst_node_ids.max()) <= spec["num_nodes"]
    assert np.all(np.diff(g.node_interact_times) >= 0)
    assert np.array_equal(g.edge_ids, np.arange(1, E + 1))
    if spec["src_side"] is not None:
        assert g.src_node_ids.max() <= spec["src_side"] < g.dst_node_ids.min()
    if spec["ties"]:
        assert len(np.unique(g.node_interact_times)) <= 122
        assert np.array_equal(g.node_interact_times, np.floor(g.node_interact_times))
    else:
        assert g.node_interact_times.max() < spec["t_span"]
    g2 = synth.make_graph(name, seed=0, num_edges=E)
    assert np.array_equal(g.src_node_ids, g2.src_node_ids) and np.array_equal(g.node_interact_times, g2.node_interact_times)
    g3 = synth.make_graph(name, seed=1, num_edges=E)
    assert not np.array_equal(g.src_node_ids, g3.src_node_ids)


def test_unique_batch_nodes_and_initial_pe():
    from lstep_b200 import synth
    src = np.array([5, 3, 5, 9], dtype=np.int64)
    dst = np.array([7, 3, 2, 9], dtype=np.int64)
    ids = synth.unique_batch_nodes(src, dst)
    assert ids.dtype == np.int64 and np.array_equal(ids, [2, 3, 5, 7, 9])  # sorted-unique, as np.unique in the loops
    pe = synth.make_initial_pe(10, 172)
    assert pe.shape == (11, 172) and pe.dtype == np.float32 and not pe[0].any() and pe[1:].any()


def _imports_of(path):
    tree = ast.parse(open(path).read(), path)
    for node in ast.walk(tree):
        if isinstance(node, ast.Import):
            for a in node.names:
                yield a.name
        elif isinstance(node, ast.ImportFrom):
            yield node.module or ""


def test_product_path_never_imports_the_oracle():
    """The oracle is test infrastructure: only tests/, __graft_entry__.smoke()/build() and bench.py's CPU legs may touch
    it. No module of the package imports it, and no C / CUDA source mentions a file under oracle/."""
    for fn in sorted(os.listdir(PKG)):
        if fn.endswith(".py"):
            mods = list(_imports_of(os.path.join(PKG, fn)))
            assert not [m for m in mods if m.split(".")[0] == "oracle"], (fn, mods)
    for fn in sorted(os.listdir(os.path.join(PKG, "csrc"))):
        text = open(os.path.join(PKG, "csrc", fn)).read()
        assert not re.search(r'#include\s+"[^"]*oracle', text), fn
    # bench.py: the oracle is imported inside the CPU legs only (never at module level)
    tree = ast.parse(open(os.path.join(ROOT, "bench.py")).read())
    top = [n for n in tree.body if isinstance(n, (ast.Import, ast.ImportFrom))]
    for n in top:
        names = [a.name for a in n.names] if isinstance(n, ast.Import) else [n.module or ""]
        assert not [m for m in names if m.split(".")[0] == "oracle"], names


def test_no_cpu_fallback_without_a_device():
    """There is no CPU fallback: without a CUDA device the library refuses to load for compute and the host-side
    entry points raise instead of computing something else."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    from lstep_b200 import NeighborSampler, _lib, synth
    with pytest.raises(_lib.LstepError, match="no CPU fallback"):
        _lib.load()
    g = synth.make_graph("tiny", seed=0)
    with pytest.raises((_lib.LstepError, RuntimeError, AssertionError)):
        NeighborSampler.from_edges(g.src_node_ids, g.dst_node_ids, g.edge_ids, g.node_interact_times, "recent",
                                   num_rows=g.num_nodes + 1)


def test_status_codes_map_to_the_reference_exception_types():
    """INTEGRATION.md: nonzero C-ABI statuses become the exception types the reference raises (IndexError for an id
    outside the tables, utils/utils.py:140-146 via adj_list[node_id]; ValueError for a bad argument)."""
    from lstep_b200 import _lib
    lib = _lib.load(require_device=False)
    _lib.check(0, "ok")
    with pytest.raises(IndexError):
        _lib.check(5, "lookup")
    seen = set()
    for code in range(0, 16):
        msg = lib.lstep_strerror(code)
        assert isinstance(msg, bytes) and msg
        seen.add(msg)
    assert len(seen) >= 6  # distinct messages for the distinct error codes


def test_header_cites_the_reference_interface_it_replaces():
    """include/lstep_b200.h: the entry points of the hot path name the reference function (file:line) they replace."""
    text = open(os.path.join(ROOT, "include", "lstep_b200.h")).read()
    for cite in ("utils/utils.py", "models/LSTEP.py", "models/modules.py"):
        assert cite in text, cite
    assert len(re.findall(r"(?:LSTEP|utils|modules|evaluate_model_utils)\.py:\d+", text)) >= 10


@pytest.mark.parametrize("args", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"],
                                  ["--workload", "scaleout", "--dump-outputs", "out"]])
def test_bench_rejects_arguments_it_cannot_honour(args, tmp_path):
    """bench.py refuses, before any work, a run with no timed step and an output dump of a path it does not dump."""
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=120,
                         cwd=tmp_path)
    assert out.returncode == 2 and "error:" in out.stderr, out.stderr[-2000:]
    assert out.stdout == "" and not os.listdir(tmp_path)


def test_reference_arm_runs_more_steps_than_the_stream_has_batches():
    """--steps is honoured exactly even when it exceeds the batches of the (sampled) stream: the port's batches wrap over the
    tail of its sample, every one a full batch (tiny_bip: 40 batches of 50 edges)."""
    import json
    import subprocess
    import sys
    import bench
    starts = bench.oracle_batch_starts(2000, 50, 60)
    assert len(starts) == 60 and min(starts) >= 1400 and max(starts) + 50 <= 2000 and starts[:3] == [1400, 1450, 1500]
    assert bench.oracle_batch_starts(40_000, 200, 10) == list(range(38_000, 40_000, 200))  # fits: the last n batches
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny_bip", "--steps", "50",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout)
    assert d["steps"] == 50 and d["value"] > 0 and np.isfinite(d["ms_per_step"])


def test_reference_arm_under_torchrun_prints_one_line_from_rank_0():
    """bench.py --impl reference launched like the driver launches it for N > 1 (torchrun, one process per rank): rank 0 alone
    runs the reference's CPU path and prints ONE JSON line, the other ranks exit 0 without work. CPU only (gloo is not even
    needed: the reference arm creates no process group)."""
    import json
    import subprocess
    import sys
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "2",
           "--warmup", "1", "--workload", "tiny_bip"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["steps"] == 2 and d["warmup"] == 1
    assert d["unit"] == "edges/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
