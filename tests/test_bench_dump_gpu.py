"""bench.py --dump-outputs: the last timed step's outputs as float32 .npy files within 64 MB, identical from run to run with
the same arguments (seeded inputs, deterministic path), and equal to an independent replay of the same steps."""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_dump(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny_bip", "--steps", str(steps), "--warmup", "2",
           "--no-scaleout", "--no-cpu-baseline", "--dump-outputs", out_dir]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    assert res.stdout.count("\n") == 1, res.stdout
    line = json.loads(res.stdout)
    assert line["steps"] == steps
    return line, {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_bench_dump_outputs_are_reproducible_and_are_the_last_steps_outputs():
    import torch
    import bench
    with tempfile.TemporaryDirectory() as tmp:
        line, a = _bench_dump(os.path.join(tmp, "a"), 7)
        _, b = _bench_dump(os.path.join(tmp, "b"), 7)
        _, c = _bench_dump(os.path.join(tmp, "c"), 8)
    assert sorted(a) == ["neighborhood_pe", "pe_history_sample", "pe_table"]
    assert sum(x.nbytes for x in a.values()) <= 64_000_000
    for k in a:
        assert a[k].dtype == np.float32 and np.isfinite(a[k]).all() and a[k].any(), k
        assert np.array_equal(a[k], b[k]), k
    assert not np.array_equal(a["neighborhood_pe"], c["neighborhood_pe"])
    # replay: the same state, every step the run made (history fill, warm-up, timed) one PEStream.step at a time
    h = bench.headline_setup("tiny_bip", 0, torch.device("cuda"))
    n = line["run_info"]["history_fill_steps_before_warmup"] + line["warmup"] + line["steps"]
    with torch.no_grad():
        for s in range(n):
            out = h.stream.step(s % h.nb, h.queries(s % h.nb))
    V1 = h.stream.V1
    assert V1 < bench.DUMP_HISTORY_ROWS  # tiny_bip: the history sample holds every row
    assert np.array_equal(a["neighborhood_pe"], out.cpu().numpy())
    assert np.array_equal(a["pe_table"], h.stream.cur.cpu().numpy())
    assert np.array_equal(a["pe_history_sample"], h.stream.export_history().cpu().numpy())
    h.stream.check_errors()
