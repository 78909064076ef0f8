"""bench.py contract pieces.  Without a GPU: the reference arm (the reference's own CPU code on a bounded sample) prints
one JSON line with the agreed keys; our arm refuses to run without a CUDA device instead of falling back; --dump-outputs
is refused for the reference arm.  On the GPU: --dump-outputs writes the last timed step's output, and --steps sets the
number of timed steps."""
import json
import os
import subprocess
import sys

import pytest

from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line():
    """the compiled reference when oracle/_ref holds it, else the oracle's port of the same path"""
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--frags", "60000", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "fragments/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert d["cpu_baseline"]["kind"] == ("reference" if O.have_ref() else "port") and d["cpu_baseline"]["cores"] == 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "fragments/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_our_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"], capture_output=True, text=True,
                       timeout=300)
    assert p.returncode != 0
    assert "no CPU fallback" in (p.stderr + p.stdout)


def test_dump_outputs_is_refused_for_the_reference_arm(tmp_path):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=300)
    assert p.returncode != 0 and "--dump-outputs" in p.stderr
    assert os.listdir(tmp_path) == []


def _bench_with_dump(out_dir, n, steps):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--n", str(n), "--steps", str(steps), "--warmup", "1",
                        "--no-e2e", "--no-cpu-baseline", "--checksum", "0", "--dump-outputs", str(out_dir)], capture_output=True,
                       text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    return json.loads([ln for ln in p.stdout.splitlines() if ln.startswith("{")][-1])


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(tmp_path):
    """--dump-outputs: the arrays of the timed path's last step, sampled at seeded line positions when the output has more
    lines than bench.DUMP_MAX_LINES, equal the oracle's output at those lines and do not depend on --steps.  --steps is the
    number of timed steps: the library counts every kernel launch of the profiled timed region, and those counts divided by
    --steps must be the launches of one step, the same for 1 and for 3 steps."""
    import numpy as np
    from repkiller_b200 import gen
    n = 1_200_000
    names = ("n_kept", "n_groups", "line", "order", "gid", "repval", "identity")
    d1 = _bench_with_dump(tmp_path / "s1", n, 1)
    d3 = _bench_with_dump(tmp_path / "s3", n, 3)
    assert d1["steps"] == 1 and d3["steps"] == 3
    per_step = {k: v["launches_per_step"] for k, v in d1["kernels"].items()}
    assert per_step and all(v >= 1 and v == int(v) for v in per_step.values())
    assert {k: v["launches_per_step"] for k, v in d3["kernels"].items()} == per_step
    w = gen.scaled(gen.WORKLOADS["c2"], n)
    g = O.group(gen.generate(w), w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio)
    got = {name: np.load(tmp_path / "s3" / f"{name}.npy") for name in names}
    for name in names:
        assert np.load(tmp_path / "s1" / f"{name}.npy").tobytes() == got[name].tobytes(), name
    assert sum(v.nbytes for v in got.values()) <= 64 << 20
    assert all(v.dtype in (np.float32, np.float64) for v in got.values())
    assert got["n_kept"].tolist() == [g.n_kept] and got["n_groups"].tolist() == [g.n_groups]
    line = got["line"].astype(np.int64)
    assert 0 < line.shape[0] < g.n_kept and (np.diff(line) > 0).all() and line[-1] < g.n_kept
    assert np.array_equal(got["order"], g.order[line]) and np.array_equal(got["gid"], g.out_gid[line])
    assert np.array_equal(got["repval"], g.repval[line])
    assert np.array_equal(got["identity"].view(np.uint32), g.identity[line].view(np.uint32))
