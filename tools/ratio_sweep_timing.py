"""Wall clock of a ratio sweep over one loaded database (tooling): 16 (len_ratio, pos_ratio) pairs grouped
  * back to back on one context (K = 1), or
  * by K threads, each on its own context of the same database (the base and K-1 views, rk_create_view), K in --ks.
Every grouping is rk_group with RK_F_HOST_RESULT (synchronous); a sweep ends when every thread's last call returned.
Modes alternate within each repeat; medians and spread over --repeats repeats.  The records are generated on the device
(C1 = 1e5, 1e6 = C2's shape scaled, C2 = 1e7 fragments) and loaded from there.

    python tools/ratio_sweep_timing.py [--sizes 1e5,1e6,1e7] [--ks 2,4] [--repeats 5] [--bench-parent DIR] [--out FILE]

--bench-parent DIR: also runs `bench.py --gpus 1` (config 2) in DIR (another checkout) and in this tree, alternating,
and reports both per-step times.  Card name and power limit are read in the same run.  Prints one JSON document (and
writes it to --out)."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from repkiller_b200 import capi, gen  # noqa: E402

PAIRS = [(lr, pr) for lr in (0.02, 0.05, 0.1, 0.2) for pr in (0.02, 0.05, 0.1, 0.3)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return [ln.strip() for ln in q.stdout.splitlines() if ln.strip()]


def workload(n):
    if n == 100_000:
        return gen.WORKLOADS["c1"]
    if n == 10_000_000:
        return gen.WORKLOADS["c2"]
    return gen.scaled(gen.WORKLOADS["c2"], n)


def group(ctx, pair, res):
    ctx._check(ctx._L.rk_group(ctx._h, pair[0], pair[1], capi.F_HOST_RESULT, C.byref(res)))
    return int(res.n_groups)


def sweep(ctxs, pool, results):
    """wall-clock seconds of grouping every pair once; thread i takes pairs i, i+K, ... on context i"""
    k = len(ctxs)

    def run(i):
        res = capi._Result()
        for j in range(i, len(PAIRS), k):
            results[j] = group(ctxs[i], PAIRS[j], res)

    t0 = time.perf_counter()
    if k == 1:
        run(0)
    else:
        for f in [pool.submit(run, i) for i in range(k)]:
            f.result()
    return time.perf_counter() - t0


def measure_size(n, ks, repeats):
    import torch
    w = workload(n)
    dev = torch.empty(n * 109 + 16, dtype=torch.uint8, device="cuda")
    base = capi.Context(0)
    base.generate_device(w, 0, n, dev.data_ptr())
    st = base.load(dev.data_ptr(), w.lx + 1, w.ly + 1, n=n)
    views = [base.view() for _ in range(max(ks) - 1)]
    modes = [1] + list(ks)
    pool = ThreadPoolExecutor(max(ks))
    groups = {}
    for k in modes:  # warm-up, and the group counts every mode must reproduce
        groups[k] = [None] * len(PAIRS)
        sweep([base] + views[:k - 1], pool, groups[k])
    times = {k: [] for k in modes}
    for _ in range(repeats):
        for k in modes:
            got = [None] * len(PAIRS)
            times[k].append(sweep([base] + views[:k - 1], pool, got))
            assert got == groups[1], f"K={k}: group counts differ from the sequential sweep"
    pool.shutdown()
    seq = statistics.median(times[1])
    out = {"fragments": n, "kept": st.n_kept, "workload": w.name, "pairs": len(PAIRS), "group_counts_equal": True, "modes": []}
    for k in modes:
        med = statistics.median(times[k])
        out["modes"].append({"contexts": k, "threads": k, "median_ms": round(med * 1e3, 3), "min_ms": round(min(times[k]) * 1e3, 3),
                             "max_ms": round(max(times[k]) * 1e3, 3), "ms_per_pair": round(med * 1e3 / len(PAIRS), 4),
                             "speedup_vs_one_context": round(seq / med, 3), "runs_ms": [round(t * 1e3, 3) for t in times[k]]})
    for v in views:
        v.close()
    base.close()
    del dev
    torch.cuda.empty_cache()
    return out


def bench_ab(parent, rounds):
    cmd = [sys.executable, "bench.py", "--gpus", "1", "--steps", "20", "--warmup", "3", "--no-cpu-baseline"]
    runs = []
    for _ in range(rounds):
        for tree, cwd in (("parent", parent), ("this change", ROOT)):
            p = subprocess.run(cmd, cwd=cwd, capture_output=True, text=True)
            line = next((ln for ln in reversed(p.stdout.splitlines()) if ln.startswith("{")), None)
            if p.returncode or line is None:
                runs.append({"tree": tree, "error": (p.stderr or p.stdout)[-400:]})
                continue
            r = json.loads(line)
            runs.append({"tree": tree, "ms_per_step": r["ms_per_step"], "value": r["value"]})
    summary = {}
    for tree in ("parent", "this change"):
        ms = [r["ms_per_step"] for r in runs if r["tree"] == tree and "ms_per_step" in r]
        if ms:
            summary[tree] = {"median_ms_per_step": round(statistics.median(ms), 4), "min": round(min(ms), 4), "max": round(max(ms), 4)}
    return {"command": " ".join(cmd[1:]) + ", parent tree and this tree alternating in one call", "runs": runs, "summary": summary}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1e5,1e6,1e7")
    ap.add_argument("--ks", default="2,4")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--bench-parent", default=None)
    ap.add_argument("--bench-rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    doc = {"card": card(), "tool": "tools/ratio_sweep_timing.py", "repeats": a.repeats, "pairs": PAIRS,
           "sizes": [measure_size(int(float(s)), [int(k) for k in a.ks.split(",")], a.repeats) for s in a.sizes.split(",")]}
    if a.bench_parent:
        doc["bench_ab"] = bench_ab(a.bench_parent, a.bench_rounds)
    text = json.dumps(doc, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
