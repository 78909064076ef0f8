"""Wall clock of a ratio sweep over one PARTITIONED load (tooling): 16 (len_ratio, pos_ratio) pairs grouped
  * back to back on one rk_multi (K = 1), or
  * by K threads, each on its own rk_multi of the same load (the base and K-1 views, rk_multi_create_view), K in --ks.
Every grouping is rk_multi_group (synchronous, host result); a sweep ends when every thread's last call returned.  Modes
alternate within each repeat; medians and spread over --repeats repeats; the group counts of every mode must equal the
sequential sweep's.  --ranks R runs R ranks; --devices picks them: "distinct" (GPUs 0..R-1, NCCL) or "same" (every rank
a thread on GPU 0, the local transport).  On a box with fewer than R GPUs "distinct" falls back to "same", and the JSON
says so: ranks on one GPU share its SMs, so such a run measures no multi-GPU gain.

    python tools/multi_ratio_sweep_timing.py [--ranks 2,8] [--per-rank 1e6,1e7] [--ks 2,4] [--repeats 5]
                                             [--bench-parent DIR] [--out FILE]

--bench-parent DIR: also runs, alternating between DIR (another checkout, already built) and this tree, `bench.py
--gpus 1` and the sequential sweep of a partitioned load (2 ranks, --ab-per-rank fragments each; the one-GPU stand-in
for `bench.py --gpus 2`), and reports both.  Card names and power limits are read in the same run.  Prints one JSON
document (and writes it to --out)."""
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
PAIRS = [(lr, pr) for lr in (0.02, 0.05, 0.1, 0.2) for pr in (0.02, 0.05, 0.1, 0.3)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return [ln.strip() for ln in q.stdout.splitlines() if ln.strip()]


def workload(gen, n):
    return gen.WORKLOADS["c2"] if n == 10_000_000 else gen.scaled(gen.WORKLOADS["c2"], n)


def group(capi, m, pair, res):
    m._check(m._L.rk_multi_group(m._h, pair[0], pair[1], 0, C.byref(res)))
    return int(res.n_groups)


def sweep(capi, ms, pool, results):
    """wall-clock seconds of grouping every pair once; thread i takes pairs i, i+K, ... on rk_multi i"""
    k = len(ms)

    def run(i):
        res = capi._Result()
        for j in range(i, len(PAIRS), k):
            results[j] = group(capi, ms[i], PAIRS[j], res)

    t0 = time.perf_counter()
    if k == 1:
        run(0)
    else:
        for f in [pool.submit(run, i) for i in range(k)]:
            f.result()
    return time.perf_counter() - t0


def load(capi, gen, ranks, per_rank, devices):
    import torch
    distinct = devices == "distinct" and torch.cuda.device_count() >= ranks
    w = workload(gen, per_rank * ranks)
    rec = gen.generate(w)
    m = capi.Multi(list(range(ranks)) if distinct else [0] * ranks)
    st = m.load(rec, w.lx + 1, w.ly + 1)
    return m, w, st, distinct


def measure(capi, gen, ranks, per_rank, ks, repeats, devices):
    m, w, st, distinct = load(capi, gen, ranks, per_rank, devices)
    views = [m.view() for _ in range(max(ks) - 1)]
    modes = [1] + list(ks)
    pool = ThreadPoolExecutor(max(ks))
    groups = {}
    for k in modes:  # warm-up, and the group counts every mode must reproduce
        groups[k] = [None] * len(PAIRS)
        sweep(capi, [m] + views[:k - 1], pool, groups[k])
        assert groups[k] == groups[1], f"K={k}: group counts differ from the sequential sweep"
    times = {k: [] for k in modes}
    for _ in range(repeats):
        for k in modes:
            got = [None] * len(PAIRS)
            times[k].append(sweep(capi, [m] + views[:k - 1], pool, got))
            assert got == groups[1], f"K={k}: group counts differ from the sequential sweep"
    pool.shutdown()
    seq = statistics.median(times[1])
    out = {"ranks": ranks, "fragments_per_rank": per_rank, "fragments": w.n, "kept": st.n_kept, "workload": w.name,
           "devices": "distinct GPUs (NCCL)" if distinct else "every rank a thread on GPU 0 (local transport)",
           "transport": m.transport, "pairs": len(PAIRS), "group_counts_equal": True, "group_counts": groups[1], "modes": []}
    for k in modes:
        med = statistics.median(times[k])
        out["modes"].append({"contexts": k, "threads": k, "median_ms": round(med * 1e3, 3), "min_ms": round(min(times[k]) * 1e3, 3),
                             "max_ms": round(max(times[k]) * 1e3, 3), "ms_per_pair": round(med * 1e3 / len(PAIRS), 4),
                             "speedup_vs_one_context": round(seq / med, 3), "runs_ms": [round(t * 1e3, 3) for t in times[k]]})
    for v in views:
        v.close()
    m.close()
    return out


def sequential_only(capi, gen, ranks, per_rank, repeats):
    """the K = 1 sweep alone (no views: runs on a tree without them too); one JSON line"""
    m, w, st, _ = load(capi, gen, ranks, per_rank, "same")
    pool = None
    first = [None] * len(PAIRS)
    sweep(capi, [m], pool, first)
    times = []
    for _ in range(repeats):
        got = [None] * len(PAIRS)
        times.append(sweep(capi, [m], pool, got))
        assert got == first
    m.close()
    print(json.dumps({"median_ms": round(statistics.median(times) * 1e3, 3), "runs_ms": [round(t * 1e3, 3) for t in times],
                      "group_counts": first}))


def bench_ab(parent, rounds, ab_per_rank):
    bench = [sys.executable, "bench.py", "--gpus", "1", "--steps", "20", "--warmup", "3", "--no-cpu-baseline"]
    runs = []
    for _ in range(rounds):
        for tree, cwd in (("parent", parent), ("this change", ROOT)):
            p = subprocess.run(bench, cwd=cwd, capture_output=True, text=True)
            line = next((ln for ln in reversed(p.stdout.splitlines()) if ln.startswith("{")), None)
            if p.returncode or line is None:
                runs.append({"tree": tree, "what": "bench", "error": (p.stderr or p.stdout)[-400:]})
            else:
                r = json.loads(line)
                runs.append({"tree": tree, "what": "bench", "ms_per_step": r["ms_per_step"], "value": r["value"], "checksum": r.get("checksum")})
            seq = [sys.executable, os.path.abspath(__file__), "--sequential-only", "--root", os.path.abspath(cwd), "--ranks", "2",
                   "--per-rank", str(ab_per_rank), "--repeats", "3"]
            p = subprocess.run(seq, cwd=cwd, capture_output=True, text=True)
            line = next((ln for ln in reversed(p.stdout.splitlines()) if ln.startswith("{")), None)
            if p.returncode or line is None:
                runs.append({"tree": tree, "what": "partitioned sweep", "error": (p.stderr or p.stdout)[-400:]})
            else:
                runs.append({"tree": tree, "what": "partitioned sweep", **json.loads(line)})
    summary = {}
    for tree in ("parent", "this change"):
        ms = [r["ms_per_step"] for r in runs if r["tree"] == tree and "ms_per_step" in r]
        sw = [r["median_ms"] for r in runs if r["tree"] == tree and "median_ms" in r]
        summary[tree] = {"bench_median_ms_per_step": round(statistics.median(ms), 4) if ms else None,
                         "bench_checksums": sorted({r["checksum"] for r in runs if r["tree"] == tree and r.get("checksum") is not None}),
                         "partitioned_sweep_median_ms": round(statistics.median(sw), 3) if sw else None,
                         "partitioned_group_counts": [r["group_counts"] for r in runs if r["tree"] == tree and "group_counts" in r][:1]}
    return {"bench": " ".join(bench[1:]), "partitioned_sweep": f"16 pairs back to back on one rk_multi, 2 ranks as threads on GPU 0, "
            f"{ab_per_rank} fragments per rank", "order": "parent tree and this tree alternating in one call", "runs": runs, "summary": summary}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ranks", default="2,8")
    ap.add_argument("--per-rank", default="1e6,1e7")
    ap.add_argument("--ks", default="2,4")
    ap.add_argument("--devices", default="distinct", choices=["distinct", "same"])
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--bench-parent", default=None)
    ap.add_argument("--bench-rounds", type=int, default=3)
    ap.add_argument("--ab-per-rank", type=float, default=5e6)
    ap.add_argument("--sequential-only", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--root", default=ROOT, help=argparse.SUPPRESS)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    sys.path.insert(0, a.root)
    from repkiller_b200 import capi, gen
    if a.sequential_only:
        return sequential_only(capi, gen, int(a.ranks), int(float(a.per_rank)), a.repeats)
    ks = [int(k) for k in a.ks.split(",")]
    doc = {"card": card(), "tool": "tools/multi_ratio_sweep_timing.py", "repeats": a.repeats, "pairs": PAIRS, "runs": []}
    for r in (int(x) for x in a.ranks.split(",")):
        for n in (int(float(x)) for x in a.per_rank.split(",")):
            doc["runs"].append(measure(capi, gen, r, n, ks, a.repeats, a.devices))
    if a.bench_parent:
        doc["bench_ab"] = bench_ab(a.bench_parent, a.bench_rounds, int(a.ab_per_rank))
    text = json.dumps(doc, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
