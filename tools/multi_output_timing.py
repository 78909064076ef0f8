"""Time of the output side of one comparison partitioned over several GPUs (tooling):
  * the extra time of rk_multi_group with RK_F_LINE_RECORDS (the line records travel to the ranks that hold the lines);
  * the device formatting of every rank's lines (rk_dist_format_lines) and of the whole text (rk_multi_format_lines);
  * the CLI under RK_DEVICES=0,..,N-1: the device writer against the host writer (RK_LEGACY_WRITER=1) on the same input.

    python tools/multi_output_timing.py [--n-per-gpu 10000000] [--worlds 2,8] [--cli-n 5000000] [--reps 5] [--out FILE]

Ranks run on distinct GPUs when the box has them; otherwise a world is run as threads on GPU 0 (with the same total
number of fragments split over the ranks), and the JSON says so.  Card name and power limit are read in the same run.
Prints one JSON document (and writes it to --out)."""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from repkiller_b200 import capi, gen  # noqa: E402

CLI = os.path.join(ROOT, "repkiller_b200", "bin", "repkiller")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return [ln.strip() for ln in q.stdout.splitlines() if ln.strip()]


def generate_host(w, chunk=8_000_000):
    """the records of workload w in host memory, generated on GPU 0 (the same bytes as gen.generate(w))"""
    import torch
    out = np.empty(w.n, dtype=gen.generate(w, 0, 1).dtype)
    raw = out.view(np.uint8).reshape(-1)
    buf = torch.empty(min(chunk, w.n) * 109, dtype=torch.uint8, device="cuda:0")
    with capi.Context(0) as ctx:
        for s in range(0, w.n, chunk):
            k = min(chunk, w.n - s)
            ctx.generate_device(w, s, k, buf.data_ptr())
            torch.cuda.synchronize()
            raw[s * 109:(s + k) * 109] = buf[:k * 109].cpu().numpy()
    return out


def multi_group(m, w, flags):
    r = capi._Result()
    t0 = time.perf_counter()
    m._check(m._L.rk_multi_group(m._h, w.len_ratio, w.pos_ratio, flags | capi.F_TIMING, C.byref(r)))
    return time.perf_counter() - t0, r.ms_device


def time_world(world, n_per_gpu, reps, n_gpus):
    distinct = n_gpus >= world
    devices = list(range(world)) if distinct else [0] * world
    n_total = n_per_gpu * world if distinct else n_per_gpu
    w = gen.scaled(gen.WORKLOADS["c2"], n_total)
    rec = generate_host(w)
    out = {"world": world, "devices": devices, "ranks": "distinct GPUs" if distinct else "threads on GPU 0", "fragments": n_total}
    with capi.Multi(devices) as m:
        out["transport"] = m.transport
        m.load(rec, w.lx + 1, w.ly + 1)
        multi_group(m, w, capi.F_LINE_RECORDS)   # warm-up of both forms
        multi_group(m, w, 0)
        walls = {0: [], capi.F_LINE_RECORDS: []}
        dev = {0: [], capi.F_LINE_RECORDS: []}
        for _ in range(reps):   # alternating
            for f in (0, capi.F_LINE_RECORDS):
                a, b = multi_group(m, w, f)
                walls[f].append(a * 1e3)
                dev[f].append(b)
        lines = [m.info(r)["n_lines"] for r in range(world)]
        out["lines_per_rank"] = lines
        out["group_ms_device_median"] = {"without_flag": statistics.median(dev[0]), "with_flag": statistics.median(dev[capi.F_LINE_RECORDS])}
        out["group_ms_wall_median"] = {"without_flag": statistics.median(walls[0]), "with_flag": statistics.median(walls[capi.F_LINE_RECORDS])}
        out["group_ms_wall_all"] = {"without_flag": walls[0], "with_flag": walls[capi.F_LINE_RECORDS]}
        out["line_records_extra_ms_device"] = out["group_ms_device_median"]["with_flag"] - out["group_ms_device_median"]["without_flag"]
        out["line_records_extra_ms_wall"] = out["group_ms_wall_median"]["with_flag"] - out["group_ms_wall_median"]["without_flag"]
        # counted bytes: a 16-byte request out and a 64-byte row back per line (most of them between GPUs)
        out["line_records_bytes"] = int(sum(lines)) * (16 + 64)
        # the last grouping had the flag: format every rank's lines on its GPU, then the whole text through one buffer
        L = m._L
        per_rank = []
        for r in range(world):
            h = L.rk_multi_ctx(m._h, r)
            ms, nbytes, t0 = 0.0, 0, time.perf_counter()
            for s in range(0, lines[r], capi.FORMAT_MAX_LINES):
                t = capi._Text()
                rc = L.rk_dist_format_lines(h, s, min(capi.FORMAT_MAX_LINES, lines[r] - s), C.byref(t))
                assert rc == 0, L.rk_last_error(h)
                ms += t.ms_device
                nbytes += t.n_bytes
            per_rank.append({"rank": r, "lines": lines[r], "bytes": nbytes, "ms_device": ms, "ms_wall": (time.perf_counter() - t0) * 1e3})
        out["format_per_rank"] = per_rank
        t0 = time.perf_counter()
        text = m.format_lines(0, sum(lines))
        out["multi_format_all_lines_ms_wall"] = (time.perf_counter() - t0) * 1e3
        out["multi_format_all_lines_ms_device_max_rank_sum"] = m.ms_format
        out["text_bytes"] = len(text)
    return out


def time_cli(n, devices, reps):
    from oracle import oracle as O
    w = gen.scaled(gen.WORKLOADS["c2"], n)
    rec = generate_host(w)
    res = {"fragments": n, "devices": ",".join(str(d) for d in devices)}
    with tempfile.TemporaryDirectory() as d:
        inp = os.path.join(d, "in.csv")
        O.write_input_csv(inp, rec, w.lx, w.ly)
        res["input_bytes"] = os.path.getsize(inp)
        runs = {"device": [], "host": []}
        md5 = {}
        for _ in range(reps):   # alternating
            for writer in ("device", "host"):
                env = dict(os.environ, RK_TIMING="1", RK_DEVICES=res["devices"])
                if writer == "host":
                    env["RK_LEGACY_WRITER"] = "1"
                outp = os.path.join(d, f"out_{writer}.csv")
                t0 = time.perf_counter()
                p = subprocess.run([CLI, inp, outp, "0.05", "0.05"], capture_output=True, env=env)
                wall = time.perf_counter() - t0
                assert p.returncode == 0, p.stderr.decode()[-2000:]
                with open(outp, "rb") as f:
                    md5[writer] = hashlib.md5(f.read()).hexdigest()
                runs[writer].append({"wall_s": wall, "stderr": [ln for ln in p.stderr.decode().splitlines() if ln.startswith("[rk]")]})
                os.remove(outp)
        res["runs"] = runs
        res["wall_s_median"] = {k: statistics.median(x["wall_s"] for x in v) for k, v in runs.items()}
        res["same_bytes"] = md5["device"] == md5["host"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-per-gpu", type=int, default=10_000_000)
    ap.add_argument("--worlds", default="2,8")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cli-n", type=int, default=5_000_000, help="fragments of the CLI input (0: skip the CLI)")
    ap.add_argument("--cli-reps", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures on the GPU")
    n_gpus = torch.cuda.device_count()
    doc = {"card": card(), "gpus": n_gpus, "worlds": []}
    for world in (int(x) for x in a.worlds.split(",")):
        doc["worlds"].append(time_world(world, a.n_per_gpu, a.reps, n_gpus))
        print(json.dumps(doc["worlds"][-1])[:400], file=sys.stderr, flush=True)
    if a.cli_n:
        doc["cli"] = time_cli(a.cli_n, list(range(min(n_gpus, 8))) if n_gpus > 1 else [0, 0, 0], a.cli_reps)
    text = json.dumps(doc, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
