"""CSV ingest over several GPUs (tooling): rk_multi_load_csv on config 2 scaled to --per-rank rows per rank, written once as
a GECKO CSV, and the CLI of this tree against another tree's CLI under RK_DEVICES, alternating, with identical output bytes.

    python tools/multi_csv_ingest_timing.py [--per-rank 10000000] [--ranks 2,4,8] [--parent-cli PATH] [--out FILE]

* rk_multi_load_csv: three calls on one rk_multi per rank count; upload and parse are the largest rank's device times
  (rk_csv_stats), call the host wall clock of the whole call (local halves, capacity, count exchange, emit, partitioned load);
* per rank: three rounds of rk_dist_load_csv on the same ranks' contexts (rk_multi_ctx), one host thread per rank, each on
  the slice rk_multi_load_csv cuts for it: every rank's upload and parse device times and its rows;
* CLI: `RK_DEVICES=<the ranks' devices> RK_TIMING=1 repkiller` of this tree and of the other tree alternating, --reps runs
  each: wall clock, the `[rk] loaded=` line and the output md5 (the other tree parses the rows on the host cores).
With as many distinct GPUs as ranks the ranks are those GPUs.  Otherwise the ranks are threads on GPU 0, which share its one
PCIe link and its SMs: such numbers say nothing about distinct GPUs, and the output marks them so.
The card name and power limit are read in the same run and stored with the numbers.
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from oracle import oracle as O  # noqa: E402
from repkiller_b200 import capi, gen  # noqa: E402

BIN = os.path.join(ROOT, "repkiller_b200", "bin")


def cards():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return [ln for ln in q.stdout.strip().split("\n") if ln]


def split_head(text: bytes):
    pos = 0
    lines = []
    for _ in range(16):
        nl = text.find(b"\n", pos)
        lines.append(text[pos:len(text) if nl < 0 else nl])
        pos = len(text) if nl < 0 else nl + 1
    return text[pos:], int(lines[12].split(b":")[1])


def cuts(body: bytes, k: int):
    """rk_multi_load_csv's cuts: one byte past the first newline at or after len(body) * r / k"""
    out = [0]
    for r in range(1, k):
        nl = body.find(b"\n", len(body) * r // k)
        out.append(len(body) if nl < 0 else nl + 1)
    return out + [len(body)]


def per_rank(m, body: bytes, lx1: int, ly1: int, total: int):
    """one rk_dist_load_csv round on the ranks of m: every rank's csv stats and the round's wall clock"""
    L = m._L
    hs = [L.rk_multi_ctx(m._h, r) for r in range(m.n)]
    c = cuts(body, m.n)
    parts = [np.frombuffer(body, dtype=np.uint8, count=c[r + 1] - c[r], offset=c[r]) for r in range(m.n)]
    st = [capi._LoadStats() for _ in hs]
    cs = [capi._CsvStats() for _ in hs]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(m.n) as ex:
        rcs = list(ex.map(lambda r: L.rk_dist_load_csv(hs[r], C.c_void_p(parts[r].ctypes.data) if parts[r].size else None,
                                                         parts[r].size, lx1, ly1, total, capi.F_TIMING, C.byref(st[r]),
                                                         C.byref(cs[r])), range(m.n)))
    wall = (time.perf_counter() - t0) * 1e3
    assert rcs == [0] * m.n, [L.rk_last_error(h) for h in hs]
    return {"wall_ms": round(wall, 2), "ranks": [{"bytes": int(parts[r].size), "upload_ms": cs[r].ms_upload, "parse_ms": cs[r].ms_parse,
                                                  "n_rows": cs[r].n_rows, "n_host_rows": cs[r].n_host_rows, "wide": cs[r].wide}
                                                 for r in range(m.n)]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--per-rank", type=int, default=10_000_000)
    ap.add_argument("--ranks", default="2,4,8")
    ap.add_argument("--parent-cli", default=None, help="the other tree's repkiller binary")
    ap.add_argument("--reps", type=int, default=2, help="CLI runs per tree, alternating")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    n_gpus = torch.cuda.device_count()
    res = {"cards": cards(), "gpus": n_gpus, "config": "c2", "rows_per_rank": a.per_rank, "runs": []}
    tmp = tempfile.mkdtemp(prefix="multi_csv_ingest_")
    for k in [int(x) for x in a.ranks.split(",")]:
        distinct = n_gpus >= k
        devices = list(range(k)) if distinct else [0] * k
        w = gen.scaled(gen.WORKLOADS["c2"], a.per_rank * k)
        inp = os.path.join(tmp, "in.csv")
        O.write_input_csv(inp, gen.generate(w), w.lx, w.ly)
        text = open(inp, "rb").read()
        body, total = split_head(text)
        run = {"ranks": k, "devices": devices, "distinct_gpus": distinct, "rows": w.n, "csv_bytes": len(text)}
        if not distinct:
            run["note"] = "ranks are threads on GPU 0 sharing one PCIe link and one GPU's SMs; distinct-GPU numbers: not measured"
        calls = []
        with capi.Multi(devices) as m:
            for _ in range(3):
                t0 = time.perf_counter()
                st, cs = m.load_csv(body, w.lx + 1, w.ly + 1, total, timing=True)
                wall = (time.perf_counter() - t0) * 1e3
                calls.append({"upload_ms_max": cs.ms_upload, "parse_ms_max": cs.ms_parse, "call_ms": round(wall, 2),
                              "n_rows": cs.n_rows, "n_host_rows": cs.n_host_rows, "wide": cs.wide, "n_loaded": st.n_loaded})
            run["rk_dist_load_csv_per_rank"] = [per_rank(m, body, w.lx + 1, w.ly + 1, total) for _ in range(3)]
        run["rk_multi_load_csv"] = calls
        del text, body
        clis = [("this", os.path.join(BIN, "repkiller"))] + ([("parent", a.parent_cli)] if a.parent_cli else [])
        runs, digests = [], set()
        env = dict(os.environ, RK_TIMING="1", RK_DEVICES=",".join(map(str, devices)))
        for rep in range(a.reps):
            for name, cli in clis:
                outp = os.path.join(tmp, f"out_{name}.csv")
                t0 = time.perf_counter()
                p = subprocess.run([cli, inp, outp, str(w.len_ratio), str(w.pos_ratio)], capture_output=True, text=True, env=env)
                wall = time.perf_counter() - t0
                assert p.returncode == 0, p.stderr
                digests.add(hashlib.md5(open(outp, "rb").read()).hexdigest())
                load_line = next(ln for ln in p.stderr.splitlines() if ln.startswith("[rk] loaded="))
                runs.append({"tree": name, "rep": rep, "wall_s": round(wall, 3), "load_line": load_line})
                os.unlink(outp)
        run["cli"] = runs
        run["cli_outputs_identical"] = len(digests) == 1
        run["cli_md5"] = sorted(digests)
        os.unlink(inp)
        res["runs"].append(run)
        print(json.dumps(run, indent=1), flush=True)
        if a.out:   # after every rank count: a cut-short run keeps what it measured
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
