"""CSV ingest timing (tooling): the host parser against rk_load_csv on a generated GECKO CSV, and the CLI of this tree
against another tree's CLI, alternating, with identical output bytes.

    python tools/csv_ingest_timing.py [--n 10000000] [--parent-cli PATH] [--out FILE]

* host route: `RK_TIMING=1 rk_hostcheck ingest` (read_frags_head + read_frags_records on all cores: the parse the CLI
  made before rk_load_csv), three runs;
* rk_load_csv: three calls on one context; upload and parse are device times (rk_csv_stats), load the rk_load_stats
  device time, call the host wall clock of the whole call.  Bytes/s of the parse count what the kernels must move: the
  text three times (newline count, classify, emit) and per row the start offset (written once, read twice), the status
  byte (written, read twice), the slot word (written, read) and the 33 bytes of compact arrays;
* CLI: this tree's and the other tree's `repkiller` alternating, --reps runs each, wall clock and the `[rk] loaded=` line.
The card name and power limit are read in the same run and stored with the numbers.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import oracle as O  # noqa: E402
from repkiller_b200 import capi, gen  # noqa: E402

BIN = os.path.join(ROOT, "repkiller_b200", "bin")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().split("\n")[0]


def split_head(text: bytes):
    pos = 0
    lines = []
    for _ in range(16):
        nl = text.find(b"\n", pos)
        lines.append(text[pos:len(text) if nl < 0 else nl])
        pos = len(text) if nl < 0 else nl + 1
    return text[pos:], int(lines[12].split(b":")[1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=10_000_000)
    ap.add_argument("--parent-cli", default=None, help="the other tree's repkiller binary")
    ap.add_argument("--reps", type=int, default=2, help="CLI runs per tree, alternating")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = {"card": card(), "rows": a.n, "config": "c2"}
    w = gen.scaled(gen.WORKLOADS["c2"], a.n)
    tmp = tempfile.mkdtemp(prefix="csv_ingest_")
    inp = os.path.join(tmp, "in.csv")
    O.write_input_csv(inp, gen.generate(w), w.lx, w.ly)
    text = open(inp, "rb").read()
    body, total = split_head(text)
    res["csv_bytes"] = len(text)

    host = []
    for _ in range(3):
        p = subprocess.run([os.path.join(BIN, "rk_hostcheck"), "ingest", inp, os.path.join(tmp, "r.bin"), os.path.join(tmp, "r.hdr")],
                           capture_output=True, text=True, env=dict(os.environ, RK_TIMING="1"))
        assert p.returncode == 0, p.stderr
        host.append(float(re.search(r"records_ms=([\d.]+)", p.stderr).group(1)))
    res["host_parse_ms"] = host
    res["host_cores"] = os.cpu_count()

    calls = []
    with capi.Context(0) as ctx:
        for _ in range(3):
            t0 = time.perf_counter()
            st, cs = ctx.load_csv(body, w.lx + 1, w.ly + 1, total)
            wall = (time.perf_counter() - t0) * 1e3
            moved = 3 * len(body) + cs.n_rows * (3 * 8 + 3 + 2 * 4 + 33)
            calls.append({"upload_ms": cs.ms_upload, "parse_ms": cs.ms_parse, "load_device_ms": st.ms_device, "call_ms": wall,
                          "n_rows": cs.n_rows, "n_host_rows": cs.n_host_rows, "wide": cs.wide,
                          "upload_GBps": len(body) / cs.ms_upload / 1e6 if cs.ms_upload else None,
                          "parse_alg_bytes": moved, "parse_GBps": moved / cs.ms_parse / 1e6 if cs.ms_parse else None})
    res["rk_load_csv"] = calls

    clis = [("this", os.path.join(BIN, "repkiller"))] + ([("parent", a.parent_cli)] if a.parent_cli else [])
    runs, digests = [], set()
    for rep in range(a.reps):
        for name, cli in clis:
            outp = os.path.join(tmp, f"out_{name}.csv")
            t0 = time.perf_counter()
            p = subprocess.run([cli, inp, outp, str(w.len_ratio), str(w.pos_ratio)], capture_output=True, text=True,
                               env=dict(os.environ, RK_TIMING="1"))
            wall = time.perf_counter() - t0
            assert p.returncode == 0, p.stderr
            digests.add(hashlib.md5(open(outp, "rb").read()).hexdigest())
            load_line = next(ln for ln in p.stderr.splitlines() if ln.startswith("[rk] loaded="))
            runs.append({"tree": name, "rep": rep, "wall_s": round(wall, 3), "load_line": load_line})
            os.unlink(outp)
    res["cli"] = runs
    res["cli_outputs_identical"] = len(digests) == 1
    res["cli_md5"] = sorted(digests)
    os.unlink(inp)
    out = json.dumps(res, indent=1)
    print(out)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
