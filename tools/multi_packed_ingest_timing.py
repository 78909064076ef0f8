"""Compact ingest over several GPUs (tooling): rk_dist_load_packed against rk_dist_load_aos on the same comparison, config
2 at --per-rank fragments per rank, alternating step by step.  A step is one load from pinned host slices + rk_dist_group
with host results (RK_F_HOST_RESULT), timed by the host clock (both calls end in a stream synchronisation); the output
checksum is computed after the timed window.

    python tools/multi_packed_ingest_timing.py [--per-rank 10000000] [--ranks 2,3] [--steps 5] [--modes threads,torchrun] [--out FILE]

* threads: the ranks are threads of rk_create_multi, each calling rk_dist_load_* / rk_dist_group on its context from its
  own host thread.  With as many distinct GPUs as ranks the ranks are those GPUs; otherwise they are threads on GPU 0, which
  share its one PCIe link and its SMs, and the output marks them so.
* torchrun: one process per GPU (python -m torch.distributed.run --standalone), NCCL between them; only rank counts up to
  the number of GPUs run, the others are recorded as not measured.
Every step's group count and output checksum (the sum of multi.output_checksum over the ranks' ranges) must be equal
between the two loads.  The H2D bytes per rank are the arrays each load copies: 33 B per fragment against 109 B.  The card
name and power limit are read in the same run and stored with the numbers.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from repkiller_b200 import capi, gen, multi  # noqa: E402


def cards():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return [ln for ln in q.stdout.strip().split("\n") if ln]


def pinned(nbytes: int) -> np.ndarray:
    import torch
    return torch.empty(max(nbytes, 1), dtype=torch.uint8, pin_memory=True).numpy()[:nbytes]


class Slice:
    """records lo .. hi of the file in pinned host memory, as 109-byte records and as the compact arrays"""

    def __init__(self, w, lo: int, hi: int):
        self.lo, self.n = lo, hi - lo
        self.aos, self.key4, self.strand, self.rest4 = pinned(self.n * 109), pinned(self.n * 16), pinned(self.n), pinned(self.n * 16)
        step = 1 << 22
        for a in range(0, self.n, step):  # (generated in chunks: the whole slice never exists twice in pageable memory)
            b = min(self.n, a + step)
            rec = gen.generate(w, start=lo + a, count=b - a)
            self.aos[a * 109:b * 109] = np.ascontiguousarray(rec).view(np.uint8).reshape(-1)
            k, s, r = capi.pack_records(rec)
            self.key4[a * 16:b * 16], self.strand[a:b], self.rest4[a * 16:b * 16] = k.view(np.uint8).reshape(-1), s, r.view(np.uint8).reshape(-1)

    def part(self, lo: int, hi: int) -> "Slice":
        """records lo .. hi of the file, a view of this slice's arrays"""
        p = Slice.__new__(Slice)
        a, b = lo - self.lo, hi - self.lo
        p.lo, p.n = lo, hi - lo
        p.aos, p.key4, p.strand, p.rest4 = self.aos[a * 109:b * 109], self.key4[a * 16:b * 16], self.strand[a:b], self.rest4[a * 16:b * 16]
        return p

    def load(self, L, h, packed: bool, lx1: int, ly1: int) -> int:
        if packed:
            return L.rk_dist_load_packed(h, C.c_void_p(self.key4.ctypes.data), C.c_void_p(self.strand.ctypes.data),
                                         C.c_void_p(self.rest4.ctypes.data), self.n, self.lo, lx1, ly1, 0, None)
        return L.rk_dist_load_aos(h, C.c_void_p(self.aos.ctypes.data), self.n, self.lo, lx1, ly1, 0, None)


def group(L, h, w):
    """rk_dist_group with host results on one rank: (status, n_groups, its lines (views of the pinned result, valid until
    the rank's next grouping), their line offset)"""
    r, info = capi._Result(), capi._DistInfo()
    rc = L.rk_dist_group(h, w.len_ratio, w.pos_ratio, capi.F_HOST_RESULT, C.byref(r), C.byref(info))
    return (rc, 0, None, 0) if rc else (0, int(r.n_groups), capi._groups_of(r, True, False), int(info.line_offset))


def checksum(g, line_offset: int) -> int:
    """(after the timed window) the checksum of one rank's range of lines"""
    return multi.output_checksum(g.order, g.gid, g.repval, g.identity, line_offset)


def summary(steps: dict, n_rank: list) -> dict:
    out = {}
    for name in ("packed", "aos"):
        ms = [s["ms"] for s in steps[name]]
        out[name] = {"median_ms": round(statistics.median(ms), 2), "ms": ms,
                     "h2d_bytes_per_rank": [n * (33 if name == "packed" else 109) for n in n_rank]}
    keys = {(s["n_groups"], s["checksum"]) for name in ("packed", "aos") for s in steps[name]}
    out["groups_and_checksums_equal"] = len(keys) == 1
    out["n_groups"], out["checksum"] = [list(k) for k in keys][0] if len(keys) == 1 else (None, None)
    out["packed_over_aos"] = round(out["packed"]["median_ms"] / out["aos"]["median_ms"], 3)
    return out


def run_threads(k: int, per_rank: int, n_steps: int, n_gpus: int) -> dict:
    distinct = n_gpus >= k
    devices = list(range(k)) if distinct else [0] * k
    w = gen.scaled(gen.WORKLOADS["c2"], per_rank * k)
    whole = Slice(w, 0, w.n)
    sl = [whole.part(*multi.slice_bounds(w.n, r, k)) for r in range(k)]   # (rk_multi_load_aos's slices)
    run = {"mode": "threads", "ranks": k, "devices": devices, "distinct_gpus": distinct, "fragments": w.n}
    if not distinct:
        run["note"] = "ranks are threads on GPU 0 sharing one PCIe link and one GPU's SMs; distinct-GPU numbers: not measured"
    steps = {"packed": [], "aos": []}
    with capi.Multi(devices) as m:
        L = m._L
        hs = [L.rk_multi_ctx(m._h, r) for r in range(k)]
        # rk_multi_load_aos sizes and maps the ranks' buffers; then one warm-up step of each load, and the timed steps
        assert L.rk_multi_load_aos(m._h, C.c_void_p(whole.aos.ctypes.data), w.n, w.lx + 1, w.ly + 1, 0, None) == 0
        with ThreadPoolExecutor(k) as ex:
            for i in range(2 * (n_steps + 1)):
                packed = i % 2 == 0
                t0 = time.perf_counter()
                rcs = list(ex.map(lambda r: sl[r].load(L, hs[r], packed, w.lx + 1, w.ly + 1), range(k)))
                gr = list(ex.map(lambda r: group(L, hs[r], w), range(k)))
                ms = (time.perf_counter() - t0) * 1e3
                assert rcs == [0] * k and all(g[0] == 0 for g in gr), [L.rk_last_error(h) for h in hs]
                if i >= 2:
                    steps["packed" if packed else "aos"].append({"ms": round(ms, 2), "n_groups": gr[0][1],
                                                                 "checksum": sum(checksum(g[2], g[3]) for g in gr) & ((1 << 64) - 1)})
    run.update(summary(steps, [s.n for s in sl]))
    return run


def worker(a):
    """one process of the torchrun mode: this rank's slice, alternating steps; rank 0 writes the run to a.part"""
    import torch
    import torch.distributed as dist
    dist.init_process_group("gloo")
    rank, k = dist.get_rank(), dist.get_world_size()
    torch.cuda.set_device(rank)
    w = gen.scaled(gen.WORKLOADS["c2"], a.per_rank * k)
    lo, hi = multi.slice_bounds(w.n, rank, k)
    s = Slice(w, lo, hi)
    ctx = capi.Context(rank)
    multi.bootstrap(ctx, multi.default_capacity(w.n // k + 16))
    L, h = ctx._L, ctx._h
    steps = {"packed": [], "aos": []}
    for i in range(2 * (a.steps + 1)):
        packed = i % 2 == 0
        dist.barrier()
        t0 = time.perf_counter()
        rc = s.load(L, h, packed, w.lx + 1, w.ly + 1)
        assert rc == 0, L.rk_last_error(h)
        rc, n_groups, g, line_offset = group(L, h, w)
        assert rc == 0, L.rk_last_error(h)
        ms = (time.perf_counter() - t0) * 1e3
        cs = checksum(g, line_offset)
        box = [None] * k
        dist.all_gather_object(box, (ms, cs))
        if i >= 2:
            steps["packed" if packed else "aos"].append({"ms": round(max(b[0] for b in box), 2), "n_groups": n_groups,
                                                         "checksum": sum(b[1] for b in box) & ((1 << 64) - 1)})
    ns = [None] * k
    dist.all_gather_object(ns, s.n)
    if rank == 0:
        run = {"mode": "torchrun", "ranks": k, "devices": list(range(k)), "distinct_gpus": True, "fragments": w.n,
               "note": "step time = the slowest rank's"}
        run.update(summary(steps, ns))
        with open(a.part, "w") as f:
            json.dump(run, f)
    dist.barrier()
    ctx.close()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--per-rank", type=int, default=10_000_000)
    ap.add_argument("--ranks", default="2,3")
    ap.add_argument("--steps", type=int, default=5, help="timed steps of each load, alternating, after one warm-up each")
    ap.add_argument("--modes", default="threads,torchrun")
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--part", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        return worker(a)
    import torch
    n_gpus = torch.cuda.device_count()
    res = {"cards": cards(), "gpus": n_gpus, "config": "c2", "fragments_per_rank": a.per_rank, "runs": []}

    def save():
        if a.out:  # after every run: a cut-short run keeps what it measured
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                f.write(json.dumps(res, indent=1) + "\n")

    ranks = [int(x) for x in a.ranks.split(",")]
    modes = a.modes.split(",")
    if "threads" in modes:
        for k in ranks:
            res["runs"].append(run_threads(k, a.per_rank, a.steps, n_gpus))
            print(json.dumps(res["runs"][-1]), flush=True)
            save()
    if "torchrun" in modes:
        for k in sorted(set([1] + ranks)):
            if k > n_gpus:
                res["runs"].append({"mode": "torchrun", "ranks": k, "measured": False,
                                    "note": f"not measured: one process per GPU needs {k} GPUs, the box has {n_gpus}"})
                continue
            part = os.path.join(tempfile.mkdtemp(prefix="multi_packed_"), "run.json")
            p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--standalone", f"--nproc_per_node={k}", __file__,
                                "--worker", "--per-rank", str(a.per_rank), "--steps", str(a.steps), "--part", part],
                               capture_output=True, text=True)
            assert p.returncode == 0, p.stderr[-4000:]
            with open(part) as f:
                res["runs"].append(json.load(f))
            print(json.dumps(res["runs"][-1]), flush=True)
            save()
    save()


if __name__ == "__main__":
    main()
