"""K8 timing (tooling): the device time of rk_group_statistics (k_stats_init + k_group_stats + k_stats_final, one
profiler scope: KID_STATS, reported as "k_group_stats") at C2 and C3 on one GPU, for this tree's library and for other
builds of it, alternating, each in its own process.

    python tools/group_stats_timing.py [--variants "",_parent] [--rounds 2] [--reps 20] [--out FILE]

A variant is an RK_LIB_SUFFIX: "" is repkiller_b200/librk_b200.so, "_parent" repkiller_b200/librk_b200_parent.so (a
library built from another commit and copied there).  The records are generated on the device, loaded and grouped once;
then --reps calls of rk_group_statistics without the host copy, after two warm-up calls.  The card name and power limit
are read in the same run and stored with the numbers.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().split("\n")[0]


def child(reps: int) -> dict:
    import torch
    from repkiller_b200 import capi, gen
    out = {}
    with capi.Context(0) as ctx:
        for wl in ("c2", "c3"):
            w = gen.WORKLOADS[wl]
            buf = torch.empty(w.n * 109, dtype=torch.uint8, device="cuda:0")
            ctx.generate_device(w, 0, w.n, buf.data_ptr())
            torch.cuda.synchronize()
            ctx.load(buf.data_ptr(), w.lx + 1, w.ly + 1, n=w.n, timing=False)
            res = ctx.group(w.len_ratio, w.pos_ratio, host_result=False, timing=False)
            ng = C.c_uint64()

            def stats():
                rc = ctx._L.rk_group_statistics(ctx._h, 0, None, None, C.byref(ng))
                if rc:
                    raise capi.RkError(rc, ctx._L.rk_last_error(ctx._h).decode())
            stats(), stats()
            ctx.profile_enable(True)
            ctx.profile_read(reset=True)
            for _ in range(reps):
                stats()
            prof = ctx.profile_read(reset=True)
            ctx.profile_enable(False)
            launches, ms, units = prof["k_group_stats"]
            out[wl] = {"n_lines": res.n_kept, "n_groups": int(ng.value), "calls": reps, "launches": launches,
                       "ms_per_call": ms / reps}
            del buf
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--variants", default=",_parent")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        print(json.dumps(child(a.reps)))
        return
    runs = []
    for r in range(a.rounds):
        for v in a.variants.split(","):
            env = dict(os.environ, RK_LIB_SUFFIX=v)
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--reps", str(a.reps)], env=env,
                               capture_output=True, text=True, check=True)
            res = json.loads(p.stdout.strip().splitlines()[-1])
            runs.append({"round": r, "variant": v or "(this tree)", **res})
            print(json.dumps(runs[-1]), flush=True)
    rec = {"card": card(), "runs": runs}
    if a.out:
        with open(a.out, "w") as f:
            json.dump(rec, f, indent=1)
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
