#!/usr/bin/env python
"""bench.py — fragments grouped per second on B200 (BASELINE.json metric), the reference's CPU path beside it.

A "step" is one pass of the whole hot path over one synthetic comparison of the named workload shape:
rk_load_aos (K1 decode, K2 processing-order and occupation-bucket sorts) + rk_group (K3 X/Y passes, K4 forest,
K5 diag/sort/labels) for len_ratio = pos_ratio = 0.05.
  value : records already resident in HBM, result left in HBM; CUDA events on the launching stream.
  e2e   : the same step through the C ABI with HOST buffers: pinned records -> H2D -> kernels -> D2H of
          order/gid/repval/identity into pinned host arrays.
N > 1: one process per GPU (torchrun).  Default: ONE comparison of N x the per-GPU size, partitioned over the GPUs inside
the library (rk_dist_*: range partition by xStart/10, X pass at home with a halo, Y exchange, forest over peer memory,
output exchange; NCCL over NVLink; weak scaling: per-GPU fragments fixed).  Its checksum is printed next to the checksum
of the SAME comparison grouped on one GPU (outside the timed region).  --multi independent: one independent
sequence-pair comparison per GPU.
`--impl reference` times the reference's own CPU code (oracle/_ref, built from /root/reference) on host cores.
`--dump-outputs DIR` (one GPU) writes what the last timed step left in HBM, as DIR/<name>.npy, so that two builds can be
compared output for output on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from dataclasses import replace

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "fragments grouped/sec (device-timed)"
UNIT = "fragments/s"
CPU_SAMPLE_N = 1_000_000
# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` captures (profiles/)
NCU_TRAFFIC = {  # profiles/r02_ncu_full_top_kernels.json (C2, 10M fragments), mean over the captured launches
    "k_radix_scatter": 98700000, "k_match_small": 441900000, "k_keys": 947500000, "k_decode": 1428600000,
    "k_order_tile": 416200000, "k_hkey": 313600000, "k_chase": 118700000, "k_groupsort_warp": 133600000,
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2")
    ap.add_argument("--n", "--frags", dest="n", type=int, default=0, help="override the fragment count (same shape, scaled); testing only")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--total-n", type=float, default=0, help="partitioned mode: total fragments of the one comparison (e.g. 1e9)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (very large slices)")
    ap.add_argument("--checksum", type=int, default=1, help="position-dependent checksum of the whole output; N > 1: also of the same comparison on one GPU")
    ap.add_argument("--multi", default="partitioned", choices=["partitioned", "independent"],
                    help="N > 1: one comparison range-partitioned over the GPUs (default) or one independent comparison per GPU")
    ap.add_argument("--profile-kernels", type=int, default=1, help="CUDA-event pairs around every kernel launch in the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the output arrays of the last timed step to DIR/<name>.npy (float32/float64; our arm on one GPU only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the output of our arm; the reference arm writes none")
    return args


def workload(args, rank=0):
    from repkiller_b200 import gen
    w = gen.WORKLOADS[args.workload]
    if args.n:
        w = gen.scaled(w, args.n)
    if rank:
        w = replace(w, seed=w.seed + 1000 * rank)  # another sequence pair of the same shape
    return w


def workload_text(w):
    return (f"{w.name}: {w.n:,} synthetic fragments, {w.lx / 1e6:g} Mbp x {w.ly / 1e6:g} Mbp, {int(w.p_rep * 100)}% repeat-family "
            f"fragments in {w.families} families, len_ratio={w.len_ratio} pos_ratio={w.pos_ratio}")


# ---------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own CPU implementation on the host cores
# ---------------------------------------------------------------------------------------------------------
def cpu_reference_run(w_sample, steps, warmup):
    """Times generate_fragment_groups + generate_diagonal_func + sort_groups of the compiled reference
    (oracle/_ref/repkiller_ref) — or of the oracle port when the reference binary is absent — on a bounded
    sample.  Returns (fragments/s, kind, per-step ms list)."""
    from repkiller_b200 import gen
    from oracle import oracle as O
    rec = gen.generate(w_sample)
    times = []
    if O.have_ref():
        kind = "reference"
        tmp = tempfile.mkdtemp(prefix="rkbench")
        inp = os.path.join(tmp, "in.csv")
        O.write_input_csv(inp, rec, w_sample.lx, w_sample.ly)
        for i in range(warmup + steps):
            info = O.run_ref(inp, os.path.join(tmp, "out.csv"), w_sample.len_ratio, w_sample.pos_ratio, nosave=True)
            if i >= warmup:
                times.append(info["group_ms"] + info["diag_ms"] + info["sort_ms"])
        os.remove(inp)
    else:
        kind = "port"
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            O.group(rec, w_sample.lx + 1, w_sample.ly + 1, w_sample.len_ratio, w_sample.pos_ratio)
            if i >= warmup:
                times.append((time.perf_counter() - t0) * 1e3)
    ms = sum(times) / len(times)
    return w_sample.n / (ms / 1e3), kind, times


REF_ARM_BUDGET_S = float(os.environ.get("RK_REF_ARM_BUDGET_S", "600"))   # wall-clock bound of the timed repetitions
REF_ARM_MAX_N = int(os.environ.get("RK_REF_ARM_MAX_N", "20000000"))       # largest comparison the host leg builds (CSV + RAM)


def reference_full_run(w, steps, warmup, budget_s):
    """The compiled, unmodified reference on the WHOLE workload w: the CSV is loaded once (FragmentsDatabase), then
    generate_fragment_groups + generate_diagonal_func + sort_groups are repeated warmup + steps times on one core
    (oracle/ref_driver.cpp, RK_REF_REPEAT).  Returns the per-repetition ms list of the timed repetitions, the number of
    warm-up repetitions that ran, and the load time."""
    from repkiller_b200 import gen
    from oracle import oracle as O
    tmp = tempfile.mkdtemp(prefix="rkbench")
    inp = os.path.join(tmp, "in.csv")
    t0 = time.perf_counter()
    chunk = 2_000_000
    with open(inp, "wb") as f:   # written in chunks: the records of a 10M-fragment comparison are 1.09 GB
        for c0 in range(0, w.n, chunk):
            part = os.path.join(tmp, "part.csv")
            O.write_input_csv(part, gen.generate(w, start=c0, count=min(chunk, w.n - c0)), w.lx, w.ly)
            with open(part, "rb") as g:
                data = g.read()
            if c0:   # drop the 16 header lines of every part but the first
                pos = 0
                for _ in range(16):
                    pos = data.index(b"\n", pos) + 1
                data = data[pos:]
            else:    # the header announces the fragments of the whole file
                head, body = data.split(b"\n", 16)[:16], data.split(b"\n", 16)[16]
                head[12] = b"Total fragments : %d" % w.n
                data = b"\n".join(head) + b"\n" + body
            f.write(data)
            os.remove(part)
    gen_s = time.perf_counter() - t0
    env = dict(os.environ, RK_REF_NOSAVE="1", RK_REF_REPEAT=str(warmup + steps), RK_REF_BUDGET_S=str(budget_s))
    p = subprocess.run([O.REF_BIN, inp, os.path.join(tmp, "out.csv"), repr(w.len_ratio), repr(w.pos_ratio)], env=env,
                       capture_output=True)
    os.remove(inp)
    if p.returncode != 0:
        raise RuntimeError(f"repkiller_ref rc={p.returncode}: {p.stderr[-400:]!r}")
    infos = [json.loads(ln) for ln in p.stderr.decode().strip().splitlines() if ln.startswith("{")]
    times = [i["group_ms"] + i["diag_ms"] + i["sort_ms"] for i in infos]
    n_warm = min(warmup, max(0, len(times) - 1))
    return times[n_warm:], n_warm, infos[0]["load_ms"], gen_s


def reference_arm(args):
    """The reference's own CPU implementation of the path on the SAME config as our arm (the whole comparison, not a
    sample), one core: the grouping loop is sequential; the reference's three threads only run different ratio pairs."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from repkiller_b200 import gen
    from oracle import oracle as O
    base = workload(args)
    world = max(1, args.gpus)
    w = gen.scaled(base, args.total_n) if args.total_n else (gen.scaled(base, base.n * world) if world > 1 else base)
    capped = w.n > REF_ARM_MAX_N
    wr = gen.scaled(w, REF_ARM_MAX_N) if capped else w
    t0 = time.perf_counter()
    if O.have_ref():
        kind = "reference"
        times, n_warm, load_ms, gen_s = reference_full_run(wr, args.steps, args.warmup, REF_ARM_BUDGET_S)
    else:   # the compiled reference did not travel: the oracle port on the same records
        kind, n_warm, load_ms, gen_s = "port", 0, 0.0, 0.0
        rec = gen.generate(wr)
        times = []
        for i in range(args.warmup + args.steps):
            t1 = time.perf_counter()
            O.group(rec, wr.lx + 1, wr.ly + 1, wr.len_ratio, wr.pos_ratio)
            if i >= args.warmup:
                times.append((time.perf_counter() - t1) * 1e3)
            if time.perf_counter() - t0 > REF_ARM_BUDGET_S and times:
                break
    ms = sum(times) / len(times)
    value = wr.n / (ms / 1e3)
    sample = (f"the whole comparison ({wr.n:,} fragments, {wr.lx / 1e6:g} Mbp x {wr.ly / 1e6:g} Mbp), loaded once, "
              f"generate_fragment_groups + generate_diagonal_func + sort_groups repeated {len(times)} times "
              f"(+{n_warm} warm-up), CSV parse/format excluded")
    if capped:
        sample = (f"CAPPED: our arm groups {w.n:,} fragments, the host leg {wr.n:,} of the same shape and density "
                  f"(CSV + {wr.n * 330 / 1e9:.0f} GB of host memory bound); " + sample)
    cfg = {"workload": workload_text(w), "reference_workload": workload_text(wr), "sample": sample,
           "steps_timed": len(times), "warmup_run": n_warm,
           "note": None if len(times) == args.steps and n_warm == args.warmup else
           f"the {REF_ARM_BUDGET_S:.0f} s budget ended the loop after {n_warm} warm-up + {len(times)} timed repetitions"}
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
        "warmup": n_warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64+u64", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "load_ms": load_ms, "input_build_s": gen_s, "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                       "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.p = None

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        out, _ = self.p.communicate(timeout=10)
        sm, mx, reasons = [], [], set()
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# Algorithmic HBM bytes per unit a kernel processes (DESIGN.md §4): what it must read and write once.
ALG_BYTES_PER_UNIT = {
    "k_decode": 109 + 36,        # record in; 32-byte {xs, ys, len, flags, identity} record + key0 u32 out
    "k_radix_hist": 4,           # one read of the keys for all digit histograms of a sort
    "k_radix_scatter": 16,       # (key, value) in, (key, value) out, per pass
    "k_keys": 4 + 32 + 32,       # file index, one 32-byte record gather; {c,len} x 2, ys, kx, ky, identity out
    "k_match_small": 20,         # key, rank, {center, length} in, owner out (+ 1 bit per rank of the X-match map)
    "k_chase": 12,
    "k_scan": 12,
    "k_hkey": 16 + 20,           # bucket key, ys, file index, identity in; h + 16-byte {h, fidx, identity} record out
    "k_order_tile": 8 + 16 + 13, # gid, rank, one 16-byte record gather in; four output arrays out
}


DUMP_MAX_LINES = 1 << 20   # --dump-outputs: larger outputs are sampled at this many seeded line positions (32 MB in all)


class _DeviceArray:
    """A 1-D array in the library's device memory, as torch.as_tensor sees it (no copy)."""

    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}


def dump_outputs(out_dir, res, device):
    """The arrays a caller of rk_group receives (order, gid, repval, identity; the last step's device buffers), plus n_kept
    and n_groups, as DIR/<name>.npy.  Integers become float64 (exact), repval and identity float32.  Outputs of more than
    DUMP_MAX_LINES lines are sampled at sorted line positions drawn with a fixed seed from n_kept alone, so two builds that
    agree on n_kept sample the same lines; `line` holds the positions."""
    import numpy as np
    import torch
    m = res.n_kept
    line = np.arange(m, dtype=np.int64)
    if m > DUMP_MAX_LINES:
        line = np.sort(np.random.default_rng(0).choice(m, DUMP_MAX_LINES, replace=False))
    out = {"n_kept": np.array([m], np.float64), "n_groups": np.array([res.n_groups], np.float64), "line": line.astype(np.float64)}
    idx = torch.from_numpy(line).to(device)
    for name, typestr, dt, ft in (("order", "<i4", np.uint32, np.float64), ("gid", "<i4", np.uint32, np.float64),
                                  ("repval", "|u1", np.uint8, np.float32), ("identity", "<f4", np.float32, np.float32)):
        v = np.zeros(0, dt)
        if m:
            t = torch.as_tensor(_DeviceArray(res.d_ptrs[name], m, typestr), device=device)
            v = t[idx].cpu().numpy().view(dt)
        out[name] = v.astype(ft)
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), v)


def ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from repkiller_b200 import capi, gen, multi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the output of one process: run it with one GPU")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    partitioned = world > 1 and args.multi == "partitioned"

    base = workload(args)
    if partitioned:
        # ONE comparison, range-partitioned over the GPUs: world x the per-GPU size of the named shape (same density;
        # weak scaling), or with --total-n exactly that many fragments in all (config 5: --workload c5 --total-n 1e9)
        w = gen.scaled(base, args.total_n) if args.total_n else gen.scaled(base, base.n * world)
        lo, hi = multi.slice_bounds(w.n, rank, world)
        n_total = w.n
    else:
        w = workload(args, rank)   # rank r: its own sequence pair of the same shape
        lo, hi = 0, w.n
        n_total = w.n * world
    n = hi - lo
    lx1, ly1 = w.lx + 1, w.ly + 1
    ctx = capi.Context(local)
    device_generated = n > 20_000_000   # large slices: same bytes from the device generator (tests pin it to gen.py)
    if device_generated:
        dev = torch.empty(n * 109 + 16, dtype=torch.uint8, device=device)
        ctx.generate_device(w, lo, n, dev.data_ptr())
        host = None
    else:
        rec = gen.generate(w, start=lo, count=n)
        host = torch.from_numpy(rec.view(np.uint8).reshape(-1)).pin_memory()
        dev = host.to(device)
    do_e2e = not args.no_e2e
    if host is None and do_e2e:
        host = torch.empty(n * 109, dtype=torch.uint8).pin_memory()
        host.copy_(dev[: n * 109])
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak_gbs, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "fallback (B200_PROFILING.md)")

    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    if partitioned:
        multi.bootstrap(ctx, multi.default_capacity(n_total // world + 16))   # NCCL id + peer-memory handles, once

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        if partitioned:
            st = ctx.dist_load(dev.data_ptr(), n, lo, lx1, ly1)
            return st, ctx.dist_group(w.len_ratio, w.pos_ratio, host_result=False, timing=True)
        st = ctx.load(dev.data_ptr(), lx1, ly1, n=n)
        return st, ctx.group(w.len_ratio, w.pos_ratio, host_result=False)

    # e2e: pinned HOST buffers in, pinned host result out, through the C-ABI calls a C++ caller makes.  Single GPU: the
    # compact ingest the drop-in CLI uses (rk_load_packed: the parser fills {xStart, yStart, length, ident} + strand +
    # {xEnd, yEnd, score, similarity}, 33 B per fragment) — and, reported beside it, the 109-byte record ingest
    # (rk_load_aos).  N > 1: rk_dist_load_aos takes the records.
    packed = None
    if do_e2e and not partitioned:
        from repkiller_b200.frags import FRAG_DTYPE
        k4, sd, r4 = capi.pack_records(host.numpy().view(FRAG_DTYPE))
        packed = [torch.from_numpy(a).pin_memory() for a in (k4, sd, r4)]

    def step_e2e():
        if partitioned:
            st = ctx.dist_load(host.data_ptr(), n, lo, lx1, ly1)
            return st, ctx.dist_group(w.len_ratio, w.pos_ratio, host_result=True, copy=False, timing=True)
        st = ctx.load_packed(packed[0].data_ptr(), packed[1].data_ptr(), packed[2].data_ptr(), lx1, ly1, n=n)
        return st, ctx.group(w.len_ratio, w.pos_ratio, host_result=True, copy=False)   # pinned result buffers, as a C caller sees them

    def step_e2e_aos():
        st = ctx.load(host.data_ptr(), lx1, ly1, n=n)
        return st, ctx.group(w.len_ratio, w.pos_ratio, host_result=True, copy=False)

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            last = None
            for _ in range(k):
                last = fn()
            e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=device, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, last

    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            step_resident()
    # timed region 1: the metric.  K steps bracketed by barrier + synchronize, CUDA events on the launching stream.
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_total, last = timed(step_resident, args.steps)
    # timed region 2: the same K steps again with a CUDA-event pair around every kernel launch (rk_profile_enable).  The
    # ~90 extra event records per step cost about 0.2 ms, so `value` comes from region 1 and the per-kernel durations,
    # the roofline and gpu_launches from region 2; both step times are reported.
    prof, ms_profiled = {}, None
    if args.profile_kernels:
        ctx.profile_enable(True)
        ctx.profile_read(reset=True)
        ms_profiled, last = timed(step_resident, args.steps)
        prof = ctx.profile_read(reset=True)
        ctx.profile_enable(False)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:   # before the e2e and checksum calls below overwrite the result buffers
        dump_outputs(args.dump_outputs, last[1], device)

    if do_e2e:
        with torch.cuda.stream(stream):
            for _ in range(max(1, args.warmup // 2)):
                step_e2e()
        ms_e2e, last_e = timed(step_e2e, args.steps)
        ms_e2e_aos = None
        if not partitioned:
            with torch.cuda.stream(stream):
                step_e2e_aos()
            ms_e2e_aos, _ = timed(step_e2e_aos, args.steps)
    else:
        ms_e2e, ms_e2e_aos = float("nan"), None

    # Checksum of the whole output (position-dependent, 64 bit), outside the timed regions.  N > 1: the sum over the ranks'
    # ranges of lines, and beside it the checksum of the SAME comparison grouped by rank 0 alone on its one GPU
    # (rk_load_aos + rk_group on all N x per-GPU fragments): the two must be equal.
    checksum = checksum_1gpu = None
    if args.checksum:
        with torch.cuda.stream(stream):
            if partitioned:
                st_h = ctx.dist_load(dev.data_ptr(), n, lo, lx1, ly1)
                res_h, info_h = ctx.dist_group(w.len_ratio, w.pos_ratio, host_result=True)
                cs_local = multi.output_checksum(res_h.order, res_h.gid, res_h.repval, res_h.identity, info_h["line_offset"])
                halves = torch.tensor([cs_local & 0xFFFFFFFF, cs_local >> 32], dtype=torch.int64, device=device)
                dist.all_reduce(halves)
                lo32, hi32 = int(halves[0].item()), int(halves[1].item())
                checksum = (lo32 + (hi32 << 32)) & ((1 << 64) - 1)
                if rank == 0 and n_total * 450 < 150e9:   # the whole comparison fits one B200
                    ctx1 = capi.Context(local)
                    whole = torch.empty(n_total * 109 + 16, dtype=torch.uint8, device=device)
                    ctx1.generate_device(w, 0, n_total, whole.data_ptr())
                    ctx1.load(whole.data_ptr(), lx1, ly1, n=n_total)
                    r1 = ctx1.group(w.len_ratio, w.pos_ratio, host_result=True)
                    checksum_1gpu = multi.output_checksum(r1.order, r1.gid, r1.repval, r1.identity)
                    ctx1.close()
                    del whole, r1
            else:
                res_h = ctx.group(w.len_ratio, w.pos_ratio, host_result=True)
                checksum = multi.output_checksum(res_h.order, res_h.gid, res_h.repval, res_h.identity)

    value = n_total * args.steps / (ms_total / 1e3)
    e2e_value = n_total * args.steps / (ms_e2e / 1e3)
    st, res_info = last
    if partitioned:
        res, info = res_info
        kept, groups, lines = info["total_kept"], res.n_groups, info["n_lines"]
        exchanged = info["bytes_sent"]
    else:
        res = res_info
        kept, groups, lines = res.n_kept, res.n_groups, res.n_kept
        exchanged = 0
    stage_ms = {k: round(v, 4) for k, v in {**st.ms_stage, **{k2: v2 for k2, v2 in res.ms_stage.items() if v2}}.items() if v}

    # partitioned: the per-kernel times of the LAST rank as well (its forest walks leave the GPU most often)
    kernels_last = None
    if partitioned and prof:
        box = [None] * world
        dist.all_gather_object(box, {k: round(v[1] / args.steps, 4) for k, v in prof.items()})
        kernels_last = box[-1]

    line = None
    if rank == 0:
        kernels, total_alg, total_ms = {}, 0.0, 0.0
        for name, (launches, ms, units) in prof.items():
            b = ALG_BYTES_PER_UNIT.get(name, 0) * units
            total_alg += b
            total_ms += ms
            kernels[name] = {"launches_per_step": launches / args.steps, "ms_per_step": round(ms / args.steps, 4),
                             "alg_gbs": round(b / ms / 1e6, 1) if b and ms > 0 else None}
        roofline = None
        if prof:
            top = max(prof.items(), key=lambda kv: kv[1][1])[0]
            launches, ms, units = prof[top]
            b = ALG_BYTES_PER_UNIT.get(top, 0) * units
            achieved = b / (ms / 1e3) / 1e9 if ms > 0 else 0.0
            roofline = {"bound": "hbm", "kernel": top, "achieved": round(achieved, 1), "peak": peak_gbs, "unit": "GB/s",
                        "frac": round(achieved / peak_gbs, 4), "traffic": NCU_TRAFFIC.get(top), "peak_source": peak_src,
                        "alg_bytes_per_launch": round(b / max(launches, 1)), "avg_launch_ms": round(ms / max(launches, 1), 5),
                        "share_of_kernel_time": round(ms / max(total_ms, 1e-9), 3)}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "ms_per_step_with_kernel_events": (ms_profiled / args.steps) if ms_profiled else None,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32+f64", "data": "synthetic",
            "config": {"workload": workload_text(w), "per_gpu_fragments": n, "kept": int(kept), "groups": int(groups),
                       "l2": "inputs larger than L2 (1.09 GB of records per GPU and step vs 126 MB)" if n * 109 > 200e6 else "inputs smaller than L2 (reduced --n run)",
                       "multi_gpu": ("one comparison partitioned over the GPUs inside librk_b200 (rk_dist_*): records to the owner of their "
                                     "xStart/10 range, X pass at home with a halo, Y exchange, forest over peer memory, output exchange; "
                                     f"NCCL send/recv, {exchanged / 1e6:.0f} MB sent by rank 0 in the grouping call of a step" if partitioned else
                                     "independent sequence pairs per rank, no data-path collective") if world > 1 else "single GPU"},
            "checksum": checksum, "checksum_same_comparison_on_1_gpu": checksum_1gpu,
            "checksum_match": (checksum == checksum_1gpu) if checksum_1gpu is not None else None,
            "e2e": {"value": e2e_value if do_e2e else None, "unit": UNIT,
                    "h2d_bytes_per_step": int(n * 109) if partitioned else int(n * 33), "d2h_bytes_per_step": int(lines * 13 + 40),
                    "ms_per_step": ms_e2e / args.steps if do_e2e else None,
                    "ingest": "rk_dist_load_aos: 109-byte records" if partitioned else
                              "rk_load_packed: 33 B per fragment (what the drop-in CLI's parser hands over)",
                    "record_ingest": None if ms_e2e_aos is None else {
                        "ms_per_step": ms_e2e_aos / args.steps, "value": n_total * args.steps / (ms_e2e_aos / 1e3),
                        "h2d_bytes_per_step": int(n * 109), "ingest": "rk_load_aos: 109-byte FragFile records"}},
            # kernels of this library launched inside timed region 1 (the C ABI counts them per call); the partitioned
            # path reports its timed launch groups (torch's own kernels and NCCL are not counted)
            # (partitioned: rank 0's kernels; NCCL's own kernels are not counted)
            "gpu_launches": int((st.n_launches + res.n_launches) * args.steps),
            "clocks": clocks,
            "roofline": roofline,
            "pipeline_alg_bytes_per_fragment": round(total_alg / args.steps / n, 1),
            "pipeline_hbm_frac": round(total_alg / (ms_total / 1e3) / 1e9 / peak_gbs, 4),
            "stage_ms": stage_ms,
            "kernels": kernels,
            "kernels_ms_per_step_last_rank": kernels_last,
        }
    if world > 1:
        dist.barrier()
    ctx.close()

    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            ws = gen.scaled(workload(args), min(n, CPU_SAMPLE_N))
            v, kind, times = cpu_reference_run(ws, 2, 1)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": 1, "kind": kind,
                                    "sample": f"{ws.n:,}-fragment sample of the {w.name} shape (same density): generate_fragment_groups + "
                                              f"generate_diagonal_func + sort_groups of the compiled reference, CSV parse/format excluded; "
                                              f"{sum(times) / len(times):.0f} ms per run"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    args.total_n = int(args.total_n)
    if args.impl == "reference":
        reference_arm(args)
    else:
        ours(args)


if __name__ == "__main__":
    main()
