"""One comparison partitioned over several ranks (csrc/multi.cu) against the oracle, bit for bit:
  * rk_create_multi with the same device listed several times — ranks are threads of one process that exchange the small
    tables through host memory and push their rows into each other's buffers as the NCCL transport does — so the whole
    partitioned path (cuts, halo and Y row exchanges, forest over peer pointers, output exchange) is checked on a one-GPU
    box for 1, 2, 3, 5 and 8 ranks;
  * rk_dist_* with one process per GPU over NCCL where the box has the GPUs (2, 4, 8)."""
import os
import socket
import sys
from dataclasses import replace

import numpy as np
import pytest

from oracle import oracle as O
from repkiller_b200 import capi, gen, multi

pytestmark = pytest.mark.gpu


def _workload(name):
    if name == "dense":    # cross-bucket links, giant families, groups > 16 with tied h, many fragments near the cuts
        return replace(gen.WORKLOADS["c1"], n=60_000, lx=400_000, ly=300_000, families=40, p_rep=0.6, seed=31)
    if name == "tiny":     # sequences so short that fragments reach over several ranks' X ranges
        return replace(gen.WORKLOADS["c1"], n=3_000, lx=30_000, ly=25_000, families=12, p_rep=0.6, seed=21)
    if name == "c3":
        return gen.scaled(gen.WORKLOADS["c3"], 200_000)
    if name == "c2_6m":    # large enough that the row exchanges spread their copies over several streams
        return gen.scaled(gen.WORKLOADS["c2"], 6_000_000)
    return gen.scaled(gen.WORKLOADS["c2"], 300_000)


def _assert_same(res, g):
    assert res.n_kept == g.n_kept and res.n_groups == g.n_groups, (res.n_kept, g.n_kept, res.n_groups, g.n_groups)
    for name, got, want in (("order", res.order, g.order), ("gid", res.gid, g.out_gid), ("repval", res.repval, g.repval),
                            ("identity", res.identity.view(np.uint32), g.identity.view(np.uint32))):
        d = np.nonzero(got != want)[0]
        assert d.size == 0, f"{name}: {d.size} differences, first at {d[:5]}: got {got[d[:5]]} want {want[d[:5]]}"


@pytest.mark.parametrize("world", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("wl", ["dense", "tiny", "c2", "c3"])
def test_ranks_as_threads_match_oracle(world, wl):
    w = _workload(wl)
    rec = gen.generate(w)
    g = O.group(rec, w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio)
    with capi.Multi([0] * world) as m:
        assert m.transport == "local"
        st = m.load(rec, w.lx + 1, w.ly + 1)
        assert st.n_loaded == w.n and st.n_kept == g.n_kept
        res = m.group(w.len_ratio, w.pos_ratio)
        _assert_same(res, g)
        infos = [m.info(r) for r in range(world)]
        assert sum(i["n_lines"] for i in infos) == g.n_kept
        assert sum(i["n_halo_in"] for i in infos) == sum(i["n_halo_out"] for i in infos)
        # a second pair of ratios on the loaded database, then the first again: nothing of a grouping leaks into the next
        g2 = O.group(rec, w.lx + 1, w.ly + 1, 0.5, 0.5)
        _assert_same(m.group(0.5, 0.5), g2)
        _assert_same(m.group(w.len_ratio, w.pos_ratio), g)


@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("wl", ["dense", "c2", "c3"])
def test_forest_bulk_rounds_match_oracle(monkeypatch, world, wl):
    """RK_DIST_BULK_MIN=1: every chain that leaves its GPU is resolved by the ask/answer rounds (what a dense 1e9-fragment
    comparison uses) instead of by walking through peer memory; chains over several GPUs need several rounds"""
    monkeypatch.setenv("RK_DIST_BULK_MIN", "1")
    w = _workload(wl)
    rec = gen.generate(w)
    g = O.group(rec, w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio)
    with capi.Multi([0] * world) as m:
        m.load(rec, w.lx + 1, w.ly + 1)
        _assert_same(m.group(w.len_ratio, w.pos_ratio), g)
        _assert_same(m.group(0.5, 0.5), O.group(rec, w.lx + 1, w.ly + 1, 0.5, 0.5))


@pytest.mark.parametrize("world,wl", [(8, "c2"), (3, "dense"), (5, "c2"), (2, "tiny"), (3, "c2_6m")])
def test_output_ranges_respect_the_row_capacity(monkeypatch, world, wl):
    """the output ranges are cut by estimated sort_groups work, which gives the ranks with small groups more lines; no rank
    may get more lines than it has rows for (RK_DIST_LINE_CAP stands in for a tight capacity).
    (3, c2_6m) also takes the row exchange's spread over several copy streams, which needs at least 2 destination peers
    and 8 MiB per exchange: each of the 3 ranks holds about 2M fragments and sends about 2/3 of its Y rows, 16 B each, to
    the other two: about 21 MB, more than twice the threshold."""
    w = _workload(wl)
    rec = gen.generate(w)
    g = O.group(rec, w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio)
    with capi.Multi([0] * world) as m:
        m.load(rec, w.lx + 1, w.ly + 1)
        m.group(w.len_ratio, w.pos_ratio)
        free = max(m.info(r)["n_lines"] for r in range(world))
    cap = -(-g.n_kept // world)
    cap += cap // 8 + 64             # 12 % over an even split (the cuts fall on boundaries of 1/4096 of the group ids)
    monkeypatch.setenv("RK_DIST_LINE_CAP", str(cap))
    with capi.Multi([0] * world) as m:
        m.load(rec, w.lx + 1, w.ly + 1)
        _assert_same(m.group(w.len_ratio, w.pos_ratio), g)
        lines = [m.info(r)["n_lines"] for r in range(world)]
    assert sum(lines) == g.n_kept and max(lines) <= cap, (lines, cap)
    print(f"largest range without the bound: {free} lines; bound {cap}; with it: {max(lines)}")


def test_ranks_as_threads_unsorted_members():
    w = _workload("dense")
    rec = gen.generate(w)
    g = O.group(rec, w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio)
    with capi.Multi([0, 0, 0]) as m:
        m.load(rec, w.lx + 1, w.ly + 1)
        res = m.group(w.len_ratio, w.pos_ratio, sort=False)
    # members in push_back (processing) order: group by gid, stable
    order = np.argsort(g.gid, kind="stable")
    assert np.array_equal(res.order, g.rank_fidx[order])
    assert np.array_equal(res.gid, g.gid[order])


def test_fuzz_inputs_two_and_three_ranks(tmp_path, fuzz_cases):
    """the adversarial CSV inputs of the golden set (tiny sequences, odd strands, length 0, duplicates) through 2 and 3 ranks"""
    done = 0
    with capi.Multi([0, 0]) as m2, capi.Multi([0, 0, 0]) as m3:
        for c in fuzz_cases[::2]:
            inp = tmp_path / "in.csv"
            inp.write_text(c["csv"], newline="")
            rec, lx1, ly1, _ = O.load_csv(str(inp))
            if rec.shape[0] == 0:
                continue
            try:
                g = O.group(rec, lx1, ly1, c["len_ratio"], c["pos_ratio"])
            except ValueError:
                continue   # input the reference itself cannot process (undefined behaviour there)
            for m in (m2, m3):
                try:
                    m.load(rec, lx1, ly1)
                except capi.RkError as e:
                    assert e.code == -3, e      # RK_ERR_RANGE, as on one GPU
                    break
                _assert_same(m.group(c["len_ratio"], c["pos_ratio"]), g)
            else:
                done += 1
    assert done > 20


# ---- one process per GPU over NCCL -------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, wl, out_dir):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(rank)
    w = _workload(wl)
    lo, hi = multi.slice_bounds(w.n, rank, world)
    rec = gen.generate(w, start=lo, count=hi - lo)
    ctx = capi.Context(rank)
    multi.bootstrap(ctx, multi.default_capacity(w.n // world + 16))
    host = np.ascontiguousarray(rec)
    ctx.dist_load(host.ctypes.data, hi - lo, lo, w.lx + 1, w.ly + 1)
    res, info = ctx.dist_group(w.len_ratio, w.pos_ratio)
    np.savez(os.path.join(out_dir, f"r{rank}.npz"), order=res.order, gid=res.gid, repval=res.repval, identity=res.identity,
             n_groups=res.n_groups, line_offset=info["line_offset"], total_kept=info["total_kept"])
    dist.barrier()
    ctx.close()
    dist.destroy_process_group()


def _gpu_count():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_nccl_processes_match_oracle(tmp_path, world):
    if _gpu_count() < world:
        pytest.skip(f"needs {world} GPUs")
    import torch.multiprocessing as mp
    wl = "c2"
    mp.spawn(_worker, args=(world, _free_port(), wl, str(tmp_path)), nprocs=world, join=True)
    w = _workload(wl)
    rec = gen.generate(w)
    g = O.group(rec, w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio)
    parts = [np.load(os.path.join(tmp_path, f"r{r}.npz")) for r in range(world)]
    assert int(parts[0]["n_groups"]) == g.n_groups and int(parts[0]["total_kept"]) == g.n_kept
    off = 0
    for p in parts:
        assert int(p["line_offset"]) == off
        off += p["order"].shape[0]
    assert off == g.n_kept
    for name, want in (("order", g.order), ("gid", g.out_gid), ("repval", g.repval)):
        assert np.array_equal(np.concatenate([p[name] for p in parts]), want), name
    assert np.array_equal(np.concatenate([p["identity"] for p in parts]).view(np.uint32), g.identity.view(np.uint32))
    # the checksum bench.py prints: sum over the ranks' ranges == checksum of the whole output
    whole = multi.output_checksum(g.order, g.out_gid, g.repval, g.identity)
    summed = sum(multi.output_checksum(p["order"], p["gid"], p["repval"], p["identity"], int(p["line_offset"])) for p in parts) & ((1 << 64) - 1)
    assert whole == summed
