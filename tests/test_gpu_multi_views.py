"""Views of a comparison partitioned over several ranks (rk_multi_create_view / capi.Multi.view, rk_dist_create_view /
capi.Context.dist_view): a second grouping context per rank over the partition database the ranks loaded.  Ranks are
threads on one GPU (capi.Multi([0] * N)), so the whole partitioned path of every context runs on a one-GPU box.
  * several ratio pairs grouped at the same time from one thread per context (base + 1 or 3 views) give, for every
    pair, the oracle's and one GPU's order, gid, repval, identity and group count, one GPU's text and statistics;
  * a view's line rows and statistics are its own: a grouping on the base does not change them, and the other way round;
  * the lifetime rules: no view before a load, no load on a view or on a base with live views, no rk_dist_init on either,
    the database outlives the base, and creating and destroying views leaves no device memory behind;
  * one process per GPU over NCCL (where the box has the GPUs), a base and a view grouping at once in every process;
  * group_and_sort from several threads on a partitioned FragmentsDatabase (rk_hostcheck group_pool) against the same
    calls from one thread and on one GPU."""
import ctypes as C
import os
import re
import socket
import subprocess
import threading
from concurrent.futures import ThreadPoolExecutor
from dataclasses import replace
from functools import lru_cache

import numpy as np
import pytest

from oracle import oracle as O
from repkiller_b200 import capi, gen, multi

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOSTCHECK = os.path.join(ROOT, "repkiller_b200", "bin", "rk_hostcheck")
RK_ERR_STATE = -4
# ordinary pairs, t < 1, a clamped threshold, a huge position ratio
PAIRS = [(0.05, 0.05), (0.1, 0.02), (1e-3, 1e-3), (2.0, 0.3), (0.05, 1e9), (0.3, 0.1), (0.02, 0.5), (1.0, 1.0)]


def _workload(name):  # the workloads of test_gpu_multi.py, and config 2 at 10M
    if name == "dense":
        return replace(gen.WORKLOADS["c1"], n=60_000, lx=400_000, ly=300_000, families=40, p_rep=0.6, seed=31)
    if name == "tiny":
        return replace(gen.WORKLOADS["c1"], n=3_000, lx=30_000, ly=25_000, families=12, p_rep=0.6, seed=21)
    if name == "c3":
        return gen.scaled(gen.WORKLOADS["c3"], 200_000)
    if name == "c2_10m":
        return gen.scaled(gen.WORKLOADS["c2"], 10_000_000)
    return gen.scaled(gen.WORKLOADS["c2"], 300_000)


@lru_cache(maxsize=1)
def _records(wl):
    w = _workload(wl)
    return w, gen.generate(w)


def _equal_groups(a, b, what):
    assert a.n_kept == b.n_kept and a.n_groups == b.n_groups, (what, a.n_kept, b.n_kept, a.n_groups, b.n_groups)
    for name in ("order", "gid", "repval"):
        d = np.nonzero(getattr(a, name) != getattr(b, name))[0]
        assert d.size == 0, f"{what} {name}: {d.size} differences, first at {d[:5]}"
    assert np.array_equal(a.identity.view(np.uint32), b.identity.view(np.uint32)), (what, "identity")


def _equal_oracle(res, g, what):
    assert res.n_kept == g.n_kept and res.n_groups == g.n_groups, (what, res.n_kept, g.n_kept, res.n_groups, g.n_groups)
    for name, got, want in (("order", res.order, g.order), ("gid", res.gid, g.out_gid), ("repval", res.repval, g.repval),
                            ("identity", res.identity.view(np.uint32), g.identity.view(np.uint32))):
        d = np.nonzero(got != want)[0]
        assert d.size == 0, f"{what} {name}: {d.size} differences, first at {d[:5]}"


def _one_gpu(w, rec, pairs):
    """{pair: (groups, text, statistics)} of rk_load_aos + rk_group on one GPU"""
    out = {}
    with capi.Context(0) as c:
        c.load(rec, w.lx + 1, w.ly + 1)
        for p in pairs:
            out[p] = (c.group(*p), c.format_lines(), c.group_statistics())
    return out


def _multi_pair(m, p):
    res = m.group(*p, line_records=True)
    return res, m.format_lines(), m.group_statistics()


def _check(got, want, what):
    res, text, stats = got
    _equal_groups(res, want[0], what)
    assert text == want[1], f"{what}: text differs"
    assert np.array_equal(stats, want[2]), f"{what}: statistics differ"


# ---- 1. concurrent pairs ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world,wl,n_views", [(2, "dense", 1), (2, "tiny", 3), (3, "c2", 1), (3, "c2", 3), (5, "c3", 1),
                                              (5, "dense", 3), (3, "c2_10m", 3)])
def test_concurrent_pairs(world, wl, n_views):
    w, rec = _records(wl)
    pairs = PAIRS if wl != "c2_10m" else PAIRS[:4]
    want = _one_gpu(w, rec, pairs)
    if wl != "c2_10m":  # (at 10M the one-GPU result stands for the oracle, which test_gpu_views.py checks it against)
        for p in pairs:
            _equal_oracle(want[p][0], O.group(rec, w.lx + 1, w.ly + 1, *p), f"one GPU {p}")
    with capi.Multi([0] * world) as m:
        m.load(rec, w.lx + 1, w.ly + 1)
        ctxs = [m] + [m.view() for _ in range(n_views)]
        assert [c.transport for c in ctxs] == ["local"] * len(ctxs)
        start = threading.Barrier(len(ctxs))

        def run(k):  # context k groups pairs k, k + len(ctxs), ... back to back
            start.wait()
            return {p: _multi_pair(ctxs[k], p) for p in pairs[k::len(ctxs)]}

        with ThreadPoolExecutor(len(ctxs)) as ex:
            results = list(ex.map(run, range(len(ctxs))))
        for k, got in enumerate(results):
            for p, g in got.items():
                _check(g, want[p], f"{world} ranks, context {k}, pair {p}")
        # every context reports its own last grouping, rank by rank
        for k, c in enumerate(ctxs):
            last = pairs[k::len(ctxs)][-1]
            assert sum(c.info(r)["n_lines"] for r in range(world)) == want[last][0].n_kept
        for v in ctxs[1:]:
            v.close()


# ---- 2. independent line rows ----------------------------------------------------------------------------------------
def test_line_rows_are_per_context():
    w, rec = _records("c2")
    a, b = PAIRS[0], PAIRS[3]
    want = _one_gpu(w, rec, [a, b])
    with capi.Multi([0] * 3) as m:
        m.load(rec, w.lx + 1, w.ly + 1)
        with m.view() as v:
            for first, second in ((v, m), (m, v)):  # pair A on one context, then pair B on the other
                _equal_groups(first.group(*a, line_records=True), want[a][0], "A")
                _equal_groups(second.group(*b, line_records=True), want[b][0], "B")
                assert first.format_lines() == want[a][1], "the first context's text changed"
                assert np.array_equal(first.group_statistics(), want[a][2]), "the first context's statistics changed"
                assert second.format_lines() == want[b][1]
                assert np.array_equal(second.group_statistics(), want[b][2])


# ---- 3. lifetime and refusals ----------------------------------------------------------------------------------------
def _dist_init(L, ctx_handle, world):
    return L.rk_dist_init(ctx_handle, 0, world, C.c_char_p(bytes(capi.DIST_ID_BYTES)), 4096)


def test_lifetime_and_refusals():
    w, rec = _records("c2")
    p = PAIRS[1]
    want = _one_gpu(w, rec, [p])[p]
    L = capi.load_library()
    with capi.Multi([0, 0]) as m:
        with pytest.raises(capi.RkError, match="no partition database"):
            m.view()  # before a load
    m = capi.Multi([0] * 3)
    m.load(rec, w.lx + 1, w.ly + 1)
    v1, v2 = m.view(), m.view()
    vv = v1.view()  # a view of a view shares the same database
    # a load on a view
    for v in (v1, vv):
        with pytest.raises(capi.RkError) as e:
            v.load(rec, w.lx + 1, w.ly + 1)
        assert e.value.code == RK_ERR_STATE and "view" in str(e.value)
    # a load on the base with live views: the count in the message, and nothing changed
    small = gen.generate(gen.scaled(gen.WORKLOADS["c2"], 20_000))
    for load in (lambda: m.load(small, w.lx + 1, w.ly + 1), lambda: m.load_csv(b"", w.lx + 1, w.ly + 1, 0)):
        with pytest.raises(capi.RkError) as e:
            load()
        assert e.value.code == RK_ERR_STATE and "3 views" in str(e.value), str(e.value)
    _check(_multi_pair(m, p), want, "base after the refused load")
    # rk_dist_init on a view and on a base with live views; rk_create_view on a rank context of a view
    for c in (v1, m):
        assert _dist_init(L, c.ctx(0), 3) == RK_ERR_STATE
        assert "view" in L.rk_last_error(c.ctx(0)).decode()
    assert not L.rk_create_view(v1.ctx(0))
    # the base destroyed first: the views still group exactly
    m.close()
    v2.close()
    _check(_multi_pair(v1, p), want, "view after the base")
    _check(_multi_pair(vv, p), want, "view of a view after the base")
    vv.close()
    _check(_multi_pair(v1, p), want, "last view")
    v1.close()


def test_views_leave_no_device_memory():
    import torch
    w, rec = _records("c2")
    with capi.Multi([0] * 3) as m:
        m.load(rec, w.lx + 1, w.ly + 1)
        with m.view() as v:  # warm-up: every lazily made buffer of the process exists after this
            v.group(*PAIRS[0], line_records=True)
            v.format_lines()
            v.group_statistics()
        torch.cuda.synchronize()
        before = torch.cuda.mem_get_info(0)[0]
        grown = []
        for _ in range(5):
            with m.view() as v:
                v.group(*PAIRS[0], line_records=True)
                v.format_lines()
                v.group_statistics()
                grown.append(before - torch.cuda.mem_get_info(0)[0])
        after = torch.cuda.mem_get_info(0)[0]
    assert min(grown) > 64 << 20, grown  # a view holds its own workspace ...
    assert before - after < 64 << 20, (before, after)  # ... and gives it all back


# ---- 4. one process per GPU ------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, out_dir):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(rank)
    w = _workload("c2")
    lo, hi = multi.slice_bounds(w.n, rank, world)
    rec = np.ascontiguousarray(gen.generate(w, start=lo, count=hi - lo))
    ctx = capi.Context(rank)
    multi.bootstrap(ctx, multi.default_capacity(w.n // world + 16))
    ctx.dist_load(rec.ctypes.data, hi - lo, lo, w.lx + 1, w.ly + 1)
    box = [capi.dist_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    view = ctx.dist_view(box[0])
    blobs = [None] * world
    dist.all_gather_object(blobs, view.dist_export())
    view.dist_import(b"".join(blobs))
    sums = {}

    def run(c, p):
        res, info = c.dist_group(*p)
        sums[p] = multi.output_checksum(res.order, res.gid, res.repval, res.identity, info["line_offset"])

    th = [threading.Thread(target=run, args=(c, p)) for c, p in ((ctx, PAIRS[0]), (view, PAIRS[3]))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    np.save(os.path.join(out_dir, f"r{rank}.npy"), np.array([sums[PAIRS[0]], sums[PAIRS[3]]], dtype=np.uint64))
    dist.barrier()
    view.close()
    ctx.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2])
def test_nccl_processes_with_views(tmp_path, world):
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs: one process per GPU over NCCL")
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    w = _workload("c2")
    rec = gen.generate(w)
    want = _one_gpu(w, rec, [PAIRS[0], PAIRS[3]])
    got = sum(np.load(os.path.join(tmp_path, f"r{r}.npy")).astype(object) for r in range(world))
    for k, p in enumerate((PAIRS[0], PAIRS[3])):
        g = want[p][0]
        assert int(got[k]) & ((1 << 64) - 1) == multi.output_checksum(g.order, g.gid, g.repval, g.identity), p


# ---- 5. the facade -------------------------------------------------------------------------------------------------
def _group_pool(csv, devices, threads, pairs):
    args = [HOSTCHECK, "group_pool", str(csv), devices, str(threads)] + [f"{x!r}" for p in pairs for x in p]
    out = subprocess.run(args, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr
    lines = out.stdout.splitlines()
    return lines[:-1], int(re.match(r"(\d+) grouping contexts", lines[-1]).group(1))


def test_group_and_sort_from_threads(tmp_path):
    w, rec = _records("c2")
    csv = tmp_path / "in.csv"
    O.write_input_csv(str(csv), rec, w.lx, w.ly)
    pairs = PAIRS[:6]
    one_gpu, _ = _group_pool(csv, "0", 1, pairs)
    sequential, n1 = _group_pool(csv, "0,0,0", 1, pairs)
    threaded, n4 = _group_pool(csv, "0,0,0", 4, pairs)
    assert sequential == one_gpu, (one_gpu, sequential)
    assert threaded == one_gpu, (one_gpu, threaded)
    assert n1 == 1 and 1 <= n4 <= 4, (n1, n4)
