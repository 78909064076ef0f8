"""The compact ingest for a comparison partitioned over several GPUs (rk_dist_load_packed, rk_multi_load_packed): 33 B per
fragment (key4, strand, rest4) instead of the 109-byte records.  The groups, the output text and the statistics equal
rk_multi_load_aos on the same records, rk_load_packed + rk_group on one GPU and the oracle; every refusal reaches every
rank with the same code and message and leaves nothing loaded.  The ranks are threads on GPU 0 (capi.Multi([0] * k)); the
caller-slice cases call rk_dist_load_packed on the ranks' contexts from a thread pool.
Run on the B200 box: python -m pytest tests -m gpu"""
import ctypes as C
import hashlib
import os
import socket
import sys
import threading
from concurrent.futures import ThreadPoolExecutor
from dataclasses import replace
from functools import lru_cache

import numpy as np
import pytest

from oracle import oracle as O
from repkiller_b200 import capi, gen, multi

pytestmark = pytest.mark.gpu

RK_ERR_ARG, RK_ERR_RANGE, RK_ERR_NOMEM = -2, -3, -5
PAIRS = [(0.05, 0.05), (0.1, 0.02), (2.0, 0.3)]  # the workload's own pair goes first


def _workload(name):  # the workloads of test_gpu_multi.py
    if name == "dense":
        return replace(gen.WORKLOADS["c1"], n=60_000, lx=400_000, ly=300_000, families=40, p_rep=0.6, seed=31)
    if name == "tiny":
        return replace(gen.WORKLOADS["c1"], n=3_000, lx=30_000, ly=25_000, families=12, p_rep=0.6, seed=21)
    if name == "c3":
        return gen.scaled(gen.WORKLOADS["c3"], 200_000)
    return gen.scaled(gen.WORKLOADS["c2"], 300_000)


@lru_cache(maxsize=None)
def _case(wl):
    """(workload, records, compact arrays, [(groups, text, statistics) of rk_load_packed on one GPU per pair], pairs)"""
    w = _workload(wl)
    rec = gen.generate(w)
    pk = capi.pack_records(rec)
    pairs = [(w.len_ratio, w.pos_ratio)] + PAIRS[1:]
    with capi.Context(0) as c:
        c.load_packed(*pk, w.lx + 1, w.ly + 1)
        want = [(c.group(*p), c.format_lines(), c.group_statistics()) for p in pairs]
    return w, rec, pk, want, pairs


def _same(res, want, what=""):
    assert res.n_kept == want.n_kept and res.n_groups == want.n_groups, (what, res.n_kept, want.n_kept, res.n_groups, want.n_groups)
    for name in ("order", "gid", "repval", "identity"):
        a, b = getattr(res, name), getattr(want, name)
        if name == "identity":
            a, b = a.view(np.uint32), b.view(np.uint32)
        d = np.nonzero(a != b)[0]
        assert d.size == 0, f"{what} {name}: {d.size} differences, first at {d[:5]}"


def _oracle(res, g):
    assert res.n_kept == g.n_kept and res.n_groups == g.n_groups
    assert np.array_equal(res.order, g.order) and np.array_equal(res.gid, g.out_gid) and np.array_equal(res.repval, g.repval)
    assert np.array_equal(res.identity.view(np.uint32), g.identity.view(np.uint32))


def _same_stats(got, want):
    """integers exact, the two means to the tolerance of the partitioned statistics tests"""
    assert got.shape == want.shape
    for f in ("count", "x_lo", "x_hi", "y_lo", "y_hi", "first_line"):
        assert np.array_equal(got[f], want[f]), f
    for f in ("mean_identity", "multiplicity"):
        rel = np.abs(got[f] - want[f]) / np.maximum(np.abs(want[f]), 1e-300)
        assert rel.max(initial=0.0) <= 1e-6, (f, float(rel.max()))


def _first_diff(a: bytes, b: bytes) -> str:
    i = next((k for k in range(min(len(a), len(b))) if a[k] != b[k]), min(len(a), len(b)))
    return f"{len(a)} vs {len(b)} bytes, first difference at byte {i}: {a[max(0, i - 60):i + 60]!r} vs {b[max(0, i - 60):i + 60]!r}"


def _handles(m):
    return [m._L.rk_multi_ctx(m._h, r) for r in range(m.n)]


def _host_parts(pk, bounds, rest=True):
    """rk_dist_load_packed arguments of host slices (lo, hi) of the compact arrays: (key4, strand, rest4, n, file_offset)"""
    key4, strand, rest4 = pk
    return [(key4.ctypes.data + lo * 16, strand.ctypes.data + lo, rest4.ctypes.data + lo * 16 if rest else 0, hi - lo, lo)
            for lo, hi in bounds]


def _dist_load(m, parts, lx1, ly1):
    """rk_dist_load_packed on every rank's context at once: (return codes, messages)"""
    L, hs = m._L, _handles(m)

    def one(r):
        k, s, rr, n, off = parts[r]
        return L.rk_dist_load_packed(hs[r], C.c_void_p(k) if k else None, C.c_void_p(s) if s else None, C.c_void_p(rr) if rr else None,
                                     n, off, lx1, ly1, 0, None)

    with ThreadPoolExecutor(m.n) as ex:
        rcs = list(ex.map(one, range(m.n)))
    return rcs, [L.rk_last_error(h).decode() for h in hs]


def _dist_group(m, lr, pr, flags):
    """rk_dist_group on every rank at once: (return codes, messages, results, infos)"""
    L, hs = m._L, _handles(m)
    res = [capi._Result() for _ in hs]
    info = [capi._DistInfo() for _ in hs]
    with ThreadPoolExecutor(m.n) as ex:
        rcs = list(ex.map(lambda r: L.rk_dist_group(hs[r], lr, pr, flags, C.byref(res[r]), C.byref(info[r])), range(m.n)))
    return rcs, [L.rk_last_error(h).decode() for h in hs], res, info


def _dist_text(m, lr, pr):
    """rk_dist_group with RK_F_LINE_RECORDS on every rank, then every rank's lines: (n_groups, text)"""
    L, hs = m._L, _handles(m)
    rcs, errs, res, info = _dist_group(m, lr, pr, capi.F_LINE_RECORDS)
    assert rcs == [0] * m.n, errs
    parts = []
    for r in range(m.n):
        t = capi._Text()
        assert L.rk_dist_format_lines(hs[r], 0, info[r].n_lines, C.byref(t)) == 0, L.rk_last_error(hs[r])
        parts.append(C.string_at(t.text, t.n_bytes) if t.n_bytes else b"")
    return res[0].n_groups, b"".join(parts)


def _check_parts(m, wl, parts):
    w, _, _, want, _ = _case(wl)
    rcs, errs = _dist_load(m, parts, w.lx + 1, w.ly + 1)
    assert rcs == [0] * m.n, errs
    n_groups, text = _dist_text(m, w.len_ratio, w.pos_ratio)
    assert n_groups == want[0][0].n_groups
    assert text == want[0][1], _first_diff(text, want[0][1])


# ---- 1. parity: Multi.load_packed against Multi.load, one GPU and the oracle -------------------------------------------
@pytest.mark.parametrize("world", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("wl", ["tiny", "dense", "c2", "c3"])
def test_multi_load_packed_equals_aos_and_one_gpu(world, wl):
    w, rec, pk, want, pairs = _case(wl)
    lx1, ly1 = w.lx + 1, w.ly + 1
    with capi.Multi([0] * world) as m:
        st = m.load_packed(*pk, lx1, ly1)
        assert st.n_loaded == rec.shape[0]
        res = m.group(*pairs[0], line_records=True)
        _oracle(res, O.group(rec, lx1, ly1, *pairs[0]))
        _same(res, want[0][0])
        text = m.format_lines()
        assert text == want[0][1], _first_diff(text, want[0][1])
        _same_stats(m.group_statistics(), want[0][2])
        info = [m.info(r) for r in range(world)]
        for p, (g1, t1, s1) in zip(pairs[1:], want[1:]):  # a second and a third pair on the same load
            _same(m.group(*p, line_records=True), g1, p)
            assert m.format_lines() == t1, p
            _same_stats(m.group_statistics(), s1)
        # the same records through rk_multi_load_aos on the same ranks: the same partition, groups and text
        m.load(rec, lx1, ly1)
        _same(m.group(*pairs[0], line_records=True), want[0][0])
        assert [m.info(r) for r in range(world)] == info
        assert m.format_lines() == want[0][1]


def test_c2_full_size_three_ranks():
    w = gen.WORKLOADS["c2"]
    pk = capi.pack_records(gen.generate(w))
    lx1, ly1 = w.lx + 1, w.ly + 1
    with capi.Context(0) as ctx:
        ctx.load_packed(*pk, lx1, ly1)
        res1 = ctx.group(w.len_ratio, w.pos_ratio)
        md5_1 = hashlib.md5(ctx.format_lines()).hexdigest()
    with capi.Multi([0, 0, 0]) as m:
        st = m.load_packed(*pk, lx1, ly1, timing=True)
        print(f"\nC2 10M over 3 ranks on one GPU: H2D {st.ms_stage['h2d']:.2f} ms (largest rank)")
        assert st.n_loaded == w.n
        _same(m.group(w.len_ratio, w.pos_ratio, line_records=True), res1)
        assert hashlib.md5(m.format_lines()).hexdigest() == md5_1


# ---- 2. caller slices through rk_dist_load_packed ----------------------------------------------------------------------
def test_uneven_empty_and_whole_slices():
    w, _, pk, _, _ = _case("dense")
    n = w.n
    with capi.Multi([0] * 4) as m:
        m.load_packed(*pk, w.lx + 1, w.ly + 1)   # sizes the ranks' buffers and maps them into each other
        for cuts in ([0, 7, 20_003, 41_999, n],          # uneven, at odd record counts
                     [0, 0, n // 2, n, n],               # empty first and last
                     [0, n // 3, n // 3, n // 3, n],     # empty middle
                     [0, 0, n, n, n],                    # one rank holds everything
                     [0, 0, 0, 0, n]):
            _check_parts(m, "dense", _host_parts(pk, list(zip(cuts, cuts[1:]))))


def test_slices_out_of_file_order():
    """rank 0 loads the second half, rank 1 the first: the grouping runs and equals rk_dist_load_aos on the same slices;
    RK_F_LINE_RECORDS is refused on every rank, as for rk_dist_load_aos"""
    w, rec, pk, _, _ = _case("dense")
    c = w.n // 2
    bounds = [(c, w.n), (0, c)]
    host = np.ascontiguousarray(rec)
    with capi.Multi([0, 0]) as m:
        m.load(rec, w.lx + 1, w.ly + 1)
        L, hs = m._L, _handles(m)
        with ThreadPoolExecutor(2) as ex:
            rcs = list(ex.map(lambda r: L.rk_dist_load_aos(hs[r], C.c_void_p(host.ctypes.data + bounds[r][0] * 109),
                                                             bounds[r][1] - bounds[r][0], bounds[r][0], w.lx + 1, w.ly + 1, 0, None),
                              range(2)))
        assert rcs == [0, 0]
        rcs, errs, res, _ = _dist_group(m, w.len_ratio, w.pos_ratio, capi.F_HOST_RESULT)
        assert rcs == [0, 0], errs
        want = [capi._groups_of(r, True, True) for r in res]
        rcs, errs = _dist_load(m, _host_parts(pk, bounds), w.lx + 1, w.ly + 1)
        assert rcs == [0, 0], errs
        rcs, errs, res, _ = _dist_group(m, w.len_ratio, w.pos_ratio, capi.F_HOST_RESULT)
        assert rcs == [0, 0], errs
        for r in range(2):
            _same(capi._groups_of(res[r], True, True), want[r], f"rank {r}")
        rcs, errs, _, _ = _dist_group(m, w.len_ratio, w.pos_ratio, capi.F_LINE_RECORDS)
        assert rcs == [RK_ERR_ARG] * 2 and len(set(errs)) == 1 and "rank order" in errs[0], errs


# ---- 3. device arrays in place -----------------------------------------------------------------------------------------
def _device_arrays(pk):
    import torch
    key4, strand, rest4 = (torch.from_numpy(np.ascontiguousarray(a).view(np.int32 if a.dtype == np.uint32 else np.uint8)).cuda()
                           for a in pk)
    torch.cuda.synchronize()
    return key4, strand, rest4


def test_device_arrays_in_place_and_a_misaligned_one():
    import torch
    w, _, pk, want, _ = _case("dense")
    key4, strand, rest4 = _device_arrays(pk)
    world = 3
    bounds = [multi.slice_bounds(w.n, r, world) for r in range(world)]
    with capi.Multi([0] * world) as m:
        m.load_packed(*pk, w.lx + 1, w.ly + 1)
        parts = [(key4.data_ptr() + lo * 16, strand.data_ptr() + lo, rest4.data_ptr() + lo * 16, hi - lo, lo) for lo, hi in bounds]
        _check_parts(m, "dense", parts)
        # the rows are read from the caller's arrays at grouping time: a second grouping still sees them
        n_groups, text = _dist_text(m, w.len_ratio, w.pos_ratio)
        assert text == want[0][1]
        # key4 of rank 1 four bytes off its 16-byte boundary: every rank refuses with the same code and message, no hang
        for bad in ((parts[1][0] + 4,) + parts[1][1:], parts[1][:2] + (parts[1][2] + 4,) + parts[1][3:]):
            rcs, errs = _dist_load(m, [parts[0], bad, parts[2]], w.lx + 1, w.ly + 1)
            assert rcs == [RK_ERR_ARG] * world and len(set(errs)) == 1, errs
            assert errs[0].startswith("rank 1: ") and "16-byte aligned" in errs[0], errs
            rcs, errs, _, _ = _dist_group(m, w.len_ratio, w.pos_ratio, 0)
            assert rcs == [-4] * world, errs   # nothing is loaded
            _check_parts(m, "dense", _host_parts(pk, bounds))   # the contexts still load
        # arrays partly on the host: refused alike
        mixed = (parts[2][0], pk[1].ctypes.data + bounds[2][0]) + parts[2][2:]
        rcs, errs = _dist_load(m, [parts[0], parts[1], mixed], w.lx + 1, w.ly + 1)
        assert rcs == [RK_ERR_ARG] * world and len(set(errs)) == 1 and errs[0].startswith("rank 2: "), errs
        _check_parts(m, "dense", parts)
        # rk_multi_load_packed takes host arrays only
        with pytest.raises(capi.RkError) as e:
            m.load_packed(key4.data_ptr(), strand.data_ptr(), rest4.data_ptr(), w.lx + 1, w.ly + 1, n=w.n)
        assert e.value.code == RK_ERR_ARG
    del key4, strand, rest4
    torch.cuda.empty_cache()


def test_device_arrays_on_another_device():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    w, _, pk, _, _ = _case("tiny")
    with torch.cuda.device(1):
        key4, strand, rest4 = _device_arrays(pk)
    bounds = [multi.slice_bounds(w.n, r, 2) for r in range(2)]
    with capi.Multi([0, 0]) as m:
        m.load_packed(*pk, w.lx + 1, w.ly + 1)
        parts = _host_parts(pk, bounds)
        lo, hi = bounds[1]
        parts[1] = (key4.data_ptr() + lo * 16, strand.data_ptr() + lo, rest4.data_ptr() + lo * 16, hi - lo, lo)
        rcs, errs = _dist_load(m, parts, w.lx + 1, w.ly + 1)
        assert rcs == [RK_ERR_ARG] * 2 and len(set(errs)) == 1 and "device 1" in errs[0], errs
        _check_parts(m, "tiny", _host_parts(pk, bounds))


# ---- 4. collective refusals: the same code and message on every rank, then a normal load works ------------------------
def test_refusals_reach_every_rank():
    w, rec, pk, want, _ = _case("tiny")
    lx1, ly1 = w.lx + 1, w.ly + 1
    world = 3
    bounds = [multi.slice_bounds(w.n, r, world) for r in range(world)]
    parts = _host_parts(pk, bounds)
    with capi.Multi([0] * world) as m:
        m.load_packed(*pk, lx1, ly1)

        def refused(bad, code, *words):
            rcs, errs = _dist_load(m, bad, lx1, ly1)
            assert rcs == [code] * world and len(set(errs)) == 1, errs
            for s in words:
                assert s in errs[0], errs
            rcs, errs, _, _ = _dist_group(m, w.len_ratio, w.pos_ratio, 0)
            assert rcs == [-4] * world, errs   # nothing is loaded
            _check_parts(m, "tiny", parts)

        # a null array on one rank
        refused([parts[0], (0,) + parts[1][1:], parts[2]], RK_ERR_ARG, "rank 1: ", "null array")
        refused([parts[0], parts[1], (parts[2][0], 0) + parts[2][2:]], RK_ERR_ARG, "rank 2: ", "null array")
        # one rank over the capacity the tiny load gave the ranks
        big = capi.pack_records(gen.generate(replace(_workload("c2"), n=400_000)))
        refused([parts[0], (big[0].ctypes.data, big[1].ctypes.data, big[2].ctypes.data, 400_000, bounds[1][0]), parts[2]],
                RK_ERR_NOMEM, "rank 1: ", "capacity")
        # a coordinate beyond the sequence on one rank (found by K1; every rank returns with the count exchange)
        k2 = pk[0].copy()
        k2[bounds[2][0] + 5, 0] = lx1 + 1000
        refused([parts[0], parts[1], (k2.ctypes.data + bounds[2][0] * 16,) + parts[2][1:]], RK_ERR_RANGE)
        # more than 2^32-16 records by one rank's file offset
        refused([parts[0], parts[1], parts[2][:4] + (0xFFFFFFF0,)], RK_ERR_ARG, "rank 2: ", "2^32-16")
        # through rk_multi_load_packed: coordinates beyond the sequence
        with pytest.raises(capi.RkError) as e:
            m.load_packed(*big, 1000, ly1)
        assert e.value.code == RK_ERR_RANGE
        m.load_packed(*pk, lx1, ly1)
        _oracle(m.group(w.len_ratio, w.pos_ratio), O.group(rec, lx1, ly1, w.len_ratio, w.pos_ratio))


# ---- 5. the arrays belong to the caller again when the call returns ----------------------------------------------------
def test_pinned_arrays_overwritten_right_after_the_call():
    import torch
    w, _, pk, want, _ = _case("c2")
    pinned = [torch.empty(a.shape, dtype={np.uint32: torch.int32, np.uint8: torch.uint8}[a.dtype.type], pin_memory=True) for a in pk]
    arrs = [t.numpy().view(a.dtype) for t, a in zip(pinned, pk)]
    world = 3
    bounds = [multi.slice_bounds(w.n, r, world) for r in range(world)]
    with capi.Multi([0] * world) as m:
        for a, src in zip(arrs, pk):
            a[...] = src
        m.load_packed(*arrs, w.lx + 1, w.ly + 1)
        for a in arrs:
            a[...] = 0xFF
        _same(m.group(w.len_ratio, w.pos_ratio, line_records=True), want[0][0])
        assert m.format_lines() == want[0][1]
        # the same through rk_dist_load_packed, each rank overwriting its slice as soon as its call returns
        for a, src in zip(arrs, pk):
            a[...] = src
        L, hs = m._L, _handles(m)
        parts = _host_parts(arrs, bounds)

        def one(r):
            k, s, rr, n, off = parts[r]
            rc = L.rk_dist_load_packed(hs[r], C.c_void_p(k), C.c_void_p(s), C.c_void_p(rr), n, off, w.lx + 1, w.ly + 1, 0, None)
            lo, hi = bounds[r]
            for a in arrs:
                a[lo:hi] = 0xFF
            return rc

        with ThreadPoolExecutor(world) as ex:
            assert list(ex.map(one, range(world))) == [0] * world
        n_groups, text = _dist_text(m, w.len_ratio, w.pos_ratio)
        assert n_groups == want[0][0].n_groups and text == want[0][1], _first_diff(text, want[0][1])


# ---- 6. rest4 == NULL --------------------------------------------------------------------------------------------------
def test_without_rest4():
    w, rec, pk, want, _ = _case("c3")
    lx1, ly1 = w.lx + 1, w.ly + 1
    world = 3
    bounds = [multi.slice_bounds(w.n, r, world) for r in range(world)]
    with capi.Multi([0] * world) as m:
        m.load_packed(pk[0], pk[1], None, lx1, ly1)
        _same(m.group(w.len_ratio, w.pos_ratio), want[0][0])
        with pytest.raises(capi.RkError) as e:
            m.group(w.len_ratio, w.pos_ratio, line_records=True)
        assert e.value.code == RK_ERR_ARG and "rest4" in str(e.value)
        # one rank without rest4: every rank refuses RK_F_LINE_RECORDS with the same message; grouping without it works
        parts = _host_parts(pk, bounds)
        parts[1] = parts[1][:2] + (0,) + parts[1][3:]
        rcs, errs = _dist_load(m, parts, lx1, ly1)
        assert rcs == [0] * world, errs
        rcs, errs, _, _ = _dist_group(m, w.len_ratio, w.pos_ratio, capi.F_LINE_RECORDS)
        assert rcs == [RK_ERR_ARG] * world and len(set(errs)) == 1 and "rank 1" in errs[0] and "rest4" in errs[0], errs
        rcs, errs, res, _ = _dist_group(m, w.len_ratio, w.pos_ratio, capi.F_HOST_RESULT)
        assert rcs == [0] * world, errs
        assert sum(r.n_kept for r in res) == want[0][0].n_kept and res[0].n_groups == want[0][0].n_groups
        # a later load with every array clears the refusal
        m.load(rec, lx1, ly1)
        m.group(w.len_ratio, w.pos_ratio, line_records=True)
        assert m.format_lines() == want[0][1]


# ---- 7. load order on one base -----------------------------------------------------------------------------------------
def _csv_body(w, rec, tmp_dir):
    """(body, total_frags) of the records written as a GECKO CSV: the bytes after the 16 header lines"""
    path = os.path.join(tmp_dir, f"{w.name}_{w.n}.csv")
    O.write_input_csv(path, rec, w.lx, w.ly)
    with open(path, "rb") as f:
        text = f.read()
    pos = 0
    for _ in range(16):
        pos = text.index(b"\n", pos) + 1
    return text[pos:], w.n


def test_load_order_aos_packed_csv_packed(tmp_path):
    """every load replaces the last one's rows: no stale records or compact rows leak into the next grouping's text"""
    cases = {wl: _case(wl) for wl in ("tiny", "dense", "c3")}
    wc, rec_c = cases["c3"][:2]
    body, total = _csv_body(wc, rec_c, str(tmp_path))
    with capi.Context(0) as c:  # the CSV load's own reference: rk_load_csv on one GPU
        c.load_csv(body, wc.lx + 1, wc.ly + 1, total)
        want_csv = (c.group(wc.len_ratio, wc.pos_ratio), c.format_lines(), c.group_statistics())
    with capi.Multi([0] * 3) as m:
        def check(wl, want):
            w = cases[wl][0]
            _same(m.group(w.len_ratio, w.pos_ratio, line_records=True), want[0], wl)
            assert m.format_lines() == want[1], wl
            _same_stats(m.group_statistics(), want[2])

        w, rec, pk, want, _ = cases["tiny"]
        m.load(rec, w.lx + 1, w.ly + 1)
        check("tiny", want[0])
        w, rec, pk, want, _ = cases["dense"]
        m.load_packed(*pk, w.lx + 1, w.ly + 1)
        check("dense", want[0])
        m.load_csv(body, wc.lx + 1, wc.ly + 1, total)
        check("c3", want_csv)
        w, rec, pk, want, _ = cases["tiny"]
        m.load_packed(*pk, w.lx + 1, w.ly + 1)
        check("tiny", want[0])
        w, rec, pk, want, _ = cases["dense"]
        m.load(rec, w.lx + 1, w.ly + 1)
        check("dense", want[0])


# ---- 8. views of a packed load -----------------------------------------------------------------------------------------
def test_views_of_a_packed_load():
    w, rec, pk, want, pairs = _case("c2")
    with capi.Multi([0] * 3) as m:
        m.load_packed(*pk, w.lx + 1, w.ly + 1)
        ctxs = [m, m.view(), m.view()]
        start = threading.Barrier(len(ctxs))

        def run(k):
            start.wait()
            res = ctxs[k].group(*pairs[k], line_records=True)
            return res, ctxs[k].format_lines(), ctxs[k].group_statistics()

        with ThreadPoolExecutor(len(ctxs)) as ex:
            got = list(ex.map(run, range(len(ctxs))))
        for k, (res, text, stats) in enumerate(got):
            _same(res, want[k][0], f"context {k}")
            assert text == want[k][1], f"context {k}"
            _same_stats(stats, want[k][2])
        for v in ctxs[1:]:
            v.close()


# ---- 9. one process per GPU over NCCL, each passing its own slice -------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out_dir):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(rank)
    w = _workload("c2")
    lo, hi = multi.slice_bounds(w.n, rank, world)
    key4, strand, rest4 = capi.pack_records(gen.generate(w, start=lo, count=hi - lo))
    ctx = capi.Context(rank)
    multi.bootstrap(ctx, multi.default_capacity(w.n // world + 16))
    ctx.dist_load_packed(key4, strand, rest4, lo, w.lx + 1, w.ly + 1)
    del key4, strand, rest4   # the rank's rows are its own
    ctx.dist_group(w.len_ratio, w.pos_ratio, line_records=True)
    with open(os.path.join(out_dir, f"r{rank}.txt"), "wb") as f:
        f.write(ctx.dist_format_lines())
    dist.barrier()
    ctx.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_nccl_processes_pass_their_own_slices(tmp_path, world):
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    text = b"".join(open(os.path.join(tmp_path, f"r{r}.txt"), "rb").read() for r in range(world))
    want = _case("c2")[3][0][1]
    assert text == want, _first_diff(text, want)
