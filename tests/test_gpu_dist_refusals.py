"""Capacity refusals of the partitioned load (csrc/multi.cu) on ranks that are threads of one process: every rank returns
RK_ERR_NOMEM with the same message, and the same rk_multi then loads and groups a normal comparison exactly, so no rank
was left behind in a collective step."""
import ctypes as C
from concurrent.futures import ThreadPoolExecutor
from dataclasses import replace

import numpy as np
import pytest

from oracle import oracle as O
from repkiller_b200 import capi, gen, multi
from repkiller_b200.frags import FRAG_DTYPE

pytestmark = pytest.mark.gpu

RK_ERR_NOMEM = -5
WORLD = 3
TINY = replace(gen.WORKLOADS["c1"], n=3_000, lx=30_000, ly=25_000, families=12, p_rep=0.6, seed=21)
N_BIG = 600_000  # about 1.6 times the capacity Multi.load gives 3 ranks for it
LX = LY = 2_000_000


def _rank_handles(m):
    return [m._L.rk_multi_ctx(m._h, r) for r in range(m.n)]


def _errors(m):
    return [m._L.rk_last_error(h).decode() for h in _rank_handles(m)]


def _records(xs, ys, length=100):
    rec = np.zeros(len(xs), dtype=FRAG_DTYPE)
    rec["xStart"], rec["yStart"], rec["length"] = xs, ys, length
    rec["xEnd"], rec["yEnd"] = rec["xStart"] + length - 1, rec["yStart"] + length - 1
    rec["diag"] = rec["xStart"].astype(np.int64) - rec["yStart"].astype(np.int64)
    rec["ident"] = length * 9 // 10
    rec["similarity"] = 90.0
    rec["strand"] = b"f"
    return rec


def _assert_tiny_groups_exactly(m):
    rec = gen.generate(TINY)
    g = O.group(rec, TINY.lx + 1, TINY.ly + 1, TINY.len_ratio, TINY.pos_ratio)
    m.load(rec, TINY.lx + 1, TINY.ly + 1)
    res = m.group(TINY.len_ratio, TINY.pos_ratio)
    assert res.n_kept == g.n_kept and res.n_groups == g.n_groups
    assert np.array_equal(res.order, g.order) and np.array_equal(res.gid, g.out_gid)
    assert np.array_equal(res.repval, g.repval)
    assert np.array_equal(res.identity.view(np.uint32), g.identity.view(np.uint32))


def _assert_load_refused(m, rec, text):
    with pytest.raises(capi.RkError) as e:
        m.load(rec, LX + 1, LY + 1)
    assert e.value.code == RK_ERR_NOMEM, str(e.value)
    errs = _errors(m)
    assert all(text in s for s in errs), errs
    assert len(set(errs)) == 1, errs


def test_slice_larger_than_the_capacity():
    """one rank's slice holds more records than the capacity the rk_multi was sized for: the rank publishes an error word
    with the first count exchange, and every rank returns RK_ERR_NOMEM"""
    with capi.Multi([0] * WORLD) as m:
        _assert_tiny_groups_exactly(m)  # sizes the capacity for the tiny comparison: well below 100k rows per rank
        L, hs = m._L, _rank_handles(m)
        big = np.ascontiguousarray(_records(np.arange(100_000) * 7 % 1_000_000, np.arange(100_000) * 11 % 1_000_000))
        small = np.ascontiguousarray(gen.generate(TINY))
        lo1, hi1 = multi.slice_bounds(TINY.n, 1, WORLD)
        lo2, hi2 = multi.slice_bounds(TINY.n, 2, WORLD)
        args = [(big.ctypes.data, big.size, 0), (small.ctypes.data + lo1 * 109, hi1 - lo1, big.size + lo1),
                (small.ctypes.data + lo2 * 109, hi2 - lo2, big.size + lo2)]
        st = [capi._LoadStats() for _ in range(WORLD)]
        with ThreadPoolExecutor(WORLD) as ex:
            rcs = list(ex.map(lambda r: L.rk_dist_load_aos(hs[r], C.c_void_p(args[r][0]), args[r][1], args[r][2], LX + 1, LY + 1, 0,
                                                           C.byref(st[r])), range(WORLD)))
        errs = _errors(m)
        assert rcs == [RK_ERR_NOMEM] * WORLD, (rcs, errs)
        assert all("more records than the capacity" in s for s in errs), errs
        _assert_tiny_groups_exactly(m)


def _spread_centres(i):
    """starts of 100-long fragments whose centres spread over 19k buckets of 100, away from the bucket edges (a centre
    within 2 of an edge links two buckets, and a run of linked buckets is never split between ranks)"""
    return (1 + i % 18_999) * 100 + 2 + (i // 18_999) % 90 - 50


def test_exchange_one_over_capacity():
    """every record in one xStart/10 bucket: the rank that owns it would hold all of them"""
    i = np.arange(N_BIG)
    with capi.Multi([0] * WORLD) as m:
        _assert_load_refused(m, _records(50_000 + i % 10, _spread_centres(i)), "would own")
        assert "fragments, capacity is" in _errors(m)[0]
        _assert_tiny_groups_exactly(m)


def test_y_pass_over_capacity():
    """X spread out, every Y centre in one /100 bucket: the owner of that Y range would hold all of them"""
    i = np.arange(N_BIG)
    with capi.Multi([0] * WORLD) as m:
        _assert_load_refused(m, _records(_spread_centres(i), 70_000 + i % 40), "in the Y pass")
        _assert_tiny_groups_exactly(m)
