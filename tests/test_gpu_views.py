"""Concurrent ratio pairs on one loaded database (rk_create_view / capi.Context.view): a view is a second grouping context
with its own stream and workspace over the load of another context.  Groupings on different contexts of one database run
from different threads at once, and every result must be the one that pair gives alone:
  * order, gid, repval and the identity bits equal the oracle's, the device text its writer's bytes, the statistics the
    base's for the same pair run alone — with 4 contexts running 8 pairs from 4 threads on three workloads;
  * the same at 10M fragments against the base's sequential results;
  * the compact load's side copy, device-pointer records, rk_sort_groups, debug_fetch and diagonal_func on a view;
  * the lifetime rules (reference-counted database, refused loads) and per-view streams;
  * the host facades from a thread pool (rk_hostcheck pool) against the single-threaded facade calls.
The test without the gpu mark checks the exported symbol."""
import ctypes as C
import hashlib
import os
import re
import subprocess
from concurrent.futures import ThreadPoolExecutor
from dataclasses import replace
from functools import lru_cache

import numpy as np
import pytest

from oracle import oracle as O
from repkiller_b200 import capi, gen

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOSTCHECK = os.path.join(ROOT, "repkiller_b200", "bin", "rk_hostcheck")
RK_ERR_STATE = -4
# ordinary pairs, t < 1, a clamped threshold, a huge position ratio
PAIRS = [(0.05, 0.05), (0.1, 0.02), (1e-3, 1e-3), (2.0, 0.3), (0.05, 1e9), (0.3, 0.1), (0.02, 0.5), (1.0, 1.0)]


def _workload(name):  # the workloads of test_gpu_multi_output.py
    if name == "dense":
        return replace(gen.WORKLOADS["c1"], n=60_000, lx=400_000, ly=300_000, families=40, p_rep=0.6, seed=31)
    if name == "c3":
        return gen.scaled(gen.WORKLOADS["c3"], 200_000)
    return gen.scaled(gen.WORKLOADS["c2"], 300_000)


@lru_cache(maxsize=1)
def _records(wl):
    w = _workload(wl)
    return w, gen.generate(w)


def _oracle_body(rec, g, tmp_dir):
    path = os.path.join(tmp_dir, "oracle_body.csv")
    O.write_output(path, b"", rec, g)
    with open(path, "rb") as f:
        body = f.read()
    os.remove(path)
    return body


def _assert_same(res, g, what=""):
    assert res.n_kept == g.n_kept and res.n_groups == g.n_groups, (what, res.n_kept, g.n_kept, res.n_groups, g.n_groups)
    for name, got, want in (("order", res.order, g.order), ("gid", res.gid, g.out_gid), ("repval", res.repval, g.repval),
                            ("identity", res.identity.view(np.uint32), g.identity.view(np.uint32))):
        d = np.nonzero(got != want)[0]
        assert d.size == 0, f"{what} {name}: {d.size} differences, first at {d[:5]}"


def _assert_equal_groups(a, b, what=""):
    assert a.n_kept == b.n_kept and a.n_groups == b.n_groups, what
    for name in ("order", "gid", "repval", "identity"):
        assert np.array_equal(getattr(a, name).view(np.uint32) if name == "identity" else getattr(a, name),
                              getattr(b, name).view(np.uint32) if name == "identity" else getattr(b, name)), (what, name)


def _oracle(rec, w, lr, pr, tmp_dir):
    g = O.group(rec, w.lx + 1, w.ly + 1, lr, pr)
    return g, _oracle_body(rec, g, tmp_dir)


# ---- 1. concurrent parity --------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("wl", ["dense", "c2", "c3"])
def test_concurrent_pairs_match_oracle(wl, tmp_path):
    w, rec = _records(wl)
    want = [_oracle(rec, w, lr, pr, str(tmp_path)) for lr, pr in PAIRS]
    base = capi.Context(0)
    base.load(rec, w.lx + 1, w.ly + 1)
    alone = []
    for lr, pr in PAIRS:  # statistics of every pair run alone on the base
        base.group(lr, pr)
        alone.append(base.group_statistics())
    ctxs = [base] + [base.view() for _ in range(3)]

    def run(i):  # thread i owns context i and runs two pairs in a row
        out = []
        for k in (2 * i, 2 * i + 1):
            res = ctxs[i].group(*PAIRS[k])
            out.append((k, res, ctxs[i].format_lines(), ctxs[i].group_statistics()))
        return out

    with ThreadPoolExecutor(4) as ex:
        outs = [o for part in ex.map(run, range(4)) for o in part]
    assert sorted(k for k, *_ in outs) == list(range(len(PAIRS)))
    for k, res, text, stats in outs:
        g, body = want[k]
        _assert_same(res, g, f"pair {PAIRS[k]}")
        assert text == body, f"pair {PAIRS[k]}: text differs"
        assert stats.tobytes() == alone[k].tobytes(), f"pair {PAIRS[k]}: statistics differ"
    for c in ctxs[1:]:
        c.close()
    base.close()


# ---- 2. full size ----------------------------------------------------------------------------------------------------
@gpu
def test_concurrent_pairs_at_10m_equal_sequential():
    import torch
    w = gen.WORKLOADS["c2"]
    n = w.n
    pairs = [(w.len_ratio, w.pos_ratio), (0.1, 0.02), (2.0, 0.3), (0.05, 1e9)]
    base = capi.Context(0)
    dev = torch.empty(n * 109 + 16, dtype=torch.uint8, device="cuda")
    base.generate_device(w, 0, n, dev.data_ptr())
    base.load(dev.data_ptr(), w.lx + 1, w.ly + 1, n=n)
    seq = [base.group(lr, pr) for lr, pr in pairs]
    ctxs = [base] + [base.view() for _ in range(3)]
    for rnd in range(2):
        with ThreadPoolExecutor(4) as ex:
            got = list(ex.map(lambda i: ctxs[i].group(*pairs[(i + rnd) % 4]), range(4)))
        for i, res in enumerate(got):
            _assert_equal_groups(res, seq[(i + rnd) % 4], f"round {rnd}, context {i}")
    for c in ctxs[1:]:
        c.close()
    base.close()
    del dev


# ---- 3. compact load: every context waits for the side copy ----------------------------------------------------------
@gpu
def test_view_of_compact_load_formats_after_the_side_copy(tmp_path):
    w, rec = _records("c2")
    key4, strand, rest4 = capi.pack_records(rec)
    (g0, body0), (g1, body1) = (_oracle(rec, w, *PAIRS[k], str(tmp_path)) for k in (0, 3))
    base = capi.Context(0)
    base.load_packed(key4, strand, rest4, w.lx + 1, w.ly + 1)
    view = base.view()  # right away: the side copy may still be running

    def on_view():
        res = view.group(*PAIRS[0])
        return res, view.format_lines()

    def on_base():
        res = base.group(*PAIRS[3])
        return res, base.format_lines()

    with ThreadPoolExecutor(2) as ex:
        fv, fb = ex.submit(on_view), ex.submit(on_base)
        (rv, tv), (rb, tb) = fv.result(), fb.result()
    _assert_same(rv, g0, "view")
    _assert_same(rb, g1, "base")
    assert tv == body0
    assert tb == body1
    view.close()
    base.close()


# ---- 4. device records -----------------------------------------------------------------------------------------------
@gpu
def test_views_format_device_records(tmp_path):
    import torch
    w, rec = _records("dense")
    dev = torch.empty(rec.shape[0] * 109 + 16, dtype=torch.uint8, device="cuda")
    base = capi.Context(0)
    base.generate_device(w, 0, rec.shape[0], dev.data_ptr())
    base.load(dev.data_ptr(), w.lx + 1, w.ly + 1, n=rec.shape[0])
    views = [base.view(), base.view()]
    want = [_oracle(rec, w, *PAIRS[k], str(tmp_path)) for k in (1, 2)]

    def run(i):
        views[i].group(*PAIRS[1 + i])
        return views[i].format_lines()

    with ThreadPoolExecutor(2) as ex:
        texts = list(ex.map(run, range(2)))
    for (g, body), t in zip(want, texts):
        assert t == body
    for v in views:
        v.close()
    base.close()
    del dev


# ---- 5. the other calls on a view ------------------------------------------------------------------------------------
@gpu
def test_other_calls_on_a_view(tmp_path):
    w, rec = _records("c3")
    lr, pr = PAIRS[1]
    g = O.group(rec, w.lx + 1, w.ly + 1, lr, pr, want_diag=True)
    base = capi.Context(0)
    st = base.load(rec, w.lx + 1, w.ly + 1)
    view = base.view()
    # RK_F_NO_SORT, then rk_sort_groups on the view
    view.group(lr, pr, sort=False)
    r = capi._Result()
    assert view._L.rk_sort_groups(C.c_void_p(view._h), C.c_uint(capi.F_HOST_RESULT), C.byref(r)) == 0, view._L.rk_last_error(view._h)
    _assert_same(capi._groups_of(r, True, True), g, "rk_sort_groups on a view")
    # the arrays of one grouping equal the base's for the same pair
    base.group(lr, pr)
    view.group(lr, pr)
    for name in ("parent", "gid_rank", "rank_fidx", "hkey"):
        assert np.array_equal(view.debug_fetch(name), base.debug_fetch(name)), name
    dv, db = view.diagonal_func(st.vsize), base.diagonal_func(st.vsize)
    assert np.array_equal(dv, db)
    assert np.array_equal(dv, g.diag_func)
    assert np.array_equal(view.diagonal_func(st.vsize), dv)  # the table buffer is reused
    view.close()
    base.close()


# ---- 6. lifetime and refusals ----------------------------------------------------------------------------------------
@gpu
def test_view_refusals():
    w, rec = _records("dense")
    with capi.Context(0) as empty:
        with pytest.raises(capi.RkError, match="holds no database"):
            empty.view()
    with capi.Multi([0, 0]) as m:
        L = m._L
        assert not L.rk_create_view(L.rk_multi_ctx(m._h, 0))  # before the load
        m.load(rec, w.lx + 1, w.ly + 1)
        for r in range(m.n):
            assert not L.rk_create_view(L.rk_multi_ctx(m._h, r))
        assert b"partitioned" in L.rk_create_error()
    base = capi.Context(0)
    base.load(rec, w.lx + 1, w.ly + 1)
    view = base.view()
    with pytest.raises(capi.RkError) as e:
        view.load(rec, w.lx + 1, w.ly + 1)
    assert e.value.code == RK_ERR_STATE
    res = view.group(*PAIRS[0])
    text, stats = view.format_lines(), view.group_statistics()
    other = replace(w, seed=w.seed + 1)
    with pytest.raises(capi.RkError) as e:
        base.load(gen.generate(other), other.lx + 1, other.ly + 1)
    assert e.value.code == RK_ERR_STATE and "1 view" in str(e.value)
    # nothing changed: the view's last result (its device arrays) and the database are as they were
    assert view.format_lines() == text
    assert view.group_statistics().tobytes() == stats.tobytes()
    _assert_equal_groups(base.group(*PAIRS[0]), res, "base after the refused load")
    view.close()
    base.close()


@gpu
def test_view_lifetime(tmp_path):
    w, rec = _records("dense")
    (g0, body0), (g1, _) = (_oracle(rec, w, *PAIRS[k], str(tmp_path)) for k in (0, 4))
    # the base closed first: its views keep the database
    base = capi.Context(0)
    base.load(rec, w.lx + 1, w.ly + 1)
    view = base.view()
    vv = view.view()  # a view of a view shares the same database
    with pytest.raises(capi.RkError, match="2 views"):
        base.load(rec, w.lx + 1, w.ly + 1)
    base.close()
    _assert_same(view.group(*PAIRS[0]), g0, "view after the base was closed")
    assert view.format_lines() == body0
    view.close()
    _assert_same(vv.group(*PAIRS[4]), g1, "view of a view, alone")
    vv.close()
    # after every view is closed, the base loads another workload, and a new view groups that one
    base = capi.Context(0)
    base.load(rec, w.lx + 1, w.ly + 1)
    view = base.view()
    view.group(*PAIRS[0])
    view.close()
    other = replace(gen.scaled(gen.WORKLOADS["c2"], 50_000), seed=7)
    orec = gen.generate(other)
    base.load(orec, other.lx + 1, other.ly + 1)
    view = base.view()
    _assert_same(view.group(*PAIRS[1]), O.group(orec, other.lx + 1, other.ly + 1, *PAIRS[1]), "new view of a reloaded base")
    view.close()
    base.close()


# ---- 7. streams ------------------------------------------------------------------------------------------------------
@gpu
def test_views_on_their_own_torch_streams():
    import torch
    w, rec = _records("c2")
    base = capi.Context(0)
    base.load(rec, w.lx + 1, w.ly + 1)
    seq = [base.group(*p) for p in PAIRS[:4]]
    views = [base.view() for _ in range(4)]
    streams = [torch.cuda.Stream() for _ in views]
    for v, s in zip(views, streams):
        v.set_stream(s.cuda_stream)
    with ThreadPoolExecutor(4) as ex:
        got = list(ex.map(lambda i: views[i].group(*PAIRS[i]), range(4)))
    for i, res in enumerate(got):
        _assert_equal_groups(res, seq[i], f"view {i}")
    for v in views:
        v.close()
    base.close()


# ---- 8. the host facades from a thread pool --------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("threads", [3, 1])
def test_hostcheck_pool_equals_steps(medium_cases, tmp_path, threads):
    c = medium_cases["c1"]
    w = gen.Workload(**c["workload"])
    rec = gen.generate(w)
    inp = tmp_path / "c1.csv"
    O.write_input_csv(str(inp), rec, w.lx, w.ly)
    pairs = [(0.05, 0.05), (0.1, 0.02), (1e-3, 1e-3), (2.0, 0.3), (0.05, 1e9), (0.3, 0.1)]
    prefix = tmp_path / "pool"
    args = [a for p in pairs for a in map(repr, p)]
    p = subprocess.run([HOSTCHECK, "pool", str(inp), str(prefix), str(threads), *args], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    used = int(re.search(r"(\d+) grouping contexts", p.stdout).group(1))
    assert 1 <= used <= threads, p.stdout
    for k, (lr, pr) in enumerate(pairs):
        alone = tmp_path / f"steps-{k}.csv"
        q = subprocess.run([HOSTCHECK, "steps", str(inp), str(alone), repr(lr), repr(pr)], capture_output=True, text=True)
        assert q.returncode == 0, q.stderr
        got = (tmp_path / f"pool-{k}.csv").read_bytes()
        assert got == alone.read_bytes(), f"pair {k}"
        if (lr, pr) == (0.05, 0.05):
            assert hashlib.md5(got).hexdigest() == c["ref_md5"]


# ---- 9. without a GPU ------------------------------------------------------------------------------------------------
def test_create_view_is_exported():
    lib = capi.LIB_PATH
    if not os.path.exists(lib):
        pytest.skip("library not built")
    out = subprocess.run(["nm", "-D", "--defined-only", lib], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r"\bT (rk_\w+)$", out, flags=re.M))
    assert "rk_create_view" in exported
    assert "rk_create_view" in capi.SYMBOLS
