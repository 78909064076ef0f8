"""The grow-only buffers of a context (text, statistics, diagonal table, rk_sort_members scratch, host result) as they
grow, on a context that loads, on a view (whose workspace and host result are allocated in rk_create_view and never
grow) and through rk_multi:
  * format_lines hands back one of two alternating text buffers: chunk k stays readable through its own pointer while
    chunk k+1 is formatted, also when the next chunk makes a buffer grow (chunks of 1, FORMAT_MAX_LINES and 1 lines);
  * group_statistics after a grouping with more groups, diagonal_func after a reload with a larger vsize, sort_members
    with increasing m, and the host result after a reload with more records equal the oracle's."""
import ctypes as C
import os
from dataclasses import replace

import numpy as np
import pytest

from oracle import oracle as O
from repkiller_b200 import capi, gen

gpu = pytest.mark.gpu
LOOSE, STRICT = (2.0, 0.3), (0.05, 0.05)  # STRICT gives 3.7x the groups of LOOSE on these workloads


def _workload(n):
    return gen.scaled(gen.WORKLOADS["c2"], n)


def _oracle(rec, w, pair, tmp_dir, body=False):
    g = O.group(rec, w.lx + 1, w.ly + 1, *pair, want_diag=True)
    if not body:
        return g, None
    path = os.path.join(tmp_dir, "oracle_body.csv")
    O.write_output(path, b"", rec, g)
    with open(path, "rb") as f:
        text = f.read()
    os.remove(path)
    return g, text


def _assert_same(res, g, what):
    assert res.n_kept == g.n_kept and res.n_groups == g.n_groups, what
    for name, got, want in (("order", res.order, g.order), ("gid", res.gid, g.out_gid), ("repval", res.repval, g.repval),
                            ("identity", res.identity.view(np.uint32), g.identity.view(np.uint32))):
        assert np.array_equal(got, want), f"{what}: {name}"


def _assert_stats_grow(ctx, rec, w, tmp_dir, g_strict=None):
    """statistics of a grouping with LOOSE, then of one with STRICT: enough more groups that both buffers grow"""
    loose = ctx.group(*LOOSE)
    ctx.group_statistics()
    strict = ctx.group(*STRICT)
    assert strict.n_groups > loose.n_groups + loose.n_groups // 8 + 1024
    g = g_strict if g_strict is not None else _oracle(rec, w, STRICT, tmp_dir)[0]
    _assert_same(strict, g, "STRICT")
    assert ctx.group_statistics().tobytes() == O.group_statistics(rec, g).tobytes()


def _assert_sort_members_grows(ctx):
    rng = np.random.default_rng(11)
    for m in (1_000, 40_000, 1_500_000):  # the scratch grows on every call
        sizes = np.diff(np.r_[0, np.sort(rng.choice(np.arange(1, m), 7, replace=False)), m])
        gid = np.repeat(np.arange(sizes.size), sizes).astype(np.uint32)
        h = rng.integers(0, 1 << 16, m).astype(np.uint64)  # ties: std::sort's order, not a stable one
        d = rng.integers(1 << 30, 1 << 31, m).astype(np.uint64)
        perm = ctx.sort_members(gid, d + h, d)
        pos = 0
        for n in sizes:
            idx = np.arange(pos, pos + n, dtype=np.uint32)
            assert np.array_equal(perm[pos:pos + n], O.std_sort_by_key(idx, h)), (m, pos, n)
            pos += n


def _assert_text_alternates(call, body, chunks):
    """format the chunks [(first line, lines)] in a row with call(first, lines, byref(rk_text)); read every chunk through
    the pointer it was handed back with only after the next one is formatted"""
    nl = np.flatnonzero(np.frombuffer(body, np.uint8) == 10)

    def want(a, k):
        return body[0 if a == 0 else nl[a - 1] + 1:nl[a + k - 1] + 1]

    def check(i):
        (a, k), t = chunks[i], texts[i]
        assert C.string_at(t.text, t.n_bytes) == want(a, k), f"chunk of {k} lines at {a}"

    texts = []
    for i, (a, k) in enumerate(chunks):
        texts.append(capi._Text())
        call(a, k, C.byref(texts[i]))
        if i:
            check(i - 1)
    check(len(chunks) - 1)


def _ctx_format(ctx):
    return lambda a, k, t: ctx._check(ctx._L.rk_format_lines(ctx._h, a, k, t))


@gpu
def test_buffers_grow_on_a_context_and_a_view(tmp_path):
    small = _workload(300_000)
    big = replace(_workload(capi.FORMAT_MAX_LINES + 50_000), seed=small.seed + 1)
    srec, brec = gen.generate(small), gen.generate(big)
    assert big.lx > small.lx
    ctx = capi.Context(0)
    st = ctx.load(srec, small.lx + 1, small.ly + 1)
    _assert_stats_grow(ctx, srec, small, str(tmp_path))
    g, body = _oracle(srec, small, LOOSE, str(tmp_path), body=True)
    _assert_same(ctx.group(*LOOSE), g, "small load")
    assert np.array_equal(ctx.diagonal_func(st.vsize), g.diag_func)
    _assert_text_alternates(_ctx_format(ctx), body, [(0, 1), (1, 5_000), (5_001, 1)])
    _assert_sort_members_grows(ctx)

    # a reload with more records and a larger vsize: host result, statistics, diagonal table and text grow
    gb, bbody = _oracle(brec, big, STRICT, str(tmp_path), body=True)
    st = ctx.load(brec, big.lx + 1, big.ly + 1)
    assert st.n_kept >= capi.FORMAT_MAX_LINES + 2 and st.vsize > small.lx // 10
    _assert_same(ctx.group(*STRICT), gb, "larger load")
    assert ctx.group_statistics().tobytes() == O.group_statistics(brec, gb).tobytes()
    assert np.array_equal(ctx.diagonal_func(st.vsize), gb.diag_func)
    chunks = [(0, 1), (1, capi.FORMAT_MAX_LINES), (1 + capi.FORMAT_MAX_LINES, 1)]
    _assert_text_alternates(_ctx_format(ctx), bbody, chunks)

    # a view: the same calls on buffers that start empty (the base is closed first; the view keeps the database)
    view = ctx.view()
    ctx.close()
    _assert_stats_grow(view, brec, big, str(tmp_path), g_strict=gb)
    assert np.array_equal(view.diagonal_func(st.vsize), gb.diag_func)
    _assert_text_alternates(_ctx_format(view), bbody, chunks)
    _assert_sort_members_grows(view)
    view.close()


@gpu
def test_buffers_grow_through_multi(tmp_path):
    small, big = _workload(60_000), replace(_workload(400_000), seed=5)
    srec, brec = gen.generate(small), gen.generate(big)
    with capi.Multi([0, 0, 0]) as mg:
        mg.load(srec, small.lx + 1, small.ly + 1)
        _assert_same(mg.group(*LOOSE, line_records=True), _oracle(srec, small, LOOSE, str(tmp_path))[0], "small load")
        mg.group_statistics()
        # the merged host result, the statistics and the text after a larger load
        mg.load(brec, big.lx + 1, big.ly + 1)
        g, body = _oracle(brec, big, STRICT, str(tmp_path), body=True)
        res = mg.group(*STRICT, line_records=True)
        _assert_same(res, g, "larger load")
        assert mg.group_statistics().tobytes() == O.group_statistics(brec, g).tobytes()
        call = lambda a, k, t: mg._check(mg._L.rk_multi_format_lines(mg._h, a, k, t))
        _assert_text_alternates(call, body, [(0, 1), (1, 5_000), (5_001, res.n_kept - 5_002), (res.n_kept - 1, 1)])
