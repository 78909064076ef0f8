"""GECKO CSV rows parsed on the device for a comparison partitioned over several GPUs (rk_dist_load_csv, rk_multi_load_csv):
the groups, the output text and the statistics equal rk_load_csv + rk_group on one GPU (and the oracle), the row counts
add up to one GPU's, and every refusal reaches every rank with the same code and message.  The ranks are threads on
GPU 0 (capi.Multi([0] * k)); the caller-slice cases call rk_dist_load_csv on the ranks' contexts from a thread pool.
Run on the B200 box: python -m pytest tests -m gpu"""
import ctypes as C
import hashlib
import os
import socket
import sys
from concurrent.futures import ThreadPoolExecutor
from dataclasses import replace

import numpy as np
import pytest

from oracle import oracle as O
from repkiller_b200 import capi, gen, multi

pytestmark = pytest.mark.gpu

RK_ERR_ARG, RK_ERR_RANGE, RK_ERR_NOMEM = -2, -3, -5


def _workload(name):  # the workloads of test_gpu_multi.py
    if name == "dense":
        return replace(gen.WORKLOADS["c1"], n=60_000, lx=400_000, ly=300_000, families=40, p_rep=0.6, seed=31)
    if name == "tiny":
        return replace(gen.WORKLOADS["c1"], n=3_000, lx=30_000, ly=25_000, families=12, p_rep=0.6, seed=21)
    if name == "c3":
        return gen.scaled(gen.WORKLOADS["c3"], 200_000)
    return gen.scaled(gen.WORKLOADS["c2"], 300_000)


def split_head(text: bytes):
    """(body, total_frags): 16 header lines, then the rest; "Total fragments" is line 13"""
    pos = 0
    lines = []
    for _ in range(16):
        nl = text.find(b"\n", pos)
        lines.append(text[pos:len(text) if nl < 0 else nl])
        pos = len(text) if nl < 0 else nl + 1
    s = lines[12]
    s = s[s.index(b":") + 1:] if b":" in s else s
    digits = s.strip()
    return text[pos:], int(digits) if digits.isdigit() else 0


def _csv_case(w, tmp_dir):
    """(csv path, loaded records, lx1, ly1, header, body, total) of a generated workload written as CSV"""
    path = os.path.join(tmp_dir, f"{w.name}_{w.n}.csv")
    O.write_input_csv(path, gen.generate(w), w.lx, w.ly)
    rec, lx1, ly1, hdr = O.load_csv(path)
    with open(path, "rb") as f:
        body, total = split_head(f.read())
    return path, rec, lx1, ly1, hdr, body, total


def _one_gpu(body, lx1, ly1, total, lr, pr):
    """rk_load_csv + rk_group on one GPU: (csv stats, groups, text, statistics)"""
    with capi.Context(0) as ctx:
        _, cs = ctx.load_csv(body, lx1, ly1, total)
        res = ctx.group(lr, pr)
        return cs, res, ctx.format_lines(), ctx.group_statistics()


def _assert_same(res, want):
    assert res.n_kept == want.n_kept and res.n_groups == want.n_groups, (res.n_kept, want.n_kept, res.n_groups, want.n_groups)
    for name in ("order", "gid", "repval", "identity"):
        a, b = getattr(res, name), getattr(want, name)
        if name == "identity":
            a, b = a.view(np.uint32), b.view(np.uint32)
        d = np.nonzero(a != b)[0]
        assert d.size == 0, f"{name}: {d.size} differences, first at {d[:5]}"


def _assert_oracle(res, g):
    assert res.n_kept == g.n_kept and res.n_groups == g.n_groups
    assert np.array_equal(res.order, g.order) and np.array_equal(res.gid, g.out_gid) and np.array_equal(res.repval, g.repval)
    assert np.array_equal(res.identity.view(np.uint32), g.identity.view(np.uint32))


def _same_stats(got, want):
    """every field bit for bit: the statistics are exact, whatever the partition"""
    assert got.shape == want.shape
    for f in got.dtype.names:
        assert got[f].tobytes() == want[f].tobytes(), f


def _first_diff(a: bytes, b: bytes) -> str:
    i = next((k for k in range(min(len(a), len(b))) if a[k] != b[k]), min(len(a), len(b)))
    return f"{len(a)} vs {len(b)} bytes, first difference at byte {i}: {a[max(0, i - 60):i + 60]!r} vs {b[max(0, i - 60):i + 60]!r}"


def _handles(m):
    return [m._L.rk_multi_ctx(m._h, r) for r in range(m.n)]


def _dist_load(m, slices, lx1, ly1, total):
    """rk_dist_load_csv on every rank's context at once: (return codes, messages, csv stats)"""
    L, hs = m._L, _handles(m)
    st = [capi._LoadStats() for _ in hs]
    cs = [capi._CsvStats() for _ in hs]

    def one(r):
        s = slices[r]
        if isinstance(s, (bytes, bytearray)):
            arr = np.frombuffer(bytes(s), dtype=np.uint8)
            ptr, n = arr.ctypes.data, arr.nbytes
        else:   # a CUDA tensor (view) of the body
            ptr, n = s.data_ptr(), s.numel()
        return L.rk_dist_load_csv(hs[r], C.c_void_p(ptr) if n else None, n, lx1, ly1, total, 0, C.byref(st[r]), C.byref(cs[r]))

    with ThreadPoolExecutor(m.n) as ex:
        rcs = list(ex.map(one, range(m.n)))
    return rcs, [L.rk_last_error(h).decode() for h in hs], cs


def _dist_text(m, lr, pr):
    """rk_dist_group with RK_F_LINE_RECORDS on every rank, then every rank's lines: (n_groups, text)"""
    L, hs = m._L, _handles(m)
    res = [capi._Result() for _ in hs]
    info = [capi._DistInfo() for _ in hs]
    with ThreadPoolExecutor(m.n) as ex:
        rcs = list(ex.map(lambda r: L.rk_dist_group(hs[r], lr, pr, capi.F_LINE_RECORDS, C.byref(res[r]), C.byref(info[r])),
                          range(m.n)))
    assert rcs == [0] * m.n, [L.rk_last_error(h) for h in hs]
    parts = []
    for r in range(m.n):
        t = capi._Text()
        assert L.rk_dist_format_lines(hs[r], 0, info[r].n_lines, C.byref(t)) == 0, L.rk_last_error(hs[r])
        parts.append(C.string_at(t.text, t.n_bytes) if t.n_bytes else b"")
    return res[0].n_groups, b"".join(parts)


def _even_cuts(body: bytes, k: int):
    """rk_multi_load_csv's cuts"""
    cuts = [0]
    for r in range(1, k):
        a = len(body) * r // k
        nl = body.find(b"\n", a)
        cuts.append(len(body) if nl < 0 else nl + 1)
    return cuts + [len(body)]


def _slices(body, cuts):
    return [body[a:b] for a, b in zip(cuts, cuts[1:])]


# ---- 1. parity: Multi.load_csv against one GPU, the oracle and Multi.load --------------------------------------------
@pytest.fixture(scope="module")
def cases(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("csv"))
    out = {}
    for wl in ("tiny", "dense", "c2", "c3"):
        w = _workload(wl)
        _, rec, lx1, ly1, _, body, total = _csv_case(w, d)
        g = O.group(rec, lx1, ly1, w.len_ratio, w.pos_ratio)
        out[wl] = (w, rec, lx1, ly1, body, total, g, _one_gpu(body, lx1, ly1, total, w.len_ratio, w.pos_ratio))
    return out


@pytest.mark.parametrize("world", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("wl", ["tiny", "dense", "c2", "c3"])
def test_multi_load_csv_equals_one_gpu(cases, world, wl):
    w, rec, lx1, ly1, body, total, g, (cs1, res1, text1, stats1) = cases[wl]
    with capi.Multi([0] * world) as m:
        st, cs = m.load_csv(body, lx1, ly1, total)
        assert (cs.n_rows, cs.n_accepted, cs.n_host_rows, cs.wide) == (cs1.n_rows, cs1.n_accepted, cs1.n_host_rows, cs1.wide)
        assert st.n_loaded == rec.shape[0]
        res = m.group(w.len_ratio, w.pos_ratio, line_records=True)
        _assert_oracle(res, g)
        _assert_same(res, res1)
        text = m.format_lines()
        assert text == text1, _first_diff(text, text1)
        _same_stats(m.group_statistics(), stats1)
        # the same records through rk_multi_load_aos on the same ranks
        m.load(rec, lx1, ly1)
        _assert_same(m.group(w.len_ratio, w.pos_ratio, line_records=True), res1)
        assert m.format_lines() == text1


def test_c2_full_size_three_ranks(tmp_path):
    w = gen.WORKLOADS["c2"]
    path = str(tmp_path / "c2.csv")
    O.write_input_csv(path, gen.generate(w), w.lx, w.ly)
    with open(path, "rb") as f:
        body, total = split_head(f.read())
    os.remove(path)
    lx1, ly1 = w.lx + 1, w.ly + 1
    with capi.Context(0) as ctx:
        _, cs1 = ctx.load_csv(body, lx1, ly1, total)
        res1 = ctx.group(w.len_ratio, w.pos_ratio)
        md5_1 = hashlib.md5(ctx.format_lines()).hexdigest()
    with capi.Multi([0, 0, 0]) as m:
        _, cs = m.load_csv(body, lx1, ly1, total, timing=True)
        print(f"\nC2 10M over 3 ranks on one GPU: upload {cs.ms_upload:.2f} ms, parse {cs.ms_parse:.2f} ms (largest rank)")
        assert (cs.n_rows, cs.n_accepted, cs.n_host_rows) == (cs1.n_rows, cs1.n_accepted, cs1.n_host_rows)
        assert (cs.n_rows, cs.n_accepted) == (w.n + 1, w.n)
        res = m.group(w.len_ratio, w.pos_ratio, line_records=True)
        _assert_same(res, res1)
        assert hashlib.md5(m.format_lines()).hexdigest() == md5_1


# ---- 2. the 120 fuzz CSVs over 2 and 3 ranks -------------------------------------------------------------------------
def _outcome(fn):
    try:
        return 0, fn()
    except capi.RkError as e:
        return e.code, str(e)


def test_fuzz_cases_two_and_three_ranks(fuzz_cases):
    refused = grouped = 0
    with capi.Context(0) as ctx, capi.Multi([0, 0]) as m2, capi.Multi([0, 0, 0]) as m3:
        for c in fuzz_cases:
            text = c["csv"].encode("latin1")
            body, total = split_head(text)
            lx1 = ly1 = None
            try:
                import tempfile
                with tempfile.NamedTemporaryFile(suffix=".csv") as f:
                    f.write(text)
                    f.flush()
                    _, lx1, ly1, _ = O.load_csv(f.name)
            except RuntimeError:
                lx1, ly1 = 1000, 1000   # more rows than "Total fragments": refused before the lengths matter
            rc1, got1 = _outcome(lambda: ctx.load_csv(body, lx1, ly1, total)[1])
            for m in (m2, m3):
                rc, got = _outcome(lambda: m.load_csv(body, lx1, ly1, total)[1])
                assert rc == rc1, (c["seed"], m.n, got, got1)
                if rc:
                    if rc1 == RK_ERR_RANGE and "Unexpected number of fragments" in got1:
                        assert "Unexpected number of fragments" in got, (c["seed"], got)
                    refused += 1
                    continue
                assert (got.n_rows, got.n_accepted, got.n_host_rows, got.wide) == \
                    (got1.n_rows, got1.n_accepted, got1.n_host_rows, got1.wide), c["seed"]
                g1 = _outcome(lambda: ctx.group(c["len_ratio"], c["pos_ratio"]))
                g = _outcome(lambda: m.group(c["len_ratio"], c["pos_ratio"], line_records=True))
                assert g[0] == g1[0], (c["seed"], g, g1)
                if g[0]:
                    continue
                _assert_same(g[1], g1[1])
                assert m.format_lines() == ctx.format_lines(), (c["seed"], m.n)
                grouped += 1
    assert grouped > 100


# ---- 3. caller slices through rk_dist_load_csv -----------------------------------------------------------------------
def _mixed_body(body: bytes) -> bytes:
    """rows in the host parser's grammar spread over the whole body: signs, exponents, CRLF, plus rejected rows"""
    rows = body.split(b"\n")
    for i in range(0, len(rows) - 1, 37):
        t = rows[i].split(b",")
        if len(t) < 14:
            continue
        k = i // 37 % 4
        if k == 0:
            t[1] = b"+" + t[1]
        elif k == 1:
            t[10] = b"%.6e" % float(t[10])
        elif k == 2:
            t[-1] = t[-1] + b"\r"
        else:
            t[0] = b"Frog"
        rows[i] = b",".join(t)
    return b"\n".join(rows)


@pytest.fixture(scope="module")
def sliced(tmp_path_factory):
    w = _workload("dense")
    _, _, lx1, ly1, _, body, total = _csv_case(w, str(tmp_path_factory.mktemp("sl")))
    body = _mixed_body(body)
    cs1, res1, text1, _ = _one_gpu(body, lx1, ly1, total, w.len_ratio, w.pos_ratio)
    assert cs1.n_host_rows > 0
    return w, body, lx1, ly1, total, cs1, res1, text1


def _check_slices(m, sliced, slices, n_rows_each=None):
    w, body, lx1, ly1, total, cs1, res1, text1 = sliced
    rcs, errs, cs = _dist_load(m, slices, lx1, ly1, total)
    assert rcs == [0] * m.n, errs
    assert sum(c.n_rows for c in cs) == cs1.n_rows
    assert sum(c.n_accepted for c in cs) == cs1.n_accepted
    assert sum(c.n_host_rows for c in cs) == cs1.n_host_rows
    if n_rows_each is not None:
        assert [c.n_rows for c in cs] == n_rows_each
    n_groups, text = _dist_text(m, w.len_ratio, w.pos_ratio)
    assert n_groups == res1.n_groups
    assert text == text1, _first_diff(text, text1)
    return cs


def test_cuts_at_every_row_boundary_near_the_even_split(sliced):
    body = sliced[1]
    with capi.Multi([0, 0, 0]) as m:
        m.load_csv(body, sliced[2], sliced[3], sliced[4])   # sizes the ranks' buffers
        even = _even_cuts(body, 3)
        for d in range(-3, 4):
            cut = even[1]
            for _ in range(abs(d)):   # d rows before / after the even cut
                cut = body.rfind(b"\n", 0, cut - 1) + 1 if d < 0 else body.find(b"\n", cut) + 1
            _check_slices(m, sliced, _slices(body, [0, cut, even[2], len(body)]))


def test_empty_slices_and_the_final_empty_row(sliced):
    body = sliced[1]
    assert body.endswith(b"\n")
    n_nl = body.count(b"\n")
    with capi.Multi([0] * 4) as m:
        m.load_csv(body, sliced[2], sliced[3], sliced[4])
        c = _even_cuts(body, 2)
        _check_slices(m, sliced, [b"", body[:c[1]], body[c[1]:], b""])         # empty first and last
        _check_slices(m, sliced, [body[:c[1]], b"", b"", body[c[1]:]])         # empty middle
        # the last rank holds only the final empty row
        cs = _check_slices(m, sliced, [body[:c[1]], body[c[1]:], b"", b""])
        assert [x.n_rows for x in cs][2:] == [0, 1]
        # all of it on one rank
        _check_slices(m, sliced, [b"", body, b"", b""], [0, n_nl, 0, 1])
        _check_slices(m, sliced, [b"", b"", b"", body], [0, 0, 0, n_nl + 1])


def test_a_slice_of_rejected_rows_only(sliced):
    w, body, lx1, ly1, total = sliced[:5]
    c = _even_cuts(body, 2)[1]
    junk = b"Junk,1,2,3\n" * 40 + b"\n" * 3 + b"Frag,,2,3\n" * 5   # (an empty token rejects a row; a short one does not)
    body2 = body[:c] + junk + body[c:]
    want = _one_gpu(body2, lx1, ly1, total, w.len_ratio, w.pos_ratio)
    with capi.Multi([0, 0, 0]) as m:
        m.load_csv(body2, lx1, ly1, total)
        cs = _check_slices(m, (w, body2, lx1, ly1, total) + want[:2] + (want[2],),
                           [body2[:c], body2[c:c + len(junk)], body2[c + len(junk):]])
        assert cs[1].n_accepted == 0 and cs[1].n_rows == junk.count(b"\n")


def test_one_wide_rank_among_compact_ones(sliced, tmp_path):
    """a 40-bit xEnd on a row of rank 1: that rank keeps 109-byte records, the others compact rows; same text and groups"""
    w, body, lx1, ly1, total = sliced[:5]
    c = _even_cuts(body, 3)
    row_start = body.find(b"\n", (c[1] + c[2]) // 2) + 1
    while not body.startswith(b"Frag,", row_start):   # a row the parser accepts
        row_start = body.find(b"\n", row_start) + 1
    row_end = body.find(b"\n", row_start)
    t = body[row_start:row_end].split(b",")
    t[3] = str(1 << 40).encode()
    body2 = body[:row_start] + b",".join(t) + body[row_end:]
    want = _one_gpu(body2, lx1, ly1, total, w.len_ratio, w.pos_ratio)
    assert want[0].wide and b"1099511627776" in want[2]
    with capi.Multi([0, 0, 0]) as m:
        m.load_csv(body2, lx1, ly1, total)
        cs = _check_slices(m, (w, body2, lx1, ly1, total) + want[:2] + (want[2],), _slices(body2, _even_cuts(body2, 3)))
        assert [bool(x.wide) for x in cs] == [False, True, False]
        _, csm = m.load_csv(body2, lx1, ly1, total)
        assert csm.wide


def test_device_slices_aligned_and_at_odd_offsets(sliced):
    import torch
    body = sliced[1]
    dev = torch.frombuffer(bytearray(body), dtype=torch.uint8).cuda()
    with capi.Multi([0, 0, 0]) as m:
        m.load_csv(body, sliced[2], sliced[3], sliced[4])
        cuts = _even_cuts(body, 3)
        assert any(x % 16 for x in cuts[1:-1])
        views = [dev[a:b] for a, b in zip(cuts, cuts[1:])]            # views of one resident body: odd offsets
        _check_slices(m, sliced, views)
        own = [v.clone() for v in views]                               # each slice in its own (aligned) allocation
        torch.cuda.synchronize()
        rcs, errs, _ = _dist_load(m, own, sliced[2], sliced[3], sliced[4])
        assert rcs == [0] * 3, errs
        del own, views, dev                                            # the parsed rows are the ranks' own
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        n_groups, text = _dist_text(m, sliced[0].len_ratio, sliced[0].pos_ratio)
        assert n_groups == sliced[6].n_groups and text == sliced[7], _first_diff(text, sliced[7])


# ---- 4. refusals: the same code and message on every rank, then a normal load works ----------------------------------
def _tiny(tmp_dir):
    w = _workload("tiny")
    _, rec, lx1, ly1, _, body, total = _csv_case(w, tmp_dir)
    return w, rec, lx1, ly1, body, total


def _still_works(m, tiny):
    w, rec, lx1, ly1, body, total = tiny
    m.load_csv(body, lx1, ly1, total)
    _assert_oracle(m.group(w.len_ratio, w.pos_ratio, line_records=True), O.group(rec, lx1, ly1, w.len_ratio, w.pos_ratio))


def test_refusals_reach_every_rank(tmp_path):
    tiny = _tiny(str(tmp_path))
    w, rec, lx1, ly1, body, total = tiny
    with capi.Multi([0, 0, 0]) as m:
        m.load_csv(body, lx1, ly1, total)
        cuts = _even_cuts(body, 3)
        # a non-last slice that does not end with '\n'
        bad = [body[:cuts[1] - 5], body[cuts[1] - 5:cuts[2]], body[cuts[2]:]]
        rcs, errs, _ = _dist_load(m, bad, lx1, ly1, total)
        assert rcs == [RK_ERR_ARG] * 3 and len(set(errs)) == 1 and "does not end with" in errs[0], errs
        _still_works(m, tiny)
        # every rank within "Total fragments", the sum over it
        rcs, errs, _ = _dist_load(m, _slices(body, cuts), lx1, ly1, total - 1)
        assert rcs == [RK_ERR_RANGE] * 3 and set(errs) == {"Unexpected number of fragments"}, errs
        _still_works(m, tiny)
        # one rank over the capacity the tiny load gave the ranks
        big = replace(_workload("c2"), n=400_000)
        _, _, _, _, _, big_body, big_total = _csv_case(big, str(tmp_path))
        rcs, errs, _ = _dist_load(m, [b"", big_body, b""], big.lx + 1, big.ly + 1, big_total)
        assert rcs == [RK_ERR_NOMEM] * 3 and len(set(errs)) == 1 and "capacity" in errs[0], errs
        _still_works(m, tiny)
        # one rank's own parse fails (a null text pointer): every rank returns its code and the same message
        hs = _handles(m)
        with ThreadPoolExecutor(3) as ex:
            arr = np.frombuffer(body, dtype=np.uint8)
            rcs = list(ex.map(lambda r: m._L.rk_dist_load_csv(hs[r], None if r == 1 else C.c_void_p(arr.ctypes.data), 10 if r == 1 else 0,
                                                                lx1, ly1, total, 0, None, None), range(3)))
        errs = [m._L.rk_last_error(h).decode() for h in hs]
        assert rcs == [RK_ERR_ARG] * 3 and len(set(errs)) == 1 and errs[0].startswith("rank 1 could not parse") \
            and "null text pointer" in errs[0], errs
        _still_works(m, tiny)
        # rk_multi_load_csv refuses device text
        import torch
        with pytest.raises(capi.RkError) as e:
            m.load_csv(torch.frombuffer(bytearray(body), dtype=torch.uint8).cuda(), lx1, ly1, total)
        assert e.value.code == RK_ERR_ARG
        _still_works(m, tiny)


# ---- 5. the CLI under RK_DEVICES ---------------------------------------------------------------------------------------
CLI = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "repkiller_b200", "bin", "repkiller")


def _cli(inp, outp, *ratios, **env):
    import subprocess
    e = dict(os.environ, RK_DEVICES="0,0,0", RK_TIMING="1")
    e.update(env)
    return subprocess.run([CLI, str(inp), str(outp), *ratios], capture_output=True, env=e)


def test_cli_medium_goldens_parse_on_every_device(tmp_path, medium_cases):
    done = 0
    for name in ("c1", "c1_loose", "dense"):
        if name not in medium_cases:
            continue
        c = medium_cases[name]
        w = gen.Workload(**c["workload"])
        inp = tmp_path / f"{name}.csv"
        O.write_input_csv(str(inp), gen.generate(w), w.lx, w.ly)
        for env in ({}, {"RK_LEGACY_WRITER": "1"}):
            outp = tmp_path / "out.csv"
            p = _cli(inp, outp, str(w.len_ratio), str(w.pos_ratio), **env)
            assert p.returncode == 0, p.stderr
            assert hashlib.md5(outp.read_bytes()).hexdigest() == c["ref_md5"], (name, env)
            assert b" parser=device " in p.stderr and b"device_parse_ms=" in p.stderr and b"host_rows=" in p.stderr, p.stderr
            done += 1
    assert done


def test_cli_fuzz_under_rk_devices(tmp_path, fuzz_cases):
    ok = refused = 0
    for c in fuzz_cases[::3]:
        inp, outp = tmp_path / "in.csv", tmp_path / "out.csv"
        inp.write_bytes(c["csv"].encode("latin1"))
        if outp.exists():
            outp.unlink()
        try:
            O.load_csv(str(inp))
            want_ok = True
        except RuntimeError:
            want_ok = False
        for env in ({}, {"RK_LEGACY_WRITER": "1"}):
            p = _cli(inp, outp, str(c["len_ratio"]), str(c["pos_ratio"]), **env)
            if not want_ok:   # the reference's uncaught exception, as on one GPU
                assert p.returncode != 0 and b"Unexpected number of fragments" in p.stderr, c["seed"]
                refused += 1
                continue
            assert p.returncode == 0, p.stderr
            assert b" parser=device " in p.stderr
            assert outp.read_bytes() == c["ref_out"].encode("latin1"), (c["seed"], env)
            ok += 1
    assert ok > 20


def test_cli_over_count_file_fails_as_on_one_gpu(tmp_path):
    from repkiller_b200 import frags
    w = gen.scaled(gen.WORKLOADS["c1"], 2_000)
    inp = tmp_path / "short.csv"
    frags.write_csv(str(inp), gen.generate(w), w.lx, w.ly, total_frags=w.n - 1)
    p = _cli(inp, tmp_path / "o.csv", "0.05", "0.05")
    one = _cli(inp, tmp_path / "o1.csv", "0.05", "0.05", RK_DEVICES="0")
    assert p.returncode == one.returncode != 0
    assert b"Unexpected number of fragments" in p.stderr and b"Unexpected number of fragments" in one.stderr


def test_cli_frags_input_keeps_the_host_parser(tmp_path):
    from repkiller_b200 import frags
    w = gen.scaled(gen.WORKLOADS["c1"], 3_000)
    rec = gen.generate(w)
    binp = tmp_path / "in.frags"
    frags.write_gecko_binary(str(binp), rec, w.lx, w.ly)
    p = _cli(binp, tmp_path / "o.csv", "0.05", "0.05")
    assert p.returncode == 0, p.stderr
    assert b" parser=host" in p.stderr and b"parser=device" not in p.stderr


# ---- 6. one process per GPU over NCCL, each reading its own bytes of the file ----------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, path, body_pos, lx1, ly1, total, lr, pr, out_dir):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(rank)
    lo, hi = multi.csv_slice_bounds(path, body_pos, rank, world)
    with open(path, "rb") as f:
        f.seek(lo)
        mine = f.read(hi - lo)
    ctx = capi.Context(rank)
    multi.bootstrap(ctx, multi.default_capacity(total // world + 16))   # (the same capacity on every rank)
    ctx.dist_load_csv(mine, lx1, ly1, total)
    ctx.dist_group(lr, pr, line_records=True)
    with open(os.path.join(out_dir, f"r{rank}.txt"), "wb") as f:
        f.write(ctx.dist_format_lines())
    dist.barrier()
    ctx.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_nccl_processes_read_their_own_slices(tmp_path, world):
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    import torch.multiprocessing as mp
    w = _workload("c2")
    path, rec, lx1, ly1, _, body, total = _csv_case(w, str(tmp_path))
    body_pos = os.path.getsize(path) - len(body)
    g = O.group(rec, lx1, ly1, w.len_ratio, w.pos_ratio)
    want = os.path.join(str(tmp_path), "oracle.csv")
    O.write_output(want, b"", rec, g)
    mp.spawn(_worker, args=(world, _free_port(), path, body_pos, lx1, ly1, total, w.len_ratio, w.pos_ratio, str(tmp_path)),
             nprocs=world, join=True)
    text = b"".join(open(os.path.join(tmp_path, f"r{r}.txt"), "rb").read() for r in range(world))
    assert text == open(want, "rb").read()
