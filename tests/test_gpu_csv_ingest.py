"""GECKO CSV rows parsed on the device (rk_load_csv, k9_csv.cu) against the oracle's restatement of the reference's loader
(oracle.load_csv) and the reference's golden bytes: the loaded arrays bit for bit, the processing order, the groups and the
output text; the rows outside the fast-path grammar go to the host parser and nowhere else.
Run on the B200 box: python -m pytest tests -m gpu"""
import hashlib
import os
import re
import struct
import subprocess

import numpy as np
import pytest

from oracle import oracle as O
from repkiller_b200 import capi, gen
from repkiller_b200.frags import make_header

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "repkiller_b200", "bin", "repkiller")
HOSTCHECK = os.path.join(ROOT, "repkiller_b200", "bin", "rk_hostcheck")
TEXT_FIELDS = ("xStart", "yStart", "length", "ident", "xEnd", "yEnd", "score")


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def ref_ctx():
    c = capi.Context(0)
    yield c
    c.close()


def split_head(text: bytes):
    """(body, total_frags) as the reference reads them: 16 lines, then the rest; line 13's value through atoll"""
    pos = 0
    lines = []
    for _ in range(16):
        nl = text.find(b"\n", pos)
        lines.append(text[pos:len(text) if nl < 0 else nl])
        pos = len(text) if nl < 0 else nl + 1
    s = lines[12]
    s = s[s.index(b":") + 1:] if b":" in s else s
    m = re.match(rb"[ \t\n\v\f\r]*([+-]?\d+)", s)
    return text[pos:], int(m.group(1)) if m else 0


def wide(rec):
    return rec.shape[0] and any(int(rec[f].max()) >> 32 for f in TEXT_FIELDS)


def compact(rec):
    key4 = np.stack([rec[f].astype(np.uint32) for f in ("xStart", "yStart", "length", "ident")], axis=1)
    rest4 = np.stack([rec["xEnd"].astype(np.uint32), rec["yEnd"].astype(np.uint32), rec["score"].astype(np.uint32),
                      rec["similarity"].view(np.uint32)], axis=1)
    return key4, rec["strand"].view(np.uint8), rest4


def load_both(ctx, ref_ctx, text: bytes, tmp_path, body_arg=None):
    """load the text through rk_load_csv and the oracle's records through rk_load_aos; the same outcome either way.
    Returns (records, lx1, ly1, header, csv stats) or None when both refused the records alike."""
    path = tmp_path / "in.csv"
    path.write_bytes(text)
    body, total = split_head(text)
    try:
        rec, lx1, ly1, hdr = O.load_csv(str(path))
    except RuntimeError as e:   # more accepted rows than "Total fragments"
        assert str(e) == "Unexpected number of fragments"
        with pytest.raises(capi.RkError) as ei:
            ctx.load_csv(body, 1000, 1000, total)
        assert ei.value.code == -3 and "Unexpected number of fragments" in str(ei.value)
        return None
    ref_err = got_err = None
    try:
        ref = ref_ctx.load(rec, lx1, ly1)
    except capi.RkError as e:
        ref_err = (e.code, str(e))
    try:
        st, cs = ctx.load_csv(body if body_arg is None else body_arg(body), lx1, ly1, total)
    except capi.RkError as e:
        got_err = (e.code, str(e))
    assert got_err == ref_err
    if ref_err:
        return None
    assert (st.n_loaded, st.n_kept, st.vsize) == (ref.n_loaded, ref.n_kept, ref.vsize)
    assert cs.n_accepted == rec.shape[0] and cs.n_rows == body.count(b"\n") + 1
    assert cs.wide == bool(wide(rec))
    if not cs.wide:
        key4, strand, rest4 = compact(rec)
        assert np.array_equal(ctx.debug_fetch("key4").reshape(-1, 4), key4)
        assert np.array_equal(ctx.debug_fetch("strand", np.uint8), strand)
        assert np.array_equal(ctx.debug_fetch("rest4").reshape(-1, 4), rest4)
    else:
        with pytest.raises(capi.RkError):
            ctx.debug_fetch("key4")
    if st.n_kept:
        assert np.array_equal(ctx.debug_fetch("rank_fidx"), ref_ctx.debug_fetch("rank_fidx"))
    return rec, lx1, ly1, hdr, cs


def same_groups(ctx, ref_ctx, rec, lx1, ly1, lr, pr):
    a, b = ctx.group(lr, pr), ref_ctx.group(lr, pr)
    g = O.group(rec, lx1, ly1, lr, pr)
    assert a.n_groups == b.n_groups == g.n_groups
    for name in ("order", "gid", "repval"):
        assert np.array_equal(getattr(a, name), getattr(b, name)), name
    assert np.array_equal(a.order, g.order) and np.array_equal(a.gid, g.out_gid)
    assert np.array_equal(a.identity.view(np.uint32), b.identity.view(np.uint32))
    text = ctx.format_lines()
    assert text == ref_ctx.format_lines()
    if a.n_groups:
        sa, sb = ctx.group_statistics(), ref_ctx.group_statistics()
        assert sa.tobytes() == sb.tobytes()
    return text


# ---- the fast-path grammar restated, to count the rows the host parser must see -------------------------------------
def _plain_u64(t: bytes) -> bool:
    return 1 <= len(t) <= 18 and all(48 <= c <= 57 for c in t)


def _plain_float(t: bytes) -> bool:
    m = digits = frac = 0
    dot = False
    for c in t:
        if 48 <= c <= 57:
            digits += 1
            if digits > 18:
                return False
            m = m * 10 + c - 48
            frac += dot
        elif c == 46 and not dot:
            dot = True
        else:
            return False
    if digits == 0 or frac > 22 or m >= 1 << 53:
        return False
    d = m / 10 ** frac   # the correctly rounded quotient = IEEE division of the two exact doubles
    low = struct.unpack("<Q", struct.pack("<d", d))[0] & 0x1FFFFFFF
    return not (0x0FFFFFFF <= low <= 0x10000001)


def row_kind(row: bytes) -> str:
    """'reject', 'device' or 'host': what the device decides for one row (readFragment's token walk)"""
    parts = row.split(b",")
    toks = [parts[i] if i < len(parts) else parts[-1] for i in range(14)]
    if any(len(t) == 0 for t in toks) or toks[0] != b"Frag":
        return "reject"
    ok = all(_plain_u64(toks[i]) for i in (1, 2, 3, 4, 6, 7, 8)) and _plain_float(toks[10])
    return "device" if ok else "host"


def host_rows(body: bytes) -> int:
    return sum(row_kind(r) == "host" for r in body.split(b"\n"))


# ---- 1. the 120 fuzz CSVs --------------------------------------------------------------------------------------------
def test_fuzz_cases(ctx, ref_ctx, fuzz_cases, tmp_path):
    decided = 0
    for c in fuzz_cases:
        text = c["csv"].encode("latin1")
        got = load_both(ctx, ref_ctx, text, tmp_path)
        if got is None:
            continue
        rec, lx1, ly1, hdr, cs = got
        body, _ = split_head(text)
        assert cs.n_host_rows == host_rows(body), c["seed"]
        decided += cs.n_accepted - cs.n_host_rows
        lines = same_groups(ctx, ref_ctx, rec, lx1, ly1, c["len_ratio"], c["pos_ratio"])
        assert hdr + lines == c["ref_out"].encode("latin1"), f"fuzz seed {c['seed']}"
    assert decided > 100


# ---- 2. grammar cases built on purpose ----------------------------------------------------------------------------------
INT_TOKENS = [b"7", b"12", b"123456789", b"123456789012345678", b"1234567890123456789", b"12345678901234567890", b"+5", b"-5",
              b" 5", b"\t5", b"5 ", b"0005", b"1" * 80, b"1\x002", b"\xe95"]
FLOAT_TOKENS = [b"87.5", b".5", b"5.", b"5..0", b"1e3", b"0x1p3", b"nan", b"inf", b"-3.5", b"+2", b" 7.25",
                b"1." + b"0" * 21 + b"1", b"1." + b"0" * 22 + b"1", b"0.0000000000000000000001", b"16777217", b"33554435",
                b"16777217.0", b"1e-50", b"1e39", b"99.999999999", b"7" * 75, b"5\x00", b"5\r", b"\xb5"]
BASE = [b"Frag", b"100", b"200", b"150", b"250", b"f", b"3", b"51", b"40", b"30", b"60.5", b"60.5", b"0", b"0"]


def _row(fields):
    return b",".join(fields)


def grammar_texts():
    """(name, text) of files that each hold plain rows plus one token kind in a full row and in short rows of 1..13
    fields (the token last, so that the padding repeats it)"""
    rng = np.random.default_rng(3)
    plain = []
    for i in range(300):
        x, y, ln = int(rng.integers(0, 9000)), int(rng.integers(0, 9000)), int(rng.integers(1, 200))
        sim = f"{rng.integers(1, 100)}.{rng.integers(0, 100):02d}".encode()
        plain.append(_row([b"Frag", b"%d" % x, b"%d" % y, b"%d" % (x + ln - 1), b"%d" % (y + ln - 1), b"fr"[i % 2:i % 2 + 1],
                           b"%d" % (i % 5), b"%d" % ln, b"%d" % (4 * ln), b"0", sim, sim, b"0", b"0"]))
    cases = []
    for kind, tokens, field in (("int", INT_TOKENS, 6), ("float", FLOAT_TOKENS, 10)):
        for t in tokens:
            rows = list(plain[:50])
            full = list(BASE)
            full[field] = t
            rows.append(_row(full))
            for k in range(1, 14):
                short = BASE[:k - 1] + [t] if k > 1 else [t]
                rows.append(_row(short))
            rows += plain[50:]
            cases.append((f"{kind}:{t[:20]!r}", rows))
    # the row and line structure: CRLF, no final newline, empty lines, more than 14 fields, trailing commas, "Frag" variants
    s = list(plain)
    s[3] += b"\r"
    s[4] = s[4] + b",extra,fields,9"
    s[5] = s[5] + b","
    s[6] = _row(BASE[:5]) + b","
    s[7] = b""
    s[8] = b"frag" + s[8][4:]
    s[9] = b"Frag " + s[9][4:]
    s[10] = b"Fragx" + s[10][4:]
    s[11] = b",".join(BASE[:3]) + b"\r"
    s[12] = s[12].replace(b",f,", b",\xff,").replace(b",r,", b",\x00,")
    cases.append(("structure", s))
    cases.append(("structure, final newline", s + [b""]))
    cases.append(("structure, blank lines at the end", s + [b"", b"", b""]))
    for name, rows in cases:
        body = b"\n".join(rows)
        yield name, make_header(20000, 20000, len(rows)).encode("latin1") + body


def test_grammar_cases(ctx, ref_ctx, tmp_path):
    checked = 0
    for name, text in grammar_texts():
        got = load_both(ctx, ref_ctx, text, tmp_path)
        if got is None:
            continue
        rec, lx1, ly1, hdr, cs = got
        body, _ = split_head(text)
        assert cs.n_host_rows == host_rows(body), name
        assert cs.n_accepted - cs.n_host_rows >= 290, name   # the plain rows were decided on the device
        same_groups(ctx, ref_ctx, rec, lx1, ly1, 0.05, 0.05)
        checked += 1
    assert checked > 30


# ---- 3. wide values ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("value", [2**32, 2**40, 10**18 - 1])
def test_wide_values_take_the_record_route(ctx, ref_ctx, tmp_path, value):
    w = gen.scaled(gen.WORKLOADS["c1"], 5_000)
    rec = gen.generate(w)
    rec["score"][17] = value
    rec["xEnd"][300] = value
    path = tmp_path / "w.csv"
    O.write_input_csv(str(path), rec, w.lx, w.ly)
    got = load_both(ctx, ref_ctx, path.read_bytes(), tmp_path)
    assert got is not None and got[4].wide
    rec2, lx1, ly1, hdr, _ = got
    text = same_groups(ctx, ref_ctx, rec2, lx1, ly1, 0.05, 0.05)
    assert str(value).encode() in text


# ---- 4. one row more than "Total fragments" ----------------------------------------------------------------------------
def test_total_frags_one_short(ctx, tmp_path):
    w = gen.scaled(gen.WORKLOADS["c1"], 2_000)
    rec = gen.generate(w)
    path = tmp_path / "s.csv"
    O.write_input_csv(str(path), rec, w.lx, w.ly)
    body, total = split_head(path.read_bytes())
    assert total == w.n
    with pytest.raises(capi.RkError) as e:
        ctx.load_csv(body, w.lx + 1, w.ly + 1, total - 1)
    assert e.value.code == -3 and "Unexpected number of fragments" in str(e.value)
    with pytest.raises(capi.RkError) as e:
        ctx.group(0.05, 0.05)
    assert e.value.code == -4
    st, cs = ctx.load_csv(body, w.lx + 1, w.ly + 1, total)
    assert st.n_loaded == w.n and cs.n_host_rows == 0
    g = O.group(rec, w.lx + 1, w.ly + 1, 0.05, 0.05)
    assert np.array_equal(ctx.group(0.05, 0.05).order, g.order)


# ---- 5. full size: config 2, 10M rows ------------------------------------------------------------------------------------
def test_c2_full_size(ctx, ref_ctx, tmp_path):
    w = gen.WORKLOADS["c2"]
    rec = gen.generate(w)
    path = tmp_path / "c2.csv"
    O.write_input_csv(str(path), rec, w.lx, w.ly)
    loaded, lx1, ly1, hdr = O.load_csv(str(path))
    body, total = split_head(path.read_bytes())
    del rec
    st, cs = ctx.load_csv(body, lx1, ly1, total)
    key4, strand, rest4 = compact(loaded)
    ref = ref_ctx.load_packed(key4, strand, rest4, lx1, ly1)
    print(f"\nC2 10M: n_host_rows={cs.n_host_rows} upload {cs.ms_upload:.2f} ms, parse {cs.ms_parse:.2f} ms, "
          f"{len(body) / 1e6:.0f} MB of text")
    assert (st.n_loaded, st.n_kept, st.vsize) == (ref.n_loaded, ref.n_kept, ref.vsize) == (w.n, ref.n_kept, ref.vsize)
    for name, dt in (("key4", np.uint32), ("strand", np.uint8), ("rest4", np.uint32), ("rank_fidx", np.uint32), ("skx", np.uint32),
                     ("rx", np.uint32), ("sky", np.uint32), ("ry", np.uint32), ("hkey", np.uint32)):
        assert np.array_equal(ctx.debug_fetch(name, dt), ref_ctx.debug_fetch(name, dt)), name
    a, b = ctx.group(w.len_ratio, w.pos_ratio), ref_ctx.group(w.len_ratio, w.pos_ratio)
    assert a.n_groups == b.n_groups
    for name in ("order", "gid", "repval"):
        assert np.array_equal(getattr(a, name), getattr(b, name)), name
    assert hashlib.md5(ctx.format_lines()).hexdigest() == hashlib.md5(ref_ctx.format_lines()).hexdigest()


# ---- 6. the text as a CUDA tensor ----------------------------------------------------------------------------------------
def test_text_on_the_device(ctx, ref_ctx, tmp_path, fuzz_cases):
    import torch
    w = gen.scaled(gen.WORKLOADS["c1"], 40_000)
    rec = gen.generate(w)
    path = tmp_path / "d.csv"
    O.write_input_csv(str(path), rec, w.lx, w.ly)
    texts = [path.read_bytes()] + [c["csv"].encode("latin1") for c in fuzz_cases[::10]]
    for text in texts:
        on_host = load_both(ctx, ref_ctx, text, tmp_path)
        if on_host is None:
            continue
        rec2, lx1, ly1, _, cs_host = on_host
        host_text = same_groups(ctx, ref_ctx, rec2, lx1, ly1, 0.05, 0.05)
        for misalign in (0, 1):   # a 16-byte aligned tensor is read in place, another one copied first
            def as_cuda(body, k=misalign):
                t = torch.frombuffer(bytearray(b"x" * k + body + b"\0"), dtype=torch.uint8).cuda()
                return t[k:k + len(body)]
            got = load_both(ctx, ref_ctx, text, tmp_path, body_arg=as_cuda)
            assert got[4].n_host_rows == cs_host.n_host_rows and got[4].ms_upload == 0.0
            assert same_groups(ctx, ref_ctx, rec2, lx1, ly1, 0.05, 0.05) == host_text


# ---- 7. views --------------------------------------------------------------------------------------------------------------
def test_views_of_a_csv_load(tmp_path):
    w = gen.scaled(gen.WORKLOADS["c1"], 30_000)
    rec = gen.generate(w)
    path = tmp_path / "v.csv"
    O.write_input_csv(str(path), rec, w.lx, w.ly)
    body, total = split_head(path.read_bytes())
    with capi.Context(0) as base:
        base.load_csv(body, w.lx + 1, w.ly + 1, total)
        want = base.group(0.05, 0.05)
        want_text = base.format_lines()
        v = base.view()
        got = v.group(0.05, 0.05)
        assert np.array_equal(got.order, want.order) and np.array_equal(got.gid, want.gid)
        assert v.format_lines() == want_text
        with pytest.raises(capi.RkError) as e:
            v.load_csv(body, w.lx + 1, w.ly + 1, total)
        assert e.value.code == -4
        with pytest.raises(capi.RkError) as e:
            base.load_csv(b"garbage that is never uploaded", w.lx + 1, w.ly + 1, total)
        assert e.value.code == -4 and "1 view of this context is live" in str(e.value)
        assert np.array_equal(base.group(0.05, 0.05).order, want.order) and base.format_lines() == want_text
        v.close()


# ---- 8. the CLI on one GPU ---------------------------------------------------------------------------------------------
def _cli(inp, outp, *ratios, **env):
    return subprocess.run([CLI, str(inp), str(outp), *ratios], capture_output=True, env=dict(os.environ, **env))


def test_cli_medium_goldens_parse_on_the_device(tmp_path, medium_cases):
    for name in ("c1", "c1_loose", "dense"):
        if name not in medium_cases:
            continue
        c = medium_cases[name]
        w = gen.Workload(**c["workload"])
        inp = tmp_path / f"{name}.csv"
        O.write_input_csv(str(inp), gen.generate(w), w.lx, w.ly)
        for env in ({}, {"RK_LEGACY_WRITER": "1"}):
            outp = tmp_path / "out.csv"
            p = _cli(inp, outp, str(w.len_ratio), str(w.pos_ratio), RK_TIMING="1", **env)
            assert p.returncode == 0, p.stderr
            assert hashlib.md5(outp.read_bytes()).hexdigest() == c["ref_md5"], (name, env)
            assert b" parser=device " in p.stderr and b"device_parse_ms=" in p.stderr, p.stderr
        outp = tmp_path / "steps.csv"
        p = subprocess.run([HOSTCHECK, "steps_device", str(inp), str(outp), str(w.len_ratio), str(w.pos_ratio)], capture_output=True)
        assert p.returncode == 0, p.stderr
        assert hashlib.md5(outp.read_bytes()).hexdigest() == c["ref_md5"], name


def test_cli_fuzz_exit_status_and_bytes(tmp_path, fuzz_cases):
    ok = 0
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
        p = _cli(inp, outp, str(c["len_ratio"]), str(c["pos_ratio"]), RK_TIMING="1")
        if not want_ok:   # the reference's uncaught exception
            assert p.returncode != 0 and b"Unexpected number of fragments" in p.stderr, c["seed"]
            continue
        assert p.returncode == 0, p.stderr
        assert b" parser=device " in p.stderr
        assert outp.read_bytes() == c["ref_out"].encode("latin1"), f"fuzz seed {c['seed']}"
        q = subprocess.run([HOSTCHECK, "steps_device", str(inp), str(outp), str(c["len_ratio"]), str(c["pos_ratio"])], capture_output=True)
        assert q.returncode == 0, q.stderr
        assert outp.read_bytes() == c["ref_out"].encode("latin1"), f"steps_device, fuzz seed {c['seed']}"
        ok += 1
    assert ok > 20


def test_cli_frags_input_keeps_the_host_parser(tmp_path):
    from repkiller_b200 import frags
    w = gen.scaled(gen.WORKLOADS["c1"], 3_000)
    rec = gen.generate(w)
    binp = tmp_path / "in.frags"
    frags.write_gecko_binary(str(binp), rec, w.lx, w.ly)
    p = _cli(binp, tmp_path / "o.csv", "0.05", "0.05", RK_TIMING="1")
    assert p.returncode == 0, p.stderr
    assert b" parser=host" in p.stderr and b"parser=device" not in p.stderr
