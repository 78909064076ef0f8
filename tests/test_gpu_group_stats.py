"""K8 (k8_stats.cu: rk_group_statistics, rk_dist_group_statistics, rk_multi_group_statistics) against the definition of
rk_group_stats in include/rk_b200.h, evaluated exactly by oracle.group_statistics from K8's own inputs (the output lines'
order, gid and identity): every array byte for byte, never to a tolerance.

1  the reference itself against a fractions.Fraction brute force, on random and adversarial columns with NaN and +inf;
2  warp and CTA layout: groups of 1 .. 5000 members whose first lines sit at residues 0, 1, 31 mod 32 and 0, 1, 255 mod
   256, line counts 1 and 255 mod 256, identities 0, NaN, +inf, ident 1, ident 2^64-1, percentages and absorption groups
   (huge identities among thousands of small ones, whose left-to-right double sum is not the rounded exact sum);
3  the 32-bit top: ends past 2^32 on X and Y, in groups that mix ends below and above it;
4  a length sum past 2^53 (one group of 2^21+3 fragments of length 2^32-3; one GPU: all of them in one X bucket exceed
   the rows one rank of a partitioned load may own);
5  the same bytes from every path: rk_load_aos, rk_load_packed, rk_load_csv, a view, rk_group with RK_F_NO_SORT then
   rk_sort_groups, the same call twice, and 1, 2, 3, 5 and 8 ranks with each rank's rk_dist_group_statistics slice.

Length-0 fragments (the only NaN and +inf identities) never join a group, so those members are always singletons.
The builders' claims are checked without the gpu mark, with the oracle where the geometry is small."""
import ctypes as C
import functools
import math
import os
import tempfile
from dataclasses import replace
from fractions import Fraction

import numpy as np
import pytest

from oracle import oracle as O
from repkiller_b200 import capi, gen
from test_gpu_edges import Axis, records

gpu = pytest.mark.gpu
TOP = (1 << 32) - 1           # the largest loaded length K1 takes
BIG_IDENT = (1 << 64) - 1


# ---- 1. the reference -------------------------------------------------------------------------------------------------
def left_to_right(vals):
    """binary64 sum in list order, one rounding per add (the built-in sum() compensates)"""
    s = 0.0
    for v in vals:
        s += v
    return s


def brute_force(rec, order, gid, identity):
    """rk_group_stats by its definition with Fractions and Python ints, one group at a time"""
    out = np.zeros(0 if len(gid) == 0 else int(gid[-1] - gid[0]) + 1, capi.GROUP_STATS_DTYPE)
    j = 0
    for k in range(out.shape[0]):
        lines = []
        while j < len(gid) and gid[j] == gid[0] + k:
            lines.append(j)
            j += 1
        r = [rec[int(order[i])] for i in lines]
        xs, ys, ln = ([int(q[f]) for q in r] for f in ("xStart", "yStart", "length"))
        vals = [float(identity[i]) for i in lines]
        span = max(a + b for a, b in zip(xs, ln)) - min(xs)
        if any(math.isnan(v) for v in vals):
            mean = np.uint64(O.NAN_BITS).view(np.float64)
        elif any(v == math.inf for v in vals):
            mean = math.inf
        else:
            mean = float(sum(Fraction(v) for v in vals)) / len(vals)
        out[k] = (len(lines), min(xs), min(ys), lines[0], max(a + b for a, b in zip(xs, ln)), max(a + b for a, b in zip(ys, ln)),
                  mean, float(sum(ln)) / float(span) if span else 0.0)
    return out


def random_columns(rng, m, kinds):
    """m output lines over random group sizes; records with 32-bit coordinates and lengths; identities of the kinds"""
    sizes = []
    while sum(sizes) < m:
        sizes.append(int(rng.choice([1, 1, 2, 3, 5, 31, 33, 70])))
    gid = np.repeat(np.arange(len(sizes)), sizes)[:m]
    rec = np.zeros(m, capi_frag_dtype())
    rec["xStart"] = rng.integers(0, 1 << 32, m, dtype=np.uint64)
    rec["yStart"] = rng.integers(0, 1 << 32, m, dtype=np.uint64)
    rec["length"] = rng.integers(0, 1 << 32, m, dtype=np.uint64)
    order = rng.permutation(m).astype(np.uint32)
    pick = rng.choice(len(kinds), m)
    ident = np.array([kinds[p](rng) for p in pick], np.float32)
    return rec, order, gid, ident


def capi_frag_dtype():
    from repkiller_b200.frags import FRAG_DTYPE
    return FRAG_DTYPE


KINDS = {
    "percent": lambda r: np.float32(r.integers(0, 10001) / 100),
    "zero": lambda r: np.float32(0),
    "small": lambda r: np.float32(100) / np.float32(r.integers(1 << 31, 1 << 32)),   # ident 1 over a long fragment
    "large": lambda r: np.float32(100) * np.float32(r.integers(1 << 60, BIG_IDENT, dtype=np.uint64)),
    "nan": lambda r: np.uint32(0xFFC00000).view(np.float32),
    "inf": lambda r: np.float32(np.inf),
}


@pytest.mark.parametrize("kinds", [("percent",), ("percent", "small", "large"), ("small", "large", "zero"),
                                   ("percent", "small", "large", "zero", "nan"), ("percent", "large", "inf"),
                                   ("percent", "small", "large", "nan", "inf")])
def test_reference_matches_fraction_brute_force(kinds):
    rng = np.random.default_rng(sum(map(ord, "".join(kinds))))
    for m in (1, 2, 37, 1500):
        rec, order, gid, ident = random_columns(rng, m, [KINDS[k] for k in kinds])
        got = O.group_statistics(rec, order, gid, ident)
        assert got.tobytes() == brute_force(rec, order, gid, ident).tobytes(), (kinds, m)


def test_reference_adversarial_sums():
    """absorption (1e21 then thousands of 100s), cancellation-free near-ties and a half-way case, against Fractions"""
    rec = np.zeros(8000, capi_frag_dtype())
    rec["length"] = 1
    big = float(np.float32(100) * np.float32(BIG_IDENT))
    cases = [[big] + [100.0] * 3000, [100.0] * 3000 + [big], [big, 100.0, big] + [100.0] * 1500,
             [2.0 ** 53, 1.0, 1.0], [2.0 ** 53, 1.0], [1.0, 2.0 ** -49, 2.0 ** 60, 2.0 ** -49],
             [float(np.float32(100) / np.float32(TOP))] * 7 + [70.0] * 5]
    for vals in cases:
        m = len(vals)
        ident = np.array(vals, np.float32)
        order, gid = np.arange(m, dtype=np.uint32), np.zeros(m, np.uint32)
        got = O.group_statistics(rec, order, gid, ident)
        assert got.tobytes() == brute_force(rec, order, gid, ident).tobytes(), vals[:4]
    ident = np.array([big] + [100.0] * 3000, np.float32)
    assert left_to_right(ident.astype(np.float64).tolist()) != math.fsum(ident.astype(np.float64).tolist())


# ---- 2. warp and CTA layout ---------------------------------------------------------------------------------------------
SIZES = [1, 2, 31, 32, 33, 63, 64, 65, 255, 256, 257, 1023, 1024, 1025, 5000]
RESIDUES = [(0, 32), (1, 32), (31, 32), (0, 256), (1, 256), (255, 256)]
GROUP_KINDS = ["percent", "mixed", "large", "absorb", "small", "zero"]
SINGLE_KINDS = ["percent", "nan", "inf", "zero", "small", "large"]


def _ident_of(kind, n, ln, rng):
    """ident column of n members of length ln"""
    if kind == "percent":
        return rng.integers(0, ln + 1, n, dtype=np.uint64)
    if kind == "zero":
        return np.zeros(n, np.uint64)
    if kind == "small":
        return np.ones(n, np.uint64)
    if kind == "large":
        return np.full(n, BIG_IDENT, np.uint64) - rng.integers(0, 1 << 20, n, dtype=np.uint64)
    if kind == "mixed":
        return rng.choice(np.array([0, 1, ln // 3, ln, BIG_IDENT, 1 << 40], np.uint64), n)
    if kind == "absorb":     # identity ~3 * 2^61 (ulp 1024 and more) every n/5 members, 100 elsewhere: each 100 added
        a = np.ones(n, np.uint64)  # after it is lost to rounding, thousands of them are not
        a[::max(n // 5, 1)] = 3 * (1 << 61) // 100
        return a
    raise ValueError(kind)


@functools.lru_cache(maxsize=None)
def build_layout(tail):
    """groups of SIZES members (same xStart and length: all join the first) whose first output line lies at each of
    RESIDUES, shifted there by leading singletons (length 0 for NaN and +inf); the line count ends at `tail` mod 256.
    Everything is laid out left to right on X, so the output order is the file order.  Returns (case, plan) with plan
    = [(first line, size, kind)] of the groups."""
    rng = np.random.default_rng(tail)
    X, Y = Axis(), Axis()
    rows, idents, plan = [], [], []
    line, nsingle = 0, 0

    def single():
        nonlocal line, nsingle
        kind = SINGLE_KINDS[nsingle % len(SINGLE_KINDS)]
        nsingle += 1
        ln = 0 if kind in ("nan", "inf") else 100
        rows.append((X.take(2000), Y.take(2000), ln, b"f" if nsingle % 3 else b"r"))
        idents.append({"nan": 0, "inf": 7, "zero": 0, "small": 1, "large": BIG_IDENT}.get(kind, int(rng.integers(0, 101))))
        line += 1

    g = 0
    for r, mod in RESIDUES:
        for n in SIZES:
            while line % mod != r:
                single()
            kind = GROUP_KINDS[g % len(GROUP_KINDS)] if n > 2 else ("mixed" if g % 2 else "percent")
            if kind == "absorb" and n < 1000:
                kind = "mixed"
            g += 1
            ln = 1 if kind in ("absorb", "large") else 1000
            x, y = X.take(3 * ln + 2000), Y.take(n + 3 * ln + 2000)
            for i in range(n):
                rows.append((x, y + i, ln, b"f"))
            idents.extend(_ident_of(kind, n, ln, rng).tolist())
            plan.append((line, n, kind))
            line += n
    while line % 256 != tail:
        single()
    rec = records(rows)
    rec["ident"] = np.array(idents, np.uint64)
    lx1 = int(rec["xStart"].max()) + 5000
    ly1 = int(rec["yStart"].max()) + 5000
    return (rec, lx1, ly1, 0.05, 0.05), plan


@pytest.mark.parametrize("tail", [1, 255])
def test_layout_builder_self_check(tail):
    (rec, lx1, ly1, lr, pr), plan = build_layout(tail)
    g = O.group(rec, lx1, ly1, lr, pr)
    assert g.n_kept == rec.shape[0] and g.n_kept % 256 == tail
    starts = np.r_[0, np.flatnonzero(np.diff(g.out_gid)) + 1]
    sizes = np.diff(np.r_[starts, g.n_kept])
    at = dict(zip(starts.tolist(), sizes.tolist()))
    for first, n, _ in plan:
        assert at.get(first) == n, (first, n, at.get(first))
    for r, mod in RESIDUES:
        assert {n for first, n, _ in plan if first % mod == r} >= set(SIZES)
    bits = g.identity.view(np.uint32)
    kinds = {"nan": bits == 0xFFC00000, "inf": bits == 0x7F800000, "zero": bits == 0}
    for k, sel in kinds.items():
        lines = np.flatnonzero(sel)
        assert {int(v) % 32 for v in lines} & {0, 31}, k          # on both sides of warp boundaries
    assert np.any(g.identity > 1e21) and np.any((g.identity > 0) & (g.identity < 0.2))
    # every absorption group: the left-to-right double sum in line order is not the rounded exact sum
    absorb = [(first, n) for first, n, kind in plan if kind == "absorb"]
    assert absorb
    vals = g.identity.astype(np.float64).tolist()
    for first, n in absorb:
        assert left_to_right(vals[first:first + n]) != math.fsum(vals[first:first + n]), first


# ---- 3. the 32-bit top ---------------------------------------------------------------------------------------------------
def _straddle(cx, cy, lengths, rows, idents, ident_of):
    for ln in lengths:
        rows.append((cx - ln // 2, cy - ln // 2, ln, b"f"))
        idents.append(ident_of(ln))


@functools.lru_cache(maxsize=None)
def build_top32():
    """loaded lengths 2^32-1: the two-record reproducer (ends 2^32+15); groups around one centre whose X and Y ends
    straddle 2^32 (lengths 2,000 .. 12,000 rising, falling and shuffled, 40 .. 70 members: over warp boundaries; length
    ratio 10 keeps each in one group, position ratio 0.05 keeps the groups 2,000 apart); a group of ident 1 .. 2^64-1 over lengths 2^32-3 (the smallest identity among ordinary
    ones).  Returns (case, groups) with groups = the file indices meant to form one group each."""
    rng = np.random.default_rng(32)
    rows, idents, groups = [], [], []

    def add(fn, *a):
        i0 = len(rows)
        fn(*a)
        groups.append(list(range(i0, len(rows))))

    def repro():
        rows.extend([(4_294_967_279, 100, 32, b"f")] * 2)
        idents.extend([25, 26])
    add(repro)
    pct = lambda ln: int(rng.integers(0, ln + 1))                                  # noqa: E731
    top = TOP - 3000
    add(_straddle, top, top, list(range(2000, 12000, 250)), rows, idents, pct)                        # 40 rising
    add(_straddle, top - 2000, top - 7_000_000, list(range(12000, 2000, -150))[:70], rows, idents, pct)   # X straddles
    lens = rng.permutation(np.arange(2000, 12000, 200)).tolist()
    add(_straddle, top - 6_000_000, top - 2000, lens, rows, idents, lambda ln: BIG_IDENT if ln % 3 else pct(ln))  # Y straddles

    def smallest():
        for i in range(40):
            rows.append((3, 5_000_000, TOP - 3, b"f"))
            idents.append([1, 3_000_000_000, BIG_IDENT, 0, 1][i % 5])
    add(smallest)
    rec = records(rows)
    rec["ident"] = np.array(idents, np.uint64)
    return (rec, TOP, TOP, 10.0, 0.05), groups


def test_top32_builder_self_check():
    (rec, lx1, ly1, _, _), groups = build_top32()
    xe = rec["xStart"] + rec["length"]
    ye = rec["yStart"] + rec["length"]
    cx = rec["xStart"] + rec["length"] // np.uint64(2)
    cy = rec["yStart"] + rec["length"] // np.uint64(2)
    assert int(cx.max()) < 1 << 32 and int(cy.max()) < 1 << 32 and int(rec["length"].max()) < 1 << 32
    assert int(xe[groups[0]][0]) == (1 << 32) + 15 and (int(xe[groups[0]][0]) & 0xFFFFFFFF) < 4_294_967_279
    for gi, axis in ((1, "xy"), (2, "x"), (3, "y")):
        sel = groups[gi]
        assert len(sel) > 32
        for e, name in ((xe, "x"), (ye, "y")):
            if name in axis:
                assert (e[sel] > np.uint64(TOP)).any() and (e[sel] <= np.uint64(TOP)).any(), (gi, name)
                assert len({int(v) // 100 for v in (cx if name == "x" else cy)[sel]}) == 1   # one centre bucket
    assert (rec["ident"][groups[4]] == np.uint64(1)).any() and (rec["length"][groups[4]] == np.uint64(TOP - 3)).all()


# ---- 4. a length sum past 2^53 ---------------------------------------------------------------------------------------------
N_LONG = (1 << 21) + 3


@functools.lru_cache(maxsize=None)
def build_len_sum():
    """one group of 2^21+3 identical fragments of length 2^32-3 (ident varies): the sum of the lengths is 2^53 + 3 * 2^32
    - 3 * 2^21 - 9, an odd 54-bit number"""
    rng = np.random.default_rng(53)
    rec = records([(1000, 2000, TOP - 2, b"f")])
    rec = np.repeat(rec, N_LONG)
    rec["ident"] = rng.integers(0, 1 << 32, N_LONG, dtype=np.uint64)
    return rec, TOP, TOP, 0.05, 0.05


def test_len_sum_builder_self_check():
    total = N_LONG * (TOP - 2)
    assert total > 1 << 53 and total % 2 == 1 and total.bit_length() == 54
    assert float(total) != total


# ---- 5. every path ---------------------------------------------------------------------------------------------------------
def fits32(rec):
    return all(int(rec[f].max()) < 1 << 32 for f in ("xStart", "yStart", "length", "ident", "xEnd", "yEnd", "score"))


def csv_case(rec, lx1, ly1):
    """(body, records) of the rendered GECKO CSV: the records as the reference's parser reads them back"""
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "in.csv")
        O.write_input_csv(p, rec, lx1 - 1, ly1 - 1)
        text = open(p, "rb").read()
        crec = O.load_csv(p)[0]
    pos = 0
    for _ in range(16):
        pos = text.index(b"\n", pos) + 1
    return text[pos:], crec


def assert_bytes(name, got, want):
    if got.tobytes() == want.tobytes():
        return
    assert got.shape == want.shape, f"{name}: {got.shape} vs {want.shape}"
    bad = np.flatnonzero([a.tobytes() != b.tobytes() for a, b in zip(got, want)])
    k = int(bad[0])
    raise AssertionError(f"{name}: {bad.size} of {got.shape[0]} groups differ, first group {k}: got {got[k]} want {want[k]}")


def same_groups(name, res, ref):
    for f in ("order", "gid"):
        assert np.array_equal(getattr(res, f), getattr(ref, f)), f"{name}: {f}"
    assert np.array_equal(res.identity.view(np.uint32), ref.identity.view(np.uint32)), f"{name}: identity"


def check_paths(ctx, case, worlds=(1, 2, 3, 5, 8), csv=True, groups=None):
    """statistics of every path equal the reference over the one-GPU grouping, byte for byte"""
    rec, lx1, ly1, lr, pr = case
    ctx.load(rec, lx1, ly1)
    ref = ctx.group(lr, pr)
    want = O.group_statistics(rec, ref.order, ref.gid, ref.identity)
    assert want.shape[0] == ref.n_groups and int(want["count"].sum()) == ref.n_kept
    if groups:   # the groups the builder meant: one gid each
        line_of = np.empty(rec.shape[0], np.int64)
        line_of[ref.order] = np.arange(ref.n_kept)
        for sel in groups:
            assert np.unique(ref.gid[line_of[sel]]).size == 1, sel[:3]
    assert_bytes("rk_load_aos", ctx.group_statistics(), want)
    assert_bytes("the same call twice", ctx.group_statistics(), want)
    with ctx.view() as v:
        same_groups("view", v.group(lr, pr), ref)
        assert_bytes("view", v.group_statistics(), want)
    ctx.group(lr, pr, sort=False)
    assert_bytes("rk_group with RK_F_NO_SORT", ctx.group_statistics(), want)
    same_groups("rk_sort_groups", ctx.sort_groups(), ref)
    assert_bytes("rk_sort_groups", ctx.group_statistics(), want)
    if fits32(rec):
        ctx.load_packed(*capi.pack_records(rec), lx1, ly1)
        same_groups("rk_load_packed", ctx.group(lr, pr), ref)
        assert_bytes("rk_load_packed", ctx.group_statistics(), want)
    if csv:   # the text's records, parsed on the device, against rk_load_aos of the same records
        body, crec = csv_case(rec, lx1, ly1)
        ctx.load_csv(body, lx1, ly1, crec.shape[0])
        cres = ctx.group(lr, pr)
        cwant = O.group_statistics(crec, cres.order, cres.gid, cres.identity)
        assert_bytes("rk_load_csv", ctx.group_statistics(), cwant)
        ctx.load(crec, lx1, ly1)
        same_groups("rk_load_aos of the CSV's records", ctx.group(lr, pr), cres)
        assert_bytes("rk_load_aos of the CSV's records", ctx.group_statistics(), cwant)
    for world in worlds:
        with capi.Multi([0] * world) as m:
            m.load(rec, lx1, ly1)
            same_groups(f"{world} ranks", m.group(lr, pr, line_records=True), ref)
            got = m.group_statistics()
            assert_bytes(f"{world} ranks", got, want)
            L = m._L
            for r in range(world):
                h = L.rk_multi_ctx(m._h, r)
                fg, ng, hp = C.c_uint64(), C.c_uint64(), C.c_void_p()
                assert L.rk_dist_group_statistics(h, capi.F_HOST_RESULT, C.byref(hp), None, C.byref(fg), C.byref(ng)) == 0
                part = capi._stats_array(hp.value, ng.value)
                assert_bytes(f"{world} ranks, rank {r}", part, want[fg.value:fg.value + ng.value])
    return ref, want


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


@gpu
@pytest.mark.parametrize("tail", [1, 255])
def test_layout_and_identity_kinds(ctx, tail):
    case, plan = build_layout(tail)
    ref, want = check_paths(ctx, case)
    first = {int(s): k for k, s in enumerate(want["first_line"])}
    for line, n, kind in plan:
        assert want["count"][first[line]] == n, (line, n, kind)
    assert (want["mean_identity"].view(np.uint64) == np.uint64(O.NAN_BITS)).any()
    assert np.isposinf(want["mean_identity"]).any()


@gpu
def test_top32_ends_and_smallest_identity(ctx):
    case, groups = build_top32()
    ref, want = check_paths(ctx, case, worlds=(1, 3), groups=groups)
    assert (want["x_hi"] > TOP).any() and (want["y_hi"] > TOP).any()
    k = int(ref.gid[np.flatnonzero(ref.order == groups[0][0])[0]])
    assert want["x_hi"][k] == (1 << 32) + 15 and want["x_lo"][k] == 4_294_967_279


@gpu
def test_length_sum_past_2pow53(ctx):
    case = build_len_sum()
    ref, want = check_paths(ctx, case, worlds=(), csv=False)   # one X bucket: beyond a rank's capacity when partitioned
    assert want.shape[0] == 1 and want["count"][0] == N_LONG
    assert want["multiplicity"][0] == float(N_LONG * (TOP - 2)) / float(TOP - 2)


WORKLOADS = {"c1": gen.WORKLOADS["c1"],
             "dense": replace(gen.WORKLOADS["c1"], n=60_000, lx=400_000, ly=300_000, families=40, p_rep=0.6, seed=31),
             "c3": gen.scaled(gen.WORKLOADS["c3"], 300_000)}


@gpu
@pytest.mark.parametrize("wl", sorted(WORKLOADS))
def test_workloads_every_path(ctx, wl):
    w = WORKLOADS[wl]
    rec = gen.generate(w)
    ref, want = check_paths(ctx, (rec, w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio))
    assert want["count"].max() > 16


@gpu
def test_c2_full_size(ctx):
    """config 2 at its full 10M fragments: one GPU, a view, packed ingest, twice, and three ranks"""
    w = gen.WORKLOADS["c2"]
    rec = gen.generate(w)
    check_paths(ctx, (rec, w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio), worlds=(3,), csv=False)
