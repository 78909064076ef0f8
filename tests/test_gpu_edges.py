"""Inputs built on purpose at the exact decisions of the grouping kernels, each checked bit for bit against the oracle on one
GPU (every intermediate, every output array, the device text) and on three ranks (cuts, halo and forest see the same edges).

A  candidate test of deviation() and the tie rule (k3_match.cu:139-156 thresholds, :186-192 band, :196-217 best_of,
   :225-234 is_candidate, :426-509 k_match_long prune / phases A and B) — tier 1, tier 2 and the Y pass;
B  the "next bucket" probe (rk_common.cuh:65-74) around max_index on both axes and strand classes;
C  tier-1 windows and tiles (k3_match.cu:245-293) and run_start over the link bitmap (rk_common.cuh:79-90);
D  the size classes of sort_groups through rk_group's gathered layout (k5_order.cu, OrderArgs::srank);
E  32-bit geometry: 4-pass rank and X/Y sorts with digit counts from K1/k_keys (capi.cu:352-421), the 2^32 refusal
   (k1_decode.cu:83-87), 4-pass gid sorts (capi.cu:494-501);
F  the single-call occupation lists rk_sol_* (sol.cu) against the restatement's lists (rko_sol_*).

The builders assert what they built using Python floats (binary64, round to nearest, no contraction: the kernels'
arithmetic) and the oracle only; those self-checks are the tests without the gpu mark."""
import functools
import math
import os
import tempfile

import numpy as np
import pytest

from oracle import oracle as O
from repkiller_b200 import capi, gen
from repkiller_b200.frags import FRAG_DTYPE

gpu = pytest.mark.gpu
BAND = 2.0 ** -40
U32MAX = 0xFFFFFFFF


# ---- shared helpers ------------------------------------------------------------------------------------------------------
def records(rows):
    """rows of (xStart, yStart, length, strand) -> FRAG_DTYPE records with consistent xEnd/yEnd/score/similarity"""
    n = len(rows)
    rec = np.zeros(n, FRAG_DTYPE)
    if not n:
        return rec
    a = np.array([(r[0], r[1], r[2]) for r in rows], dtype=np.uint64)
    ln = a[:, 2]
    ident = (ln * np.uint64(4)) // np.uint64(5)
    rec["xStart"], rec["yStart"], rec["length"] = a[:, 0], a[:, 1], ln
    rec["xEnd"] = a[:, 0] + np.maximum(ln, np.uint64(1)) - np.uint64(1)
    rec["yEnd"] = a[:, 1] + np.maximum(ln, np.uint64(1)) - np.uint64(1)
    rec["diag"] = a[:, 0].astype(np.int64) - a[:, 1].astype(np.int64)
    rec["score"] = np.uint64(4) * ident
    sim = (100.0 * ident.astype(np.float64) / np.maximum(ln, np.uint64(1)).astype(np.float64)).astype(np.float32)
    rec["similarity"] = sim
    rec["ident"] = sim.astype(np.uint64)
    rec["seqX"], rec["seqY"] = 0, 1
    rec["strand"] = [r[3] for r in rows]
    return rec


def deviation(ec, el, c, ln, lr, pr):
    """SequenceOcupationList.cpp:20-31 in binary64 (Python floats round to nearest, no contraction)"""
    q1 = abs(ln - el) / (ln * lr)
    sl = -abs(q1) + 1.0
    if sl < 0:
        return 0.0
    q2 = abs(c - ec) / (ln * pr)
    sp = -abs(q2) + 1.0
    if sp < 0:
        return 0.0
    return sl * 0.4 + sp * 0.6


def proc_rank(rec):
    """processing rank of every record: xStart/10 bucket, file order inside (FragmentsDatabase.cpp:96-97)"""
    order = np.argsort(rec["xStart"] // np.uint64(10), kind="stable")
    rank = np.empty(rec.shape[0], np.int64)
    rank[order] = np.arange(rec.shape[0])
    return rank


def parents_by_file(rec, g):
    """file index -> file index of the owner the oracle found (X or Y), -1 for none"""
    parent = np.full(rec.shape[0], -1, np.int64)
    p = g.parent.astype(np.int64)
    has = g.parent != O.NONE
    parent[g.rank_fidx] = np.where(has, g.rank_fidx[np.where(has, p, 0)].astype(np.int64), -1)
    return parent


def x_segments(rec, lx1):
    """per record: (segment id, position in the segment, segment size) of the X pass — segments are runs of linked
    centre buckets per strand class (rk_common.cuh:65-90), members in processing order"""
    mx = lx1 // 100
    nbx = mx + 2
    c = (rec["xStart"] + rec["length"] // np.uint64(2)).astype(np.int64)
    key = (rec["strand"] != b"f").astype(np.int64) * nbx + c // 100
    r = c % 100
    linked = set(key[(r <= 1) & (c >= 100)].tolist()) | set((key[((r == 99) & (c < mx)) | ((r == 98) & (c < mx - 1))] + 1).tolist())
    start = {}
    for k in set(key.tolist()):
        j = k
        while j in linked:           # link bit j: bucket j is processed together with j-1
            j -= 1
        start[k] = j
    seg = np.array([start[k] for k in key.tolist()], np.int64)
    order = np.lexsort((proc_rank(rec), seg))
    pos = np.empty(rec.shape[0], np.int64)
    sseg = seg[order]
    first = np.r_[0, np.nonzero(sseg[1:] != sseg[:-1])[0] + 1]
    size = np.diff(np.r_[first, rec.shape[0]])
    idx = np.repeat(np.arange(first.size), size)
    pos[order] = np.arange(rec.shape[0]) - first[idx]
    sz = np.empty(rec.shape[0], np.int64)
    sz[order] = size[idx]
    return seg, pos, sz


def first_diff(name, got, want):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, f"{name}: shape {got.shape} vs {want.shape}"
    d = np.nonzero(got != want)[0]
    assert d.size == 0, f"{name}: {d.size} diffs, first at {d[:4]}: got {got[d[:4]]} want {want[d[:4]]}"


def check_one_gpu(ctx, rec, lx1, ly1, lr, pr, g=None, text=True):
    st = ctx.load(rec, lx1, ly1)
    g = g if g is not None else O.group(rec, lx1, ly1, lr, pr)
    assert st.n_kept == g.n_kept and st.vsize == g.vsize
    if g.n_kept:
        first_diff("rank_fidx", ctx.debug_fetch("rank_fidx"), g.rank_fidx)
    res = ctx.group(lr, pr)
    if g.n_kept:
        first_diff("parent", ctx.debug_fetch("parent"), g.parent)
        first_diff("gid_rank", ctx.debug_fetch("gid_rank"), g.gid)
        first_diff("hkey", ctx.debug_fetch("hkey"), g.h.astype(np.uint32))
    assert res.n_groups == g.n_groups
    first_diff("order", res.order, g.order)
    first_diff("gid", res.gid, g.out_gid)
    first_diff("repval", res.repval, g.repval)
    first_diff("identity", res.identity.view(np.uint32), g.identity.view(np.uint32))
    if text:
        with tempfile.TemporaryDirectory() as d:
            p = os.path.join(d, "o.csv")
            O.write_output(p, b"", rec, g)
            assert open(p, "rb").read() == ctx.format_lines(), "device text"
    return g


def check_three_ranks(m3, rec, lx1, ly1, lr, pr, g):
    st = m3.load(rec, lx1, ly1)
    assert st.n_kept == g.n_kept
    res = m3.group(lr, pr)
    assert res.n_kept == g.n_kept and res.n_groups == g.n_groups
    first_diff("3 ranks order", res.order, g.order)
    first_diff("3 ranks gid", res.gid, g.out_gid)
    first_diff("3 ranks repval", res.repval, g.repval)
    first_diff("3 ranks identity", res.identity.view(np.uint32), g.identity.view(np.uint32))


def check_both(ctx, m3, case):
    rec, lx1, ly1, lr, pr = case[:5]
    g = check_one_gpu(ctx, rec, lx1, ly1, lr, pr)
    check_three_ranks(m3, rec, lx1, ly1, lr, pr, g)


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def m3():
    m = capi.Multi([0, 0, 0])
    yield m
    m.close()


# ---- A. thresholds and ties ----------------------------------------------------------------------------------------------
RATIOS = [(0.1, 0.1), (0.3, 0.7), (0.7, 0.3), (1 / 3, 2 / 3), (0.05, 0.05), (1e-3, 1e-3), (1e4, 1e4), (2048.0, 0.5)]
LENGTHS = list(range(1, 65)) + [100, 1000, 1 << 20]
MAX_DL = 1 << 18             # larger length differences are left out: they only lengthen the axes


def thresh(ln, ratio):
    """Thresh of k3_match.cu:143-149: (t, pass, rej)"""
    t = ln * ratio
    return t, min(math.ceil(min(t * (1 - BAND), 4294967295.0)), U32MAX), min(math.floor(min(t * (1 + BAND), 4294967295.0)), U32MAX)


def diffs(t):
    f, c = math.floor(t), math.ceil(t)
    return sorted({d for d in (0, f - 1, f, c, c + 1) if d >= 0})


class Axis:
    """allocates isolated windows (>= 300 bp apart, starting on a bucket boundary) along one axis"""

    def __init__(self, start=1000):
        self.pos = start

    def take(self, span):
        base = -(-self.pos // 100) * 100
        self.pos = base + span + 300
        return base


def place(spec, lq, bx, by, rows, strand=b"f", x_far=None):
    """One query and its entries.  spec: [(center offset from the query, entry length)], oldest first; the query centre
    sits at residue `res` of its bucket.  Entries are written before the query (file order) and every xStart/10 must be
    non-decreasing in that order, so the processing order is the intended one (asserted by the self-checks).
    x_far: (list of X bases) puts every fragment alone on X (Y pass), else X mirrors Y."""
    ents, res = spec
    left = max([lq // 2] + [el // 2 - off for off, el in ents]) + 1
    cq = -(-(left - res) // 100) * 100 + res
    out = []
    for i, (off, el) in enumerate(ents + [(0, lq)]):
        c = cq + off
        xy = c - el // 2
        out.append((xy, el))
    idx0 = len(rows)
    for i, (xy, el) in enumerate(out):
        if x_far is None:
            rows.append((bx + xy, by + xy, el, strand))
        else:
            rows.append((x_far[i], by + xy, el, strand))
    return idx0, by + cq, bx + cq


def cases_for(lr, pr):
    """(spec, lq, kind) of the threshold table and the tie cases for one ratio pair"""
    out = []
    for lq in LENGTHS:
        tl, _, _ = thresh(lq, lr)
        tp, _, _ = thresh(lq, pr)
        for dl in diffs(tl):
            for dc in diffs(tp):
                if dl > MAX_DL or dc > 99:
                    continue   # dc > 99 from a residue-99 centre is another bucket: never a candidate
                out.append((([(-dc, lq + dl)], 99), lq, "grid"))
    # ties and dominance, at a query length where both t are >= 8
    lq = max(40, math.ceil(8 / min(lr, pr)))
    if lq <= 100_000:
        # own bucket vs neighbour (the query at residue 1 probes the previous bucket), neighbour newer: own wins
        out.append((([(2, lq + 6), (-2, lq - 6)], 1), lq, "tie_own_vs_neighbour"))
        for kind in ("tie_mirrored", "tie_equal_score", "dominance"):
            spec = find_pair(lq, lr, pr, kind)
            if spec:
                out.append(((spec, 50), lq, kind))
    # the same tie where length * ratio >= 2^30 (k_match_long without its prune, clamped thresholds for 1e4)
    lq = 1 << 20
    if lq * max(lr, pr) >= 1 << 30:
        out.append((([(2, lq + 6), (-2, lq - 6)], 1), lq, "tie_own_vs_neighbour_big_t"))
    return out


def find_pair(lq, lr, pr, kind):
    """two entries (older, newer) in the query's bucket, both inserted (the newer is no candidate of the older), processed
    in that order before the query (centre at residue 50, so xStart/10 follows xStart):
      tie_mirrored     centres q-d and q+d, the same score;
      tie_equal_score  distinct (dl, dc), the same rounded score (searched);
      dominance        the older is strictly better although its dl is larger (a prune on either difference alone is wrong)"""
    cq = 100_050
    lim = 12
    for a in range(lim + 1):
        for b in range(lim + 1):
            for a2 in range(lim + 1):
                for b2 in range(lim + 1):
                    if kind == "tie_mirrored" and (b2 != b or b == 0):
                        continue
                    if kind == "tie_equal_score" and (a, b) == (a2, b2):
                        continue
                    if kind == "dominance" and not (a > a2 and b < b2):
                        continue
                    for s1, t1, s2, t2 in ((1, -1, -1, 1), (1, 1, -1, -1), (-1, 1, 1, -1), (1, -1, 1, 1), (-1, -1, 1, 1),
                                           (1, 1, 1, -1), (-1, 1, -1, -1), (-1, -1, -1, 1)):
                        if kind == "tie_mirrored" and t1 == t2:
                            continue
                        e1, e2 = (t1 * b, lq + s1 * a), (t2 * b2, lq + s2 * a2)
                        if e1[1] < 1 or e2[1] < 1:
                            continue
                        sc1 = deviation(cq + e1[0], e1[1], cq, lq, lr, pr)
                        sc2 = deviation(cq + e2[0], e2[1], cq, lq, lr, pr)
                        if sc2 <= 0 or (sc1 != sc2 if kind != "dominance" else sc1 <= sc2):
                            continue
                        if deviation(cq + e1[0], e1[1], cq + e2[0], e2[1], lr, pr) > 0:
                            continue
                        x1, x2, xq = (cq + e1[0] - e1[1] // 2) // 10, (cq + e2[0] - e2[1] // 2) // 10, (cq - lq // 2) // 10
                        if x1 <= x2 <= xq:
                            return [e1, e2]
    return None


def pads(xq_or_xe, yq_or_ye, bq):
    """33 members of the same super-bucket that no query of the case can see: centres at residues 0/1 of bucket bq+1 (they
    link it to bq), xStart equal to the given one (so their processing rank is fixed by file order).  The case's queries
    sit at or above max_index, so a residue-98/99 query does not probe bq+1 either."""
    out = []
    for k in range(33):
        cp = 100 * (bq + 1) + k % 2
        out.append((xq_or_xe, yq_or_ye, 2 * (cp - xq_or_xe), b"f"))
    return out


WAYS = ("tier1", "tier2_phaseA", "tier2_phaseB", "ypass")


def _layout_thresholds(lr, pr, start):
    rows, meta = [], []
    X = Y = Axis(start)          # one allocator: every window is isolated on both axes
    for spec, lq, kind in cases_for(lr, pr):
        span = max([lq] + [el for _, el in spec[0]]) + 400
        ne = len(spec[0])
        # tier 1
        bx = X.take(span)
        i0, _, _ = place(spec, lq, bx, bx, rows)
        meta.append((kind, "tier1", list(range(i0, i0 + ne)), i0 + ne))
        # tier 2, phase A: 33 pads between the entries and the query (entries in an earlier chunk of 32)
        b = X.take(span + 300)
        i0, _, cq = place(spec, lq, b, b, rows)
        q = rows.pop()
        rows.extend(pads(q[0], q[1], cq // 100))
        rows.append(q)
        meta.append((kind, "tier2_phaseA", list(range(i0, i0 + ne)), len(rows) - 1))
        # tier 2, phase B: 33 pads before the entries (entries and query in one chunk)
        b = X.take(span + 300)
        i0, _, cq = place(spec, lq, b, b, rows)
        rows[i0:i0] = pads(rows[i0][0], rows[i0][1], cq // 100)
        meta.append((kind, "tier2_phaseB", list(range(i0 + 33, i0 + 33 + ne)), len(rows) - 1))
        # Y pass: G then F identical on X (F X-matched, an entry of the query's Y segment), entries and query alone on X
        xs = [X.take(el + 100) for el in [el for _, el in spec[0]] + [lq]]
        gx = X.take(span)
        by = Y.take(span)
        rej = thresh(lq, lr)[2]
        lf = lq + rej + 5 if rej < 1 << 20 else lq + 5     # inert to the query where the axis allows it
        i0, ycq, _ = place(spec, lq, 0, by, rows, x_far=xs)
        q = rows.pop()
        gy = Y.take(lf + 400)
        rows.append((gx, gy, lf, b"f"))
        rows.append((gx, max(0, (ycq // 100) * 100 + 10 - lf // 2), lf, b"f"))
        rows.append(q)
        meta.append((kind, "ypass", list(range(i0, i0 + ne)), len(rows) - 1))
    rec = records(rows)
    lx1 = int(rec["xStart"].max() + rec["length"].max()) + 1000
    ly1 = int(rec["yStart"].max() + rec["length"].max()) + 1000
    return rec, lx1, ly1, lr, pr, meta


@functools.lru_cache(maxsize=None)
def build_thresholds(lr, pr):
    """every case four ways: tier 1 (the case's segment alone), tier 2 with the entries in an earlier 32-member chunk than
    the query (phase A) and in the query's chunk (phase B), and the Y pass (far apart on X, with an X-matched member in the
    Y segment).  Every query lies at or above max_index (laid out twice: the axis length sets max_index)."""
    rec, lx1, ly1, *_ = _layout_thresholds(lr, pr, 1000)
    return _layout_thresholds(lr, pr, max(lx1, ly1) // 99 + 2000)


@pytest.mark.parametrize("lr,pr", RATIOS)
def test_threshold_builder_self_check(lr, pr):
    """the table contains what it is for: quotients exactly 1 (both, and one), pairs inside the 2^-40 band, exact ties
    decided by the rule the case names, entries processed before their query"""
    rec, lx1, ly1, lr, pr, meta = build_thresholds(lr, pr)
    assert lx1 < 1 << 32 and ly1 < 1 << 32
    rank = proc_rank(rec)
    seg, pos, size = x_segments(rec, lx1)
    parent = parents_by_file(rec, O.group(rec, lx1, ly1, lr, pr))
    both_one = one_one = band = 0
    seen = set()
    ways = {}
    for kind, way, ents, q in meta:
        ways.setdefault(kind, []).append(way)
        if way.startswith("tier2"):   # more than 32 members; the entries in an earlier chunk (A) or the query's (B)
            assert all(seg[e] == seg[q] for e in ents) and size[q] > 32, (kind, way, size[q])
            chunk_e = {int(pos[e]) // 32 for e in ents}
            assert chunk_e == ({int(pos[q]) // 32} if way == "tier2_phaseB" else chunk_e - {int(pos[q]) // 32}), (kind, way)
        elif way == "tier1":
            assert size[q] <= 32
        assert all(rank[e] < rank[q] for e in ents), (kind, way)
        assert all(rank[a] < rank[b] for a, b in zip(ents, ents[1:])), (kind, way)
        ax = "yStart" if way == "ypass" else "xStart"
        c = int(rec[ax][q]) + int(rec["length"][q]) // 2
        ln = int(rec["length"][q])
        assert c >= (lx1 if ax == "xStart" else ly1) // 100, (kind, way)   # no next-bucket probe from the query
        if kind == "grid":
            e = ents[0]
            dl, dc = abs(ln - int(rec["length"][e])), abs(c - int(rec[ax][e]) - int(rec["length"][e]) // 2)
            ql, qp = dl / (ln * lr), dc / (ln * pr)
            both_one += ql == 1.0 and qp == 1.0
            one_one += (ql == 1.0) != (qp == 1.0) and max(ql, qp) <= 1.0
            band += any(abs(d - ln * r) <= ln * r * BAND for d, r in ((dl, lr), (dc, pr)))
        else:
            seen.add(kind)
            sc = [deviation(int(rec[ax][e]) + int(rec["length"][e]) // 2, int(rec["length"][e]), c, ln, lr, pr) for e in ents]
            if kind.startswith("tie"):
                assert sc[0] == sc[1] > 0, (kind, sc)
                want = ents[0] if kind.startswith("tie_own_vs_neighbour") else ents[1]
            else:
                assert sc[0] > sc[1] > 0, sc
                want = ents[0]
            assert parent[q] == want, (kind, way, parent[q], want)
    assert band > 0
    if lr <= 1 and pr <= 1:
        assert both_one > 0 and one_one > 0
    if lr < 100:
        assert {"tie_own_vs_neighbour", "tie_mirrored", "dominance"} <= seen
    assert "tie_own_vs_neighbour" in seen
    if (1 << 20) * max(lr, pr) >= 1 << 30:
        assert "tie_own_vs_neighbour_big_t" in seen
    # every case runs every way, the same number of times
    for kind, w in ways.items():
        assert sorted(w) == sorted(WAYS * (len(w) // len(WAYS))) and len(w) % len(WAYS) == 0, (kind, sorted(set(w)))


@gpu
@pytest.mark.parametrize("lr,pr", RATIOS)
def test_thresholds_and_ties_match_oracle(ctx, m3, lr, pr):
    """k3_match.cu:139-156 (make_thresh, quotient_vs_one), :186-192 (band_candidate), :196-217 (best_of), :225-234
    (is_candidate), :426-509 (k_match_long: prune or, for t >= 2^30, none; phase A :460-467 and phase B :500-505 tie
    rules) at dl, dc in {0, floor(t)-1, floor(t), ceil(t), ceil(t)+1} for lengths 1..64, 100, 1000, 2^20, in tier 1, tier 2 (phase A and phase B) and the Y pass"""
    check_both(ctx, m3, build_thresholds(lr, pr))


# ---- B. the "next bucket" probe --------------------------------------------------------------------------------------------
B_RATIO = (2.0, 2.0)


def probe_query(c, rows, x_of, y_of, strand):
    """query at centre c with an own-bucket entry and, where the probe can reach one, a neighbour entry that scores higher
    (next bucket for residues 98/99, previous for 0/1): the query's owner shows whether the probe fired.  The entries are
    processed before the query and never see each other.  x_of / y_of give the coordinates on each axis (the other axis
    puts every fragment alone).  Returns the file indices (neighbour, own, query)."""
    def add(v, ln):
        rows.append((*x_of(v, c), *y_of(v, c), ln, strand))
        return len(rows) - 1
    if c < 20:                                   # first bucket: no neighbour below, the own entry one to the right
        lq = 2 * c + 1
        return None, add(c + 1 - lq // 2, lq), add(c - lq // 2, lq)
    lq = 40
    if c % 100 >= 98:                            # neighbour at the start of the next bucket, then the own entry, same xStart
        cn = (c // 100 + 1) * 100
        nb = add(c - lq // 2, lq + 2 * (cn - c))
        own = add(c - lq // 2, lq - 20)
    else:                                        # neighbour at the end of the previous bucket
        nb = add((c // 100) * 100 - 1 - lq // 2, lq) if c >= 100 else None
        own = add(c - lq // 2, lq + 20)
    return nb, own, add(c - lq // 2, lq)


@functools.lru_cache(maxsize=None)
def build_probes(mres):
    """M = lx1/100 = ly1/100 = 1000 + mres (mres in 97, 98, 99, 100, 101).  The two centres in M-3 .. M+2 with residue 98/99:
    on X (residue 98 forward, 99 reverse) and on Y (99 forward, 98 reverse), the other axis far away; then the residue 0/1
    and first-bucket centres on both axes."""
    M = 1000 + mres
    lx1 = 100 * M + 37
    cs = [c for c in range(M - 3, M + 3) if c % 100 in (98, 99)]
    assert len(cs) == 2
    rows = []
    far = Axis(5000)
    cases = []
    for axis, strands in (("x", (b"f", b"r")), ("y", (b"r", b"f"))):
        for c, s in zip(cs, strands):
            if axis == "x":
                idx = probe_query(c, rows, lambda v, c: (v,), lambda v, c: (far.take(100) + 10,), s)
            else:
                idx = probe_query(c, rows, lambda v, c: (far.take(100) + 10,), lambda v, c: (v,), s)
            cases.append((axis, c, s, idx))
    extra = [0, 1, 98, 99, 100, 101, 200, 201, 5000, 5001]
    for i, c in enumerate(extra):
        # one slot per centre: alternate axis and strand so that no two of these centres meet in one list
        axis, s = ("x", "y")[i % 2], (b"f", b"r")[(i // 2) % 2]
        if any(abs(c - c2) < 300 for a2, c2, s2, _ in cases if (a2, s2) == (axis, s)):
            axis = "y" if axis == "x" else "x"
            if any(abs(c - c2) < 300 for a2, c2, s2, _ in cases if (a2, s2) == (axis, s)):
                s = b"r" if s == b"f" else b"f"
                if any(abs(c - c2) < 300 for a2, c2, s2, _ in cases if (a2, s2) == (axis, s)):
                    continue
        if axis == "x":
            idx = probe_query(c, rows, lambda v, c: (v,), lambda v, c: (far.take(100) + 10,), s)
        else:
            idx = probe_query(c, rows, lambda v, c: (far.take(100) + 10,), lambda v, c: (v,), s)
        cases.append((axis, c, s, idx))
    rec = records(rows)
    assert int(rec["xStart"].max()) < lx1 - 100 and int(rec["yStart"].max()) < lx1 - 100
    return rec, lx1, lx1, B_RATIO[0], B_RATIO[1], cases


@pytest.mark.parametrize("mres", [97, 98, 99, 100, 101])
def test_probe_builder_self_check(mres):
    rec, lx1, ly1, lr, pr, cases = build_probes(mres)
    M = lx1 // 100
    assert M % 100 == mres % 100
    near = [c for a, c, s, _ in cases if M - 3 <= c <= M + 2]
    assert sorted(c % 100 for c in near) == [98, 98, 99, 99]
    assert {(a, s) for a, c, s, _ in cases if c in near} == {("x", b"f"), ("x", b"r"), ("y", b"f"), ("y", b"r")}
    # the query joins the neighbour entry exactly where get_associated_group probes it (:47, :58, :80), else the own entry
    parent = parents_by_file(rec, O.group(rec, lx1, ly1, lr, pr))
    for axis, c, s, (nb, own, q) in cases:
        r = c % 100
        fires = (r == 99 and c < M) or (r == 98 and c < M - 1) or (r <= 1 and c >= 100)
        assert parent[q] == (nb if fires else own), (axis, c, s, parent[q], nb, own)


@gpu
@pytest.mark.parametrize("mres", [97, 98, 99, 100, 101])
def test_probe_edges_match_oracle(ctx, m3, mres):
    """rk_common.cuh:65-74 (probes_next / probes_prev) as K1 raises link bits (k1_decode.cu:109-112) and K3 picks the
    neighbour bucket (k3_match.cu:115-120): centres M-3 .. M+2 with residue 98/99 for M = 1097 .. 1101, residues 0/1, and
    centres 0, 1, 98, 99, 100, 101"""
    check_both(ctx, m3, build_probes(mres))


# ---- C. tier-1 windows, tiles and linked runs --------------------------------------------------------------------------------
SEG_SIZES = [1, 2, 31, 32, 33, 34, 63, 64, 65]
SEG_OFFSETS = [0, 1, 31, 32, 63, 224, 255]
SEG_RATIO = (0.05, 0.05)


@functools.lru_cache(maxsize=None)
def build_segments():
    """every segment size at every start offset mod 256 of the sorted X positions: fillers alone in unlinked buckets move
    the next segment's first position.  Members: length 200 (t = 10), centres 7 apart with every third one 13 apart, so
    neighbours are candidates and the chains need several phase-2 rounds; a few lengths differ by 15 (not candidates)."""
    rows, pos, heads = [], 0, []
    b = 10
    for k in SEG_SIZES:
        for off in SEG_OFFSETS:
            while pos % 256 != off:
                rows.append((100 * b + 50 - 50, 100 * b + 50 - 50, 100, b"f"))   # centre at residue 50, alone
                b += 3
                pos += 1
            heads.append((k, off, pos))
            c = 100 * b + 5
            for j in range(k):
                ln = 200 if j % 5 != 4 else 215
                cc = c + (j * 7 + (j // 3) * 6) % 90
                rows.append((cc - ln // 2, cc - ln // 2, ln, b"f"))
            pos += k
            b += 3
    rec = records(rows)
    lx1 = int(rec["xStart"].max()) + 5000
    return rec, lx1, lx1, SEG_RATIO[0], SEG_RATIO[1], heads


def run_rows(rows, start_bucket, n, strand, ln=20):
    """a run of n linked buckets: a residue-98 entry in every bucket and a residue-1 query in every bucket after the first,
    which joins the previous bucket's entry (dc = 3)"""
    for b in range(start_bucket, start_bucket + n):
        rows.append((100 * b + 98 - ln // 2, 100 * b + 98 - ln // 2, ln, strand))
        if b > start_bucket:
            rows.append((100 * b + 1 - ln // 2, 100 * b + 1 - ln // 2, ln, strand))
    if start_bucket == 0:
        rows.append((50 - ln // 2, 50 - ln // 2, ln, strand))


RUN_LENGTHS = [31, 32, 33, 64, 65, 1000]


@functools.lru_cache(maxsize=None)
def build_runs(rev_start):
    """forward runs of every length starting at buckets = 31, 32, 33 (mod 2048); reverse-class runs of every length, one
    starting at bucket rev_start (0 or 1: the base of the reverse class, bit nbx of the link map) and the rest after it"""
    rows, starts = [], []
    for i, n in enumerate(RUN_LENGTHS):
        for j, s in enumerate((31, 32, 33)):
            sb = 2048 * (3 * i + j + 1) + s
            run_rows(rows, sb, n, b"f")
            starts.append(("f", sb, n))
    rb = rev_start
    for n in RUN_LENGTHS:
        run_rows(rows, rb, n, b"r")
        starts.append(("r", rb, n))
        rb = -(-(rb + n + 40) // 32) * 32 + (rev_start + 31) % 32
    rec = records(rows)
    lx1 = int(rec["xStart"].max()) + 20_000
    return rec, lx1, lx1, 0.5, 0.5, starts


def test_segment_builder_self_check():
    rec, lx1, ly1, lr, pr, heads = build_segments()
    # sorted X positions: (strand class, bucket of the centre) — no probes fire (residues 5..94, centres >= max_index)
    cx = rec["xStart"] + rec["length"] // np.uint64(2)
    assert ((cx % np.uint64(100) >= np.uint64(2)) & (cx % np.uint64(100) <= np.uint64(97))).all()
    key = cx // np.uint64(100)
    order = np.lexsort((proc_rank(rec), key))
    skey = key[order]
    seg_start = np.r_[0, np.nonzero(skey[1:] != skey[:-1])[0] + 1]
    sizes = np.diff(np.r_[seg_start, rec.shape[0]])
    got = {(int(sz), int(s % 256)) for s, sz in zip(seg_start, sizes) if sz > 1 or s in {h[2] for h in heads}}
    for k, off, pos in heads:
        assert (k, off) in got and pos % 256 == off
    g = O.group(rec, lx1, ly1, lr, pr)
    assert g.n_groups < rec.shape[0] and np.bincount(g.gid).max() >= 2


@pytest.mark.parametrize("rev_start", [0, 1])
def test_run_builder_self_check(rev_start):
    rec, lx1, ly1, lr, pr, starts = build_runs(rev_start)
    g = O.group(rec, lx1, ly1, lr, pr)
    sizes = np.bincount(g.gid)
    assert (sizes == 2).sum() >= sum(n - 1 for _, _, n in starts) - 2   # every residue-1 query joined across a bucket edge
    assert {s % 32 for k, s, n in starts if k == "f"} == {31, 0, 1}
    assert min(s for k, s, n in starts if k == "r") == rev_start


@gpu
def test_segment_alignment_matches_oracle(ctx, m3):
    """k3_match.cu:245-293 (k_match_small phase 0: heads, the window straddle, tier-2 hand-off) and :256,273 (tile and
    halo): segments of 1..65 members starting at positions 0, 1, 31, 32, 63, 224, 255 mod 256"""
    check_both(ctx, m3, build_segments())


@gpu
@pytest.mark.parametrize("rev_start", [0, 1])
def test_linked_runs_match_oracle(ctx, m3, rev_start):
    """rk_common.cuh:79-90 (run_start over several link words) and k3_match.cu:70-71 (k_keys): runs of 31 .. 1000 linked
    buckets across 32-bucket words, and runs at the base of the reverse strand class"""
    check_both(ctx, m3, build_runs(rev_start))


# ---- D. size classes through rk_group ----------------------------------------------------------------------------------------
GROUP_SIZES = [1, 2, 15, 16, 17, 31, 32, 33, 127, 128, 129, 1023, 1024, 1025, 1026, 2049]


def _killer(n):
    """median-of-three killer (Musser 1997): drives libstdc++'s introsort to its depth limit and into heap sort"""
    k = n // 2
    a = np.zeros(n, np.int64)
    for i in range(1, k + 1):
        if i % 2:
            a[i - 1] = i
            a[i] = k + i
        a[k + i - 1] = 2 * i
    return a[:n]


@functools.lru_cache(maxsize=None)
def build_size_classes():
    """groups of exactly GROUP_SIZES members (same xStart and length: all join the first member in X), with h random, tied,
    constant, sorted, reversed or a median-of-three killer; a last fragment of the xStart/10 bucket of another length (not a
    candidate) fixes diag_func, so h is the pattern itself.  Every group in its own Y region."""
    rng = np.random.default_rng(17)
    patterns = {"random": lambda n: rng.integers(0, 4 * n + 8, n), "tied": lambda n: rng.integers(0, 4, n),
                "constant": lambda n: np.full(n, 5), "sorted": lambda n: np.arange(n), "reversed": lambda n: np.arange(n)[::-1],
                "killer": _killer}
    rows, want = [], []
    X, Y = Axis(), Axis()
    ln = 1000
    for name, fn in patterns.items():
        for n in GROUP_SIZES:
            k = np.asarray(fn(n), np.int64)
            x = X.take(3 * ln)
            y = Y.take(int(k.max()) + 3 * ln)
            for kk in k:
                rows.append((x, y + ln + int(kk), ln, b"f"))
            rows.append((x, y + ln, 2 * ln, b"f"))
            want.append((name, n))
    rec = records(rows)
    lx1 = int(rec["xStart"].max()) + 5000
    ly1 = int(rec["yStart"].max()) + 5000
    return rec, lx1, ly1, 0.05, 0.05, want


def test_size_class_builder_self_check():
    rec, lx1, ly1, lr, pr, want = build_size_classes()
    g = O.group(rec, lx1, ly1, lr, pr)
    sizes = np.bincount(g.gid)
    got = sorted(int(s) for s in sizes)
    expect = sorted([n for _, n in want] + [1] * len(want))
    assert got == expect


@gpu
def test_size_classes_through_group_match_oracle(ctx, m3):
    """k5_order.cu through rk_group's gathered layout (OrderArgs::srank, hfi_r): groups of 1 .. 2049 members around the
    16 / 128 / 1024 class boundaries under random, tied, constant, sorted, reversed and killer keys"""
    check_both(ctx, m3, build_size_classes())


# ---- E. 32-bit geometry ------------------------------------------------------------------------------------------------------
def _host_bytes():
    """MemAvailable: what the host can give without swapping (free pages plus reclaimable cache)"""
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 0


@functools.lru_cache(maxsize=None)
def build_full32(lx_header):
    """gen-style background over the whole axis plus copies of the threshold (ratios 0.05), probe, segment, run and
    size-class inputs moved to the top of the axes (by multiples of 100,000: residues and xStart/10 relations stay), centres
    up to 2^32-1, rows in the last visited X bucket (vsize-2) and in the dropped one (vsize-1)"""
    lx1 = lx_header + 1
    w = gen.Workload("full32", 250_000, lx_header, lx_header, 0.3, 20_000, seed=9)
    parts = [gen.generate(w)]
    top = []
    for rec, *_ in (build_thresholds(0.05, 0.05), build_probes(100), build_segments(), build_runs(1), build_size_classes()):
        top.append(rec)
    span = max(int(max(r["xStart"].max(), r["yStart"].max()) + r["length"].max()) for r in top)
    base = 0
    for r in top:
        r = r.copy()
        shift = np.uint64(((lx1 - span - 100_000) // 100_000 - base) * 100_000)
        r["xStart"] += shift
        r["yStart"] += shift
        r["xEnd"] += shift
        r["yEnd"] += shift
        parts.append(r)
        base += -(-span // 100_000) + 1
    vs = 1 + lx1 // 10
    edge = []
    xl = 10 * (vs - 2)                       # last visited X bucket
    for i in range(10):
        x = xl + i
        ln = 2 * (lx1 - x)                   # centre lx1 = 2^32 - 1 at the full geometry
        edge.append((x, lx1 - 1 - ln // 2 - i * 3, ln, b"f" if i % 2 else b"r"))
    for i in range(6):
        edge.append((10 * (vs - 1) + min(i, lx1 - 1 - 10 * (vs - 1)), 1000 + 50 * i, 1, b"f"))   # dropped bucket
    parts.append(records(edge))
    rec = np.concatenate(parts)
    return rec, lx1, lx1, 0.05, 0.05


def full32_header():
    """4,294,967,294 (loaded length 2^32-1) when the host can hold the oracle's ~10 GB of per-bucket tables; otherwise
    config 5's 3 Gbp, whose rank and X/Y keys also need 4 radix passes"""
    return 4_294_967_294 if _host_bytes() > 24 << 30 else 3_000_000_000


def test_full32_builder_self_check():
    lx_header = 4_294_967_294
    lx1 = lx_header + 1
    vs = 1 + lx1 // 10
    assert math.ceil(math.log2(vs)) == 29 and math.ceil(math.log2(2 * (lx1 // 100 + 2))) == 27
    assert math.ceil(math.log2(1 + 3_000_000_001 // 10)) > 24 and math.ceil(math.log2(2 * (3_000_000_001 // 100 + 2))) > 24
    if _host_bytes() > 24 << 30:
        rec, lx1, ly1, lr, pr = build_full32(lx_header)
        cx = rec["xStart"] + rec["length"] // np.uint64(2)
        assert int(cx.max()) == (1 << 32) - 1
        assert ((rec["xStart"] // np.uint64(10)) == np.uint64(vs - 2)).any()
        assert ((rec["xStart"] // np.uint64(10)) == np.uint64(vs - 1)).any()


@gpu
def test_full_32bit_geometry_matches_oracle(ctx, m3):
    """capi.cu:352-354 (bits_rank 29, bits_x/bits_y 27: four radix passes) with K1's digit counts (k1_decode.cu HistOut,
    capi.cu:391-421), k_keys' (k3_match.cu:76-85), centres up to 2^32-1, the last visited and the dropped X bucket.  The
    geometry that ran is printed (3 Gbp when the host has less than 24 GB available)."""
    lx_header = full32_header()
    print(f"full geometry: loaded lengths {lx_header + 1:,}")
    rec, lx1, ly1, _, _ = build_full32(lx_header)
    for lr, pr in ((0.05, 0.05), B_RATIO):   # the threshold and segment copies' ratios, then the probe copies'
        check_both(ctx, m3, (rec, lx1, ly1, lr, pr))


@gpu
def test_centre_2pow32_is_refused(ctx):
    """k1_decode.cu:83-87: a centre of 2^32 does not fit the 32-bit kernels and is refused (RK_ERR_RANGE), the context
    stays usable"""
    lx1 = (1 << 32) - 1
    rec = records([(4_294_967_280, 100, 32, b"f")])      # centre 2^32
    with pytest.raises(capi.RkError) as e:
        ctx.load(rec, lx1, lx1)
    assert e.value.code == -3
    rec = records([(4_294_967_279, 100, 32, b"f"), (4_294_967_279, 100, 32, b"f")])   # centre 2^32-1
    check_one_gpu(ctx, rec, lx1, lx1, 0.05, 0.05)


@gpu
def test_c2_shape_above_2pow24_kept_fragments(ctx):
    """capi.cu:494-501: more than 2^24 kept fragments, so the gid sort takes 4 passes (255 Mbp: the rank sort too)"""
    w = gen.scaled(gen.WORKLOADS["c2"], 17_000_000)
    rec = gen.generate(w)
    g = check_one_gpu(ctx, rec, w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio, text=False)
    assert g.n_kept > 1 << 24


# ---- F. single-call occupation lists --------------------------------------------------------------------------------------------
def sol_ops(seed, seq_size, n_ops):
    """interleaved inserts and queries: centres near max_index, at residues 0, 1, 98, 99, and anywhere in the list"""
    rng = np.random.default_rng(seed)
    mi = seq_size // 100
    ops = []
    for i in range(n_ops):
        kind = rng.integers(0, 4)
        if kind == 0:
            c = int(rng.integers(max(0, mi - 3), mi + 3))
        elif kind == 1:
            c = int(rng.integers(0, max(1, seq_size // 100 - 1))) * 100 + int(rng.choice([0, 1, 98, 99]))
        else:
            c = int(rng.integers(0, seq_size))
        c = min(c, seq_size - 1)
        ln = int(rng.integers(1, 60))
        ops.append(("i" if rng.random() < 0.55 else "q", c, ln, i + 1))
    return ops


def run_sol(sol, ops, get):
    out = []
    for op, c, ln, tag in ops:
        if op == "i":
            sol.insert(c, ln, tag)
        else:
            out.append(get(sol, c, ln))
    return out


SOL_GEOMS = [(100 * (1000 + r) + 37) for r in (97, 98, 99, 100, 101)] + [10_037, 250]


def test_sol_oracle_self_check():
    o = O.Sol(0.5, 0.5, 100_037)
    o.insert(1000, 20, 7)
    o.insert(1002, 20, 9)
    assert o.get(1001, 20) == 9           # equal score, newest first
    assert o.get(5000, 20) == 0
    with pytest.raises(IndexError):
        o.insert(100_037 + 100, 20, 1)
    o.close()


@gpu
@pytest.mark.parametrize("seq_size", SOL_GEOMS)
def test_sol_matches_oracle(seq_size):
    """sol.cu:44-78 (k_sol_apply, k_sol_query: the +1 / +2 probes under center < max_index, max_index-1) and :207-232
    against the restatement's lists, queries interleaved with inserts, around max_index"""
    for lr, pr in [(0.5, 0.5), (2.0, 2.0), (0.05, 1.0)]:
        ops = sol_ops(seq_size, seq_size, 4000)
        with capi.Sol(0, lr, pr, seq_size) as s:
            got = run_sol(s, ops, lambda s, c, ln: s.get_associated(c, ln))
        o = O.Sol(lr, pr, seq_size)
        want = run_sol(o, ops, lambda s, c, ln: s.get(c, ln))
        o.close()
        assert got == want, (lr, pr, next(i for i, (a, b) in enumerate(zip(got, want)) if a != b))
        assert sum(1 for t in want if t) > len(want) // 10


@gpu
def test_sol_flush_pool_growth_and_u64_operands():
    """sol.cu:130-162 (more than 65,536 inserts between two queries: a flush inside rk_sol_insert, pool growth) and
    sol.cu:33-41 (deviation64: lengths and tags above 2^53); tag 0 and centres beyond the list are refused"""
    seq = 1_000_037
    rng = np.random.default_rng(3)
    with capi.Sol(0, 0.3, 0.7, seq) as s:
        o = O.Sol(0.3, 0.7, seq)
        for i in range(70_000):
            c, ln = int(rng.integers(0, seq)), int(rng.integers(1, 200))
            s.insert(c, ln, i + 1)
            o.insert(c, ln, i + 1)
        for _ in range(300):
            c, ln = int(rng.integers(0, seq)), int(rng.integers(1, 200))
            assert s.get_associated(c, ln) == o.get(c, ln)
        with pytest.raises(capi.RkError) as e:
            s.insert(5, 5, 0)
        assert e.value.code == -2
        with pytest.raises(capi.RkError) as e:
            s.insert(seq + 100, 5, 1)
        assert e.value.code == -3
        with pytest.raises(capi.RkError) as e:
            s.get_associated(seq + 100, 5)
        assert e.value.code == -3
        o.close()
    # lengths above 2^53 (a unit of difference is below the resolution of the conversion to binary64); centres above 2^53
    # would need a list of 2^53/100 heads, so the centres stay within a list of 10 Mbp
    seq = 10_000_037
    with capi.Sol(0, 0.5, 0.5, seq) as s:
        o = O.Sol(0.5, 0.5, seq)
        for i in range(3000):
            c = int(rng.integers(0, seq))
            ln = (1 << 54) + int(rng.integers(0, 1 << 20))
            if i % 3 == 2:
                assert s.get_associated(c, ln) == o.get(c, ln)
            else:
                s.insert(c, ln, (1 << 63) + i)
                o.insert(c, ln, (1 << 63) + i)
        for k in range(50):
            c = 12345 + 1000 * k
            s.insert(c, (1 << 55) + k, 100_000 + k)
            o.insert(c, (1 << 55) + k, 100_000 + k)
            assert s.get_associated(c + 1, (1 << 55) + k + 3) == o.get(c + 1, (1 << 55) + k + 3)
        o.close()
