"""Parity of the CUDA path (through the C ABI) against the oracle and the reference's golden outputs.
Run on the B200 box: python -m pytest tests -m gpu"""
import hashlib
import os

import numpy as np
import pytest

from oracle import oracle as O
from repkiller_b200 import capi, gen
from repkiller_b200.frags import FRAG_DTYPE, make_header

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def first_diff(a, b):
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape:
        return f"shape {a.shape} vs {b.shape}"
    d = np.nonzero(a != b)[0]
    if d.size == 0:
        return None
    i = int(d[0])
    return f"{d.size} diffs, first at {i}: got {a[max(0, i - 2):i + 3]} want {b[max(0, i - 2):i + 3]}"


def assert_same(name, got, want):
    msg = first_diff(got, want)
    assert msg is None, f"{name}: {msg}"


def check_against_oracle(ctx, rec, lx1, ly1, lr, pr, stages=True):
    st = ctx.load(rec, lx1, ly1)
    g = O.group(rec, lx1, ly1, lr, pr)
    assert st.n_kept == g.n_kept
    assert st.vsize == g.vsize
    if stages and g.n_kept:
        assert_same("rank_fidx", ctx.debug_fetch("rank_fidx"), g.rank_fidx)
    res = ctx.group(lr, pr)
    if stages and g.n_kept:
        assert_same("parent", ctx.debug_fetch("parent"), g.parent)
        assert_same("gid_rank", ctx.debug_fetch("gid_rank"), g.gid)
        assert_same("hkey", ctx.debug_fetch("hkey"), g.h.astype(np.uint32))
    assert res.n_groups == g.n_groups
    assert_same("out_gid", res.gid, g.out_gid)
    assert_same("order", res.order, g.order)
    assert_same("repval", res.repval, g.repval)
    assert_same("identity(bits)", res.identity.view(np.uint32), g.identity.view(np.uint32))
    return res, g


def test_sort_pairs_matches_stable_sort(ctx):
    import torch
    dev = torch.device("cuda:0")
    gen_ = torch.Generator(device="cpu").manual_seed(5)
    for n, bits in [(1, 1), (33, 5), (4096, 8), (4097, 9), (100_003, 17), (1_000_000, 24), (300_000, 32), (70_000, 3)]:
        keys = torch.randint(0, 2 ** bits, (n,), generator=gen_, dtype=torch.int64).to(torch.int32).to(dev) if bits < 32 else \
            torch.randint(-2 ** 31, 2 ** 31, (n,), generator=gen_, dtype=torch.int64).to(torch.int32).to(dev)
        ko, vo, kt, vt = (torch.empty(n, dtype=torch.int32, device=dev) for _ in range(4))
        work = torch.empty(ctx.sort_pairs_work_bytes(n), dtype=torch.uint8, device=dev)
        torch.cuda.synchronize()
        ctx.sort_pairs_device(keys.data_ptr(), None, ko.data_ptr(), vo.data_ptr(), kt.data_ptr(), vt.data_ptr(), n, bits,
                              work.data_ptr())
        ku = keys.cpu().numpy().view(np.uint32)
        perm = np.argsort(ku, kind="stable")
        assert_same(f"sorted keys n={n} bits={bits}", ko.cpu().numpy().view(np.uint32), ku[perm])
        assert_same(f"sorted values n={n} bits={bits}", vo.cpu().numpy().view(np.uint32), perm.astype(np.uint32))


def test_c1_every_stage(ctx):
    w = gen.WORKLOADS["c1"]
    rec = gen.generate(w)
    check_against_oracle(ctx, rec, w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio)


def test_fuzz_golden_bytes(ctx, fuzz_cases, tmp_path):
    """Tiny adversarial inputs: the CUDA result, written with the reference's line format, must reproduce the
    bytes the reference itself produced (tests/golden/fuzz.json.gz)."""
    for c in fuzz_cases:
        inp = tmp_path / "in.csv"
        inp.write_text(c["csv"], newline="")
        rec, lx1, ly1, hdr = O.load_csv(str(inp))
        res, g = check_against_oracle(ctx, rec, lx1, ly1, c["len_ratio"], c["pos_ratio"])
        g.order, g.out_gid, g.repval, g.identity = res.order, res.gid, res.repval, res.identity
        outp = tmp_path / "out.csv"
        O.write_output(str(outp), hdr, rec, g)
        assert outp.read_bytes() == c["ref_out"].encode("latin1"), f"fuzz seed {c['seed']}"
        # K6: the same bytes formatted on the device (the header lines are the host's)
        assert hdr + ctx.format_lines() == c["ref_out"].encode("latin1"), f"device text, fuzz seed {c['seed']}"


@pytest.mark.parametrize("name", ["c1_loose", "c3_small", "dense", "c2_small"])
def test_medium_golden_md5(ctx, medium_cases, tmp_path, name):
    c = medium_cases[name]
    w = gen.Workload(**c["workload"])
    rec = gen.generate(w)
    res, g = check_against_oracle(ctx, rec, w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio)
    g.order, g.out_gid, g.repval, g.identity = res.order, res.gid, res.repval, res.identity
    outp = tmp_path / "out.csv"
    O.write_output(str(outp), make_header(w.lx, w.ly, w.n).encode(), rec, g)
    assert hashlib.md5(outp.read_bytes()).hexdigest() == c["ref_md5"]
    text = ctx.format_lines()   # K6: device-side formatter, byte for byte the reference's lines
    assert hashlib.md5(make_header(w.lx, w.ly, w.n).encode() + text).hexdigest() == c["ref_md5"]
    # chunked calls return the same bytes
    k = res.n_kept // 3
    assert ctx.format_lines(0, k) + ctx.format_lines(k, res.n_kept - k) == text


def test_device_text_float_formats(ctx, tmp_path):
    """printf("%g") of every kind of float the two float columns can hold (similarity is whatever the input carried):
    denormals, powers of ten and their neighbours, rounding ties, inf, nan, -0; and 20-digit integers."""
    rng = np.random.default_rng(11)
    n = 40_000
    rec = np.zeros(n, FRAG_DTYPE)
    rec["xStart"] = rng.integers(0, 9_000, n)
    rec["yStart"] = rng.integers(0, 9_000, n)
    rec["length"] = rng.integers(0, 400, n)            # length 0: identity is inf or -nan
    rec["ident"] = rng.integers(0, 400, n)
    rec["xEnd"] = rng.integers(0, 2 ** 63, n, dtype=np.uint64) * 2 + 1   # 19/20-digit integers
    rec["yEnd"] = rng.integers(0, 2 ** 40, n)
    rec["score"] = rng.integers(0, 2 ** 63, n, dtype=np.uint64)
    rec["strand"] = rng.choice([b"f", b"r"], n)
    bits = rng.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32)
    special = np.array([0, 0x80000000, 1, 0x007FFFFF, 0x00800000, 0x7F7FFFFF, 0x7F800000, 0xFF800000, 0x7FC00000, 0xFFC00000,
                        0x49742400, 0x49742408, 0x497423F8, 0x38D1B717, 0x38D1B716, 0x3A83126F, 0x42AFD70A], dtype=np.uint32)
    bits[: special.size] = special
    pct = (rng.integers(0, 10001, n // 2) / np.float32(100)).astype(np.float32)   # "87.92"-like values
    bits[n // 2:] = pct.view(np.uint32)
    rec["similarity"] = bits.view(np.float32)
    res, g = check_against_oracle(ctx, rec, 10_001, 10_001, 0.05, 0.05)
    g.order, g.out_gid, g.repval, g.identity = res.order, res.gid, res.repval, res.identity
    outp = tmp_path / "out.csv"
    O.write_output(str(outp), b"", rec, g)
    want, got = outp.read_bytes(), ctx.format_lines()
    if want != got:
        wl, gl = want.split(b"\n"), got.split(b"\n")
        bad = [(a, b) for a, b in zip(wl, gl) if a != b][:5]
        raise AssertionError(f"{len(wl)} vs {len(gl)} lines; first differences: {bad}")


def test_edge_inputs(ctx):
    # empty database
    st = ctx.load(np.zeros(0, FRAG_DTYPE), 1001, 1001)
    assert st.n_kept == 0
    res = ctx.group(0.05, 0.05)
    assert res.n_groups == 0 and res.n_kept == 0
    # everything in the dropped last bucket (vsize-1 == xStart/10)
    rec = np.zeros(5, FRAG_DTYPE)
    rec["xStart"] = 1000
    rec["length"] = 1
    rec["strand"] = b"f"
    st = ctx.load(rec, 1001, 1001)
    assert st.n_kept == 0
    assert ctx.group(0.5, 0.5).n_kept == 0
    # one fragment; duplicates (exact ties: newest entry wins)
    rec = np.zeros(7, FRAG_DTYPE)
    rec["xStart"] = [10, 10, 10, 500, 10, 10, 10]
    rec["yStart"] = [20, 20, 700, 20, 20, 20, 20]
    rec["length"] = 30
    rec["ident"] = 7
    rec["strand"] = [b"f", b"f", b"f", b"f", b"r", b"x", b"f"]
    check_against_oracle(ctx, rec[:1], 1001, 1001, 0.05, 0.05)
    check_against_oracle(ctx, rec, 1001, 1001, 0.05, 0.05)
    # no sort: members stay in processing order
    res = ctx.group(0.05, 0.05, sort=False)
    g = O.group(rec, 1001, 1001, 0.05, 0.05)
    assert_same("gid multiset", np.sort(res.gid), np.sort(g.out_gid))


def test_error_behaviour(ctx):
    rec = np.zeros(3, FRAG_DTYPE)
    rec["xStart"] = [5, 20000, 7]
    rec["length"] = 10
    with pytest.raises(capi.RkError) as e:
        ctx.load(rec, 1001, 1001)           # xStart/10 >= vsize: the reference writes out of bounds
    assert e.value.code == -3
    with pytest.raises(capi.RkError) as e:
        ctx.group(0.05, 0.05)               # nothing loaded after a failed load
    assert e.value.code == -4
    rec["xStart"] = [5, 6, 7]
    ctx.load(rec, 1001, 1001)
    for bad in [(0.0, 0.1), (0.1, -1.0)]:
        with pytest.raises(capi.RkError) as e:
            ctx.group(*bad)                 # init_args rejects non-positive ratios (commonFunctions.cpp:26-27)
        assert e.value.code == -2
    rec["length"] = [10, 5000, 10]          # center beyond the occupation list
    with pytest.raises(capi.RkError) as e:
        ctx.load(rec, 1001, 1001)
    assert e.value.code == -3


def test_device_pointer_input(ctx):
    import torch
    w = gen.scaled(gen.WORKLOADS["c2"], 200_000)
    rec = gen.generate(w)
    t = torch.from_numpy(rec.view(np.uint8).copy()).cuda()
    torch.cuda.synchronize()
    ctx.load(t.data_ptr(), w.lx + 1, w.ly + 1, n=w.n)
    res = ctx.group(w.len_ratio, w.pos_ratio)
    g = O.group(rec, w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio)
    assert_same("order", res.order, g.order)
    assert_same("gid", res.gid, g.out_gid)


def test_diagonal_func_table(ctx):
    w = gen.scaled(gen.WORKLOADS["c1"], 20_000)
    rec = gen.generate(w)
    st = ctx.load(rec, w.lx + 1, w.ly + 1)
    g = O.group(rec, w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio, want_diag=True)
    assert_same("diag_func", ctx.diagonal_func(st.vsize), g.diag_func)


def test_ratio_sweep_reuses_loaded_database(ctx):
    """One loaded database, several (len_ratio, pos_ratio) pairs (src/repkiller.cpp:60-72)."""
    w = gen.scaled(gen.WORKLOADS["c1"], 50_000)
    rec = gen.generate(w)
    ctx.load(rec, w.lx + 1, w.ly + 1)
    for lr, pr in [(0.05, 0.05), (0.5, 0.5), (1.0, 0.1), (2.5, 3.0)]:
        res = ctx.group(lr, pr)
        g = O.group(rec, w.lx + 1, w.ly + 1, lr, pr)
        assert res.n_groups == g.n_groups
        assert_same(f"order {lr},{pr}", res.order, g.order)
        assert_same(f"gid {lr},{pr}", res.gid, g.out_gid)


# ---- the drop-in CLI and the reference-named facades (host C++ over the C ABI) ----------------------------
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "repkiller_b200", "bin", "repkiller")
HOSTCHECK = os.path.join(ROOT, "repkiller_b200", "bin", "rk_hostcheck")
BANNER = ("--- Running REPKILLER v0.9.b ---\n     Bitlab - Arquitectura de Computadores\n"
          "           Universidad de Málaga 2018\n\nRepkiller finished with no errors\n").encode()


def test_cli_bytes_equal_reference_on_fuzz(fuzz_cases, tmp_path):
    import subprocess
    for c in fuzz_cases[::3]:
        inp = tmp_path / "in.csv"
        inp.write_text(c["csv"], newline="")
        outp = tmp_path / "out.csv"
        p = subprocess.run([CLI, str(inp), str(outp), repr(c["len_ratio"]), repr(c["pos_ratio"])], capture_output=True)
        assert p.returncode == 0, p.stderr
        assert p.stdout == BANNER
        assert outp.read_bytes() == c["ref_out"].encode("latin1"), f"fuzz seed {c['seed']}"


def test_cli_and_facade_steps_on_c1(medium_cases, tmp_path):
    import subprocess
    c = medium_cases["c1"]
    w = gen.Workload(**c["workload"])
    rec = gen.generate(w)
    inp = tmp_path / "c1.csv"
    O.write_input_csv(str(inp), rec, w.lx, w.ly)
    # the reference's golden md5 was produced from this same CSV shape (tests/golden/make_golden.py)
    for tool, args in [(CLI, []), (HOSTCHECK, ["steps"])]:
        outp = tmp_path / "out.csv"
        cmd = [tool, *args, str(inp), str(outp), "0.05", "0.05"]
        p = subprocess.run(cmd, capture_output=True)
        assert p.returncode == 0, p.stderr
        assert hashlib.md5(outp.read_bytes()).hexdigest() == c["ref_md5"], tool
        outp.unlink()


def test_cli_unwritable_output_falls_back(tmp_path, fuzz_cases):
    import subprocess
    c = fuzz_cases[0]
    inp = tmp_path / "in.csv"
    inp.write_text(c["csv"], newline="")
    p = subprocess.run([CLI, str(inp), "/nonexistent-dir/out.csv", repr(c["len_ratio"]), repr(c["pos_ratio"])],
                       capture_output=True, cwd=tmp_path)
    assert p.returncode == 0
    assert b"Couldn't access /nonexistent-dir/out.csv, saving into represults-1.csv" in p.stderr
    assert (tmp_path / "represults-1.csv").read_bytes() == c["ref_out"].encode("latin1")


@pytest.mark.parametrize("name", ["c2", "c3"])
def test_full_size_workloads_match_oracle(ctx, name):
    """BASELINE configs 2 and 3 at their full 10M fragments: every output array bit-exact vs the oracle, plus the
    size-independent properties (each kept fragment exactly once, gids non-decreasing and dense, repval pattern)."""
    w = gen.WORKLOADS[name]
    rec = gen.generate(w)
    res, g = check_against_oracle(ctx, rec, w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio, stages=False)
    assert np.array_equal(np.sort(res.order), np.sort(g.rank_fidx))
    assert (np.diff(res.gid.astype(np.int64)) >= 0).all() and res.gid[-1] + 1 == res.n_groups
    head = np.r_[True, res.gid[1:] != res.gid[:-1]]
    size = np.bincount(res.gid)[res.gid]
    assert np.array_equal(res.repval, np.where(size == 1, 0, np.where(head, 1, 2)).astype(np.uint8))
    print(name, "groups", res.n_groups, "max group", int(size.max()), "device ms", res.ms_device)


def test_device_generator_matches_host_generator(ctx):
    """rk_gen_workload (device) must produce the bytes of repkiller_b200.gen.generate (host) — it is what the
    1e9-fragment benchmark uses instead of a host-generated file."""
    import torch
    from dataclasses import replace
    for w, start, count in [(gen.WORKLOADS["c2"], 9_000_000, 300_001), (gen.WORKLOADS["c3"], 123, 200_000),
                            (gen.WORKLOADS["c5"], 999_000_000, 100_000), (replace(gen.WORKLOADS["c1"], seed=77), 0, 100_000)]:
        host = gen.generate(w, start=start, count=count)
        out = torch.empty(count * 109, dtype=torch.uint8, device="cuda:0")
        ctx.generate_device(w, start, count, out.data_ptr())
        got = out.cpu().numpy()
        want = host.view(np.uint8).reshape(-1)
        d = np.nonzero(got != want)[0]
        assert d.size == 0, f"{w.name}: {d.size} bytes differ, first at record {d[0] // 109} byte {d[0] % 109}"


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


def test_group_order_is_libstdcxx_sort_for_every_size_and_pattern(ctx):
    """K5b alone through rk_sort_members (sort_groups as a function of its arguments): groups of every size class (<= 16
    stable, 17..128 and 129..1024 by one warp, > 1024 split in global memory) with keys that are random, heavily tied,
    constant, sorted, reversed, organ-pipe and median-of-three killers (depth limit -> heap sort) must come out in the
    order std::sort leaves them (oracle: rko_std_sort_by_key runs the real std::sort)."""
    rng = np.random.default_rng(5)
    sizes = list(range(1, 40)) + [63, 64, 65, 100, 127, 128, 129, 130, 200, 255, 256, 257, 500, 1000, 1023, 1024, 1025, 1026,
                                   1500, 2047, 2048, 2049, 3000, 5000, 9000, 20000]
    patterns = {
        "random": lambda n: rng.integers(0, 1 << 30, n),
        "ties8": lambda n: rng.integers(0, 8, n),
        "ties_sqrt": lambda n: rng.integers(0, max(2, int(n ** 0.5)), n),
        "constant": lambda n: np.full(n, 7),
        "sorted": lambda n: np.arange(n),
        "reversed": lambda n: np.arange(n)[::-1].copy(),
        "organ": lambda n: np.minimum(np.arange(n), np.arange(n)[::-1]),
        "killer": _killer,
        "sorted_ties": lambda n: np.arange(n) // 3,
    }
    hs, gids = [], []
    g = 0
    for name, fn in patterns.items():
        for n in sizes:
            hs.append(np.asarray(fn(n), dtype=np.int64))
            gids.append(np.full(n, g, np.int64))
            g += 1
    h64 = np.concatenate(hs).astype(np.uint64)
    gid = np.concatenate(gids).astype(np.uint32)
    # h = |y - d|: half of the members get their key from above the table value, half from below
    d = rng.integers(1 << 30, 1 << 31, h64.shape[0]).astype(np.uint64)
    y = np.where(rng.integers(0, 2, h64.shape[0]) == 0, d + h64, d - h64)
    perm = ctx.sort_members(gid, y, d)
    pos = 0
    for hh in hs:
        n = hh.shape[0]
        idx = np.arange(pos, pos + n, dtype=np.uint32)
        want = O.std_sort_by_key(idx, h64) if n > 1 else idx
        msg = first_diff(perm[pos:pos + n], want)
        assert msg is None, f"group of {n} at {pos}: {msg}"
        pos += n


def test_packed_ingest_equals_record_ingest(ctx, fuzz_cases, tmp_path):
    """rk_load_packed (33 B per fragment: what the CLI sends) must give the arrays AND the output text of rk_load_aos"""
    from dataclasses import replace
    cases = [(gen.generate(w), w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio) for w in (
        gen.scaled(gen.WORKLOADS["c2"], 200_003), replace(gen.WORKLOADS["c1"], n=60_000, lx=400_000, ly=300_000, families=40, p_rep=0.6, seed=31))]
    for c in fuzz_cases[::5]:
        inp = tmp_path / "in.csv"
        inp.write_text(c["csv"], newline="")
        rec, lx1, ly1, _ = O.load_csv(str(inp))
        cases.append((rec, lx1, ly1, c["len_ratio"], c["pos_ratio"]))
    for rec, lx1, ly1, lr, pr in cases:
        ctx.load(rec, lx1, ly1)
        a = ctx.group(lr, pr)
        text_a = ctx.format_lines()
        st = ctx.load_packed(*capi.pack_records(rec), lx1, ly1)
        assert st.n_loaded == rec.shape[0] and st.n_kept == a.n_kept
        b = ctx.group(lr, pr)
        for f in ("order", "gid", "repval"):
            assert_same(f, getattr(b, f), getattr(a, f))
        assert_same("identity", b.identity.view(np.uint32), a.identity.view(np.uint32))
        assert ctx.format_lines() == text_a
        # without the output-only array the grouping still works and the formatter says why it cannot
        key4, strand, _ = capi.pack_records(rec)
        ctx.load_packed(key4, strand, None, lx1, ly1)
        assert_same("order (no rest4)", ctx.group(lr, pr).order, a.order)
        if a.n_kept:
            with pytest.raises(capi.RkError):
                ctx.format_lines()


@pytest.mark.parametrize("wl", ["c1", "dense", "c3"])
def test_group_statistics_match_oracle_reduction(ctx, wl):
    """K8 (north_star kernel 5): every field bit for bit against the exact evaluation of its definition over the
    reference's groups."""
    from dataclasses import replace
    w = {"c1": gen.WORKLOADS["c1"],
         "dense": replace(gen.WORKLOADS["c1"], n=60_000, lx=400_000, ly=300_000, families=40, p_rep=0.6, seed=31),
         "c3": gen.scaled(gen.WORKLOADS["c3"], 300_000)}[wl]
    rec = gen.generate(w)
    res, g = check_against_oracle(ctx, rec, w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio, stages=False)
    got = ctx.group_statistics()
    want = O.group_statistics(rec, g)
    assert got.shape[0] == g.n_groups
    for f in got.dtype.names:
        assert_same(f, got[f].view(np.uint64) if got[f].dtype == np.float64 else got[f],
                    want[f].view(np.uint64) if want[f].dtype == np.float64 else want[f])
    assert got["count"].sum() == g.n_kept and got["count"].max() > 16


def test_two_giant_families_small_input(ctx):
    """60k fragments, 90 % of them in two repeat families: segments and groups of tens of thousands of members on a
    small input (tier 2 of K3, the giant-group path of K5b) — every stage against the oracle, and the device text."""
    from dataclasses import replace
    w = replace(gen.scaled(gen.WORKLOADS["c3"], 60_000), families=2)
    rec = gen.generate(w)
    res, g = check_against_oracle(ctx, rec, w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio)
    assert np.bincount(res.gid).max() > 1024
    g.order, g.out_gid, g.repval, g.identity = res.order, res.gid, res.repval, res.identity
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        O.write_output(os.path.join(d, "o.csv"), b"", rec, g)
        assert open(os.path.join(d, "o.csv"), "rb").read() == ctx.format_lines()


def test_config4_shape_dense_y_axis(ctx):
    """BASELINE config 4 at 1/50 of its size (same densities): a 1.45 Gbp concatenation of contigs against a 150 Mbp
    sequence puts ~17 fragments per strand into every Y bucket, so most Y segments exceed 32 fragments (tier 2)."""
    w = gen.scaled(gen.WORKLOADS["c4"], 1_000_000)
    rec = gen.generate(w)
    check_against_oracle(ctx, rec, w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio)
