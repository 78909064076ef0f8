"""The output side of one comparison partitioned over several ranks (RK_F_LINE_RECORDS): every rank formats the text of its
own output lines (K6, rk_dist_format_lines / rk_multi_format_lines) and reduces its own groups (K8,
rk_dist_group_statistics / rk_multi_group_statistics) from line rows that the grouping brought to it.  The text must be
byte for byte what one GPU writes and what the oracle's writer writes; the statistics must be one GPU's.
  * ranks as threads of one process on one device (capi.Multi([0] * k)), as in test_gpu_multi.py;
  * rk_dist_* with one process per GPU over NCCL where the box has the GPUs (2, 4, 8);
  * the CLI under RK_DEVICES, which now writes through the device writer unless RK_LEGACY_WRITER=1.
The two tests without the gpu mark check the exported symbols and the flag bits."""
import ctypes as C
import hashlib
import os
import re
import socket
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from dataclasses import replace
from functools import lru_cache

import numpy as np
import pytest

from oracle import oracle as O
from repkiller_b200 import capi, gen, multi

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "repkiller_b200", "bin", "repkiller")
RK_ERR_STATE = -4
NEW_SYMBOLS = ["rk_dist_format_lines", "rk_dist_group_statistics", "rk_multi_format_lines", "rk_multi_group_statistics"]


def _workload(name):  # the workloads of test_gpu_multi.py
    if name == "dense":
        return replace(gen.WORKLOADS["c1"], n=60_000, lx=400_000, ly=300_000, families=40, p_rep=0.6, seed=31)
    if name == "tiny":
        return replace(gen.WORKLOADS["c1"], n=3_000, lx=30_000, ly=25_000, families=12, p_rep=0.6, seed=21)
    if name == "c3":
        return gen.scaled(gen.WORKLOADS["c3"], 200_000)
    if name == "c2_6m":
        return gen.scaled(gen.WORKLOADS["c2"], 6_000_000)
    return gen.scaled(gen.WORKLOADS["c2"], 300_000)


def _oracle_body(rec, g, tmp_dir):
    """the lines the oracle's writer writes (no header)"""
    path = os.path.join(tmp_dir, "oracle_body.csv")
    O.write_output(path, b"", rec, g)
    with open(path, "rb") as f:
        body = f.read()
    os.remove(path)
    return body


@lru_cache(maxsize=2)
def _case(wl, len_ratio=None, pos_ratio=None):
    """(workload, records, oracle groups, oracle text, one-GPU device text and statistics) of one comparison"""
    import tempfile
    w = _workload(wl)
    lr, pr = (w.len_ratio, w.pos_ratio) if len_ratio is None else (len_ratio, pos_ratio)
    rec = gen.generate(w)
    g = O.group(rec, w.lx + 1, w.ly + 1, lr, pr)
    with tempfile.TemporaryDirectory() as d:
        body = _oracle_body(rec, g, d)
    with capi.Context(0) as ctx:
        ctx.load(rec, w.lx + 1, w.ly + 1)
        ctx.group(lr, pr)
        one = ctx.format_lines()
        stats = ctx.group_statistics()
    return w, rec, g, body, one, stats


def _assert_same(res, g):
    assert res.n_kept == g.n_kept and res.n_groups == g.n_groups, (res.n_kept, g.n_kept, res.n_groups, g.n_groups)
    for name, got, want in (("order", res.order, g.order), ("gid", res.gid, g.out_gid), ("repval", res.repval, g.repval),
                            ("identity", res.identity.view(np.uint32), g.identity.view(np.uint32))):
        d = np.nonzero(got != want)[0]
        assert d.size == 0, f"{name}: {d.size} differences, first at {d[:5]}"


def _first_diff(a: bytes, b: bytes) -> str:
    i = next((k for k in range(min(len(a), len(b))) if a[k] != b[k]), min(len(a), len(b)))
    return f"{len(a)} vs {len(b)} bytes, first difference at byte {i}: {a[max(0, i - 60):i + 60]!r} vs {b[max(0, i - 60):i + 60]!r}"


def _chunkings(total, offsets):
    """two ways to cut lines 0..total into chunks: (a) at every rank boundary b: [b-1, b], [b, b] (empty), [b, b+1], with
    one-line chunks; (b) chunks that cross the rank boundaries (cut halfway between them)"""
    bounds = sorted(set(o for o in offsets if 0 < o < total))
    pts = sorted(set([0, total] + [min(max(b + d, 0), total) for b in bounds for d in (-1, 0, 1)]))
    a = []
    for lo, hi in zip(pts, pts[1:]):
        a.append((lo, hi))
        if lo in bounds:
            a.append((lo, lo))
    mids = [0] + [(x + y) // 2 for x, y in zip([0] + bounds, bounds + [total])] + [total]
    b = [(lo, hi) for lo, hi in zip(mids, mids[1:])]
    return a, b


def _rank_handles(m):
    """the rk_ctx of every rank of a capi.Multi"""
    L = m._L
    return [L.rk_multi_ctx(m._h, r) for r in range(m.n)]


def _dist_text(L, h, first, count):
    t = capi._Text()
    rc = L.rk_dist_format_lines(h, first, count, C.byref(t))
    return rc, (C.string_at(t.text, t.n_bytes) if rc == 0 and t.n_bytes else b"")


# ---- 1. text parity, ranks as threads on one GPU ---------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("world,wl", [(k, wl) for wl in ("dense", "tiny", "c2", "c3") for k in (1, 2, 3, 5, 8)] + [(3, "c2_6m")])
def test_text_equals_one_gpu_and_oracle(world, wl):
    w, rec, g, body, one, _ = _case(wl)
    assert one == body, "one GPU: " + _first_diff(one, body)
    with capi.Multi([0] * world) as m:
        m.load(rec, w.lx + 1, w.ly + 1)
        _assert_same(m.group(w.len_ratio, w.pos_ratio, line_records=True), g)
        text = m.format_lines()
        assert text == one, _first_diff(text, one)
        offsets = [m.info(r)["line_offset"] for r in range(world)]
        for chunks in _chunkings(g.n_kept, offsets):
            parts = [m.format_lines(lo, hi - lo) for lo, hi in chunks]
            assert all(p == b"" for (lo, hi), p in zip(chunks, parts) if lo == hi)
            assert b"".join(parts) == text, chunks
        # every rank's own lines, local indices
        L, hs = m._L, _rank_handles(m)
        infos = [m.info(r) for r in range(world)]
        for r in range(world):
            rc, t = _dist_text(L, hs[r], 0, infos[r]["n_lines"])
            assert rc == 0, L.rk_last_error(hs[r])
            lo = infos[r]["line_offset"]
            assert t == m.format_lines(lo, infos[r]["n_lines"])


# ---- 2. 64-bit fields survive the row --------------------------------------------------------------------------------
@gpu
def test_fuzz_inputs_two_and_three_ranks(fuzz_cases, tmp_path):
    """the adversarial CSV inputs of the golden set: header + device text over 2 and 3 ranks == the reference's bytes"""
    done = 0
    with capi.Multi([0, 0]) as m2, capi.Multi([0, 0, 0]) as m3:
        for c in fuzz_cases[::2]:
            inp = tmp_path / "in.csv"
            inp.write_text(c["csv"], newline="")
            rec, lx1, ly1, hdr = O.load_csv(str(inp))
            if rec.shape[0] == 0:
                continue
            try:
                O.group(rec, lx1, ly1, c["len_ratio"], c["pos_ratio"])
            except ValueError:
                continue   # input the reference itself cannot process
            for m in (m2, m3):
                try:
                    m.load(rec, lx1, ly1)
                except capi.RkError as e:
                    assert e.code == -3, e
                    break
                m.group(c["len_ratio"], c["pos_ratio"], line_records=True)
                assert hdr + m.format_lines() == c["ref_out"].encode("latin1"), f"fuzz seed {c['seed']}, {m.n} ranks"
            else:
                done += 1
    assert done > 20


@gpu
@pytest.mark.parametrize("world", [2, 3])
def test_values_beyond_32_bits(world, tmp_path):
    """xEnd, yEnd, score and ident of 40 bits (printed, never used for grouping) come out digit for digit"""
    w = gen.scaled(gen.WORKLOADS["c1"], 20_000)
    rec = gen.generate(w)
    for f, step in (("xEnd", 5), ("yEnd", 11), ("score", 7), ("ident", 3)):
        rec[f][::step] = (1 << 40) + np.arange(rec[::step].shape[0], dtype=np.uint64) * 977
    g = O.group(rec, w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio)
    body = _oracle_body(rec, g, str(tmp_path))
    assert b"1099511627776" in body
    with capi.Multi([0] * world) as m:
        m.load(rec, w.lx + 1, w.ly + 1)
        _assert_same(m.group(w.len_ratio, w.pos_ratio, line_records=True), g)
        text = m.format_lines()
    assert text == body, _first_diff(text, body)


# ---- 3. statistics parity --------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("world", [1, 3, 8])
@pytest.mark.parametrize("wl", ["dense", "c2", "c3"])
def test_statistics_equal_one_gpu(world, wl):
    w, rec, g, _, _, want = _case(wl)
    with capi.Multi([0] * world) as m:
        m.load(rec, w.lx + 1, w.ly + 1)
        res = m.group(w.len_ratio, w.pos_ratio, line_records=True)
        got = m.group_statistics()
        assert got.shape[0] == g.n_groups == want.shape[0]
        for f in ("count", "x_lo", "x_hi", "y_lo", "y_hi", "first_line"):
            d = np.nonzero(got[f] != want[f])[0]
            assert d.size == 0, f"{f}: {d.size} differences, first at {d[:5]}"
        for f in ("mean_identity", "multiplicity"):
            rel = np.abs(got[f] - want[f]) / np.maximum(np.abs(want[f]), 1e-300)
            assert rel.max() <= 1e-6, (f, float(rel.max()))   # the tolerance of the one-GPU statistics test
        # per rank: its own groups, from the gid of its first line on; the ranks' ranges tile [0, n_groups)
        L, hs = m._L, _rank_handles(m)
        run = 0
        for r in range(world):
            info = m.info(r)
            fg, ng = C.c_uint64(), C.c_uint64()
            hp = C.c_void_p()
            assert L.rk_dist_group_statistics(hs[r], capi.F_HOST_RESULT, C.byref(hp), None, C.byref(fg), C.byref(ng)) == 0
            if info["n_lines"]:
                assert fg.value == res.gid[info["line_offset"]] == run, (r, fg.value, run)
                part = capi._stats_array(hp.value, ng.value)
                assert part.tobytes() == got[fg.value:fg.value + ng.value].tobytes()
            else:
                assert ng.value == 0
            run += ng.value
        assert run == g.n_groups


# ---- 4. lifetimes and the flag ---------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("world", [2, 3])
def test_rows_follow_every_grouping_of_a_load(world, tmp_path):
    """three ratio pairs on one load: the line rows reuse regions the load wrote, and the later groupings must not need them"""
    w = _workload("dense")
    rec = gen.generate(w)
    with capi.Multi([0] * world) as m:
        m.load(rec, w.lx + 1, w.ly + 1)
        for lr, pr in ((w.len_ratio, w.pos_ratio), (0.5, 0.5), (0.2, 0.9)):
            g = O.group(rec, w.lx + 1, w.ly + 1, lr, pr)
            _assert_same(m.group(lr, pr, line_records=True), g)
            text = m.format_lines()
            body = _oracle_body(rec, g, str(tmp_path))
            assert text == body, (lr, pr, _first_diff(text, body))


@gpu
def test_the_flag_changes_no_result_and_is_needed():
    w = _workload("c2")
    rec = gen.generate(w)
    with capi.Multi([0, 0, 0]) as m:
        m.load(rec, w.lx + 1, w.ly + 1)
        with_rows = m.group(w.len_ratio, w.pos_ratio, line_records=True)
        infos_with = [m.info(r) for r in range(3)]
        plain = m.group(w.len_ratio, w.pos_ratio)
        for f in ("order", "gid", "repval", "identity"):
            assert getattr(with_rows, f).tobytes() == getattr(plain, f).tobytes(), f
        assert with_rows.n_groups == plain.n_groups
        for r in range(3):
            a, b = infos_with[r], m.info(r)
            assert {k: v for k, v in a.items() if k != "bytes_sent"} == {k: v for k, v in b.items() if k != "bytes_sent"}
        # after a grouping without the flag there are no line rows: every rank refuses
        with pytest.raises(capi.RkError) as e:
            m.format_lines()
        assert e.value.code == RK_ERR_STATE
        with pytest.raises(capi.RkError) as e:
            m.group_statistics()
        assert e.value.code == RK_ERR_STATE
        L, hs = m._L, _rank_handles(m)
        for r in range(3):
            rc, _ = _dist_text(L, hs[r], 0, 0)
            assert rc == RK_ERR_STATE, r
            assert L.rk_dist_group_statistics(hs[r], 0, None, None, None, None) == RK_ERR_STATE, r


@gpu
@pytest.mark.parametrize("world", [2, 3])
def test_device_records_kept_resident(world):
    """rk_dist_load_aos from DEVICE slices (the rows are read from the caller's memory at grouping time) gives the text of
    host input; the ranks are the threads of a Multi, each calling rk_dist_* on its own context"""
    import torch
    w, rec, g, body, _, _ = _case("dense")
    dev = torch.from_numpy(np.ascontiguousarray(rec).view(np.uint8).reshape(-1).copy()).cuda()
    torch.cuda.synchronize()
    with capi.Multi([0] * world) as m:
        m.load(rec, w.lx + 1, w.ly + 1)   # sizes the ranks' buffers and maps them into each other
        L, hs = m._L, _rank_handles(m)
        bounds = [multi.slice_bounds(w.n, r, world) for r in range(world)]
        st = [capi._LoadStats() for _ in range(world)]
        res = [capi._Result() for _ in range(world)]
        info = [capi._DistInfo() for _ in range(world)]
        with ThreadPoolExecutor(world) as ex:
            rcs = list(ex.map(lambda r: L.rk_dist_load_aos(hs[r], C.c_void_p(dev.data_ptr() + bounds[r][0] * 109),
                                                             bounds[r][1] - bounds[r][0], bounds[r][0], w.lx + 1, w.ly + 1, 0,
                                                             C.byref(st[r])), range(world)))
            assert rcs == [0] * world, [L.rk_last_error(h) for h in hs]
            rcs = list(ex.map(lambda r: L.rk_dist_group(hs[r], w.len_ratio, w.pos_ratio, capi.F_LINE_RECORDS, C.byref(res[r]),
                                                         C.byref(info[r])), range(world)))
            assert rcs == [0] * world, [L.rk_last_error(h) for h in hs]
        parts = []
        for r in range(world):
            rc, t = _dist_text(L, hs[r], 0, info[r].n_lines)
            assert rc == 0, L.rk_last_error(hs[r])
            parts.append(t)
    assert [i.line_offset for i in info] == list(np.cumsum([0] + [i.n_lines for i in info[:-1]]))
    text = b"".join(parts)
    assert text == body, _first_diff(text, body)
    del dev


@gpu
def test_line_records_need_slices_in_rank_order():
    """the rank that loaded a record is found by the slices' file offsets: slices that overlap (every rank says its slice
    starts at record 0) are refused with RK_ERR_ARG by every rank, before any collective step; grouping without the flag
    still runs"""
    w, rec, _, _, _, _ = _case("tiny")
    world = 3
    with capi.Multi([0] * world) as m:
        m.load(rec, w.lx + 1, w.ly + 1)
        L, hs = m._L, _rank_handles(m)
        bounds = [multi.slice_bounds(w.n, r, world) for r in range(world)]
        host = np.ascontiguousarray(rec)
        st = [capi._LoadStats() for _ in range(world)]
        res = [capi._Result() for _ in range(world)]
        with ThreadPoolExecutor(world) as ex:
            rcs = list(ex.map(lambda r: L.rk_dist_load_aos(hs[r], C.c_void_p(host.ctypes.data + bounds[r][0] * 109), bounds[r][1] - bounds[r][0],
                                                             0, w.lx + 1, w.ly + 1, 0, C.byref(st[r])), range(world)))
            assert rcs == [0] * world, [L.rk_last_error(h) for h in hs]
            rcs = list(ex.map(lambda r: L.rk_dist_group(hs[r], w.len_ratio, w.pos_ratio, capi.F_LINE_RECORDS, C.byref(res[r]), None),
                              range(world)))
            assert rcs == [-2] * world, [L.rk_last_error(h) for h in hs]
            assert b"rank order" in L.rk_last_error(hs[0])
            rcs = list(ex.map(lambda r: L.rk_dist_group(hs[r], w.len_ratio, w.pos_ratio, 0, C.byref(res[r]), None), range(world)))
            assert rcs == [0] * world, [L.rk_last_error(h) for h in hs]


# ---- 5. capacity -----------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("world,wl", [(8, "c2"), (3, "dense"), (2, "tiny")])
def test_rows_fit_a_tight_line_capacity(monkeypatch, world, wl):
    """RK_DIST_LINE_CAP as in test_output_ranges_respect_the_row_capacity: the fullest rank holds about as many lines as the
    bound allows, and its rows (64 B per line in the 72 B per row the load used) give the right text"""
    w, rec, g, body, _, _ = _case(wl)
    cap = -(-g.n_kept // world)
    cap += cap // 8 + 64
    monkeypatch.setenv("RK_DIST_LINE_CAP", str(cap))
    with capi.Multi([0] * world) as m:
        m.load(rec, w.lx + 1, w.ly + 1)
        _assert_same(m.group(w.len_ratio, w.pos_ratio, line_records=True), g)
        lines = [m.info(r)["n_lines"] for r in range(world)]
        text = m.format_lines()
    assert max(lines) <= cap and max(lines) > cap // 2, (lines, cap)
    assert text == body, _first_diff(text, body)


# ---- 6. the CLI ------------------------------------------------------------------------------------------------------
def _cli(inp, outp, lr, pr, **env):
    return subprocess.run([CLI, str(inp), str(outp), lr, pr], capture_output=True, env=dict(os.environ, RK_DEVICES="0,0,0", **env))


@gpu
def test_cli_over_several_ranks_both_writers(tmp_path, medium_cases):
    c = medium_cases["c1"]
    w = gen.Workload(**c["workload"])
    inp = tmp_path / "c1.csv"
    O.write_input_csv(str(inp), gen.generate(w), w.lx, w.ly)
    for env, writer in (({}, "device"), ({"RK_LEGACY_WRITER": "1"}, "host")):
        outp = tmp_path / f"out_{writer}.csv"
        p = _cli(inp, outp, "0.05", "0.05", RK_TIMING="1", **env)
        assert p.returncode == 0, p.stderr
        assert hashlib.md5(outp.read_bytes()).hexdigest() == c["ref_md5"], writer
        lines = [ln for ln in p.stderr.decode().splitlines() if "len_ratio=" in ln]
        assert len(lines) == 1 and f" writer={writer}" in lines[0], p.stderr


@gpu
def test_cli_over_several_ranks_fuzz(tmp_path, fuzz_cases):
    """device writer and host writer over 3 ranks: the same exit status and, where the run succeeds, the reference's bytes"""
    done = 0
    for c in fuzz_cases[::6]:
        inp = tmp_path / "in.csv"
        inp.write_text(c["csv"], newline="")
        lr, pr = repr(c["len_ratio"]), repr(c["pos_ratio"])
        dev, host = _cli(inp, tmp_path / "dev.csv", lr, pr), _cli(inp, tmp_path / "host.csv", lr, pr, RK_LEGACY_WRITER="1")
        assert dev.returncode == host.returncode, (c["seed"], dev.stderr, host.stderr)
        if dev.returncode == 0:
            assert (tmp_path / "dev.csv").read_bytes() == c["ref_out"].encode("latin1"), f"fuzz seed {c['seed']}"
            done += 1
    assert done > 10


# ---- 7. one process per GPU over NCCL --------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, wl, out_dir):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(rank)
    w = _workload(wl)
    lo, hi = multi.slice_bounds(w.n, rank, world)
    rec = gen.generate(w, start=lo, count=hi - lo)
    ctx = capi.Context(rank)
    multi.bootstrap(ctx, multi.default_capacity(w.n // world + 16))
    # odd ranks hand in device memory (kept resident until the text is formatted), even ranks host memory
    host = np.ascontiguousarray(rec)
    dev = torch.from_numpy(host.view(np.uint8).reshape(-1).copy()).cuda() if rank % 2 else None
    torch.cuda.synchronize()
    ctx.dist_load(dev.data_ptr() if dev is not None else host.ctypes.data, hi - lo, lo, w.lx + 1, w.ly + 1)
    res, info = ctx.dist_group(w.len_ratio, w.pos_ratio, line_records=True)
    text = ctx.dist_format_lines()
    first_gid, stats = ctx.dist_group_statistics()
    with open(os.path.join(out_dir, f"r{rank}.txt"), "wb") as f:
        f.write(text)
    np.savez(os.path.join(out_dir, f"r{rank}.npz"), first_gid=first_gid, stats=stats, line_offset=info["line_offset"],
             n_lines=info["n_lines"], gid0=res.gid[0] if res.n_kept else -1)
    dist.barrier()
    ctx.close()
    dist.destroy_process_group()


@gpu
@pytest.mark.parametrize("world", [2, 4, 8])
def test_nccl_processes_format_their_lines(tmp_path, world):
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    import torch.multiprocessing as mp
    wl = "c2"
    mp.spawn(_worker, args=(world, _free_port(), wl, str(tmp_path)), nprocs=world, join=True)
    _, _, g, body, one, want = _case(wl)
    text = b"".join(open(os.path.join(tmp_path, f"r{r}.txt"), "rb").read() for r in range(world))
    assert text == one == body, _first_diff(text, body)
    parts = [np.load(os.path.join(tmp_path, f"r{r}.npz")) for r in range(world)]
    got = np.concatenate([p["stats"] for p in parts])
    assert got.shape[0] == g.n_groups
    for p in parts:
        if int(p["n_lines"]):
            assert int(p["first_gid"]) == int(p["gid0"])
    for f in ("count", "x_lo", "x_hi", "y_lo", "y_hi", "first_line"):
        assert np.array_equal(got[f], want[f]), f


# ---- 8. without a GPU ------------------------------------------------------------------------------------------------
def test_new_symbols_are_exported():
    lib = capi.LIB_PATH
    if not os.path.exists(lib):
        pytest.skip("library not built")
    out = subprocess.run(["nm", "-D", "--defined-only", lib], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r"\bT (rk_\w+)$", out, flags=re.M))
    for name in NEW_SYMBOLS:
        assert name in exported, name
        assert name in capi.SYMBOLS, name


def test_line_records_flag_is_a_bit_of_its_own():
    text = open(os.path.join(ROOT, "include", "rk_b200.h")).read()
    flags = {k: int(v, 0) for k, v in re.findall(r"#define (RK_F_\w+) (0x[0-9a-fA-F]+|\d+)u", text)}
    assert "RK_F_LINE_RECORDS" in flags and flags["RK_F_LINE_RECORDS"] == capi.F_LINE_RECORDS, flags
    seen = 0
    for v in flags.values():   # one bit each, no bit shared
        assert v and v & (v - 1) == 0, flags
        assert not seen & v, flags
        seen |= v
