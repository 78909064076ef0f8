"""tests/native/database_glue_check.cpp: the FragmentsDatabase constructors linked against a recording stand-in for the
library (no GPU, nothing computed).  One run builds one database and prints the load call and what the database answers,
so two runs on the same file compare two routes.  The host parser's route must hand the library the same arrays for a CSV
and its .frags rendering; the device parser's route must hand rk_load_csv / rk_multi_load_csv exactly the bytes after the
16 header lines, the loaded lengths and the stated count, and answer like the host parser's route on the same file."""
import os
import subprocess

import numpy as np
import pytest

from repkiller_b200 import frags, gen
from test_host_cpu import _binary_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "repkiller_b200", "csrc", "host")
NOTHING_LIVE = "live ctx=0 multi=0 host=0"


def _fnv(b: bytes) -> str:
    h = 1469598103934665603
    for v in b:
        h = ((h ^ v) * 1099511628211) & ((1 << 64) - 1)
    return f"{h:016x}"


def _body(data: bytes) -> bytes:
    pos = 0
    for _ in range(16):
        nl = data.find(b"\n", pos)
        pos = len(data) if nl < 0 else nl + 1
    return data[pos:]


@pytest.fixture(scope="module")
def glue(tmp_path_factory):
    exe = tmp_path_factory.mktemp("glue") / "ingest_glue"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-I", os.path.join(ROOT, "include"), "-o", str(exe),
                           os.path.join(ROOT, "tests", "native", "database_glue_check.cpp"),
                           os.path.join(HOST, "FragmentsDatabase.cpp"), os.path.join(HOST, "GeckoFrags.cpp")])
    return str(exe)


def _run(exe, path, ranks=1, parser="host"):
    p = subprocess.run([exe, str(path), str(ranks), parser], capture_output=True, text=True)
    return p.returncode, p.stdout.strip().split("\n")


def _device_route_hands_the_body_and_equals_the_host_route(glue, tmp_path, fuzz_cases, ranks):
    w = gen.scaled(gen.WORKLOADS["c1"], 3_000)
    rec = gen.generate(w)
    csv_path = tmp_path / "in.csv"
    frags.write_csv(str(csv_path), rec, w.lx, w.ly)
    cases = [(csv_path, w.lx + 1, w.ly + 1, w.n)]
    for c in fuzz_cases[::12]:   # short rows, bad tokens, CRLF, odd headers
        p = tmp_path / f"f{c['seed']}.csv"
        p.write_text(c["csv"], newline="")
        cases.append((p, None, None, None))
    call_head = ["call", "rk_load_csv"] if ranks == 1 else ["call", "rk_multi_load_csv", f"ranks={ranks}"]
    for path, lx1, ly1, total in cases:
        rc, dev = _run(glue, path, ranks, "device")
        rc_host, host = _run(glue, path, ranks, "host")
        if rc or rc_host:   # the stated count is too small: both routes refuse alike and release what they made
            for r, out in ((rc, dev), (rc_host, host)):
                assert r == 1 and out[-2:] == ["exception: Unexpected number of fragments", NOTHING_LIVE], (path, out)
            continue
        body = _body(path.read_bytes())
        call = dev[0].split()
        assert call[:len(call_head) + 2] == call_head + [f"bytes={len(body)}", f"body={_fnv(body)}"], (path, dev[0])
        if lx1 is not None:
            assert call[len(call_head) + 2:] == [f"seqx_len={lx1}", f"seqy_len={ly1}", f"total_frags={total}"]
        if ranks > 1:
            assert host[0].startswith(f"call rk_multi_load_aos ranks={ranks} "), host
        facts_dev, facts_host = dev[1].split(), host[1].split()
        assert facts_dev[:-2] == facts_host[:-2], (path, dev, host)   # getA, total, sequences, lengths
        assert facts_dev[-2:] == ["parser=1", f"multi={int(ranks > 1)}"] and facts_host[-2:] == ["parser=0", f"multi={int(ranks > 1)}"]
        assert dev[2:] == host[2:], (path, dev, host)                 # records, buckets (one device), header, live objects
        assert len(dev) == (6 if ranks == 1 else 5) and dev[-1] == NOTHING_LIVE


def _device_route_refuses_more_rows_than_stated(glue, tmp_path, ranks):
    w = gen.scaled(gen.WORKLOADS["c1"], 500)
    rec = gen.generate(w)
    path = tmp_path / "short.csv"
    frags.write_csv(str(path), rec, w.lx, w.ly, total_frags=w.n - 1)
    rc, out = _run(glue, path, ranks, "device")
    assert rc == 1 and out[-2:] == ["exception: Unexpected number of fragments", NOTHING_LIVE], out
    frags.write_csv(str(path), rec, w.lx, w.ly, total_frags=w.n)
    rc, out = _run(glue, path, ranks, "device")
    assert rc == 0 and out[1].split()[1] == f"total={w.n}" and out[-1] == NOTHING_LIVE, out


def test_device_csv_constructor_hands_the_body_and_equals_the_host_route(glue, tmp_path, fuzz_cases):
    _device_route_hands_the_body_and_equals_the_host_route(glue, tmp_path, fuzz_cases, 1)   # rk_load_csv


def test_multi_csv_constructor_hands_the_body_and_equals_the_host_route(glue, tmp_path, fuzz_cases):
    _device_route_hands_the_body_and_equals_the_host_route(glue, tmp_path, fuzz_cases, 3)   # rk_multi_load_csv


def test_device_csv_constructor_refuses_more_rows_than_stated(glue, tmp_path):
    _device_route_refuses_more_rows_than_stated(glue, tmp_path, 1)


def test_multi_csv_constructor_refuses_more_rows_than_stated(glue, tmp_path):
    _device_route_refuses_more_rows_than_stated(glue, tmp_path, 3)


def test_constructor_hands_the_same_arrays_to_the_library_for_both_containers(glue, tmp_path):
    """CSV and .frags input must lead to the same load call — count, sequence lengths, compact arrays — and to the same
    records and accessors; wide values take the 109-byte route; several devices the partitioned one."""
    w, rec = _binary_case(n=4_000, seed=11)
    csv_path, bin_path = tmp_path / "in.csv", tmp_path / "in.frags"
    frags.write_csv(str(csv_path), rec, w.lx, w.ly)
    frags.write_gecko_binary(str(bin_path), rec, w.lx, w.ly)
    want, _, _ = frags.gecko_binary_as_loaded(bin_path.read_bytes())

    def run(path, *extra):
        rc, out = _run(glue, path, *extra)
        assert rc == 0, out
        return out

    a, b = run(csv_path), run(bin_path)
    assert a[:4] == b[:4] and a[5] == b[5]             # load call, accessors, records, buckets, live objects; only the header text differs
    key4 = np.stack([want["xStart"], want["yStart"], want["length"], want["ident"]], axis=1).astype(np.uint32)
    rest4 = np.stack([want["xEnd"].astype(np.uint32), want["yEnd"].astype(np.uint32), want["score"].astype(np.uint32),
                      want["similarity"].view(np.uint32)], axis=1)
    assert a[0] == (f"call rk_load_packed n={w.n} seqx_len={w.lx + 1} seqy_len={w.ly + 1} key4={_fnv(key4.tobytes())} "
                    f"strand={_fnv(want['strand'].tobytes())} rest4={_fnv(rest4.tobytes())}")
    assert a[1] == (f"getA={1 + (w.lx + 1) // 10} total={w.n} seqs=2 len0={w.lx + 1} len1={w.ly + 1} max={max(w.lx, w.ly) + 1} "
                    "parser=0 multi=0")
    assert a[2] == f"records={_fnv(want.tobytes())}"
    assert a[4].startswith("header_lines=16 ") and b[4].startswith("header_lines=16 ")
    assert a[5] == NOTHING_LIVE
    # several devices: the records go to the partitioned load
    m = run(bin_path, 3)
    assert m[0] == f"call rk_multi_load_aos ranks=3 n={w.n} seqx_len={w.lx + 1} seqy_len={w.ly + 1} records={_fnv(want.tobytes())}"
    # a value beyond 32 bits: the 109-byte records instead of the compact arrays
    rec["score"][7] = 2**40
    frags.write_gecko_binary(str(bin_path), rec, w.lx, w.ly)
    frags.write_csv(str(csv_path), rec, w.lx, w.ly)
    want, _, _ = frags.gecko_binary_as_loaded(bin_path.read_bytes())
    a, b = run(csv_path), run(bin_path)
    assert a[0] == b[0] == f"call rk_load_aos n={w.n} seqx_len={w.lx + 1} seqy_len={w.ly + 1} records={_fnv(want.tobytes())}"
    # "Total fragments" smaller than the accepted rows: the reference's exception (FragmentsDatabase.cpp:99)
    frags.write_csv(str(csv_path), rec, w.lx, w.ly, total_frags=w.n - 1)
    rc, out = _run(glue, csv_path)
    assert rc == 1 and out[-2:] == ["exception: Unexpected number of fragments", NOTHING_LIVE], out
