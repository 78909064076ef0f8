"""tests/native/multi_csv_glue_check.cpp: the FragmentsDatabase constructor that parses the CSV rows on several devices
(CsvOnDevice with a device list, host/FragmentsDatabaseMultiCsv.cpp) linked against a recording stand-in for the library
(no GPU).  It must hand rk_multi_load_csv exactly the bytes after the 16 header lines, the loaded lengths and the stated
count, and give the same records and accessors as the host parser's constructor for several devices on the same file."""
import os
import subprocess

import pytest

from repkiller_b200 import frags, gen

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "repkiller_b200", "csrc", "host")


def _fnv(b: bytes) -> str:
    h = 1469598103934665603
    for v in b:
        h = ((h ^ v) * 1099511628211) & ((1 << 64) - 1)
    return f"{h:016x}"


@pytest.fixture(scope="module")
def glue(tmp_path_factory):
    exe = tmp_path_factory.mktemp("glue") / "multi_csv_glue"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-I", os.path.join(ROOT, "include"), "-o", str(exe),
                           os.path.join(ROOT, "tests", "native", "multi_csv_glue_check.cpp"),
                           os.path.join(HOST, "FragmentsDatabase.cpp"), os.path.join(HOST, "FragmentsDatabaseMultiCsv.cpp"),
                           os.path.join(HOST, "GeckoFrags.cpp")])
    return str(exe)


def _run(exe, path, *extra):
    p = subprocess.run([exe, str(path), *extra], capture_output=True, text=True)
    return p.returncode, p.stdout.strip().split("\n")


def _body(data: bytes) -> bytes:
    pos = 0
    for _ in range(16):
        nl = data.find(b"\n", pos)
        pos = len(data) if nl < 0 else nl + 1
    return data[pos:]


def test_multi_csv_constructor_hands_the_body_and_equals_the_host_route(glue, tmp_path, fuzz_cases):
    w = gen.scaled(gen.WORKLOADS["c1"], 3_000)
    rec = gen.generate(w)
    csv_path = tmp_path / "in.csv"
    frags.write_csv(str(csv_path), rec, w.lx, w.ly)
    cases = [(csv_path, w.lx + 1, w.ly + 1, w.n)]
    for c in fuzz_cases[::12]:   # short rows, bad tokens, CRLF, odd headers
        p = tmp_path / f"f{c['seed']}.csv"
        p.write_text(c["csv"], newline="")
        cases.append((p, None, None, None))
    for path, lx1, ly1, total in cases:
        rc, out = _run(glue, path)
        if rc:   # the stated count is too small: both routes refuse alike
            assert out[-1] == "exception: Unexpected number of fragments", (path, out)
            continue
        body = _body(path.read_bytes())
        call = out[0].split()
        assert call[:4] == ["call", "rk_multi_load_csv", "ranks=3", f"bytes={len(body)}"], out[0]
        assert call[4] == f"body={_fnv(body)}", path
        if lx1 is not None:
            assert call[5:] == [f"seqx_len={lx1}", f"seqy_len={ly1}", f"total_frags={total}"]
        assert out[1].startswith("call rk_multi_load_aos ranks=3"), out   # (the host route's call)
        dev, host = out[2].split(), out[3].split()
        assert dev[0] == "device" and host[0] == "host" and dev[1:5] == host[1:5], (path, out)
        assert dev[5:] == ["parser=1", "multi=1"] and host[5:] == ["parser=0", "multi=1"]
        assert out[4].endswith("same_records=1 same_header=1"), (path, out)


def test_multi_csv_constructor_refuses_more_rows_than_stated(glue, tmp_path):
    w = gen.scaled(gen.WORKLOADS["c1"], 500)
    rec = gen.generate(w)
    path = tmp_path / "short.csv"
    frags.write_csv(str(path), rec, w.lx, w.ly, total_frags=w.n - 1)
    rc, out = _run(glue, path, "device")
    assert rc == 1 and out[-1] == "exception: Unexpected number of fragments"
    frags.write_csv(str(path), rec, w.lx, w.ly, total_frags=w.n)
    rc, out = _run(glue, path, "device")
    assert rc == 0 and out[-1] == f"device total={w.n}"
