"""Host-side logic of the drop-in that needs no GPU: the CSV row parser (readFragment rules) and the output
writer's line format, through the rk_hostcheck helper, against the oracle and the reference's golden bytes."""
import os
import subprocess

import numpy as np

from oracle import oracle as O
from repkiller_b200 import frags, gen
from repkiller_b200.frags import FRAG_DTYPE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOSTCHECK = os.path.join(ROOT, "repkiller_b200", "bin", "rk_hostcheck")
CLI = os.path.join(ROOT, "repkiller_b200", "bin", "repkiller")


def test_csv_parser_matches_oracle_on_fuzz(tmp_path, fuzz_cases):
    for c in fuzz_cases:
        inp = tmp_path / "in.csv"
        inp.write_text(c["csv"], newline="")
        out = tmp_path / "recs.bin"
        subprocess.check_call([HOSTCHECK, "parse", str(inp), str(out)])
        got = np.fromfile(out, dtype=FRAG_DTYPE)
        want, _, _, _ = O.load_csv(str(inp))
        assert got.tobytes() == want.tobytes(), f"fuzz seed {c['seed']}"


def test_parallel_parser_matches_oracle_for_any_thread_count(tmp_path, fuzz_cases):
    """FragmentsDatabase parses the rows with all host cores (ranges cut at row boundaries, concatenated in order): the
    records must be those of the row-by-row loop for every thread count, also when there are more threads than rows."""
    for c in fuzz_cases[::3]:
        inp = tmp_path / "in.csv"
        inp.write_text(c["csv"], newline="")
        want, _, _, _ = O.load_csv(str(inp))
        for threads in (1, 2, 3, 7, 16, 64):
            out = tmp_path / "recs.bin"
            subprocess.check_call([HOSTCHECK, "parse", str(inp), str(out), str(threads)])
            got = np.fromfile(out, dtype=FRAG_DTYPE)
            assert got.tobytes() == want.tobytes(), f"fuzz seed {c['seed']}, {threads} threads"


def test_float_fast_path_equals_strtof():
    """readFragment parses plain `digits[.digits]` similarity tokens without strtof; the result must be strtof's
    (correctly rounded float) on every token the fast path accepts."""
    p = subprocess.run([HOSTCHECK, "floatcheck", "3000000", "7"], capture_output=True, text=True)
    assert p.returncode == 0, p.stdout[-1500:]
    assert " 0 mismatches" in p.stdout


def test_writer_line_format_matches_reference(tmp_path, fuzz_cases):
    """Every line the reference wrote for a singleton group (repval 0) must be reproduced byte for byte by the
    host writer from the same record (float formatting of similarity and identity, '-nan', strand bytes)."""
    checked = 0
    for c in fuzz_cases[:60]:
        inp = tmp_path / "in.csv"
        inp.write_text(c["csv"], newline="")
        out = tmp_path / "w.csv"
        subprocess.check_call([HOSTCHECK, "write", str(inp), str(out)])
        mine = out.read_bytes().split(b"\n")
        ref = c["ref_out"].encode("latin1").split(b"\n")
        assert mine[:16] == ref[:16]                      # header echoed verbatim
        def key(line):                                    # everything but the gid and repval columns
            f = line.split(b",")
            return tuple(f[:6] + f[7:13])
        mine_keys = {key(l) for l in mine[16:] if l}
        for l in ref[16:]:
            if l:
                assert key(l) in mine_keys, (c["seed"], l)
                checked += 1
    assert checked > 1000


def test_cli_argument_errors():
    p = subprocess.run([CLI], capture_output=True)
    assert p.returncode == 1
    assert b"Invalid number of arguments." in p.stderr
    assert p.stdout.startswith(b"Repkiller v0.9.b\nUsage: ./repkiller <input_file_path> <output_file_path> <length_ratio> <position_ratio>\n")
    p = subprocess.run([CLI, "/nonexistent.csv", "/tmp/o.csv", "0.05", "0.05"], capture_output=True)
    assert p.returncode != 0 and b"Could not open input file /nonexistent.csv." in p.stderr


# ---- GECKO's binary container (SURVEY §8f N4; csrc/host/GeckoFrags.h) -- parity unpinned: the reference reads CSV only ----
def _binary_case(n=20_000, seed=5):
    from dataclasses import replace
    w = replace(gen.WORKLOADS["c1"], n=n, seed=seed)
    rec = gen.generate(w)
    rec["block"] = np.arange(n) % 7 - 3              # a signed field with both signs
    rec["strand"][::5] = b"r"
    return w, rec


def test_binary_file_loads_like_its_csv_rendering(tmp_path):
    """the definition of the binary route: the records a .frags file loads as are the records readFragment builds from the CSV
    rows printing the same values (ident from the similarity column, diag recomputed, seqX/seqY/evalue fixed)"""
    w, rec = _binary_case()
    rec["ident"] += 3                                  # the stored ident is NOT what loads (FragmentsDatabase.cpp:39)
    rec["seqX"], rec["seqY"] = 4, 9
    rec["evalue"] = np.frombuffer(bytes(range(16)), dtype="V16")[0]
    csv_path, bin_path = tmp_path / "in.csv", tmp_path / "in.frags"
    frags.write_csv(str(csv_path), rec, w.lx, w.ly)
    frags.write_gecko_binary(str(bin_path), rec, w.lx, w.ly)
    out_csv, out_bin = tmp_path / "csv.bin", tmp_path / "bin.bin"
    subprocess.check_call([HOSTCHECK, "parse", str(csv_path), str(out_csv)])
    p = subprocess.run([HOSTCHECK, "fragsbin", str(bin_path), str(out_bin)], capture_output=True, text=True, check=True)
    assert p.stdout.split() == [str(w.lx), str(w.ly), str(rec.shape[0])]
    from_csv = np.fromfile(out_csv, dtype=FRAG_DTYPE)
    from_bin = np.fromfile(out_bin, dtype=FRAG_DTYPE)
    assert from_csv.shape[0] == rec.shape[0]
    assert from_bin.tobytes() == from_csv.tobytes()
    # and the numpy statement of the same rule (used by the GPU tests)
    want, lx, ly = frags.gecko_binary_as_loaded(bin_path.read_bytes())
    assert (lx, ly) == (w.lx, w.ly) and want.tobytes() == from_bin.tobytes()


def test_binary_encode_is_the_inverse_of_decode(tmp_path):
    """rk_hostcheck tofrags (C++ encoder) and frags.write_gecko_binary (numpy) produce the same file from the same records"""
    w, rec = _binary_case(n=3_000, seed=9)
    loaded = rec.copy()
    loaded["ident"] = loaded["similarity"].astype(np.uint64)   # what the CSV parser makes of the records
    loaded["seqX"], loaded["seqY"] = 0, 1
    csv_path = tmp_path / "in.csv"
    frags.write_csv(str(csv_path), rec, w.lx, w.ly)
    out = tmp_path / "out.frags"
    subprocess.check_call([HOSTCHECK, "tofrags", str(csv_path), str(out)])
    assert out.read_bytes() == frags.records_to_gecko_binary(loaded, w.lx, w.ly)


def test_binary_layout_edge_cases(tmp_path):
    empty = tmp_path / "empty.frags"
    empty.write_bytes((1000).to_bytes(8, "big") + (2000).to_bytes(8, "big"))
    out = tmp_path / "o.bin"
    p = subprocess.run([HOSTCHECK, "fragsbin", str(empty), str(out)], capture_output=True, text=True, check=True)
    assert p.stdout.split() == ["1000", "2000", "0"] and out.read_bytes() == b""
    for bad in (b"", b"\0" * 15, b"\0" * (16 + 108), b"\0" * (16 + 110)):
        f = tmp_path / "bad.frags"
        f.write_bytes(bad)
        assert subprocess.run([HOSTCHECK, "fragsbin", str(f), str(out)]).returncode == 4
    # values beyond 32 bits and the extreme bit patterns survive the byte reversal
    rec = frags.empty_records(4)
    rec["xStart"] = [0, 1, 2**40 + 5, 2**63 - 1]
    rec["yStart"] = [2**33, 0, 7, 1]
    rec["length"] = [1, 2**32, 3, 4]
    rec["score"] = [2**64 - 1, 0, 1, 2]
    rec["block"] = [-(2**63), -1, 0, 2**63 - 1]
    rec["similarity"] = np.array([0.0, 99.99, 100.0, 1e-30], dtype=np.float32)
    rec["strand"] = [b"f", b"r", b"\xff", b"\x00"]
    f = tmp_path / "wide.frags"
    frags.write_gecko_binary(str(f), rec, 2**41, 2**35)
    p = subprocess.run([HOSTCHECK, "fragsbin", str(f), str(out)], capture_output=True, text=True, check=True)
    assert p.stdout.split() == [str(2**41), str(2**35), "4"]
    want, _, _ = frags.gecko_binary_as_loaded(f.read_bytes())
    assert np.fromfile(out, dtype=FRAG_DTYPE).tobytes() == want.tobytes()


def _ingest(path, tmp_path, threads=None, env=None):
    out, hdr = tmp_path / "ing.bin", tmp_path / "ing.hdr"
    cmd = [HOSTCHECK, "ingest", str(path), str(out), str(hdr)] + ([str(threads)] if threads else [])
    p = subprocess.run(cmd, capture_output=True, text=True, env=dict(os.environ, **(env or {})))
    if p.returncode:
        return p.returncode, None, None, None
    lx1, ly1, total, binary = (int(v) for v in p.stdout.split())
    return 0, np.fromfile(out, dtype=FRAG_DTYPE), hdr.read_bytes(), (lx1, ly1, total, binary)


def test_constructor_input_stage_csv_and_binary(tmp_path, fuzz_cases):
    """the device-free half of the FragmentsDatabase constructor on both containers: same records, same sequence lengths,
    a 16-line header either way; any thread count"""
    w, rec = _binary_case(n=50_000, seed=2)
    csv_path, bin_path = tmp_path / "in.csv", tmp_path / "in.frags"
    frags.write_csv(str(csv_path), rec, w.lx, w.ly)
    frags.write_gecko_binary(str(bin_path), rec, w.lx, w.ly)
    rc, from_csv, hdr_csv, info_csv = _ingest(csv_path, tmp_path)
    assert rc == 0 and info_csv == (w.lx + 1, w.ly + 1, w.n, 0)
    assert hdr_csv == frags.make_header(w.lx, w.ly, w.n).encode("latin1")
    want, _, _ = frags.gecko_binary_as_loaded(bin_path.read_bytes())
    assert from_csv.tobytes() == want.tobytes()
    for threads in (None, 1, 3, 7, 64):
        rc, from_bin, hdr_bin, info_bin = _ingest(bin_path, tmp_path, threads)
        assert rc == 0 and info_bin == (w.lx + 1, w.ly + 1, w.n, 1)
        assert from_bin.tobytes() == want.tobytes(), threads
        lines = hdr_bin.decode("latin1").split("\n")
        assert len(lines) == 17 and lines[16] == ""
        assert lines[6] == f"SeqX length : {w.lx}" and lines[7] == f"SeqY length : {w.ly}" and lines[12] == f"Total fragments : {w.n}"
        assert lines[14] == frags.HEADER_TEMPLATE.split("\n")[14]
    # the CSV route through the same entry still equals the row-by-row parser on the adversarial inputs
    for c in fuzz_cases[::10]:
        inp = tmp_path / "f.csv"
        inp.write_text(c["csv"], newline="")
        want_f, _, _, _ = O.load_csv(str(inp))
        rc, got, _, _ = _ingest(inp, tmp_path, 3)
        assert rc == 0 and got.tobytes() == want_f.tobytes(), c["seed"]


def test_input_format_detection(tmp_path):
    """binary only when the name says .frags AND the content has the layout AND starts with a zero byte; RK_INPUT_FORMAT decides
    otherwise; a file that claims to be binary and is not is an error, never a guess"""
    w, rec = _binary_case(n=500, seed=3)
    blob = frags.records_to_gecko_binary(rec, w.lx, w.ly)
    text = (frags.make_header(w.lx, w.ly, w.n) + frags.records_to_csv_rows(rec)).encode("latin1")
    want, _, _ = frags.gecko_binary_as_loaded(blob)
    (tmp_path / "a.frags").write_bytes(blob)
    (tmp_path / "a.dat").write_bytes(blob)
    (tmp_path / "csv_named.frags").write_bytes(text)
    (tmp_path / "short.frags").write_bytes(blob[:-1])
    rc, got, _, info = _ingest(tmp_path / "a.frags", tmp_path)
    assert rc == 0 and info[3] == 1 and got.tobytes() == want.tobytes()
    rc, got, _, info = _ingest(tmp_path / "a.dat", tmp_path)                  # not named .frags: read as the reference would
    assert rc == 0 and info[3] == 0 and got.shape[0] == 0
    rc, got, _, info = _ingest(tmp_path / "a.dat", tmp_path, env={"RK_INPUT_FORMAT": "frags"})
    assert rc == 0 and info[3] == 1 and got.tobytes() == want.tobytes()
    rc, got, _, info = _ingest(tmp_path / "csv_named.frags", tmp_path)        # a CSV under a .frags name stays a CSV
    assert rc == 0 and info[3] == 0 and got.tobytes() == want.tobytes()
    rc, got, _, info = _ingest(tmp_path / "short.frags", tmp_path)            # layout broken: CSV rules (nothing accepted)
    assert rc == 0 and info[3] == 0
    rc, _, _, _ = _ingest(tmp_path / "short.frags", tmp_path, env={"RK_INPUT_FORMAT": "frags"})
    assert rc == 4
    rc, got, _, info = _ingest(tmp_path / "a.frags", tmp_path, env={"RK_INPUT_FORMAT": "csv"})
    assert rc == 0 and info[3] == 0

