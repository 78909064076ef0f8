"""The oracle (oracle/rk_oracle.c) against the committed outputs of the reference itself (tests/golden)."""
import hashlib
import os

import numpy as np
import pytest

from oracle import oracle as O
from repkiller_b200 import gen


def _oracle_bytes(tmp_path, csv_text, lr, pr):
    inp = tmp_path / "in.csv"
    inp.write_text(csv_text, newline="")
    rec, lx1, ly1, hdr = O.load_csv(str(inp))
    g = O.group(rec, lx1, ly1, lr, pr)
    outp = tmp_path / "out.csv"
    O.write_output(str(outp), hdr, rec, g)
    return outp.read_bytes(), g


def test_fuzz_outputs_match_reference(tmp_path, fuzz_cases):
    assert len(fuzz_cases) >= 100
    for c in fuzz_cases:
        got, g = _oracle_bytes(tmp_path, c["csv"], c["len_ratio"], c["pos_ratio"])
        assert got == c["ref_out"].encode("latin1"), f"fuzz seed {c['seed']}"
        assert g.n_groups == c["n_groups"] and g.n_kept == c["n_kept"]


@pytest.mark.parametrize("name", ["c1", "c1_loose", "c3_small", "dense", "c2_small"])
def test_medium_md5_matches_reference(tmp_path, medium_cases, name):
    c = medium_cases[name]
    w = gen.Workload(**c["workload"])
    rec = gen.generate(w)
    assert hashlib.md5(rec.tobytes()).hexdigest() == c["records_md5"], "generator drifted from the committed fixtures"
    g = O.group(rec, w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio)
    assert g.n_groups == c["n_groups"]
    outp = tmp_path / "out.csv"
    from repkiller_b200.frags import make_header
    O.write_output(str(outp), make_header(w.lx, w.ly, w.n).encode(), rec, g)
    data = outp.read_bytes()
    assert len(data) == c["ref_bytes"]
    assert hashlib.md5(data).hexdigest() == c["ref_md5"]


def test_decomposition_invariants(medium_cases):
    """SURVEY.md §3.3: parent rank < own rank, gid = number of roots before the root, members in rank order."""
    w = gen.Workload(**medium_cases["c1"]["workload"])
    rec = gen.generate(w)
    g = O.group(rec, w.lx + 1, w.ly + 1, w.len_ratio, w.pos_ratio)
    r = np.arange(g.n_kept, dtype=np.int64)
    has = g.parent != O.NONE
    assert (g.parent[has].astype(np.int64) < r[has]).all()
    roots = ~has
    gid_of_root = np.cumsum(roots) - 1
    root = r.copy()
    for _ in range(64):
        p = g.parent[root]
        nxt = np.where(p != O.NONE, p, root)
        if (nxt == root).all():
            break
        root = nxt
    assert (gid_of_root[root] == g.gid).all()
    assert int(roots.sum()) == g.n_groups


@pytest.mark.skipif(not O.have_ref(), reason="needs the compiled original repkiller in oracle/_ref; its output on this "
                                                "workload is not stored in tests/golden")
def test_oracle_vs_live_reference(tmp_path):
    """When the compiled reference is present, run it live on a fresh workload the fixtures do not hold."""
    from dataclasses import replace
    w = replace(gen.WORKLOADS["c1"], n=50_000, seed=99, p_rep=0.5, families=30)
    rec = gen.generate(w)
    inp = tmp_path / "in.csv"
    O.write_input_csv(str(inp), rec, w.lx, w.ly)
    ref_out = tmp_path / "ref.out"
    O.run_ref(str(inp), str(ref_out), w.len_ratio, w.pos_ratio)
    rec2, lx1, ly1, hdr = O.load_csv(str(inp))
    assert rec2.tobytes() == rec.tobytes()
    g = O.group(rec2, lx1, ly1, w.len_ratio, w.pos_ratio)
    out = tmp_path / "orc.out"
    O.write_output(str(out), hdr, rec2, g)
    assert out.read_bytes() == ref_out.read_bytes()
