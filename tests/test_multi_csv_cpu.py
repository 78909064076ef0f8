"""multi.csv_slice_bounds: the byte range of a GECKO CSV file one process loads with rk_dist_load_csv, by the cut rule of
rk_multi_load_csv (one byte past the first newline at or after body byte bytes * r / world).  No GPU."""
import pytest

from repkiller_b200 import multi


def _cuts(body: bytes, world: int):
    """the rule restated over the body in memory"""
    cuts = [0]
    for r in range(1, world):
        a = len(body) * r // world
        nl = body.find(b"\n", a)
        cuts.append(len(body) if nl < 0 else nl + 1)
    return cuts + [len(body)]


def _bounds(tmp_path, head: bytes, body: bytes, world: int, window: int = 1 << 16):
    p = tmp_path / "in.csv"
    p.write_bytes(head + body)
    return [multi.csv_slice_bounds(str(p), len(head), r, world, window) for r in range(world)]


@pytest.mark.parametrize("world", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("body", [
    b"",                                         # no rows at all
    b"Frag,1,2,3",                               # no newline
    b"Frag,1,2,3\n",                             # one row and the empty one after it
    b"a\nb\n",                                   # more ranks than rows
    b"\n" * 7,                                   # cuts that fall on a newline
    b"row one\nrow two is longer\nr3\n\nr5\r\nlast without newline",
    b"".join(b"Frag,%d,%d,0\n" % (i, i * 7) for i in range(1000)),
])
def test_bounds_follow_the_cut_rule(tmp_path, world, body):
    head = b"".join(b"header line %d\n" % i for i in range(16))
    got = _bounds(tmp_path, head, body, world)
    want = _cuts(body, world)
    assert got == [(len(head) + a, len(head) + b) for a, b in zip(want, want[1:])]
    # the slices tile the body, and every one but the last non-empty one ends with a newline
    assert b"".join(body[a - len(head):b - len(head)] for a, b in got) == body
    nonempty = [r for r, (a, b) in enumerate(got) if b > a]
    for r in nonempty[:-1]:
        assert body[got[r][1] - len(head) - 1:got[r][1] - len(head)] == b"\n"


def test_a_small_window_reads_on_to_the_newline(tmp_path):
    """a row longer than the window: the cut still falls after the row's newline"""
    body = b"x" * 5000 + b"\n" + b"y" * 3000 + b"\n" + b"z" * 10
    head = b"h\n" * 16
    assert _bounds(tmp_path, head, body, 3, window=64) == _bounds(tmp_path, head, body, 3)
    got = _bounds(tmp_path, head, body, 3, window=64)
    want = _cuts(body, 3)
    assert got == [(len(head) + a, len(head) + b) for a, b in zip(want, want[1:])]
