"""TEST INFRASTRUCTURE — NOT part of the product path.

ctypes front end of the C restatement (oracle/rk_oracle.c) and a runner for the compiled reference
(oracle/_ref/repkiller_ref).  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
``--impl reference`` legs may import this module.
"""
from __future__ import annotations

import ctypes as C
import json
import os
import subprocess
from dataclasses import dataclass

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "_build", "librk_oracle.so")
REF_BIN = os.path.join(HERE, "_ref", "repkiller_ref")
NONE = 0xFFFFFFFF


def build(ref: bool = True) -> None:
    """Compile the C restatement and, when /root/reference is present, the reference behind ref_driver.cpp."""
    subprocess.check_call(["make", "-s", "-C", HERE, "lib"] + (["ref", "refbody"] if ref else []))


class _Result(C.Structure):
    _fields_ = [
        ("n_kept", C.c_uint64), ("n_groups", C.c_uint64), ("vsize", C.c_uint64),
        ("rank_fidx", C.POINTER(C.c_uint32)), ("xowner", C.POINTER(C.c_uint32)), ("yowner", C.POINTER(C.c_uint32)),
        ("parent", C.POINTER(C.c_uint32)), ("gid", C.POINTER(C.c_uint32)), ("h", C.POINTER(C.c_uint64)),
        ("order", C.POINTER(C.c_uint32)), ("out_gid", C.POINTER(C.c_uint32)), ("repval", C.POINTER(C.c_uint8)),
        ("identity", C.POINTER(C.c_float)), ("diag_func", C.POINTER(C.c_uint64)),
    ]


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            build(ref=False)
        L = C.CDLL(LIB_PATH)
        L.rko_parse_row.argtypes = [C.c_char_p, C.c_size_t, C.c_void_p]
        L.rko_parse_row.restype = C.c_int
        L.rko_load_csv.argtypes = [C.c_char_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64),
                                   C.POINTER(C.c_uint64), C.POINTER(C.c_void_p)]
        L.rko_load_csv.restype = C.c_int
        L.rko_group.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_double, C.c_double, C.c_int,
                                C.POINTER(_Result)]
        L.rko_group.restype = C.c_int
        L.rko_result_free.argtypes = [C.POINTER(_Result)]
        L.rko_write_output.argtypes = [C.c_char_p, C.c_char_p, C.c_void_p, C.POINTER(_Result)]
        L.rko_write_output.restype = C.c_int
        L.rko_write_input_csv.argtypes = [C.c_char_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64]
        L.rko_write_input_csv.restype = C.c_int
        L.rko_free.argtypes = [C.c_void_p]
        L.rko_std_sort_by_key.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
        _lib = L
    return _lib


@dataclass
class OracleGroups:
    n_kept: int
    n_groups: int
    vsize: int
    rank_fidx: np.ndarray
    xowner: np.ndarray
    yowner: np.ndarray
    parent: np.ndarray
    gid: np.ndarray
    h: np.ndarray
    order: np.ndarray
    out_gid: np.ndarray
    repval: np.ndarray
    identity: np.ndarray
    diag_func: np.ndarray | None


def _arr(ptr, n, dtype):
    if n == 0:
        return np.zeros(0, dtype=dtype)
    return np.ctypeslib.as_array(ptr, shape=(n,)).astype(dtype, copy=True)


def _frag_dtype():
    from repkiller_b200.frags import FRAG_DTYPE
    return FRAG_DTYPE


def load_csv(path: str):
    """(records, lx1, ly1, header) the way the reference's FragmentsDatabase loads them (lengths are header + 1)."""
    L = lib()
    recs, hdr = C.c_void_p(), C.c_void_p()
    n, lx1, ly1 = C.c_uint64(), C.c_uint64(), C.c_uint64()
    rc = L.rko_load_csv(path.encode(), C.byref(recs), C.byref(n), C.byref(lx1), C.byref(ly1), C.byref(hdr))
    if rc == -1:
        raise FileNotFoundError(path)
    dt = _frag_dtype()
    out = np.frombuffer(C.string_at(recs.value, n.value * dt.itemsize), dtype=dt).copy() if n.value else np.zeros(0, dt)
    header = C.string_at(hdr.value)
    L.rko_free(recs)
    L.rko_free(hdr)
    if rc == -2:
        raise RuntimeError("Unexpected number of fragments")
    return out, lx1.value, ly1.value, header


def group(records: np.ndarray, lx1: int, ly1: int, len_ratio: float, pos_ratio: float, want_diag: bool = False) -> OracleGroups:
    L = lib()
    rec = np.ascontiguousarray(records)
    assert rec.dtype.itemsize == 109
    r = _Result()
    rc = L.rko_group(rec.ctypes.data, rec.shape[0], lx1, ly1, len_ratio, pos_ratio, int(want_diag), C.byref(r))
    if rc:
        raise ValueError(f"rko_group failed: {rc}")
    m = r.n_kept
    out = OracleGroups(
        n_kept=m, n_groups=r.n_groups, vsize=r.vsize,
        rank_fidx=_arr(r.rank_fidx, m, np.uint32), xowner=_arr(r.xowner, m, np.uint32),
        yowner=_arr(r.yowner, m, np.uint32), parent=_arr(r.parent, m, np.uint32), gid=_arr(r.gid, m, np.uint32),
        h=_arr(r.h, m, np.uint64), order=_arr(r.order, m, np.uint32), out_gid=_arr(r.out_gid, m, np.uint32),
        repval=_arr(r.repval, m, np.uint8), identity=_arr(r.identity, m, np.float32),
        diag_func=_arr(r.diag_func, r.vsize - 1, np.uint64) if want_diag else None,
    )
    L.rko_result_free(C.byref(r))
    return out


def write_output(path: str, header: bytes, records: np.ndarray, g: OracleGroups) -> None:
    L = lib()
    r = _Result()
    r.n_kept = g.n_kept
    keep = [np.ascontiguousarray(g.order), np.ascontiguousarray(g.out_gid), np.ascontiguousarray(g.repval),
            np.ascontiguousarray(g.identity)]
    r.order = keep[0].ctypes.data_as(C.POINTER(C.c_uint32))
    r.out_gid = keep[1].ctypes.data_as(C.POINTER(C.c_uint32))
    r.repval = keep[2].ctypes.data_as(C.POINTER(C.c_uint8))
    r.identity = keep[3].ctypes.data_as(C.POINTER(C.c_float))
    rec = np.ascontiguousarray(records)
    if L.rko_write_output(path.encode(), header, rec.ctypes.data, C.byref(r)):
        raise OSError(f"cannot write {path}")


def write_input_csv(path: str, records: np.ndarray, lx_header: int, ly_header: int) -> None:
    rec = np.ascontiguousarray(records)
    if lib().rko_write_input_csv(path.encode(), rec.ctypes.data, rec.shape[0], lx_header, ly_header):
        raise OSError(f"cannot write {path}")


NAN_BITS = 0xFFF8000000000000   # the identity column's NaN (0xFFC00000) widened to binary64


def _to_f64(v: np.ndarray) -> np.ndarray:
    """uint64 -> float64 rounded to nearest even (Python's int -> float) for the values above 2^53"""
    out = v.astype(np.float64)
    big = np.flatnonzero(v >= np.uint64(1 << 53))
    out[big] = [float(int(x)) for x in v[big]]
    return out


def group_statistics(records: np.ndarray, order, gid=None, identity=None) -> np.ndarray:
    """rk_group_statistics by its definition (include/rk_b200.h), evaluated exactly: one row per group of the output lines
    (order: file index of each line, gid: nondecreasing dense group ids, identity: the float32 identity column).
    Integers from uint64 reductions; mean_identity = math.fsum of the members (the exactly rounded sum) / count, NaN
    (NAN_BITS) if a member is NaN, else +inf if one is +inf; multiplicity = float(sum of lengths) / float(X span).
    `order` may also be the OracleGroups of group(): its order, out_gid and identity are used."""
    import math
    from repkiller_b200.capi import GROUP_STATS_DTYPE
    if isinstance(order, OracleGroups):
        order, gid, identity = order.order, order.out_gid, order.identity
    order = np.asarray(order, np.int64)
    gid = np.asarray(gid, np.int64)
    ident = np.asarray(identity, np.float32).astype(np.float64)
    m = order.shape[0]
    if m == 0:
        return np.zeros(0, GROUP_STATS_DTYPE)
    starts = np.r_[0, np.flatnonzero(gid[1:] != gid[:-1]) + 1]
    n_groups = starts.shape[0]
    if (gid[starts] != gid[0] + np.arange(n_groups)).any():
        raise ValueError("group ids are not dense and nondecreasing")
    count = np.diff(np.r_[starts, m])
    xs, ys, ln = (np.asarray(records[f])[order].astype(np.uint64) for f in ("xStart", "yStart", "length"))
    out = np.zeros(n_groups, GROUP_STATS_DTYPE)
    out["count"], out["first_line"] = count, starts
    out["x_lo"], out["y_lo"] = np.minimum.reduceat(xs, starts), np.minimum.reduceat(ys, starts)
    out["x_hi"], out["y_hi"] = np.maximum.reduceat(xs + ln, starts), np.maximum.reduceat(ys + ln, starts)
    span = out["x_hi"] - np.minimum.reduceat(xs, starts)
    total = np.add.reduceat(ln, starts)
    mult = np.zeros(n_groups)
    nz = span > 0
    mult[nz] = _to_f64(total[nz]) / _to_f64(span[nz])
    out["multiplicity"] = mult
    has_nan = np.add.reduceat(np.isnan(ident).astype(np.int64), starts) > 0
    has_inf = np.add.reduceat(np.isposinf(ident).astype(np.int64), starts) > 0
    s = ident[starts].copy()                      # singletons
    vals = ident.tolist()
    for k in np.flatnonzero((count > 1) & ~has_nan & ~has_inf).tolist():
        a = int(starts[k])
        s[k] = math.fsum(vals[a:a + int(count[k])])
    s[has_inf] = math.inf
    mean = s / count.astype(np.float64)
    mean.view(np.uint64)[has_nan] = np.uint64(NAN_BITS)
    out["mean_identity"] = mean
    return out


def std_sort_by_key(idx: np.ndarray, h: np.ndarray) -> np.ndarray:
    """libstdc++ std::sort order of idx under comp(a, b) = h[a] < h[b]."""
    out = np.ascontiguousarray(idx, dtype=np.uint32).copy()
    hh = np.ascontiguousarray(h, dtype=np.uint64)
    lib().rko_std_sort_by_key(out.ctypes.data, out.shape[0], hh.ctypes.data)
    return out


class Sol:
    """One SequenceOcupationList of the restatement (rko_sol_*): the checker of repkiller_b200.capi.Sol"""

    def __init__(self, len_ratio: float, pos_ratio: float, seq_size: int):
        L = lib()
        L.rko_sol_create.argtypes = [C.c_double, C.c_double, C.c_uint64]
        L.rko_sol_create.restype = C.c_void_p
        L.rko_sol_insert.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64]
        L.rko_sol_get.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(C.c_uint64)]
        L.rko_sol_destroy.argtypes = [C.c_void_p]
        self._L = L
        self._h = L.rko_sol_create(len_ratio, pos_ratio, seq_size)
        if not self._h:
            raise MemoryError("rko_sol_create")

    def insert(self, center: int, length: int, tag: int) -> None:
        rc = self._L.rko_sol_insert(self._h, center, length, tag)
        if rc == -1:
            raise IndexError(f"center {center} lies beyond the lists")
        if rc:
            raise MemoryError("rko_sol_insert")

    def get(self, center: int, length: int) -> int:
        """tag of the entry get_associated_group returns, 0 for none"""
        t = C.c_uint64()
        if self._L.rko_sol_get(self._h, center, length, C.byref(t)):
            raise IndexError(f"a probe of center {center} reads beyond the lists")
        return t.value

    def close(self):
        if self._h:
            self._L.rko_sol_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()


def have_ref() -> bool:
    return os.path.exists(REF_BIN) and os.access(REF_BIN, os.X_OK)


def run_ref(in_csv: str, out_csv: str, len_ratio: float, pos_ratio: float, nosave: bool = False, timeout: float | None = None) -> dict:
    """Run the compiled reference (oracle/_ref/repkiller_ref); returns its per-phase timing line."""
    env = dict(os.environ)
    if nosave:
        env["RK_REF_NOSAVE"] = "1"
    p = subprocess.run([REF_BIN, in_csv, out_csv, repr(len_ratio), repr(pos_ratio)], env=env, capture_output=True,
                       timeout=timeout)
    if p.returncode != 0:
        raise RuntimeError(f"repkiller_ref rc={p.returncode}: {p.stderr[-400:]!r}")
    return json.loads(p.stderr.decode().strip().splitlines()[-1])
