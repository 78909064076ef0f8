"""ctypes binding of librk_b200.so (include/rk_b200.h).

This is plumbing: the product is the CUDA library behind the C ABI.  There is no CPU path — importing works
anywhere (so the symbol table can be checked), but creating a Context without a CUDA device raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "librk_b200%s.so" % os.environ.get("RK_LIB_SUFFIX", ""))  # suffix: tuning variants only

RK_NONE = 0xFFFFFFFF
F_HOST_RESULT, F_NO_SORT, F_TIMING, F_LINE_RECORDS = 1, 2, 4, 8
STAGES = ["h2d", "decode", "ranksort", "keys", "xsort", "ysort", "xmatch", "ymatch", "forest", "hkey", "gsort",
          "final", "d2h"]
NSTAGES = len(STAGES)

# every symbol include/rk_b200.h declares
SYMBOLS = ["rk_create", "rk_create_view", "rk_create_error", "rk_destroy", "rk_last_error", "rk_set_stream", "rk_load_aos", "rk_load_packed", "rk_load_csv", "rk_group", "rk_sort_groups", "rk_host_alloc", "rk_host_free",
           "rk_diagonal_func", "rk_format_lines", "rk_debug_fetch", "rk_profile_enable", "rk_profile_read", "rk_sort_pairs_work_bytes", "rk_sort_pairs", "rk_version",
           "rk_gen_workload", "rk_sort_members", "rk_group_statistics", "rk_sol_create", "rk_sol_destroy", "rk_sol_insert", "rk_sol_get_associated", "rk_sol_last_error",
           # one comparison over several GPUs
           "rk_dist_unique_id", "rk_dist_init", "rk_dist_export", "rk_dist_import", "rk_dist_load_aos", "rk_dist_load_csv", "rk_dist_load_packed",
           "rk_dist_group", "rk_dist_format_lines", "rk_dist_group_statistics", "rk_dist_create_view",
           "rk_create_multi", "rk_destroy_multi", "rk_multi_last_error", "rk_multi_ranks", "rk_multi_ctx", "rk_multi_transport",
           "rk_multi_load_aos", "rk_multi_load_csv", "rk_multi_load_packed", "rk_multi_group", "rk_multi_info", "rk_multi_format_lines", "rk_multi_group_statistics",
           "rk_multi_create_view"]
DIST_ID_BYTES, DIST_BLOB_BYTES = 128, 128
GROUP_STATS_DTYPE = np.dtype([("count", "<u4"), ("x_lo", "<u4"), ("y_lo", "<u4"), ("first_line", "<u4"), ("x_hi", "<u8"), ("y_hi", "<u8"),
                              ("mean_identity", "<f8"), ("multiplicity", "<f8")])


class RkError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"rk status {code}: {msg}")
        self.code = code


class _LoadStats(C.Structure):
    _fields_ = [("n_loaded", C.c_uint64), ("n_kept", C.c_uint64), ("vsize", C.c_uint64),
                ("ms_stage", C.c_float * NSTAGES), ("ms_device", C.c_float), ("n_launches", C.c_uint64)]


class _CsvStats(C.Structure):
    _fields_ = [("n_rows", C.c_uint64), ("n_accepted", C.c_uint64), ("n_host_rows", C.c_uint64), ("wide", C.c_int),
                ("ms_upload", C.c_float), ("ms_parse", C.c_float)]


class _KernelTime(C.Structure):
    _fields_ = [("name", C.c_char_p), ("launches", C.c_uint64), ("ms_total", C.c_double), ("units", C.c_uint64)]


class _Result(C.Structure):
    _fields_ = [("n_kept", C.c_uint64), ("n_groups", C.c_uint64),
                ("order", C.POINTER(C.c_uint32)), ("gid", C.POINTER(C.c_uint32)), ("repval", C.POINTER(C.c_uint8)),
                ("identity", C.POINTER(C.c_float)),
                ("d_order", C.c_void_p), ("d_gid", C.c_void_p), ("d_repval", C.c_void_p), ("d_identity", C.c_void_p),
                ("ms_stage", C.c_float * NSTAGES), ("ms_device", C.c_float), ("n_launches", C.c_uint64)]


class _DistInfo(C.Structure):
    _fields_ = [("rank", C.c_int), ("world", C.c_int)] + [(k, C.c_uint64) for k in (
        "total_loaded", "total_kept", "total_groups", "line_offset", "n_lines", "rank_offset", "n_ranked", "n_halo_in",
        "n_halo_out", "n_y", "bytes_sent")]


def _info_dict(i: "_DistInfo") -> dict:
    return {k: int(getattr(i, k)) for k, _ in _DistInfo._fields_}


_lib = None


def load_library():
    """dlopen the in-tree library (building it is __graft_entry__.build()'s job; fail loudly if it is missing)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RkError(-1, f"{LIB_PATH} is missing: run `python -m repkiller_b200.build` (there is no fallback path)")
    L = C.CDLL(LIB_PATH)
    L.rk_create.argtypes = [C.c_int]
    L.rk_create.restype = C.c_void_p
    L.rk_create_view.argtypes = [C.c_void_p]
    L.rk_create_view.restype = C.c_void_p
    L.rk_create_error.restype = C.c_char_p
    L.rk_destroy.argtypes = [C.c_void_p]
    L.rk_last_error.argtypes = [C.c_void_p]
    L.rk_last_error.restype = C.c_char_p
    L.rk_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    L.rk_load_aos.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint, C.POINTER(_LoadStats)]
    L.rk_load_packed.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint, C.POINTER(_LoadStats)]
    L.rk_load_csv.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint, C.POINTER(_LoadStats),
                              C.POINTER(_CsvStats)]
    L.rk_group.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_uint, C.POINTER(_Result)]
    L.rk_sort_groups.argtypes = [C.c_void_p, C.c_uint, C.POINTER(_Result)]
    L.rk_diagonal_func.argtypes = [C.c_void_p, C.c_void_p]
    L.rk_debug_fetch.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_uint64]
    L.rk_debug_fetch.restype = C.c_int64
    L.rk_sort_pairs_work_bytes.argtypes = [C.c_uint64]
    L.rk_sort_pairs_work_bytes.restype = C.c_uint64
    L.rk_sort_pairs.argtypes = [C.c_void_p] + [C.c_void_p] * 6 + [C.c_uint64, C.c_int, C.c_void_p]
    L.rk_version.restype = C.c_char_p
    L.rk_format_lines.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(_Text)]
    L.rk_profile_enable.argtypes = [C.c_void_p, C.c_int]
    L.rk_profile_read.argtypes = [C.c_void_p, C.POINTER(_KernelTime), C.c_int, C.c_int]
    L.rk_group_statistics.argtypes = [C.c_void_p, C.c_uint, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
    L.rk_sort_members.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.rk_dist_unique_id.argtypes = [C.c_void_p]
    L.rk_dist_init.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_uint64]
    L.rk_dist_export.argtypes = [C.c_void_p, C.c_void_p]
    L.rk_dist_import.argtypes = [C.c_void_p, C.c_void_p]
    L.rk_dist_load_aos.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint, C.POINTER(_LoadStats)]
    L.rk_dist_load_csv.argtypes = L.rk_load_csv.argtypes
    L.rk_dist_load_packed.argtypes = [C.c_void_p] * 4 + [C.c_uint64] * 4 + [C.c_uint, C.POINTER(_LoadStats)]
    L.rk_dist_group.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_uint, C.POINTER(_Result), C.POINTER(_DistInfo)]
    L.rk_dist_format_lines.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(_Text)]
    L.rk_dist_group_statistics.argtypes = [C.c_void_p, C.c_uint, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_uint64),
                                           C.POINTER(C.c_uint64)]
    L.rk_dist_create_view.argtypes = [C.c_void_p, C.c_void_p]
    L.rk_dist_create_view.restype = C.c_void_p
    L.rk_create_multi.argtypes = [C.POINTER(C.c_int), C.c_int]
    L.rk_create_multi.restype = C.c_void_p
    L.rk_destroy_multi.argtypes = [C.c_void_p]
    L.rk_multi_last_error.argtypes = [C.c_void_p]
    L.rk_multi_last_error.restype = C.c_char_p
    L.rk_multi_ranks.argtypes = [C.c_void_p]
    L.rk_multi_ctx.argtypes = [C.c_void_p, C.c_int]
    L.rk_multi_ctx.restype = C.c_void_p
    L.rk_multi_transport.argtypes = [C.c_void_p]
    L.rk_multi_transport.restype = C.c_char_p
    L.rk_multi_load_aos.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint, C.POINTER(_LoadStats)]
    L.rk_multi_load_csv.argtypes = L.rk_load_csv.argtypes
    L.rk_multi_load_packed.argtypes = L.rk_load_packed.argtypes
    L.rk_multi_group.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_uint, C.POINTER(_Result)]
    L.rk_multi_info.argtypes = [C.c_void_p, C.c_int, C.POINTER(_DistInfo)]
    L.rk_multi_format_lines.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(_Text)]
    L.rk_multi_group_statistics.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
    L.rk_multi_create_view.argtypes = [C.c_void_p]
    L.rk_multi_create_view.restype = C.c_void_p
    L.rk_sol_create.argtypes = [C.c_int, C.c_double, C.c_double, C.c_uint64]
    L.rk_sol_create.restype = C.c_void_p
    L.rk_sol_destroy.argtypes = [C.c_void_p]
    L.rk_sol_insert.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64]
    L.rk_sol_get_associated.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(C.c_uint64)]
    L.rk_sol_last_error.argtypes = [C.c_void_p]
    L.rk_sol_last_error.restype = C.c_char_p
    _lib = L
    return L


class _Text(C.Structure):
    _fields_ = [("text", C.c_void_p), ("n_bytes", C.c_uint64), ("ms_device", C.c_float)]


FORMAT_MAX_LINES = 8_000_000


@dataclass
class LoadStats:
    n_loaded: int
    n_kept: int
    vsize: int
    ms_stage: dict
    ms_device: float
    n_launches: int = 0


@dataclass
class CsvStats:
    """what rk_load_csv saw in the text: rows (the empty one after a final newline included), records loaded, rows left
    to the host parser, whether the 109-byte route was taken, and the device times of the upload and the parse"""
    n_rows: int
    n_accepted: int
    n_host_rows: int
    wide: bool
    ms_upload: float
    ms_parse: float


@dataclass
class Groups:
    """Result of one (len_ratio, pos_ratio) grouping, in the reference's output order."""
    n_kept: int
    n_groups: int
    order: np.ndarray | None      # file index of each output line
    gid: np.ndarray | None        # the `block` column
    repval: np.ndarray | None
    identity: np.ndarray | None
    d_ptrs: dict = field(default_factory=dict)
    ms_stage: dict = field(default_factory=dict)
    ms_device: float = 0.0
    n_launches: int = 0


class Context:
    """One GPU-resident fragment database + grouping workspace (FragmentsDatabase's role on the device)."""

    def __init__(self, device: int = 0):
        self._L = load_library()
        self._h = self._L.rk_create(device)
        if not self._h:
            raise RkError(-1, self._L.rk_create_error().decode())
        self.device = device

    @classmethod
    def _wrap(cls, handle: int, device: int) -> "Context":
        c = cls.__new__(cls)
        c._L, c._h, c.device = load_library(), handle, device
        return c

    def view(self) -> "Context":
        """A second grouping context over this context's loaded database (rk_create_view): its own stream and workspace,
        the load shared.  Different contexts may group concurrently from different threads; close() releases the view,
        and the database lives until the last context that shares it is closed."""
        h = self._L.rk_create_view(self._h)
        if not h:
            raise RkError(-1, self._L.rk_create_error().decode())
        v = Context._wrap(h, self.device)
        v._keep = getattr(self, "_keep", None)  # records the load reads in place stay alive while the view uses them
        return v

    def close(self):
        if getattr(self, "_h", None):
            self._L.rk_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc: int):
        if rc != 0:
            raise RkError(rc, self._L.rk_last_error(self._h).decode())

    def set_stream(self, cuda_stream_ptr: int):
        self._check(self._L.rk_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    def load(self, records, seqx_len: int, seqy_len: int, n: int | None = None, timing: bool = True) -> LoadStats:
        """records: numpy array of 109-byte FragFile records (host), or an int device/host pointer with n given.
        seqx_len/seqy_len are the LOADED lengths (header value + 1)."""
        if isinstance(records, np.ndarray):
            rec = np.ascontiguousarray(records)
            assert rec.dtype.itemsize == 109 or rec.dtype == np.uint8
            n = rec.nbytes // 109
            ptr = rec.ctypes.data
            self._keep = rec
        else:
            ptr = int(records)
            assert n is not None
        st = _LoadStats()
        self._check(self._L.rk_load_aos(self._h, C.c_void_p(ptr), n, seqx_len, seqy_len, F_TIMING if timing else 0, C.byref(st)))
        return LoadStats(st.n_loaded, st.n_kept, st.vsize, {STAGES[i]: st.ms_stage[i] for i in range(NSTAGES)}, st.ms_device,
                         st.n_launches)

    def load_packed(self, key4, strand, rest4, seqx_len: int, seqy_len: int, n: int | None = None, timing: bool = True) -> LoadStats:
        """The compact ingest (rk_load_packed): numpy arrays key4 [n,4] u32, strand [n] u8, rest4 [n,4] u32 or None — or int
        pointers (host or device) with n given."""
        keep, pk, ps, pr, n = _packed_args(key4, strand, rest4, n)
        if keep is not None:
            self._keep = keep
        st = _LoadStats()
        self._check(self._L.rk_load_packed(self._h, C.c_void_p(pk), C.c_void_p(ps), C.c_void_p(pr) if pr else None, n, seqx_len, seqy_len,
                                           F_TIMING if timing else 0, C.byref(st)))
        return LoadStats(st.n_loaded, st.n_kept, st.vsize, {STAGES[i]: st.ms_stage[i] for i in range(NSTAGES)}, st.ms_device,
                         st.n_launches)

    def load_csv(self, body, seqx_len: int, seqy_len: int, total_frags: int, timing: bool = True):
        """The body of a GECKO CSV (the bytes after its 16 header lines) parsed and loaded on the device (rk_load_csv):
        bytes, a uint8 numpy array, or a uint8 torch tensor on the CPU or on this context's GPU.  seqx_len/seqy_len are the
        LOADED lengths (header value + 1), total_frags the header's "Total fragments".  Returns (LoadStats, CsvStats)."""
        arr, ptr, n = _text_arg(body, "load_csv")
        st, cs = _LoadStats(), _CsvStats()
        self._check(self._L.rk_load_csv(self._h, C.c_void_p(ptr) if n else None, n, seqx_len, seqy_len, total_frags,
                                        F_TIMING if timing else 0, C.byref(st), C.byref(cs)))
        self._keep = None  # the parsed rows are the database's own: the text may go
        return _csv_result(st, cs)

    def group(self, len_ratio: float, pos_ratio: float, host_result: bool = True, sort: bool = True, timing: bool = True,
              copy: bool = True) -> Groups:
        """copy=False: the host arrays are views of the library-owned pinned result buffers (what a C caller gets);
        they are valid until the next call on this context."""
        flags = (F_HOST_RESULT if host_result else 0) | (0 if sort else F_NO_SORT) | (F_TIMING if timing else 0)
        r = _Result()
        self._check(self._L.rk_group(self._h, len_ratio, pos_ratio, flags, C.byref(r)))
        m = r.n_kept
        self._last_m = m

        def arr(p, dt):
            if not host_result:
                return None
            if m == 0:
                return np.zeros(0, dt)
            v = np.ctypeslib.as_array(p, shape=(m,))
            return v.copy() if copy else v

        return Groups(m, r.n_groups, arr(r.order, np.uint32), arr(r.gid, np.uint32), arr(r.repval, np.uint8),
                      arr(r.identity, np.float32),
                      {"order": r.d_order, "gid": r.d_gid, "repval": r.d_repval, "identity": r.d_identity},
                      {STAGES[i]: r.ms_stage[i] for i in range(NSTAGES)}, r.ms_device, r.n_launches)

    def sort_groups(self, host_result: bool = True, copy: bool = True) -> Groups:
        """rk_sort_groups: after group(..., sort=False), the members of every group ordered on the device (sort_groups)"""
        r = _Result()
        self._check(self._L.rk_sort_groups(self._h, F_HOST_RESULT if host_result else 0, C.byref(r)))
        return _groups_of(r, host_result, copy)

    def format_lines(self, first_line: int = 0, n_lines: int | None = None) -> bytes:
        """Text of the output lines of the last group() (commonFunctions.cpp:101-115), formatted on the device; the
        16 header lines are the caller's.  Chunks of FORMAT_MAX_LINES lines are concatenated."""
        text, self.ms_format = _format_chunks(lambda a, k, t: self._check(self._L.rk_format_lines(self._h, a, k, t)), first_line,
                                              self._last_m if n_lines is None else n_lines)
        return text

    def generate_device(self, w, start: int, count: int, out_ptr: int):
        """Records start..start+count of workload `w` (repkiller_b200.gen.Workload) written to device memory at out_ptr
        (count * 109 bytes).  Same bytes as gen.generate(w, start, count)."""
        f = self._L.rk_gen_workload
        f.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_double] + [C.c_uint64] * 6 + [C.c_void_p]
        self._check(f(self._h, w.seed, w.lx, w.ly, w.p_rep, w.families, w.ax, w.ay, w.tandem_every, start, count,
                      C.c_void_p(out_ptr)))

    def profile_enable(self, on: bool = True):
        self._check(self._L.rk_profile_enable(self._h, int(on)))

    def profile_read(self, reset: bool = True) -> dict:
        """{kernel name: (launches, total ms, units processed)} accumulated since the last reset."""
        buf = (_KernelTime * 32)()
        k = self._L.rk_profile_read(self._h, buf, 32, int(reset))
        return {buf[i].name.decode(): (int(buf[i].launches), float(buf[i].ms_total), int(buf[i].units)) for i in range(k)}

    def diagonal_func(self, vsize: int) -> np.ndarray:
        out = np.zeros(max(vsize - 1, 0), dtype=np.uint64)
        if out.size:
            self._check(self._L.rk_diagonal_func(self._h, C.c_void_p(out.ctypes.data)))
        return out

    def debug_fetch(self, name: str, dtype=np.uint32) -> np.ndarray:
        """a device array of the last load/group (rk_debug_fetch); "strand" is bytes (dtype=np.uint8), "key4" and "rest4"
        four uint32 per record"""
        sz = self._L.rk_debug_fetch(self._h, name.encode(), None, 0)
        if sz < 0:
            self._check(int(sz))
        out = np.zeros(sz // np.dtype(dtype).itemsize, dtype=dtype)
        if sz:
            got = self._L.rk_debug_fetch(self._h, name.encode(), C.c_void_p(out.ctypes.data), out.nbytes)
            if got < 0:
                self._check(int(got))
        return out

    def sort_pairs_device(self, keys_in: int, values_in: int | None, keys_out: int, values_out: int, keys_tmp: int,
                          values_tmp: int, n: int, key_bits: int, work: int):
        self._check(self._L.rk_sort_pairs(self._h, C.c_void_p(keys_in), C.c_void_p(values_in) if values_in else None,
                                          C.c_void_p(keys_out), C.c_void_p(values_out), C.c_void_p(keys_tmp),
                                          C.c_void_p(values_tmp), n, key_bits, C.c_void_p(work)))

    def sort_pairs_work_bytes(self, n: int) -> int:
        return int(self._L.rk_sort_pairs_work_bytes(n))

    def group_statistics(self) -> np.ndarray:
        """per-group statistics of the last group() as a structured array (GROUP_STATS_DTYPE), one row per group id"""
        hp, dp, ng = C.c_void_p(), C.c_void_p(), C.c_uint64()
        self._check(self._L.rk_group_statistics(self._h, F_HOST_RESULT, C.byref(hp), C.byref(dp), C.byref(ng)))
        return _stats_array(hp.value, ng.value)

    def sort_members(self, gid: np.ndarray, y: np.ndarray, d: np.ndarray) -> np.ndarray:
        """sort_groups as a pure function: perm[j] = index of the member std::sort leaves at position j (members given
        group by group, h = |y - d|)"""
        g = np.ascontiguousarray(gid, dtype=np.uint32)
        yy, dd = np.ascontiguousarray(y, dtype=np.uint64), np.ascontiguousarray(d, dtype=np.uint64)
        perm = np.zeros(g.shape[0], dtype=np.uint32)
        self._check(self._L.rk_sort_members(self._h, g.shape[0], C.c_void_p(g.ctypes.data), C.c_void_p(yy.ctypes.data),
                                            C.c_void_p(dd.ctypes.data), C.c_void_p(perm.ctypes.data)))
        return perm

    # ---- one comparison over several GPUs, one process per GPU (rk_dist_*; collective calls) ----
    def dist_init(self, rank: int, world: int, unique_id: bytes, cap_per_rank: int):
        assert len(unique_id) == DIST_ID_BYTES
        self._check(self._L.rk_dist_init(self._h, rank, world, C.c_char_p(unique_id), cap_per_rank))

    def dist_view(self, unique_id: bytes) -> "Context":
        """A view of this rank's partitioned load (rk_dist_create_view; collective): a second grouping context with its
        own stream, NCCL communicator and workspace.  unique_id: a fresh dist_unique_id() of rank 0, broadcast; then
        every rank calls dist_export / dist_import on the view, as after dist_init."""
        assert len(unique_id) == DIST_ID_BYTES
        h = self._L.rk_dist_create_view(self._h, C.c_char_p(unique_id))
        if not h:
            raise RkError(-1, self._L.rk_create_error().decode())
        v = Context._wrap(h, self.device)
        v._keep = getattr(self, "_keep", None)
        return v

    def dist_export(self) -> bytes:
        buf = C.create_string_buffer(DIST_BLOB_BYTES)
        self._check(self._L.rk_dist_export(self._h, buf))
        return buf.raw

    def dist_import(self, blobs: bytes):
        self._check(self._L.rk_dist_import(self._h, C.c_char_p(blobs)))

    def dist_load(self, ptr: int, n_local: int, file_offset: int, seqx_len: int, seqy_len: int, timing: bool = False) -> LoadStats:
        st = _LoadStats()
        self._check(self._L.rk_dist_load_aos(self._h, C.c_void_p(ptr), n_local, file_offset, seqx_len, seqy_len,
                                             F_TIMING if timing else 0, C.byref(st)))
        return LoadStats(st.n_loaded, st.n_kept, st.vsize, {STAGES[i]: st.ms_stage[i] for i in range(NSTAGES)}, st.ms_device,
                         st.n_launches)

    def dist_load_csv(self, body, seqx_len: int, seqy_len: int, total_frags: int, timing: bool = False):
        """This rank's slice of a GECKO CSV body (rk_dist_load_csv; collective): the body types of load_csv.  Every slice
        before the last non-empty one ends with a newline; the library works out the file offsets.  Returns (LoadStats,
        CsvStats) with this rank's counts."""
        arr, ptr, n = _text_arg(body, "dist_load_csv")
        st, cs = _LoadStats(), _CsvStats()
        self._check(self._L.rk_dist_load_csv(self._h, C.c_void_p(ptr) if n else None, n, seqx_len, seqy_len, total_frags,
                                             F_TIMING if timing else 0, C.byref(st), C.byref(cs)))
        return _csv_result(st, cs)

    def dist_load_packed(self, key4, strand, rest4, file_offset: int, seqx_len: int, seqy_len: int, n: int | None = None,
                         timing: bool = False) -> LoadStats:
        """This rank's slice of the file in the compact form (rk_dist_load_packed; collective): the arguments of load_packed,
        file_offset = the file index of the slice's first fragment.  Host arrays are copied before the call returns;
        device arrays (int pointers on this rank's device, key4 and rest4 16-byte aligned) are used in place."""
        _, pk, ps, pr, n = _packed_args(key4, strand, rest4, n)
        st = _LoadStats()
        self._check(self._L.rk_dist_load_packed(self._h, C.c_void_p(pk) if pk else None, C.c_void_p(ps) if ps else None,
                                                C.c_void_p(pr) if pr else None, n, file_offset, seqx_len, seqy_len,
                                                F_TIMING if timing else 0, C.byref(st)))
        return LoadStats(st.n_loaded, st.n_kept, st.vsize, {STAGES[i]: st.ms_stage[i] for i in range(NSTAGES)}, st.ms_device,
                         st.n_launches)

    def dist_group(self, len_ratio: float, pos_ratio: float, host_result: bool = True, sort: bool = True, timing: bool = False,
                   copy: bool = True, line_records: bool = False):
        """(Groups of THIS rank's range of output lines, info dict); line_records: for dist_format_lines /
        dist_group_statistics"""
        flags = ((F_HOST_RESULT if host_result else 0) | (0 if sort else F_NO_SORT) | (F_TIMING if timing else 0)
                 | (F_LINE_RECORDS if line_records else 0))
        r, info = _Result(), _DistInfo()
        self._check(self._L.rk_dist_group(self._h, len_ratio, pos_ratio, flags, C.byref(r), C.byref(info)))
        self._dist_lines = info.n_lines
        return _groups_of(r, host_result, copy), _info_dict(info)

    def dist_format_lines(self, first_line: int = 0, n_lines: int | None = None) -> bytes:
        """text of THIS rank's lines first_line .. (local indices) after dist_group(..., line_records=True)"""
        text, self.ms_format = _format_chunks(lambda a, k, t: self._check(self._L.rk_dist_format_lines(self._h, a, k, t)), first_line,
                                              self._dist_lines if n_lines is None else n_lines)
        return text

    def dist_group_statistics(self):
        """(first gid, statistics of THIS rank's groups) after dist_group(..., line_records=True)"""
        hp, dp, fg, ng = C.c_void_p(), C.c_void_p(), C.c_uint64(), C.c_uint64()
        self._check(self._L.rk_dist_group_statistics(self._h, F_HOST_RESULT, C.byref(hp), C.byref(dp), C.byref(fg), C.byref(ng)))
        return fg.value, _stats_array(hp.value, ng.value)


def _format_chunks(call, first_line: int, n_lines: int):
    """(text, device ms) of lines first_line .. first_line + n_lines in calls of at most FORMAT_MAX_LINES lines;
    call(first, count, byref(_Text)) formats one chunk"""
    out, ms, done = [], 0.0, 0
    while True:
        cnt = min(FORMAT_MAX_LINES, n_lines - done)
        t = _Text()
        call(first_line + done, cnt, C.byref(t))
        out.append(C.string_at(t.text, t.n_bytes) if t.n_bytes else b"")
        ms += t.ms_device
        done += cnt
        if done >= n_lines:
            return b"".join(out), ms


def _stats_array(ptr, n: int) -> np.ndarray:
    if n == 0:
        return np.zeros(0, dtype=GROUP_STATS_DTYPE)
    return np.frombuffer(C.string_at(ptr, n * GROUP_STATS_DTYPE.itemsize), dtype=GROUP_STATS_DTYPE).copy()


def _groups_of(r: "_Result", host_result: bool, copy: bool) -> Groups:
    m = r.n_kept

    def arr(p, dt):
        if not host_result:
            return None
        if m == 0:
            return np.zeros(0, dt)
        v = np.ctypeslib.as_array(p, shape=(m,))
        return v.copy() if copy else v

    return Groups(m, r.n_groups, arr(r.order, np.uint32), arr(r.gid, np.uint32), arr(r.repval, np.uint8), arr(r.identity, np.float32),
                  {"order": r.d_order, "gid": r.d_gid, "repval": r.d_repval, "identity": r.d_identity},
                  {STAGES[i]: r.ms_stage[i] for i in range(NSTAGES)}, r.ms_device, r.n_launches)


def _packed_args(key4, strand, rest4, n):
    """(arrays to keep alive or None, key4, strand, rest4 addresses (rest4 None when absent), n) of the compact arrays:
    numpy arrays key4 [n,4] u32, strand [n] u8, rest4 [n,4] u32 or None — or int pointers with n given"""
    if isinstance(key4, np.ndarray):
        k, s_ = np.ascontiguousarray(key4, dtype=np.uint32), np.ascontiguousarray(strand, dtype=np.uint8)
        r = np.ascontiguousarray(rest4, dtype=np.uint32) if rest4 is not None else None
        return (k, s_, r), k.ctypes.data, s_.ctypes.data, (r.ctypes.data if r is not None else None), s_.shape[0]
    assert n is not None
    return None, int(key4), int(strand), (int(rest4) if rest4 else None), n


def pack_records(rec: np.ndarray):
    """(key4, strand, rest4) of 109-byte FragFile records for Context.load_packed; every value must fit in 32 bits"""
    for f in ("xStart", "yStart", "length", "ident", "xEnd", "yEnd", "score"):
        if rec.shape[0] and int(rec[f].max()) >> 32:
            raise ValueError(f"{f} does not fit in 32 bits: use Context.load (rk_load_aos)")
    key4 = np.stack([rec["xStart"], rec["yStart"], rec["length"], rec["ident"]], axis=1).astype(np.uint32)
    rest4 = np.stack([rec["xEnd"].astype(np.uint32), rec["yEnd"].astype(np.uint32), rec["score"].astype(np.uint32),
                      rec["similarity"].view(np.uint32)], axis=1)
    strand = rec["strand"].view(np.uint8).copy()
    return np.ascontiguousarray(key4), strand, np.ascontiguousarray(rest4)


class Sol:
    """One device-resident SequenceOcupationList (rk_sol_*): inserts are queued and applied in order before the next
    query; a query returns the tag of the entry get_associated_group picks, 0 for none.  Tags must be non-zero."""

    def __init__(self, device: int, len_ratio: float, pos_ratio: float, seq_size: int):
        self._L = load_library()
        self._h = self._L.rk_sol_create(device, len_ratio, pos_ratio, seq_size)
        if not self._h:
            raise RkError(-1, f"rk_sol_create({device}, {len_ratio}, {pos_ratio}, {seq_size}) failed")

    def _check(self, rc: int):
        if rc != 0:
            raise RkError(rc, self._L.rk_sol_last_error(self._h).decode())

    def insert(self, center: int, length: int, tag: int):
        self._check(self._L.rk_sol_insert(self._h, center, length, tag))

    def get_associated(self, center: int, length: int) -> int:
        t = C.c_uint64()
        self._check(self._L.rk_sol_get_associated(self._h, center, length, C.byref(t)))
        return t.value

    def close(self):
        if getattr(self, "_h", None):
            self._L.rk_sol_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def dist_unique_id() -> bytes:
    """rank 0: the NCCL unique id every rank hands to Context.dist_init (broadcast it with whatever the application has)"""
    L = load_library()
    buf = C.create_string_buffer(DIST_ID_BYTES)
    rc = L.rk_dist_unique_id(buf)
    if rc:
        raise RkError(rc, "NCCL is not available")
    return buf.raw


def _text_arg(body, what: str):
    """(object to keep alive, address, bytes) of a text argument: bytes, a uint8 numpy array or a uint8 torch tensor"""
    if isinstance(body, (bytes, bytearray)):
        arr = np.frombuffer(bytes(body), dtype=np.uint8)
        return arr, arr.ctypes.data, arr.nbytes
    if isinstance(body, np.ndarray):
        arr = np.ascontiguousarray(body).view(np.uint8)
        return arr, arr.ctypes.data, arr.nbytes
    if type(body).__module__.startswith("torch"):
        arr = body.contiguous()
        assert arr.element_size() == 1
        return arr, arr.data_ptr(), arr.numel()
    raise TypeError(f"{what} takes bytes, a uint8 numpy array or a uint8 torch tensor")


def _csv_result(st: "_LoadStats", cs: "_CsvStats"):
    return (LoadStats(st.n_loaded, st.n_kept, st.vsize, {STAGES[i]: st.ms_stage[i] for i in range(NSTAGES)}, st.ms_device,
                      st.n_launches),
            CsvStats(cs.n_rows, cs.n_accepted, cs.n_host_rows, bool(cs.wide), cs.ms_upload, cs.ms_parse))


class Multi:
    """One comparison over several GPUs of one process (rk_create_multi): the library runs one host thread per GPU."""

    def __init__(self, devices):
        self._L = load_library()
        arr = (C.c_int * len(devices))(*devices)
        self._h = self._L.rk_create_multi(arr, len(devices))
        if not self._h:
            raise RkError(-1, self._L.rk_create_error().decode())
        self.n = len(devices)

    @property
    def transport(self) -> str:
        return self._L.rk_multi_transport(self._h).decode()

    def view(self) -> "Multi":
        """A second grouping context per rank over this comparison's load (rk_multi_create_view): its own streams,
        transport, workspace and result buffers.  Different Multi objects of one load may group at the same time from
        different threads; the load lives until the last of them is closed."""
        h = self._L.rk_multi_create_view(self._h)
        if not h:
            raise RkError(-1, self._L.rk_create_error().decode())
        v = Multi.__new__(Multi)
        v._L, v._h, v.n = self._L, h, self.n
        v._keep = getattr(self, "_keep", None)
        return v

    def ctx(self, rank: int) -> int:
        """the handle of rank's context (rk_multi_ctx), for calls on one rank"""
        return self._L.rk_multi_ctx(self._h, rank)

    def close(self):
        if getattr(self, "_h", None):
            self._L.rk_destroy_multi(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise RkError(rc, self._L.rk_multi_last_error(self._h).decode())

    def load(self, records: np.ndarray, seqx_len: int, seqy_len: int) -> LoadStats:
        rec = np.ascontiguousarray(records)
        self._keep = rec
        st = _LoadStats()
        self._check(self._L.rk_multi_load_aos(self._h, C.c_void_p(rec.ctypes.data), rec.nbytes // 109, seqx_len, seqy_len, 0, C.byref(st)))
        return LoadStats(st.n_loaded, st.n_kept, st.vsize, {}, st.ms_device, st.n_launches)

    def load_csv(self, body, seqx_len: int, seqy_len: int, total_frags: int, timing: bool = False):
        """A whole GECKO CSV body in host memory (bytes or a uint8 numpy array), cut into one slice per rank at row starts
        and parsed by every rank on its GPU (rk_multi_load_csv).  Returns (LoadStats, CsvStats): the counts summed over
        the ranks, the upload and parse times the largest of the ranks'."""
        arr, ptr, n = _text_arg(body, "Multi.load_csv")
        st, cs = _LoadStats(), _CsvStats()
        self._check(self._L.rk_multi_load_csv(self._h, C.c_void_p(ptr) if n else None, n, seqx_len, seqy_len, total_frags,
                                              F_TIMING if timing else 0, C.byref(st), C.byref(cs)))
        return _csv_result(st, cs)

    def load_packed(self, key4, strand, rest4, seqx_len: int, seqy_len: int, n: int | None = None, timing: bool = False) -> LoadStats:
        """The whole file in the compact form of Context.load_packed, in host memory (numpy arrays, or int host pointers with
        n given), cut into load()'s slices (rk_multi_load_packed); the arrays may go when this returns."""
        _, pk, ps, pr, n = _packed_args(key4, strand, rest4, n)
        st = _LoadStats()
        self._check(self._L.rk_multi_load_packed(self._h, C.c_void_p(pk) if pk else None, C.c_void_p(ps) if ps else None,
                                                 C.c_void_p(pr) if pr else None, n, seqx_len, seqy_len, F_TIMING if timing else 0,
                                                 C.byref(st)))
        return LoadStats(st.n_loaded, st.n_kept, st.vsize, {STAGES[i]: st.ms_stage[i] for i in range(NSTAGES)}, st.ms_device,
                         st.n_launches)

    def group(self, len_ratio: float, pos_ratio: float, sort: bool = True, line_records: bool = False) -> Groups:
        """line_records: every rank also gets the records of its output lines, for format_lines / group_statistics"""
        r = _Result()
        flags = (0 if sort else F_NO_SORT) | (F_LINE_RECORDS if line_records else 0)
        self._check(self._L.rk_multi_group(self._h, len_ratio, pos_ratio, flags, C.byref(r)))
        self._last_m = r.n_kept
        return _groups_of(r, True, True)

    def format_lines(self, first_line: int = 0, n_lines: int | None = None) -> bytes:
        """Context.format_lines over the whole comparison (global line indices), after group(..., line_records=True)"""
        text, self.ms_format = _format_chunks(lambda a, k, t: self._check(self._L.rk_multi_format_lines(self._h, a, k, t)), first_line,
                                              self._last_m if n_lines is None else n_lines)
        return text

    def group_statistics(self) -> np.ndarray:
        """Context.group_statistics over the whole comparison (all groups in gid order), after group(..., line_records=True)"""
        hp, ng = C.c_void_p(), C.c_uint64()
        self._check(self._L.rk_multi_group_statistics(self._h, C.byref(hp), C.byref(ng)))
        return _stats_array(hp.value, ng.value)

    def info(self, rank: int) -> dict:
        i = _DistInfo()
        self._check(self._L.rk_multi_info(self._h, rank, C.byref(i)))
        return _info_dict(i)
