"""ctypes binding of libgrakel_b200.so (the C-ABI declared in include/grakel_b200.h).

There is no CPU fallback: if the shared library or a B200 is missing, every
compute entry point raises.  The library is built in-tree by
``__graft_entry__.build()`` (``grakel_b200/csrc/build.sh``).
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgrakel_b200.so")

GK_F32, GK_F64 = 0, 1
GK_NORMALIZE, GK_NAN_TO_NUM, GK_GRAM_SIMT, GK_OUT_DEVICE, GK_FULL_TILES, GK_DENSE_ALL = 1, 2, 4, 8, 16, 32
GK_DIST, GK_DIST_GATHER = 64, 128
GK_SP_WITH_LABELS, GK_SP_KEEP_DIST, GK_SP_DIJKSTRA_ORDER = 1, 2, 4
GK_ERR_RANGE, GK_ERR_UNSUPPORTED = -4, -5
GK_NH_COUNT_SENSITIVE = 1


class GkStats(C.Structure):
    _fields_ = [
        ("n_graphs", C.c_int64), ("n_vertices", C.c_int64), ("n_edges", C.c_int64),
        ("n_levels", C.c_int64), ("level_dims", C.c_int64 * 64),
        ("n_columns", C.c_int64), ("n_entries", C.c_int64), ("n_dense_columns", C.c_int64),
        ("n_tail_columns", C.c_int64), ("tail_updates", C.c_int64), ("threshold", C.c_int64),
        ("max_count", C.c_int64), ("max_diag", C.c_int64), ("hash_retries", C.c_int64),
        ("gram_path", C.c_int64), ("gemm_tiles", C.c_int64), ("gemm_launches", C.c_int64),
        ("kernel_launches", C.c_int64),
        ("ms_h2d", C.c_float), ("ms_features", C.c_float), ("ms_panel", C.c_float),
        ("ms_gemm", C.c_float), ("ms_tail", C.c_float), ("ms_d2h", C.c_float), ("ms_total", C.c_float),
    ]

    def as_dict(self):
        d = {}
        for name, _ in self._fields_:
            v = getattr(self, name)
            d[name] = list(v)[: max(int(self.n_levels), 1)] if name == "level_dims" else v
        return d


class GrakelB200Error(RuntimeError):
    pass


_P = C.c_void_p
_SYMBOLS = {
    "gk_version": (C.c_int, []),
    "gk_last_error": (C.c_char_p, []),
    "gk_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "gk_destroy": (C.c_int, [_P]),
    "gk_sync": (C.c_int, [_P]),
    "gk_pack_csr": (C.c_int, [_P, C.c_int64, _P, _P, _P, _P, _P, _P, C.c_int32]),
    "gk_wl_features": (C.c_int, [_P, C.c_int32, C.POINTER(GkStats)]),
    "gk_sp_features": (C.c_int, [_P, C.c_int32, C.POINTER(GkStats)]),
    "gk_spattr_features": (C.c_int, [_P, C.c_int32, C.POINTER(GkStats)]),
    "gk_wl_sp_features": (C.c_int, [_P, C.c_int32, C.c_int32, C.POINTER(GkStats)]),
    "gk_wl_oa_features": (C.c_int, [_P, C.c_int32, C.POINTER(GkStats)]),
    "gk_nh_features": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, _P, C.POINTER(GkStats)]),
    "gk_nh_gram": (C.c_int, [_P, C.c_int64, C.c_int32, _P, C.c_int32, C.c_int64, C.POINTER(GkStats)]),
    "gk_nh_labels": (C.c_int, [_P, C.c_int32, _P]),
    "gk_gram": (C.c_int, [_P, C.c_int64, C.c_int32, C.c_int64, C.c_int64, _P, C.c_int32, C.c_int64, _P, _P,
                          C.POINTER(GkStats)]),
    "gk_fetch": (C.c_int, [_P, _P, C.c_int32, C.c_int64]),
    "gk_set_row_map": (C.c_int, [_P, C.c_int64, _P]),
    "gk_wl_labels": (C.c_int, [_P, C.c_int32, _P]),
    "gk_sp_distances": (C.c_int, [_P, C.c_int64, _P]),
    "gk_wl_fit_transform": (C.c_int, [_P, C.c_int64, _P, _P, _P, _P, C.c_int32, C.c_int32, _P, C.c_int32, C.c_int64,
                                      _P, C.POINTER(GkStats)]),
    "gk_wl_gram": (C.c_int, [_P, C.c_int32, C.c_int32, _P, C.c_int32, C.c_int64, _P, C.POINTER(GkStats)]),
    "gk_sp_fit_transform": (C.c_int, [_P, C.c_int64, _P, _P, _P, _P, _P, C.c_int32, C.c_int32, _P, C.c_int32,
                                      C.c_int64, _P, C.POINTER(GkStats)]),
    "gk_event_record": (C.c_int, [_P, C.c_int32]),
    "gk_event_elapsed": (C.c_int, [_P, C.c_int32, C.c_int32, C.POINTER(C.c_float)]),
    "gk_profiler_range": (C.c_int, [C.c_int32]),
    "gk_selftest_gram": (C.c_int, [_P, C.c_int64, C.c_int64, _P, _P, _P]),
    "gk_tu_open": (C.c_int, [C.c_char_p, C.c_char_p, C.c_int32, C.POINTER(_P)]),
    "gk_tu_info": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "gk_tu_pack": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "gk_tu_fill": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "gk_tu_close": (C.c_int, [_P]),
    "gk_comm_unique_id": (C.c_int, [_P]),
    "gk_comm_init": (C.c_int, [_P, C.c_int32, C.c_int32, _P]),
    "gk_comm_destroy": (C.c_int, [_P]),
    "gk_comm_rows": (C.c_int, [_P, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "gk_result_device": (C.c_int, [_P, C.POINTER(_P), C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                   C.POINTER(C.c_int32)]),
    "gk_selftest_dist_tiles": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "gk_host_alloc": (C.c_int, [C.c_int64, C.POINTER(_P)]),
    "gk_host_free": (C.c_int, [_P, C.c_int64]),
    "gk_selftest_deliver": (C.c_int, [C.c_int32, C.c_int64, C.c_int64, _P, _P, C.c_int32, _P]),
}

_lib = None
_lib_lock = threading.Lock()


def load_library():
    """Load the shared library and bind every symbol of include/grakel_b200.h."""
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise GrakelB200Error(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(grakel_b200 has no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SYMBOLS.items():
            fn = getattr(lib, name)  # AttributeError here = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def exported_symbols():
    return sorted(_SYMBOLS)


def _ptr(a):
    if a is None:
        return None
    return a.ctypes.data_as(_P)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


class _HostBlock:
    """Owner of one gk_host_alloc mapping; the ndarray returned to the user keeps it alive through `.base`."""

    def __init__(self, lib, nbytes):
        p = _P()
        if lib.gk_host_alloc(nbytes, C.byref(p)) != 0:
            raise MemoryError("gk_host_alloc(%d) failed: %s" % (nbytes, lib.gk_last_error().decode()))
        self._lib, self.ptr, self.nbytes = lib, p.value, nbytes
        self.__array_interface__ = {"data": (self.ptr, False), "shape": (nbytes,), "typestr": "|u1", "version": 3}

    def __del__(self):
        try:
            if self.ptr:
                self._lib.gk_host_free(self.ptr, self.nbytes)
                self.ptr = None
        except Exception:
            pass


def host_matrix(rows, cols, dtype=np.float64):
    """Fresh C-order (rows, cols) ndarray in a huge-page-backed, pooled host mapping (gk_host_alloc); small
    results come from numpy directly."""
    dt = np.dtype(dtype)
    nbytes = int(rows) * int(cols) * dt.itemsize
    if nbytes < (8 << 20) or os.environ.get("GRAKEL_B200_HOST_ALLOC", "1") == "0":
        return np.empty((rows, cols), dtype=dt)
    block = _HostBlock(load_library(), nbytes)
    return np.asarray(block).view(dt).reshape(rows, cols)


class Engine:
    """One device context (opaque gk_handle + CUDA stream).  Not picklable on
    purpose: estimators keep only host-side state and fetch an engine lazily."""

    def __init__(self, device=None):
        self.lib = load_library()
        if device is None:
            device = int(os.environ.get("GRAKEL_B200_DEVICE", os.environ.get("LOCAL_RANK", "0")))
        self.device = int(device)
        h = _P()
        rc = self.lib.gk_create(self.device, C.byref(h))
        if rc != 0:
            raise GrakelB200Error("gk_create failed: " + self.lib.gk_last_error().decode())
        self.h = h
        self._lock = threading.RLock()

    def close(self):
        """Destroy the handle now (collective when a communicator exists: every rank calls it)."""
        if getattr(self, "h", None):
            self.lib.gk_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            msg = self.lib.gk_last_error().decode()
            if rc == GK_ERR_UNSUPPORTED:
                raise NotImplementedError(msg)
            raise GrakelB200Error(f"[{rc}] {msg}")

    # ---- raw entry points -------------------------------------------------
    def pack(self, graph_ptr, row_ptr, col_idx, labels=None, weights=None, attrs=None):
        gp, rp, ci = _i32(graph_ptr), _i32(row_ptr), _i32(col_idx)
        lab = None if labels is None else _i32(labels)
        w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
        at, ad = None, 0
        if attrs is not None:
            at = np.ascontiguousarray(attrs, dtype=np.float64)
            ad = at.shape[1]
        with self._lock:
            self._check(self.lib.gk_pack_csr(self.h, len(gp) - 1, _ptr(gp), _ptr(rp), _ptr(ci), _ptr(lab), _ptr(w),
                                             _ptr(at), ad))
            self.n_graphs = len(gp) - 1

    def set_row_map(self, n_rows, row_of_graph):
        m = None if row_of_graph is None else _i32(row_of_graph)
        with self._lock:
            self._check(self.lib.gk_set_row_map(self.h, int(n_rows), _ptr(m)))

    def wl_features(self, n_iter):
        st = GkStats()
        with self._lock:
            self._check(self.lib.gk_wl_features(self.h, int(n_iter), C.byref(st)))
        return st

    def wl_oa_features(self, n_iter):
        st = GkStats()
        with self._lock:
            self._check(self.lib.gk_wl_oa_features(self.h, int(n_iter), C.byref(st)))
        return st

    def nh_features(self, R, bits, count_sensitive, labels0):
        """NeighborhoodHash levels of the packed block; labels0 = int64 hashed level-0 label per vertex, -1 = None."""
        st = GkStats()
        lab = np.ascontiguousarray(labels0, dtype=np.int64)
        with self._lock:
            self._check(self.lib.gk_nh_features(self.h, int(R), int(bits), GK_NH_COUNT_SENSITIVE if count_sensitive else 0,
                                                _ptr(lab), C.byref(st)))
        return st

    def nh_gram(self, n_graphs, n_fit=None, out=None, simt=False, dense_all=False, device_ptr=None, ld=0, stats=None):
        """fp64 NeighborhoodHash matrix: a fresh host array, `out`, `device_ptr` (raw device pointer) or, with
        out=False, left on the device (result_device / fetch)."""
        n_fit = n_graphs if n_fit is None else int(n_fit)
        rows = n_graphs if n_fit == n_graphs else n_graphs - n_fit
        flags = (GK_GRAM_SIMT if simt else 0) | (GK_DENSE_ALL if dense_all else 0)
        K, kptr = None, None
        if device_ptr is not None:
            flags |= GK_OUT_DEVICE
            kptr = C.c_void_p(int(device_ptr))
        elif out is None:
            K = host_matrix(rows, n_fit, np.float64)
            kptr = _ptr(K)
        elif out is not False:
            K = out
            assert K.dtype == np.float64 and K.flags.c_contiguous and K.shape == (rows, n_fit)
            kptr = _ptr(K)
        st = stats if stats is not None else GkStats()
        with self._lock:
            self._check(self.lib.gk_nh_gram(self.h, n_fit, flags, kptr, GK_F64, int(ld), C.byref(st)))
        return K

    def nh_labels(self, level, n_vertices):
        """u64 labels of one level (2^64 - 1 = None)."""
        out = np.empty(n_vertices, dtype=np.uint64)
        with self._lock:
            self._check(self.lib.gk_nh_labels(self.h, int(level), _ptr(out)))
        return out

    def sp_features(self, with_labels=True, keep_dist=False, dijkstra_order=False):
        st = GkStats()
        flags = (GK_SP_WITH_LABELS if with_labels else 0) | (GK_SP_KEEP_DIST if keep_dist else 0)
        flags |= GK_SP_DIJKSTRA_ORDER if dijkstra_order else 0
        with self._lock:
            self._check(self.lib.gk_sp_features(self.h, flags, C.byref(st)))
        return st

    def wl_sp_features(self, n_iter, keep_dist=False, dijkstra_order=True):
        st = GkStats()
        flags = GK_SP_WITH_LABELS | (GK_SP_KEEP_DIST if keep_dist else 0) | (GK_SP_DIJKSTRA_ORDER if dijkstra_order else 0)
        with self._lock:
            self._check(self.lib.gk_wl_sp_features(self.h, int(n_iter), flags, C.byref(st)))
        return st

    def spattr_features(self, dijkstra_order=False):
        st = GkStats()
        with self._lock:
            self._check(self.lib.gk_spattr_features(self.h, GK_SP_DIJKSTRA_ORDER if dijkstra_order else 0, C.byref(st)))
        return st

    def gram(self, n_graphs, n_fit=None, normalize=False, nan_to_num=False, out=None, dtype=np.float64,
             row_range=None, simt=False, full_tiles=False, stats=None, want_diag=True, device_ptr=None, ld=0,
             dense_all=False, dist=False, gather=False):
        """Returns (K, xdiag, ydiag).  K is a fresh C-order numpy array unless
        `out` (host array) or `device_ptr` (raw device pointer) is given."""
        n_fit = n_graphs if n_fit is None else int(n_fit)
        square = n_fit == n_graphs
        rows_total = n_graphs if square else n_graphs - n_fit
        rb, re_ = (0, rows_total) if row_range is None else row_range
        dt = np.dtype(dtype)
        code = GK_F64 if dt == np.float64 else GK_F32
        flags = (GK_NORMALIZE if normalize else 0) | (GK_NAN_TO_NUM if nan_to_num else 0)
        flags |= (GK_GRAM_SIMT if simt else 0) | (GK_FULL_TILES if full_tiles else 0) | (GK_DENSE_ALL if dense_all else 0)
        flags |= (GK_DIST if dist else 0) | (GK_DIST_GATHER if gather else 0)
        K = None
        kptr = None
        if device_ptr is not None:
            flags |= GK_OUT_DEVICE
            kptr = C.c_void_p(int(device_ptr))
        elif out is not None:
            if out is not False:
                K = out
                assert K.dtype == dt and K.flags.c_contiguous and K.shape == (re_ - rb, n_fit)
                kptr = _ptr(K)
        else:
            K = host_matrix(re_ - rb, n_fit, dt)
            kptr = _ptr(K)
        xd = np.empty(n_fit, dtype=np.float64) if want_diag else None
        yd = np.empty(n_graphs - n_fit, dtype=np.float64) if (want_diag and not square) else None
        st = stats if stats is not None else GkStats()
        with self._lock:
            self._check(self.lib.gk_gram(self.h, n_fit, flags, rb, re_, kptr, code, int(ld), _ptr(xd), _ptr(yd),
                                         C.byref(st)))
        return K, xd, yd

    # ---- multi-GPU (one process per GPU; collective calls)
    @staticmethod
    def comm_unique_id():
        """128-byte NCCL id created by one rank; hand it to every rank (torch.distributed, MPI, a file ...)."""
        buf = C.create_string_buffer(128)
        lib = load_library()
        if lib.gk_comm_unique_id(buf) != 0:
            raise GrakelB200Error("gk_comm_unique_id: " + lib.gk_last_error().decode())
        return bytes(buf.raw)

    def comm_init(self, nranks, rank, unique_id):
        buf = C.create_string_buffer(bytes(unique_id), 128)
        self._check(self.lib.gk_comm_init(self.h, int(nranks), int(rank), buf))
        self.nranks, self.rank = int(nranks), int(rank)

    def comm_rows(self, n_rows):
        a, b = C.c_int64(), C.c_int64()
        self._check(self.lib.gk_comm_rows(self.h, int(n_rows), C.byref(a), C.byref(b)))
        return a.value, b.value

    def result_device(self):
        """(device pointer, rows, cols, ld, dtype code) of the library-owned result of the last gram()."""
        p, r, c, ld, dt = _P(), C.c_int64(), C.c_int64(), C.c_int64(), C.c_int32()
        self._check(self.lib.gk_result_device(self.h, C.byref(p), C.byref(r), C.byref(c), C.byref(ld), C.byref(dt)))
        return p.value, r.value, c.value, ld.value, dt.value

    def fetch(self, out):
        code = GK_F64 if out.dtype == np.float64 else GK_F32
        self._check(self.lib.gk_fetch(self.h, _ptr(out), code, out.shape[1]))
        return out

    def wl_labels(self, level, n_vertices):
        out = np.empty(n_vertices, dtype=np.int32)
        with self._lock:
            self._check(self.lib.gk_wl_labels(self.h, int(level), _ptr(out)))
        return out

    def sp_distances(self, g, n):
        out = np.empty((n, n), dtype=np.float64)
        with self._lock:
            self._check(self.lib.gk_sp_distances(self.h, int(g), _ptr(out)))
        return out

    def wl_fit_transform_raw(self, graph_ptr, row_ptr, col_idx, labels, n_iter, out, normalize=False):
        """One C call, host buffers in / host buffer out (the e2e path of bench.py)."""
        st = GkStats()
        code = GK_F64 if out.dtype == np.float64 else GK_F32
        flags = (GK_NORMALIZE | GK_NAN_TO_NUM) if normalize else 0
        with self._lock:
            self._check(self.lib.gk_wl_fit_transform(self.h, len(graph_ptr) - 1, _ptr(graph_ptr), _ptr(row_ptr),
                                                     _ptr(col_idx), _ptr(labels), int(n_iter), flags, _ptr(out), code,
                                                     out.shape[1], None, C.byref(st)))
        return st

    def wl_gram(self, n_iter, out=None, dtype=np.float64, device_ptr=None, ld=0, dense_all=False, want_diag=False,
                stats=None):
        """WL features + square Gram of the packed block in ONE C call (gk_wl_gram): the asynchronous pass -- one host
        synchronisation, head/tail decision on the device -- when it applies, else gk_wl_features + gk_gram.
        Returns (K, xdiag, stats); `out` / `device_ptr` as in gram()."""
        n = self.n_graphs
        dt = np.dtype(dtype)
        code = GK_F64 if dt == np.float64 else GK_F32
        flags = GK_DENSE_ALL if dense_all else 0
        K, kptr = None, None
        if device_ptr is not None:
            flags |= GK_OUT_DEVICE
            kptr = C.c_void_p(int(device_ptr))
        elif out is not None:
            if out is not False:
                K = out
                assert K.dtype == dt and K.flags.c_contiguous and K.shape == (n, n)
                kptr = _ptr(K)
        else:
            K = host_matrix(n, n, dt)
            kptr = _ptr(K)
        xd = np.empty(n, dtype=np.float64) if want_diag else None
        st = stats if stats is not None else GkStats()
        with self._lock:
            self._check(self.lib.gk_wl_gram(self.h, int(n_iter), flags, kptr, code, int(ld), _ptr(xd), C.byref(st)))
        return K, xd, st

    def selftest_gram(self, counts):
        counts = np.ascontiguousarray(counts, dtype=np.uint16)
        n, d = counts.shape
        a = np.empty((n, n), dtype=np.float64)
        b = np.empty((n, n), dtype=np.float64)
        with self._lock:
            self._check(self.lib.gk_selftest_gram(self.h, n, d, _ptr(counts), _ptr(a), _ptr(b)))
        return a, b

    def selftest_deliver(self, src, mode=0, diag=None, nan_to_num=False):
        """Host-only: fp32 matrix -> float64 through the delivery code of gk_gram (no device work).  mode 0: upper
        triangle as fp32, 1: all rows, 2: all rows + normalisation, 3: upper triangle band-packed as u16."""
        src = np.ascontiguousarray(src, dtype=np.float32)
        rows, cols = src.shape
        dst = np.full((rows, cols), np.nan)
        dg = None if diag is None else np.ascontiguousarray(diag, dtype=np.float64)
        self._check(self.lib.gk_selftest_deliver(int(mode), rows, cols, _ptr(src), _ptr(dg), 1 if nan_to_num else 0, _ptr(dst)))
        return dst

    def event_record(self, slot):
        self._check(self.lib.gk_event_record(self.h, slot))

    def event_elapsed(self, a, b):
        ms = C.c_float()
        self._check(self.lib.gk_event_elapsed(self.h, a, b, C.byref(ms)))
        return ms.value

    def profiler_range(self, on):
        self._check(self.lib.gk_profiler_range(1 if on else 0))

    def sync(self):
        self._check(self.lib.gk_sync(self.h))


_engines = {}
_engines_lock = threading.Lock()
_default_device = None


def set_default_device(device):
    """Device ordinal new estimator runs use (default: GRAKEL_B200_DEVICE, else LOCAL_RANK, else 0)."""
    global _default_device
    _default_device = None if device is None else int(device)


def default_device():
    if _default_device is not None:
        return _default_device
    return int(os.environ.get("GRAKEL_B200_DEVICE", os.environ.get("LOCAL_RANK", "0")))


def get_engine(device=None):
    """The process-wide engine of a device (bench / tools / tests that drive the C-ABI step by step)."""
    if device is None:
        device = default_device()
    with _engines_lock:
        e = _engines.get(device)
        if e is None:
            e = Engine(device)
            _engines[device] = e
        return e


class _EnginePool:
    """Engines of one device handed out to estimator runs: a run holds one engine (one handle + stream) for its
    pack -> features -> gram sequence, so estimators used from several Python threads (sklearn's threading
    backend) run concurrently on separate streams instead of serialising on one handle.  At most
    GRAKEL_B200_MAX_ENGINES (default 4) engines per device; further threads wait for a free one."""

    def __init__(self, device):
        self.device = device
        self.free = []
        self.count = 0
        self.cv = threading.Condition()
        self.limit = max(1, int(os.environ.get("GRAKEL_B200_MAX_ENGINES", "4")))

    def acquire(self):
        with self.cv:
            while True:
                if self.free:
                    return self.free.pop()
                if self.count < self.limit:
                    self.count += 1
                    break
                self.cv.wait()
        try:
            # the first engine of the pool is the process-wide one, so step-by-step users share its buffers
            return get_engine(self.device) if self.count == 1 else Engine(self.device)
        except Exception:
            with self.cv:
                self.count -= 1
                self.cv.notify()
            raise

    def release(self, eng):
        with self.cv:
            self.free.append(eng)
            self.cv.notify()


_pools = {}


class engine:
    """`with engine(device) as eng:` -- exclusive use of one engine of the device for the duration."""

    def __init__(self, device=None):
        self.device = default_device() if device is None else int(device)
        self.eng = None

    def __enter__(self):
        with _engines_lock:
            pool = _pools.get(self.device)
            if pool is None:
                pool = _pools[self.device] = _EnginePool(self.device)
        self.pool = pool
        self.eng = pool.acquire()
        self.eng._lock.acquire()
        return self.eng

    def __exit__(self, *exc):
        self.eng._lock.release()
        self.pool.release(self.eng)
        return False
