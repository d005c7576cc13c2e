"""ctypes bindings for the oracle libraries (TEST INFRASTRUCTURE).

Only tests/, ``__graft_entry__.smoke()`` and bench.py's CPU arms import this module. The product
package ``usearch_b200`` never does.

* :class:`RefIndex`  — the unmodified reference (oracle/_ref/libusearch_ref_*.so, built from
  /root/reference by oracle/build.py).
* :class:`PortIndex`, :func:`port_exact_search` — the plain-C restatement (oracle/liboracle.so).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

HERE = os.path.dirname(os.path.abspath(__file__))

# enum values from /root/reference/include/usearch/index_plugins.hpp:113-159
METRIC = {"ip": ord("i"), "cos": ord("c"), "l2sq": ord("e"), "hamming": ord("b"),
          "tanimoto": ord("t"), "sorensen": ord("s"), "jaccard": ord("j")}
SCALAR = {"b1": 1, "bf16": 4, "f64": 10, "f32": 11, "f16": 12, "i8": 23}
SCALAR_NP = {"b1": np.uint8, "bf16": np.uint16, "f32": np.float32, "f16": np.float16, "i8": np.int8}

_u64p = C.POINTER(C.c_uint64)
_f32p = C.POINTER(C.c_float)


def bytes_per_vector(dims: int, scalar: str) -> int:
    bits = {"b1": 1, "i8": 8, "f16": 16, "bf16": 16, "f32": 32, "f64": 64}[scalar]
    return (dims * bits + 7) // 8


def _ptr(a: np.ndarray, typ=C.c_void_p):
    return a.ctypes.data_as(typ)


def _check(err: C.c_char_p):
    if err.value:
        raise RuntimeError(err.value.decode())


_ref_libs: dict[str, C.CDLL] = {}


def ref_lib(flavour: str = "parity") -> C.CDLL | None:
    if flavour in _ref_libs:
        return _ref_libs[flavour]
    path = _build.build_reference(flavour)
    if path is None or not os.path.exists(path):
        return None
    lib = C.CDLL(path)
    lib.ref_make.restype = C.c_void_p
    lib.ref_make.argtypes = [C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(C.c_char_p)]
    lib.ref_make_empty.restype = C.c_void_p
    lib.ref_free.argtypes = [C.c_void_p]
    for name in ("ref_size", "ref_dimensions", "ref_connectivity", "ref_max_level", "ref_bytes_per_vector",
                 "ref_expansion_search", "ref_serialized_length"):
        getattr(lib, name).restype = C.c_size_t
        getattr(lib, name).argtypes = [C.c_void_p]
    lib.ref_change_expansion_search.argtypes = [C.c_void_p, C.c_size_t]
    lib.ref_metric_kind.argtypes = [C.c_void_p]
    lib.ref_scalar_kind.argtypes = [C.c_void_p]
    lib.ref_isa_name.restype = C.c_char_p
    lib.ref_isa_name.argtypes = [C.c_void_p]
    lib.ref_pin_metric.argtypes = [C.c_void_p, C.c_int]
    lib.ref_distance.restype = C.c_float
    lib.ref_distance.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.ref_add_many.restype = C.c_size_t
    lib.ref_add_many.argtypes = [C.c_void_p, _u64p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(C.c_char_p)]
    lib.ref_remove.restype = C.c_size_t
    lib.ref_remove.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_char_p)]
    lib.ref_save_buffer.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_char_p)]
    lib.ref_load_buffer.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_char_p)]
    lib.ref_view_buffer.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_char_p)]
    lib.ref_save_path.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_char_p)]
    lib.ref_load_path.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_char_p)]
    lib.ref_search_many.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int,
                                    _u64p, _f32p, _u64p, _u64p, _u64p, C.POINTER(C.c_char_p)]
    lib.ref_filtered_search_many_f32.argtypes = [C.c_void_p, _f32p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, _u64p,
                                                 C.c_size_t, _u64p, _f32p, _u64p, _u64p, _u64p, C.POINTER(C.c_char_p)]
    lib.ref_cluster_many.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, _u64p, _f32p, _u64p, _u64p,
                                     C.POINTER(C.c_char_p)]
    lib.ref_exact_search.restype = C.c_int
    lib.ref_exact_search.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.c_int,
                                     C.c_size_t, C.c_size_t, C.c_int, _u64p, _f32p]
    lib.ref_cast_from_f32.restype = C.c_size_t
    lib.ref_cast_from_f32.argtypes = [C.c_int, _f32p, C.c_size_t, C.c_void_p]
    lib.ref_hardware_threads.restype = C.c_size_t
    _ref_libs[flavour] = lib
    return lib


class RefIndex:
    """The reference ``index_dense_gt<u64,u32>`` behind oracle/ref_driver.cpp."""

    def __init__(self, flavour: str = "parity", *, metric: str | None = None, scalar: str = "f32", dims: int = 0,
                 connectivity: int = 16, expansion_add: int = 128, expansion_search: int = 64):
        self.lib = ref_lib(flavour)
        if self.lib is None:
            raise RuntimeError("reference library unavailable (oracle/_ref not built and /root/reference absent)")
        self.flavour = flavour
        err = C.c_char_p()
        if metric is None:
            self.h = C.c_void_p(self.lib.ref_make_empty())
        else:
            self.h = C.c_void_p(self.lib.ref_make(METRIC[metric], SCALAR[scalar], dims, connectivity, expansion_add,
                                                  expansion_search, C.byref(err)))
            _check(err)
        self._keep = None

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.ref_free(self.h)
            self.h = None

    size = property(lambda s: s.lib.ref_size(s.h))
    dims = property(lambda s: s.lib.ref_dimensions(s.h))
    connectivity = property(lambda s: s.lib.ref_connectivity(s.h))
    max_level = property(lambda s: s.lib.ref_max_level(s.h))
    bytes_per_vector = property(lambda s: s.lib.ref_bytes_per_vector(s.h))
    isa_name = property(lambda s: s.lib.ref_isa_name(s.h).decode())

    def pin_metric(self, pinned: bool = True) -> None:
        rc = self.lib.ref_pin_metric(self.h, 1 if pinned else 0)
        if rc != 0:
            raise RuntimeError(f"ref_pin_metric failed ({rc})")

    def change_expansion_search(self, ef: int) -> None:
        self.lib.ref_change_expansion_search(self.h, ef)

    def distance(self, a: np.ndarray, b: np.ndarray) -> float:
        a = np.ascontiguousarray(a)
        b = np.ascontiguousarray(b)
        return float(self.lib.ref_distance(self.h, _ptr(a), _ptr(b)))

    def add(self, keys: np.ndarray, vectors: np.ndarray, threads: int = 1) -> int:
        keys = np.ascontiguousarray(keys, dtype=np.uint64)
        vectors = np.ascontiguousarray(vectors)
        err = C.c_char_p()
        n = self.lib.ref_add_many(self.h, _ptr(keys, _u64p), _ptr(vectors), len(keys), vectors.strides[0], threads,
                                  C.byref(err))
        _check(err)
        return n

    def remove(self, key: int) -> int:
        err = C.c_char_p()
        n = self.lib.ref_remove(self.h, key, C.byref(err))
        _check(err)
        return n

    def save(self) -> np.ndarray:
        n = self.lib.ref_serialized_length(self.h)
        buf = np.empty(n, dtype=np.uint8)
        err = C.c_char_p()
        self.lib.ref_save_buffer(self.h, _ptr(buf), n, C.byref(err))
        _check(err)
        return buf

    def load(self, blob: np.ndarray) -> None:
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        err = C.c_char_p()
        self.lib.ref_load_buffer(self.h, _ptr(blob), blob.size, C.byref(err))
        _check(err)

    def view(self, blob: np.ndarray) -> None:
        """`view` over the caller's buffer: nothing is copied, the buffer is kept alive by this object."""
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        err = C.c_char_p()
        self.lib.ref_view_buffer(self.h, _ptr(blob), blob.size, C.byref(err))
        _check(err)
        self._keep = blob

    def save_path(self, path: str) -> None:
        err = C.c_char_p()
        self.lib.ref_save_path(self.h, path.encode(), C.byref(err))
        _check(err)

    def load_path(self, path: str) -> None:
        err = C.c_char_p()
        self.lib.ref_load_path(self.h, path.encode(), C.byref(err))
        _check(err)

    def search(self, queries: np.ndarray, k: int, threads: int = 1, exact: bool = False, counters: bool = True):
        queries = np.ascontiguousarray(queries)
        nq = queries.shape[0]
        keys = np.zeros((nq, k), dtype=np.uint64)
        dist = np.zeros((nq, k), dtype=np.float32)
        counts = np.zeros(nq, dtype=np.uint64)
        computed = np.zeros(nq, dtype=np.uint64)
        visited = np.zeros(nq, dtype=np.uint64)
        err = C.c_char_p()
        self.lib.ref_search_many(self.h, _ptr(queries), nq, queries.strides[0], k, threads, int(exact),
                                 _ptr(keys, _u64p), _ptr(dist, _f32p), _ptr(counts, _u64p),
                                 _ptr(computed, _u64p) if counters else None,
                                 _ptr(visited, _u64p) if counters else None, C.byref(err))
        _check(err)
        return keys, dist, counts, computed, visited


def _ref_filtered_search(self, queries: np.ndarray, k: int, allowed_keys: np.ndarray, threads: int = 1):
    queries = np.ascontiguousarray(queries, dtype=np.float32)
    allowed = np.sort(np.ascontiguousarray(allowed_keys, dtype=np.uint64))
    nq = queries.shape[0]
    keys = np.zeros((nq, k), dtype=np.uint64)
    dist = np.zeros((nq, k), dtype=np.float32)
    counts, computed, visited = (np.zeros(nq, dtype=np.uint64) for _ in range(3))
    err = C.c_char_p()
    self.lib.ref_filtered_search_many_f32(self.h, _ptr(queries, _f32p), nq, queries.strides[0], k, threads,
                                          _ptr(allowed, _u64p), allowed.size, _ptr(keys, _u64p), _ptr(dist, _f32p),
                                          _ptr(counts, _u64p), _ptr(computed, _u64p), _ptr(visited, _u64p), C.byref(err))
    _check(err)
    return keys, dist, counts, computed, visited


RefIndex.filtered_search = _ref_filtered_search


def _ref_cluster(self, queries: np.ndarray, level: int):
    """index_dense_gt::cluster(vector, level) per row: (keys, distances, computed_distances, visited_members)."""
    queries = np.ascontiguousarray(queries)
    nq = queries.shape[0]
    keys = np.zeros(nq, dtype=np.uint64)
    dist = np.zeros(nq, dtype=np.float32)
    computed = np.zeros(nq, dtype=np.uint64)
    visited = np.zeros(nq, dtype=np.uint64)
    err = C.c_char_p()
    self.lib.ref_cluster_many(self.h, _ptr(queries), nq, queries.strides[0], level, _ptr(keys, _u64p), _ptr(dist, _f32p),
                              _ptr(computed, _u64p), _ptr(visited, _u64p), C.byref(err))
    _check(err)
    return keys, dist, computed, visited


RefIndex.cluster = _ref_cluster

def ref_exact_search(dataset: np.ndarray, queries: np.ndarray, k: int, *, metric: str, scalar: str, dims: int,
                     pinned: bool = True, flavour: str = "parity"):
    """exact_search_t of the reference over raw matrices (rows in `scalar` kind); keys are dataset row numbers."""
    lib = ref_lib(flavour)
    dataset = np.ascontiguousarray(dataset)
    queries = np.ascontiguousarray(queries)
    nq = queries.shape[0]
    keys = np.zeros((nq, k), dtype=np.uint64)
    dist = np.zeros((nq, k), dtype=np.float32)
    rc = lib.ref_exact_search(dataset.ctypes.data_as(C.c_void_p), dataset.shape[0], dataset.strides[0],
                              queries.ctypes.data_as(C.c_void_p), nq, queries.strides[0], METRIC[metric],
                              SCALAR[scalar], dims, k, int(pinned), _ptr(keys, _u64p), _ptr(dist, _f32p))
    if rc:
        raise RuntimeError(f"ref_exact_search failed: {rc}")
    return keys, dist


_port_lib: C.CDLL | None = None


def port_lib() -> C.CDLL:
    global _port_lib
    if _port_lib is not None:
        return _port_lib
    lib = C.CDLL(_build.build_port())
    lib.oracle_open.restype = C.c_void_p
    lib.oracle_open.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_char_p)]
    lib.oracle_close.argtypes = [C.c_void_p]
    for name in ("oracle_size", "oracle_dimensions", "oracle_connectivity", "oracle_max_level",
                 "oracle_bytes_per_vector"):
        getattr(lib, name).restype = C.c_size_t
        getattr(lib, name).argtypes = [C.c_void_p]
    lib.oracle_metric_kind.argtypes = [C.c_void_p]
    lib.oracle_scalar_kind.argtypes = [C.c_void_p]
    lib.oracle_change_expansion_search.argtypes = [C.c_void_p, C.c_size_t]
    lib.oracle_distance.restype = C.c_float
    lib.oracle_distance.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.oracle_search_many.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int,
                                       _u64p, _f32p, _u64p, _u64p, _u64p]
    lib.oracle_filtered_search_many.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int,
                                                _u64p, C.c_size_t, _u64p, _f32p, _u64p, _u64p, _u64p]
    lib.oracle_exact_search.restype = C.c_int
    lib.oracle_exact_search.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t, C.c_int,
                                        C.c_int, C.c_size_t, C.c_size_t, _u64p, _f32p]
    lib.oracle_cluster_many.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, _u64p, _f32p, _u64p, _u64p]
    lib.oracle_cast_from_f32.restype = C.c_size_t
    lib.oracle_cast_from_f32.argtypes = [C.c_int, _f32p, C.c_size_t, C.c_void_p]
    _port_lib = lib
    return lib


class PortIndex:
    """The plain-C restatement over a serialised v2 blob (borrowed, kept alive here)."""

    def __init__(self, blob: np.ndarray, expansion_search: int = 64):
        self.lib = port_lib()
        self.blob = np.ascontiguousarray(blob, dtype=np.uint8)
        err = C.c_char_p()
        self.h = C.c_void_p(self.lib.oracle_open(_ptr(self.blob), self.blob.size, C.byref(err)))
        _check(err)
        self.lib.oracle_change_expansion_search(self.h, expansion_search)

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.oracle_close(self.h)
            self.h = None

    size = property(lambda s: s.lib.oracle_size(s.h))
    dims = property(lambda s: s.lib.oracle_dimensions(s.h))
    connectivity = property(lambda s: s.lib.oracle_connectivity(s.h))
    max_level = property(lambda s: s.lib.oracle_max_level(s.h))
    bytes_per_vector = property(lambda s: s.lib.oracle_bytes_per_vector(s.h))

    def change_expansion_search(self, ef: int) -> None:
        self.lib.oracle_change_expansion_search(self.h, ef)

    def distance(self, a: np.ndarray, b: np.ndarray) -> float:
        a = np.ascontiguousarray(a)
        b = np.ascontiguousarray(b)
        return float(self.lib.oracle_distance(self.h, _ptr(a), _ptr(b)))

    def search(self, queries: np.ndarray, k: int, threads: int = 1, exact: bool = False):
        queries = np.ascontiguousarray(queries)
        nq = queries.shape[0]
        keys = np.zeros((nq, k), dtype=np.uint64)
        dist = np.zeros((nq, k), dtype=np.float32)
        counts = np.zeros(nq, dtype=np.uint64)
        computed = np.zeros(nq, dtype=np.uint64)
        visited = np.zeros(nq, dtype=np.uint64)
        self.lib.oracle_search_many(self.h, _ptr(queries), nq, queries.strides[0] if nq else 0, k, threads,
                                    int(exact), _ptr(keys, _u64p), _ptr(dist, _f32p), _ptr(counts, _u64p),
                                    _ptr(computed, _u64p), _ptr(visited, _u64p))
        return keys, dist, counts, computed, visited

    def filtered_search(self, queries: np.ndarray, k: int, allowed_keys: np.ndarray, threads: int = 1):
        """filtered_search with the predicate "key in allowed_keys"."""
        queries = np.ascontiguousarray(queries)
        allowed = np.sort(np.ascontiguousarray(allowed_keys, dtype=np.uint64))
        nq = queries.shape[0]
        keys = np.zeros((nq, k), dtype=np.uint64)
        dist = np.zeros((nq, k), dtype=np.float32)
        counts, computed, visited = (np.zeros(nq, dtype=np.uint64) for _ in range(3))
        self.lib.oracle_filtered_search_many(self.h, _ptr(queries), nq, queries.strides[0] if nq else 0, k, threads, 0,
                                             _ptr(allowed, _u64p), allowed.size, _ptr(keys, _u64p), _ptr(dist, _f32p),
                                             _ptr(counts, _u64p), _ptr(computed, _u64p), _ptr(visited, _u64p))
        return keys, dist, counts, computed, visited

    def cluster(self, queries: np.ndarray, level: int):
        queries = np.ascontiguousarray(queries)
        nq = queries.shape[0]
        keys = np.zeros(nq, dtype=np.uint64)
        dist = np.zeros(nq, dtype=np.float32)
        computed = np.zeros(nq, dtype=np.uint64)
        visited = np.zeros(nq, dtype=np.uint64)
        self.lib.oracle_cluster_many(self.h, _ptr(queries), nq, queries.strides[0] if nq else 0, level, _ptr(keys, _u64p),
                                     _ptr(dist, _f32p), _ptr(computed, _u64p), _ptr(visited, _u64p))
        return keys, dist, computed, visited


def port_exact_search(dataset: np.ndarray, queries: np.ndarray, k: int, *, metric: str, scalar: str, dims: int):
    """The plain-C restatement of exact_search_t over raw matrices (pinned metrics); keys are dataset row numbers."""
    lib = port_lib()
    dataset = np.ascontiguousarray(dataset)
    queries = np.ascontiguousarray(queries)
    nq = queries.shape[0]
    keys = np.zeros((nq, k), dtype=np.uint64)
    dist = np.zeros((nq, k), dtype=np.float32)
    rc = lib.oracle_exact_search(_ptr(dataset), dataset.shape[0], dataset.strides[0], _ptr(queries), nq, queries.strides[0],
                                 METRIC[metric], SCALAR[scalar], dims, k, _ptr(keys, _u64p), _ptr(dist, _f32p))
    if rc:
        raise RuntimeError(f"oracle_exact_search failed: {rc}")
    return keys, dist
