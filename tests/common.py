"""Shared helpers for the parity tests: build an index, hand the SAME serialised graph to the oracle(s) and
to the GPU backend, compare bit-for-bit."""
from __future__ import annotations

import hashlib
import io
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import bindings  # noqa: E402
from usearch_b200 import datagen  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def have_reference() -> bool:
    return bindings.ref_lib("parity") is not None


def make_collection(n: int, d: int, scalar: str, nq: int, *, seed: int = 42, rank: int = 16, iid: bool = False):
    if scalar == "b1":
        base = datagen.latent(n, d, seed=seed, rank=min(rank, d))
        queries = datagen.latent(nq, d, seed=seed + 1, rank=min(rank, d))
    elif iid:
        base = np.random.default_rng(seed).standard_normal((n, d), dtype=np.float32)
        queries = np.random.default_rng(seed + 1).standard_normal((nq, d), dtype=np.float32)
    else:
        base = datagen.latent(n, d, seed=seed, rank=min(rank, d))
        queries = datagen.latent(nq, d, seed=seed + 1, rank=min(rank, d))
    return datagen.to_scalar(base, scalar), datagen.to_scalar(queries, scalar)


def build_reference_blob(base: np.ndarray, metric: str, scalar: str, d: int, connectivity: int, expansion_add: int = 128,
                         threads: int = 8, keys: np.ndarray | None = None):
    ref = bindings.RefIndex("parity", metric=metric, scalar=scalar, dims=d, connectivity=connectivity,
                            expansion_add=expansion_add, expansion_search=64)
    keys = np.arange(len(base), dtype=np.uint64) if keys is None else keys
    ref.add(keys, base, threads=threads)
    return ref, ref.save()


def build_graph_blob(base: np.ndarray, metric: str, scalar: str, d: int, connectivity: int, expansion_add: int = 128,
                     keys: np.ndarray | None = None, removed=()) -> np.ndarray:
    """The collection linked into a graph by this project's GPU builder, the members in `removed` deleted by this
    project's `remove`, serialised in the v2 format. Search parity does not depend on who built the graph: the GPU search
    and the plain-C oracle (itself pinned to the reference's outputs by tests/golden) are handed the same serialised
    file. A wrong tombstone written by `remove` would be read the same way by both; tombstones written by the reference
    are covered by the golden fixture ip_f32_n1500_d48_removed and reference_cases.npz's small cases."""
    from usearch_b200.index import Index
    index = Index(ndim=d, metric=metric, dtype=scalar, connectivity=connectivity, expansion_add=expansion_add)
    index.add(np.arange(len(base), dtype=np.uint64) if keys is None else keys, base)
    for key in removed:
        assert index.remove(int(key)) == 1
    return index.save()


def assert_same_results(a, b, what: str = ""):
    """(keys, distances, counts, computed, visited) tuples must agree bit-for-bit."""
    ak, ad, ac = a[0], a[1], a[2]
    bk, bd, bc = b[0], b[1], b[2]
    assert np.array_equal(ac.astype(np.uint64), bc.astype(np.uint64)), f"{what}: counts differ"
    bad = np.nonzero((ak != bk).any(axis=1))[0]
    assert bad.size == 0, f"{what}: labels differ for {bad.size} queries, first {bad[:5]}"
    assert np.array_equal(ad.view(np.uint32), bd.view(np.uint32)), f"{what}: distance bits differ"
    if len(a) > 3 and len(b) > 3 and a[3] is not None and b[3] is not None:
        assert np.array_equal(np.asarray(a[3], dtype=np.uint64), np.asarray(b[3], dtype=np.uint64)), f"{what}: computed_distances differ"
        assert np.array_equal(np.asarray(a[4], dtype=np.uint64), np.asarray(b[4], dtype=np.uint64)), f"{what}: visited_members differ"


# ---- tests/golden/reference_cases.npz (made by tests/golden/make_golden_reference_cases.py) ----------------------------
GOLDEN_NQ = 24
GOLDEN_SMALL_CASES = 20  # the first of small_random_cases(): every scalar kind twice
GOLDEN_SEARCH_CASES = [
    # name, metric, scalar, n, d, M, ef, k
    ("l2sq_f32", "l2sq", "f32", 200, 24, 16, 64, 10),
    ("cos_f32_ef16", "cos", "f32", 200, 100, 8, 16, 10),    # ef barely above k
    ("ip_f32_absurd", "ip", "f32", 200, 17, 3, 5, 10),      # M=3, ef < k (cpp/test.cpp:820-865)
    ("cos_f16", "cos", "f16", 200, 64, 16, 64, 10),
    ("l2sq_bf16", "l2sq", "bf16", 200, 40, 16, 64, 10),
    ("ip_i8", "ip", "i8", 200, 128, 16, 64, 10),
    ("cos_i8", "cos", "i8", 200, 100, 16, 64, 10),
    ("l2sq_i8", "l2sq", "i8", 200, 100, 16, 64, 10),
    ("hamming_b1_d64", "hamming", "b1", 300, 64, 16, 64, 10),   # 64-bit codes: ties everywhere
    ("hamming_b1_m64", "hamming", "b1", 200, 256, 64, 64, 20),
    ("sorensen_b1", "sorensen", "b1", 200, 128, 8, 32, 5),
]
GOLDEN_CLUSTER_CASES = [("cluster_cos_f32", "cos", "f32", 500, 32, 4), ("cluster_hamming_b1", "hamming", "b1", 500, 64, 4)]


def digest(*arrays) -> str:
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def strip_vectors(blob: np.ndarray) -> np.ndarray:
    """A serialised v2 index without its vector matrix (the graph alone); `with_vectors` puts the matrix back."""
    rows, cols = (int(x) for x in blob[:8].view(np.uint32))
    return np.concatenate([blob[:8], blob[8 + rows * cols:]])


def with_vectors(graph: np.ndarray, vectors: np.ndarray) -> np.ndarray:
    rows, cols = (int(x) for x in graph[:8].view(np.uint32))
    matrix = np.ascontiguousarray(vectors).view(np.uint8).reshape(-1)
    assert matrix.size == rows * cols, (matrix.size, rows, cols)
    return np.concatenate([graph[:8], matrix, graph[8:]])


def golden_case(name: str):
    """One case of tests/golden/reference_cases.npz (each case is an uncompressed .npz stored as one uint8 array)."""
    with np.load(os.path.join(GOLDEN, "reference_cases.npz")) as outer:
        return np.load(io.BytesIO(outer[name].tobytes()))


def native_metric_rows():
    """(metric, scalar, dims, rows) of the pinned-vs-native metric comparison: i.i.d. Gaussian rows, seed 7."""
    rng = np.random.default_rng(7)
    for metric, scalar, d in [("l2sq", "f32", 768), ("ip", "f32", 100), ("cos", "f32", 768), ("ip", "i8", 1024),
                              ("l2sq", "i8", 100), ("hamming", "b1", 256), ("tanimoto", "b1", 200)]:
        yield metric, scalar, d, datagen.to_scalar(rng.standard_normal((64, d), dtype=np.float32), scalar)


def small_random_cases(count: int = 40):
    """Seeded random configurations at the small end: n from 1, k > n, ef < k, removed members, a duplicate vector, every
    scalar kind."""
    rng = np.random.default_rng(2026)
    kinds = [("l2sq", "f32"), ("cos", "f32"), ("ip", "f32"), ("cos", "f16"), ("l2sq", "bf16"), ("ip", "i8"), ("cos", "i8"),
             ("hamming", "b1"), ("tanimoto", "b1"), ("sorensen", "b1")]
    for case in range(count):
        metric, scalar = kinds[case % len(kinds)]
        n = int(rng.integers(1, 200))
        d = int(rng.integers(1, 6)) * 8 if scalar == "b1" else int(rng.integers(1, 41))
        m = int(rng.integers(2, 9))
        ef = int(rng.integers(1, 40))
        k = int(rng.integers(1, 25))
        base, q = make_collection(n, d, scalar, 16, seed=100 + case, rank=min(4, d))
        if n > 4:
            base[n // 2] = base[0]                                  # a duplicate: equal distances
        keys = rng.permutation(np.arange(10 * n, dtype=np.uint64))[:n]
        expansion_add = int(rng.integers(2, 40))
        removed = keys[:int(rng.integers(0, max(1, n // 3)))]
        yield dict(metric=metric, scalar=scalar, n=n, d=d, m=m, ef=ef, k=k, base=base, q=q, keys=keys,
                   expansion_add=expansion_add, removed=removed)
