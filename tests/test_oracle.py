"""CPU tests that PIN the oracle: the plain-C restatement (oracle/hnsw_oracle.c) against
  (a) the committed golden fixtures produced by the unmodified reference (tests/golden/make_golden*.py),
  (b) the tiny known-answer vectors the reference's own test-suites hold,
  (c) the live reference library when oracle/_ref is available (the same configurations, smaller, are in (a))."""
import glob
import os

import numpy as np
import pytest

import common
from oracle import bindings
from usearch_b200 import v2format

FIXTURES = sorted(glob.glob(os.path.join(common.GOLDEN, "*_n*.npz")))


def ulp_distance(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    ai = a.view(np.int32).astype(np.int64)
    bi = b.view(np.int32).astype(np.int64)
    return np.abs(ai - bi)


@pytest.mark.parametrize("path", FIXTURES, ids=[os.path.basename(p)[:-4] for p in FIXTURES])
def test_port_matches_golden(path):
    g = np.load(path)
    port = bindings.PortIndex(g["blob"], int(g["ef"]))
    keys, dist, counts, computed, visited = port.search(g["queries"], int(g["k"]), threads=4)
    # pinned arithmetic: everything the reference returned, bit for bit
    assert np.array_equal(counts, g["counts_pinned"])
    assert np.array_equal(keys, g["keys_pinned"])
    assert np.array_equal(dist.view(np.uint32), g["distances_pinned"].view(np.uint32))
    assert np.array_equal(computed, g["computed_pinned"])
    assert np.array_equal(visited, g["visited_pinned"])
    # the reference's NATIVE SimSIMD dispatch on the generating host: same labels, distances <= 1 ULP,
    # except i8/f16-style cosine whose native kernel uses the 12-bit rsqrt_ps (not among the fixtures)
    assert np.array_equal(keys, g["keys_native"])
    found = np.arange(keys.shape[1])[None, :] < counts[:, None]
    assert ulp_distance(dist, g["distances_native"])[found].max() <= 1


def test_golden_has_padding_and_removed_entries():
    g = np.load(os.path.join(common.GOLDEN, "ip_f32_n1500_d48_removed.npz"))
    graph = v2format.loads(g["blob"])
    assert (graph.keys == v2format.FREE_KEY).sum() == 150
    assert not np.isin(g["keys_pinned"], [v2format.FREE_KEY]).any()


def _tiny(metric, scalar, vectors, keys, dims):
    """Fully connected single-level graph over a handful of vectors."""
    n = len(keys)
    nb = [[[j for j in range(n) if j != i]] for i in range(n)]
    graph = v2format.Graph(metric, scalar, dims, 2 if n <= 3 else n, max(4, 2 * n), np.asarray(vectors), np.asarray(keys, dtype=np.uint64),
                           np.zeros(n, dtype=np.int16), nb, 0, 0)
    return v2format.dumps(graph)


def test_known_answers_from_reference_tests():
    # javascript/usearch.test.js:60-84 — l2sq is NOT square-rooted
    blob = _tiny("l2sq", "f32", np.array([[10, 20], [10, 25]], dtype=np.float32), [15, 16], 2)
    keys, dist, counts, *_ = bindings.PortIndex(blob).search(np.array([[13, 14]], dtype=np.float32), 2)
    assert keys.tolist() == [[15, 16]] and dist.tolist() == [[45.0, 130.0]] and counts.tolist() == [2]
    # golang/lib_test.go:835-877 — cos of orthogonal unit vectors is 1, l2sq is 2, i8 l2sq {10,0,0}/{0,10,0} = 200
    blob = _tiny("cos", "f32", np.array([[1, 0, 0], [0, 1, 0]], dtype=np.float32), [1, 2], 3)
    _, dist, *_ = bindings.PortIndex(blob).search(np.array([[1, 0, 0]], dtype=np.float32), 2)
    assert dist.tolist() == [[0.0, 1.0]]
    blob = _tiny("l2sq", "i8", np.array([[10, 0, 0], [0, 10, 0]], dtype=np.int8), [1, 2], 3)
    _, dist, *_ = bindings.PortIndex(blob).search(np.array([[10, 0, 0]], dtype=np.int8), 2)
    assert dist.tolist() == [[0.0, 200.0]]
    # cpp/test.cpp:1071-1099 — 1-D l2sq keeps exact key order 42, 43, 44
    blob = _tiny("l2sq", "f32", np.array([[10.1], [10.2], [10.3]], dtype=np.float32), [42, 43, 44], 1)
    keys, *_ = bindings.PortIndex(blob).search(np.array([[10.0]], dtype=np.float32), 3)
    assert keys.tolist() == [[42, 43, 44]]


def test_edge_cases_port():
    # empty index: count 0, padding with key 0 and a signalling NaN (index.hpp:2715-2720)
    empty = v2format.dumps(v2format.Graph("cos", "f32", 8, 16, 32, np.zeros((0, 32), np.uint8), np.zeros(0, np.uint64),
                                          np.zeros(0, np.int16), [], 0, 0))
    keys, dist, counts, *_ = bindings.PortIndex(empty).search(np.ones((2, 8), dtype=np.float32), 3)
    assert counts.tolist() == [0, 0] and (keys == 0).all() and (dist.view(np.uint32) == 0x7FA00000).all()
    # fewer members than k: short rows are padded
    blob = _tiny("l2sq", "f32", np.array([[0.0], [1.0]], dtype=np.float32), [7, 8], 1)
    keys, dist, counts, *_ = bindings.PortIndex(blob).search(np.array([[0.25]], dtype=np.float32), 5)
    assert counts.tolist() == [2] and keys[0, :2].tolist() == [7, 8] and (keys[0, 2:] == 0).all()
    assert np.isnan(dist[0, 2:]).all()


@pytest.mark.skipif(not common.have_reference(), reason="oracle/_ref not built")
@pytest.mark.parametrize("metric,scalar,n,d,m,ef,k", [
    ("l2sq", "f32", 3000, 24, 16, 64, 10),
    ("cos", "f32", 2000, 100, 8, 16, 10),      # ef barely above k
    ("ip", "f32", 1000, 17, 3, 5, 10),        # "absurd" config: M=3, ef < k (cpp/test.cpp:820-865)
    ("cos", "f16", 1500, 64, 16, 64, 10),
    ("l2sq", "bf16", 1500, 40, 16, 64, 10),
    ("ip", "i8", 2000, 128, 16, 64, 10),
    ("hamming", "b1", 5000, 64, 16, 64, 10),   # 64-bit codes: ties everywhere
    ("hamming", "b1", 3000, 256, 64, 64, 20),
    ("sorensen", "b1", 1500, 128, 8, 32, 5),
])
def test_port_matches_live_reference(metric, scalar, n, d, m, ef, k):
    base, q = common.make_collection(n, d, scalar, 200, iid=(d < 32))
    ref, blob = common.build_reference_blob(base, metric, scalar, d, m, threads=4)
    ref.pin_metric(True)
    ref.change_expansion_search(ef)
    want = ref.search(q, k, threads=4)
    got = bindings.PortIndex(blob, ef).search(q, k, threads=4)
    common.assert_same_results(want, got, f"{metric}/{scalar}")
    # exact (brute-force) path: index.hpp:4251-4268
    want = ref.search(q[:20], k, threads=2, exact=True)
    got = bindings.PortIndex(blob, ef).search(q[:20], k, threads=2, exact=True)
    common.assert_same_results(want[:3], got[:3], f"exact {metric}/{scalar}")


@pytest.mark.skipif(not common.have_reference(), reason="oracle/_ref not built")
def test_pinned_metrics_equal_native_where_exact():
    """On an AVX-512 host the pinned restatement IS the native kernel for every exactly
    reproducible metric (SURVEY.md §2.2); cosine differs by the rsqrt approximation only."""
    rng = np.random.default_rng(7)
    for metric, scalar, d, exact in [("l2sq", "f32", 768, True), ("ip", "f32", 100, True), ("cos", "f32", 768, False),
                                     ("ip", "i8", 1024, True), ("l2sq", "i8", 100, True), ("hamming", "b1", 256, True),
                                     ("tanimoto", "b1", 200, True)]:
        ref = bindings.RefIndex("parity", metric=metric, scalar=scalar, dims=d, connectivity=4)
        if ref.isa_name not in ("skylake", "ice", "sapphire", "genoa"):
            pytest.skip(f"host selects {ref.isa_name} kernels")
        x = common.datagen.to_scalar(rng.standard_normal((64, d), dtype=np.float32), scalar)
        native = np.array([ref.distance(x[i], x[i + 1]) for i in range(63)], dtype=np.float32)
        ref.pin_metric(True)
        pinned = np.array([ref.distance(x[i], x[i + 1]) for i in range(63)], dtype=np.float32)
        if exact:
            assert np.array_equal(native.view(np.uint32), pinned.view(np.uint32)), (metric, scalar)
        else:
            assert ulp_distance(native, pinned).max() <= 1, (metric, scalar)


def test_v2format_roundtrip():
    g = np.load(FIXTURES[0])
    graph = v2format.loads(g["blob"])
    assert np.array_equal(v2format.dumps(graph), g["blob"])


@pytest.mark.skipif(not common.have_reference(), reason="oracle/_ref not built")
def test_exact_search_oracles_agree():
    """The two brute-force oracles (exact_search_t over raw matrices, index search(exact=True)) give the same distance
    bits for a symmetric metric, and the port's exact path matches the reference's bit for bit."""
    base, q = common.make_collection(1500, 48, "f32", 32, iid=True)
    ref, blob = common.build_reference_blob(base, "l2sq", "f32", 48, 8, expansion_add=16, threads=4)
    ref.pin_metric(True)
    want = ref.search(q, 10, threads=2, exact=True)
    port = bindings.PortIndex(blob, 64).search(q, 10, threads=2, exact=True)
    common.assert_same_results(want[:3], port[:3], "port exact vs reference exact")
    fk, fd = bindings.ref_exact_search(base, q, 10, metric="l2sq", scalar="f32", dims=48, pinned=True)
    assert np.array_equal(fd.view(np.uint32), want[1].view(np.uint32))
    assert np.array_equal(fk, want[0])  # iid floats: no equal distances


@pytest.mark.skipif(not common.have_reference(), reason="oracle/_ref not built")
@pytest.mark.parametrize("metric,scalar,n,d,m", [("cos", "f32", 4000, 32, 4), ("hamming", "b1", 4000, 64, 4)])
def test_port_cluster_matches_live_reference(metric, scalar, n, d, m):
    """index_gt::cluster (index.hpp:3092-3125): small connectivity -> several graph levels to stop at."""
    base, q = common.make_collection(n, d, scalar, 100)
    ref, blob = common.build_reference_blob(base, metric, scalar, d, m, threads=4)
    ref.pin_metric(True)
    port = bindings.PortIndex(blob, 64)
    assert ref.max_level >= 3
    for level in (0, 1, 2, ref.max_level, ref.max_level + 3):
        want = ref.cluster(q, level)
        got = port.cluster(q, level)
        for a, b in zip(want, got):
            assert np.array_equal(a.view(np.uint32) if a.dtype == np.float32 else a, b.view(np.uint32) if b.dtype == np.float32 else b)
    # level 0 and level 1 are the same stop; beyond the top level the entry point is the answer
    assert np.array_equal(ref.cluster(q, 0)[0], ref.cluster(q, 1)[0])
    assert len(set(ref.cluster(q, ref.max_level + 3)[0].tolist())) == 1


@pytest.mark.parametrize("path", FIXTURES, ids=[os.path.basename(p)[:-4] for p in FIXTURES])
def test_port_next_rows_match_golden(path):
    """Exact search and cluster of the plain-C port against what the reference returned for the fixture graphs
    (tests/golden/next_rows.npz, made by make_golden_next_rows.py)."""
    name = os.path.basename(path)[:-4]
    g, nr = np.load(path), np.load(os.path.join(common.GOLDEN, "next_rows.npz"))
    port = bindings.PortIndex(g["blob"], int(g["ef"]))
    keys, dist, counts = port.search(g["queries"], int(g["k"]), threads=2, exact=True)[:3]
    assert np.array_equal(keys, nr[f"{name}/exact_keys"]) and np.array_equal(counts, nr[f"{name}/exact_counts"])
    assert np.array_equal(dist.view(np.uint32), nr[f"{name}/exact_distances"].view(np.uint32))
    for i, level in enumerate(nr[f"{name}/cluster_levels"]):
        ck, cd, cc, cv = port.cluster(g["queries"], int(level))
        assert np.array_equal(ck, nr[f"{name}/cluster_keys"][i]), f"level {level}"
        assert np.array_equal(cd.view(np.uint32), nr[f"{name}/cluster_distances"][i].view(np.uint32))
        assert np.array_equal(cc, nr[f"{name}/cluster_computed"][i]) and np.array_equal(cv, nr[f"{name}/cluster_visited"][i])


@pytest.mark.parametrize("path", FIXTURES, ids=[os.path.basename(p)[:-4] for p in FIXTURES])
def test_port_filtered_and_free_exact_search_match_golden(path):
    """filtered_search and exact_search_t over raw matrices of the plain-C port against what the reference returned on the
    fixture graphs (tests/golden/port_extras.npz, made by make_golden_port_extras.py)."""
    name = os.path.basename(path)[:-4]
    g, px = np.load(path), np.load(os.path.join(common.GOLDEN, "port_extras.npz"))
    graph = v2format.loads(g["blob"])
    q, k = g["queries"], int(g["k"])
    vectors = graph.vectors.view(bindings.SCALAR_NP[graph.scalar]).reshape(graph.size, -1)
    fk, fd = bindings.port_exact_search(vectors, q, k + 1, metric=graph.metric, scalar=graph.scalar, dims=graph.dimensions)
    wk, wd = px[f"{name}/free_keys"], px[f"{name}/free_distances"]
    assert np.array_equal(fd.view(np.uint32), wd.view(np.uint32))
    unique = wd[:, :k] != wd[:, 1:k + 1]  # std::partial_sort leaves the order of equal distances unspecified
    unique[:, 1:] &= wd[:, 1:k] != wd[:, :k - 1]
    assert np.array_equal(fk[:, :k][unique], wk[:, :k][unique])
    if graph.scalar != "f32":
        return
    port = bindings.PortIndex(g["blob"], int(g["ef"]))
    for i in range(3):
        want = tuple(px[f"{name}/filtered_{i}_{f}"] for f in ("keys", "distances", "counts", "computed", "visited"))
        got = port.filtered_search(q, k, px[f"{name}/filtered_{i}_allowed"], threads=2)
        common.assert_same_results(want, got, f"{name} filtered {i}")


def test_casts_match_golden():
    """datagen.to_scalar (how the tests quantise f32 rows) and the port's casts equal the reference's cast_gt
    (index_plugins.hpp:1105-1224) on the rows of tests/golden/port_extras.npz."""
    import ctypes as C
    px = np.load(os.path.join(common.GOLDEN, "port_extras.npz"))
    x = px["cast/input"]
    for scalar in ("f16", "bf16", "i8", "b1"):
        want = px[f"cast/{scalar}"]
        assert np.array_equal(common.datagen.to_scalar(x, scalar).view(np.uint8), want.view(np.uint8)), scalar
        if scalar in ("i8", "b1"):
            lib = bindings.port_lib()
            for row, expect in zip(x, want):
                out = np.zeros(bindings.bytes_per_vector(x.shape[1], scalar), dtype=np.uint8)
                lib.oracle_cast_from_f32(bindings.SCALAR[scalar], row.ctypes.data_as(bindings._f32p), x.shape[1],
                                         out.ctypes.data_as(C.c_void_p))
                assert np.array_equal(out, expect.view(np.uint8)), scalar


@pytest.mark.skipif(not common.have_reference(), reason="oracle/_ref not built")
def test_port_matches_live_reference_on_random_small_cases():
    """Forty seeded random configurations at the small end (n from 1, k > n, ef < k, removed members, duplicate vectors,
    every scalar kind): graph search, exact search and cluster of the port against the reference, bit for bit."""
    for case, c in enumerate(common.small_random_cases()):
        metric, scalar, n, d, m, ef, k, q = (c[f] for f in ("metric", "scalar", "n", "d", "m", "ef", "k", "q"))
        ref, _ = common.build_reference_blob(c["base"], metric, scalar, d, m, expansion_add=c["expansion_add"], threads=1,
                                             keys=c["keys"])
        for key in c["removed"]:
            ref.remove(int(key))
        blob = ref.save()
        ref.pin_metric(True)
        ref.change_expansion_search(ef)
        port = bindings.PortIndex(blob, ef)
        what = f"case {case}: {metric}/{scalar} n={n} d={d} M={m} ef={ef} k={k}"
        common.assert_same_results(ref.search(q, k, threads=1), port.search(q, k, threads=2), what)
        common.assert_same_results(ref.search(q, k, threads=1, exact=True)[:3], port.search(q, k, threads=2, exact=True)[:3], what + " exact")
        if ref.size:
            for level in (0, 1, ref.max_level + 1):
                for a, b in zip(ref.cluster(q, level), port.cluster(q, level)):
                    assert np.array_equal(a.view(np.uint32) if a.dtype == np.float32 else a,
                                          b.view(np.uint32) if b.dtype == np.float32 else b), what + f" cluster {level}"


# ---- the same configurations against tests/golden/reference_cases.npz (make_golden_reference_cases.py) -----------------

def _golden_blob(g, *inputs):
    assert common.digest(*inputs) == str(g["inputs_sha256"]), "the seeded collection came out different on this host"
    return common.with_vectors(g["graph"], inputs[0])


def _assert_search_and_exact(g, port, q, k, what):
    want = tuple(g[f"search_{f}"] for f in ("keys", "distances", "counts", "computed", "visited"))
    common.assert_same_results(want, port.search(q, k, threads=2), what)
    want = tuple(g[f"exact_{f}"] for f in ("keys", "distances", "counts"))
    common.assert_same_results(want, port.search(q, k, threads=2, exact=True)[:3], what + " exact")


def _assert_cluster(g, port, q, what):
    for i, level in enumerate(g["cluster_levels"]):
        got = port.cluster(q, int(level))
        for field, b in zip(("keys", "distances", "computed", "visited"), got):
            a = g[f"cluster_{field}"][i]
            assert np.array_equal(a.view(np.uint32) if a.dtype == np.float32 else a,
                                  b.view(np.uint32) if b.dtype == np.float32 else b), f"{what} cluster level {level} {field}"


@pytest.mark.parametrize("name,metric,scalar,n,d,m,ef,k", common.GOLDEN_SEARCH_CASES, ids=[c[0] for c in common.GOLDEN_SEARCH_CASES])
def test_port_matches_golden_reference_cases(name, metric, scalar, n, d, m, ef, k):
    """The configurations of test_port_matches_live_reference (every scalar kind, ef < k, M = 3, 64-bit codes, M = 64):
    graph and exact search of the port on the reference's graph against what the reference returned."""
    g = common.golden_case(name)
    base, q = common.make_collection(n, d, scalar, common.GOLDEN_NQ, iid=(d < 32))
    port = bindings.PortIndex(_golden_blob(g, base, q), ef)
    assert (port.size, port.dims, port.connectivity) == (n, d, m)
    _assert_search_and_exact(g, port, q, k, name)


@pytest.mark.parametrize("name,metric,scalar,n,d,m", common.GOLDEN_CLUSTER_CASES, ids=[c[0] for c in common.GOLDEN_CLUSTER_CASES])
def test_port_cluster_matches_golden_reference_cases(name, metric, scalar, n, d, m):
    """index_gt::cluster on several graph levels (up to and beyond the top) against what the reference returned."""
    g = common.golden_case(name)
    base, q = common.make_collection(n, d, scalar, common.GOLDEN_NQ)
    port = bindings.PortIndex(_golden_blob(g, base, q), 64)
    assert port.max_level >= 3 and int(g["cluster_levels"][3]) == port.max_level
    _assert_cluster(g, port, q, name)


def test_exact_search_oracles_agree_golden():
    """The port's two brute-force paths against the reference's: index search(exact=True) and exact_search_t over the raw
    rows; for this symmetric metric the reference's two give the same distance bits."""
    g = common.golden_case("free_l2sq_f32")
    base, q = common.make_collection(300, 48, "f32", common.GOLDEN_NQ, iid=True)
    port = bindings.PortIndex(_golden_blob(g, base, q), 64)
    want = tuple(g[f"exact_{f}"] for f in ("keys", "distances", "counts"))
    common.assert_same_results(want, port.search(q, 10, threads=2, exact=True)[:3], "port exact vs reference exact")
    fk, fd = bindings.port_exact_search(base, q, 10, metric="l2sq", scalar="f32", dims=48)
    assert np.array_equal(fd.view(np.uint32), g["free_distances"].view(np.uint32))
    assert np.array_equal(fk, g["free_keys"])  # iid floats: no equal distances
    assert np.array_equal(g["free_distances"].view(np.uint32), g["exact_distances"].view(np.uint32))


def test_pinned_metrics_equal_native_golden():
    """The reference's NATIVE SimSIMD kernels on an AVX-512 host (distances stored in the golden file) against the pinned
    restatement: bit for bit for every exactly reproducible metric, cosine within the rsqrt approximation (1 ULP)."""
    g = common.golden_case("native")
    assert str(g["isa"]) in ("skylake", "ice", "sapphire", "genoa"), str(g["isa"])
    for metric, scalar, d, x in common.native_metric_rows():
        assert common.digest(x) == str(g[f"{metric}_{scalar}_sha256"]), (metric, scalar)
        empty = v2format.Graph(metric, scalar, d, 4, 8, np.zeros((0, x.shape[1] * x.itemsize), np.uint8),
                               np.zeros(0, np.uint64), np.zeros(0, np.int16), [], 0, 0)
        port = bindings.PortIndex(v2format.dumps(empty))
        pinned = np.array([port.distance(x[i], x[i + 1]) for i in range(len(x) - 1)], dtype=np.float32)
        native = g[f"{metric}_{scalar}"]
        if metric == "cos":
            assert ulp_distance(native, pinned).max() <= 1, (metric, scalar)
        else:
            assert np.array_equal(native.view(np.uint32), pinned.view(np.uint32)), (metric, scalar)


def test_port_matches_golden_random_small_cases():
    """The first seeded random configurations of test_port_matches_live_reference_on_random_small_cases (n from 1, k > n,
    ef < k, removed members, duplicate vectors, every scalar kind): graph search, exact search and cluster of the port
    against what the reference returned."""
    for case, c in zip(range(common.GOLDEN_SMALL_CASES), common.small_random_cases()):
        g = common.golden_case(f"small_{case}")
        what = f"case {case}: {c['metric']}/{c['scalar']} n={c['n']} d={c['d']} M={c['m']} ef={c['ef']} k={c['k']}"
        port = bindings.PortIndex(_golden_blob(g, c["base"], c["q"]), c["ef"])
        _assert_search_and_exact(g, port, c["q"], c["k"], what)
        if "cluster_levels" in g:
            _assert_cluster(g, port, c["q"], what)
