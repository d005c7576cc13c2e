"""GPU parity of the brute-force path (SURVEY.md §8 N1): `search(exact=True)` on a frozen index against
index_gt::search_exact_ (index.hpp:4251-4268), and `usearch_exact_search` against exact_search_t
(index_plugins.hpp:2071-2164), both as the pinned plain-C oracle restates them (pinned to the reference's own outputs
by tests/golden). Graphs come from this project's builder, removed members from its `remove` (common.build_graph_blob)."""
import numpy as np
import pytest

import common
from oracle import bindings

pytestmark = pytest.mark.gpu

INDEX_CASES = [
    # metric, scalar, n, d, k, nq, removed
    ("cos", "f32", 5000, 768, 10, 70, 0),
    ("l2sq", "f32", 3000, 97, 33, 64, 100),      # ragged dimension, k > 32, removed members
    ("ip", "f32", 4096, 128, 256, 17, 0),        # the largest k whose lists live in registers
    ("l2sq", "f32", 3000, 64, 300, 24, 10),      # count > 256: lists in L2 (tiled scan + exact_merge_big_kernel)
    ("ip", "i8", 2500, 128, 700, 9, 0),          # count > 256 on i8: the tiled dp4a kernel instead of the IMMA one
    ("hamming", "b1", 3000, 128, 1000, 5, 0),    # a third of the collection, ties everywhere
    ("cos", "f16", 3000, 256, 10, 64, 50),
    ("l2sq", "bf16", 2000, 100, 10, 64, 0),
    ("ip", "i8", 3000, 1024, 10, 64, 0),
    ("cos", "i8", 2000, 100, 10, 33, 20),
    ("hamming", "b1", 6000, 64, 20, 64, 100),    # 64-bit codes: ties everywhere
    ("tanimoto", "b1", 3000, 200, 10, 64, 0),
    ("sorensen", "b1", 3000, 256, 10, 64, 0),
    ("l2sq", "f32", 1500, 2048, 10, 40, 30),     # 8 KB vectors: the tiled stage does not fit, one-query-per-warp scan kernel
    ("cos", "f32", 20000, 64, 10, 300, 0),       # many tiles per segment, several query groups
    ("l2sq", "i8", 20000, 200, 10, 300, 50),     # IMMA path: 3 query tiles, ragged K slice, removed members
    ("cos", "i8", 9000, 768, 40, 130, 0),        # IMMA path: k > 32
]


@pytest.mark.parametrize("metric,scalar,n,d,k,nq,removed", INDEX_CASES)
def test_index_exact_search_matches_reference(metric, scalar, n, d, k, nq, removed):
    from usearch_b200.index import Index
    base, q = common.make_collection(n, d, scalar, nq)
    base[n // 2:n // 2 + 40] = base[:40]          # duplicated vectors under different keys: equal distances
    keys = np.arange(n, dtype=np.uint64) * 7 + 3
    blob = common.build_graph_blob(base, metric, scalar, d, 8, expansion_add=16, keys=keys, removed=keys[5:5 + removed])
    want = bindings.PortIndex(blob).search(q, k, threads=8, exact=True)
    index = Index.restore(blob)
    got = index.search(q, k, exact=True)
    common.assert_same_results(want[:3], (got.keys, got.distances, got.counts), f"exact gpu vs reference [{metric}/{scalar}]")
    if removed:
        assert not np.isin(got.keys, keys[5:5 + removed]).any()


def test_index_exact_search_with_fewer_members_than_wanted():
    from usearch_b200.index import Index
    base, q = common.make_collection(7, 32, "f32", 5)
    blob = common.build_graph_blob(base, "l2sq", "f32", 32, 8)
    want = bindings.PortIndex(blob).search(q, 10, threads=1, exact=True)
    got = Index.restore(blob).search(q, 10, exact=True)
    assert (got.counts == 7).all()
    common.assert_same_results(want[:3], (got.keys, got.distances, got.counts), "exact, k > n")


def test_index_exact_search_agrees_with_graph_search_at_full_expansion():
    """Both kernels share metrics.cuh: a member found by the graph search carries the distance bits of the scan, and
    with ef = n the graph search finds (nearly) everything the scan does."""
    from usearch_b200.index import Index
    base, q = common.make_collection(2000, 64, "f32", 64, iid=True)
    blob = common.build_graph_blob(base, "l2sq", "f32", 64, 16)
    index = Index.restore(blob)
    exact = index.search(q, 10, exact=True)
    index.expansion_search = 2000
    graph = index.search(q, 10)
    found = 0
    for row in range(len(q)):  # members unreachable through the graph shift positions: compare by key
        scan = dict(zip(exact.keys[row].tolist(), exact.distances[row].view(np.uint32).tolist()))
        for key, bits in zip(graph.keys[row].tolist(), graph.distances[row].view(np.uint32).tolist()):
            if key in scan:
                found += 1
                assert scan[key] == bits
    assert found > 0.8 * exact.keys.size
    assert (exact.distances <= graph.distances).all()


FREE_CASES = [
    ("cos", "f32", 4000, 768, 10, 50),
    ("l2sq", "f32", 3000, 97, 5, 64),
    ("ip", "f16", 3000, 128, 10, 64),
    ("cos", "bf16", 2000, 96, 10, 64),
    ("cos", "i8", 2000, 256, 10, 64),     # asymmetric rounding: metric(dataset, query) order matters
    ("l2sq", "i8", 2000, 100, 10, 64),
    ("hamming", "b1", 4000, 256, 10, 64),
    ("tanimoto", "b1", 2000, 200, 1, 64),  # wanted == 1: std::min_element branch
]


@pytest.mark.parametrize("metric,scalar,n,d,k,nq", FREE_CASES)
def test_free_exact_search_matches_reference(metric, scalar, n, d, k, nq):
    from usearch_b200.index import exact_search
    base, q = common.make_collection(n, d, scalar, nq)
    wk, wd = bindings.port_exact_search(base, q, k + 1, metric=metric, scalar=scalar, dims=d)
    got = exact_search(base, q, k, metric=metric, dtype=scalar)
    assert np.array_equal(got.distances.view(np.uint32), wd[:, :k].view(np.uint32)), "distance bits differ"
    # labels are defined wherever the distance is unique in the row (std::partial_sort leaves ties unspecified)
    unique = (wd[:, :k] != wd[:, 1:k + 1])
    unique[:, 1:] &= wd[:, 1:k] != wd[:, :k - 1]
    assert unique.any()
    assert np.array_equal(got.keys[unique], wk[:, :k][unique])
    # and every reported label really has the reported distance
    for row in range(0, nq, 7):
        members = base[got.keys[row].astype(np.int64)]
        again = bindings.port_exact_search(members, q[row:row + 1], k, metric=metric, scalar=scalar, dims=d)[1]
        assert np.array_equal(again[0].view(np.uint32), got.distances[row].view(np.uint32))


def test_free_exact_search_rejects_more_neighbours_than_rows():
    from usearch_b200.index import exact_search
    base, q = common.make_collection(5, 16, "f32", 2)
    with pytest.raises(RuntimeError):
        exact_search(base, q, 6, metric="l2sq")


@pytest.mark.parametrize("metric,scalar,n,d,m", [
    ("cos", "f32", 6000, 768, 4),      # STAGED kernel
    ("l2sq", "f32", 6000, 32, 4),      # DIRECT kernel
    ("ip", "f16", 4000, 256, 4),
    ("hamming", "b1", 6000, 128, 4),
])
def test_cluster_matches_reference(metric, scalar, n, d, m):
    """index_dense_gt::cluster(vector, level): the descent of the search kernel stopped at `level`."""
    from usearch_b200.index import Index
    base, q = common.make_collection(n, d, scalar, 300)
    blob = common.build_graph_blob(base, metric, scalar, d, m)
    ref = bindings.PortIndex(blob)
    index = Index.restore(blob)
    assert index.max_level == ref.max_level >= 3
    for level in (0, 1, 2, ref.max_level, ref.max_level + 2):
        wk, wd, wc, wv = ref.cluster(q, level)
        gk, gd = index.cluster(q, level, stats=True)
        assert np.array_equal(gk, wk), f"level {level}: members differ"
        assert np.array_equal(gd.view(np.uint32), wd.view(np.uint32)), f"level {level}: distance bits differ"
        assert np.array_equal(index.last_computed, wc) and np.array_equal(index.last_visited, wv), f"level {level}: counters"
    # the graph search is unaffected by a cluster call in between
    ref.change_expansion_search(64)
    index.expansion_search = 64
    want = ref.search(q, 10, threads=8)
    got = index.search(q, 10, stats=True)
    common.assert_same_results(want, (got.keys, got.distances, got.counts, index.last_computed, index.last_visited), "after cluster")



@pytest.mark.parametrize("kernel", ["imma", "umma", "tiled"])
def test_i8_exact_kernels_agree_with_the_reference(kernel):
    """The three i8 scans — tcgen05 with TMEM accumulators (default), mma.sync, dp4a — forced one at a time
    (USEARCH_B200_EXACT is read once per process, hence the subprocess): same bits, index mode and free function."""
    import os
    import subprocess
    import sys
    code = (
        "import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "import numpy as np, common\n"
        "from oracle import bindings\n"
        "from usearch_b200.index import Index, exact_search\n"
        "for metric, n, d, k, nq, removed in (('ip', 5000, 1024, 10, 150, 0), ('l2sq', 7000, 200, 33, 300, 40), ('cos', 3000, 768, 100, 70, 10), ('ip', 700, 96, 256, 9, 0)):\n"
        "    base, q = common.make_collection(n, d, 'i8', nq)\n"
        "    base[n // 2:n // 2 + 30] = base[:30]\n"
        "    keys = np.arange(n, dtype=np.uint64) * 5 + 1\n"
        "    blob = common.build_graph_blob(base, metric, 'i8', d, 8, expansion_add=16, keys=keys, removed=keys[3:3 + removed])\n"
        "    want = bindings.PortIndex(blob).search(q, k, threads=8, exact=True)\n"
        "    got = Index.restore(blob).search(q, k, exact=True)\n"
        "    common.assert_same_results(want[:3], (got.keys, got.distances, got.counts), metric)\n"
        "    wk, wd = bindings.port_exact_search(base, q, k, metric=metric, scalar='i8', dims=d)\n"
        "    free = exact_search(base, q, k, metric=metric, dtype='i8')\n"
        "    assert np.array_equal(free.distances.view(np.uint32), wd.view(np.uint32)), metric\n"
        "print('I8_EXACT_OK')\n"
    ) % (common.ROOT, os.path.join(common.ROOT, "tests"))
    env = dict(os.environ, USEARCH_B200_EXACT=kernel)
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "I8_EXACT_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-3000:]
