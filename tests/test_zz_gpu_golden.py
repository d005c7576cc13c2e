"""GPU parity against the COMMITTED golden vectors (tests/golden/*.npz: outputs of the unmodified reference, made by
make_golden.py / make_golden_next_rows.py): nothing of the reference or the oracle is involved at run time.
Collected last (file name) so that every other GPU test has reported before these start."""
import glob
import os

import numpy as np
import pytest

import common
from oracle import bindings

pytestmark = pytest.mark.gpu

GOLDEN_FIXTURES = sorted(glob.glob(os.path.join(common.GOLDEN, "*_n*.npz")))
IDS = [os.path.basename(p)[:-4] for p in GOLDEN_FIXTURES]


@pytest.mark.parametrize("path", GOLDEN_FIXTURES, ids=IDS)
def test_search_matches_golden(path):
    """Labels, distance bits, counts and both counters of the graph search."""
    from usearch_b200.index import Index
    g = np.load(path)
    index = Index.restore(g["blob"])
    index.expansion_search = int(g["ef"])
    got = index.search(g["queries"], int(g["k"]), stats=True)
    want = (g["keys_pinned"], g["distances_pinned"], g["counts_pinned"], g["computed_pinned"], g["visited_pinned"])
    common.assert_same_results(want, (got.keys, got.distances, got.counts, index.last_computed, index.last_visited), "gpu vs golden")
    # the reference's native SimSIMD dispatch on the generating host: same labels
    assert np.array_equal(got.keys, g["keys_native"])


# Round 1 never saw this test finish: cluster(level = top) on a graph whose top level holds ONE member walks an empty
# list, and an empty list used to arm an mbarrier phase nobody waited for (search_kernel.cu, measure_list) - the next
# wait of that warp deadlocked. Fixed in round 2; the case below (levels up to and beyond the top) is the regression test.
@pytest.mark.parametrize("path", GOLDEN_FIXTURES, ids=IDS)
def test_next_rows_match_golden(path):
    """Exact search (index mode and free function) and cluster against tests/golden/next_rows.npz."""
    from usearch_b200 import v2format
    from usearch_b200.index import Index, exact_search
    name = os.path.basename(path)[:-4]
    g, nr = np.load(path), np.load(os.path.join(common.GOLDEN, "next_rows.npz"))
    q, k = g["queries"], int(g["k"])
    index = Index.restore(g["blob"])
    got = index.search(q, k, exact=True)
    assert np.array_equal(got.keys, nr[f"{name}/exact_keys"]) and np.array_equal(got.counts, nr[f"{name}/exact_counts"])
    assert np.array_equal(got.distances.view(np.uint32), nr[f"{name}/exact_distances"].view(np.uint32))
    for i, level in enumerate(nr[f"{name}/cluster_levels"]):
        ck, cd = index.cluster(q, int(level), stats=True)
        assert np.array_equal(ck, nr[f"{name}/cluster_keys"][i]), f"level {level}"
        assert np.array_equal(cd.view(np.uint32), nr[f"{name}/cluster_distances"][i].view(np.uint32))
        assert np.array_equal(index.last_computed, nr[f"{name}/cluster_computed"][i])
        assert np.array_equal(index.last_visited, nr[f"{name}/cluster_visited"][i])
    graph = v2format.loads(g["blob"])
    vectors = graph.vectors.view(bindings.SCALAR_NP[graph.scalar]).reshape(graph.size, -1)
    free = exact_search(vectors, q, k, metric=graph.metric, dtype=graph.scalar)
    wd, wk = nr[f"{name}/free_distances"], nr[f"{name}/free_keys"]
    assert np.array_equal(free.distances.view(np.uint32), wd[:, :k].view(np.uint32))
    unique = wd[:, :k] != wd[:, 1:k + 1]
    unique[:, 1:] &= wd[:, 1:k] != wd[:, :k - 1]
    assert np.array_equal(free.keys[unique], wk[:, :k][unique])


@pytest.mark.parametrize("metric,scalar,n,d,m,ef,k,nq", [
    ("cos", "f16", 6000, 768, 32, 128, 10, 128),     # WORD metrics: 4 lanes per vector split by accumulator
    ("l2sq", "f16", 4000, 200, 16, 64, 10, 128),     # 400-byte vectors: ragged last chunk group
    ("ip", "bf16", 4000, 256, 16, 64, 10, 128),
    ("cos", "bf16", 3000, 136, 16, 300, 20, 64),     # ef > 256: shared-memory `top`
    ("ip", "i8", 8000, 1024, 16, 128, 10, 256),      # 16 resident warps per SM, one stage set
    ("cos", "i8", 4000, 256, 16, 64, 10, 128),
    ("l2sq", "i8", 4000, 512, 16, 64, 10, 128),
    ("cos", "f16", 6000, 768, 32, 256, 10, 128),     # C3's ef
    ("cos", "f16", 3000, 1536, 16, 64, 10, 64),      # 3 KB half vectors: two stage sets again
    ("ip", "i8", 3000, 4096, 16, 64, 10, 64),        # 4 KB i8 vectors
])
def test_short_vector_kernels_match_reference(metric, scalar, n, d, m, ef, k, nq):
    """The kernels that became the default in round 2 for f16 / bf16 / i8 (search_kernel.cu, dispatch) against the pinned
    oracle: labels, distance bits, counts, both counters."""
    from usearch_b200.index import Index
    base, q = common.make_collection(n, d, scalar, nq)
    blob = common.build_graph_blob(base, metric, scalar, d, m)
    want = bindings.PortIndex(blob, ef).search(q, k, threads=16)
    index = Index.restore(blob)
    index.expansion_search = ef
    got = index.search(q, k, stats=True)
    common.assert_same_results(want, (got.keys, got.distances, got.counts, index.last_computed, index.last_visited), "gpu vs oracle")
