"""GPU parity: the CUDA search (through the C ABI) against the CPU search of the oracle (the plain-C restatement of the
reference search, pinned to the reference's own outputs by tests/golden) on the SAME serialised graph, bit-for-bit:
labels, distance bits, counts and the reference's two counters. Graphs come from this project's builder, removed members
from its `remove` (common.build_graph_blob)."""
import numpy as np
import pytest

import common
from oracle import bindings

pytestmark = pytest.mark.gpu

CASES = [
    # metric, scalar, n, d, M, ef, k, nq
    ("l2sq", "f32", 20000, 128, 16, 64, 10, 512),
    ("cos", "f32", 8000, 768, 32, 128, 10, 256),
    ("ip", "f32", 6000, 96, 16, 64, 10, 256),
    ("cos", "f32", 3000, 97, 13, 32, 7, 128),     # ragged dimension, odd connectivity
    ("ip", "i8", 8000, 1024, 16, 128, 10, 256),
    ("l2sq", "i8", 4000, 100, 16, 64, 10, 128),
    ("cos", "i8", 4000, 256, 16, 64, 10, 128),
    ("hamming", "b1", 20000, 256, 64, 64, 10, 256),
    ("tanimoto", "b1", 6000, 200, 16, 64, 10, 128),
    ("sorensen", "b1", 6000, 256, 16, 64, 10, 128),
    ("l2sq", "f32", 5000, 32, 16, 300, 40, 64),     # ef > 256: shared-memory `top`, k > 32, DIRECT kernel
    ("ip", "f32", 6000, 128, 16, 300, 50, 64),      # ef > 256 on the STAGED (TMA) kernel
    ("cos", "f32", 4000, 64, 40, 256, 100, 64),     # M0 = 80 > 64 neighbours per row, ef == 256
    ("cos", "f16", 6000, 768, 32, 128, 10, 128),    # one lane per vector, 32 TMA slots per pass
    ("l2sq", "f16", 4000, 100, 16, 64, 10, 128),    # 200-byte vectors: DIRECT kernel, ragged tail
    ("ip", "bf16", 4000, 256, 16, 64, 10, 128),
    ("cos", "bf16", 3000, 96, 16, 64, 10, 128),
]


@pytest.mark.parametrize("metric,scalar,n,d,m,ef,k,nq", CASES)
def test_search_matches_reference(metric, scalar, n, d, m, ef, k, nq):
    from usearch_b200.index import Index
    base, q = common.make_collection(n, d, scalar, nq)
    blob = common.build_graph_blob(base, metric, scalar, d, m)
    want = bindings.PortIndex(blob, ef).search(q, k, threads=16)
    index = Index.restore(blob)
    index.expansion_search = ef
    assert index.size == n and index.ndim == d and index.connectivity == m
    got = index.search(q, k, stats=True)
    common.assert_same_results(want, (got.keys, got.distances, got.counts, index.last_computed, index.last_visited),
                               f"gpu vs reference [{metric}/{scalar}]")
    assert index.kernel_launches >= 1


@pytest.mark.parametrize("mode,shrink", [("hash", 64), ("bitmap", 64), ("bitmap_log", 64), ("bitmap_log", 1)])
def test_visited_modes_and_scratch_retry(mode, shrink, tmp_path):
    """All `visits` implementations are exact: open-addressing table (undersized on purpose: flag-and-retry path of
    frozen_index_t::search_device), bitmap wiped per query, bitmap cleaned through the per-query log of set bits
    (with a 64x undersized log: fall back to a full wipe). 8192 queries: every warp serves several in a row, so a
    bitmap left dirty by one query would corrupt the next. The graph is built here, outside the process whose search
    runs under the test hooks."""
    import os
    import subprocess
    import sys
    base, _ = common.make_collection(30000, 64, "f32", 1, iid=True)
    path = str(tmp_path / "graph.usearch")
    common.build_graph_blob(base, "l2sq", "f32", 64, 16).tofile(path)
    code = (
        "import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "import numpy as np, common\n"
        "from oracle import bindings\n"
        "from usearch_b200.index import Index\n"
        "base, q = common.make_collection(30000, 64, 'f32', 8192, iid=True)\n"
        "blob = np.fromfile(%r, dtype=np.uint8)\n"
        "want = bindings.PortIndex(blob, 64).search(q, 10, threads=16)\n"
        "index = Index.restore(blob); index.expansion_search = 64\n"
        "got = index.search(q, 10, stats=True)\n"
        "common.assert_same_results(want, (got.keys, got.distances, got.counts, index.last_computed, index.last_visited), 'mode')\n"
        "print('launches', index.kernel_launches, 'maxD', int(want[3].max()))\n"
    ) % (common.ROOT, os.path.join(common.ROOT, "tests"), path)
    env = dict(os.environ, USEARCH_B200_VISITED=mode, USEARCH_B200_SCRATCH_SHRINK=str(shrink))
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    launches = int(out.stdout.split("launches")[1].split()[0])
    if mode == "hash":  # bitmap `visits` cannot overflow; its heap head alone (shared memory) holds these searches
        assert launches >= 2, "expected at least one retry launch with 64x undersized scratch: " + out.stdout


@pytest.mark.parametrize("fraction", [0.5, 0.05, 0.0])
def test_filtered_search_matches_reference(fraction):
    """Device-side `key in set` predicate vs the oracle's filtered_search with the same predicate (cpp/test.cpp:1105-1145,
    the oracle pinned to the reference's filtered_search by tests/golden/port_extras.npz): rejected members are traversed
    but never returned; some keys are also removed."""
    from usearch_b200.index import Index
    n, d, m, ef, k = 8000, 96, 16, 64, 10
    base, q = common.make_collection(n, d, "f32", 200)
    blob = common.build_graph_blob(base, "cos", "f32", d, m, keys=np.arange(n, dtype=np.uint64) * 7 + 3,
                                   removed=range(3, 3 + 7 * 400, 7 * 4))
    rng = np.random.default_rng(5)
    allowed = (rng.permutation(n)[: int(n * fraction)].astype(np.uint64) * 7 + 3)
    want = bindings.PortIndex(blob, ef).filtered_search(q, k, allowed, threads=16)
    index = Index.restore(blob)
    index.expansion_search = ef
    got = index.filtered_search(q, k, allowed)
    common.assert_same_results(want, (got.keys, got.distances, got.counts, index.last_computed, index.last_visited),
                               f"filtered {fraction}")
    if fraction:
        assert np.isin(got.keys[got.distances == got.distances], allowed).all()
    else:
        assert (got.counts == 0).all()


@pytest.mark.parametrize("metric,scalar,d", [("cos", "f16", 128), ("ip", "bf16", 96), ("cos", "i8", 256), ("hamming", "b1", 256)])
def test_f32_queries_are_cast_like_the_reference(metric, scalar, d):
    """Queries arrive as f32 while the index stores another scalar kind: the host cast of the C ABI must equal
    the reference's `cast_gt` (index_plugins.hpp:1105-1224) — here the oracle searches the queries cast by
    datagen.to_scalar, which test_oracle.py pins to the reference's casts (tests/golden/port_extras.npz)."""
    from usearch_b200.index import Index
    n, m, ef, k = 4000, 16, 64, 10
    base, _ = common.make_collection(n, d, scalar, 8)
    q32 = common.datagen.latent(100, d, seed=77, rank=16)
    blob = common.build_graph_blob(base, metric, scalar, d, m)
    want = bindings.PortIndex(blob, ef).search(common.datagen.to_scalar(q32, scalar), k, threads=16)
    index = Index.restore(blob)
    index.expansion_search = ef
    got = index.search(q32, k, stats=True)
    common.assert_same_results(want, (got.keys, got.distances, got.counts, index.last_computed, index.last_visited),
                               f"f32 -> {scalar}")


