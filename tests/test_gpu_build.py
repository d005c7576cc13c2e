"""GPU-assisted add (SURVEY.md §8f N4; csrc/builder.cu) and the by-key half of the C ABI, on one GPU.

A GPU-built graph is not bit-identical to a reference-built one (neither are two multi-threaded reference builds), so the
bar is DESIGN.md §9: structure invariants, and the reference search (the pinned plain-C oracle) on the GPU-built file
reaching the recall and the work per query the reference reached on its own file of the same collection
(tests/golden/build_quality.json). Our own search on our own graph must still equal the oracle's search on that same
graph bit for bit."""
import json
import os
import sys
import threading

import numpy as np
import pytest

import common
from oracle import bindings

sys.path.insert(0, os.path.join(common.ROOT, "tools"))
from build_check import exact_truth, hamming_truth, recall, structure_report  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("metric,scalar,n,d,m", [
    ("cos", "f32", 12000, 96, 16),
    ("l2sq", "f32", 8000, 128, 16),
    ("cos", "f16", 8000, 256, 16),
    ("ip", "i8", 8000, 256, 16),
    ("hamming", "b1", 12000, 256, 32),
    ("cos", "f32", 6000, 768, 32),
])
def test_gpu_built_graph_is_as_good_as_a_reference_built_one(metric, scalar, n, d, m):
    from usearch_b200.index import Index
    base, queries = common.make_collection(n, d, scalar, 400)
    keys = np.arange(n, dtype=np.uint64)
    index = Index(ndim=d, metric=metric, dtype=scalar, connectivity=m, expansion_add=128)
    index.add(keys, base)
    assert len(index) == n
    gpu_blob = index.save()
    rep = structure_report(gpu_blob)
    assert rep["n_problems"] == 0, rep["problems"]
    truth = hamming_truth(base, queries, 10) if scalar == "b1" else exact_truth(base, queries, metric, 10)
    with open(os.path.join(common.GOLDEN, "build_quality.json")) as f:
        ref = json.load(f)[f"{metric}/{scalar}/{n}/{d}/{m}"]  # the reference's search of its own graph, ef = 64
    want = bindings.PortIndex(gpu_blob, 64).search(queries, 10, threads=16)
    got = {"ref": (ref["recall"], ref["computed_per_query"]), "gpu": (recall(want[0], truth), float(want[3].mean()))}
    assert got["gpu"][0] >= got["ref"][0] - 0.01, got
    assert abs(got["gpu"][1] - got["ref"][1]) <= 0.08 * got["ref"][1], got
    # same graph => our search and the oracle's agree bit for bit
    index.expansion_search = 64
    mine = index.search(queries, 10, stats=True)
    common.assert_same_results(want, (mine.keys, mine.distances, mine.counts, index.last_computed, index.last_visited), "gpu graph")


def test_incremental_adds_grow_the_index_and_find_themselves():
    """cpp/test.cpp:358-361: a stored vector is its own nearest neighbour; capacity grows on demand; single adds work."""
    from usearch_b200.index import Index
    n, d = 5000, 64
    base, _ = common.make_collection(n, d, "f32", 1)
    index = Index(ndim=d, metric="cos", dtype="f32", connectivity=16)
    index.add(7, base[0])                                    # one member, no reserve
    index.add(np.arange(100, 1100, dtype=np.uint64), base[1:1001])
    index.reserve(2500)
    index.add(np.arange(5000, 5000 + n - 1001, dtype=np.uint64), base[1001:])
    assert len(index) == n and index.capacity >= n
    index.expansion_search = 64
    res = index.search(base[:2000], 1)
    expect = np.concatenate([[7], np.arange(100, 1100), np.arange(5000, 5999)]).astype(np.uint64)
    assert (res.keys[:, 0] == expect).mean() > 0.995
    assert float(np.nanmax(res.distances[:, 0])) < 1e-5
    with pytest.raises(RuntimeError, match="Duplicate"):
        index.add(7, base[3])
    with pytest.raises(RuntimeError, match="Duplicate"):   # twice within one call
        index.add(np.array([777777, 777777], dtype=np.uint64), base[3:5])
    assert len(index) == n and not index.contains(777777)
    # f64 input is cast on the device; the round trip through `get` returns the stored f32
    index.add(99999, base[5].astype(np.float64))
    assert np.array_equal(index.get(99999), base[5])


def test_lookups_and_edits_by_key():
    from usearch_b200 import v2format
    from usearch_b200.index import Index, load_library
    import ctypes as C
    n, d = 3000, 48
    base, queries = common.make_collection(n, d, "f32", 64)
    blob = common.build_graph_blob(base, "ip", "f32", d, 16, keys=np.arange(n, dtype=np.uint64) * 3)
    index = Index.restore(blob)                             # lookups work on a loaded file too
    assert index.contains(30) and not index.contains(31) and index.count(30) == 1 and index.count(31) == 0
    assert np.array_equal(index.get(30), base[10]) and index.get(31) is None
    assert np.allclose(index.get(30, dtype="f64"), base[10].astype(np.float64))
    # usearch_distance == the distance the search reports for that pair == the pinned oracle's
    lib = load_library()
    err = C.c_char_p()
    dist = lib.usearch_distance(queries[0].ctypes.data_as(C.c_void_p), base[10].ctypes.data_as(C.c_void_p), 1, d, 2, C.byref(err))
    assert not err.value
    port = bindings.PortIndex(blob, 64)
    assert np.float32(dist).view(np.uint32) == np.float32(port.distance(queries[0], base[10])).view(np.uint32)
    # remove: tombstone, gone from results, size shrinks, slot is not recycled
    index.expansion_search = 64
    before = index.search(queries, 10)
    victim = int(before.keys[0, 0])
    assert index.remove(victim) == 1 and index.remove(victim) == 0
    assert len(index) == n - 1 and not index.contains(victim)
    after = index.search(queries, 10)
    assert victim not in after.keys.tolist()[0]
    # the file after the same removal, modelled as the reference's remove does it (the key becomes the free key, the
    # links stay; golden fixture ip_f32_n1500_d48_removed): same answers
    graph = v2format.loads(blob)
    graph.keys[graph.keys == victim] = v2format.FREE_KEY
    want = bindings.PortIndex(v2format.dumps(graph), 64).search(queries, 10, threads=8)
    assert np.array_equal(after.keys, want[0]) and np.array_equal(after.distances.view(np.uint32), want[1].view(np.uint32))
    # rename
    other = int(before.keys[1, 0])
    assert index.rename(other, 10**12) == 1 and index.contains(10**12) and not index.contains(other)
    again = index.search(queries[1], 10)
    assert int(again.keys[0]) == 10**12
    # save -> load keeps the tombstone and the new key
    copy = Index.restore(index.save())
    assert len(copy) == n - 1 and copy.contains(10**12) and not copy.contains(victim)


def test_concurrent_single_query_callers_are_gathered():
    from usearch_b200.index import Index
    n, d = 4000, 64
    base, queries = common.make_collection(n, d, "f32", 256)
    blob = common.build_graph_blob(base, "cos", "f32", d, 16)
    index = Index.restore(blob)
    index.expansion_search = 64
    want = index.search(queries, 10)
    out = [None] * len(queries)

    def worker(lo, hi):
        for i in range(lo, hi):
            out[i] = index.search(queries[i], 10)

    threads = [threading.Thread(target=worker, args=(i * 32, (i + 1) * 32)) for i in range(8)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    for i, m in enumerate(out):
        assert np.array_equal(m.keys, want.keys[i, :int(want.counts[i])])
        assert np.array_equal(m.distances.view(np.uint32), want.distances[i, :int(want.counts[i])].view(np.uint32))


def _cpu_indexes_merge(per_shard, k):
    """`Indexes`-style merge of per-shard CPU results (python/lib.cpp:350-391) with the deterministic order."""
    nq = per_shard[0][0].shape[0]
    out_k = np.zeros((nq, k), np.uint64)
    out_d = np.full((nq, k), np.array(0x7FA00000, dtype=np.uint32).view(np.float32), np.float32)
    out_c = np.zeros(nq, np.uint64)
    for q in range(nq):
        items = []
        for r, (keys, d, c) in enumerate(per_shard):
            items += [(float(d[q, i]), r, i, int(keys[q, i])) for i in range(int(c[q]))]
        items.sort(key=lambda t: (t[0], t[1], t[2]))
        items = items[:k]
        out_c[q] = len(items)
        for i, (dd, _, _, kk) in enumerate(items):
            out_k[q, i], out_d[q, i] = kk, dd
    return out_k, out_d, out_c


@pytest.mark.parametrize("metric,scalar,d,m,G", [("cos", "f32", 96, 16, 3), ("hamming", "b1", 128, 16, 4), ("ip", "i8", 128, 16, 2)])
def test_sharded_search_matches_the_cpu_indexes_merge(metric, scalar, d, m, G):
    """SURVEY §8e parity target: the CPU `Indexes` search (the pinned oracle per shard) over the SAME G serialised shards,
    merged by (distance, shard, position). Each shard is searched on the GPU; the merge kernel does the exchange step's
    second half."""
    from usearch_b200.index import Index, merge_topk
    n, k, ef = 9000, 10, 64
    base, queries = common.make_collection(n, d, scalar, 200)
    keys = np.arange(n, dtype=np.uint64)
    cpu, gpu = [], []
    for r in range(G):
        blob = common.build_graph_blob(base[r::G], metric, scalar, d, m, keys=keys[r::G])
        want = bindings.PortIndex(blob, ef).search(queries, k, threads=16)
        cpu.append((want[0], want[1], want[2]))
        index = Index.restore(blob)
        index.expansion_search = ef
        got = index.search(queries, k)
        gpu.append((got.keys, got.distances, got.counts))
    want_k, want_d, want_c = _cpu_indexes_merge(cpu, k)
    merged = merge_topk(gpu, k)
    assert np.array_equal(merged.counts, want_c)
    assert np.array_equal(merged.distances.view(np.uint32), want_d.view(np.uint32))  # distance multisets AND order
    assert np.array_equal(merged.keys, want_k)


def test_merge_kernel_equals_its_torch_specification():
    import torch
    from usearch_b200.index import merge_topk
    from usearch_b200.sharded import merge_gathered
    rng = np.random.default_rng(5)
    nq, k, world = 300, 10, 8
    shards = []
    for r in range(world):
        d = np.sort(rng.integers(0, 5, size=(nq, k)).astype(np.float32), axis=1)   # heavy ties, like Hamming
        keys = (rng.permutation(nq * k).reshape(nq, k) * world + r).astype(np.uint64)
        c = rng.integers(0, k + 1, size=nq).astype(np.uint64)
        c[0], c[1] = 0, k
        shards.append((keys, d, c))
    got = merge_topk(shards, k)
    wk, wd, wc = merge_gathered([torch.from_numpy(s[0].astype(np.int64)) for s in shards], [torch.from_numpy(s[1]) for s in shards],
                                [torch.from_numpy(s[2].astype(np.int64)) for s in shards], k)
    assert np.array_equal(got.counts, wc.numpy().astype(np.uint64))
    assert np.array_equal(got.keys, wk.numpy().astype(np.uint64))
    assert np.array_equal(got.distances.view(np.uint32), wd.numpy().view(np.uint32))


def test_enqueue_then_finish_equals_the_blocking_calls(tmp_path):
    """usearch_b200_search_many_enqueue x3 + one _finish == three usearch_b200_search_many_device calls, with scratch small
    enough (test hook) that some queries overflow and have to be retried by _finish. The graph is built here, outside
    the process whose search runs under the test hooks."""
    import subprocess
    base, _ = common.make_collection(6000, 64, "f32", 1)
    path = str(tmp_path / "graph.usearch")
    common.build_graph_blob(base, "cos", "f32", 64, 16).tofile(path)
    code = (
        "import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "import numpy as np, torch, common\n"
        "from usearch_b200.index import Index\n"
        "base, q = common.make_collection(6000, 64, 'f32', 384)\n"
        "blob = np.fromfile(%r, dtype=np.uint8)\n"
        "index = Index.restore(blob); index.expansion_search = 64\n"
        "dev = torch.device('cuda', 0)\n"
        "qd = torch.from_numpy(q).to(dev)\n"
        "def bufs(): return (torch.zeros((128, 10), dtype=torch.int64, device=dev), torch.zeros((128, 10), dtype=torch.float32, device=dev), torch.zeros(128, dtype=torch.int32, device=dev))\n"
        "sync, deferred = [bufs() for _ in range(3)], [bufs() for _ in range(3)]\n"
        "for i, (k, d, c) in enumerate(sync): index.search_device(qd[i*128:(i+1)*128].data_ptr(), 128, 256, 10, k.data_ptr(), d.data_ptr(), c.data_ptr())\n"
        "for i, (k, d, c) in enumerate(deferred): index.search_enqueue(qd[i*128:(i+1)*128].data_ptr(), 128, 256, 10, k.data_ptr(), d.data_ptr(), c.data_ptr())\n"
        "index.search_finish()\n"
        "torch.cuda.synchronize()\n"
        "for a, b in zip(sync, deferred):\n"
        "    assert torch.equal(a[0], b[0]) and torch.equal(a[1].view(torch.int32), b[1].view(torch.int32)) and torch.equal(a[2], b[2])\n"
        "want = index.search(q, 10)\n"
        "assert np.array_equal(torch.cat([s[0] for s in deferred]).cpu().numpy().astype(np.uint64), want.keys)\n"
        "print('ENQUEUE_OK')\n"
    ) % (common.ROOT, os.path.join(common.ROOT, "tests"), path)
    env = dict(os.environ, USEARCH_B200_VISITED="hash", USEARCH_B200_SCRATCH_SHRINK="64")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ENQUEUE_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


def test_adding_to_a_loaded_reference_built_index():
    """`load` a file written by the reference (a committed golden fixture), then keep adding on the GPU (capacity grows
    from the file's size), save, and let the reference search (the pinned oracle) search the result: every member, old
    and new, is its own nearest neighbour."""
    from usearch_b200 import v2format
    from usearch_b200.index import Index
    blob = np.load(os.path.join(common.GOLDEN, "cos_f32_n2000_d64.npz"))["blob"]
    graph = v2format.loads(blob)
    n0, n1, d = graph.size, 3000, graph.dimensions
    assert graph.metric == "cos" and graph.scalar == "f32" and np.array_equal(graph.keys, np.arange(n0, dtype=np.uint64))
    added, _ = common.make_collection(n1, d, "f32", 1, seed=7)
    base = np.concatenate([graph.vectors.view(np.float32).reshape(n0, d), added])
    index = Index.restore(blob)
    assert len(index) == n0
    index.add(np.arange(n0, n0 + n1, dtype=np.uint64), base[n0:])
    assert len(index) == n0 + n1
    rep = structure_report(index.save())
    assert rep["n_problems"] == 0, rep["problems"]
    keys, dist, _, _, _ = bindings.PortIndex(index.save(), 64).search(base, 1, threads=16)
    assert (keys[:, 0] == np.arange(n0 + n1, dtype=np.uint64)).mean() > 0.995
    # clear -> the handle is reusable for a new collection
    index.clear()
    assert len(index) == 0
    index.add(np.arange(100, dtype=np.uint64), base[:100])
    assert len(index) == 100 and index.contains(99)
