"""Generate tests/golden/port_extras.npz and tests/golden/build_quality.json by RUNNING THE UNMODIFIED REFERENCE
(oracle/_ref, needs the reference sources):  python tests/golden/make_golden_port_extras.py

port_extras.npz, on the graphs and queries of the committed search fixtures (metric pinned):
  * ``<name>/filtered_<i>_{allowed,keys,distances,counts,computed,visited}``: filtered_search with the predicate
    "key in allowed" for three sizes of the allowed set (f32 fixtures: the reference's filtered search takes f32 queries),
  * ``<name>/free_{keys,distances}``: exact_search_t over the fixture's raw vectors, k + 1 columns,
  * ``cast/{input,f16,bf16,i8,b1}``: the reference's casts of f32 rows into each scalar kind.
build_quality.json: recall@10 and computed distances per query of the reference's search (ef 64, native metric) over
the graph the reference builds, for the collections of test_gpu_build.py."""
import glob
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import common  # noqa: E402
from oracle import bindings  # noqa: E402
from usearch_b200 import v2format  # noqa: E402

BUILD_CASES = [("cos", "f32", 12000, 96, 16), ("l2sq", "f32", 8000, 128, 16), ("cos", "f16", 8000, 256, 16),
               ("ip", "i8", 8000, 256, 16), ("hamming", "b1", 12000, 256, 32), ("cos", "f32", 6000, 768, 32)]


def port_extras():
    out = {}
    for path in sorted(glob.glob(os.path.join(HERE, "*_n*.npz"))):
        name = os.path.basename(path)[:-4]
        g = np.load(path)
        graph = v2format.loads(g["blob"])
        q, k = g["queries"], int(g["k"])
        vectors = graph.vectors.view(bindings.SCALAR_NP[graph.scalar]).reshape(graph.size, -1)
        fk, fd = bindings.ref_exact_search(vectors, q, k + 1, metric=graph.metric, scalar=graph.scalar, dims=graph.dimensions)
        out[f"{name}/free_keys"], out[f"{name}/free_distances"] = fk, fd
        if graph.scalar != "f32":
            continue
        ref = bindings.RefIndex("parity")
        ref.load(g["blob"])
        ref.pin_metric(True)
        ref.change_expansion_search(int(g["ef"]))
        live = graph.keys[graph.keys != v2format.FREE_KEY]
        rng = np.random.default_rng(5)
        for i, fraction in enumerate((0.5, 0.05, 0.0)):
            allowed = np.sort(rng.permutation(live)[:int(len(live) * fraction)])
            res = ref.filtered_search(q, k, allowed, threads=1)
            out[f"{name}/filtered_{i}_allowed"] = allowed
            for field, value in zip(("keys", "distances", "counts", "computed", "visited"), res):
                out[f"{name}/filtered_{i}_{field}"] = value
    x = np.random.default_rng(9).standard_normal((16, 256), dtype=np.float32) * np.float32(3.0)
    x[1, ::2] = 1e-30  # subnormal-sized inputs
    out["cast/input"] = x
    lib = bindings.ref_lib("parity")
    for scalar in ("f16", "bf16", "i8", "b1"):
        rows = []
        for row in x:
            buf = np.zeros(bindings.bytes_per_vector(x.shape[1], scalar), dtype=np.uint8)
            lib.ref_cast_from_f32(bindings.SCALAR[scalar], row.ctypes.data_as(bindings._f32p), x.shape[1],
                                  buf.ctypes.data_as(bindings.C.c_void_p))
            rows.append(buf.view(bindings.SCALAR_NP[scalar]))
        out[f"cast/{scalar}"] = np.stack(rows)
    np.savez_compressed(os.path.join(HERE, "port_extras.npz"), **out)


def build_quality():
    from build_check import exact_truth, hamming_truth, recall
    out = {}
    for metric, scalar, n, d, m in BUILD_CASES:
        base, queries = common.make_collection(n, d, scalar, 400)
        ref, _ = common.build_reference_blob(base, metric, scalar, d, m, threads=8)
        ref.change_expansion_search(64)
        truth = hamming_truth(base, queries, 10) if scalar == "b1" else exact_truth(base, queries, metric, 10)
        keys, _, _, computed, _ = ref.search(queries, 10, threads=8)
        out[f"{metric}/{scalar}/{n}/{d}/{m}"] = {"recall": round(float(recall(keys, truth)), 4),
                                                 "computed_per_query": round(float(computed.mean()), 1)}
        print(metric, scalar, out[f"{metric}/{scalar}/{n}/{d}/{m}"])
    with open(os.path.join(HERE, "build_quality.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    port_extras()
    build_quality()
