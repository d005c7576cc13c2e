"""Generate tests/golden/reference_cases.npz by RUNNING THE UNMODIFIED REFERENCE (oracle/_ref, needs the reference
sources):  python tests/golden/make_golden_reference_cases.py

Each case is one uint8 array holding an uncompressed .npz of its arrays (common.golden_case reads one), which keeps
the per-array overhead of the outer archive small.

The configurations of test_oracle.py's live-reference tests (common.GOLDEN_*_CASES, the first
common.GOLDEN_SMALL_CASES of common.small_random_cases), at sizes that keep the file small. Graphs are built by the
reference single-threaded (reproducible) from common.make_collection; each case stores the serialised graph WITHOUT
its vector matrix (`graph`: the vectors are regenerated from the same seeds; `inputs_sha256` checks that they came out
the same), and what the reference returned with the metric pinned:
  * ``search_{keys,distances,counts,computed,visited}`` and ``exact_{keys,distances,counts}``,
  * ``cluster_{levels,keys,distances,computed,visited}``,
  * ``free_{keys,distances}``: exact_search_t over the raw rows, next to the index's exact search,
  * case ``native``: ``<metric>_<scalar>``: the reference's NATIVE SimSIMD distances of consecutive rows of
    common.native_metric_rows() (regenerated, checked by ``<metric>_<scalar>_sha256``), and the host's ``isa``.
"""
import io
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import common  # noqa: E402
from oracle import bindings  # noqa: E402

digest, strip_vectors = common.digest, common.strip_vectors


def pack(arrays: dict) -> np.ndarray:
    buf = io.BytesIO()
    np.savez(buf, **arrays)
    return np.frombuffer(buf.getvalue(), dtype=np.uint8)


def searched(ref, blob, base, q, k) -> dict:
    c = {"graph": strip_vectors(blob), "inputs_sha256": digest(base, q)}
    for field, v in zip(("keys", "distances", "counts", "computed", "visited"), ref.search(q, k, threads=1)):
        c[f"search_{field}"] = v
    for field, v in zip(("keys", "distances", "counts"), ref.search(q, k, threads=1, exact=True)[:3]):
        c[f"exact_{field}"] = v
    return c


def clustered(ref, q, levels) -> dict:
    res = [ref.cluster(q, level) for level in levels]
    c = {"cluster_levels": np.array(levels)}
    for i, field in enumerate(("keys", "distances", "computed", "visited")):
        c[f"cluster_{field}"] = np.stack([r[i] for r in res])
    return c


def main():
    out = {}
    for name, metric, scalar, n, d, m, ef, k in common.GOLDEN_SEARCH_CASES:
        base, q = common.make_collection(n, d, scalar, common.GOLDEN_NQ, iid=(d < 32))
        ref, blob = common.build_reference_blob(base, metric, scalar, d, m, threads=1)
        ref.pin_metric(True)
        ref.change_expansion_search(ef)
        out[name] = pack(searched(ref, blob, base, q, k))
    for name, metric, scalar, n, d, m in common.GOLDEN_CLUSTER_CASES:
        base, q = common.make_collection(n, d, scalar, common.GOLDEN_NQ)
        ref, blob = common.build_reference_blob(base, metric, scalar, d, m, threads=1)
        ref.pin_metric(True)
        assert ref.max_level >= 3
        out[name] = pack({"graph": strip_vectors(blob), "inputs_sha256": digest(base, q),
                          **clustered(ref, q, [0, 1, 2, ref.max_level, ref.max_level + 3])})
    # the two brute-force oracles on one collection: exact_search_t over the raw rows and the index's exact search
    base, q = common.make_collection(300, 48, "f32", common.GOLDEN_NQ, iid=True)
    ref, blob = common.build_reference_blob(base, "l2sq", "f32", 48, 8, expansion_add=16, threads=1)
    ref.pin_metric(True)
    c = searched(ref, blob, base, q, 10)
    c["free_keys"], c["free_distances"] = bindings.ref_exact_search(base, q, 10, metric="l2sq", scalar="f32", dims=48)
    out["free_l2sq_f32"] = pack(c)
    # the reference's native kernels on this host's ISA, for the pinned-vs-native comparison
    c = {}
    for metric, scalar, d, x in common.native_metric_rows():
        ref = bindings.RefIndex("parity", metric=metric, scalar=scalar, dims=d, connectivity=4)
        c[f"{metric}_{scalar}"] = np.array([ref.distance(x[i], x[i + 1]) for i in range(len(x) - 1)], np.float32)
        c[f"{metric}_{scalar}_sha256"] = digest(x)
        c["isa"] = ref.isa_name
    out["native"] = pack(c)
    # the seeded random small cases
    for case, c in enumerate(common.small_random_cases(common.GOLDEN_SMALL_CASES)):
        ref, _ = common.build_reference_blob(c["base"], c["metric"], c["scalar"], c["d"], c["m"],
                                             expansion_add=c["expansion_add"], threads=1, keys=c["keys"])
        for key in c["removed"]:
            ref.remove(int(key))
        blob = ref.save()
        ref.pin_metric(True)
        ref.change_expansion_search(c["ef"])
        g = searched(ref, blob, c["base"], c["q"], c["k"])
        if ref.size:
            g.update(clustered(ref, c["q"], [0, 1, ref.max_level + 1]))
        out[f"small_{case}"] = pack(g)
    path = os.path.join(HERE, "reference_cases.npz")
    np.savez_compressed(path, **out)
    print(f"{len(out)} cases, {os.path.getsize(path)} bytes")


if __name__ == "__main__":
    main()
