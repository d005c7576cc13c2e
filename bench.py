#!/usr/bin/env python
"""bench.py — the reference's headline metric (QPS of batched HNSW search at recall@10 >= 0.95) on B200.

One "step" = one batched `search()` over a fresh batch of synthetic queries against the index in HBM.
Default workload = the configuration BASELINE.json's metric is quoted on: 10M x 768 f32 cosine (M=32, ef=128,
batch 4096, k=10). The collection is generated on the GPU and the graph is BUILT on the GPU by the batched builder
(`usearch_b200_add_many_device`, csrc/builder.cu) in about a minute — the reference needs more than half an hour of
16-core time for the same graph — and both arms search that same graph.

  python bench.py --gpus 1 --steps K --warmup W            # our arm: CUDA path through the C ABI
  python bench.py --impl reference --steps K --warmup W    # the reference's own CPU search (oracle/_ref) of that graph
  torchrun ... bench.py --gpus N                           # N > 1: replicas (index fits one GPU) or shards (--parallelism)

See DESIGN.md §6 for what each JSON key means and how the roofline figure is derived.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from usearch_b200 import datagen  # noqa: E402

METRIC = "QPS @ recall@10>=0.95"
_REAL_STDOUT = sys.stdout
CHUNK = 262144  # rows generated at a time; chunk c of a collection is a pure function of (seed, c)
WORKLOADS = {  # BASELINE.json configs + the configuration its metric is quoted on (NS)
    "NS": dict(n=10_000_000, dim=768, metric="cos", dtype="f32", connectivity=32, ef=128, batch=4096),
    "C1": dict(n=100_000, dim=128, metric="l2sq", dtype="f32", connectivity=16, ef=64, batch=4096),
    "C2": dict(n=1_000_000, dim=768, metric="cos", dtype="f32", connectivity=32, ef=128, batch=4096),
    "C3": dict(n=10_000_000, dim=768, metric="cos", dtype="f16", connectivity=32, ef=256, batch=65536),
    "C4": dict(n=10_000_000, dim=1024, metric="ip", dtype="i8", connectivity=16, ef=128, batch=16384, parallelism="shard"),
    "C5": dict(n=100_000_000, dim=256, metric="hamming", dtype="b1", connectivity=64, ef=64, batch=32768, parallelism="shard"),
}


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


def host_threads() -> int:
    """Usable host cores: min(affinity, cgroup CPU quota)."""
    n = len(os.sched_getaffinity(0))
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--workload", default="NS", choices=sorted(WORKLOADS), help="a named configuration of BASELINE.json")
    # overrides of the named workload, for development runs only
    p.add_argument("--n", type=int)
    p.add_argument("--dim", type=int)
    p.add_argument("--metric")
    p.add_argument("--dtype")
    p.add_argument("--connectivity", type=int)
    p.add_argument("--ef", type=int)
    p.add_argument("--batch", type=int)
    p.add_argument("--expansion-add", type=int, default=128)
    p.add_argument("--k", type=int, default=10)
    p.add_argument("--rank-latent", type=int, default=16)
    p.add_argument("--cpu-sample-seconds", type=float, default=12.0)
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-next-rows", action="store_true")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="write what the last timed step returned (keys, distances, counts, both counters) as DIR/<name>.npy")
    p.add_argument("--builder", default="gpu", choices=["gpu", "reference"],
                   help="who builds the graph both arms search: the GPU builder (default) or the reference on the host cores")
    p.add_argument("--parallelism", default=None, choices=["replica", "shard"],
                   help="N > 1 only. replica (default when the index fits one GPU): every rank holds the whole index and serves "
                        "its own batches, no exchange step. shard (C4/C5: capacity): the collection is split by key, every "
                        "rank searches every query, ONE NCCL all-gather + merge kernel (csrc/shards.cu).")
    a = p.parse_args()
    w = WORKLOADS[a.workload]
    for key in ("n", "dim", "metric", "dtype", "connectivity", "ef", "batch"):
        if getattr(a, key) is None:
            setattr(a, key, w[key])
    if a.parallelism is None:
        a.parallelism = w.get("parallelism", "replica")
    return a


def workload_name(a) -> str:
    return (f"{a.n}x{a.dim} {a.dtype} {a.metric}, M={a.connectivity} ef={a.ef} batch={a.batch} k={a.k}, "
            f"rank-{a.rank_latent} latent synthetic")


# ------------------------------------------------------------------------------------------------
#  synthetic collection, generated chunk by chunk on the device (SURVEY.md §8d)
# ------------------------------------------------------------------------------------------------

class Collection:
    """Rank-r latent Gaussian rows x = z W + 0.1 eps (seeds 42 base / 43 queries / 44 mixing matrix), quantised to the
    index's scalar kind the way a user would before `add`. Chunk c is a pure function of (seed, c): the builder, the
    ground truth and the other arm regenerate exactly the same rows without keeping 30 GB around."""

    def __init__(self, a, device):
        import torch
        self.a, self.device, self.torch = a, device, torch
        w = np.random.default_rng(44).standard_normal((a.rank_latent, a.dim)).astype(np.float32)
        self.w = torch.from_numpy(w).to(device)

    def rows_f32(self, seed: int, chunk: int, rows: int):
        torch = self.torch
        g = torch.Generator(device=self.device)
        g.manual_seed(seed * 1_000_003 + chunk)
        z = torch.randn((rows, self.a.rank_latent), generator=g, device=self.device)
        e = torch.randn((rows, self.a.dim), generator=g, device=self.device)
        return z @ self.w + 0.1 * e

    def quantise(self, x):
        """f32 rows -> the tensor whose bytes are the vectors in the index's scalar kind."""
        torch, kind = self.torch, self.a.dtype
        if kind == "f32":
            return x.contiguous()
        if kind == "f16":
            return x.half().contiguous()
        if kind == "bf16":
            return x.bfloat16().contiguous()
        if kind == "i8":
            xd = x.double()
            return torch.clamp(torch.trunc(xd * 127.0 / xd.norm(dim=1, keepdim=True)), -127, 127).to(torch.int8).contiguous()
        if kind == "b1":
            bits = (x > 0).reshape(x.shape[0], -1, 8).to(torch.int32)
            weights = torch.tensor([128, 64, 32, 16, 8, 4, 2, 1], device=x.device, dtype=torch.int32)
            return (bits * weights).sum(dim=2).to(torch.uint8).contiguous()
        raise ValueError(kind)

    def as_float(self, q):
        """What the metric sees, as f32 (for ground truth): b1 -> +-1 per bit."""
        torch, kind = self.torch, self.a.dtype
        if kind == "b1":
            shifts = torch.tensor([7, 6, 5, 4, 3, 2, 1, 0], device=q.device, dtype=torch.int32)
            bits = ((q.to(torch.int32)[:, :, None] >> shifts) & 1).reshape(q.shape[0], -1)
            return bits.float() * 2 - 1
        return q.float()

    def base_chunks(self, shard: int = 0, shards: int = 1):
        """Yields (global row ids int64, quantised rows) of this shard (keys congruent to `shard` mod `shards`)."""
        torch = self.torch
        for c, lo in enumerate(range(0, self.a.n, CHUNK)):
            rows = min(CHUNK, self.a.n - lo)
            x = self.quantise(self.rows_f32(42, c, rows))
            ids = torch.arange(lo, lo + rows, device=self.device, dtype=torch.int64)
            if shards > 1:
                first = (shard - lo) % shards
                x, ids = x[first::shards].contiguous(), ids[first::shards].contiguous()
            yield ids, x

    def queries(self, total: int, stream: int = 0):
        out = []
        for c, lo in enumerate(range(0, total, CHUNK)):
            out.append(self.quantise(self.rows_f32(43 + 1000 * stream, c, min(CHUNK, total - lo))))
        return self.torch.cat(out, 0)


def build_index_gpu(a, coll: Collection, shard: int, shards: int):
    """Generate this shard's rows on the device and link them into the graph with the batched GPU builder."""
    import torch
    from usearch_b200.index import Index
    index = Index(ndim=a.dim, metric=a.metric, dtype=a.dtype, connectivity=a.connectivity, expansion_add=a.expansion_add,
                  expansion_search=a.ef)
    index.reserve((a.n + shards - 1) // shards)
    t0 = time.time()
    for ids, x in coll.base_chunks(shard, shards):
        index.add_device(ids.data_ptr(), x.data_ptr(), x.shape[0], x.stride(0) * x.element_size(), a.dtype)
    torch.cuda.synchronize()
    return index, time.time() - t0


def build_index_reference(a, coll: Collection, shard: int, shards: int, threads: int):
    """The same rows built by the UNMODIFIED reference on the host cores (small collections / cross-checks)."""
    import torch
    from oracle import bindings
    from usearch_b200.index import Index
    keys, rows = [], []
    for ids, x in coll.base_chunks(shard, shards):
        keys.append(ids.cpu().numpy().astype(np.uint64))
        rows.append(x.view(torch.uint8).reshape(x.shape[0], -1).cpu().numpy() if a.dtype == "bf16" else x.cpu().numpy())
    base = np.concatenate(rows, 0)
    if a.dtype == "bf16":
        base = base.view(np.uint16)
    ref = bindings.RefIndex("perf", metric=a.metric, scalar=a.dtype, dims=a.dim, connectivity=a.connectivity,
                            expansion_add=a.expansion_add, expansion_search=a.ef)
    t0 = time.time()
    ref.add(np.concatenate(keys), base, threads=threads)
    dt = time.time() - t0
    blob = ref.save()
    index = Index.restore(blob)
    index.expansion_search = a.ef
    return index, dt, blob


def exact_topk_gpu(a, coll: Collection, queries_q, k: int):
    """Brute-force ground truth over the WHOLE collection with torch (setup only, never timed)."""
    import torch
    q = coll.as_float(queries_q)
    if a.metric == "cos":
        q = torch.nn.functional.normalize(q, dim=1)
    torch.backends.cuda.matmul.allow_tf32 = False
    best_d = best_i = None
    for ids, xq in coll.base_chunks():
        x = coll.as_float(xq)
        if a.metric == "cos":
            x = torch.nn.functional.normalize(x, dim=1)
        if a.metric in ("cos", "ip"):
            dist = 1.0 - q @ x.T
        elif a.metric == "hamming":
            dist = (x.shape[1] - q @ x.T) * 0.5
        else:
            dist = (q * q).sum(1, keepdim=True) - 2.0 * (q @ x.T) + (x * x).sum(1)[None, :]
        d, i = torch.topk(dist, min(k, x.shape[0]), dim=1, largest=False)
        i = ids[i]
        if best_d is None:
            best_d, best_i = d, i
        else:
            cat_d, cat_i = torch.cat([best_d, d], 1), torch.cat([best_i, i], 1)
            best_d, sel = torch.topk(cat_d, k, dim=1, largest=False)
            best_i = torch.gather(cat_i, 1, sel)
    return best_i, best_d


def recall_at_k(found_keys: np.ndarray, counts: np.ndarray, truth: np.ndarray) -> float:
    hits = 0
    for i in range(found_keys.shape[0]):
        hits += len(set(found_keys[i, :int(counts[i])].tolist()) & set(truth[i].tolist()))
    return hits / float(truth.size)


def recall_at_k_with_ties(found_d: np.ndarray, counts: np.ndarray, truth_d: np.ndarray) -> float:
    """Binary codes have 257 possible Hamming distances: the k-th neighbour is usually one of many at the same distance and
    set intersection punishes an arbitrary choice among them. Here a found entry counts when its distance does not exceed the
    true k-th smallest distance (both sides count the same integer)."""
    kth = truth_d[:, -1:]
    ok = (found_d <= kth + 0.25) & (np.arange(found_d.shape[1])[None, :] < counts[:, None])
    return float(ok.sum()) / float(truth_d.size)


def to_numpy_queries(a, q):
    """Device query tensor -> the host array the C ABI / the reference take (bf16 travels as uint16)."""
    import torch
    if a.dtype == "bf16":
        return q.view(torch.uint16).cpu().numpy() if hasattr(torch, "uint16") else q.view(torch.int16).cpu().numpy().view(np.uint16)
    return q.cpu().numpy()


# ------------------------------------------------------------------------------------------------
#  clocks sampling (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------------

class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.samples = []
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 6 and parts[0].isdigit():
                self.samples.append(parts)

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(int(s[0]) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(s[2 + j].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(self.samples[0][1]), "reasons": reasons,
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
#  CPU reference timing
# ------------------------------------------------------------------------------------------------

def cpu_reference_qps(ref, queries: np.ndarray, k: int, threads: int):
    t0 = time.perf_counter()
    res = ref.search(queries, k, threads=threads, counters=True)
    dt = time.perf_counter() - t0
    return len(queries) / dt, dt, res


def run_reference_arm(a):
    """The reference's own CPU implementation of the path, all usable host threads, on the SAME graph as our arm
    (built on the GPU unless --builder reference, saved in the v2 format, `view`ed by the reference: no copy)."""
    import torch
    from oracle import bindings
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl reference: the collection is generated and its graph built on a GPU")
    threads = host_threads()
    device = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    os.environ["USEARCH_B200_DEVICE"] = "0"
    coll = Collection(a, device)
    info = {"builder": a.builder}
    if a.builder == "gpu":
        index, dt = build_index_gpu(a, coll, 0, 1)
        info["build_s"] = round(dt, 1)
        t0 = time.time()
        blob = index.save()
        info["save_s"] = round(time.time() - t0, 1)
    else:
        index, dt, blob = build_index_reference(a, coll, 0, 1, threads)
        info.update(build_s=round(dt, 1), build_threads=threads)
    ref = bindings.RefIndex("perf")
    ref.view(blob)
    ref.change_expansion_search(a.ef)
    total = (a.warmup + a.steps) * a.batch
    q_dev = coll.queries(total)
    queries = to_numpy_queries(a, q_dev)
    for s in range(a.warmup):
        cpu_reference_qps(ref, queries[s * a.batch:(s + 1) * a.batch], a.k, threads)
    t0 = time.perf_counter()
    found = []
    for s in range(a.warmup, a.warmup + a.steps):
        _, _, res = cpu_reference_qps(ref, queries[s * a.batch:(s + 1) * a.batch], a.k, threads)
        found.append(res)
    dt = time.perf_counter() - t0
    qps = a.steps * a.batch / dt
    recall = None
    try:
        R = min(a.batch, 2048)
        gt, _ = exact_topk_gpu(a, coll, q_dev[a.warmup * a.batch:a.warmup * a.batch + R], a.k)
        recall = round(recall_at_k(found[0][0][:R], found[0][2][:R], gt.cpu().numpy().astype(np.uint64)), 4)
    except Exception as e:  # ground truth is optional for this arm
        log("ground truth skipped:", e)
    line = {
        "impl": "reference", "metric": METRIC, "value": round(qps, 1), "unit": "queries/s", "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": round(1000 * dt / a.steps, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": a.dtype, "data": "synthetic",
        "config": {"workload": workload_name(a), "isa": ref.isa_name, "index_build": info,
                   "computed_distances_per_query": round(float(np.mean([r[3].mean() for r in found])), 1)},
        "recall_at_10": recall,
        "cpu_baseline": {"value": round(qps, 1), "unit": "queries/s", "cores": threads, "kind": "reference",
                         "sample": f"{a.steps} batches of {a.batch} queries, reference built -O3 -ffast-math -march=native, SimSIMD {ref.isa_name}"},
        "e2e": {"value": round(qps, 1), "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), file=_REAL_STDOUT, flush=True)


# ------------------------------------------------------------------------------------------------
#  our arm
# ------------------------------------------------------------------------------------------------

def measure_next_rows(a, index, ref, batch: np.ndarray, k: int, threads: int) -> dict:
    """SURVEY §8(f) rows on the bench collection, outside the timed region of the headline metric: wall clock of one
    call through the host API, the reference timed on a bounded sample of the same batch, and label agreement on that
    sample. Never raises: a failure is reported in the JSON instead of losing the line."""
    out = {}
    batch = batch[:4096]
    try:
        index.search(batch[:256], k, exact=True)  # warm-up (scratch allocation)
        t0 = time.perf_counter()
        exact = index.search(batch, k, exact=True)
        dt = time.perf_counter() - t0
        sample = batch[:max(threads // 2, 4)]  # the reference scans 10M x 768 at ~1 query/s on 16 cores: keep this leg to seconds
        t0 = time.perf_counter()
        want = ref.search(sample, k, threads=threads, exact=True)
        dt_cpu = time.perf_counter() - t0
        out["exact_search"] = {
            "value": round(len(batch) / dt, 1), "unit": "queries/s", "ms_per_batch": round(dt * 1e3, 1),
            "multiply_adds_per_s": round(len(batch) * index.size * a.dim / dt / 1e12, 2), "multiply_adds_unit": "T/s",
            "cpu_reference": {"value": round(len(sample) / dt_cpu, 1), "unit": "queries/s", "cores": threads,
                              "sample": f"{len(sample)} queries in {dt_cpu:.1f} s, index.search(exact=True)"},
            "rows_with_identical_labels": round(float((want[0] == exact.keys[:len(sample)]).all(axis=1).mean()), 4),
        }
    except Exception as e:  # noqa: BLE001
        out["exact_search"] = {"error": str(e)}
    try:
        level = 1
        index.cluster(batch[:256], level)
        t0 = time.perf_counter()
        gk, gd = index.cluster(batch, level, stats=True)
        dt = time.perf_counter() - t0
        sample = batch[:1024]
        t0 = time.perf_counter()
        wk, wd, wc, wv = ref.cluster(sample, level)
        dt_cpu = time.perf_counter() - t0
        out["cluster"] = {
            "value": round(len(batch) / dt, 1), "unit": "queries/s", "level": level, "ms_per_batch": round(dt * 1e3, 2),
            "cpu_reference": {"value": round(len(sample) / dt_cpu, 1), "unit": "queries/s", "cores": 1,
                              "sample": f"{len(sample)} queries in {dt_cpu:.2f} s, index.cluster(vector, {level})"},
            "rows_with_identical_members": round(float((wk == gk[:len(sample)]).mean()), 4),
            "counters_identical": bool(np.array_equal(wc, index.last_computed[:len(sample)])),
        }
    except Exception as e:  # noqa: BLE001
        out["cluster"] = {"error": str(e)}
    try:
        allowed = np.arange(0, a.n, 10, dtype=np.uint64)  # one key in ten passes the predicate
        index.filtered_search(batch[:256], k, allowed)
        t0 = time.perf_counter()
        got = index.filtered_search(batch, k, allowed)
        dt = time.perf_counter() - t0
        row = {"value": round(len(batch) / dt, 1), "unit": "queries/s", "ms_per_batch": round(dt * 1e3, 2),
               "predicate": "key % 10 == 0 (bitmap over slots built on the device from the sorted key list)",
               "all_labels_pass_predicate": bool((got.keys[got.distances == got.distances] % 10 == 0).all())}
        if a.dtype == "f32":
            sample = batch[:512]
            t0 = time.perf_counter()
            want = ref.filtered_search(sample, k, allowed, threads=threads)
            dt_cpu = time.perf_counter() - t0
            row["cpu_reference"] = {"value": round(len(sample) / dt_cpu, 1), "unit": "queries/s", "cores": threads,
                                    "sample": f"{len(sample)} queries in {dt_cpu:.2f} s, filtered_search"}
            row["rows_with_identical_labels"] = round(float((want[0] == got.keys[:len(sample)]).all(axis=1).mean()), 4)
        out["filtered_search"] = row
    except Exception as e:  # noqa: BLE001
        out["filtered_search"] = {"error": str(e)}
    return out


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, keys, distances, counts, computed, visited) -> None:
    """The arrays search_device returned for one batch, as float64 (keys, counts, counters: exact below 2**53) and float32
    (distances, bit for bit; padding stays NaN). A 4096-query batch at k = 10 is about 0.6 MB. A batch larger than
    DUMP_LIMIT_BYTES in all is cut to a fixed, seeded sample of its rows, whose numbers go to rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    b, k = keys.shape
    per_row = k * (8 + 4) + 3 * 8
    rows = None
    if b * per_row > DUMP_LIMIT_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(b, (DUMP_LIMIT_BYTES - 4096) // (per_row + 8), replace=False))
        np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))
    for name, t, dtype in (("keys", keys, np.float64), ("distances", distances, np.float32), ("counts", counts, np.float64),
                           ("computed_distances", computed, np.float64), ("visited_members", visited, np.float64)):
        a = t.cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), (a if rows is None else a[rows]).astype(dtype))


def run_b200_arm(a):
    import torch
    import torch.distributed as dist
    from usearch_b200 import sharded

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 arm has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    os.environ["USEARCH_B200_DEVICE"] = str(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    # replica: every rank holds the whole index and serves its own batches; shard: rank r holds the keys congruent to r
    shards = world if (a.parallelism == "shard" and world > 1) else 1
    shard_id = rank if shards > 1 else 0
    threads = max(1, host_threads() // world)
    coll = Collection(a, device)
    info = {"builder": a.builder}
    blob = None
    if a.builder == "gpu":
        index, dt = build_index_gpu(a, coll, shard_id, shards)
        info["build_s"] = round(dt, 1)
    else:
        index, dt, blob = build_index_reference(a, coll, shard_id, shards, threads)
        info.update(build_s=round(dt, 1), build_threads=threads)
    index.expansion_search = a.ef
    log(f"rank {rank}: {len(index)} vectors in HBM ({index.memory_usage / 1e9:.2f} GB), graph built by '{a.builder}' in {info['build_s']} s")
    if shards > 1:
        sharded.join(index)

    B, k, W, K = a.batch, a.k, a.warmup, a.steps
    total = (W + K) * B
    # shards: the batch is replicated; replicas serve different batches
    q_dev = coll.queries(total, stream=0 if (shards > 1 or world == 1) else rank)
    bpv = q_dev.stride(0) * q_dev.element_size()
    vs = (bpv + 15) // 16 * 16
    if vs != bpv:
        padded = torch.zeros((total, vs), dtype=torch.uint8, device=device)
        padded[:, :bpv] = q_dev.view(torch.uint8).reshape(total, bpv)
        q_bytes = padded
    else:
        q_bytes = q_dev.view(torch.uint8).reshape(total, bpv)

    keys_dev = torch.zeros((B, k), dtype=torch.int64, device=device)
    dist_dev = torch.zeros((B, k), dtype=torch.float32, device=device)
    cnt_dev = torch.zeros(B, dtype=torch.int32, device=device)
    comp_dev = torch.zeros(B, dtype=torch.int32, device=device)
    vis_dev = torch.zeros(B, dtype=torch.int32, device=device)
    # An explicit stream for everything that follows: the library launches on the stream it is given (0 / the legacy default
    # stream would mean "the handle's own stream", which torch's events and copies are not ordered with).
    stream = torch.cuda.Stream(device)
    torch.cuda.synchronize(device)
    torch.cuda.set_stream(stream)
    search_device = index.sharded_search_device if shards > 1 else index.search_device

    def step_device(s: int):
        qs = q_bytes[s * B:(s + 1) * B]
        search_device(qs.data_ptr(), B, vs, k, keys_dev.data_ptr(), dist_dev.data_ptr(), cnt_dev.data_ptr(),
                      comp_dev.data_ptr(), vis_dev.data_ptr(), stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    # ---- warm-up ----
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.5)  # nvidia-smi needs a moment before its first sample
    for s in range(W):
        step_device(s)
        comp_dev.sum(dtype=torch.int64), vis_dev.sum(dtype=torch.int64), keys_dev.clone(), cnt_dev.clone()
    barrier()

    # ---- timed: device-resident ----
    launches0 = index.kernel_launches
    kernel_ms, alg_bytes = [], []
    m0 = 2 * index.connectivity
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ncu_range = os.environ.get("USEARCH_B200_NCU_RANGE") == "1"  # `ncu --profile-from-start off`: only the timed steps are listed
    if ncu_range:
        torch.cuda.profiler.start()
    ev0.record(stream)
    first_found = None
    for s in range(W, W + K):
        step_device(s)
        kernel_ms.append(index.last_kernel_ms)
        alg_bytes.append((comp_dev.sum(dtype=torch.int64), vis_dev.sum(dtype=torch.int64)))
        if first_found is None:
            first_found = (keys_dev.clone(), dist_dev.clone(), cnt_dev.clone())
            first_counters = (comp_dev.cpu().numpy().astype(np.uint64), vis_dev.cpu().numpy().astype(np.uint64))
    ev1.record(stream)
    barrier()
    if ncu_range:
        torch.cuda.profiler.stop()
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, keys_dev, dist_dev, cnt_dev, comp_dev, vis_dev)
    launches = index.kernel_launches - launches0
    elapsed_ms = ev0.elapsed_time(ev1)
    t = torch.tensor([elapsed_ms], device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    alg = [(int(D.item()) * index.bytes_per_vector + int(H.item()) * (4 + 4 * m0)) for D, H in alg_bytes]
    d_per_q = sum(int(D.item()) for D, _ in alg_bytes) / (K * B)
    h_per_q = sum(int(H.item()) for _, H in alg_bytes) / (K * B)

    # ---- timed: end to end through the host C ABI (pinned host buffers, H2D + D2H inside) ----
    q_pin = q_dev.view(torch.uint8).reshape(total, bpv).cpu().pin_memory()
    np_dtype = {"f32": np.float32, "f16": np.float16, "bf16": np.uint16, "i8": np.int8, "b1": np.uint8}[a.dtype]
    q_host = q_pin.numpy().view(np_dtype).reshape(total, -1)
    search_host = index.sharded_search if shards > 1 else index.search
    for s in range(W):
        search_host(q_host[s * B:(s + 1) * B], k)
    barrier()
    t0 = time.perf_counter()
    for s in range(W, W + K):
        res = search_host(q_host[s * B:(s + 1) * B], k)
    barrier()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], device=device)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te.item())

    # ---- quality gate: recall@10 against exact ground truth over the whole collection ----
    R = min(B, 2048)
    q0 = q_dev[W * B:W * B + R]
    gt_k, gt_d = exact_topk_gpu(a, coll, q0, k)
    found_k, found_d, found_c = first_found
    recall = recall_at_k(found_k.cpu().numpy().astype(np.uint64)[:R], found_c.cpu().numpy()[:R], gt_k.cpu().numpy().astype(np.uint64))
    recall_ties = None
    if a.dtype == "b1":
        recall_ties = recall_at_k_with_ties(found_d.cpu().numpy()[:R], found_c.cpu().numpy()[:R], gt_d.cpu().numpy())
    log(f"rank {rank}: recall@{k} of its first timed batch ({R} rows) = {recall:.4f}; row 0 found {found_k[0].tolist()} truth {gt_k[0].tolist()}")
    if world > 1:  # every rank checks its own batch (replicas) or the same merged batch (shards)
        rt = torch.tensor([recall], device=device)
        dist.all_reduce(rt, op=dist.ReduceOp.MIN)
        recall = float(rt.item())

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- CPU baseline on a bounded sample + full-size parity (rank 0, N=1 only) ----
    cpu = None
    next_rows = None
    from oracle import bindings
    if world == 1 and not a.no_cpu_baseline and bindings.ref_lib("perf") is None:
        log("cpu_baseline skipped: the reference library (oracle/_ref) is not built")
    elif world == 1 and not a.no_cpu_baseline:
        threads_all = host_threads()
        t0 = time.time()
        if blob is None:
            blob = index.save()
        info["save_s"] = round(time.time() - t0, 1)
        ref = bindings.RefIndex("perf")
        ref.view(blob)
        ref.change_expansion_search(a.ef)
        queries = q_host
        pilot_qps, _, _ = cpu_reference_qps(ref, queries[:256], k, threads_all)
        sample = int(min(total, max(512, pilot_qps * a.cpu_sample_seconds)))
        qps_cpu, dt_cpu, res_cpu = cpu_reference_qps(ref, queries[:sample], k, threads_all)
        cpu = {"value": round(qps_cpu, 1), "unit": "queries/s", "cores": threads_all, "kind": "reference",
               "sample": f"{sample} queries of the same workload in {dt_cpu:.1f} s, reference -O3 -ffast-math -march=native, SimSIMD {ref.isa_name}",
               "computed_distances_per_query": round(float(res_cpu[3].mean()), 1),
               "visited_members_per_query": round(float(res_cpu[4].mean()), 1)}
        # full-size parity property on the first timed batch (<= 4096 rows): labels + counters against the reference's
        # NATIVE SimSIMD kernels (cosine differs by <= 1 ULP from the pinned arithmetic, so near-ties may swap), and
        # labels + distance BITS + counters against the reference with the metric pinned (oracle/metrics_pinned.h)
        P = min(B, 4096)
        lo = W * B
        gpu_keys = found_k.cpu().numpy().astype(np.uint64)[:P]
        gpu_bits = found_d.cpu().numpy().view(np.uint32)[:P]
        native = ref.search(queries[lo:lo + P], k, threads=threads_all, counters=True)
        cpu["gpu_rows_with_identical_labels"] = round(float((native[0] == gpu_keys).all(axis=1).mean()), 6)
        cpu["gpu_counters_identical"] = bool(np.array_equal(native[3], first_counters[0][:P]) and
                                             np.array_equal(native[4], first_counters[1][:P]))
        try:
            pinned_ref = bindings.RefIndex("parity")
            pinned_ref.view(blob)
            pinned_ref.change_expansion_search(a.ef)
            pinned_ref.pin_metric(True)
            pinned = pinned_ref.search(queries[lo:lo + P], k, threads=threads_all, counters=True)
            cpu["parity_rows_checked"] = P
            cpu["parity_pinned_rows_with_identical_labels"] = round(float((pinned[0] == gpu_keys).all(axis=1).mean()), 6)
            cpu["parity_pinned_distance_bits_identical"] = bool(np.array_equal(pinned[1].view(np.uint32), gpu_bits))
            cpu["parity_pinned_counters_identical"] = bool(np.array_equal(pinned[3], first_counters[0][:P]) and
                                                           np.array_equal(pinned[4], first_counters[1][:P]))
            del pinned_ref
        except Exception as e:  # noqa: BLE001
            cpu["parity_pinned_error"] = str(e)
        if not a.no_next_rows:
            next_rows = measure_next_rows(a, index, ref, queries[lo:lo + B], k, threads_all)
        del ref

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    k_ms = float(np.mean(kernel_ms))
    achieved = float(np.mean(alg)) / (k_ms * 1e-3) / 1e9
    traffic = None  # DRAM bytes per launch from an `ncu --set full` capture of this very workload at this N, else null
    prof = os.path.join(ROOT, "profiles", "roofline_latest.json")
    if os.path.exists(prof):
        try:
            pj = json.load(open(prof))
            if pj.get("workload") == workload_name(a) and int(pj.get("n_gpus", 1)) == world and pj.get("parallelism", "replica") == a.parallelism:
                traffic = pj.get("dram_bytes_per_launch")
        except Exception:
            pass

    # the metric is job throughput: queries answered per second. Replicas answer `world` different batches per step,
    # shards answer ONE batch per step between them.
    queries_per_step = B * (world if shards == 1 else 1)
    value = queries_per_step * K / (elapsed_ms * 1e-3)
    parallelism = "single GPU" if world == 1 else (
        f"shard-by-key x{world}: every rank searches the whole batch in its shard, one NCCL all-gather + merge kernel" if shards > 1
        else f"{world} replicas of the whole index, one batch of {B} per replica per step, no exchange step")
    line = {
        "metric": METRIC, "value": round(value, 1), "unit": "queries/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": round(elapsed_ms / K, 3), "higher_is_better": True, "scaling": "weak" if shards == 1 else "strong",
        "vs_baseline": None, "dtype": a.dtype, "data": "synthetic",
        "config": {
            "workload": workload_name(a), "parallelism": parallelism, "queries_per_step": queries_per_step,
            "l2_policy": "index (vectors+graph) larger than the 126 MB L2; every step uses a fresh query batch",
            "index_hbm_gb": round(index.memory_usage / 1e9, 3), "index_build": info,
            "computed_distances_per_query": round(d_per_q, 1), "visited_members_per_query": round(h_per_q, 1),
        },
        "recall_at_10": round(recall, 4),
        **({"recall_at_10_counting_ties": round(recall_ties, 4)} if recall_ties is not None else {}),
        "gpu_launches": int(launches),
        "clocks": clocks,
        "e2e": {"value": round(queries_per_step * K / e2e_s, 1), "unit": "queries/s", "h2d_bytes_per_step": int(B * bpv),
                "d2h_bytes_per_step": int(B * k * 12 + B * 4),
                "note": ("usearch_b200_sharded_search_many" if shards > 1 else "usearch_search_many") +
                        " on pinned host buffers; H2D of queries and D2H of keys/distances/counts inside the timed call"},
        "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                     "frac": round(achieved / peak, 4), "traffic": traffic, "peak_source": peak_src,
                     "kernel": "hnsw_search_kernel", "kernel_ms_per_launch": round(k_ms, 3),
                     "algorithmic_bytes_per_launch": int(np.mean(alg)),
                     "formula": "sum_q D_q*bytes_per_vector + H_q*(4+4*M0), D/H = the reference's computed_distances/visited_members; rank 0's launch"},
        "cpu_baseline": cpu,
    }
    if shards > 1:  # what the exchange step costs: the step minus this rank's search kernel
        line["config"]["exchange_ms_per_step"] = round(elapsed_ms / K - k_ms, 3)
    if next_rows:
        line["next_rows"] = next_rows
    print(json.dumps(line), file=_REAL_STDOUT, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    a = parse_args()
    # The contract is ONE JSON line on stdout. Libraries (NCCL prints its version on fd 1 at communicator creation) must not
    # get in its way: everything that writes to fd 1 goes to stderr, only the JSON line goes to the real stdout.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if a.impl == "reference":
        run_reference_arm(a)
    else:
        run_b200_arm(a)


if __name__ == "__main__":
    main()
