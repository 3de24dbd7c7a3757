#!/usr/bin/env python
"""bench.py -- batched HNSW search throughput of the B200 engine (and of the reference on the host cores).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg3|cfg2|cfg4|cfg5s|...]

One "step" = one batch of queries through the hot path (greedy descent + ef-wide base-layer beam + top-k) over a
synthetic corpus resident in HBM.  Default workload = the configuration BASELINE.json's metric is quoted on ("d=768 fp32,
10M vectors, batch 4096", configs[2], "cfg3"; 30.7 GB, fits one B200): 10 M x d768 fp32, structured synthetic
(x = z P + 0.05 eps, 32-d latent, SURVEY.md 8d), cosine, M=32, ef_construction=128, ef=128, batch 4096, k=10, on
1/2/4/8 GPUs (row-range shards).  `--workload cfg2` = configs[1] (1 M, l2sq, M=16, ef=64, batch 1024), and so on.
The graph is built by the engine itself on the GPU (lb200_add_batch_device + lb200_build) before the timed region.

`value`  : queries/s, queries already resident in HBM (lb200_search_batch_device), CUDA events on the launching stream.
`e2e`    : the same through the reference-facing host call (lb200_search_batch: pinned host buffers in and out,
           H2D/D2H inside the timed region).
`roofline`: algorithmic bytes (SURVEY.md 8d: n_dist*row_bytes + pops*(4+4*M0) + hops*(4+4*M) + query bytes, counters
           returned by the kernel itself and equal to usearch's computed_distances) / search-kernel device time,
           against the measured HBM copy bandwidth in MEASURED_PEAKS.json.
`cpu_baseline`: the UNMODIFIED reference (oracle/_ref, usearch compiled from /root/reference) on all host cores,
           loading the very index file the engine wrote (usearch file format) and searching the same queries --
           which also yields the same-graph id parity reported under `parity`.  Corpora above 8 GB (cfg3): the engine
           builds a second graph over the first --cpu-prefix-rows rows for this purpose (bounded sample).
--impl reference: the reference alone on the host cores: builds its own graph over a bounded number of rows of the
           corpus generator (sized for ~1 minute of multi-threaded adds) and searches the same query batches.
Steps cycle through a pool of distinct query batches; the corpus (30.7 GB; 3 GB for cfg2), gathered at random, is far
larger than L2 (126 MB).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (n, dim, metric, M, efc, ef, batch, k, description)
    "cfg2": dict(n=1_000_000, dim=768, metric="l2sq", M=16, efc=128, ef=64, batch=1024, k=10,
                 desc="cfg2: 1M x d768 f32 l2sq, M=16 efc=128 ef=64, batch-1024 k=10"),
    "cfg2s": dict(n=100_000, dim=768, metric="l2sq", M=16, efc=128, ef=64, batch=1024, k=10,
                  desc="cfg2s (smoke-size): 100k x d768 f32 l2sq, M=16 efc=128 ef=64, batch-1024 k=10"),
    # recall_1gpu: recall@10 of the unsharded graph at this ef as measured by the 1-GPU run of this very bench
    # (profiles/r01_bench_cfg3_10M_cos.json); the sharded runs match it when --recall-target is not given
    "cfg3": dict(n=10_000_000, dim=768, metric="cos", M=32, efc=128, ef=128, batch=4096, k=10, recall_1gpu=0.88125,
                 desc="cfg3: 10M x d768 f32 cosine, M=32 efc=128 ef=128, batch-4096 k=10"),
    "cfg3s": dict(n=1_000_000, dim=768, metric="cos", M=32, efc=128, ef=128, batch=4096, k=10,
                  desc="cfg3s (1/10 scale): 1M x d768 f32 cosine, M=32 efc=128 ef=128, batch-4096 k=10"),
    "cfg4": dict(n=10_000_000, dim=1536, metric="l2sq", M=16, efc=128, ef=64, batch=4096, k=100, pq=(96, 256),
                 desc="cfg4: 10M x d1536 f32 -> PQ 96 subvectors x 256 centroids, l2sq, M=16 efc=128 ef=64 (expansion 100), batch-4096 k=100"),
    "cfg4s": dict(n=1_000_000, dim=1536, metric="l2sq", M=16, efc=128, ef=64, batch=4096, k=100, pq=(96, 256),
                  desc="cfg4s (1/10 scale): 1M x d1536 f32 -> PQ 96x256, l2sq, M=16 efc=128 ef=64 (expansion 100), batch-4096 k=100"),
    # BASELINE configs[4] is 50M x 768-byte binary vectors over 8 GPUs: one shard's worth (6.25M) on one GPU
    "cfg5": dict(n=50_000_000, dim=6144, kind="b1", metric="hamming", M=16, efc=128, ef=64, batch=4096, k=10,
                 desc="cfg5: 50M x 6144-bit (768 B) hamming, M=16 efc=128 ef=64, batch-4096 k=10 (build + search, 8 GPUs)"),
    "cfg5s": dict(n=6_250_000, dim=6144, kind="b1", metric="hamming", M=16, efc=128, ef=64, batch=4096, k=10,
                  desc="cfg5s (one of 8 shards of cfg5): 6.25M x 6144-bit (768 B) hamming, M=16 efc=128 ef=64, batch-4096 k=10"),
    "cfg5t": dict(n=500_000, dim=6144, kind="b1", metric="hamming", M=16, efc=128, ef=64, batch=4096, k=10,
                  desc="cfg5t (small): 500k x 6144-bit (768 B) hamming, M=16 efc=128 ef=64, batch-4096 k=10"),
}
METRIC_NAME = "queries/sec @ recall@10, d=768 fp32, 10M vectors, batch 4096, 1/2/4/8 B200"
LATENT, NOISE = 32, 0.05
BIG_CORPUS_BYTES = 8e9  # above this the index file is not handed to the reference whole (cpu_baseline) nor rebuilt unsharded per rank
DEVICE_TYPE, DIST_BACKEND = "cuda", "nccl"  # tests/test_bench_dryrun.py walks run_ours on the CPU with a stand-in engine
SEED_P, SEED_CORPUS, SEED_QUERY = 1234, 42, 43


# --------------------------------------------------------------------------------------- synthetic data
def projection_np(dim):
    return (np.random.default_rng(SEED_P).standard_normal((LATENT, dim)) / np.sqrt(LATENT)).astype(np.float32)


def structured_np(n, dim, seed, chunk=100_000):
    """Host generator (reference arm): x = z P + NOISE * eps."""
    P = projection_np(dim)
    out = np.empty((n, dim), np.float32)
    rng = np.random.default_rng(seed)
    for lo in range(0, n, chunk):
        hi = min(n, lo + chunk)
        z = rng.standard_normal((hi - lo, LATENT), dtype=np.float32)
        out[lo:hi] = z @ P + NOISE * rng.standard_normal((hi - lo, dim), dtype=np.float32)
    return out


def structured_torch(n, dim, seed, device, chunk=200_000):
    """Device generator (our arm).  Same distribution as structured_np (different random stream)."""
    import torch
    P = torch.from_numpy(projection_np(dim)).to(device)
    out = torch.empty((n, dim), dtype=torch.float32, device=device)
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    for lo in range(0, n, chunk):
        hi = min(n, lo + chunk)
        z = torch.randn((hi - lo, LATENT), generator=g, device=device)
        out[lo:hi] = z @ P
        out[lo:hi] += NOISE * torch.randn((hi - lo, dim), generator=g, device=device)
    return out


def bits_torch(n, bits, seed, device, chunk=100_000, protos=64, flip=0.10):
    """Binary vectors (SURVEY.md 8d cfg 5): one of 64 random prototypes XOR 10 % random bit flips, packed MSB-first."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(SEED_P)
    proto = torch.randint(0, 256, (protos, bits // 8), generator=g, device=device, dtype=torch.uint8)
    g.manual_seed(seed)
    out = torch.empty((n, bits // 8), dtype=torch.uint8, device=device)
    w = torch.tensor([128, 64, 32, 16, 8, 4, 2, 1], device=device, dtype=torch.uint8)
    for lo in range(0, n, chunk):
        hi = min(n, lo + chunk)
        which = torch.randint(0, protos, (hi - lo,), generator=g, device=device)
        flips = (torch.rand((hi - lo, bits // 8, 8), generator=g, device=device) < flip).to(torch.uint8)
        out[lo:hi] = proto[which] ^ (flips * w).sum(dim=2).to(torch.uint8)
    return out


def bits_np(n, bits, seed, chunk=100_000, protos=64, flip=0.10):
    proto = np.random.default_rng(SEED_P).integers(0, 256, (protos, bits // 8), dtype=np.uint8)
    rng = np.random.default_rng(seed)
    out = np.empty((n, bits // 8), np.uint8)
    for lo in range(0, n, chunk):
        hi = min(n, lo + chunk)
        which = rng.integers(0, protos, hi - lo)
        out[lo:hi] = proto[which] ^ np.packbits(rng.random((hi - lo, bits)) < flip, axis=1)
    return out


# --------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "20"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def recall_at_k(found, truth):
    hits = 0
    for f, t in zip(found, truth):
        hits += len(set(f.tolist()) & set(t.tolist()))
    return hits / float(truth.size)


def usable_cores():
    """Host threads this process may actually run on: the affinity mask, capped by the cgroup CPU quota (a container on a
    128-core box may be limited to far fewer; std::thread::hardware_concurrency() reports the box)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        pass
    return max(1, n)


def parity_block(gk, gd, rk, rd, rtol=1e-5, atol=1e-6):
    """Same-graph parity of two result sets.  Position-wise id equality, plus a tie-aware row test: ids may be permuted
    inside groups of (near-)equal distances (the reference's binary heap and the engine's sorted list pop equal-distance
    candidates in different orders -- DESIGN.md 4.1), and an id may be swapped at the tail against another of the same
    distance.  Distances are compared position-wise, which is meaningful because both lists are sorted ascending."""
    nq = len(gk)
    rows_ok = 0
    for q in range(nq):
        ka, kb, da, db = gk[q], rk[q], gd[q], rd[q]
        if np.array_equal(ka, kb):
            rows_ok += 1
            continue
        if not np.allclose(da, db, rtol=10 * rtol, atol=10 * atol):
            continue
        good = True
        for i in np.nonzero(ka != kb)[0]:
            pos = np.nonzero(ka == kb[i])[0]
            ref_d = da[pos[0]] if len(pos) else da[-1]
            if not np.isclose(ref_d, db[i], rtol=10 * rtol, atol=10 * atol):
                good = False
                break
        rows_ok += good
    fin = np.isfinite(rd) & np.isfinite(gd)
    rel = np.abs(gd - rd)[fin] / np.maximum(np.abs(rd[fin]), 1e-12)
    return {"identical_id_rows": float(np.mean(np.all(gk == rk, axis=1))), "identical_ids": float(np.mean(gk == rk)),
            "rows_identical_up_to_distance_ties": rows_ok / float(nq),
            "max_rel_dist_err": float(rel.max()) if rel.size else 0.0}


def dump_outputs(out_dir, **arrays):
    """--dump-outputs DIR: what the timed path returned to its caller in the last timed step, one DIR/<name>.npy per array,
    distances as float32 and keys / counts as float64 (exact: keys stay far below 2**53).  The inputs depend only on the
    arguments (seeded generators), so two builds of the project can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32 if a.dtype == np.float32 else np.float64))


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------------------- reference arm
def run_reference(args, wl):
    """The reference's own CPU path (oracle/_ref = usearch compiled unmodified) on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import reflib
    if not reflib.available():
        return run_reference_port(args, wl)
    cores = min(usable_cores(), reflib.lib().refx_hardware_threads())
    # bounded sample, the SAME on every box and every N: the reference builds its own graph over the first --ref-rows rows
    # of the corpus generator (default 200 000; 10 M rows would take it the better part of an hour) with all usable host
    # threads, then answers the bench's query batches
    gen = bits_np if wl.get("kind") == "b1" else structured_np
    nsteps = args.steps + args.warmup
    pool = min(nsteps, args.query_pool)
    Q = gen(pool * wl["batch"], wl["dim"], SEED_QUERY)
    n_ref = min(wl["n"], args.ref_rows)
    Xp = gen(n_ref, wl["dim"], SEED_CORPUS)
    pqkw = {}
    if wl.get("pq"):  # codebook for the reference arm: 256 corpus rows (a valid, if untrained, codebook), stated in `sample`
        nsub, ncent = wl["pq"]
        pqkw = dict(pq=True, num_centroids=ncent, num_subvectors=nsub,
                    codebook=Xp[np.random.default_rng(7).choice(len(Xp), ncent, replace=False)].copy())
    idx = reflib.RefIndex(wl["dim"], wl["metric"], wl.get("kind", "f32"), M=wl["M"], efc=wl["efc"], ef=wl["ef"], threads=cores, **pqkw)
    idx.reserve(n_ref)
    t0 = time.perf_counter()
    idx.add_batch(np.arange(1, n_ref + 1, dtype=np.uint64), Xp, threads=cores)
    t_build = time.perf_counter() - t0
    Xr = None
    del Xp, Xr
    # each timed step is a bounded sample of the batch, sized from the warm-up rate so that K steps take about a minute
    B = wl["batch"]
    t0 = time.perf_counter()
    for s in range(args.warmup):
        idx.search_batch(Q[(s % pool) * B:((s % pool) + 1) * B], wl["k"], threads=cores)
    qps_est = args.warmup * B / (time.perf_counter() - t0)
    per_step = int(max(min(B, 64), min(B, args.ref_seconds * qps_est / max(1, args.steps))))
    times = []
    for s in range(args.steps):
        q = Q[(s % pool) * B:(s % pool) * B + per_step]
        t0 = time.perf_counter()
        keys, dists, counts, comp, vis = idx.search_batch(q, wl["k"], threads=cores)
        times.append(time.perf_counter() - t0)
    if args.dump_outputs:  # per_step follows the measured rate: the first min(B, 64) queries of the step are always in it
        m = min(B, 64)
        dump_outputs(args.dump_outputs, keys=keys[:m], distances=dists[:m], counts=counts[:m])
    total = sum(times)
    value = args.steps * per_step / total
    sample = ("reference builds its own graph over the first %d rows of the %d-row corpus generator (%.0f s, %d threads); each step = "
              "the first %d queries of a %d-query batch" % (n_ref, wl["n"], t_build, cores, per_step, B))
    line = {
        "impl": "reference", "metric": METRIC_NAME, "value": value, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u8 (popcount)" if wl.get("kind") == "b1" else "f32", "data": "synthetic",
        "config": {"workload": wl["desc"], "corpus_rows_indexed": n_ref, "ef": wl["ef"], "k": wl["k"], "batch": wl["batch"],
                   "queries_per_step": per_step},
        "cpu_baseline": {"value": value, "unit": "queries/s", "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "build_vectors_per_s": n_ref / t_build,
    }
    print(json.dumps(line))


def run_reference_port(args, wl):
    """oracle/_ref is not built: time the plain-C restatement of the reference (oracle/hnsw_oracle.c, single thread) on a
    small bounded sample instead."""
    from oracle import portlib
    gen = bits_np if wl.get("kind") == "b1" else structured_np
    n_ref = min(wl["n"], args.ref_rows or 20_000)
    X = gen(n_ref, wl["dim"], SEED_CORPUS)
    per_step = min(wl["batch"], 64)
    Q = gen((args.steps + args.warmup) * per_step, wl["dim"], SEED_QUERY)
    idx = portlib.PortIndex(wl["dim"], wl["metric"], wl.get("kind", "f32"), M=wl["M"], efc=wl["efc"], ef=wl["ef"])
    idx.reserve(n_ref)
    t0 = time.perf_counter()
    for i in range(n_ref):
        idx.add(i + 1, X[i])
    t_build = time.perf_counter() - t0
    times = []
    for s in range(args.steps + args.warmup):
        t0 = time.perf_counter()
        keys, dists, counts, _ = idx.search_batch(Q[s * per_step:(s + 1) * per_step], wl["k"])
        if s >= args.warmup:
            times.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, keys=keys, distances=dists, counts=counts)
    value = args.steps * per_step / sum(times)
    sample = "oracle PORT (oracle/_ref missing): 1 thread, own graph over the first %d rows (%.0f s), %d queries per step" % (
        n_ref, t_build, per_step)
    print(json.dumps({
        "impl": "reference", "metric": METRIC_NAME, "value": value, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u8 (popcount)" if wl.get("kind") == "b1" else "f32", "data": "synthetic",
        "config": {"workload": wl["desc"], "corpus_rows_indexed": n_ref, "ef": wl["ef"], "k": wl["k"], "batch": wl["batch"],
                   "queries_per_step": per_step},
        "cpu_baseline": {"value": value, "unit": "queries/s", "cores": 1, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# --------------------------------------------------------------------------------------- our arm
def run_ours(args, wl):
    import torch
    import torch.distributed as dist
    from lantern_b200 import api

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group(DIST_BACKEND, device_id=torch.device(DEVICE_TYPE, local) if DEVICE_TYPE == "cuda" else None)
    torch.cuda.set_device(local)
    dev = torch.device(DEVICE_TYPE, local if DEVICE_TYPE == "cuda" else 0)
    api.lib()

    n, dim, k, ef, B = wl["n"], wl["dim"], wl["k"], wl["ef"], wl["batch"]
    kind = wl.get("kind", "f32")
    rowb = dim // 8 if kind == "b1" else dim * 4  # bytes of one input row
    gen_t = bits_torch if kind == "b1" else structured_torch
    args.warmup = max(3, args.warmup)  # timing rules: at least 3 warm-up steps (the JSON line reports the value used)
    nsteps = args.steps + args.warmup  # after the clamp: exactly args.steps timed iterations
    pool = min(nsteps, args.query_pool)  # distinct query batches, cycled: step s uses batch s % pool

    # ---- corpus shard of this rank: contiguous row range (SURVEY.md 8e) ----
    lo, hi = (n * rank) // world, (n * (rank + 1)) // world
    pq = wl.get("pq")
    stream = torch.cuda.current_stream()
    nrec = min(B, 1024)
    expand = max(1, args.search_expand)
    t0 = time.perf_counter()
    Q = gen_t(pool * B, dim, SEED_QUERY, dev)
    ef_shard = args.shard_ef if (world > 1 and args.shard_ef > 0) else ef
    pq_info = None
    if not pq:
        X = gen_t(n, dim, SEED_CORPUS, dev)[lo:hi].contiguous() if world > 1 else gen_t(n, dim, SEED_CORPUS, dev)
        torch.cuda.synchronize()
        t_gen = time.perf_counter() - t0
        idx = api.Index(dim, wl["metric"], kind, M=wl["M"], efc=wl["efc"], ef=ef)
        idx.reserve(hi - lo)
        keys_host = np.arange(lo + 1, hi + 1, dtype=np.uint64)  # global keys = row + 1
        t0 = time.perf_counter()
        idx.add_batch_device(keys_host, X.data_ptr(), hi - lo, rowb, kind)
        idx.build()
        torch.cuda.synchronize()
        t_build = time.perf_counter() - t0
        bst = idx.last_build_stats()
        build_work = [bst["computed_distances"], bst["algorithmic_bytes"], bst["device_ms"]]
    else:
        # PQ storage (cfg4): the raw fp32 corpus (61 GB at 10M x d1536) is never resident as a whole: it is generated
        # chunk by chunk; each chunk feeds (a) the running exact top-k used as recall ground truth, (b) lb200_add_batch +
        # lb200_build (PQ encode + insertion), and is then dropped.  The codebook is trained once by the engine's own
        # k-means (lb200_train_pq_device) on the first 200k rows and given to both sides.
        assert world == 1, "PQ workloads run on one GPU"
        nsub, ncent = pq
        chunk = 500_000
        sample = gen_t(min(n, 200_000), dim, SEED_CORPUS * 1000, dev)
        t1 = time.perf_counter()
        codebook, rounds = api.train_pq_device(sample.data_ptr(), dim * 4, len(sample), dim, nsub, ncent, wl["metric"], 15, 7)
        t_train = time.perf_counter() - t1
        del sample
        idx = api.Index(dim, wl["metric"], "f32", M=wl["M"], efc=wl["efc"], ef=ef, pq=True, num_centroids=ncent,
                        num_subvectors=nsub, codebook=codebook)
        idx.reserve(n)
        run_k = torch.full((2, nrec, k), -1, dtype=torch.int64, device=dev)
        run_d = torch.full((2, nrec, k), float("inf"), dtype=torch.float32, device=dev)
        t_gen, t_build = 0.0, 0.0
        build_work = [0, 0, 0.0]
        for c, clo in enumerate(range(0, n, chunk)):
            chi = min(n, clo + chunk)
            t1 = time.perf_counter()
            Xc = gen_t(chi - clo, dim, SEED_CORPUS * 1000 + c, dev)
            torch.cuda.synchronize()
            t_gen += time.perf_counter() - t1
            api.exact_search_device(Xc.data_ptr(), chi - clo, rowb, Q.data_ptr(), nrec, rowb, k, run_k[1].data_ptr(),
                                    run_d[1].data_ptr(), wl["metric"], "f32", dim, stream.cuda_stream)
            run_k[1] += clo + 1
            mk = torch.empty((nrec, k), dtype=torch.int64, device=dev)
            md = torch.empty((nrec, k), dtype=torch.float32, device=dev)
            api.merge_shards_device(run_k.data_ptr(), run_d.data_ptr(), 2, nrec, k, mk.data_ptr(), md.data_ptr(), stream.cuda_stream)
            run_k[0], run_d[0] = mk, md
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            idx.add_batch_device(np.arange(clo + 1, chi + 1, dtype=np.uint64), Xc.data_ptr(), chi - clo, rowb, "f32")
            idx.build()
            torch.cuda.synchronize()
            t_build += time.perf_counter() - t1
            bst = idx.last_build_stats()
            build_work = [build_work[0] + bst["computed_distances"], build_work[1] + bst["algorithmic_bytes"],
                          build_work[2] + bst["device_ms"]]
            del Xc
        pq_truth = run_k[0].cpu().numpy()
        pq_info = {"num_subvectors": nsub, "num_centroids": ncent, "kmeans_rounds": rounds, "kmeans_seconds": t_train,
                   "codebook": "trained by lb200_train_pq_device on 200k rows, compat128 encode (reference quirk)"}

    if expand > 1:
        idx.set_option("search_expand", expand)
    out_keys = torch.empty((B, k), dtype=torch.int64, device=dev)
    out_dists = torch.empty((B, k), dtype=torch.float32, device=dev)
    out_counts = torch.empty((B,), dtype=torch.int32, device=dev)
    if world > 1:
        g_keys = torch.empty((world, B, k), dtype=torch.int64, device=dev)
        g_dists = torch.empty((world, B, k), dtype=torch.float32, device=dev)
        m_keys = torch.empty((B, k), dtype=torch.int64, device=dev)
        m_dists = torch.empty((B, k), dtype=torch.float32, device=dev)

    state = {"ef": ef_shard}

    def step_device(s):
        q = Q[(s % pool) * B:((s % pool) + 1) * B]
        idx.search_batch_device(q.data_ptr(), B, rowb, kind, k, state["ef"], out_keys.data_ptr(), out_dists.data_ptr(),
                                out_counts.data_ptr(), stream.cuda_stream)
        if world > 1:  # the one exchange step: all-gather of per-shard top-k over NVLink, then a G-way merge
            dist.all_gather_into_tensor(g_keys, out_keys)
            dist.all_gather_into_tensor(g_dists, out_dists)
            api.merge_shards_device(g_keys.data_ptr(), g_dists.data_ptr(), world, B, k, m_keys.data_ptr(), m_dists.data_ptr(),
                                    stream.cuda_stream)
            return m_keys
        return out_keys

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- ground truth for recall (untimed): brute force on this rank's shard, merged like the search results ----
    tk = torch.empty((nrec, k), dtype=torch.int64, device=dev)
    td = torch.empty((nrec, k), dtype=torch.float32, device=dev)
    gt_info = None
    if not pq:
        ge = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ge[0].record(stream)
        api.exact_search_device(X.data_ptr(), hi - lo, rowb, Q.data_ptr(), nrec, rowb, k, tk.data_ptr(), td.data_ptr(),
                                wl["metric"], kind, dim, stream.cuda_stream)
        ge[1].record(stream)
        torch.cuda.synchronize()
        gt_ms = ge[0].elapsed_time(ge[1])
        tc = kind == "f32" and wl["metric"] in ("l2sq", "cos") and (hi - lo) >= 32768 and nrec >= 16 and not os.environ.get("LB200_EXACT")
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                tf32_peak = float(json.load(f)["bf16_tflops"]) / 2.0
        except Exception:
            tf32_peak = 1590.0 / 2.0
        gt_info = {"rows": hi - lo, "queries": nrec, "k": k, "seconds": gt_ms / 1e3,
                   "path": "tcgen05 3xTF32 filter + exact fp32 re-rank (csrc/exact_tc.cu)" if tc else "SIMT fp32 (csrc/exact.cu)"}
        if tc:
            tfl = 3 * 2.0 * (hi - lo) * nrec * dim / (gt_ms / 1e3) / 1e12
            gt_info["roofline"] = {"bound": "tensor", "achieved": tfl, "unit": "TFLOP/s", "peak": tf32_peak,
                                   "frac": tfl / tf32_peak, "flops": "3 tf32 MMAs per product (hi*hi + hi*lo + lo*hi), whole search incl. norms and re-rank",
                                   "peak_source": "MEASURED_PEAKS.json bf16_tflops / 2 (dense tf32 runs at half the bf16 rate)"}
        tk += lo + 1  # offsets -> global keys
    if world > 1:
        gk = torch.empty((world, nrec, k), dtype=torch.int64, device=dev)
        gd = torch.empty((world, nrec, k), dtype=torch.float32, device=dev)
        dist.all_gather_into_tensor(gk, tk)
        dist.all_gather_into_tensor(gd, td)
        tk2 = torch.empty_like(tk)
        td2 = torch.empty_like(td)
        api.merge_shards_device(gk.data_ptr(), gd.data_ptr(), world, nrec, k, tk2.data_ptr(), td2.data_ptr(), stream.cuda_stream)
        tk = tk2
    torch.cuda.synchronize()
    truth = pq_truth if pq else tk.cpu().numpy()

    # ---- multi-GPU: per-shard beam width (SURVEY.md 8e).  Every query visits every shard, so throughput only grows
    #      if the per-shard beam shrinks: pick the smallest ef_s >= k whose MERGED recall@10 reaches the recall of
    #      the unsharded single-GPU graph at the workload's ef (measured here on rank 0), and report both. ----
    shard_info = None
    if world > 1:
        # recall target = recall of the UNSHARDED graph at the workload's ef.  Small corpora: every rank builds the full
        # graph (rank 0 takes the target from it; all ranks use it for the labelled "replicated" comparison below).
        # Large corpora: pass the 1-GPU bench's recall with --recall-target instead of rebuilding 10M+ rows per rank.
        target = torch.zeros(1, dtype=torch.float64, device=dev)
        full = None
        build_full = args.recall_target <= 0 and args.shard_ef >= 0 or args.replicated_comparison
        if build_full and n * rowb <= BIG_CORPUS_BYTES:
            Xfull = gen_t(n, dim, SEED_CORPUS, dev)
            full = api.Index(dim, wl["metric"], kind, M=wl["M"], efc=wl["efc"], ef=ef)
            full.reserve(n)
            full.add_batch_device(np.arange(1, n + 1, dtype=np.uint64), Xfull.data_ptr(), n, rowb, kind)
            full.build()
            del Xfull
            fk = torch.empty((B, k), dtype=torch.int64, device=dev)
            fd = torch.empty((B, k), dtype=torch.float32, device=dev)
            full.search_batch_device(Q.data_ptr(), B, rowb, kind, k, ef, fk.data_ptr(), fd.data_ptr(), 0, stream.cuda_stream)
            torch.cuda.synchronize()
            if rank == 0:
                target[0] = recall_at_k(fk[:nrec].cpu().numpy(), truth)
        target_src = "unsharded graph built and searched in this run (rank 0)"
        if args.recall_target > 0:
            target[0] = args.recall_target
            target_src = "--recall-target"
        elif full is None and args.shard_ef == 0 and wl.get("recall_1gpu"):
            target[0] = wl["recall_1gpu"]
            target_src = "recorded 1-GPU run of this bench (WORKLOADS[...]['recall_1gpu']); corpus too large to rebuild unsharded per rank"
        dist.broadcast(target, 0)
        target = float(target.item())
        sweep = {}
        cands = sorted(set([e for e in (k, 12, 16, 20, 24, 28, 32, 36, 40, 44, 48, 52, 56, 64, 72, 80, 96, 112, 128) if k <= e <= ef] + [ef]))
        chosen = ef
        for e in (cands if args.shard_ef == 0 else []):
            state["ef"] = e
            res = step_device(0)
            torch.cuda.synchronize()
            r = recall_at_k(res[:nrec].cpu().numpy(), truth)
            sweep[e] = r
            if r >= target and target > 0:
                chosen = e
                break
        if args.shard_ef > 0:
            chosen = args.shard_ef
        elif args.shard_ef < 0:
            chosen = ef  # "same-ef" mode
        state["ef"] = chosen
        ef_shard = chosen
        shard_info = {"recall_target_unsharded_1gpu": target, "recall_target_source": target_src,
                      "sweep_merged_recall_by_ef": sweep, "ef_per_shard": chosen}
        def timed(fn, reps):
            for s_ in range(3):
                fn(s_)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for s_ in range(reps):
                fn(s_)
            e1.record(stream)
            barrier()
            tr = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
            dist.all_reduce(tr, op=dist.ReduceOp.MAX)
            return float(tr.item()) / 1e3

        reps = max(10, min(args.steps, 100))
        if chosen != ef:  # (i) of SURVEY 8e: same ef on every shard (higher recall, little speed-up)
            state["ef"] = ef
            res = step_device(0)
            torch.cuda.synchronize()
            r_same = recall_at_k(res[:nrec].cpu().numpy(), truth)
            shard_info["same_ef"] = {"ef_per_shard": ef, "value": reps * B / timed(step_device, reps), "unit": "queries/s",
                                     "merged_recall": r_same}
            state["ef"] = chosen
        if full is not None:
            # replicated comparison (NOT the headline): every GPU holds the whole graph and serves its own B-query batches,
            # no exchange step; weak scaling in queries.  Same kernel, same ef as 1 GPU, same recall as 1 GPU.
            def rep_step(s_):
                full.search_batch_device(Q[((s_ + rank) % pool) * B].data_ptr(), B, rowb, kind, k, ef, fk.data_ptr(), fd.data_ptr(), 0,
                                         stream.cuda_stream)
            shard_info["replicated_comparison"] = {
                "value": world * reps * B / timed(rep_step, reps), "unit": "queries/s", "scaling": "weak",
                "what": "NOT the headline: full corpus replicated on every GPU, each GPU serves its own %d-query batches at ef=%d, "
                        "no collective; recall = the 1-GPU recall" % (B, ef)}
            full.close()
            del full
            torch.cuda.empty_cache()

    # ---- warm-up, then K timed steps on the device ----
    for s in range(args.warmup):
        res = step_device(s)
        if s == 0:
            torch.cuda.synchronize()
            rec = recall_at_k(res[:nrec].cpu().numpy(), truth)
    barrier()
    launches0 = api.kernel_launches()
    sampler = ClockSampler(local) if rank == 0 else None
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    alg_bytes, kern_ms, n_dist = 0, 0.0, 0
    barrier()
    ev[0].record(stream)
    for s in range(args.warmup, nsteps):
        step_device(s)
        if args.per_step_stats:
            st = idx.last_stats()
            alg_bytes += st["algorithmic_bytes"]; kern_ms += st["kernel_ms"]; n_dist += st["computed_distances"]
    ev[1].record(stream)
    barrier()
    ms = ev[0].elapsed_time(ev[1])
    launches = api.kernel_launches() - launches0
    if args.dump_outputs and rank == 0:  # the last timed step's results, before anything else reuses the buffers
        if world > 1:
            dump_outputs(args.dump_outputs, keys=m_keys, distances=m_dists)
        else:
            dump_outputs(args.dump_outputs, keys=out_keys, distances=out_dists, counts=out_counts)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = args.steps * B / (ms / 1e3)

    # ---- roofline of the search kernel: separate pass with per-step counters (the stats call synchronises) ----
    alg_bytes, kern_ms, n_dist, pops = 0, 0.0, 0, 0
    for s in range(args.warmup, nsteps):
        q = Q[(s % pool) * B:((s % pool) + 1) * B]
        idx.search_batch_device(q.data_ptr(), B, rowb, kind, k, ef_shard, out_keys.data_ptr(), out_dists.data_ptr(),
                                out_counts.data_ptr(), stream.cuda_stream)
        st = idx.last_stats()
        alg_bytes += st["algorithmic_bytes"]; kern_ms += st["kernel_ms"]; n_dist += st["computed_distances"]; pops += st["base_pops"]
    # The clock sampler (nvidia-smi, 20 ms period, ~0.1 s to start) covers the timed region, this pass over the same steps
    # and -- when both together are shorter than 0.6 s -- further untimed repetitions of the same steps, so that even short
    # runs (small --steps) yield samples taken under the benchmark's own load.  `ms` is identical on all ranks.
    extra = int(np.ceil(max(0.0, 600.0 - 2.0 * ms) / max(ms / args.steps, 1e-3)))
    for s in range(extra):
        step_device(args.warmup + s)
    torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    if clocks is not None:
        clocks["sampled_over"] = "timed steps + stats pass + %d identical untimed steps" % extra
    peak, peak_src = peaks()
    achieved = alg_bytes / (kern_ms / 1e3) / 1e9
    traffic = None
    prof = os.path.join(ROOT, "profiles", "search_kernel_traffic.json")
    if os.path.exists(prof) and world == 1:
        try:
            with open(prof) as f:
                traffic = json.load(f).get(wl["desc"].split(":")[0])
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "peak_source": peak_src, "kernel": "hnsw_search_kernel<%s,%s>" % (wl["metric"], "pq" if pq else kind),
                "kernel_ms_per_step": kern_ms / args.steps,
                "timing": "kernel_ms_per_step: CUDA events around the one kernel launch, in a SEPARATE pass over the same steps whose "
                          "stats read-back synchronises after every step (slightly slower than the back-to-back `ms_per_step`)", "algorithmic_bytes_per_step": alg_bytes / args.steps,
                "dist_evals_per_query": n_dist / (args.steps * B), "pops_per_query": pops / (args.steps * B),
                "limbo_overflows_last_step": st.get("limbo_overflows", 0)}

    # ---- e2e through the reference-facing host call: pinned host buffers in/out, copies inside the timed region ----
    e2e = None
    if world > 1:
        hq = torch.empty(Q.shape, dtype=Q.dtype).pin_memory()
        hq.copy_(Q)
        dq = torch.empty((B, Q.shape[1]), dtype=Q.dtype, device=dev)
        hk = torch.empty((B, k), dtype=torch.int64).pin_memory()
        hd = torch.empty((B, k), dtype=torch.float32).pin_memory()

        def step_e2e(s):
            dq.copy_(hq[(s % pool) * B:((s % pool) + 1) * B], non_blocking=True)  # every shard needs every query
            idx.search_batch_device(dq.data_ptr(), B, rowb, kind, k, ef_shard, out_keys.data_ptr(), out_dists.data_ptr(),
                                    out_counts.data_ptr(), stream.cuda_stream)
            dist.all_gather_into_tensor(g_keys, out_keys)
            dist.all_gather_into_tensor(g_dists, out_dists)
            api.merge_shards_device(g_keys.data_ptr(), g_dists.data_ptr(), world, B, k, m_keys.data_ptr(), m_dists.data_ptr(),
                                    stream.cuda_stream)
            if rank == 0:
                hk.copy_(m_keys, non_blocking=True)
                hd.copy_(m_dists, non_blocking=True)
            torch.cuda.synchronize()

        for s in range(args.warmup):
            step_e2e(s)
        barrier()
        t0 = time.perf_counter()
        for s in range(args.warmup, nsteps):
            step_e2e(s)
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        dt = float(dt.item())
        e2e = {"value": args.steps * B / dt, "unit": "queries/s", "h2d_bytes_per_step": world * B * rowb,
               "d2h_bytes_per_step": B * k * 12, "ms_per_step": 1e3 * dt / args.steps,
               "note": "every rank uploads the query batch from pinned host memory; rank 0 downloads the merged top-k"}
    if world == 1:
        hq = torch.empty(Q.shape, dtype=Q.dtype).pin_memory()
        hq.copy_(Q)
        hk = torch.empty((B, k), dtype=torch.int64).pin_memory()
        hd = torch.empty((B, k), dtype=torch.float32).pin_memory()
        hc = torch.empty((B,), dtype=torch.int64).pin_memory()
        for s in range(args.warmup):
            idx.search_batch_raw(hq[(s % pool) * B].data_ptr(), B, rowb, kind, k, ef, hk.data_ptr(), hd.data_ptr(), hc.data_ptr())
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for s in range(args.warmup, nsteps):
            idx.search_batch_raw(hq[(s % pool) * B].data_ptr(), B, rowb, kind, k, ef, hk.data_ptr(), hd.data_ptr(), hc.data_ptr())
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        e2e = {"value": args.steps * B / dt, "unit": "queries/s", "h2d_bytes_per_step": B * rowb,
               "d2h_bytes_per_step": B * k * 8 + B * k * 4 + B * 4, "ms_per_step": 1e3 * dt / args.steps}

    # ---- CPU baseline (rank 0, N=1): the unmodified reference on the host cores over the SAME index file ----
    cpu_baseline, parity = None, None
    if world == 1 and not args.no_cpu_baseline and pq:
        # the reference refuses to LOAD pq index files (lantern_storage.hpp:550-551), so it builds its own pq graph, with
        # the same codebook, over a bounded prefix of the corpus and searches the bench's query batches
        from oracle import reflib
        if reflib.available():
            cores = min(usable_cores(), reflib.lib().refx_hardware_threads())
            n_ref = min(n, args.pq_ref_rows)
            Xr = gen_t(n_ref, dim, SEED_CORPUS * 1000, dev).cpu().numpy()
            ridx = reflib.RefIndex(dim, wl["metric"], M=wl["M"], efc=wl["efc"], ef=ef, threads=cores, pq=True,
                                   num_centroids=pq[1], num_subvectors=pq[0], codebook=codebook)
            ridx.reserve(n_ref)
            t0 = time.perf_counter()
            ridx.add_batch(np.arange(1, n_ref + 1, dtype=np.uint64), Xr, threads=cores)
            t_rb = time.perf_counter() - t0
            qh = Q.cpu().numpy()
            spent, done, s, first = 0.0, 0, 0, None
            while spent < args.cpu_seconds and s < pool:
                t0 = time.perf_counter()
                rres = ridx.search_batch(qh[s * B:(s + 1) * B], k, threads=cores)
                spent += time.perf_counter() - t0
                if first is None:
                    first = rres
                done += B
                s += 1
            cpu_baseline = {"value": done / spent, "unit": "queries/s", "cores": cores, "kind": "reference",
                            "sample": "unmodified usearch (oracle/_ref) builds its own pq graph over the first %d of %d rows (%.0f s) "
                                      "with the same codebook and searches %d queries (%.1f s) on %d threads" % (
                                          n_ref, n, t_rb, done, spent, cores)}
            # parity at this geometry.  The reference cannot LOAD a pq index file (lantern_storage.hpp:550-551), so a same-graph
            # comparison is impossible: the engine builds its own pq graph over the SAME rows with the same codebook, both answer
            # the same queries, both are scored against the raw-fp32 exact top-k of those rows (the +-0.5 % recall contract)
            Xd = torch.from_numpy(Xr).to(dev)
            eidx = api.Index(dim, wl["metric"], "f32", M=wl["M"], efc=wl["efc"], ef=ef, pq=True, num_centroids=pq[1],
                             num_subvectors=pq[0], codebook=codebook)
            eidx.reserve(n_ref)
            eidx.add_batch_device(np.arange(1, n_ref + 1, dtype=np.uint64), Xd.data_ptr(), n_ref, rowb, "f32")
            eidx.build()
            ptk = torch.empty((nrec, k), dtype=torch.int64, device=dev)
            ptd = torch.empty((nrec, k), dtype=torch.float32, device=dev)
            api.exact_search_device(Xd.data_ptr(), n_ref, rowb, Q.data_ptr(), nrec, rowb, k, ptk.data_ptr(), ptd.data_ptr(), wl["metric"],
                                    "f32", dim, stream.cuda_stream)
            eidx.search_batch_device(Q.data_ptr(), B, rowb, "f32", k, ef, out_keys.data_ptr(), out_dists.data_ptr(),
                                     out_counts.data_ptr(), stream.cuda_stream)
            torch.cuda.synchronize()
            ptruth = (ptk + 1).cpu().numpy()
            ek = out_keys[:nrec].cpu().numpy().astype(np.uint64)
            rk = first[0][:nrec]
            parity = {"graph_rows": n_ref, "queries": nrec, "same_graph": False,
                      "why": "the reference refuses to load pq index files; each side builds its own graph over the same rows with the "
                             "same codebook",
                      "reference_recall_at_k": recall_at_k(rk, ptruth), "engine_recall_at_k": recall_at_k(ek, ptruth),
                      "mean_id_overlap_at_k": float(np.mean([len(set(a.tolist()) & set(b.tolist())) / float(k) for a, b in zip(ek, rk)])),
                      "ground_truth": "raw fp32 exact top-%d of the %d rows (lb200_exact_search_device)" % (k, n_ref)}
            eidx.close()
            del Xd
    cpu_note = None
    if world == 1 and not args.no_cpu_baseline and not pq:
        from oracle import reflib
        if reflib.available():
            b_idx = idx
            try:
                cores = min(usable_cores(), reflib.lib().refx_hardware_threads())
                b_n, b_truth, b_what = n, truth, "the engine's %d-node index file" % n
                if n * rowb > BIG_CORPUS_BYTES:
                    # The reference needs the index file twice in host RAM (35 GB each for cfg3) and half a minute to parse it:
                    # bounded sample instead.  The engine builds a second graph, same parameters, over the first
                    # --cpu-prefix-rows corpus rows; the reference loads THAT file and answers the same query batches.
                    b_n = min(n, args.cpu_prefix_rows)
                    b_idx = api.Index(dim, wl["metric"], kind, M=wl["M"], efc=wl["efc"], ef=ef)
                    b_idx.reserve(b_n)
                    b_idx.add_batch_device(np.arange(1, b_n + 1, dtype=np.uint64), X.data_ptr(), b_n, rowb, kind)
                    b_idx.build()
                    btk = torch.empty((nrec, k), dtype=torch.int64, device=dev)
                    btd = torch.empty((nrec, k), dtype=torch.float32, device=dev)
                    api.exact_search_device(X.data_ptr(), b_n, rowb, Q.data_ptr(), nrec, rowb, k, btk.data_ptr(), btd.data_ptr(),
                                            wl["metric"], kind, dim, stream.cuda_stream)
                    btk += 1  # offsets -> keys
                    torch.cuda.synchronize()
                    b_truth = btk.cpu().numpy()
                    b_what = ("the index file the engine built over the first %d of the %d corpus rows (same M/efc/ef; the full file "
                              "would not fit twice in host RAM next to the corpus)" % (b_n, n))
                t0 = time.perf_counter()
                buf = b_idx.save_buffer()
                ridx = reflib.RefIndex(dim, wl["metric"], kind, M=wl["M"], efc=wl["efc"], ef=ef, threads=cores)
                ridx.load_buffer(buf)
                t_load = time.perf_counter() - t0
                del buf
                ridx._loaded = None
                qh = Q.cpu().numpy()
                spent, done, first = 0.0, 0, None
                s = 0
                while spent < args.cpu_seconds and s < pool:
                    qb = qh[s * B:(s + 1) * B]
                    t0 = time.perf_counter()
                    rkeys, rd, rc, comp, vis = ridx.search_batch(qb, k, threads=cores)
                    spent += time.perf_counter() - t0
                    done += B
                    if first is None:
                        first = (rkeys, rd, comp)
                    s += 1
                cpu_qps = done / spent
                cpu_baseline = {"value": cpu_qps, "unit": "queries/s", "cores": cores, "kind": "reference",
                                "sample": "unmodified usearch (oracle/_ref) loads %s (%.0f s) and searches %d of the bench's query "
                                          "batches (%d queries, %.1f s) on %d threads" % (b_what, t_load, s, done, spent, cores)}
                # same-graph parity at that size: step-0 queries, ids position-wise
                b_idx.search_batch_device(Q.data_ptr(), B, rowb, kind, k, ef, out_keys.data_ptr(), out_dists.data_ptr(),
                                          out_counts.data_ptr(), stream.cuda_stream)
                torch.cuda.synchronize()
                st0 = b_idx.last_stats()
                gk = out_keys.cpu().numpy().astype(np.uint64)
                gd = out_dists.cpu().numpy()
                rk0, rd0, comp0 = first
                parity = {"graph_rows": b_n, "queries": B}
                parity.update(parity_block(gk, gd, rk0, rd0))
                parity.update({"reference_computed_distances": int(comp0), "engine_computed_distances": int(st0["computed_distances"]),
                               "reference_recall_at_10": recall_at_k(rk0[:nrec], b_truth),
                               "engine_recall_at_10": recall_at_k(gk[:nrec], b_truth)})
            except Exception as e:  # the baseline is a side measurement: never lose the GPU numbers over it
                cpu_note = "cpu_baseline failed: %r" % (e,)
                print(cpu_note, file=sys.stderr)
            finally:
                if b_idx is not idx:
                    b_idx.close()

    if world == 1 and not args.no_cpu_baseline and cpu_baseline is None and not pq:
        # oracle/_ref unavailable (or the index file too large for host RAM): the plain-C restatement on one core, on a
        # bounded sample of the same queries; it loads the engine's index file when that is small enough, else skips
        from oracle import portlib
        if n * rowb <= 2e9:
            pidx = portlib.PortIndex(dim, wl["metric"], kind, M=wl["M"], efc=wl["efc"], ef=ef)
            pidx.reserve(n)
            pidx.load_buffer(idx.save_buffer())
            qh = Q[:256].cpu().numpy()
            t0 = time.perf_counter()
            pidx.search_batch(qh, k)
            dt = time.perf_counter() - t0
            cpu_baseline = {"value": len(qh) / dt, "unit": "queries/s", "cores": 1, "kind": "port",
                            "sample": "oracle port (hnsw_oracle.c, 1 thread) loads the engine's index file and searches %d queries" % len(qh)}
    if rank == 0:
        line = {
            "metric": METRIC_NAME, "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",  # the corpus is fixed; shards shrink as N grows
            "vs_baseline": None, "dtype": "u8 (popcount)" if kind == "b1" else "f32", "data": "synthetic",
            "config": {"workload": wl["desc"], "corpus_rows": n, "rows_per_gpu": hi - lo, "ef": ef, "ef_per_shard": ef_shard, "k": k, "search_order": "exact (reference order)" if expand == 1 else "relaxed: %d candidates per round" % expand,
                       "batch": B, "parallelism": "row-range shards x%d + NCCL all-gather of top-k + merge" % world if world > 1 else "1 GPU",
                       "l2_policy": "inputs larger than L2: %.1f GB corpus gathered at random; %d distinct query batches cycled" % ((hi - lo) * rowb / 1e9, pool),
                       "generator": ("64 random prototypes XOR 10%% bit flips, seeds %d/%d/%d" % (SEED_P, SEED_CORPUS, SEED_QUERY)) if kind == "b1" else
                       "x = z P + %.2f eps, z~N(0,I_%d), seeds %d/%d/%d" % (NOISE, LATENT, SEED_P, SEED_CORPUS, SEED_QUERY)},
            "recall_at_10": rec if k == 10 else None, "recall_at_k": rec, "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
            "cpu_baseline": cpu_baseline, "cpu_baseline_note": cpu_note, "parity": parity, "sharding": shard_info, "pq": pq_info,
            "ground_truth": gt_info,
            "build": {"vectors_per_s": (hi - lo) / t_build, "seconds": t_build, "datagen_seconds": t_gen,
                      # SURVEY 8d build metric: sum of computed_distances(add) x bytes per stored vector / device time
                      "dist_evals_per_vector": build_work[0] / max(1, hi - lo), "device_seconds": build_work[2] / 1e3,
                      "roofline": {"bound": "hbm+l2 (the heuristic re-reads rows that mostly hit L2)",
                                   "achieved": build_work[1] / max(build_work[2] / 1e3, 1e-9) / 1e9, "peak": peaks()[0], "unit": "GB/s",
                                   "frac": build_work[1] / max(build_work[2] / 1e3, 1e-9) / 1e9 / peaks()[0]}},
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()

# --------------------------------------------------------------------------------------- our arm, N > 1: row-sharded group
def run_group(args, wl):
    """--gpus N > 1 (default mode "rows"): ONE graph over the whole corpus, vectors sharded by row range across the N GPUs,
    every distance evaluated on the GPU that holds the row (lb200_group_*, csrc/group.cu).  Rank 0 generates the corpus and
    builds the graph exactly as the 1-GPU run does; lb200_group_distribute hands every rank its row range and a copy of the
    adjacency lists over NVLink.  Total work == the 1-GPU search; results == the 1-GPU results on the same graph (checked
    in this run, `same_graph_as_1gpu`); recall therefore equals the 1-GPU recall at the same ef by construction."""
    import torch
    import torch.distributed as dist
    from lantern_b200 import api

    world, rank, local = int(os.environ["WORLD_SIZE"]), int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev, timeout=__import__("datetime").timedelta(minutes=30))
    api.lib()
    n, dim, k, ef, B = wl["n"], wl["dim"], wl["k"], wl["ef"], wl["batch"]
    kind = wl.get("kind", "f32")
    rowb = dim // 8 if kind == "b1" else dim * 4
    gen_t = bits_torch if kind == "b1" else structured_torch
    args.warmup = max(3, args.warmup)
    nsteps = args.steps + args.warmup
    pool = min(nsteps, args.query_pool)
    stream = torch.cuda.current_stream()
    nrec = min(B, 1024)

    def allgather_bytes(send):  # bootstrap collective of the group (creation / distribution only)
        t = torch.frombuffer(bytearray(send), dtype=torch.uint8).to(dev)
        out = torch.empty((world, len(send)), dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(out, t)
        return out.cpu().numpy().tobytes()

    grp = api.Group.ranked(rank, world, allgather_bytes)
    idx, Q, truth, t_gen, t_build, build_work = None, None, None, 0.0, 0.0, [0, 0, 0.0]
    if rank == 0:
        t0 = time.perf_counter()
        Q = gen_t(pool * B, dim, SEED_QUERY, dev)
        X = gen_t(n, dim, SEED_CORPUS, dev)
        torch.cuda.synchronize()
        t_gen = time.perf_counter() - t0
        idx = api.Index(dim, wl["metric"], kind, M=wl["M"], efc=wl["efc"], ef=ef)
        idx.reserve(n)
        t0 = time.perf_counter()
        idx.add_batch_device(np.arange(1, n + 1, dtype=np.uint64), X.data_ptr(), n, rowb, kind)
        idx.build()
        torch.cuda.synchronize()
        t_build = time.perf_counter() - t0
        bst = idx.last_build_stats()
        build_work = [bst["computed_distances"], bst["algorithmic_bytes"], bst["device_ms"]]
        tk = torch.empty((nrec, k), dtype=torch.int64, device=dev)
        td = torch.empty((nrec, k), dtype=torch.float32, device=dev)
        api.exact_search_device(X.data_ptr(), n, rowb, Q.data_ptr(), nrec, rowb, k, tk.data_ptr(), td.data_ptr(), wl["metric"], kind,
                                dim, stream.cuda_stream)
        torch.cuda.synchronize()
        truth = (tk + 1).cpu().numpy()
        del X
        torch.cuda.empty_cache()
    t0 = time.perf_counter()
    grp.distribute(idx, root=0, max_batch=B, max_results=B * k)
    torch.cuda.synchronize()
    t_dist = time.perf_counter() - t0

    out_keys = torch.empty((B, k), dtype=torch.int64, device=dev)
    out_dists = torch.empty((B, k), dtype=torch.float32, device=dev)
    out_counts = torch.empty((B,), dtype=torch.int32, device=dev)

    def step_device(s):
        qp = Q[(s % pool) * B:((s % pool) + 1) * B].data_ptr() if rank == 0 else 0
        grp.search_batch_device(qp, B, rowb, kind, k, ef, out_keys.data_ptr(), out_dists.data_ptr(), out_counts.data_ptr(),
                                stream.cuda_stream)

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    # same graph => same answer as the 1-GPU kernel (rank 0 still holds the whole index)
    same, rec, one_gpu = None, None, None
    step_device(0)
    torch.cuda.synchronize()
    if rank == 0:
        k1 = torch.empty((B, k), dtype=torch.int64, device=dev)
        d1 = torch.empty((B, k), dtype=torch.float32, device=dev)
        idx.search_batch_device(Q.data_ptr(), B, rowb, kind, k, ef, k1.data_ptr(), d1.data_ptr(), 0, stream.cuda_stream)
        torch.cuda.synchronize()
        st1 = idx.last_stats()
        same = {"identical_id_rows": float((k1 == out_keys).all(dim=1).float().mean().item()),
                "bit_identical_distances": bool(torch.equal(d1.view(torch.int32), out_dists.view(torch.int32))),
                "one_gpu_computed_distances": int(st1["computed_distances"])}
        rec = recall_at_k(out_keys[:nrec].cpu().numpy(), truth)
        # the 1-GPU kernel on the same graph, same queries, same box: the denominator of this run's own speed-up
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = max(3, min(20, args.steps))
        for s_ in range(2):
            idx.search_batch_device(Q[(s_ % pool) * B].data_ptr(), B, rowb, kind, k, ef, k1.data_ptr(), d1.data_ptr(), 0, stream.cuda_stream)
        e0.record(stream)
        for s_ in range(reps):
            idx.search_batch_device(Q[(s_ % pool) * B].data_ptr(), B, rowb, kind, k, ef, k1.data_ptr(), d1.data_ptr(), 0, stream.cuda_stream)
        e1.record(stream)
        torch.cuda.synchronize()
        idx.search_batch_device(Q.data_ptr(), B, rowb, kind, k, ef, k1.data_ptr(), d1.data_ptr(), 0, stream.cuda_stream)
        torch.cuda.synchronize()
        one_gpu = {"value": reps * B / (e0.elapsed_time(e1) / 1e3), "unit": "queries/s",
                   "recall_at_k": recall_at_k(k1[:nrec].cpu().numpy(), truth),
                   "what": "lb200_search_batch_device on rank 0's unsharded copy of the same graph, %d steps" % reps}
    for s in range(args.warmup):
        step_device(s)
    barrier()
    launches0 = api.kernel_launches()
    sampler = ClockSampler(local) if rank == 0 else None
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    barrier()
    ev[0].record(stream)
    for s in range(args.warmup, nsteps):
        step_device(s)
    ev[1].record(stream)
    barrier()
    if args.dump_outputs and rank == 0:  # the last timed step's results, before anything else reuses the buffers
        dump_outputs(args.dump_outputs, keys=out_keys, distances=out_dists, counts=out_counts)
    t = torch.tensor([ev[0].elapsed_time(ev[1])], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    launches = api.kernel_launches() - launches0
    value = args.steps * B / (ms / 1e3)

    # per-rank work of one step (the stats call synchronises): rows each GPU read, its kernel time
    step_device(args.warmup)
    st = grp.last_stats()
    mine = torch.tensor([st["local_rows_evaluated"], st["local_row_bytes"], st["owner_computed_distances"], st["owner_base_pops"],
                         st["owner_upper_hops"], st["owner_rounds"], st["kernel_ms"] * 1e6, st["owner_cycles_produce"],
                         st["owner_cycles_local"], st["owner_cycles_wait"], st["owner_cycles_consume"]], dtype=torch.float64, device=dev)
    allst = torch.empty((world, mine.numel()), dtype=torch.float64, device=dev)
    dist.all_gather_into_tensor(allst, mine)
    allst = allst.cpu().numpy()
    extra = int(np.ceil(max(0.0, 600.0 - ms) / max(ms / args.steps, 1e-3)))
    for s in range(extra):
        step_device(args.warmup + s)
    torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    if clocks is not None:
        clocks["sampled_over"] = "timed steps + stats step + %d identical untimed steps" % extra

    # e2e: ONE upload of the query batch from pinned host memory (rank 0), results back to the host on every rank
    hq = hk = hd = hc = None
    if rank == 0:
        hq = torch.empty(Q.shape, dtype=Q.dtype).pin_memory()
        hq.copy_(Q)
    hk = torch.empty((B, k), dtype=torch.int64).pin_memory()
    hd = torch.empty((B, k), dtype=torch.float32).pin_memory()
    hc = torch.empty((B,), dtype=torch.int64).pin_memory()

    def step_e2e(s):
        grp.search_batch_raw(hq[(s % pool) * B].data_ptr() if rank == 0 else 0, B, rowb, kind, k, ef, hk.data_ptr(), hd.data_ptr(),
                             hc.data_ptr())
    for s in range(args.warmup):
        step_e2e(s)
    barrier()
    t0 = time.perf_counter()
    for s in range(args.warmup, nsteps):
        step_e2e(s)
    barrier()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    dt = float(dt.item())
    e2e = {"value": args.steps * B / dt, "unit": "queries/s", "h2d_bytes_per_step": B * rowb, "d2h_bytes_per_step": B * k * 12 + B * 4,
           "ms_per_step": 1e3 * dt / args.steps,
           "note": "rank 0 uploads the batch once from pinned host memory (the other GPUs read the queries over NVLink inside the "
                   "kernel); every rank downloads the full top-k (bytes counted for rank 0)"}
    if rank == 0:
        peak, peak_src = peaks()
        vec_bytes = rowb
        alg = float(allst[:, 2].sum() * vec_bytes + allst[:, 3].sum() * (4 + 8 * wl["M"]) + allst[:, 4].sum() * (4 + 4 * wl["M"]) + B * vec_bytes)
        kms = float(allst[:, 6].max() / 1e6)
        mhz = (clocks or {}).get("sm_mhz") or 1965.0
        per_rank = [{"rank": r, "rows_evaluated_per_query": float(allst[r, 0] / B), "row_gb_per_step": float(allst[r, 1] / 1e9),
                     "kernel_ms": float(allst[r, 6] / 1e6), "local_hbm_frac": float(allst[r, 1] / (allst[r, 6] / 1e9) / 1e9 / peak),
                     # where an owner warp's time goes, per expansion round (SM cycles / sampled SM clock)
                     "owner_us_per_round": {name: float(allst[r, 7 + i] / max(allst[r, 5], 1.0) / mhz)
                                            for i, name in enumerate(("produce_ids", "local_rows", "wait_for_peers", "insertions"))}}
                    for r in range(world)]
        roofline = {"bound": "hbm", "achieved": alg / (kms / 1e3) / 1e9, "peak": peak * world, "unit": "GB/s",
                    "frac": alg / (kms / 1e3) / 1e9 / (peak * world), "traffic": None, "peak_source": peak_src + " x %d GPUs" % world,
                    "kernel": "group_search_kernel<%s,%s> on %d GPUs" % (wl["metric"], kind, world), "kernel_ms_per_step": kms,
                    "algorithmic_bytes_per_step": alg, "dist_evals_per_query": float(allst[:, 2].sum() / B),
                    "pops_per_query": float(allst[:, 3].sum() / B), "rounds_per_query": float(allst[:, 5].sum() / B),
                    "timing": "one extra step after the timed region; kernel_ms = max over ranks of the search kernel's device time"}
        line = {
            "metric": METRIC_NAME, "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u8 (popcount)" if kind == "b1" else "f32", "data": "synthetic",
            "config": {"workload": wl["desc"], "corpus_rows": n, "rows_per_gpu": n // world, "ef": ef, "ef_per_shard": ef, "k": k,
                       "search_order": "exact (reference order)", "batch": B,
                       "parallelism": "one graph, vectors sharded by row range x%d (adjacency replicated), distances evaluated on the "
                                      "owning GPU over NVLink peer memory, top-k all-gather fused into the kernel epilogue; no NCCL on "
                                      "the search path" % world,
                       "l2_policy": "inputs larger than L2: %.1f GB of rows per GPU gathered at random; %d distinct query batches cycled" % (
                           n // world * rowb / 1e9, pool),
                       "generator": ("64 random prototypes XOR 10%% bit flips, seeds %d/%d/%d" % (SEED_P, SEED_CORPUS, SEED_QUERY)) if kind == "b1" else
                       "x = z P + %.2f eps, z~N(0,I_%d), seeds %d/%d/%d" % (NOISE, LATENT, SEED_P, SEED_CORPUS, SEED_QUERY)},
            "recall_at_10": rec if k == 10 else None, "recall_at_k": rec, "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roofline, "cpu_baseline": None, "cpu_baseline_note": "reported by the N=1 run", "parity": None,
            "sharding": {"mode": "rows (one graph)", "same_graph_as_1gpu": same, "one_gpu_same_run": one_gpu, "per_rank": per_rank,
                         "distribute_seconds": t_dist,
                         "speedup_vs_one_gpu_same_run": value / one_gpu["value"] if one_gpu else None},
            "pq": None,
            "build": {"vectors_per_s": n / t_build, "seconds": t_build, "datagen_seconds": t_gen, "where": "rank 0 (one graph)",
                      "dist_evals_per_vector": build_work[0] / max(1, n), "device_seconds": build_work[2] / 1e3},
        }
        print(json.dumps(line))
    grp.close()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--query-pool", type=int, default=32, help="distinct query batches (cycled over the steps)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("LB200_WORKLOAD", "cfg3"), choices=sorted(WORKLOADS))
    ap.add_argument("--shard-mode", default="rows", choices=["rows", "graphs"],
                    help="--gpus > 1: 'rows' = ONE graph, vectors sharded by row range, distances evaluated on the owning GPU "
                         "(lb200_group_*, results identical to 1 GPU); 'graphs' = round 1's independent graph per shard + NCCL "
                         "all-gather + merge with a recall-matched per-shard ef")
    ap.add_argument("--shard-ef", type=int, default=0,
                    help="--gpus > 1: per-shard ef; 0 = recall-matched (smallest ef_s whose merged recall reaches the unsharded "
                         "1-GPU recall at the workload's ef), -1 = same ef as the workload")
    ap.add_argument("--recall-target", type=float, default=0.0,
                    help="--gpus > 1: unsharded 1-GPU recall to match (0 = measure it here by building the full graph)")
    ap.add_argument("--replicated-comparison", action="store_true", help="--gpus > 1: force the replicated comparison")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="bound on the cpu_baseline search time")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-prefix-rows", type=int, default=1_000_000,
                    help="corpora above 8 GB: rows of the prefix graph the engine builds for the reference to load (cpu_baseline)")
    ap.add_argument("--search-expand", type=int, default=1, help="candidates expanded per search round (1 = the reference's exact order)")
    ap.add_argument("--pq-ref-rows", type=int, default=100_000, help="pq workloads: rows the reference indexes for cpu_baseline")
    ap.add_argument("--ref-seconds", type=float, default=60.0, help="--impl reference: target duration of the K timed steps")
    ap.add_argument("--ref-rows", type=int, default=200_000,
                    help="--impl reference: corpus prefix the reference indexes (fixed, so the arm is the same on every box and N)")
    ap.add_argument("--per-step-stats", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the results of the last timed step (keys, distances, counts) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl)
    elif int(os.environ.get("WORLD_SIZE", "1")) > 1 and args.shard_mode == "rows" and not wl.get("pq") and DEVICE_TYPE == "cuda":
        run_group(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
