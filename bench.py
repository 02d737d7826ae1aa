#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on its config 2 (the 1xB200 IVF_PQ case):
ANN queries/sec, 1M x 768 f32, IVF_PQ nlist=1024, PQ m=96x8bit, nprobes=20, k=10, batch=1024.

A "step" = one pass of the hot path over one batch of 1024 synthetic queries.
  value     : whole-job QPS with queries/results resident in HBM (lgpu_search_device),
              timed per step with CUDA events on the launching stream, L2 flushed
              (untimed) between steps;
  e2e       : the same metric through the host-buffer C-ABI call (lgpu_search) with pinned
              host buffers, H2D of the queries and D2H of the results inside the timed region,
              L2 flushed (untimed) between calls; `e2e.pipelined` = the same batches through
              lgpu_search_async with two calls in flight (no flush possible inside a pipeline);
  roofline  : algorithmic PQ-code bytes of the batch / the scan kernel's measured duration
              (CUDA events recorded around the kernel by the library) vs the measured HBM peak;
  cpu_baseline : the CPU oracle (a port of the reference's lance path) on the host cores the
              process may actually use (affinity and cgroup quota), best of 3 repetitions;
  gate      : before anything is timed, the GPU results of 128 ground-truth queries must be
              bit-identical to the CPU oracle's (plain and refine_factor=10); recall@k of both.
N == 1 also reports `latency` (B=1 p50/p99 through the host-buffer calls) and `extra_workloads`
(BASELINE.json configs[0], [2], [3] at full size, and config 2 on SURVEY.md 8d's clustered data).
N > 1 (torchrun): `value` = independent replicas, one batch per rank per step, no data-path
collective ("scaling": "weak").  In the same run every rank also executes the partition-sharded
path (lgpu_search_sharded_device: one in-library ncclAllGather of 16-byte top-k records + merge):
`sharded` = config 2 split N ways on ONE shared batch, gated bit-for-bit against the single-GPU
result and the oracle; `c5` = a BASELINE configs[4]-shaped shard (12.2M rows per GPU, nlist 16384,
batch 8192; the true 100M-row config at N = 8), oracle-checked on the probed partitions.
`--impl reference` times the CPU oracle alone (the reference's Rust path cannot be built
here: no cargo, lance un-vendored), rank 0 only.
`--dump-outputs DIR` writes what the timed search returned in its last timed step (rank 0) as
DIR/ids.npy, DIR/distances.npy and DIR/counts.npy.  The index, the queries and hence these arrays are the
same on every run with the same arguments, so two builds can be compared output for output.
"""
import argparse
import json
import math
import os
import stat
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# cuBLAS is only run-to-run deterministic with a fixed workspace configuration; the index training below runs with
# torch's deterministic algorithms, which require it.  Read when torch creates its first cuBLAS handle.
os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")

WORKLOADS = {
    # BASELINE.json configs[1]
    "c2": dict(n=1_000_000, dim=768, nlist=1024, m=96, nprobes=20, k=10, batch=1024, metric="l2", data="latent"),
    # the same on SURVEY.md 8d's clustered variant
    "c2c": dict(n=1_000_000, dim=768, nlist=1024, m=96, nprobes=20, k=10, batch=1024, metric="l2", data="clustered"),
    # small variant for local CPU checks of the harness itself
    "tiny": dict(n=20_000, dim=64, nlist=32, m=8, nprobes=4, k=10, batch=64, metric="l2", data="latent"),
}
# index training: the reference's defaults (rust/lancedb/src/index/vector.rs:286-297)
TRAIN = dict(max_iterations=50, sample_rate=256)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


# ------------------------------------------------------------------------------------------ host cores
def host_threads():
    """Threads the CPU arm may really use: min(affinity mask, cgroup CPU quota).  os.cpu_count() alone
    over-subscribes a quota-limited lease (round 1: 128 threads on a 4.7x smaller quota)."""
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = os.cpu_count() or 1
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:                      # cgroup v2
            a, b = f.read().split()[:2]
            if a != "max":
                quota = float(a) / float(b)
    except Exception:
        try:                                                           # cgroup v1
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                p = float(f.read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    threads = aff if quota is None else max(1, min(aff, int(math.ceil(quota))))
    model = "unknown"
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    model = line.split(":", 1)[1].strip()
                    break
    except Exception:
        pass
    return threads, {"cpu_model": model, "os_cpu_count": os.cpu_count(), "affinity": aff,
                     "cgroup_quota_cpus": quota, "threads_used": threads}


# ------------------------------------------------------------------------------------------ synthetic data
LATENT_RANK = 32
DATA_DESC = {
    "latent": ("synthetic float32: rank-32 Gaussian latent z@A (A fixed, seed 44) + N(0, 0.05^2) noise; "
               "base seed 42, queries seed 43"),
    "clustered": ("synthetic float32 (SURVEY.md 8d clustered variant): 4*nlist Gaussian blobs, centres N(0,1) "
                  "seed 44, sigma 0.3; base seed 42, queries = held-out samples seed 43"),
}


def _gen(seed, device):
    import torch
    dev = "cuda" if str(device).startswith("cuda") else "cpu"
    return torch.Generator(device=dev).manual_seed(seed), (device if dev == "cuda" else "cpu")


def synth_vectors(cfg, n, seed, device):
    """Synthetic float32[dim] vectors.
    latent: x = z A + 0.05 eps, z ~ N(0, I_32), A a fixed 32 x dim matrix -- a low intrinsic dimension like
    real embeddings.  Pure i.i.d. N(0,1) in 768-d (SURVEY.md 8d's first variant) has no neighbourhood
    structure: k-means on it degenerates (partition sizes std/mean 2.3, recall@10 ~ 0.04), so the workload
    would no longer be BASELINE.md's 1.875 MB of codes per query.
    clustered: SURVEY.md 8d's second variant, 4*nlist blobs with sigma 0.3 around N(0,1) centres.
    The generator lives on the device that holds the data (same stream on every rank / both bench arms)."""
    import torch
    g44, gdev = _gen(44, device)
    g, _ = _gen(seed, device)
    dim = cfg["dim"]
    out = torch.empty(n, dim, dtype=torch.float32, device=device)
    chunk = 1 << 17
    if cfg.get("data", "latent") == "clustered":
        nb = 4 * cfg["nlist"]
        centres = torch.randn(nb, dim, generator=g44, device=gdev).to(device)
        for s in range(0, n, chunk):
            e = min(n, s + chunk)
            a = torch.randint(0, nb, (e - s,), generator=g, device=gdev).to(device)
            out[s:e] = centres[a] + 0.3 * torch.randn(e - s, dim, generator=g, device=gdev).to(device)
        return out
    A = (torch.randn(LATENT_RANK, dim, generator=g44, device=gdev) / LATENT_RANK ** 0.5).to(device)
    for s in range(0, n, chunk):
        e = min(n, s + chunk)
        z = torch.randn(e - s, LATENT_RANK, generator=g, device=gdev).to(device)
        eps = torch.randn(e - s, dim, generator=g, device=gdev).to(device)
        out[s:e] = z @ A + 0.05 * eps
    return out


def index_cache_path(cfg, tag, device):
    """Trained indexes are cached in a temporary directory of this user's own.  On a shared host that name can
    already be taken by someone else: unless the directory is ours and private, returns None (train, do not cache)."""
    key = "_".join(f"{k}{cfg[k]}" for k in ("n", "dim", "nlist", "m", "metric", "data"))
    dev = "cuda" if str(device).startswith("cuda") else "cpu"
    d = os.path.join(tempfile.gettempdir(), f"lancedb_b200_bench_{os.getuid()}")
    try:
        os.mkdir(d, 0o700)
        os.chmod(d, 0o700)                      # whatever the umask
    except FileExistsError:
        pass
    st = os.lstat(d)
    if not stat.S_ISDIR(st.st_mode) or st.st_uid != os.getuid() or stat.S_IMODE(st.st_mode) != 0o700:
        log(f"[bench] {d} is not a private directory of this user: the index is not cached")
        return None
    return os.path.join(d, f"v3_{tag}_{key}_{dev}_it{TRAIN['max_iterations']}_sr{TRAIN['sample_rate']}.npz")


def get_index(cfg, tag, device):
    """Train (setup, untimed) or load the synthetic index; also returns exact top-k ground truth for 128
    held-out queries and the build time."""
    from lancedb_b200.index import IvfPqIndexData, train_ivf_pq
    import torch
    path = index_cache_path(cfg, tag, device)
    if path is not None and os.path.exists(path):
        z = np.load(path)
        ix = IvfPqIndexData(int(z["dim"]), int(z["nlist"]), int(z["m"]), str(z["metric"]), z["centroids"],
                            z["codebook"], z["part_offsets"], z["codes_t"], z["row_ids"], None)
        return ix, z["gt_queries"], z["gt_ids"], float(z["build_s"])
    t0 = time.time()
    x = synth_vectors(cfg, cfg["n"], 42, device)
    t1 = time.time()
    # the k-means updates (index_add_ / scatter_add_) sum with float atomics on CUDA unless torch is asked for its
    # deterministic kernels: without them every training run yields a slightly different index.  An op without a
    # deterministic kernel raises here rather than quietly making the index vary from run to run.
    mode = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())
    torch.use_deterministic_algorithms(True)
    try:
        ix = train_ivf_pq(x, num_partitions=cfg["nlist"], num_sub_vectors=cfg["m"], distance_type=cfg["metric"],
                          max_iterations=TRAIN["max_iterations"], sample_rate=TRAIN["sample_rate"], device=device)
    finally:
        torch.use_deterministic_algorithms(mode[0], warn_only=mode[1])
    build_s = time.time() - t1
    gq = synth_vectors(cfg, 128, 4343, device)
    xs = x / x.norm(dim=1, keepdim=True) if cfg["metric"] == "cosine" else x
    qs = gq / gq.norm(dim=1, keepdim=True) if cfg["metric"] == "cosine" else gq
    d = (xs * xs).sum(1)[None, :] - 2.0 * qs @ xs.T
    gt = d.topk(cfg["k"], largest=False).indices.cpu().numpy().astype(np.uint64)
    gqn = gq.cpu().numpy()
    del x, xs, d
    if path is not None:
        tmp = path + f".{os.getpid()}.tmp.npz"
        np.savez(tmp, dim=ix.dim, nlist=ix.nlist, m=ix.m, metric=ix.metric, centroids=ix.centroids,
                 codebook=ix.codebook, part_offsets=ix.part_offsets, codes_t=ix.codes_t, row_ids=ix.row_ids,
                 gt_queries=gqn, gt_ids=gt, build_s=build_s)
        os.replace(tmp, path)
    log(f"[bench] index built in {time.time() - t0:.1f}s (training+encoding {build_s:.1f}s) -> {path or 'not cached'}")
    return ix, gqn, gt, build_s


def attach_vectors(cfg, ix, device):
    """Raw vectors in the index's row order (refine_factor needs them): regenerated, not cached."""
    import torch
    x = synth_vectors(cfg, cfg["n"], 42, device)
    order = torch.as_tensor(ix.row_ids.astype(np.int64), device=x.device)
    ix.vectors = x[order].cpu().numpy()
    del x
    return ix


def synthetic_uniform_index(n, dim, nlist, m, metric, seed, owner=None, rank=0):
    """Untrained index with uniform-ish partitions (+-30 %) and random codes: throughput and parity do not
    depend on index quality, and 10M / 100M-row indexes cannot be trained inside a bench run.  Every
    partition is generated from its own seed, so any rank (and the oracle check) can rebuild any partition.
    owner: optional [nlist] rank of each partition; non-owned partitions are empty on this rank."""
    from lancedb_b200.index import IvfPqIndexData
    rng = np.random.default_rng(seed)
    dsub = dim // m
    base = n // nlist
    sizes = rng.integers(int(base * 0.7), int(base * 1.3) + 1, nlist).astype(np.int64)
    cent = rng.standard_normal((nlist, dim), dtype=np.float32)
    if metric == "cosine":
        cent /= np.linalg.norm(cent, axis=1, keepdims=True)
    cb = (rng.standard_normal((m, 256, dsub), dtype=np.float32) * 0.3).astype(np.float32)
    goff = np.zeros(nlist + 1, np.uint64)
    goff[1:] = np.cumsum(sizes)
    mine = np.ones(nlist, bool) if owner is None else (owner == rank)
    local = np.where(mine, sizes, 0)
    off = np.zeros(nlist + 1, np.uint64)
    off[1:] = np.cumsum(local)
    nloc = int(off[-1])
    codes = np.empty(nloc * m, np.uint8)
    ids = np.empty(nloc, np.uint64)
    for p in np.nonzero(mine)[0]:
        a, b = int(off[p]), int(off[p + 1])
        codes[a * m:b * m] = partition_codes(seed, int(p), b - a, m)
        ids[a:b] = np.arange(int(goff[p]), int(goff[p]) + (b - a), dtype=np.uint64)
    return IvfPqIndexData(dim, nlist, m, metric, cent, cb, off, codes, ids, None), sizes, goff


def partition_codes(seed, p, n_p, m):
    return np.random.default_rng([seed, 7, p]).integers(0, 256, size=n_p * m, dtype=np.uint8)


def sparse_oracle_index(full_desc, sizes, goff, parts, seed):
    """The oracle's view of a huge synthetic index restricted to the partitions `parts` (all others empty):
    enough to check queries whose probes fall inside `parts`."""
    from lancedb_b200.index import IvfPqIndexData
    keep = np.zeros(full_desc.nlist, bool)
    keep[np.asarray(parts, np.int64)] = True
    local = np.where(keep, sizes, 0)
    off = np.zeros(full_desc.nlist + 1, np.uint64)
    off[1:] = np.cumsum(local)
    m = full_desc.m
    codes = np.empty(int(off[-1]) * m, np.uint8)
    ids = np.empty(int(off[-1]), np.uint64)
    for p in np.nonzero(keep)[0]:
        a, b = int(off[p]), int(off[p + 1])
        codes[a * m:b * m] = partition_codes(seed, int(p), b - a, m)
        ids[a:b] = np.arange(int(goff[p]), int(goff[p]) + (b - a), dtype=np.uint64)
    return IvfPqIndexData(full_desc.dim, full_desc.nlist, m, full_desc.metric, full_desc.centroids,
                          full_desc.codebook, off, codes, ids, None)


# ------------------------------------------------------------------------------------------ clocks / peaks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i",
                 str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            j = json.load(f)
        return float(j["hbm_gbs"]), float(j["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, 1400.0, "fallback (B200_PROFILING.md)"


def profiled_traffic():
    """dram__bytes_read+write per launch of the scan kernel from the committed ncu --set full capture
    (profiles/): a profiler number, so it is read from the profile, never measured in this run."""
    try:
        cands = sorted(f for f in os.listdir(os.path.join(ROOT, "profiles")) if f.endswith("_scan_traffic.json"))
        with open(os.path.join(ROOT, "profiles", cands[-1])) as f:
            j = json.load(f)
        return float(j["dram_bytes_per_launch"]), j.get("kernel")
    except Exception:
        return None, None


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_baseline(cfg, orc, queries, seconds=4.0, reps=3):
    """The oracle (port of the lance CPU path) on the usable host cores: bounded sample, best of `reps`."""
    threads, info = host_threads()
    probe = queries[:max(threads, 8)]
    t0 = time.perf_counter()
    orc.search(probe, k=cfg["k"], nprobes=cfg["nprobes"], nthreads=threads)
    per_q = (time.perf_counter() - t0) / len(probe)
    n = int(min(len(queries), max(threads * 4, seconds / max(per_q, 1e-6))))
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        orc.search(queries[:n], k=cfg["k"], nprobes=cfg["nprobes"], nthreads=threads)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    out = {"value": n / best, "unit": "queries/s", "cores": threads, "kind": "port",
           "sample": f"{n} queries of the same workload, best of {reps} x {best:.1f}s, oracle/oracle.c "
                     f"(-O3 -mavx2 -mfma) with {threads} threads"}
    out.update(info)
    return out


def run_reference(args, cfg):
    """--impl reference: the CPU oracle alone, rank 0 only."""
    rank, local, world = dist_env()
    if rank != 0:
        return
    import oracle
    import torch
    device = f"cuda:{local}" if torch.cuda.is_available() else "cpu"
    ix, gq, gt, _ = get_index(cfg, args.workload, device)
    B = cfg["batch"]
    threads, info = host_threads()
    orc = oracle.OracleIndex.from_data(ix)
    nb = 4
    q = synth_vectors(cfg, B * nb, 43, device).cpu().numpy().reshape(nb, B, cfg["dim"])
    for i in range(args.warmup):
        orc.search(q[i % nb][: max(threads, B // 8)], k=cfg["k"], nprobes=cfg["nprobes"], nthreads=threads)
    t0 = time.perf_counter()
    for i in range(args.steps):
        res = orc.search(q[i % nb], k=cfg["k"], nprobes=cfg["nprobes"], nthreads=threads)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *res)
    qps = B * args.steps / dt
    gi, _, _ = orc.search(gq, k=cfg["k"], nprobes=cfg["nprobes"], nthreads=threads)
    recall = float(np.mean([len(set(gi[i].tolist()) & set(gt[i].tolist())) / cfg["k"] for i in range(len(gq))]))
    sample = f"{B} queries per step (the full batch), oracle/oracle.c, {threads} threads"
    cb = {"value": qps, "unit": "queries/s", "cores": threads, "kind": "port", "sample": sample}
    cb.update(info)
    _emit({
        "impl": "reference", "metric": "ANN queries/sec (IVF_PQ)", "value": qps, "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": DATA_DESC[cfg["data"]], "config": workload_config(cfg, args, 1, "cpu"),
        "recall_at_k": recall, "cpu_baseline": cb,
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


def workload_config(cfg, args, world, par):
    return {"workload": f"{cfg['n']}x{cfg['dim']} f32, IVF_PQ nlist={cfg['nlist']} m={cfg['m']}x8bit, "
                        f"nprobes={cfg['nprobes']}, k={cfg['k']}, batch={cfg['batch']}, {cfg['metric']}",
            "baseline_config": "BASELINE.json configs[1]" if args.workload in ("c2", "c2c") else args.workload,
            "batch_per_gpu": cfg["batch"], "global_batch": cfg["batch"] * (world if par == "replicas" else 1),
            "parallelism": par if world > 1 else "single",
            "index_training": f"k-means max_iterations={TRAIN['max_iterations']} sample_rate={TRAIN['sample_rate']} "
                              "(the reference's defaults, index/vector.rs:286-297)",
            "l2_flush": "512 MiB write between steps (untimed); each step uses a different query batch"}


_REAL_STDOUT = None


def _quiet_stdout():
    """The contract is ONE JSON line on stdout.  Libraries underneath (NCCL prints its version banner to
    fd 1 when NCCL_DEBUG is set in the environment) write there too, so fd 1 points at stderr until
    _emit() prints the line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def _emit(obj):
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(obj), flush=True)


def recall_of(ids, gt, k):
    return float(np.mean([len(set(ids[i].tolist()) & set(gt[i].tolist())) / k for i in range(len(gt))]))


def same(a, b):
    return bool(np.array_equal(a[0], b[0]) and np.array_equal(np.asarray(a[1]).view(np.uint32), np.asarray(b[1]).view(np.uint32))
                and np.array_equal(np.asarray(a[2]).view(np.uint32), np.asarray(b[2]).view(np.uint32)))


def dump_outputs(out_dir, ids, dist, cnt):
    """One search's results as a caller receives them: ids [B,k] u64, distances [B,k] f32, counts [B] u32.  Ids and
    counts are stored as float64 (exact below 2**53; an empty slot's id UINT64_MAX reads 2**64)."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"ids": np.asarray(ids).view(np.uint64).astype(np.float64),
              "distances": np.asarray(dist, np.float32),
              "counts": np.asarray(cnt).view(np.uint32).astype(np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ------------------------------------------------------------------------------------------ timing helpers
class DeviceRunner:
    """Device-resident timing of an IVF_PQ handle: CUDA events per step on the launching stream, 512 MiB L2
    flush (untimed) between steps."""

    def __init__(self, torch, device, flush):
        self.torch, self.device, self.flush = torch, device, flush

    def time(self, fn, steps, warmup):
        torch = self.torch
        for i in range(warmup):
            fn(i)
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for i in range(steps):
            self.flush.zero_()
            ev[i][0].record()
            fn(i)
            ev[i][1].record()
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in ev]


def ivf_extra_workload(torch, _native, name, icfg, runner, peak_gbs, steps=4, check=4, seed=11):
    """Full-size BASELINE config on a synthetic uniform index: QPS, scan roofline fraction, oracle spot check."""
    import oracle
    t0 = time.time()
    ix, sizes, goff = synthetic_uniform_index(icfg["n"], icfg["dim"], icfg["nlist"], icfg["m"], icfg["metric"], seed)
    gen_s = time.time() - t0
    gpu = _native.GpuIvfPq(ix, device=torch.cuda.current_device(), with_vectors=False)
    B, k, dim = icfg["batch"], icfg["k"], icfg["dim"]
    g = torch.Generator().manual_seed(3)
    q = torch.randn(2, B, dim, generator=g)
    dq = q.cuda()
    oi = torch.empty(B, k, dtype=torch.int64, device="cuda"); od = torch.empty(B, k, device="cuda")
    oc = torch.empty(B, dtype=torch.int32, device="cuda")
    p = _native.make_params(k=k, nprobes=icfg["nprobes"])
    st = torch.cuda.current_stream().cuda_stream
    fn = lambda i: gpu.search_device(dq[i % 2].data_ptr(), B, p, oi.data_ptr(), od.data_ptr(), oc.data_ptr(), st)
    ms = runner.time(fn, steps, 2)
    _native.set_profiling(True)
    fn(steps - 1)
    stage = _native.last_stage_ms(); code_bytes = _native.last_scanned_code_bytes()
    fstats = _native.last_filter_stats()
    _native.set_profiling(False)
    torch.cuda.synchronize()
    got = (oi.cpu().numpy().view(np.uint64)[:check], od.cpu().numpy()[:check], oc.cpu().numpy().view(np.uint32)[:check])
    threads, _ = host_threads()
    want = oracle.OracleIndex.from_data(ix).search(q[(steps - 1) % 2, :check].numpy(), k=k, nprobes=icfg["nprobes"],
                                                   nthreads=threads)
    achieved = code_bytes / (stage["scan"] / 1e3) / 1e9
    out = {"config": name, "workload": f"{icfg['n']}x{dim} f32, IVF_PQ nlist={icfg['nlist']} m={icfg['m']}, nprobes="
                                       f"{icfg['nprobes']}, k={k}, batch={B}, {icfg['metric']}; synthetic uniform "
                                       "partitions, random codes (untrained)",
           "ms_per_batch": float(np.mean(ms)), "qps": B / (float(np.mean(ms)) / 1e3), "steps": steps,
           "stage_ms": stage, "filter_stats": fstats, "oracle_check": same(got, want), "oracle_check_queries": check,
           "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                        "frac": achieved / peak_gbs, "kernel_ms": stage["scan"],
                        "algorithmic_bytes_per_launch": code_bytes,
                        "whole_step_frac": code_bytes / (float(np.mean(ms)) / 1e3) / 1e9 / peak_gbs},
           "index_rows": int(ix.nrows), "index_generate_s": gen_s}
    gpu.close()
    del dq, oi, od, oc
    torch.cuda.empty_cache()
    return out


def flat_extra_workload(torch, _native, runner, peak_tf, steps=5, check=4):
    """BASELINE configs[3]: 1M x 1536 flat L2 as a bf16 tensor-core GEMM shortlist + exact f32 re-score + top-k."""
    import oracle
    N, dim, B, k = 1_000_000, 1536, 1024, 10
    g = torch.Generator(device="cuda").manual_seed(5)
    v = torch.randn(N, dim, generator=g, device="cuda").cpu().numpy()
    fl = _native.GpuFlat(v, device=torch.cuda.current_device())
    q = torch.randn(2, B, dim, generator=g, device="cuda")
    oi = torch.empty(B, k, dtype=torch.int64, device="cuda"); od = torch.empty(B, k, device="cuda")
    oc = torch.empty(B, dtype=torch.int32, device="cuda")
    p = _native.make_params(k=k, nprobes=0)
    st = torch.cuda.current_stream().cuda_stream
    fn = lambda i: fl.search_device("l2", q[i % 2].data_ptr(), B, p, oi.data_ptr(), od.data_ptr(), oc.data_ptr(), st)
    ms = runner.time(fn, steps, 2)
    torch.cuda.synchronize()
    got = (oi.cpu().numpy().view(np.uint64)[:check], od.cpu().numpy()[:check], oc.cpu().numpy().view(np.uint32)[:check])
    threads, _ = host_threads()
    want = oracle.flat_search(v, q[(steps - 1) % 2, :check].cpu().numpy(), k=k, nthreads=threads)
    t = float(np.mean(ms)) / 1e3
    flops = 2.0 * B * N * dim
    out = {"config": "BASELINE.json configs[3]", "workload": f"{N}x{dim} f32 flat L2, batch={B}, k={k}; i.i.d. N(0,1)",
           "ms_per_batch": t * 1e3, "qps": B / t, "steps": steps, "oracle_check": same(got, want),
           "oracle_check_queries": check,
           "roofline": {"bound": "tensor", "achieved": flops / t / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
                        "frac": flops / t / 1e12 / peak_tf, "note": "whole step (GEMM shortlist + exact re-score + "
                        "top-k) over 2*B*N*d flops, vs the sustained bf16 peak"}}
    fl.close()
    del v, q
    torch.cuda.empty_cache()
    return out


def latency_lines(torch, _native, gpu, cfg, qn, flush, reps=200):
    """B=1 latency through the host-buffer calls: the IVF_PQ index (config 2) and BASELINE configs[0]
    (100k x 128 flat L2, the reference's CPU-runnable case) with the CPU port's single-query latency beside it."""
    import oracle
    k = cfg["k"]
    p = _native.make_params(k=k, nprobes=cfg["nprobes"])
    hi = torch.empty(1, k, dtype=torch.int64).pin_memory().numpy().view(np.uint64)
    hd = torch.empty(1, k, dtype=torch.float32).pin_memory().numpy()
    hc = torch.empty(1, dtype=torch.int32).pin_memory().numpy().view(np.uint32)
    q1 = torch.from_numpy(qn.reshape(-1, cfg["dim"])[:reps].copy()).pin_memory().numpy()

    def pct(fn, n):
        for i in range(10):
            fn(i)
        t = []
        for i in range(n):
            t0 = time.perf_counter()
            fn(i)
            t.append((time.perf_counter() - t0) * 1e6)
        return {"p50_us": float(np.percentile(t, 50)), "p99_us": float(np.percentile(t, 99)), "calls": n}

    out = {"ivf_pq_b1": pct(lambda i: gpu.search_into(q1[i % reps:i % reps + 1], p, hi, hd, hc), reps)}
    out["ivf_pq_b1"]["call"] = "lgpu_search, B=1, pinned host buffers, config 2 index, nprobes=20, k=10"
    # C1
    rng = np.random.default_rng(42)
    v = rng.standard_normal((100_000, 128), dtype=np.float32)
    fq = torch.from_numpy(np.random.default_rng(43).standard_normal((reps, 128), dtype=np.float32)).pin_memory().numpy()
    fl = _native.GpuFlat(v, device=torch.cuda.current_device())
    pf = _native.make_params(k=k, nprobes=0)
    c1 = pct(lambda i: fl.search_into("l2", fq[i % reps:i % reps + 1], pf, hi, hd, hc), reps)
    fi, fd, fc = fl.search(fq[:8], k=k)
    oi, od, ocn = oracle.flat_search(v, fq[:8], k=k)
    c1["oracle_check"] = same((fi, fd, fc), (oi, od, ocn))
    t = []
    for i in range(20):
        t0 = time.perf_counter()
        oracle.flat_search(v, fq[i:i + 1], k=k, nthreads=1)
        t.append((time.perf_counter() - t0) * 1e6)
    c1["cpu_port_p50_us"] = float(np.percentile(t, 50))
    c1["call"] = "lgpu_flat_search, B=1, pinned host buffers; BASELINE.json configs[0] (100k x 128 f32 flat L2); " \
                 "cpu = oracle flat_search, 1 thread"
    out["c1_flat_b1"] = c1
    fl.close()
    return out


# ------------------------------------------------------------------------------------------ main
def main():
    _quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--parallelism", default="replicas", choices=["replicas", "sharded"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip latency / extra_workloads / sharded / c5 blocks")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's ids / distances / counts as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = WORKLOADS[args.workload]
    args.warmup = max(args.warmup, 3) if args.impl == "native" else args.warmup
    if args.impl == "reference":
        return run_reference(args, cfg)

    import torch
    import oracle
    from lancedb_b200 import _native
    rank, local, world = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (lancedb_b200 has no CPU fallback)")
    torch.cuda.set_device(local)
    device = f"cuda:{local}"
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device(device))
    par = args.parallelism if world > 1 else "replicas"
    threads, _ = host_threads()
    peak_gbs, peak_tf, peak_src = measured_peaks()

    # ---- setup (untimed): index, queries ----
    if rank == 0:
        ix, gq, gt, build_s = get_index(cfg, args.workload, device)
    if world > 1:
        dist.barrier()
    if rank != 0:
        ix, gq, gt, build_s = get_index(cfg, args.workload, device)
    torch.cuda.empty_cache()
    full_ix = ix
    B, k, dim = cfg["batch"], cfg["k"], cfg["dim"]
    if rank == 0:
        attach_vectors(cfg, full_ix, device)          # refine_factor gate needs the raw vectors
    comm = None
    if par == "sharded":
        from lancedb_b200.distributed import exchange_unique_id
        gpu = _native.GpuIvfPq(ix.shard(rank, world), device=local, with_vectors=False)
        comm = _native.Comm(exchange_unique_id(), rank, world, local)
    else:
        gpu = _native.GpuIvfPq(full_ix, device=local, with_vectors=rank == 0)
    nb = 8
    qseed = 43 if par == "sharded" else 43 + 1000 * rank
    q_host = torch.empty(nb, B, dim, dtype=torch.float32).pin_memory()
    q_host.copy_(synth_vectors(cfg, nb * B, qseed, device).reshape(nb, B, dim))
    d_q = q_host.to(device)
    d_ids = torch.empty(B, k, dtype=torch.int64, device=device)     # u64 payload
    d_dist = torch.empty(B, k, dtype=torch.float32, device=device)
    d_cnt = torch.empty(B, dtype=torch.int32, device=device)
    h_ids = [torch.empty(B, k, dtype=torch.int64).pin_memory() for _ in range(2)]
    h_dist = [torch.empty(B, k, dtype=torch.float32).pin_memory() for _ in range(2)]
    h_cnt = [torch.empty(B, dtype=torch.int32).pin_memory() for _ in range(2)]
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=device)
    p = _native.make_params(k=k, nprobes=cfg["nprobes"])
    stream = torch.cuda.current_stream().cuda_stream

    def step_device(i):
        if par == "sharded":
            comm.search_device(gpu, d_q[i % nb].data_ptr(), B, p, d_ids.data_ptr(), d_dist.data_ptr(), d_cnt.data_ptr(), stream)
        else:
            gpu.search_device(d_q[i % nb].data_ptr(), B, p, d_ids.data_ptr(), d_dist.data_ptr(), d_cnt.data_ptr(), stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- correctness gate before timing (rank 0, full index): GPU == CPU oracle bit for bit on the 128
    # ground-truth queries, plain and refine_factor=10; recall@k of both arms vs exact flat top-k ----
    gate = None
    if rank == 0 and par == "replicas":
        orc = oracle.OracleIndex.from_data(full_ix)
        g_plain = gpu.search(gq, k=k, nprobes=cfg["nprobes"])
        o_plain = orc.search(gq, k=k, nprobes=cfg["nprobes"], nthreads=threads)
        g_ref = gpu.search(gq, k=k, nprobes=cfg["nprobes"], refine_factor=10)
        o_ref = orc.search(gq, k=k, nprobes=cfg["nprobes"], refine_factor=10, nthreads=threads)
        gate = {"queries": int(len(gq)), "gpu_equals_oracle_plain": same(g_plain, o_plain),
                "gpu_equals_oracle_refine10": same(g_ref, o_ref),
                "recall_at_k_gpu": recall_of(g_plain[0], gt, k), "recall_at_k_cpu": recall_of(o_plain[0], gt, k),
                "recall_at_k_refine10_gpu": recall_of(g_ref[0], gt, k),
                "recall_at_k_refine10_cpu": recall_of(o_ref[0], gt, k)}
        if not (gate["gpu_equals_oracle_plain"] and gate["gpu_equals_oracle_refine10"]):
            raise SystemExit(f"[bench] parity gate failed: {gate}")
        # what limits recall on this data: PQ error (refine removes it) or IVF coverage (more probes remove it)
        sweep = {}
        for npb in (20, 50, 100, 200):
            r = gpu.search(gq, k=k, nprobes=npb, refine_factor=10)
            sweep[str(npb)] = recall_of(r[0], gt, k)
        gate["recall_at_k_refine10_vs_nprobes"] = sweep

    sampler = ClockSampler(local)      # samples clocks / throttle reasons through regions (1) and (2)
    sampler.start()
    t_wait = time.time()
    while not sampler.rows and time.time() - t_wait < 3.0:      # rank-local work only: no collectives here
        gpu.search_device(d_q[0].data_ptr(), B, p, d_ids.data_ptr(), d_dist.data_ptr(), d_cnt.data_ptr(), stream)
        torch.cuda.synchronize()
    for i in range(args.warmup):
        step_device(i)
    barrier()
    # ---- (1) device-resident timed region ----
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    launches0 = _native.kernel_launch_count()
    for i in range(args.steps):
        flush.zero_()
        ev[i][0].record()
        step_device(i)
        ev[i][1].record()
    barrier()
    launches = _native.kernel_launch_count() - launches0
    if args.dump_outputs and rank == 0:            # before the regions below overwrite d_ids / d_dist / d_cnt
        dump_outputs(args.dump_outputs, d_ids.cpu().numpy(), d_dist.cpu().numpy(), d_cnt.cpu().numpy())
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    units = B * args.steps * (world if par == "replicas" else 1)
    value = units / (total_ms / 1e3)

    # ---- (2) end to end through the host-buffer C-ABI calls (pinned host memory) ----
    qn = q_host.numpy()
    hi = [t.numpy().view(np.uint64) for t in h_ids]; hd = [t.numpy() for t in h_dist]
    hc = [t.numpy().view(np.uint32) for t in h_cnt]
    e2e_val = e2e_pipe = None
    if par == "replicas":
        for i in range(3):
            gpu.search_into(qn[i % nb], p, hi[0], hd[0], hc[0])
        barrier()
        e2e_s = 0.0
        for i in range(args.steps):
            flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            gpu.search_into(qn[i % nb], p, hi[0], hd[0], hc[0])      # H2D + kernels + D2H + sync inside
            e2e_s += time.perf_counter() - t0
        e2e_t = torch.tensor([e2e_s], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
        e2e_val = units / float(e2e_t.item())
        # pipelined: two lgpu_search_async calls in flight (batch i+1's H2D under batch i's kernels); the warm-up
        # runs the same two-in-flight pattern so that both workspaces are allocated and captured before the clock
        prev = None
        for i in range(8):
            t = gpu.search_async(qn[i % nb], p, hi[i % 2], hd[i % 2], hc[i % 2])
            if prev is not None:
                _native.ticket_wait(prev)
            prev = t
        _native.ticket_wait(prev)
        barrier()
        t0 = time.perf_counter()
        prev = None
        for i in range(args.steps):
            t = gpu.search_async(qn[i % nb], p, hi[i % 2], hd[i % 2], hc[i % 2])
            if prev is not None:
                _native.ticket_wait(prev)
            prev = t
        _native.ticket_wait(prev)
        pipe_t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(pipe_t, op=dist.ReduceOp.MAX)
        e2e_pipe = units / float(pipe_t.item())
    clocks = sampler.stop()

    # ---- (3) per-kernel times (library CUDA events on the launching stream) -> roofline ----
    _native.set_profiling(True)
    stage = {}
    scan_ms, code_bytes = [], 0
    prof_steps = min(args.steps, 20)
    for i in range(prof_steps):
        flush.zero_()
        gpu.search_device(d_q[i % nb].data_ptr(), B, p, d_ids.data_ptr(), d_dist.data_ptr(), d_cnt.data_ptr(), stream)
        s = _native.last_stage_ms()
        for kk, v in s.items():
            stage[kk] = stage.get(kk, 0.0) + v / prof_steps
        scan_ms.append(s["scan"])
        code_bytes = _native.last_scanned_code_bytes()
    filter_stats = _native.last_filter_stats()
    _native.set_profiling(False)
    scan_avg = float(np.mean(scan_ms))
    achieved = code_bytes / (scan_avg / 1e3) / 1e9
    traffic, traffic_kernel = profiled_traffic()

    out = None
    if rank == 0:
        out = {
            "metric": "ANN queries/sec (IVF_PQ)", "value": value, "unit": "queries/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "weak" if par == "replicas" else "strong", "vs_baseline": None,
            "dtype": "f32", "data": DATA_DESC[cfg["data"]],
            "config": workload_config(cfg, args, world, par),
            "clocks": clocks,
            "gpu_launches": int(launches),        # counted by the library around region (1), this rank
            "recall_at_k": gate["recall_at_k_gpu"] if gate else None,
            "gate": gate,
            "index_build_s": build_s,
            "stage_ms": stage,
            "filter_stats": filter_stats,        # last profiled batch: candidates appended / re-scored, exact fix-ups
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs,
                         "traffic": traffic, "traffic_kernel": traffic_kernel,
                         "kernel": "PQ code scan (dominant kernel of the step; name in profiles/)",
                         "kernel_ms": scan_avg, "algorithmic_bytes_per_launch": code_bytes, "peak_source": peak_src,
                         "whole_step_frac": code_bytes / (total_ms / args.steps / 1e3) / 1e9 / peak_gbs,
                         "compulsory_bytes_per_launch": int(full_ix.codes_t.size)},
        }
        if e2e_val is not None:
            out["e2e"] = {"value": e2e_val, "unit": "queries/s", "h2d_bytes_per_step": B * dim * 4,
                          "d2h_bytes_per_step": B * k * 12 + B * 4, "call": "lgpu_search (synchronous), L2 flushed between calls",
                          "pipelined": {"value": e2e_pipe, "call": "lgpu_search_async, 2 calls in flight, no L2 flush"}}
        if not args.no_cpu_baseline and world == 1:
            full_ix.vectors = None
            out["cpu_baseline"] = cpu_baseline(cfg, oracle.OracleIndex.from_data(full_ix), qn.reshape(-1, dim))

    # ---- (4) N == 1 extras: B=1 latency, the other BASELINE configs ----
    if world == 1 and not args.no_extras and args.workload != "tiny":
        runner = DeviceRunner(torch, device, flush)
        try:
            out["latency"] = latency_lines(torch, _native, gpu, cfg, qn, flush)
        except Exception as e:                        # an extra must never take the headline line down
            out["latency"] = {"error": repr(e)}
        gpu.close(); gpu = None
        full_ix.vectors = None
        torch.cuda.empty_cache()
        extras = []
        for name, fn in (
            ("c2_clustered", lambda: clustered_workload(torch, _native, oracle, args, device, runner, peak_gbs)),
            ("c3", lambda: ivf_extra_workload(torch, _native, "BASELINE.json configs[2]", dict(
                n=10_000_000, dim=768, nlist=4096, m=96, nprobes=50, k=100, batch=4096, metric="cosine"), runner, peak_gbs)),
            ("c4", lambda: flat_extra_workload(torch, _native, runner, peak_tf)),
        ):
            try:
                t0 = time.time()
                r = fn(); r["name"] = name; r["wall_s"] = time.time() - t0
                extras.append(r)
            except Exception as e:
                extras.append({"name": name, "error": repr(e)})
        out["extra_workloads"] = extras

    # ---- (5) N > 1 extras: the partition-sharded path under the same clock ----
    if world > 1 and par == "replicas" and not args.no_extras:
        try:
            sh = sharded_block(torch, dist, _native, oracle, cfg, full_ix, gpu, rank, local, world, flush, peak_gbs)
        except Exception as e:
            sh = {"error": repr(e)}
        try:
            c5 = c5_block(torch, dist, _native, oracle, rank, local, world, flush, peak_gbs)
        except Exception as e:
            c5 = {"error": repr(e)}
        if rank == 0:
            out["sharded"] = sh
            out["c5"] = c5
    if rank == 0:
        _emit(out)
    if gpu is not None:
        gpu.close()
    if comm is not None:
        comm.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def clustered_workload(torch, _native, oracle, args, device, runner, peak_gbs):
    """Config 2 on SURVEY.md 8d's clustered data: QPS, recall (plain / refine 10), parity gate."""
    cfg = WORKLOADS["c2c"]
    ix, gq, gt, build_s = get_index(cfg, "c2c", device)
    attach_vectors(cfg, ix, device)
    gpu = _native.GpuIvfPq(ix, device=torch.cuda.current_device(), with_vectors=True)
    orc = oracle.OracleIndex.from_data(ix)
    threads, _ = host_threads()
    B, k, dim = cfg["batch"], cfg["k"], cfg["dim"]
    g_plain = gpu.search(gq, k=k, nprobes=cfg["nprobes"]); o_plain = orc.search(gq, k=k, nprobes=cfg["nprobes"], nthreads=threads)
    g_ref = gpu.search(gq, k=k, nprobes=cfg["nprobes"], refine_factor=10)
    o_ref = orc.search(gq, k=k, nprobes=cfg["nprobes"], refine_factor=10, nthreads=threads)
    dq = synth_vectors(cfg, 2 * B, 43, device).reshape(2, B, dim)
    oi = torch.empty(B, k, dtype=torch.int64, device=device); od = torch.empty(B, k, device=device)
    oc = torch.empty(B, dtype=torch.int32, device=device)
    p = _native.make_params(k=k, nprobes=cfg["nprobes"])
    st = torch.cuda.current_stream().cuda_stream
    fn = lambda i: gpu.search_device(dq[i % 2].data_ptr(), B, p, oi.data_ptr(), od.data_ptr(), oc.data_ptr(), st)
    ms = runner.time(fn, 10, 3)
    _native.set_profiling(True)
    fn(0)
    stage = _native.last_stage_ms(); code_bytes = _native.last_scanned_code_bytes()
    fstats = _native.last_filter_stats()
    _native.set_profiling(False)
    sizes = np.diff(ix.part_offsets.astype(np.int64))
    ix.vectors = None
    cpu = cpu_baseline(cfg, oracle.OracleIndex.from_data(ix), dq.reshape(-1, dim).cpu().numpy(), seconds=3.0, reps=2)
    gpu.close()
    torch.cuda.empty_cache()
    achieved = code_bytes / (stage["scan"] / 1e3) / 1e9
    return {"config": "BASELINE.json configs[1], clustered data", "data": DATA_DESC["clustered"],
            "ms_per_batch": float(np.mean(ms)), "qps": B / (float(np.mean(ms)) / 1e3), "stage_ms": stage,
            "gpu_equals_oracle_plain": same(g_plain, o_plain), "gpu_equals_oracle_refine10": same(g_ref, o_ref),
            "recall_at_k": recall_of(g_plain[0], gt, k), "recall_at_k_refine10": recall_of(g_ref[0], gt, k),
            "recall_at_k_cpu": recall_of(o_plain[0], gt, k), "recall_at_k_refine10_cpu": recall_of(o_ref[0], gt, k),
            "partition_size_std_over_mean": float(sizes.std() / sizes.mean()), "index_build_s": build_s,
            "cpu_qps": cpu["value"], "cpu_threads": cpu["cores"],
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs,
                         "kernel_ms": stage["scan"], "algorithmic_bytes_per_launch": code_bytes,
                         "note": ("algorithmic bytes count a partition's codes once per query that probes it; the kernel "
                                  "reads them from HBM once per tile of <= 8 queries, so a value above 1.0 is on-chip "
                                  "reuse (large partitions: many queries per tile), not more than the HBM peak")},
            "filter_stats": fstats}


def sharded_block(torch, dist, _native, oracle, cfg, full_ix, gpu_full, rank, local, world, flush, peak_gbs, steps=20):
    """Config 2 split `world` ways by partition, ONE shared batch per step (strong scaling), through
    lgpu_search_sharded_device.  Gate (rank 0): ids / distance bits / counts equal the single-GPU search of the
    full index on the same batch, plus an 8-query oracle spot check."""
    from lancedb_b200.distributed import exchange_unique_id
    device = f"cuda:{local}"
    B, k, dim = cfg["batch"], cfg["k"], cfg["dim"]
    shard = _native.GpuIvfPq(full_ix.shard(rank, world), device=local, with_vectors=False)
    comm = _native.Comm(exchange_unique_id(), rank, world, local)
    nb = 4
    dq = synth_vectors(cfg, nb * B, 977, device).reshape(nb, B, dim)          # identical on every rank
    oi = torch.empty(B, k, dtype=torch.int64, device=device); od = torch.empty(B, k, device=device)
    oc = torch.empty(B, dtype=torch.int32, device=device)
    p = _native.make_params(k=k, nprobes=cfg["nprobes"])
    st = torch.cuda.current_stream().cuda_stream
    fn = lambda i: comm.search_device(shard, dq[i % nb].data_ptr(), B, p, oi.data_ptr(), od.data_ptr(), oc.data_ptr(), st)
    # parity gate
    fn(0)
    torch.cuda.synchronize()
    got = (oi.cpu().numpy().view(np.uint64).copy(), od.cpu().numpy().copy(), oc.cpu().numpy().view(np.uint32).copy())
    gpu_full.search_device(dq[0].data_ptr(), B, p, oi.data_ptr(), od.data_ptr(), oc.data_ptr(), st)
    torch.cuda.synchronize()
    single = (oi.cpu().numpy().view(np.uint64).copy(), od.cpu().numpy().copy(), oc.cpu().numpy().view(np.uint32).copy())
    parity_single = same(got, single)
    parity_oracle = None
    if rank == 0:
        threads, _ = host_threads()
        full_ix.vectors = None
        want = oracle.OracleIndex.from_data(full_ix).search(dq[0, :8].cpu().numpy(), k=k, nprobes=cfg["nprobes"], nthreads=threads)
        parity_oracle = same((got[0][:8], got[1][:8], got[2][:8]), want)
    flag = torch.tensor([1 if parity_single else 0], device=device)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    for i in range(3):
        fn(i)
    dist.barrier(); torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for i in range(steps):
        flush.zero_()
        ev[i][0].record(); fn(i); ev[i][1].record()
    dist.barrier(); torch.cuda.synchronize()
    tot = torch.tensor([sum(a.elapsed_time(b) for a, b in ev)], dtype=torch.float64, device=device)
    dist.all_reduce(tot, op=dist.ReduceOp.MAX)
    ms = float(tot.item()) / steps
    _native.set_profiling(True)
    fn(0)
    cm = comm.last_stage_ms(); stg = _native.last_stage_ms()
    _native.set_profiling(False)
    dist.barrier()
    comm.close(); shard.close()
    return {"workload": "BASELINE.json configs[1] partition-sharded over %d GPUs, one shared batch of %d" % (world, B),
            "scaling": "strong", "qps": B / (ms / 1e3), "ms": ms, "steps": steps,
            "local_search_ms": cm["local_search"], "coarse_ms": stg["coarse"] + stg["select_probes"],
            "scan_ms": stg["scan"], "allgather_ms": cm["allgather"], "merge_ms": cm["merge"],
            "allgather_bytes_per_rank": B * k * 16, "collective": "one ncclAllGather of [B][k] 16-byte records (in-library)",
            "parity": bool(flag.item() == 1), "parity_vs": "single-GPU search of the full index, same batch, every rank "
            "(ids, distance bits, counts)", "oracle_check": parity_oracle, "oracle_check_queries": 8}


def c5_block(torch, dist, _native, oracle, rank, local, world, flush, peak_gbs, steps=5, seed=23):
    """BASELINE configs[4] shape: nlist 16384, m 96, 12.2M rows PER GPU (the true 100M x 768 index at N = 8),
    partitions sharded across the ranks, batch 8192, nprobes 20 / k 10 (north_star defaults; BASELINE.json
    does not state them), one ncclAllGather of per-rank top-k.  Oracle check on rank 0 over the partitions the
    checked queries probe (regenerated from their seeds)."""
    from lancedb_b200.distributed import exchange_unique_id
    from lancedb_b200.index import assign_partitions
    device = f"cuda:{local}"
    nlist, m, dim, B, k, nprobes = 16384, 96, 768, 8192, 10, 20
    n_total = 12_207_031 * world
    rng = np.random.default_rng(seed)
    base = n_total // nlist
    sizes = rng.integers(int(base * 0.7), int(base * 1.3) + 1, nlist).astype(np.int64)   # same draw as the builder
    owner = assign_partitions(sizes, world)
    t0 = time.time()
    ixs, sizes2, goff = synthetic_uniform_index(n_total, dim, nlist, m, "l2", seed, owner=owner, rank=rank)
    assert np.array_equal(sizes, sizes2)
    gen_s = time.time() - t0
    shard = _native.GpuIvfPq(ixs, device=local, with_vectors=False)
    comm = _native.Comm(exchange_unique_id(), rank, world, local)
    g = torch.Generator(device="cuda").manual_seed(99)
    dq = torch.randn(2, B, dim, generator=g, device=device)                  # identical on every rank
    oi = torch.empty(B, k, dtype=torch.int64, device=device); od = torch.empty(B, k, device=device)
    oc = torch.empty(B, dtype=torch.int32, device=device)
    p = _native.make_params(k=k, nprobes=nprobes)
    st = torch.cuda.current_stream().cuda_stream
    fn = lambda i: comm.search_device(shard, dq[i % 2].data_ptr(), B, p, oi.data_ptr(), od.data_ptr(), oc.data_ptr(), st)
    for i in range(2):
        fn(i)
    dist.barrier(); torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for i in range(steps):
        flush.zero_()
        ev[i][0].record(); fn(i); ev[i][1].record()
    dist.barrier(); torch.cuda.synchronize()
    tot = torch.tensor([sum(a.elapsed_time(b) for a, b in ev)], dtype=torch.float64, device=device)
    dist.all_reduce(tot, op=dist.ReduceOp.MAX)
    ms = float(tot.item()) / steps
    _native.set_profiling(True)
    fn(0)
    cm = comm.last_stage_ms(); stg = _native.last_stage_ms(); code_bytes = _native.last_scanned_code_bytes()
    _native.set_profiling(False)
    got = (oi.cpu().numpy().view(np.uint64)[:4].copy(), od.cpu().numpy()[:4].copy(), oc.cpu().numpy().view(np.uint32)[:4].copy())
    check = None
    if rank == 0:
        threads, _ = host_threads()
        q4 = dq[0, :4].cpu().numpy()
        probe_orc = oracle.OracleIndex.from_data(sparse_oracle_index(ixs, sizes, goff, [], seed))
        parts = sorted({int(x) for qq in q4 for x in probe_orc.find_partitions(qq, nprobes)[0]})
        sp = sparse_oracle_index(ixs, sizes, goff, parts, seed)
        want = oracle.OracleIndex.from_data(sp).search(q4, k=k, nprobes=nprobes, nthreads=threads)
        check = same(got, want)
    cb = torch.tensor([float(code_bytes)], dtype=torch.float64, device=device)
    dist.all_reduce(cb, op=dist.ReduceOp.SUM)
    dist.barrier()
    comm.close(); shard.close()
    agg = float(cb.item()) / (stg["scan"] / 1e3) / 1e9
    return {"workload": f"{n_total}x{dim} f32, IVF_PQ nlist={nlist} m={m}, nprobes={nprobes}, k={k}, batch={B}, l2; "
                        f"{world} partition shards of ~12.2M rows (BASELINE.json configs[4] is N = 8); synthetic uniform "
                        "partitions, random codes",
            "is_true_config5": world == 8, "qps": B / (ms / 1e3), "ms": ms, "steps": steps,
            "local_search_ms": cm["local_search"], "coarse_ms": stg["coarse"] + stg["select_probes"], "scan_ms": stg["scan"],
            "topk_ms": stg["topk"], "allgather_ms": cm["allgather"], "merge_ms": cm["merge"],
            "allgather_bytes_per_rank": B * k * 16, "oracle_check": check, "oracle_check_queries": 4,
            "rows_per_gpu": int(ixs.nrows), "index_generate_s": gen_s,
            "roofline": {"bound": "hbm", "achieved": agg, "peak": peak_gbs * world, "unit": "GB/s (all ranks)",
                         "frac": agg / (peak_gbs * world), "note": "all ranks' scanned code bytes / rank 0's scan kernel time"}}


if __name__ == "__main__":
    main()
