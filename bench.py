#!/usr/bin/env python
"""bench.py — HNSW k-NN queries/sec on synthetic f32 vectors (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

A step = one pass of the hot path (batched hnsw_knn) over one batch of B queries.

Workloads (SURVEY.md §8d):
  config2   (default) BASELINE configs[1]: 1M x 768 f32 per GPU, ef=200, k=10, batch 4096, index m=16 /
            ef_construction=200.  At N>1 (torchrun, one rank per GPU) every rank owns one 1M-vector shard
            with its own graph ("weak": per-GPU work fixed), the query batch is replicated and the sharded
            operator runs through the C ABI (cozo_gpu_hnsw_search_sharded[_dev]): per-shard search ->
            exchange (fused peer stores, or ONE NCCL all-gather per list with --exchange nccl) -> merge.
  config3   BASELINE configs[2]: 10M x 768, k=100, batch 65536, one GPU (roofline capture).
  config5   BASELINE configs[4]: 12.5M x 768 per GPU (100M over 8), ef=200, k=10, batch 1M tiled by 65536.
  strong10m SURVEY §8d strong-scaling series: 10M x 768 in total, split over the N GPUs, batch 65536.
  pagerank  BASELINE configs[3]: PageRank on RMAT scale 24 (separate metric, see run_pagerank).

Keys beyond the base contract: `roofline`, `cpu_baseline`, `e2e`, `clocks`, `gpu_launches`, `parity`.
Prints exactly one JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "HNSW k-NN queries/sec at recall@10"
UNIT = "queries/s"

WORKLOADS = {
    #            rows/GPU     batch     k    tile   scaling
    "config2":   (1_000_000,  4096,     10,  65536, "weak"),
    "config3":   (10_000_000, 65536,    100, 65536, "weak"),
    "config5":   (12_500_000, 1_048_576, 10, 65536, "weak"),
    "strong10m": (10_000_000, 65536,    10,  65536, "strong"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "export-graph"])
    ap.add_argument("--workload", default=os.environ.get("COZO_BENCH_WORKLOAD", "config2"),
                    choices=list(WORKLOADS) + ["pagerank"])
    # overrides for quick runs (None = the workload's value)
    ap.add_argument("--rows", dest="n", type=int, default=None)
    ap.add_argument("--dim", type=int, default=int(os.environ.get("COZO_BENCH_DIM", 768)))
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--tile", type=int, default=None)
    ap.add_argument("--ef", type=int, default=200)
    ap.add_argument("--k", type=int, default=None)
    ap.add_argument("--m", type=int, default=16)
    ap.add_argument("--efc", type=int, default=200)
    ap.add_argument("--cpu-sample", type=int, default=int(os.environ.get("COZO_BENCH_CPU_SAMPLE", 4096)))
    ap.add_argument("--ref-sample", type=int, default=int(os.environ.get("COZO_BENCH_REF_SAMPLE", 0)),
                    help="queries per step of the reference arm (0 = the GPU arm's batch)")
    ap.add_argument("--parity-sample", type=int, default=256, help="N>1: queries checked against the oracle per shard")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / oracle legs")
    ap.add_argument("--opt", action="append", default=[], help="library option name=value")
    ap.add_argument("--exchange", default=os.environ.get("COZO_BENCH_EXCHANGE", "fused"), choices=["nccl", "fused"],
                    help="N>1: one NCCL all-gather per list (north star) or peer stores fused into the search kernel")
    ap.add_argument("--also-exchange", default=None, choices=["nccl", "fused"],
                    help="N>1: time the other exchange too on the same indexes (reported under `exchange_alt`)")
    ap.add_argument("--device-gen", type=int, default=-1, help="1/0: generate the corpus in HBM / on the host (-1: HBM above 2M rows)")
    ap.add_argument("--out", default=None, help="--impl export-graph: where to write the graph")
    ap.add_argument("--scale", type=int, default=24, help="pagerank: RMAT scale")
    ap.add_argument("--watchdog-s", type=int, default=int(os.environ.get("COZO_BENCH_WATCHDOG_S", 840)),
                    help="end the process (rc 3) if the run has not finished after this many seconds: a wedged kernel "
                         "must not hold the GPU box until the caller's limit (0 = off)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float32 / float64), so that two "
                         "builds can be compared output for output on the same seeded inputs")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if a.workload in WORKLOADS:
        rows, batch, k, tile, scaling = WORKLOADS[a.workload]
        world = int(os.environ.get("WORLD_SIZE", 1))
        if a.workload == "strong10m":
            rows = rows // world
        a.n = a.n or int(os.environ.get("COZO_BENCH_N", 0)) or rows
        a.batch = a.batch or int(os.environ.get("COZO_BENCH_BATCH", 0)) or batch
        a.k = a.k or k
        a.tile = a.tile or tile
        a.scaling = scaling
    return a


def workload_name(a, n_gpus):
    s = f"{a.n}x{a.dim} f32 U[0,1) per GPU, L2, m={a.m}, ef_construction={a.efc}, ef={a.ef}, k={a.k}, batch={a.batch}"
    if a.batch > a.tile:
        s += f" (tiles of {a.tile})"
    if n_gpus > 1:
        s += f", corpus row-sharded over {n_gpus} GPUs ({a.n * n_gpus} vectors total)"
    return s


def gen_vectors(n, dim, seed):
    """i.i.d. U[0,1) f32 (the law of rand_vec, data/functions.rs:2154), generated in chunks."""
    rng = np.random.default_rng(seed)
    out = np.empty((n, dim), np.float32)
    step = max(1, (1 << 26) // dim)
    for i in range(0, n, step):
        rng.random(out=out[i:i + step], dtype=np.float32)
    return out


def gen_vectors_dev(n, dim, seed, dev):
    """the same law generated on the device (12.5M x 768 = 38 GB per shard never exists on the host)"""
    import torch
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    out = torch.empty((n, dim), dtype=torch.float32, device=dev)
    step = max(1, (1 << 28) // dim)
    for i in range(0, n, step):
        out[i:i + step].uniform_(0.0, 1.0, generator=gen)
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for t, line in self.rows:
            if t < t0 - 0.05 or t > t1 + 0.15:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(key="hnsw_search_bytes_per_launch"):
    """dram bytes per launch of the dominant kernel from the committed ncu capture (not measurable inside
    an un-profiled run); None when the capture does not cover this workload."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p)).get(key)
    except Exception:
        return None


def host_cores() -> int:
    """threads the CPU arms may use: the affinity mask, capped by a cgroup CPU quota if one is set"""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                quota, period = txt[0], float(txt[1])
            else:
                quota, period = txt[0], float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota not in ("max", "-1") and period > 0:
                n = max(1, min(n, int(-(-float(quota) // period))))
            break
        except (OSError, ValueError, IndexError):
            continue
    return n


def mem_available_bytes() -> int:
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 0


DUMP_BYTES = 64 * 10**6


def dump_outputs(out_dir, arrays):
    """--dump-outputs: one DIR/<name>.npy per array (all share their first axis).  Integer ids are written as float64,
    which holds them exactly.  When the arrays exceed 64 MB in all, the same seeded sample of rows is kept of each,
    and the sampled row numbers go to DIR/sample_rows.npy."""
    arrays = {k: np.asarray(v, np.float32 if np.asarray(v).dtype == np.float32 else np.float64) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(v.nbytes for v in arrays.values()) // n
    if n * row_bytes > DUMP_BYTES:
        keep = (DUMP_BYTES - 4096) // (row_bytes + 8)
        rows = np.sort(np.random.default_rng(0x5EED0005).choice(n, keep, replace=False))
        arrays = {k: v[rows] for k, v in arrays.items()}
        arrays["sample_rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), v)


def recall_rows(a_ids, b_ids, k):
    return float(np.mean([len(set(x.tolist()) & set(y.tolist())) / k for x, y in zip(a_ids, b_ids)]))


def save_levels(path, levels):
    ni, rp, ci, ep = levels
    d = {"n_levels": np.array(len(rp)), "entry": np.array(-1 if ep is None else ep, np.int64)}
    for i in range(len(rp)):
        d[f"rp{i}"] = rp[i]
        d[f"ci{i}"] = ci[i]
        if i:
            d[f"ni{i}"] = ni[i]
    np.savez(path, **d)


def load_levels(path):
    z = np.load(path)
    nl = int(z["n_levels"])
    ep = int(z["entry"])
    return ([None] + [z[f"ni{i}"] for i in range(1, nl)], [z[f"rp{i}"] for i in range(nl)],
            [z[f"ci{i}"] for i in range(nl)], None if ep < 0 else ep)


def export_graph(a):
    """--impl export-graph: build the configs[1] graph with the device builder and write it to --out.
    Run as a SEPARATE process by the reference arm, so that the process that times the CPU search never
    maps libcozo_gpu.so (the oracle's own sequential builder would need ~a day for 1M x 768)."""
    from cozo_b200 import capi
    capi.init(0)
    X = gen_vectors(a.n, a.dim, 0x5EED0001)
    g = capi.HnswIndex.build(X, m=a.m, ef_construction=a.efc, level_seed=0x5EED0003)
    save_levels(a.out, g.export_levels())
    g.close()


def run_reference(a, rank, world):
    """--impl reference: the reference's CPU algorithm (oracle port: the Rust crate cannot be built in this
    image) on the host cores, same config, same number of queries per step as the GPU arm."""
    if rank != 0:
        return
    if a.workload == "pagerank":
        return run_pagerank_reference(a)
    cores = host_cores()
    t0 = time.perf_counter()
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "graph.npz")
        subprocess.check_call([sys.executable, os.path.abspath(__file__), "--impl", "export-graph", "--out", path,
                               "--rows", str(a.n), "--dim", str(a.dim), "--m", str(a.m), "--efc", str(a.efc)],
                              env={**os.environ, "WORLD_SIZE": "1", "RANK": "0", "LOCAL_RANK": "0"})
        levels = load_levels(path)
    build_s = time.perf_counter() - t0
    assert "cozo_b200.capi" not in sys.modules      # this process never loads the GPU library
    X = gen_vectors(a.n, a.dim, 0x5EED0001)
    from oracle import oracle as O
    ix = O.OracleHnsw.from_levels(X, O.HnswLevels(*levels))
    sample = min(a.ref_sample or a.batch, a.batch)
    times = []
    for s in range(a.warmup + a.steps):
        Q = gen_vectors(sample, a.dim, 0x5EED0002 + s)
        t0 = time.perf_counter()
        ix.search(Q, a.k, a.ef, n_threads=cores)
        if s >= a.warmup:
            times.append(time.perf_counter() - t0)
    tot = sum(times)
    qps = sample * a.steps / tot
    line = {
        "impl": "reference", "metric": METRIC, "value": qps, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * tot / a.steps, "higher_is_better": True, "scaling": a.scaling,
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(a, 1), "queries_per_step": sample, "host_cores": cores,
                   "note": "graph built by the device builder in a separate process "
                           f"({build_s:.1f}s, not timed), searched here on the CPU by the oracle port of hnsw_knn"},
        "cpu_baseline": {"value": qps, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{sample} queries per step x {a.steps} steps, {cores} threads (one query per "
                                   "thread at a time == N concurrent read transactions)"},
        "e2e": {"value": qps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# PageRank workload (BASELINE configs[3]) — its own metric; `bench.py --workload pagerank`
PR_METRIC = "PageRank edge traversals/sec on RMAT (reference defaults: theta 0.85, 10 iterations)"


def rmat_numpy(scale, ef, seed, a=0.57, b=0.19, c=0.19):
    from tests.util import rmat_edges
    return rmat_edges(scale, ef, seed, a, b, c)


def run_pagerank_reference(a):
    from oracle import oracle as O
    cores = host_cores()
    n, src, dst = rmat_numpy(a.scale, 16, 0x5EED0004)
    m = int(src.size)
    times = []
    for s in range(min(a.warmup, 1) + min(a.steps, 3)):
        t0 = time.perf_counter()
        og = O.OracleGraph(n, src, dst)
        sc, it, err = og.pagerank(0.85, 0.0, 10, n_threads=cores)
        if s >= min(a.warmup, 1):
            times.append(time.perf_counter() - t0)
    tot = sum(times)
    val = m * 10 * len(times) / tot
    print(json.dumps({
        "impl": "reference", "metric": PR_METRIC, "value": val, "unit": "edges/s", "n_gpus": 1, "steps": len(times),
        "warmup": min(a.warmup, 1), "ms_per_step": 1e3 * tot / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"RMAT scale {a.scale} edge factor 16: n={n} m={m}, 10 iterations", "host_cores": cores},
        "cpu_baseline": {"value": val, "unit": "edges/s", "cores": cores, "kind": "port",
                         "sample": "CSR build + 10 pull iterations per step (what PageRank::run does per call)"},
        "e2e": {"value": val, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


def run_pagerank(a):
    """one step = one FixedRule call: 10 pull iterations (epsilon = 0 keeps all ten) on the staged CSR.
    value: edge traversals/s over the iterations (device-timed inside cozo_gpu_pagerank, graph resident);
    e2e:   the host-API sequence of PageRank::run: stage the edge list (H2D + CSR build) + iterate + D2H scores."""
    import torch
    from cozo_b200 import capi
    capi.init(0)
    for o in a.opt:
        name, val = o.split("=")
        capi.set_option(name, int(val))
    from tools.bench_pagerank import rmat_torch
    t0 = time.perf_counter()
    n, src, dst = rmat_torch(a.scale, 16, 0x5EED0004)
    gen_s = time.perf_counter() - t0
    m = int(src.size)
    t0 = time.perf_counter()
    g = capi.Graph(n, src, dst)
    stage_s = time.perf_counter() - t0
    iters = 10
    sampler = ClockSampler(0)
    sampler.start()
    for _ in range(max(a.warmup, 3)):
        g.pagerank(0.85, 0.0, iters)
    t_start = time.perf_counter()
    kms = []
    for _ in range(a.steps):
        scores, it, err, ms = g.pagerank(0.85, 0.0, iters)
        assert it == iters
        kms.append(ms)
    t_end = time.perf_counter()
    clocks = sampler.stop(t_start, t_end)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"scores": scores})
    tot_ms = sum(kms)
    value = m * iters * a.steps / (tot_ms / 1e3)
    bytes_iter = 8 * m + 20 * n
    peak, peak_src = peak_hbm()
    achieved = bytes_iter * iters * a.steps / (tot_ms / 1e3) / 1e9
    # e2e: stage + run + scores back, wall clock, twice
    e2e_t = []
    for _ in range(2):
        t0 = time.perf_counter()
        g2 = capi.Graph(n, src, dst)
        sc2, _, _, _ = g2.pagerank(0.85, 0.0, iters)
        e2e_t.append(time.perf_counter() - t0)
        g2.close()
    cpu = None
    if not a.no_cpu:
        from oracle import oracle as O
        cores = host_cores()
        t0 = time.perf_counter()
        og = O.OracleGraph(n, src, dst)
        build_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        os_, oit, _ = og.pagerank(0.85, 0.0, iters, n_threads=cores)
        it_s = time.perf_counter() - t0
        rel = np.abs(scores - os_) / os_
        cpu = {"value": m * iters / it_s, "unit": "edges/s", "cores": cores, "kind": "port",
               "sample": f"10 iterations of the oracle pull loop on {cores} threads ({it_s:.2f}s) after a "
                         f"{build_s:.1f}s CSR build", "max_rel_err_gpu_vs_oracle": float(rel.max()),
               "p999_rel_err": float(np.quantile(rel[::16], 0.999))}
    print(json.dumps({
        "metric": PR_METRIC, "value": value, "unit": "edges/s", "n_gpus": 1, "steps": a.steps, "warmup": max(a.warmup, 3),
        "ms_per_step": tot_ms / a.steps, "ms_per_iteration": tot_ms / a.steps / iters, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"RMAT scale {a.scale} edge factor 16 (a,b,c = .57,.19,.19), ids permuted: n={n} m={m}, "
                               "theta 0.85, 10 iterations", "l2_policy": "inputs larger than L2 (CSR 1.1 GB + vectors)",
                   "gen_s": round(gen_s, 2), "stage_s": round(stage_s, 2),
                   "options": {o.split("=")[0]: int(o.split("=")[1]) for o in a.opt}},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": ncu_traffic("pagerank_bytes_per_iteration"), "kernel": "pagerank iteration (all launches)",
                     "algorithmic_bytes_per_iteration": bytes_iter, "peak_source": peak_src},
        "cpu_baseline": cpu,
        "e2e": {"value": m * iters / min(e2e_t), "unit": "edges/s", "h2d_bytes_per_step": 8 * m,
                "d2h_bytes_per_step": 4 * n, "seconds_per_call": min(e2e_t)},
        "clocks": clocks, "gpu_launches": int(capi.get_option("pagerank.last_launches")) * a.steps}), flush=True)


# ---------------------------------------------------------------------------------------------------
def arm_watchdog(seconds):
    """A daemon thread that ends the process even when the main thread sits inside a CUDA call."""
    if seconds <= 0:
        return
    import threading

    def fire():
        sys.stderr.write(f"bench.py: watchdog: not finished after {seconds} s, exiting (rc 3)\n")
        sys.stderr.flush()
        os._exit(3)
    t = threading.Timer(seconds, fire)
    t.daemon = True
    t.start()


def main():
    a = parse()
    if a.impl == "ours":
        arm_watchdog(a.watchdog_s)
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if a.impl == "export-graph":
        return export_graph(a)
    if a.impl == "reference":
        return run_reference(a, rank, world)
    if a.workload == "pagerank":
        if rank == 0:
            run_pagerank(a)
        return
    import torch
    from cozo_b200 import capi
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback for the hot path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    capi.init(local_rank)
    capi.set_option("shard.exchange", 1 if a.exchange == "fused" else 0)
    capi.set_option("shard.tile", a.tile)
    for o in a.opt:
        name, val = o.split("=")
        capi.set_option(name, int(val))

    # ---- corpus shard + index on this GPU -----------------------------------------------
    on_device = a.n > 2_000_000 if a.device_gen < 0 else bool(a.device_gen)   # big shards are generated in HBM (38 GB at config 5)
    t0 = time.perf_counter()
    if on_device:
        Xd = gen_vectors_dev(a.n, a.dim, 0x5EED0001 + 1000 * rank, dev)
        torch.cuda.synchronize()
        X = None
    else:
        X = gen_vectors(a.n, a.dim, 0x5EED0001 + 1000 * rank)
    gen_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    if on_device:
        g = capi.HnswIndex.build(None, m=a.m, ef_construction=a.efc, level_seed=0x5EED0003 + rank,
                                 vectors_dev_ptr=Xd.data_ptr(), n_vectors=a.n, dim=a.dim, borrow=True)
    else:
        g = capi.HnswIndex.build(X, m=a.m, ef_construction=a.efc, level_seed=0x5EED0003 + rank)
    build_s = time.perf_counter() - t0
    B, k, ef, dim = a.batch, a.k, a.ef, a.dim
    nsteps = a.warmup + a.steps
    # query batches resident in HBM before the timed region; distinct per step while they fit 8 GB
    nsets = max(1, min(nsteps, (8 << 30) // (B * dim * 4)))
    if B * dim * 4 * nsets <= (1 << 30):
        Qh = gen_vectors(B * nsets, dim, 0x5EED0002).reshape(nsets, B, dim)
        Qd = torch.from_numpy(Qh).to(dev)
    else:
        Qd = gen_vectors_dev(B * nsets, dim, 0x5EED0002, dev).view(nsets, B, dim)
        Qh = None
    qstats = torch.zeros((nsteps, B, 4), dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    grp = None
    if world > 1:
        import torch.distributed as dist
        uid = [capi.ShardGroup.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        grp = capi.ShardGroup(uid[0], rank, world)
        grp.attach(g)
        out_i = torch.empty((B, k), dtype=torch.int64, device=dev)
        out_d = torch.empty((B, k), dtype=torch.float32, device=dev)
    else:
        ids = torch.empty((B, k), dtype=torch.int32, device=dev)
        dd = torch.empty((B, k), dtype=torch.float32, device=dev)

    def step(s):
        q = Qd[s % nsets]
        if grp is None:
            g.search_dev(q.data_ptr(), B, k, ef, ids.data_ptr(), dd.data_ptr(), None, qstats[s].data_ptr(), stream)
        else:   # the sharded operator of the C ABI: local search -> exchange -> merge, tile by tile
            grp.search_dev(q.data_ptr(), B, k, ef, out_i.data_ptr(), out_d.data_ptr(), qstats[s].data_ptr(), stream)

    sampler = ClockSampler(local_rank)
    sampler.start()          # nvidia-smi needs a moment to start: launch it before the warm-up
    for s in range(a.warmup):
        step(s)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    time.sleep(0.3)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    torch.cuda.synchronize()
    t_start = time.perf_counter()
    e_all0 = torch.cuda.Event(enable_timing=True)
    e_all1 = torch.cuda.Event(enable_timing=True)
    e_all0.record()
    for i in range(a.steps):
        evs[i][0].record()
        step(a.warmup + i)
        evs[i][1].record()
    e_all1.record()
    torch.cuda.synchronize()
    t_end = time.perf_counter()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop(t_start, t_end)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, {"ids": (ids if grp is None else out_i).cpu().numpy(),
                                      "distances": (dd if grp is None else out_d).cpu().numpy()})
    total_ms = e_all0.elapsed_time(e_all1)
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    step_ms = [e0.elapsed_time(e1) for e0, e1 in evs]
    # whole-job units.  weak: every rank searched B queries against its shard (per-shard searches);
    # strong: the job is B queries over the fixed corpus
    units = B * a.steps * (world if a.scaling == "weak" else 1)
    value = units / (total_ms / 1e3)

    # ---- the other exchange on the same shards (optional) ----------------------------------------------
    exchange_alt = None
    if grp is not None and a.also_exchange:
        capi.set_option("shard.exchange", 1 if a.also_exchange == "fused" else 0)
        uid2 = [capi.ShardGroup.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid2, src=0)
        grp2 = capi.ShardGroup(uid2[0], rank, world)
        grp2.attach(g)
        for s_ in range(min(a.warmup, 2)):
            grp2.search_dev(Qd[s_ % nsets].data_ptr(), B, k, ef, out_i.data_ptr(), out_d.data_ptr(), None, stream)
        torch.cuda.synchronize()
        dist.barrier()
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ea.record()
        for i in range(a.steps):
            grp2.search_dev(Qd[(a.warmup + i) % nsets].data_ptr(), B, k, ef, out_i.data_ptr(), out_d.data_ptr(), None, stream)
        eb.record()
        torch.cuda.synchronize()
        t2 = torch.tensor([ea.elapsed_time(eb)], dtype=torch.float64, device=dev)
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        exchange_alt = {"exchange": grp2.info()["exchange"], "ms_per_step": float(t2.item()) / a.steps,
                        "value": B * a.steps * (world if a.scaling == "weak" else 1) / (float(t2.item()) / 1e3)}
        grp2.close()
        capi.set_option("shard.exchange", 1 if a.exchange == "fused" else 0)

    # ---- roofline of the dominant kernel (hnsw_search_kernel) ---------------------------
    st = qstats[a.warmup:].to(torch.int64).sum(dim=(0, 1)).cpu().numpy()
    dist_evals, expanded, nbr_reads = int(st[0]), int(st[1]), int(st[2])
    alg_bytes_per_step = (dist_evals * dim * 4 + expanded * 8 + nbr_reads * 4 + a.steps * B * dim * 4) / a.steps
    # kernel duration: the search kernel alone (at N=1 and B <= tile a step is just that launch)
    kern_ms = statistics.mean(step_ms) if world == 1 else None
    if world > 1:
        lids = torch.empty((B, k), dtype=torch.int32, device=dev)
        ldd = torch.empty((B, k), dtype=torch.float32, device=dev)
        tmp = []
        for i in range(min(a.steps, 5)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g.search_dev(Qd[(a.warmup + i) % nsets].data_ptr(), B, k, ef, lids.data_ptr(), ldd.data_ptr(), None, None, stream)
            e1.record()
            torch.cuda.synchronize()
            tmp.append(e0.elapsed_time(e1))
        kern_ms = statistics.mean(tmp)
    peak, peak_src = peak_hbm()
    achieved = alg_bytes_per_step / (kern_ms / 1e3) / 1e9
    tiles = -(-B // a.tile)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": ncu_traffic() if a.workload == "config2" else None,
                "traffic_source": "profiles/traffic.json (ncu --set full capture of this kernel at this workload; "
                                  "not re-measured in this run)" if a.workload == "config2" else None,
                "kernel": "hnsw_search_kernel", "kernel_ms": kern_ms,
                "algorithmic_bytes_per_launch": alg_bytes_per_step / (tiles if world > 1 else 1),
                "launches_per_step": tiles if world > 1 else 1, "peak_source": peak_src,
                "dist_evals_per_query": dist_evals / (a.steps * B), "nodes_expanded_per_query": expanded / (a.steps * B)}

    # ---- e2e: the reference-facing C-ABI call with HOST buffers (pinned), copies inside ----
    # N=1: cozo_gpu_hnsw_search; N>1: cozo_gpu_hnsw_search_sharded, the same path as `value`
    e2e_steps = a.steps if B * dim * 4 <= (1 << 30) else min(a.steps, 2)
    e2e_warm = min(a.warmup, 2)
    hq = (torch.from_numpy(Qh) if Qh is not None else Qd[:1].cpu()).pin_memory()
    e2e_times = []
    for s in range(e2e_warm + e2e_steps):
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        if grp is None:
            hi, hd, hc, hst = g.search(hq[s % hq.shape[0]].numpy(), k, ef)
        else:
            hi, hd, hc, hst = grp.search(hq[s % hq.shape[0]].numpy(), k, ef, root=-1)
        dt = time.perf_counter() - t0
        if s >= e2e_warm:
            e2e_times.append(dt)
    e2e_s = sum(e2e_times)
    if world > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e = {"value": B * e2e_steps * (world if a.scaling == "weak" else 1) / e2e_s, "unit": UNIT,
           "h2d_bytes_per_step": B * dim * 4, "d2h_bytes_per_step": B * k * (12 if world > 1 else 8) + B * 16,
           "steps": e2e_steps,
           "call": "cozo_gpu_hnsw_search" if world == 1 else "cozo_gpu_hnsw_search_sharded (every rank passes the batch)"}

    # ---- parity vs the CPU oracle on the same graph(s) + cpu_baseline --------------------------------
    cpu_baseline = None
    recall_vs_oracle = None
    parity = None
    if not a.no_cpu:
        from oracle import oracle as O
        cores = host_cores()
        s_last = (a.warmup + a.steps - 1) % nsets
        if world == 1:
            if rank == 0:
                Xh = X if X is not None else Xd.cpu().numpy()
                levels = g.export_levels()
                sample = min(a.cpu_sample, B)
                Qs = (Qh[s_last][:sample] if Qh is not None else Qd[s_last][:sample].cpu().numpy())
                ix = O.OracleHnsw.from_levels(Xh, O.HnswLevels(*levels))
                t0 = time.perf_counter()
                oids, odist, ocnt, ost = ix.search(Qs, k, ef, n_threads=cores)
                qps = len(Qs) / (time.perf_counter() - t0)
                hi, hd, _, hst = g.search(Qs, k, ef)
                recall_vs_oracle = recall_rows(hi, oids, k)
                parity = {"queries": int(sample), "recall_at_k": recall_vs_oracle,
                          "identical_id_sets": float(np.mean([set(x.tolist()) == set(y.tolist()) for x, y in zip(hi, oids)])),
                          "dist_evals": {"gpu": int(hst.dist_evals), "oracle": int(ost[:, 0].sum())},
                          "nodes_expanded": {"gpu": int(hst.nodes_expanded), "oracle": int(ost[:, 1].sum())},
                          "traversal_counters_rel_diff": abs(int(hst.dist_evals) - int(ost[:, 0].sum())) / max(1, int(ost[:, 0].sum()))}
                cpu_baseline = {"value": qps, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"{sample} queries of the last timed batch, {cores} threads, oracle port of "
                                          "hnsw_knn on the exported graph (flat CSR + flat vectors: faster than real Cozo)"}
        else:
            # every rank: its shard's lists vs the oracle on ITS exported graph; rank 0: the operator's merged
            # result vs a numpy merge of the gathered per-shard lists (GPU lists and oracle lists)
            sample = min(a.parity_sample, B)
            Qs = (Qh[s_last][:sample] if Qh is not None else Qd[s_last][:sample].cpu().numpy())
            shard_bytes = a.n * dim * 4 + a.n * 40 * 4
            avail = mem_available_bytes()
            group = world if avail == 0 else max(1, min(world, int(0.6 * avail // max(shard_bytes, 1))))
            per, perr = None, None
            for g0 in range(0, world, group):
                if g0 <= rank < g0 + group:
                    try:      # a failure here must not desynchronise the ranks: the collectives below always run
                        Xh = X if X is not None else Xd.cpu().numpy()
                        levels = g.export_levels()
                        ix = O.OracleHnsw.from_levels(Xh, O.HnswLevels(*levels))
                        oi, od, _, ost = ix.search(Qs, k, ef, n_threads=max(1, cores // min(group, world)))
                        li, ld, _, lst = g.search(Qs, k, ef)
                        per = (li, ld, oi, od, int(lst.dist_evals), int(ost[:, 0].sum()))
                        del ix, Xh, levels
                    except Exception as e:          # noqa: BLE001
                        perr = repr(e)
                dist.barrier()
            mi, md, mc, _ = grp.search(Qs, k, ef, root=-1)
            gathered = [None] * world
            dist.all_gather_object(gathered, (per, perr))
            if rank == 0:
                try:
                    if any(p[0] is None for p in gathered):
                        raise RuntimeError("; ".join(str(p[1]) for p in gathered if p[1]))
                    gathered = [p[0] for p in gathered]
                    from cozo_b200.sharded import merge_lists as numpy_merge
                    offsets = np.arange(world, dtype=np.int64) * a.n
                    g_i, g_d = numpy_merge(np.stack([p[0] for p in gathered]), np.stack([p[1] for p in gathered]), offsets, k)
                    o_i, o_d = numpy_merge(np.stack([p[2] for p in gathered]), np.stack([p[3] for p in gathered]), offsets, k)
                    recall_vs_oracle = recall_rows(mi, o_i, k)
                    parity = {"queries_per_shard": int(sample),
                              "per_shard_recall_vs_oracle": [recall_rows(p[0], p[2], k) for p in gathered],
                              "per_shard_dist_evals": [{"gpu": p[4], "oracle": p[5]} for p in gathered],
                              "merged_equals_numpy_merge_of_gpu_lists": bool(np.array_equal(mi, g_i) and np.array_equal(md, g_d)),
                              "merged_recall_vs_merged_oracle": recall_vs_oracle,
                              "oracle_ranks_at_a_time": int(group)}
                except Exception as e:              # noqa: BLE001
                    parity = {"error": repr(e)}

    if rank == 0:
        info = grp.info() if grp is not None else None
        per_tile = 1 + 1 + (1 if (info and info["exchange"] == "fused") else 0)   # search, merge, (flag barrier)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": total_ms / a.steps, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(a, world), "name": a.workload, "l2_policy": "inputs larger than L2 (corpus "
                       f"{a.n * a.dim * 4 / 1e9:.2f} GB/GPU >> 126 MB), {nsets} distinct query batch(es) cycled per step",
                       "value_counts": ("per-shard k-NN searches per second summed over ranks (== queries/s at N=1); "
                                        "global queries/s over the whole sharded corpus = value / n_gpus")
                       if a.scaling == "weak" else "global queries/s over the fixed corpus",
                       "index_build_s": round(build_s, 2), "gen_s": round(gen_s, 2), "host_cores": host_cores(),
                       "options": {o.split("=")[0]: int(o.split("=")[1]) for o in a.opt}},
            "global_queries_per_s": value / world if a.scaling == "weak" else value,
            "recall_at_k_vs_oracle": recall_vs_oracle, "parity": parity,
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "clocks": clocks,
            "gpu_launches": a.steps * (1 if world == 1 else tiles * per_tile),
            "exchange": (info["exchange"] if info else None), "exchange_alt": exchange_alt,
            "step_ms": step_ms,
        }
        print(json.dumps(line), flush=True)
    if grp is not None:
        grp.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
