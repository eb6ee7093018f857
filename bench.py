#!/usr/bin/env python
"""Benchmark of the Harmony hot path (cluster() + moe_correct_ridge() to convergence).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload NAME] [--dump-outputs DIR]

Metric (BASELINE.json): cells/sec to convergence of the full Harmony loop.
A *step* = one complete run of the loop from the post-upload state: restore Z_cos, the
init assignment from given centroids (harmony.py:377-392) and harmonize() until the
reference's own convergence rule stops it (harmony.py:419-435) -- nothing skipped.
The k-means++ initialisation (sklearn, harmony.py:369-373) is outside the hot path and is
computed once, untimed, on a 100k-cell subsample; both arms start from the same centroids.

  value      whole-job cells/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e        same metric through run_harmony(...) with HOST arrays: H2D upload, layout
             sort, loop, D2H of Z_corr inside the timed region
  roofline   HBM roofline of the dominant kernel (k_round), from CUDA events recorded by
             the library around every round launch (live, this run)
  cpu_baseline  the CPU oracle (NumPy port of the reference's algorithm) on a bounded
             sample of the same workload, on this box's host cores

Workloads (BASELINE.json configs): syn1m (default; 1M cells x 50 PCs x 20 batches, K=100,
per GPU -- weak scaling), syn10m8 (10M x 50 x 50 batches over 8 GPUs => 1.25M per GPU),
syn5m8 (5M x 50, covariates 30+4, K=200 over 8 GPUs => 625k per GPU).

--dump-outputs DIR writes what the last timed step returned (see dump_outputs) so that two builds can be compared
output for output: the inputs, initial centroids included, depend only on the arguments.  The device's reductions
are not bitwise reproducible, so two runs of one build differ in the last bits (compare with a tolerance).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# The CPU arm runs BLAS / OpenMP code on hosts with > 100 cores: OpenBLAS aborts ("NUM_THREADS exceeded", rc 139 in
# round 1) when asked for more threads than it was built for, so the pools are capped BEFORE numpy / torch load.
CPU_THREADS = max(1, min(os.cpu_count() or 1, 32))
for _v in ("OPENBLAS_NUM_THREADS", "OMP_NUM_THREADS", "MKL_NUM_THREADS"):
    os.environ.setdefault(_v, str(CPU_THREADS))

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True              # the benchmark leaves the tree as it found it (it may be read-only)

WORKLOADS = {
    "syn1m": dict(per_gpu=1_000_000, d=50, levels=[20], K=100,
                  name="synthetic 1M cells x 50 PCs x 20 batches, K=100 (per GPU)"),
    "syn10m8": dict(per_gpu=1_250_000, d=50, levels=[50], K=100,
                    name="synthetic 10M cells x 50 PCs x 50 batches, K=100 over 8 GPUs (1.25M per GPU)"),
    "syn5m8": dict(per_gpu=625_000, d=50, levels=[30, 4], K=200,
                   name="synthetic 5M cells x 50 PCs, covariates 30+4, K=200 over 8 GPUs (625k per GPU)"),
    "tiny": dict(per_gpu=50_000, d=50, levels=[20], K=100, name="tiny debug workload (50k cells per GPU)"),
}
SEED = 0
INIT_SUBSAMPLE = 100_000
DUMP_SAMPLE_BYTES = 48 << 20      # --dump-outputs: Z_corr + R rows of the cell sample; the other outputs are small


def algorithmic_bytes(d, K, V):
    """SURVEY.md section 8(d): bytes per cell of one k-means round / one ridge pass."""
    return 4 * d + 8 * K + 4 * V + 4, 16 * d + 8 * K + 8 * V


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def init_centroids(w, N_total, seed=SEED):
    """k-means++ / 25 Lloyd iterations (the reference's sklearn settings, harmony.py:370-371)
    on the unit-normalised first INIT_SUBSAMPLE cells.  Untimed; identical for both arms.
    One thread: sklearn's multi-threaded Lloyd reduces its partial sums in scheduling order, so its
    centroids differ in the last bits from run to run, and with them every later result."""
    from sklearn.cluster import KMeans
    from threadpoolctl import threadpool_limits
    from harmonypy_b200.synthetic import make_synthetic_arrays
    n = min(N_total, INIT_SUBSAMPLE)
    Z, _ = make_synthetic_arrays(N_total, w["d"], w["levels"], seed=seed, lo=0, hi=n)
    Zc = Z / np.linalg.norm(Z, axis=1, keepdims=True)
    with threadpool_limits(limits=1):
        km = KMeans(n_clusters=w["K"], init="k-means++", n_init=1, max_iter=25, random_state=seed).fit(Zc)
    return km.cluster_centers_.astype(np.float32)


def global_level_probs(w, N_total, lo, hi, codes, dist=None):
    counts = np.concatenate([np.bincount(codes[v], minlength=int(b)) for v, b in enumerate(w["levels"])]).astype(np.float64)
    if dist is not None:
        import torch
        t = torch.from_numpy(counts).cuda()
        dist.all_reduce(t)
        counts = t.cpu().numpy()
    return (counts / N_total).astype(np.float32)


def make_problem(w, Z, codes, Pr_b, N_total, lo):
    from harmonypy_b200.harmony import Problem
    levels = np.asarray(w["levels"], dtype=np.int32)
    B = int(levels.sum())
    return Problem(Z=Z, codes=codes, levels=levels, level_names=[], Pr_b=Pr_b,
                   theta=np.full(B, 2, np.float32), lamb=np.concatenate([[0], np.ones(B)]).astype(np.float32),
                   lambda_estimation=False, sigma=np.full(w["K"], 0.1, np.float32), K=w["K"],
                   n_global=N_total, shard_lo=lo)


def harmony_step(ho, Y0):
    """One full run of the hot path on an engine that already holds the data."""
    ho._engine.set_option("reset", 1)
    for lst in (ho.objective_harmony, ho.objective_kmeans, ho.objective_kmeans_dist, ho.objective_kmeans_entropy,
                ho.objective_kmeans_cross, ho.kmeans_rounds):
        lst.clear()
    ho.init_cluster(SEED, Y0)
    ho.harmonize(ho.max_iter_harmony, False)
    return sum(ho.kmeans_rounds), len(ho.kmeans_rounds)


# ------------------------------------------------------------------------------------------------
def _oracle_run(w, Y0, n_sample):
    """One timed oracle run (see cpu_oracle_rate)."""
    from harmonypy_b200.synthetic import make_synthetic_arrays
    from oracle.harmony_oracle import HarmonyOracle, onehot_from_codes, torch_perm_source
    Z, codes = make_synthetic_arrays(max(n_sample, 1), w["d"], w["levels"], seed=SEED, lo=0, hi=n_sample)
    levels = np.asarray(w["levels"])
    B = int(levels.sum())
    Pr_b = np.concatenate([np.bincount(codes[v], minlength=int(b)) for v, b in enumerate(levels)]) / n_sample
    phi = onehot_from_codes(codes, levels, np.float32)
    orc = HarmonyOracle(Z.T, phi, Pr_b.astype(np.float32), np.full(w["K"], 0.1, np.float32), np.full(B, 2, np.float32),
                        np.concatenate([[0], np.ones(B)]).astype(np.float32), dtype=np.float32)
    t0 = time.perf_counter()
    orc.init_from_centroids(Y0.T)
    orc.harmonize(10, torch_perm_source(n_sample, SEED))
    dt = time.perf_counter() - t0
    return n_sample / dt, dt, dict(rounds=list(map(int, orc.kmeans_rounds)))


def load_reference():
    """The UNMODIFIED reference package staged under baseline/_ref (baseline/stage_reference.py), or None."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.exists(os.path.join(ref_dir, "harmonypy", "harmony.py")):
        return None
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    import harmonypy.harmony as rh
    return rh


def reference_run(rh, w, Y0, n_sample, threads):
    """One run of the reference's own run_harmony(device='cpu') on the first n_sample cells of the workload.
    Its sklearn k-means++ call (harmony.py:369-373) is answered with the SAME centroids our arm starts from
    (the module's KMeans name is pointed at a stub; no reference source is touched), so both arms time the same
    work: init assignment + harmonize() to the reference's own convergence rule.
    Returns (seconds of init_cluster + harmonize, seconds of the whole run_harmony call, kmeans_rounds)."""
    import pandas as pd
    import torch
    from harmonypy_b200.synthetic import make_synthetic_arrays
    torch.set_num_threads(threads)
    Z, codes = make_synthetic_arrays(max(n_sample, 1), w["d"], w["levels"], seed=SEED, lo=0, hi=n_sample)
    meta = pd.DataFrame({f"var{v}": [f"v{v}_{c:04d}" for c in codes[v]] for v in range(len(w["levels"]))})

    class GivenCentroids:                      # stands in for sklearn.cluster.KMeans inside the reference module
        def __init__(self, **kw):
            pass

        def fit(self, X):
            self.cluster_centers_ = np.asarray(Y0, dtype=np.float64)
            return self

    spans = {}
    orig_init, orig_harm, orig_km = rh.Harmony.init_cluster, rh.Harmony.harmonize, rh.KMeans

    def timed(name, fn):
        def wrap(self, *a, **k):
            t = time.perf_counter()
            r = fn(self, *a, **k)
            spans[name] = spans.get(name, 0.0) + time.perf_counter() - t
            return r
        return wrap
    rh.KMeans = GivenCentroids
    rh.Harmony.init_cluster = timed("init", orig_init)
    rh.Harmony.harmonize = timed("harmonize", orig_harm)
    try:
        t0 = time.perf_counter()
        ho = rh.run_harmony(Z, meta, list(meta.columns), nclust=w["K"], max_iter_harmony=10, max_iter_kmeans=20,
                            verbose=False, random_state=SEED, device="cpu")
        _ = ho.Z_corr
        total = time.perf_counter() - t0
    finally:
        rh.KMeans, rh.Harmony.init_cluster, rh.Harmony.harmonize = orig_km, orig_init, orig_harm
    return spans["init"] + spans["harmonize"], total, list(map(int, ho.kmeans_rounds))


def cpu_arm(w, Y0, n_sample):
    """The CPU arm: the staged reference when present (kind "reference"), else the NumPy port (kind "port").
    Returns dict(loop_seconds, total_seconds, rounds, kind, cores, sample)."""
    rh = load_reference()
    if rh is not None:
        loop, total, rounds = reference_run(rh, w, Y0, n_sample, CPU_THREADS)
        return dict(loop_seconds=loop, total_seconds=total, rounds=rounds, kind="reference", cores=CPU_THREADS,
                    sample=f"unmodified harmonypy.run_harmony(device='cpu', torch fp32, {CPU_THREADS} threads) from baseline/_ref on "
                           f"the first {n_sample} cells of the workload, same initial centroids as the GPU arm "
                           f"(its sklearn call is answered with them), init assignment + harmonize to convergence, rounds {rounds}")
    from threadpoolctl import threadpool_limits
    with threadpool_limits(limits=min(CPU_THREADS, 8)):
        rate, dt, info = _oracle_run(w, Y0, n_sample)
    return dict(loop_seconds=dt, total_seconds=dt, rounds=info["rounds"], kind="port", cores=min(CPU_THREADS, 8),
                sample=f"oracle/harmony_oracle.py (NumPy fp32 port; baseline/_ref is absent) on the first {n_sample} cells, "
                       f"init assignment + harmonize to convergence, rounds {info['rounds']}")


def workload_config(w, world, N_total, mode=None, rounds=None, iters=None):
    """The `config` object of the JSON line -- identical for both arms of one (workload, n_gpus)."""
    return {"workload": w["name"], "cells_total": N_total, "cells_per_gpu": w["per_gpu"], "d": w["d"],
            "levels": w["levels"], "K": w["K"], "parallelism": f"cells sharded over {world} GPU(s)",
            "perm_mode": "device", "l2": "inputs larger than L2 (R 400 MB + Z 600 MB per GPU), no flush",
            "init": f"sklearn k-means++ on a {min(N_total, INIT_SUBSAMPLE)}-cell subsample, untimed"}


def run_reference(args, w):
    """--impl reference: the reference's own CPU implementation on this box's host cores, on a bounded sample of the
    workload (rank 0 only; the other ranks exit without work)."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    n_sample = args.cpu_sample
    N_total = w["per_gpu"] * world
    Y0 = init_centroids(w, N_total)
    loops, totals = [], []
    for i in range(args.warmup + args.steps):
        r = cpu_arm(w, Y0, n_sample)
        if i >= args.warmup:
            loops.append(r["loop_seconds"]); totals.append(r["total_seconds"])
    ms = 1e3 * float(np.mean(loops))
    val = n_sample / (ms / 1e3)
    out = {
        "impl": "reference", "metric": "cells/sec to convergence (full Harmony loop)", "value": val,
        "unit": "cells/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(w, world, N_total),
        "cpu_baseline": {"value": val, "unit": "cells/s", "cores": r["cores"], "kind": r["kind"],
                         "host_cores": os.cpu_count(), "sample": r["sample"]},
        "e2e": {"value": n_sample / float(np.mean(totals)), "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def golden_parity(device_index, comm=None):
    """Second half of the metric: Z_corr max|d|/max|Z| vs the REFERENCE's stored output on the
    bundled datasets (fixtures under tests/golden, generated from the real harmonypy), through the
    public class with the reference permutation stream.  A few seconds.  With more than one rank the
    datasets run SHARDED over all ranks of the job (every rank calls this; same engine mode as the
    timed runs), so the line carries the parity of the N-GPU path, not of a single-GPU side run."""
    from harmonypy_b200.harmony import Harmony, Problem
    n_ranks = 1 if comm is None else comm.world
    out = {"tolerance": 1e-4, "norm": "max|Z - Z_ref| / max|Z_ref|", "n_ranks": n_ranks}
    for name, label in (("pbmc", "pbmc_3500"), ("ircolitis", "ircolitis_blood_cd8")):
        try:
            inp = np.load(os.path.join(ROOT, "tests", "golden", f"{name}_input.npz"))
            gold = np.load(os.path.join(ROOT, "tests", "golden", f"{name}_golden.npz"))
        except Exception:
            continue
        prob = Problem(Z=inp["Z"], codes=inp["codes"], levels=inp["levels"], level_names=[], Pr_b=inp["Pr_b"],
                       theta=inp["theta"], lamb=inp["lamb"], lambda_estimation=bool(inp["lambda_estimation"]),
                       sigma=inp["sigma"], K=int(inp["K"]))
        t0 = time.perf_counter()
        ho = Harmony(prob, float(inp["alpha"]), int(inp["max_iter_harmony"]), int(inp["max_iter_kmeans"]),
                     float(inp["epsilon_kmeans"]), float(inp["epsilon_harmony"]), float(inp["block_size"]), False,
                     int(inp["random_state"]), device_index, init_centroids=inp["Y0"], comm=comm)
        Zc = ho.Z_corr                      # gathered over the ranks
        dt = time.perf_counter() - t0
        ref, ref64 = gold["Zcorr_final"], gold["Zcorr_final_f64"]
        cells = gold["final_cells"]
        out[label] = {
            "vs_reference_fp32": float(np.abs(Zc[cells] - ref).max() / np.abs(ref).max()),
            "vs_reference_fp64_arbiter": float(np.abs(Zc[cells] - ref64).max() / np.abs(ref64).max()),
            "kmeans_rounds_equal": list(map(int, ho.kmeans_rounds)) == list(map(int, gold["kmeans_rounds"])),
            "cells": int(Zc.shape[0]), "seconds_incl_upload": dt, "n_ranks": n_ranks,
            "round_kernel": "k_round_tc5" if ho._engine.counter("tc5") == 1 else "k_round_mma",
            "fused_exchange": ho._engine.counter("fused") == 1,
        }
        del ho
    return out


def dump_outputs(out_dir, ho):
    """What the timed path returned in its last step, one DIR/<name>.npy each, under 64 MB in all: Z_corr and R on
    one fixed, seeded sample of this rank's cells in cell order (DUMP_SAMPLE_BYTES for the two), the centroids Y,
    O and E in full (float32); the objectives and kmeans_rounds (float64)."""
    from harmonypy_b200 import _cabi
    os.makedirs(out_dir, exist_ok=True)
    Zc = ho.result_local()
    n_local = Zc.shape[0]
    n = min(n_local, DUMP_SAMPLE_BYTES // (4 * (ho.d + ho.K)))
    cells = np.sort(np.random.default_rng(SEED).choice(n_local, n, replace=False))
    arrays = {"Z_corr": Zc[cells], "R": ho._engine.get(_cabi.R)[cells], "Y": ho.Y, "O": ho.O, "E": ho.E}
    arrays = {k: np.asarray(v, dtype=np.float32) for k, v in arrays.items()}
    for name in ("objective_harmony", "objective_kmeans", "objective_kmeans_dist", "objective_kmeans_entropy",
                 "objective_kmeans_cross", "kmeans_rounds"):
        arrays[name] = np.asarray(getattr(ho, name), dtype=np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ------------------------------------------------------------------------------------------------
def run_ours(args, w):
    import torch
    from harmonypy_b200.build import build
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if rank == 0:
        build(verbose=False)
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    from harmonypy_b200.harmony import Harmony, Comm
    from harmonypy_b200.synthetic import make_synthetic_arrays

    N_total = w["per_gpu"] * world
    lo, hi = N_total * rank // world, N_total * (rank + 1) // world
    t_setup = time.perf_counter()
    Z, codes = make_synthetic_arrays(N_total, w["d"], w["levels"], seed=SEED, lo=lo, hi=hi)
    Pr_b = global_level_probs(w, N_total, lo, hi, codes, dist)
    if rank == 0:
        Y0 = init_centroids(w, N_total)
    else:
        Y0 = np.zeros((w["K"], w["d"]), np.float32)
    comm = None
    if world > 1:
        comm = Comm(None)
        Y0 = comm.broadcast_array(Y0, 0)
    prob = make_problem(w, Z, codes, Pr_b, N_total, lo)
    opts = {"persistent": 0} if args.staged else {}
    for kv in args.engine_opt:
        k, v = kv.split("=")
        opts[k] = int(v)
    opts = opts or None
    ho = Harmony(prob, 0.2, 10, 20, 1e-5, 1e-4, 0.05, False, SEED, local_rank, perm_mode="device",
                 comm=comm, engine_options=opts, run=False)
    eng = ho._engine
    t_setup = time.perf_counter() - t_setup

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        harmony_step(ho, Y0)
    barrier()
    l0, r0, p0 = eng.counter("launches"), eng.counter("rounds"), eng.counter("ridge_passes")
    ms_round0, ms_ridge0, ms_init0 = eng.timer_ms("ms_round"), eng.timer_ms("ms_ridge"), eng.timer_ms("ms_init")
    stream = torch.cuda.default_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        barrier()
        e0.record(stream)
        tot_rounds = tot_iters = 0
        for _ in range(args.steps):
            r, it = harmony_step(ho, Y0)
            tot_rounds += r; tot_iters += it
        e1.record(stream)
        barrier()
    ms_total = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ho)
    if dist is not None:
        t = torch.tensor([ms_total], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    launches = eng.counter("launches") - l0
    n_rounds, n_ridge = eng.counter("rounds") - r0, eng.counter("ridge_passes") - p0
    ms_round = eng.timer_ms("ms_round") - ms_round0
    ms_ridge = eng.timer_ms("ms_ridge") - ms_ridge0
    ms_init = eng.timer_ms("ms_init") - ms_init0
    ms_per_step = ms_total / args.steps
    value = N_total / (ms_per_step / 1e3)

    # ---- roofline of the dominant kernel (k_round), live numbers from this run
    V = len(w["levels"])
    b_round, b_ridge = algorithmic_bytes(w["d"], w["K"], V)
    n_local = hi - lo
    peak, peak_src = measured_peak_gbs()
    ach_round = (b_round * n_local * n_rounds) / (ms_round / 1e3) / 1e9 if ms_round > 0 else 0.0
    ach_ridge = (b_ridge * n_local * n_ridge) / (ms_ridge / 1e3) / 1e9 if ms_ridge > 0 else 0.0
    tc5 = eng.counter("tc5") == 1
    traffic, traffic_source = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        ent = tj.get("k_round_tc5" if tc5 else "k_round_mma")
        if tj.get("workload") == args.workload and ent:
            traffic = ent.get("dram_bytes_per_launch")
            traffic_source = "static: %s; %s" % (ent.get("capture"), ent.get("note", ""))
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": ("k_round_tc5<NC> (tcgen05 / tensor-memory round kernel: producer warp + MMA warp + 16 epilogue warps)" if tc5 else
                                           "k_round_mma (one k-means round, persistent cooperative kernel, mma.sync)"),
                "achieved": ach_round, "peak": peak, "unit": "GB/s", "frac": ach_round / peak, "traffic": traffic,
                "traffic_source": traffic_source,
                "note": ("achieved = SURVEY 8(d) algorithmic bytes (4d + 8K + 4V + 4 per cell and round) / measured launch time; "
                         "the kernel itself moves fewer bytes than that definition: it never re-reads R (phase 0 folded into the "
                         "previous round's accumulation) and stores R only in the rounds after which cluster() can stop"
                         if tc5 else None),
                "peak_source": peak_src, "algorithmic_bytes_per_cell": b_round,
                "bytes_per_launch": b_round * n_local, "avg_launch_ms": ms_round / max(n_rounds, 1),
                "launches_timed": n_rounds, "share_of_step": ms_round / ms_total,
                "ridge": {"achieved": ach_ridge, "frac": ach_ridge / peak, "algorithmic_bytes_per_cell": b_ridge,
                          "avg_pass_ms": ms_ridge / max(n_ridge, 1), "share_of_step": ms_ridge / ms_total},
                "init_share_of_step": ms_init / ms_total}

    # ---- e2e through the public API with host buffers (rank-local shard in, local Z_corr out)
    e2e = None
    if not args.no_e2e:
        from harmonypy_b200.harmony import Harmony as H
        from harmonypy_b200 import pinned_empty
        # the caller's inputs live in page-locked host memory (the contract's "from pinned host memory"): the upload
        # is one DMA; the result comes back in a page-locked buffer of the wrapper's pool, re-used once the previous
        # result has been dropped (first call: allocation + pinning inside the timed region)
        Zp = pinned_empty(Z.shape, Z.dtype, local_rank); Zp[...] = Z
        codes_p = pinned_empty(codes.shape, codes.dtype, local_rank); codes_p[...] = codes
        prob_p = make_problem(w, Zp, codes_p, Pr_b, N_total, lo)
        times = []
        out = None
        for i in range(3):
            out = None                       # a caller that loops drops the previous result before the next call
            barrier()
            t0 = time.perf_counter()
            h2 = H(prob_p, 0.2, 10, 20, 1e-5, 1e-4, 0.05, False, SEED, local_rank, perm_mode="device", comm=comm,
                   engine_options=opts, init_centroids=Y0, run=True)
            out = h2.result_local()
            barrier()
            times.append(time.perf_counter() - t0)
            h2_dma = h2._engine.counter("dma_direct")
            del h2
        t_e2e = min(times)
        # the end-to-end result against the device-resident run timed above (same data, seed and centroids)
        ref = ho.result_local()
        e2e_diff = float(np.max(np.abs(out - ref)) / max(float(np.max(np.abs(ref))), 1e-30))
        del ref
        if dist is not None:
            t = torch.tensor([t_e2e], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            t_e2e = float(t.item())
        e2e = {"value": N_total / t_e2e, "unit": "cells/s", "seconds": t_e2e,
               "h2d_bytes_per_step": int(Z.nbytes + codes.nbytes + 3 * n_local * 4),
               "d2h_bytes_per_step": int(out.nbytes),
               "note": "Harmony(problem, ..., init_centroids) on host arrays: H2D upload, layout sort, "
                       "init assignment, harmonize to convergence, D2H of Z_corr; inputs in page-locked host memory "
                       "(harmonypy_b200.pinned_empty), result in a pooled page-locked buffer; best of 3",
               "seconds_all": [float(x) for x in times], "max_rel_diff_vs_resident_run": e2e_diff,
               "dma_direct": int(h2_dma)}

    # ---- CPU baseline beside it (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        r = cpu_arm(w, Y0, args.cpu_sample)
        cpu = {"value": args.cpu_sample / r["loop_seconds"], "unit": "cells/s", "cores": r["cores"], "host_cores": os.cpu_count(),
               "kind": r["kind"], "seconds": r["loop_seconds"], "sample": r["sample"]}

    parity = None
    if not args.no_parity:
        parity = golden_parity(local_rank, comm)          # all ranks: the datasets run sharded over the job's GPUs
    if rank == 0:
        out = {
            "metric": "cells/sec to convergence (full Harmony loop)", "value": value, "unit": "cells/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(w, world, N_total),
            "run": {"iterations_per_step": tot_iters / args.steps, "rounds_per_step": tot_rounds / args.steps,
                    "mode": ("persistent round kernel with in-kernel NVLink exchange of the K x B tables (fused, exact)"
                             if eng.counter("fused") == 1 else
                             "staged launches + NCCL all-reduce of the K x B tables per block (exact multi-GPU mode)" if world > 1
                             else "staged launches" if args.staged else
                             "persistent tcgen05 round kernel (k_round_tc5), one round ahead" if eng.counter("tc5") == 1
                             else "persistent round kernel")},
            "cell_rounds_per_s": n_local * world * n_rounds / (ms_round / 1e3) if ms_round > 0 else None,
            "ridge_passes_per_s": n_local * world * n_ridge / (ms_ridge / 1e3) if ms_ridge > 0 else None,
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "parity": parity, "gpu_launches": int(launches),
            "clocks": clocks.summary(), "setup_seconds": t_setup,
        }
        print(json.dumps(out), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="syn1m", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-sample", type=int, default=100_000)
    ap.add_argument("--staged", action="store_true", help="one launch per block step instead of the persistent kernel")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--engine-opt", action="append", default=[], help="name=int engine option (debug / A-B runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (rank 0's cells)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, w)
    else:
        run_ours(args, w)


if __name__ == "__main__":
    main()
