"""Centroid initialisation at scale: the device k-means++ / Lloyd (hmy_kmeans_init) on cells sharded over W GPUs
against the reference's path (sklearn KMeans on rank 0, then a broadcast of the centroids).

    python scripts/init_scaling.py [--worlds 1,2,4,8] [--cells-per-gpu 1000000] [--out FILE]

Every rank materialises its own shard of one synthetic dataset (harmonypy_b200.synthetic: d = 50 PCs, 20 batch levels,
K = 100) and creates an engine for it; no rank holds all cells.  World 1 is the single-GPU path.  Device timings are the
wall time of the slowest rank from a common start (barrier + device synchronise) to the return of kmeans_init, which ends
in a stream synchronise; the first call of each kind is a warm-up.  sklearn runs once, in the largest world, on the
first --sklearn-cells cells only (it is capped: at 1M cells it takes tens of seconds on the host), with the host's
default thread count.  Prints one JSON line; --out also writes it to FILE.  Needs as many CUDA devices as the largest
world (smaller worlds run, larger ones are skipped)."""
import argparse
import json
import os
import queue
import socket
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

D, K, LEVELS, SEED = 50, 100, [20], 0


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _worker(rank, world, port, q, a):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from harmonypy_b200 import _cabi
        from harmonypy_b200.harmony import Comm
        from harmonypy_b200.synthetic import make_synthetic_arrays
        comm = Comm(None)
        N = a.cells_per_gpu * world
        lo, hi = comm.shard(N)
        Z, codes = make_synthetic_arrays(N, D, LEVELS, seed=SEED, lo=lo, hi=hi)
        eng = _cabi.Engine(rank, hi - lo, N, lo, D, K, np.asarray(LEVELS, np.int32))
        eng.set_stream(torch.cuda.current_stream().cuda_stream)
        n_coll = [0]

        def allreduce(ptr, count, dtype, stream):
            n_coll[0] += 1
            return comm.allreduce_devptr(ptr, count, dtype, stream)
        eng.set_allreduce(allreduce)
        eng.set_rank(rank, world)
        eng.set_data(Z, codes)

        def timed(max_iter):
            torch.cuda.synchronize()
            dist.barrier()
            torch.cuda.synchronize()
            n_coll[0] = 0
            t0 = time.perf_counter()
            Y, info = eng.kmeans_init(SEED, max_iter=max_iter, tol=1e-4)
            dt = time.perf_counter() - t0
            worst = [None] * world
            dist.all_gather_object(worst, dt)
            return 1e3 * max(worst), info, n_coll[0], Y
        out = dict(world=world, n_cells=N)
        for label, max_iter in (("seeding", 0), ("init", 25)):
            timed(max_iter)                                   # warm-up
            runs = [timed(max_iter) for _ in range(a.reps)]
            out[f"{label}_ms"] = [round(r[0], 3) for r in runs]
            out[f"{label}_ms_median"] = round(float(np.median([r[0] for r in runs])), 3)
            out[f"{label}_collectives"] = runs[-1][2]
            if label == "init":
                info = runs[-1][1]
                out["lloyd_iterations"] = info["iterations"]
                out["inertia"] = info["inertia"]
                out["identical_over_repeats"] = all(np.array_equal(r[3], runs[0][3]) for r in runs)
        if a.sklearn and comm.world == a.max_world:
            out["sklearn"] = _sklearn_arm(a, comm, rank)
        if rank == 0:
            q.put(out)
    finally:
        dist.destroy_process_group()


def _sklearn_arm(a, comm, rank):
    """The reference's initialisation (harmony.py:369-373) on rank 0 over the first a.sklearn_cells cells, then the
    broadcast every other rank waits in (what Harmony.init_cluster does with init_mode="sklearn")."""
    import torch
    from harmonypy_b200.synthetic import make_synthetic_arrays
    n = min(a.sklearn_cells, a.cells_per_gpu * comm.world)
    res = None
    C = np.zeros((K, D), dtype=np.float32)
    if rank == 0:
        from sklearn.cluster import KMeans
        Z, _ = make_synthetic_arrays(a.cells_per_gpu * comm.world, D, LEVELS, seed=SEED, lo=0, hi=n)
        t0 = time.perf_counter()
        Zc = Z / np.linalg.norm(Z, axis=1, keepdims=True)
        model = KMeans(n_clusters=K, init="k-means++", n_init=1, max_iter=25, random_state=SEED).fit(Zc)
        C = model.cluster_centers_.astype(np.float32)
        t_fit = time.perf_counter() - t0
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    comm.broadcast_array(C, src=0)
    torch.cuda.synchronize()
    t_bc = time.perf_counter() - t1
    if rank == 0:
        res = dict(cells=n, capped=n < a.cells_per_gpu * comm.world, fit_s=round(t_fit, 3),
                   broadcast_ms=round(1e3 * t_bc, 3), lloyd_iterations=int(model.n_iter_),
                   inertia=float(model.inertia_), host_threads=os.cpu_count())
    return res


def _run_world(world, a):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, a)) for r in range(world)]
    try:
        for p in procs:
            p.start()
        deadline = time.time() + a.timeout
        while True:
            try:
                out = q.get(timeout=5)
                break
            except queue.Empty:
                dead = [p.exitcode for p in procs if p.exitcode not in (None, 0)]
                if dead or time.time() > deadline:
                    raise RuntimeError(f"world {world}: ranks failed (exit codes {dead}) or timed out")
        for p in procs:
            p.join(timeout=300)
            if p.exitcode != 0:
                raise RuntimeError(f"world {world}: a rank exited with {p.exitcode}")
        return out
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
            p.join(timeout=30)


def _gpu_description():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        rows = [x.strip() for x in r.stdout.strip().splitlines() if x.strip()]
        return rows[0] if rows else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--worlds", default="1,2,4,8")
    ap.add_argument("--cells-per-gpu", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sklearn-cells", type=int, default=1_000_000)
    ap.add_argument("--no-sklearn", dest="sklearn", action="store_false")
    ap.add_argument("--timeout", type=float, default=1200.0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    n_dev = torch.cuda.device_count()
    if n_dev == 0:
        raise SystemExit("init_scaling.py needs CUDA devices")
    worlds = [w for w in (int(x) for x in a.worlds.split(",")) if w <= n_dev]
    a.max_world = max(worlds)
    from harmonypy_b200.build import build
    build(verbose=False)
    result = dict(metric="init_scaling", gpu=_gpu_description(), devices=n_dev, cells_per_gpu=a.cells_per_gpu,
                  d=D, K=K, max_iter=25, tol=1e-4, runs=[_run_world(w, a) for w in worlds])
    line = json.dumps(result)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
