"""hmy_kmeans_init on cells sharded over 2 / 4 / 8 GPUs (one process per GPU, fused and staged mode, even and uneven
pre-sharded cell ranges) against the single-process oracle (oracle/kmeans_init_oracle.py: kmeans_init on all cells),
and a full pre-sharded Harmony(init_mode="device") run.  Needs as many CUDA devices as ranks (skipped otherwise)."""
import os
import queue
import socket
import time
import traceback

import numpy as np
import pytest

from conftest import load_case

pytestmark = pytest.mark.gpu

NAMES = ["pbmc", "synth", "ircolitis"]
SEEDS = (0, 7)


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _edges(world, N, uneven):
    if uneven:
        return [0, (3 * N) // 10, N]
    return [N * r // world for r in range(world + 1)]


def _problem(inp, edges, rank):
    from harmonypy_b200.harmony import Problem
    lo, hi = edges[rank], edges[rank + 1]
    N = inp["Z"].shape[0]
    return Problem(Z=np.ascontiguousarray(inp["Z"][lo:hi]), codes=np.ascontiguousarray(inp["codes"][:, lo:hi]),
                   levels=inp["levels"], level_names=[], Pr_b=inp["Pr_b"], theta=inp["theta"], lamb=inp["lamb"],
                   lambda_estimation=bool(inp["lambda_estimation"]), sigma=inp["sigma"], K=int(inp["K"]),
                   n_global=N, shard_lo=lo)


def _harmony(inp, prob, rank, **kw):
    from harmonypy_b200.harmony import Harmony
    return Harmony(prob, float(inp["alpha"]), int(inp["max_iter_harmony"]), int(inp["max_iter_kmeans"]),
                   float(inp["epsilon_kmeans"]), float(inp["epsilon_harmony"]), float(inp["block_size"]), False,
                   int(inp["random_state"]), rank, comm=True, **kw)


def _init_worker(rank, world, port, q, fused, uneven):
    """Every case's device initialisations on this rank: max_iter 0, (1, tol 0), (25, 1e-4) for each seed."""
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        out, engines = dict(rank=rank, cases={}), []
        for name in NAMES:
            inp, _ = load_case(name)
            edges = _edges(world, inp["Z"].shape[0], uneven)
            ho = _harmony(inp, _problem(inp, edges, rank), rank, run=False, engine_options={"fused": fused})
            res = dict(fused=ho._engine.counter("fused"), lo=ho._lo, hi=ho._hi)
            for seed in SEEDS:
                res[seed, 0] = ho._engine.kmeans_init(seed, max_iter=0)
                res[seed, 1] = ho._engine.kmeans_init(seed, max_iter=1, tol=0.0)
                res[seed, 25] = ho._engine.kmeans_init(seed, max_iter=25, tol=1e-4)
            out["cases"][name] = res
            engines.append(ho)                 # peers may still map its exchange buffer: released at process exit
        q.put(out)
    except BaseException:
        q.put(dict(rank=rank, error=traceback.format_exc()))
        raise
    finally:
        dist.destroy_process_group()


def _run_ranks(target, world, *args, timeout=900):
    """Spawn one process per rank, collect one result per rank; every worker is terminated and joined on the way out."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=target, args=(r, world, port, q) + args) for r in range(world)]
    try:
        for p in procs:
            p.start()
        outs, deadline = [], time.time() + timeout
        while len(outs) < world:
            try:
                o = q.get(timeout=5)
            except queue.Empty:
                dead = [p.exitcode for p in procs if p.exitcode not in (None, 0)]
                assert not dead, f"a rank exited with {dead} before reporting"
                assert time.time() < deadline, "ranks did not report in time"
                continue
            assert "error" not in o, f"rank {o['rank']} failed:\n{o['error']}"
            outs.append(o)
        for p in procs:
            p.join(timeout=120)
            assert p.exitcode == 0
        return sorted(outs, key=lambda o: o["rank"])
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
            p.join(timeout=30)


_CACHE = {}


def _sharded_results(world, fused, uneven):
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    key = (world, fused, uneven)
    if key not in _CACHE:
        try:
            _CACHE[key] = _run_ranks(_init_worker, world, fused, uneven)
        except BaseException as exc:          # one spawn per configuration, also when it failed
            _CACHE[key] = exc
    if isinstance(_CACHE[key], BaseException):
        raise _CACHE[key]
    return _CACHE[key]


_ORACLE = {}


def _oracle(name, seed, max_iter, tol):
    from oracle.kmeans_init_oracle import kmeans_init
    key = (name, seed, max_iter, tol)
    if key not in _ORACLE:
        inp, _ = load_case(name)
        _ORACLE[key] = kmeans_init(inp["Z"], int(inp["K"]), seed, max_iter=max_iter, tol=tol)
    return _ORACLE[key]


@pytest.mark.parametrize("world,fused,uneven", [(2, 1, False), (2, 0, False), (2, 1, True), (4, 1, False), (8, 1, False)],
                         ids=["2-fused", "2-staged", "2-fused-presharded-uneven", "4-fused", "8-fused"])
@pytest.mark.parametrize("name", NAMES)
def test_sharded_device_init_matches_the_oracle(name, world, fused, uneven):
    outs = _sharded_results(world, fused, uneven)
    res = [o["cases"][name] for o in outs]
    inp, _ = load_case(name)
    edges = _edges(world, inp["Z"].shape[0], uneven)
    assert [(r["lo"], r["hi"]) for r in res] == list(zip(edges[:-1], edges[1:]))
    assert all(r["fused"] == fused for r in res)
    for seed in SEEDS:
        for it in (0, 1, 25):
            Y0, info0 = res[0][seed, it]
            for r in res[1:]:                                  # bitwise the same on every rank
                np.testing.assert_array_equal(r[seed, it][0], Y0)
                assert r[seed, it][1] == info0
        C0, _ = _oracle(name, seed, 0, 1e-4)
        np.testing.assert_allclose(res[0][seed, 0][0], C0, atol=1e-6, err_msg="k-means++ picked different cells")
        C1, _ = _oracle(name, seed, 1, 0.0)
        assert np.abs(res[0][seed, 1][0] - C1).max() < 5e-3
        _, oinfo = _oracle(name, seed, 25, 1e-4)
        info = res[0][seed, 25][1]
        print(f"\n[{name} seed {seed}, {world} GPUs {'fused' if fused else 'staged'}{' uneven' if uneven else ''}] "
              f"iterations {info['iterations']} vs {oinfo['iterations']}, inertia {info['inertia']:.6f} vs {oinfo['inertia']:.6f}")
        assert abs(info["iterations"] - oinfo["iterations"]) <= 1
        assert abs(info["inertia"] - oinfo["inertia"]) <= 1e-3 * oinfo["inertia"]


def _harmony_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        inp, _ = load_case("pbmc")
        ho = _harmony(inp, _problem(inp, _edges(2, inp["Z"].shape[0], True), rank), rank, init_mode="device")
        q.put(dict(rank=rank, Z=ho.Z_corr, obj=list(ho.objective_harmony), info=ho.kmeans_init_info,
                   rounds=list(ho.kmeans_rounds)))
    except BaseException:
        q.put(dict(rank=rank, error=traceback.format_exc()))
        raise
    finally:
        dist.destroy_process_group()


def test_presharded_harmony_runs_from_device_init_on_two_gpus():
    """No rank holds all cells and no init_centroids is given: the ranks initialise together and run to the end."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    a, b = _run_ranks(_harmony_worker, 2)
    _, gold = load_case("pbmc")
    assert a["info"] == b["info"] and a["info"]["iterations"] >= 1
    assert a["rounds"] == b["rounds"] and a["obj"] == b["obj"]
    np.testing.assert_array_equal(a["Z"], b["Z"])
    assert np.isfinite(a["Z"]).all() and np.isfinite(a["obj"]).all()
    ref = float(gold["objective_harmony"][-1])
    print(f"\n[pbmc, 2 GPUs pre-sharded, device init] final objective {a['obj'][-1]:.4f} vs sklearn-initialised {ref:.4f}")
    assert abs(a["obj"][-1] - ref) < 0.03 * abs(ref)


def test_shard_without_allreduce_or_rank_fails_before_any_collective():
    from harmonypy_b200._cabi import Engine, EngineError
    inp, _ = load_case("synth")
    n, N, K = 1000, inp["Z"].shape[0], int(inp["K"])
    eng = Engine(0, n, N, 0, inp["Z"].shape[1], K, inp["levels"])
    try:
        eng.set_data(inp["Z"][:n], inp["codes"][:, :n])
        with pytest.raises(EngineError, match="all-reduce over ranks: call hmy_set_allreduce"):
            eng.kmeans_init(0)
        calls = []
        eng.set_allreduce(lambda ptr, count, dtype, stream: calls.append(count) or 1)
        with pytest.raises(EngineError, match="needs its rank: call hmy_set_rank"):
            eng.kmeans_init(0)
        assert calls == []                                    # no collective was started
        with pytest.raises(EngineError, match="rank < world"):
            eng.set_rank(2, 2)
    finally:
        eng.close()


# ---- ranks as threads on one GPU ------------------------------------------------------------------------------------
# The same C ABI path on a one-GPU machine: W contexts on device 0, one thread per context, and a sum all-reduce through
# host memory in rank order.  A rank that never arrives breaks the barrier (timeout) instead of hanging the test.

class _HostAllreduce:
    def __init__(self, world, timeout=120.0):
        import threading
        self.world, self.bufs, self.calls = world, [None] * world, [0] * world
        self.barrier = threading.Barrier(world, timeout=timeout)

    def for_rank(self, rank):
        import torch

        def fn(ptr, count, dtype, stream):
            class _Mem:
                pass
            m = _Mem()
            m.__cuda_array_interface__ = {"shape": (int(count),), "typestr": "<f4" if dtype == 0 else "<f8",
                                          "data": (int(ptr), False), "version": 2}
            t = torch.as_tensor(m, device="cuda")
            torch.cuda.synchronize()
            self.calls[rank] += 1
            self.bufs[rank] = t.cpu().numpy().copy()
            self.barrier.wait()
            total = self.bufs[0].copy()
            for r in range(1, self.world):
                total += self.bufs[r]
            self.barrier.wait()
            t.copy_(torch.from_numpy(total))
            torch.cuda.synchronize()
            return 0
        return fn


def _thread_ranks(name, edges, args_of_rank):
    """kmeans_init on every rank's context at once; returns per rank (Y, info) or the exception it raised."""
    import threading
    from harmonypy_b200._cabi import Engine
    inp, _ = load_case(name)
    Z, codes, N, K = inp["Z"], inp["codes"], inp["Z"].shape[0], int(inp["K"])
    world = len(edges) - 1
    ar = _HostAllreduce(world)
    engines = []
    for r in range(world):
        lo, hi = edges[r], edges[r + 1]
        eng = Engine(0, hi - lo, N, lo, Z.shape[1], K, inp["levels"])
        eng.set_data(Z[lo:hi], codes[:, lo:hi])
        eng.set_allreduce(ar.for_rank(r))
        eng.set_rank(r, world)
        engines.append(eng)
    out = [None] * world

    def run(r):
        try:
            out[r] = engines[r].kmeans_init(*args_of_rank(r))
        except Exception as exc:                              # noqa: BLE001 -- reported to the test
            out[r] = exc
    threads = [threading.Thread(target=run, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for e in engines:
        e.close()
    return out, ar.calls


@pytest.mark.parametrize("name,split", [("pbmc", "even"), ("synth", "uneven"), ("pbmc", "small")])
def test_ranks_on_one_gpu_match_the_oracle(name, split):
    inp, _ = load_case(name)
    N, K = inp["Z"].shape[0], int(inp["K"])
    edges = {"even": [0, N // 2, N], "uneven": [0, (3 * N) // 10, N],
             "small": [0, K // 2, N - K // 3, N]}[split]            # shards with fewer cells than clusters
    for seed in SEEDS:
        for max_iter, tol in ((0, 1e-4), (1, 0.0), (25, 1e-4)):
            out, calls = _thread_ranks(name, edges, lambda r: (seed, max_iter, tol))
            for o in out:
                assert not isinstance(o, Exception), o
                np.testing.assert_array_equal(o[0], out[0][0])
                assert o[1] == out[0][1]
            assert len(set(calls)) == 1 and calls[0] == K + 2 + 2 * out[0][1]["iterations"]
            C, oinfo = _oracle(name, seed, max_iter, tol)
            Y, info = out[0]
            if max_iter == 0:
                np.testing.assert_allclose(Y, C, atol=1e-6, err_msg="k-means++ picked different cells")
            elif max_iter == 1:
                assert np.abs(Y - C).max() < 5e-3
            else:
                assert abs(info["iterations"] - oinfo["iterations"]) <= 1
                assert abs(info["inertia"] - oinfo["inertia"]) <= 1e-3 * oinfo["inertia"]


def test_ranks_fail_together():
    """One rank's bad argument, or ranks that disagree, fail every rank after the first exchange: no rank is left
    waiting in a collective."""
    from harmonypy_b200._cabi import EngineError
    inp, _ = load_case("synth")
    N = inp["Z"].shape[0]
    edges = [0, N // 2, N]
    out, calls = _thread_ranks("synth", edges, lambda r: (0, 25 if r == 0 else -1, 1e-4))
    assert isinstance(out[0], EngineError) and "rank 1 failed its checks" in str(out[0])
    assert isinstance(out[1], EngineError) and "non-negative" in str(out[1])
    assert calls == [1, 1]
    out, calls = _thread_ranks("synth", edges, lambda r: (r, 25, 1e-4))
    assert all(isinstance(o, EngineError) and "disagree" in str(o) for o in out)
    assert calls == [1, 1]
