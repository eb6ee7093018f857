"""Device k-means initialisation on cells sharded over ranks, on CPU: the sharded oracle
(tests/kmeans_init_shard_oracle.py: kmeans_init_sharded -- per-shard passes, one slot per rank summed as an exact all-gather,
Lloyd tables summed over ranks) against the single-process oracle, and the host's init_mode="device" path over a gloo
world of 2 with a test engine whose kmeans_init is that oracle over a real all-reduce."""
import os
import socket

import numpy as np
import pandas as pd
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import load_case, rel_max
from kmeans_init_shard_oracle import kmeans_init_rank, kmeans_init_sharded
from oracle.kmeans_init_oracle import kmeans_init
from shard_engine import ShardOracleEngine


def _edges(split, N, K):
    return {"even": [0, N // 2, N],
            "uneven": [0, N // 3 + 17, N],
            "small": [0, K // 2, N - K // 3, N],          # first and last shard hold fewer cells than clusters
            "eight": [N * r // 8 for r in range(9)]}[split]


@pytest.mark.parametrize("seed", [0, 7])
@pytest.mark.parametrize("split", ["even", "uneven", "small", "eight"])
@pytest.mark.parametrize("name", ["pbmc", "synth"])
def test_sharded_oracle_matches_single_process(name, split, seed):
    inp, _ = load_case(name)
    Z, K = inp["Z"], int(inp["K"])
    edges = _edges(split, Z.shape[0], K)
    C0, i0 = kmeans_init(Z, K, seed, max_iter=0)
    S0, j0 = kmeans_init_sharded(Z, K, seed, edges, max_iter=0)
    np.testing.assert_array_equal(j0["seeds"], i0["seeds"])
    np.testing.assert_array_equal(S0, C0)
    C1, _ = kmeans_init(Z, K, seed, max_iter=1, tol=0.0)
    S1, _ = kmeans_init_sharded(Z, K, seed, edges, max_iter=1, tol=0.0)
    assert np.abs(S1 - C1).max() <= 1e-6
    C25, i25 = kmeans_init(Z, K, seed, max_iter=25, tol=1e-4)
    S25, j25 = kmeans_init_sharded(Z, K, seed, edges, max_iter=25, tol=1e-4)
    np.testing.assert_array_equal(j25["seeds"], i25["seeds"])
    assert j25["iterations"] == i25["iterations"]
    assert abs(j25["inertia"] - i25["inertia"]) <= 1e-9 * i25["inertia"]


def test_sharded_oracle_reports_too_few_distinct_cells():
    Z = np.repeat(np.eye(3, dtype=np.float32), 10, axis=0)             # 30 cells, 3 distinct
    with pytest.raises(ValueError, match="fewer distinct cells"):
        kmeans_init_sharded(Z, 4, 0, [0, 12, 30])


# ---- the host over gloo ----------------------------------------------------------------------------------------------

class KmeansShardEngine(ShardOracleEngine):
    """ShardOracleEngine plus kmeans_init: the sharded oracle over the run's all-reduce."""

    def set_data(self, Z, codes):
        super().set_data(Z, codes)
        self.Z32 = np.asarray(Z, dtype=np.float32)

    def kmeans_init(self, seed, max_iter=25, tol=1e-4):
        self.calls["kmeans_init"] = self.calls.get("kmeans_init", 0) + 1
        self.centroids, info = kmeans_init_rank(self.Z32, self.lo, self.N, self.K, seed, self.comm.rank,
                                                self.comm.world, self.comm.allreduce_numpy, max_iter, tol)
        return self.centroids, info


CASE = dict(N=3001, d=8, levels=[3], K=12, iters=2, seed=9)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q, edges):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.set_num_threads(2)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import dataclasses
        from harmonypy_b200.harmony import Harmony, prepare_problem, run_harmony
        from harmonypy_b200.synthetic import make_synthetic
        c = CASE
        Z, meta = make_synthetic(c["N"], c["d"], c["levels"], seed=4)
        if edges is None:
            ho = run_harmony(Z, meta, list(meta.columns), nclust=c["K"], max_iter_harmony=c["iters"],
                             max_iter_kmeans=6, verbose=False, random_state=c["seed"], init_mode="device",
                             comm=True, engine_factory=KmeansShardEngine)
        else:
            full, _ = prepare_problem(pd.DataFrame(Z), meta, list(meta.columns), nclust=c["K"])
            lo, hi = edges[rank], edges[rank + 1]
            mine = dataclasses.replace(full, Z=full.Z[lo:hi].copy(), codes=full.codes[:, lo:hi].copy(),
                                       n_global=c["N"], shard_lo=lo)
            ho = Harmony(mine, 0.2, c["iters"], 6, 1e-5, 1e-4, 0.05, False, c["seed"], 0, comm=True,
                         engine_factory=KmeansShardEngine, init_mode="device")
        q.put(dict(rank=rank, lo=ho._lo, hi=ho._hi, calls=ho._engine.calls.get("kmeans_init", 0),
                   C=ho._engine.centroids, info=ho.kmeans_init_info, rounds=list(ho.kmeans_rounds),
                   obj=list(ho.objective_kmeans), Z=ho.Z_corr))
    finally:
        dist.destroy_process_group()


def _run(edges, world=2):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, edges)) for r in range(world)]
    try:
        for p in procs:
            p.start()
        outs = [q.get(timeout=300) for _ in procs]
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
            p.join(timeout=30)
    return sorted(outs, key=lambda o: o["rank"])


def _single(C):
    from oracle.harmony_oracle import HarmonyOracle, onehot_from_codes, torch_perm_source
    from harmonypy_b200.harmony import prepare_problem
    from harmonypy_b200.synthetic import make_synthetic
    c = CASE
    Z, meta = make_synthetic(c["N"], c["d"], c["levels"], seed=4)
    prob, _ = prepare_problem(pd.DataFrame(Z), meta, list(meta.columns), nclust=c["K"])
    orc = HarmonyOracle(prob.Z.T, onehot_from_codes(prob.codes, prob.levels, np.float64), prob.Pr_b, prob.sigma,
                        prob.theta, prob.lamb, lambda_estimation=prob.lambda_estimation, max_iter_kmeans=6,
                        dtype=np.float64)
    orc.init_from_centroids(C.T)
    orc.harmonize(c["iters"], torch_perm_source(c["N"], c["seed"]))
    return orc, prob.Z


@pytest.mark.parametrize("edges", [None, [0, 1100, 3001]], ids=["even", "presharded_uneven"])
def test_two_ranks_initialise_on_device_and_reproduce_single_process_oracle(edges):
    a, b = _run(edges)
    if edges is not None:
        assert (a["lo"], a["hi"], b["lo"], b["hi"]) == (0, 1100, 1100, 3001)
    assert a["calls"] == b["calls"] == 1
    np.testing.assert_array_equal(a["C"], b["C"])             # bitwise: every rank starts from the same centroids
    assert a["info"]["iterations"] == b["info"]["iterations"] and a["info"]["inertia"] == b["info"]["inertia"]
    orc, Z = _single(a["C"])
    # the centroids are the sharded oracle's, whose seeds are those of one process holding every cell
    C, info = kmeans_init_sharded(Z, CASE["K"], CASE["seed"], edges or [0, CASE["N"] // 2, CASE["N"]])
    np.testing.assert_array_equal(a["C"], C)
    np.testing.assert_array_equal(info["seeds"], kmeans_init(Z, CASE["K"], CASE["seed"])[1]["seeds"])
    assert a["rounds"] == b["rounds"] == list(orc.kmeans_rounds)
    np.testing.assert_array_equal(a["Z"], b["Z"])
    np.testing.assert_allclose(a["obj"], b["obj"], rtol=0, atol=0)
    np.testing.assert_allclose(a["obj"], orc.objective_kmeans, rtol=1e-9)
    assert rel_max(a["Z"], orc.Z_corr.T) < 1e-6
