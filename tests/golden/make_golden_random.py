#!/usr/bin/env python
"""Golden fixtures for the randomised comparisons with the original harmonypy (slowkow/harmonypy).

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden_random.py <harmonypy checkout>

The inputs are the seeded random problems the tests themselves build; this script runs the unmodified package on
them and stores what it returned, so the tests compare against it without the package being present:

  * ``random_oracle.npz``   -- harmony.py restated in fp64 (the temp-copy substitution of make_golden.py) on the
    configurations of tests/test_oracle_live_reference.py: its sklearn centroids, digests of its permutations
    (the torch.manual_seed(0) stream of oracle.harmony_oracle.torch_perm_source), its parameters, kmeans_rounds,
    objectives, O, and Z_corr / R on a fixed subsample of the cells (every 4th / every 8th cell);
  * ``random_frontend.npz`` -- run_harmony(max_iter_harmony=0)'s argument normalisation on the calls of
    tests/test_frontend_live_reference.py (exact arrays as the first 16 hex digits of their SHA-1) and the exception
    types it raises;
  * ``random_lisi.npz``     -- compute_lisi on the random data of tests/test_lisi_oracle.py.
"""
import hashlib
import os
import sys

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path.insert(0, os.path.dirname(TESTS))
sys.path.insert(0, TESTS)
sys.path.insert(0, HERE)

import numpy as np
import pandas as pd

ZCORR_STEP, R_STEP = 4, 8


def digest(a):
    return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def oracle_cases(ref):
    import make_golden
    import test_oracle_live_reference as t
    from oracle.harmony_oracle import torch_perm_source
    make_golden.REF = ref
    mod64 = make_golden.load_reference_module(True)
    out = {}
    for case, (N, d, levels, kw) in enumerate(t.CASES):
        rng = np.random.default_rng(100 + case)
        Z, meta = t._problem(rng, N, d, levels)
        kw = dict(kw, max_iter_harmony=kw.get("max_iter_harmony", 3))
        ho, cap = make_golden.run_captured(mod64, pd.DataFrame(Z.astype(np.float64)), meta, list(meta.columns), kw,
                                           np.arange(0, N, 7))
        src = torch_perm_source(N, 0)
        for p in cap["perms"]:
            assert np.array_equal(p, src()), "the reference's permutations are not the torch.manual_seed(0) stream"
        p = f"c{case}_"
        out.update({
            p + "Z_digest": np.array(digest(Z)),
            p + "Phi_digest": np.array(digest(np.asarray(ho.Phi.T, dtype=np.uint8))),
            p + "Y0": np.asarray(cap["Y0"], dtype=np.float32),
            p + "perm_digests": np.array([digest(np.asarray(q, dtype=np.int64)) for q in cap["perms"]]),
            p + "Pr_b": np.asarray(ho.Pr_b, dtype=np.float64), p + "sigma": np.asarray(ho.sigma, dtype=np.float64),
            p + "theta": np.asarray(ho.theta, dtype=np.float64), p + "lamb": np.asarray(ho.lamb, dtype=np.float64),
            p + "alpha": np.float64(ho.alpha), p + "lambda_estimation": np.bool_(ho.lambda_estimation),
            p + "block_size": np.float64(ho.block_size), p + "epsilon_kmeans": np.float64(ho.epsilon_kmeans),
            p + "epsilon_harmony": np.float64(ho.epsilon_harmony), p + "max_iter_kmeans": np.int32(ho.max_iter_kmeans),
            p + "max_iter_harmony": np.int32(ho.max_iter_harmony),
            p + "kmeans_rounds": np.asarray(ho.kmeans_rounds, dtype=np.int32),
            p + "objective_harmony": np.asarray(ho.objective_harmony, dtype=np.float64),
            p + "objective_kmeans": np.asarray(ho.objective_kmeans, dtype=np.float64),
            p + "O": np.asarray(ho.O, dtype=np.float64),
            p + "Zcorr_absmax": np.float64(np.abs(ho.Z_corr).max()),
            p + "Zcorr_sub": np.asarray(ho.Z_corr[::ZCORR_STEP], dtype=np.float64),
            p + "R_sub": np.asarray(ho.R[::R_STEP], dtype=np.float64),
        })
        print(f"oracle case {case}: rounds {list(ho.kmeans_rounds)}")
    out["zcorr_step"], out["r_step"] = np.int32(ZCORR_STEP), np.int32(R_STEP)
    return out


def _exc_name(e):
    return f"{type(e).__module__}.{type(e).__qualname__}"


def frontend_calls(ref):
    sys.path.insert(0, ref)
    import harmonypy
    import test_frontend_live_reference as t
    out = {}
    for i, spec in enumerate(t.CALLS):
        rng = np.random.default_rng(40 + i)
        Z, meta = t._data(rng, spec.get("N", 400), 6, spec["levels"])
        vars_use = list(meta.columns)
        if spec.get("vars_as_str"):
            vars_use = vars_use[0]
        data = pd.DataFrame(Z.T if spec.get("transpose") else Z)
        ho = harmonypy.run_harmony(data, meta, vars_use, max_iter_harmony=0, verbose=False, device="cpu", **spec["kw"])
        p = f"call{i}_"
        out.update({
            p + "K": np.int64(ho.K), p + "N": np.int64(ho.N), p + "d": np.int64(ho.d), p + "B": np.int64(ho.B),
            p + "lambda_estimation": np.bool_(ho.lambda_estimation),
            p + "Pr_b": np.asarray(ho.Pr_b, dtype=np.float64).ravel(),
            p + "theta": np.asarray(ho.theta, dtype=np.float64).ravel(),
            p + "sigma": np.asarray(ho.sigma, dtype=np.float64).ravel(),
            p + "lamb": np.asarray(ho.lamb, dtype=np.float64).ravel(),
            p + "Z_orig_digest": np.array(digest(np.asarray(ho.Z_orig, dtype=np.float32))),
            p + "Phi_digest": np.array(digest(np.asarray(ho.Phi.T, dtype=np.uint8))),
        })
    for i, spec in enumerate(t.BAD_CALLS):
        rng = np.random.default_rng(70 + i)
        Z, meta = t._data(rng, 300, 5, [2, 3])
        if spec.get("numeric_covariate"):
            meta["c0"] = rng.integers(0, 2, 300)
        if spec.get("wrong_shape"):
            Z = Z[:250, :4]
        try:
            harmonypy.run_harmony(pd.DataFrame(Z), meta, list(meta.columns), max_iter_harmony=0, verbose=False,
                                  device="cpu", **spec["kw"])
            raise SystemExit(f"bad call {i} did not raise")
        except Exception as e:
            out[f"bad{i}_exception"] = np.array(_exc_name(e))
    rng = np.random.default_rng(5)
    Z, meta = t._data(rng, 300, 5, [2, 3])
    try:
        harmonypy.run_harmony(pd.DataFrame(Z), meta, list(meta.columns), lamb=[1.0, 2.0, 3.0], max_iter_harmony=1,
                              verbose=False, device="cpu")
        raise SystemExit("the wrong-length lambda call did not raise")
    except Exception as e:
        out["wrong_lamb_exception"] = np.array(_exc_name(e))
    return out


def lisi_cases(ref):
    sys.path.insert(0, ref)
    from harmonypy.lisi import compute_lisi
    import test_lisi_oracle as t
    out = {}
    for n, d, perp, seed in t.RANDOM_CASES:
        X, meta = t._random_problem(n, d, seed)
        out[f"seed{seed}_lisi"] = np.asarray(compute_lisi(X, meta, list(meta.columns), perp), dtype=np.float64)
    return out


def main(ref):
    for name, fn in (("random_oracle", oracle_cases), ("random_frontend", frontend_calls), ("random_lisi", lisi_cases)):
        path = os.path.join(HERE, f"{name}.npz")
        np.savez_compressed(path, **fn(ref))
        print("wrote", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    if len(sys.argv) != 2 or not os.path.exists(os.path.join(sys.argv[1], "harmonypy", "harmony.py")):
        raise SystemExit("usage: make_golden_random.py <checkout of slowkow/harmonypy>")
    main(os.path.abspath(sys.argv[1]))
