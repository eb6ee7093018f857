"""Differential test of the CPU oracle against the reference over randomised configurations.

The golden fixtures of the three datasets pin the oracle there; this test widens the pin across the argument space
(per-covariate / per-level theta and lambda, dynamic lambda, tau, sigma, block sizes, 1-3 covariates, small K).  It
runs the fp64 oracle on seeded random problems and compares with what the reference's fp64 restatement (harmonypy/
harmony.py with float32 -> float64 substituted, as tests/golden/make_golden.py does) returned on the same inputs,
the same sklearn centroids and the same permutation stream: tests/golden/random_oracle.npz, written by
tests/golden/make_golden_random.py.  Agreement is at rounding level (1e-9), not at fp32 noise level.  CPU only.
"""
import hashlib
import os

import numpy as np
import pandas as pd
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def ref64():
    return np.load(os.path.join(GOLDEN, "random_oracle.npz"))


def _digest(a):
    return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def _problem(rng, N, d, levels):
    ntype = 5
    centers = rng.normal(size=(ntype, d)) * 2.0
    t = rng.integers(0, ntype, N)
    Z = centers[t] + rng.normal(size=(N, d))
    meta = {}
    for v, L in enumerate(levels):
        b = rng.integers(0, L, N)
        Z = Z + (rng.normal(size=(L, d)) * 0.8)[b]
        meta[f"v{v}"] = pd.Categorical([f"l{v}_{x}" for x in b])
    return Z.astype(np.float32), pd.DataFrame(meta)


CASES = [
    # N, d, levels, kwargs
    (700, 8, [3], dict(nclust=9)),
    (900, 6, [4, 2], dict(nclust=12, theta=[1.5, 0.5], lamb=[0.5, 2.0], sigma=0.15)),
    (800, 10, [2, 3, 2], dict(nclust=10, theta=[2.0, 1.0, 0.7, 1.2, 0.3, 2.5, 1.1], lamb=-1, alpha=0.35)),
    (650, 5, [5], dict(nclust=8, tau=7, theta=3.0, block_size=0.2, max_iter_kmeans=6)),
    (1000, 7, [3, 3], dict(nclust=14, lamb=[0.1, 0.2, 0.3, 1.0, 2.0, 3.0], block_size=0.013, epsilon_cluster=1e-3)),
    (600, 4, [2], dict(nclust=5, sigma=0.3, block_size=0.5, epsilon_harmony=1e-2)),
]


@pytest.mark.parametrize("case", range(len(CASES)))
def test_oracle_fp64_equals_live_reference_fp64(ref64, case):
    from oracle.harmony_oracle import HarmonyOracle, onehot_from_codes, torch_perm_source
    g = {k[len(f"c{case}_"):]: ref64[k] for k in ref64.files if k.startswith(f"c{case}_")}
    N, d, levels, _ = CASES[case]                   # the keyword arguments went to the reference's run_harmony
    rng = np.random.default_rng(100 + case)
    Z, meta = _problem(rng, N, d, levels)
    assert _digest(Z) == str(g["Z_digest"]), "the seeded input is not the one the reference ran on"

    codes = np.stack([pd.Categorical(meta[v]).codes for v in meta.columns]).astype(np.int32)
    lv = np.array([len(pd.Categorical(meta[v]).categories) for v in meta.columns], dtype=np.int32)
    phi = onehot_from_codes(codes, lv, np.float64)
    assert _digest(phi.astype(np.uint8)) == str(g["Phi_digest"])
    orc = HarmonyOracle(Z.astype(np.float64).T, phi, g["Pr_b"], g["sigma"], g["theta"], g["lamb"], alpha=float(g["alpha"]),
                        lambda_estimation=bool(g["lambda_estimation"]), block_size=float(g["block_size"]),
                        epsilon_kmeans=float(g["epsilon_kmeans"]), epsilon_harmony=float(g["epsilon_harmony"]),
                        max_iter_kmeans=int(g["max_iter_kmeans"]), dtype=np.float64)
    # the reference's centroids and its permutation stream (torch.manual_seed(0), one randperm per update_R)
    src, want_perms = torch_perm_source(N, 0), iter(g["perm_digests"])

    def perms():
        p = src()
        assert _digest(p.astype(np.int64)) == str(next(want_perms)), "permutation stream differs from the reference's"
        return p
    orc.init_from_centroids(np.asarray(g["Y0"], dtype=np.float64).T)
    orc.harmonize(int(g["max_iter_harmony"]), perms)

    assert list(orc.kmeans_rounds) == list(g["kmeans_rounds"])
    assert next(want_perms, None) is None
    zs, rs = int(ref64["zcorr_step"]), int(ref64["r_step"])
    assert np.abs(orc.Z_corr.T[::zs] - g["Zcorr_sub"]).max() / float(g["Zcorr_absmax"]) < 1e-9
    np.testing.assert_allclose(orc.objective_harmony, g["objective_harmony"], rtol=1e-10)
    np.testing.assert_allclose(orc.objective_kmeans, g["objective_kmeans"], rtol=1e-10)
    np.testing.assert_allclose(orc.R.T[::rs], g["R_sub"], atol=1e-11)
    np.testing.assert_allclose(orc.O, g["O"], rtol=1e-9, atol=1e-10)
