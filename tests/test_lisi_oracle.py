"""The LISI oracle (oracle/lisi_oracle.py) against the reference's own known-answer test and against outputs of
the unmodified reference (tests/golden/make_golden_lisi.py).  CPU only."""
import os

import numpy as np
import pandas as pd
import pytest

from oracle.lisi_oracle import compute_lisi, compute_simpson, knn_exact

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _meta(g):
    return pd.DataFrame({str(c): pd.Categorical.from_codes(g["codes"][i], categories=list(range(int(g["n_categories"][i]))))
                         for i, c in enumerate(g["columns"])})


def test_oracle_matches_the_reference_known_answer_test():
    """tests/test_lisi.py:5-17 of the reference: np.allclose against data/lisi_lisi.tsv.gz (values from the R package)."""
    g = np.load(os.path.join(GOLDEN, "lisi_kat.npz"))
    got = compute_lisi(g["X"], _meta(g), [str(c) for c in g["columns"]], float(g["perplexity"]))
    assert got.shape == g["lisi_expected"].shape == (400, 2)
    assert np.allclose(got, g["lisi_expected"])                            # the reference's own criterion
    np.testing.assert_allclose(got, g["lisi_reference_python"], rtol=1e-10, atol=0)   # and its Python code, tightly


def test_oracle_matches_reference_on_pbmc_pcs():
    g = np.load(os.path.join(GOLDEN, "lisi_pbmc.npz"))
    got = compute_lisi(g["X"].astype(np.float64), _meta(g), ["donor"], 30)
    np.testing.assert_allclose(got, g["lisi_reference_python"], rtol=1e-9, atol=0)
    assert 1.0 - 1e-9 <= got.min() and got.max() <= int(g["n_categories"][0]) + 1e-9


def test_knn_exact_is_sorted_and_contains_self_first():
    rng = np.random.default_rng(0)
    X = rng.normal(size=(300, 5))
    d, i = knn_exact(X, 20, chunk=64)
    assert (i[:, 0] == np.arange(300)).all() and (d[:, 0] == 0).all()
    assert (np.diff(d, axis=1) >= 0).all()
    full = np.sqrt(((X[:, None, :] - X[None, :, :]) ** 2).sum(-1))
    np.testing.assert_allclose(d, np.sort(full, axis=1)[:, :20], rtol=1e-12)


def test_simpson_edge_cases_follow_the_reference():
    # all neighbours at distance 0: P is uniform whatever beta is, H = log(k) != log(perplexity): 50 tries, no crash
    k, n = 89, 3
    D = np.zeros((k, n))
    idx = np.tile(np.arange(k)[:, None], (1, n))
    codes = np.arange(k) % 2
    s = compute_simpson(D, idx, codes, 2, 30.0)
    np.testing.assert_allclose(s, (45 / 89) ** 2 + (44 / 89) ** 2, rtol=1e-12)
    # neighbours so far away that exp underflows at beta = 1 (lisi.py:88-90): halving beta recovers a finite answer
    D = np.full((k, n), 1e4) + np.arange(k)[:, None]
    s = compute_simpson(D, idx, codes, 2, 30.0)
    assert np.isfinite(s).all() and (s > 0).all()


RANDOM_CASES = [(600, 3, 30, 0), (900, 20, 15, 1), (500, 8, 42, 2)]


def _random_problem(n, d, seed):
    rng = np.random.default_rng(seed)
    t = rng.integers(0, 4, n)
    X = rng.normal(size=(4, d))[t] * 2.5 + rng.normal(size=(n, d))
    meta = pd.DataFrame({"type": pd.Categorical(t.astype(str)), "batch": pd.Categorical(rng.integers(0, 3, n).astype(str)),
                         "one": pd.Categorical(["a"] * n)})
    return X, meta


@pytest.mark.parametrize("n,d,perp,seed", RANDOM_CASES)
def test_oracle_equals_live_reference_on_random_data(n, d, perp, seed):
    """Against what the unmodified reference's compute_lisi returned on the same seeded data
    (tests/golden/make_golden_random.py)."""
    X, meta = _random_problem(n, d, seed)
    want = np.load(os.path.join(GOLDEN, "random_lisi.npz"))[f"seed{seed}_lisi"]
    got = compute_lisi(X, meta, ["type", "batch", "one"], perp)
    np.testing.assert_allclose(got, want, rtol=1e-9)
    np.testing.assert_allclose(got[:, 2], 1.0, rtol=1e-12)          # a single category: LISI = 1 everywhere
