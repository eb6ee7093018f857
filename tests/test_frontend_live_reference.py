"""Differential test of the host front end (harmonypy_b200.harmony.prepare_problem) against the reference's
argument normalisation (harmonypy/harmony.py:116-173) over randomised call signatures: orientation of data_mat,
str / list vars_use, theta and lamb as None / scalar / per-covariate / per-level, lamb = -1, tau, nclust, sigma.

What the reference derived, run with max_iter_harmony = 0 (it still normalises every argument and initialises), and
the exception types it raised are stored in tests/golden/random_frontend.npz (tests/golden/make_golden_random.py;
exact arrays as SHA-1 digests).  CPU only."""
import hashlib
import os

import numpy as np
import pandas as pd
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def ref():
    return np.load(os.path.join(GOLDEN, "random_frontend.npz"))


def _digest(a):
    return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def _exc_name(e):
    return f"{type(e).__module__}.{type(e).__qualname__}"


def _data(rng, N, d, levels):
    Z = rng.normal(size=(N, d)).astype(np.float32)
    meta = pd.DataFrame({f"c{v}": [f"lev{int(x):02d}" for x in rng.integers(0, L, N)] for v, L in enumerate(levels)})
    return Z, meta


CALLS = [
    dict(levels=[3], kw=dict()),
    dict(levels=[4, 2], kw=dict(theta=1.5, lamb=0.7, nclust=7)),
    dict(levels=[2, 3], kw=dict(theta=[2.0, 0.5], lamb=[0.3, 3.0], sigma=0.25, nclust=6)),
    dict(levels=[2, 3], kw=dict(theta=[1.0, 2.0, 3.0, 4.0, 5.0], lamb=[1.0, 2.0, 3.0, 4.0, 5.0], nclust=5)),
    dict(levels=[3, 2, 2], kw=dict(lamb=-1, alpha=0.4, tau=11, nclust=9)),
    dict(levels=[5], kw=dict(tau=3, theta=0.0, nclust=4), transpose=True, vars_as_str=True),
    dict(levels=[12], kw=dict(), N=1500),                          # default nclust = min(round(N / 30), 100)
]


@pytest.mark.parametrize("i", range(len(CALLS)))
def test_prepare_problem_equals_reference_normalisation(ref, i):
    from harmonypy_b200.harmony import prepare_problem
    spec = CALLS[i]
    rng = np.random.default_rng(40 + i)
    N = spec.get("N", 400)
    Z, meta = _data(rng, N, 6, spec["levels"])
    vars_use = list(meta.columns)
    if spec.get("vars_as_str"):
        vars_use = vars_use[0]
    data = pd.DataFrame(Z.T if spec.get("transpose") else Z)
    kw = dict(spec["kw"])
    ho = {k[len(f"call{i}_"):]: ref[k] for k in ref.files if k.startswith(f"call{i}_")}
    kw.pop("alpha", None)
    prob, vu = prepare_problem(data, meta, vars_use, kw.get("theta"), kw.get("lamb"), kw.get("sigma", 0.1),
                               kw.get("nclust"), kw.get("tau", 0))
    assert prob.K == ho["K"] and prob.N == ho["N"] and prob.d == ho["d"] and prob.B == ho["B"]
    assert bool(prob.lambda_estimation) == bool(ho["lambda_estimation"])
    np.testing.assert_allclose(prob.Pr_b, ho["Pr_b"], rtol=1e-6)
    np.testing.assert_allclose(prob.theta, ho["theta"], rtol=1e-6)
    np.testing.assert_allclose(prob.sigma, ho["sigma"], rtol=1e-6)
    if not prob.lambda_estimation:
        np.testing.assert_allclose(prob.lamb, ho["lamb"], rtol=1e-6)
    assert _digest(np.asarray(prob.Z, dtype=np.float32)) == str(ho["Z_orig_digest"])
    # integer codes <-> the reference's dense one-hot, same row order
    from oracle.harmony_oracle import onehot_from_codes
    assert _digest(onehot_from_codes(prob.codes, prob.levels).astype(np.uint8)) == str(ho["Phi_digest"])


BAD_CALLS = [
    dict(kw=dict(theta=[1.0, 2.0, 3.0])),                 # neither per-covariate (2) nor per-level (5)
    dict(kw=dict(), numeric_covariate=True),              # harmony.py:134: numeric column has no .unique categories
    dict(kw=dict(), wrong_shape=True),                    # data_mat matches N on neither axis
]


@pytest.mark.parametrize("i", range(len(BAD_CALLS)))
def test_bad_arguments_raise_the_same_exception_type_as_the_reference(ref, i):
    from harmonypy_b200.harmony import prepare_problem
    spec = BAD_CALLS[i]
    rng = np.random.default_rng(70 + i)
    Z, meta = _data(rng, 300, 5, [2, 3])
    if spec.get("numeric_covariate"):
        meta["c0"] = rng.integers(0, 2, 300)
    if spec.get("wrong_shape"):
        Z = Z[:250, :4]
    kw = spec["kw"]
    theirs = str(ref[f"bad{i}_exception"])
    with pytest.raises(Exception) as ours:
        prepare_problem(pd.DataFrame(Z), meta, list(meta.columns), kw.get("theta"), kw.get("lamb"), 0.1, None, 0)
    assert _exc_name(ours.value) == theirs, (_exc_name(ours.value), theirs)


def test_wrong_length_lambda_fails_earlier_than_in_the_reference(ref):
    """Deliberate difference: the reference does not validate a lamb list that is neither per-covariate nor per-level
    (harmony.py:162-165) and only fails inside the first moe_correct_ridge (shape mismatch in torch); here the front
    end refuses it up front."""
    from harmonypy_b200.harmony import prepare_problem
    rng = np.random.default_rng(5)
    Z, meta = _data(rng, 300, 5, [2, 3])
    assert str(ref["wrong_lamb_exception"]) != "builtins.AssertionError"
    with pytest.raises(AssertionError, match="lambda"):
        prepare_problem(pd.DataFrame(Z), meta, list(meta.columns), None, [1.0, 2.0, 3.0], 0.1, None, 0)
