"""CPU-side checks of the drop-in boundary: the library builds, loads, exports every symbol
include/harmony_b200.h declares, and refuses to run without a GPU (no silent CPU fallback)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from harmonypy_b200.build import build
    build(verbose=False)
    from harmonypy_b200 import _cabi
    return _cabi.load()


def header_symbols():
    text = open(os.path.join(ROOT, "include", "harmony_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(hmy_[a-z_0-9]+)\s*\(", text)))


def test_every_declared_symbol_is_exported(lib):
    names = header_symbols()
    assert "hmy_kmeans_round" in names and "hmy_ridge_correct" in names and len(names) >= 18
    for n in names:
        assert hasattr(lib, n), f"{n} declared in the header but not exported"


def test_binding_table_matches_header(lib):
    from harmonypy_b200 import _cabi
    assert sorted(_cabi.SYMBOLS) == header_symbols()


def test_version_string(lib):
    assert b"sm_100a" in lib.hmy_version()


def test_create_fails_loudly_without_gpu(lib):
    """A child process that sees no CUDA device (hidden from it where the machine has one) cannot create an engine."""
    code = ("from harmonypy_b200 import _cabi\n"
            "try:\n"
            "    _cabi.Engine(0, 100, 100, 0, 10, 8, [2])\n"
            "except _cabi.EngineError as e:\n"
            "    assert 'hmy_create' in str(e), e\n"
            "else:\n"
            "    raise SystemExit('an engine was created without a CUDA device')\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


def test_create_validates_arguments(lib):
    h = C.c_void_p()
    lv = np.array([3], dtype=np.int32)
    p = lv.ctypes.data_as(C.POINTER(C.c_int32))
    assert lib.hmy_create(C.byref(h), 0, 100, 100, 0, 300, 10, 1, p) != 0
    assert b"d must be" in lib.hmy_last_error(None)
    assert lib.hmy_create(C.byref(h), 0, 100, 100, 0, 30, 1000, 1, p) != 0
    assert b"K" in lib.hmy_last_error(None)
    assert lib.hmy_create(C.byref(h), 0, 100, 50, 0, 30, 10, 1, p) != 0
    assert b"n_global" in lib.hmy_last_error(None)


def test_lisi_entry_point_validates_and_refuses_to_run_without_gpu(lib):
    import pandas as pd
    import torch
    import harmonypy_b200 as hm
    from harmonypy_b200 import _cabi
    X = np.random.default_rng(0).normal(size=(50, 4))
    meta = pd.DataFrame({"a": pd.Categorical(["x", "y"] * 25)})
    with pytest.raises(_cabi.EngineError, match="fewer cells"):
        hm.compute_lisi(X, meta, ["a"], 30)                       # 90 neighbours of 50 cells (checked before any CUDA call)
    X = np.random.default_rng(0).normal(size=(500, 4))
    meta = pd.DataFrame({"a": pd.Categorical(["x", "y"] * 250)})
    with pytest.raises(_cabi.EngineError, match="perplexity"):
        hm.compute_lisi(X, meta, ["a"], 60)                       # 180 > 128 neighbours
    if not torch.cuda.is_available():
        with pytest.raises(_cabi.EngineError, match="hmy_lisi_compute"):
            hm.compute_lisi(X, meta, ["a"], 30)                   # no CPU fallback
