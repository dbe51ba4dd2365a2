"""CPU-side checks: the C-ABI library loads and exports every symbol include/gml_b200.h declares, the
host mirror of the reference interface behaves like the reference, and the product path fails loudly
(no CPU fallback) when there is no CUDA device."""
import ctypes
import os
import pathlib
import re
import subprocess
import sys

import numpy as np
import pytest

import gml_b200
from gml_b200 import _lib

ROOT = pathlib.Path(__file__).resolve().parent.parent


def rerun_without_device(request):
    """On a machine with a CUDA device, runs the calling test again in a child pytest that sees none
    (CUDA_VISIBLE_DEVICES=""), so the no-device behaviour is checked there too."""
    assert os.environ.get("CUDA_VISIBLE_DEVICES") != "", "a device is visible with CUDA_VISIBLE_DEVICES=\"\""
    res = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", f"{request.path}::{request.node.name}"], cwd=ROOT,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "1 passed" in res.stdout, res.stdout[-4000:] + res.stderr[-2000:]


def test_library_exports_every_header_symbol():
    header = (ROOT / "include" / "gml_b200.h").read_text()
    declared = set(re.findall(r"\b(gml_b200_[a-z_0-9]+)\s*\(", header))
    assert declared, "no declarations found"
    lib = _lib.load()
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in gml_b200.h but not exported"
    assert declared == set(_lib.EXPORTS)
    assert b"sm_100a" in lib.gml_b200_version()


def test_struct_sizes_match_header():
    # gml_b200_opts: 2 doubles, 6 int32, pointer, 8 int32 ; gml_b200_stats: see header
    assert ctypes.sizeof(_lib.Opts) == 2 * 8 + 6 * 4 + 8 + 8 * 4
    assert ctypes.sizeof(_lib.Stats) == 6 * 4 + 8 + 7 * 8 + 4 * 8


def test_defaults_match_reference():
    # src/GraphicalModelLearning.jl:28,35,49,56
    assert (gml_b200.RISE().regularizer, gml_b200.RISE().symmetrization) == (0.4, True)
    assert gml_b200.logRISE().regularizer == 0.8
    assert gml_b200.RPLE().regularizer == 0.2
    m = gml_b200.multiRISE()
    assert (m.regularizer, m.symmetrization, m.interaction_order) == (0.4, True, 2)


def test_lambda_and_data_info(golden):
    s = golden("mvt_samples.csv")
    k, n, m = gml_b200.data_info(s)
    assert (k, n, m) == (512, 9, 100_000_000)
    lam = gml_b200.regularizer_lambda(0.2, n, m)
    assert abs(lam - 0.2 * np.sqrt(np.log(81 / 0.05) / 1e8)) < 1e-18


def test_pack_histogram_layout_and_validation(golden):
    s = golden("c_samples.csv")
    counts, spins = gml_b200.pack_histogram(s)
    assert counts.dtype == np.float64 and spins.dtype == np.int8
    assert spins.shape == (4, s.shape[0]) and spins.flags["C_CONTIGUOUS"]
    assert np.array_equal(spins.T, s[:, 1:])
    # transposed input (the Adjoint the reference's sample() returns, sampling.jl:54) is accepted
    c2, s2 = gml_b200.pack_histogram(np.asfortranarray(s.astype(np.int64)))
    assert np.array_equal(c2, counts) and np.array_equal(s2, spins)
    bad = s.copy(); bad[0, 1] = 0.5
    with pytest.raises(ValueError):
        gml_b200.pack_histogram(bad)


def test_multirise_key_order():
    # (u,), (u,j) ascending, (u,j<k) lexicographic  (src/GraphicalModelLearning.jl:94-104, models.jl:228-246)
    assert gml_b200.multirise_keys(4, 2, 3) == [(2,), (2, 1), (2, 3), (2, 4), (2, 1, 3), (2, 1, 4), (2, 3, 4)]
    lib = _lib.load()
    assert lib.gml_b200_multibody_num_keys(30, 3) == 1 + 29 + 406
    assert lib.gml_b200_multibody_num_keys(4, 4) == 1 + 3 + 3 + 1


def test_factor_graph_round_trip():
    # test/runtests.jl:17-30
    from helpers import MODELS
    for m in MODELS.values():
        gm = gml_b200.FactorGraph.from_matrix(m)
        assert np.allclose(gm.to_matrix(), m)
        for key, v in gm:
            assert np.isclose(v, m[key[0] - 1, key[-1] - 1])
    assert len(gml_b200.matrix_to_dict(MODELS["b"])) == 9


def test_nlp_method_is_rejected(golden):
    with pytest.raises(NotImplementedError):
        gml_b200.learn(golden("a_samples.csv"), gml_b200.RISE(), gml_b200.NLP())


def test_no_cpu_fallback(golden, request):
    """Without a CUDA device the product must fail loudly, never compute on the CPU."""
    lib = _lib.load()
    if lib.gml_b200_device_count() > 0:
        rerun_without_device(request)
        return
    with pytest.raises(gml_b200.GMLB200Error) as e:
        gml_b200.learn(golden("a_samples.csv"))
    assert e.value.code == _lib.ECUDA and "no CPU fallback" in str(e.value)


def test_matrix_entry_fails_loudly_without_device_and_validates_layout(golden, request):
    """The reference-typed entry (Fortran-ordered K x (N+1) matrix) has no CPU path either; layout errors are host errors."""
    s = np.asfortranarray(golden("a_samples.csv"))
    with pytest.raises(ValueError):
        gml_b200.learn_matrix(np.ascontiguousarray(golden("c_samples.csv")), gml_b200.RISE(), gml_b200.B200())   # row-major
    with pytest.raises(ValueError):
        gml_b200.learn_matrix(s.astype(np.float16, order="F"), gml_b200.RISE(), gml_b200.B200())
    lib = _lib.load()
    if lib.gml_b200_device_count() > 0:
        rerun_without_device(request)
        return
    with pytest.raises(gml_b200.GMLB200Error) as e:
        gml_b200.learn(s, gml_b200.RISE(), gml_b200.B200())        # F-ordered input takes the matrix entry
    assert e.value.code == _lib.ECUDA
