"""Host side of sample(): the reference's sampler types, argument refusals that need no device, and the loud failure of the
exact sampler's C entry point without a CUDA device."""
import numpy as np
import pytest

import gml_b200
from gml_b200 import _lib
from test_host_api import rerun_without_device


def test_gibbs_sampler_is_rejected_like_nlp():
    gm = gml_b200.FactorGraph(2, 3, "spin", {(1, 2): 0.1})
    assert isinstance(gml_b200.Gibbs(), gml_b200.GMLSampler) and isinstance(gml_b200.B200Exact(), gml_b200.GMLSampler)
    with pytest.raises(NotImplementedError, match="B200Exact"):
        gml_b200.sample(gm, 10, 1, gml_b200.Gibbs())
    with pytest.raises(NotImplementedError, match="B200Exact"):
        gml_b200.sample_device(gm, 10, 1, gml_b200.Gibbs())


def test_host_refusals():
    gm = gml_b200.FactorGraph(2, 3, "spin", {(1, 2): 0.1})
    for call in (lambda: gml_b200.sample(gml_b200.FactorGraph(2, 3, "boolean", gm.terms), 10),    # src/sampling.jl:95-97
                 lambda: gml_b200.sample(gml_b200.FactorGraph(2, 41, "spin", gm.terms), 10),
                 lambda: gml_b200.sample(gm, 0),
                 lambda: gml_b200.sample(gm, 10, 0),
                 lambda: gml_b200.sample(gml_b200.FactorGraph(2, 3, "spin", {(0, 1): 0.1}), 10)):
        with pytest.raises(ValueError):
            call()


def test_exact_sampler_fails_loudly_without_device(request):
    lib = _lib.load()
    if lib.gml_b200_device_count() > 0:
        rerun_without_device(request)
        return
    idx = np.array([[0, 1], [2, -1]], dtype=np.int32)
    wts = np.array([0.3, -0.1])
    K = np.zeros(1, dtype=np.int64)
    rc = lib.gml_b200_sample_exact_device(0, 3, 2, 2, idx.ctypes.data, wts.ctypes.data, 100, 1, 0, K.ctypes.data, None,
                                          None, None, 0, None)
    assert rc == _lib.ECUDA
    # input errors are found before the device is touched
    rc = lib.gml_b200_sample_exact_device(0, 41, 2, 2, idx.ctypes.data, wts.ctypes.data, 100, 1, 0, K.ctypes.data, None,
                                          None, None, 0, None)
    assert rc == _lib.EINVAL
