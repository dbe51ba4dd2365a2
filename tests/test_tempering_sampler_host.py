"""Host side of sample(..., B200Tempering()): the sampler type, argument refusals that need no device, and the loud failure
of the replica-exchange sampler's C entry point without a CUDA device."""
import numpy as np
import pytest

import gml_b200
from gml_b200 import _lib
from test_host_api import rerun_without_device


def test_b200tempering_is_a_sampler():
    s = gml_b200.B200Tempering()
    assert isinstance(s, gml_b200.GMLSampler)
    assert (s.seed, s.device, s.chains, s.burn_in, s.thin, s.betas) == (0, 0, 0, 200, 10, None)
    assert s.last_rhat == [] and s.last_swap_rate == []


def test_host_refusals():
    gm = gml_b200.FactorGraph(2, 3, "spin", {(1, 2): 0.1})
    T = gml_b200.B200Tempering
    calls = [lambda: gml_b200.sample(gml_b200.FactorGraph(2, 3, "boolean", gm.terms), 10, sampler=T()),
             lambda: gml_b200.sample(gml_b200.FactorGraph(2, 4097, "spin", gm.terms), 10, sampler=T()),
             lambda: gml_b200.sample(gm, 0, sampler=T()),
             lambda: gml_b200.sample(gm, 10, 0, T()),
             lambda: gml_b200.sample(gm, 10, sampler=T(chains=-1)),
             lambda: gml_b200.sample(gm, 10, sampler=T(burn_in=-1)),
             lambda: gml_b200.sample(gm, 10, sampler=T(thin=0)),
             lambda: gml_b200.sample(gm, 2 ** 31, sampler=T()),
             lambda: gml_b200.sample(gml_b200.FactorGraph(2, 3, "spin", {(0, 1): 0.1}), 10, sampler=T()),
             lambda: gml_b200.sample(gm, 10, sampler=T(), return_log_z=True),
             lambda: gml_b200.sample_device(gm, 10, sampler=T(), return_log_z=True)]
    for betas in ([1.0], [1.0, 0.8, 0.5], [1.0] + list(np.linspace(0.9, 0.1, 63)), [0.9, 0.5],
                  [1.0, 1.0], [1.0, 0.5, 0.6, 0.1], [1.0, 0.5, 0.2, -0.1], [1.0, float("nan")], [1.0, float("inf")]):
        calls.append(lambda b=betas: gml_b200.sample(gm, 10, sampler=T(betas=b)))
    for call in calls:
        with pytest.raises(ValueError):
            call()


def test_tempering_sampler_fails_loudly_without_device(request):
    lib = _lib.load()
    if lib.gml_b200_device_count() > 0:
        rerun_without_device(request)
        return
    idx = np.array([[0, 1], [2, -1]], dtype=np.int32)
    wts = np.array([0.3, -0.1])
    K = np.zeros(1, dtype=np.int64)

    def call(N=3, n=100, thin=1, betas=np.array([1.0, 0.5]), n_rungs=None):
        n_rungs = len(betas) if n_rungs is None else n_rungs
        return lib.gml_b200_sample_tempering_device(0, N, 2, 2, idx.ctypes.data, wts.ctypes.data, n_rungs,
                                                    None if betas is None else betas.ctypes.data, n, 1, 0, 10, thin, 0,
                                                    K.ctypes.data, None, None, None, None, 0, None)

    assert call() == _lib.ECUDA
    assert call(betas=None, n_rungs=0) == _lib.ECUDA          # the default ladder
    # input errors are found before the device is touched
    assert call(N=4097) == _lib.EINVAL
    assert call(N=2) == _lib.EINVAL          # spin index 2 outside [0, N)
    assert call(n=0) == _lib.EINVAL
    assert call(thin=0) == _lib.EINVAL
    for betas, n_rungs in ((np.array([1.0, 0.5, 0.2]), None), (np.array([1.0]), None), (None, 2), (np.array([1.0, 0.5]), 0),
                           (np.array([0.5, 0.2]), None), (np.array([1.0, 1.0]), None), (np.array([1.0, -0.5]), None),
                           (np.array([1.0, np.nan]), None), (np.array([1.0, 0.5, 0.7, 0.1]), None)):
        assert call(betas=betas, n_rungs=n_rungs) == _lib.EINVAL, (betas, n_rungs)
