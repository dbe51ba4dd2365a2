"""Host side of sample(..., B200Gibbs()): the sampler type, argument refusals that need no device, and the loud failure of
the MCMC sampler's C entry point without a CUDA device."""
import numpy as np
import pytest

import gml_b200
from gml_b200 import _lib
from test_host_api import rerun_without_device


def test_b200gibbs_is_a_sampler():
    s = gml_b200.B200Gibbs()
    assert isinstance(s, gml_b200.GMLSampler)
    assert (s.seed, s.device, s.chains) == (0, 0, 0) and s.burn_in >= 0 and s.thin >= 1 and s.last_rhat == []


def test_host_refusals():
    gm = gml_b200.FactorGraph(2, 3, "spin", {(1, 2): 0.1})
    G = gml_b200.B200Gibbs
    for call in (lambda: gml_b200.sample(gml_b200.FactorGraph(2, 3, "boolean", gm.terms), 10, sampler=G()),
                 lambda: gml_b200.sample(gml_b200.FactorGraph(2, 4097, "spin", gm.terms), 10, sampler=G()),
                 lambda: gml_b200.sample(gm, 0, sampler=G()),
                 lambda: gml_b200.sample(gm, 10, 0, G()),
                 lambda: gml_b200.sample(gm, 10, sampler=G(chains=-1)),
                 lambda: gml_b200.sample(gm, 10, sampler=G(burn_in=-1)),
                 lambda: gml_b200.sample(gm, 10, sampler=G(thin=0)),
                 lambda: gml_b200.sample(gm, 2 ** 31, sampler=G()),
                 lambda: gml_b200.sample(gml_b200.FactorGraph(2, 3, "spin", {(0, 1): 0.1}), 10, sampler=G()),
                 lambda: gml_b200.sample(gm, 10, sampler=G(), return_log_z=True),
                 lambda: gml_b200.sample_device(gm, 10, sampler=G(), return_log_z=True)):
        with pytest.raises(ValueError):
            call()


def test_mcmc_sampler_fails_loudly_without_device(request):
    lib = _lib.load()
    if lib.gml_b200_device_count() > 0:
        rerun_without_device(request)
        return
    idx = np.array([[0, 1], [2, -1]], dtype=np.int32)
    wts = np.array([0.3, -0.1])
    K = np.zeros(1, dtype=np.int64)

    def call(N=3, n=100, thin=1):
        return lib.gml_b200_sample_mcmc_device(0, N, 2, 2, idx.ctypes.data, wts.ctypes.data, n, 1, 0, 10, thin, 0,
                                               K.ctypes.data, None, None, None, 0, None)

    assert call() == _lib.ECUDA
    # input errors are found before the device is touched
    assert call(N=4097) == _lib.EINVAL
    assert call(N=2) == _lib.EINVAL          # spin index 2 outside [0, N)
    assert call(n=0) == _lib.EINVAL
    assert call(thin=0) == _lib.EINVAL
