"""Host side of sample(..., B200SwendsenWang()): the sampler type, argument refusals that need no device, the loud failure
of the cluster sampler's C entry points without a CUDA device, and the samplers that refuse it."""
import numpy as np
import pytest

import gml_b200
from gml_b200 import _lib
from test_host_api import rerun_without_device


def test_b200swendsenwang_is_its_own_sampler():
    s = gml_b200.B200SwendsenWang()
    assert isinstance(s, gml_b200.GMLSampler)
    assert not isinstance(s, (gml_b200.B200Gibbs, gml_b200.B200Tempering, gml_b200.B200Exact))
    assert (s.seed, s.device, s.chains, s.burn_in, s.thin) == (0, 0, 0, 200, 10) and s.last_rhat == []


def test_host_refusals():
    gm = gml_b200.FactorGraph(2, 3, "spin", {(1, 2): 0.1})
    three = gml_b200.FactorGraph(3, 3, "spin", {(1, 2): 0.1, (1, 2, 3): 0.2})
    S = gml_b200.B200SwendsenWang
    calls = [lambda: gml_b200.sample(gml_b200.FactorGraph(2, 3, "boolean", gm.terms), 10, sampler=S()),
             lambda: gml_b200.sample(gml_b200.FactorGraph(2, 4097, "spin", gm.terms), 10, sampler=S()),
             lambda: gml_b200.sample(gm, 0, sampler=S()),
             lambda: gml_b200.sample(gm, 10, 0, S()),
             lambda: gml_b200.sample(gm, 10, sampler=S(chains=-1)),
             lambda: gml_b200.sample(gm, 10, sampler=S(burn_in=-1)),
             lambda: gml_b200.sample(gm, 10, sampler=S(thin=0)),
             lambda: gml_b200.sample(gm, 2 ** 31, sampler=S()),
             lambda: gml_b200.sample(gml_b200.FactorGraph(2, 3, "spin", {(0, 1): 0.1}), 10, sampler=S()),
             lambda: gml_b200.sample(gm, 10, sampler=S(), return_log_z=True),
             lambda: gml_b200.sample_device(gm, 10, sampler=S(), return_log_z=True),
             lambda: gml_b200.sample(three, 10, sampler=S()),
             lambda: gml_b200.sample_device(three, 10, sampler=S()),
             lambda: gml_b200.moments(three, S(), 10),
             lambda: gml_b200.moments(gml_b200.FactorGraph(2, 4097, "spin", gm.terms), S(), 10),
             lambda: gml_b200.moments(gm, S()),
             lambda: gml_b200.moments(gm, S(thin=0), 10)]
    for call in calls:
        with pytest.raises(ValueError):
            call()


def test_samplers_without_cluster_moves_refuse_it():
    """log_partition, log_likelihood and fit_likelihood have no Swendsen-Wang form: their TypeError paths refuse it."""
    gm = gml_b200.FactorGraph(2, 3, "spin", {(1, 2): 0.1})
    samples = np.array([[5, 1, 1, -1], [3, -1, 1, 1]])
    S = gml_b200.B200SwendsenWang
    for call in (lambda: gml_b200.log_partition(gm, S()), lambda: gml_b200.log_likelihood(gm, samples, S()),
                 lambda: gml_b200.fit_likelihood(gm, samples, S())):
        with pytest.raises(TypeError):
            call()


def test_cluster_entries_fail_loudly_without_device(request):
    lib = _lib.load()
    if lib.gml_b200_device_count() > 0:
        rerun_without_device(request)
        return
    K, mean = np.zeros(1, dtype=np.int64), np.zeros(2)
    key_idx = np.array([[0, 1], [2, -1]], dtype=np.int32)

    def terms(kind):
        if kind == "three":
            return 3, np.array([[0, 1, 2]], dtype=np.int32), np.array([0.3])
        return 2, np.array([[0, 1], [2, -1]], dtype=np.int32), np.array([0.3, -0.1])

    def sample(N=3, n=100, thin=1, burn_in=10, chains=0, kind="pair"):
        order, idx, wts = terms(kind)
        return lib.gml_b200_sample_cluster_device(0, N, order, len(wts), idx.ctypes.data, wts.ctypes.data, n, 1, chains,
                                                  burn_in, thin, 0, K.ctypes.data, None, None, None, 0, None)

    def moments(N=3, n=100, thin=1, burn_in=10, chains=0, kind="pair"):
        order, idx, wts = terms(kind)
        return lib.gml_b200_moments_cluster(0, N, order, len(wts), idx.ctypes.data, wts.ctypes.data, n, chains, burn_in, thin,
                                            0, 2, 2, key_idx.ctypes.data, mean.ctypes.data, None, None, None)

    for call in (sample, moments):
        assert call() == _lib.ECUDA
        # input errors are found before the device is touched
        assert call(N=4097) == _lib.EINVAL
        assert call(N=2) == _lib.EINVAL          # spin index 2 outside [0, N)
        assert call(n=0) == _lib.EINVAL
        assert call(thin=0) == _lib.EINVAL
        assert call(burn_in=-1) == _lib.EINVAL
        assert call(chains=-1) == _lib.EINVAL
        assert call(kind="three") == _lib.EINVAL
        # the counters: (burn_in + records * thin) * (n_terms + N + 1) reaches 2^62 with one chain and these sizes
        assert call(n=2 ** 30, chains=1, thin=2 ** 30) == _lib.EINVAL
