"""Host side of moments / empirical_moments / log_likelihood: the argument refusals that need no device, and the loud
failure of the moments C entry points without a CUDA device."""
import numpy as np
import pytest

import gml_b200
from gml_b200 import B200Exact, B200Gibbs, B200Tempering, FactorGraph, _lib
from test_host_api import rerun_without_device


def test_host_refusals():
    gm = FactorGraph(2, 3, "spin", {(1, 2): 0.1, (3,): -0.2})
    data = np.array([[2, 1, -1, 1], [1, -1, -1, 1]])
    value_errors = [
        lambda: gml_b200.moments(FactorGraph(2, 3, "boolean", gm.terms)),
        lambda: gml_b200.moments(gm, B200Exact(), 10),                      # number_sample with B200Exact
        lambda: gml_b200.moments(gm, None, 10),
        lambda: gml_b200.moments(gm, B200Gibbs()),                           # number_sample missing
        lambda: gml_b200.moments(gm, B200Tempering()),
        lambda: gml_b200.moments(gm, B200Gibbs(), 0),
        lambda: gml_b200.moments(gm, B200Gibbs(thin=0), 10),
        lambda: gml_b200.moments(gm, B200Tempering(chains=-1), 10),
        lambda: gml_b200.moments(gm, B200Tempering(betas=[1.0, 0.5, 0.1]), 10),
        lambda: gml_b200.moments(FactorGraph(2, 41, "spin", gm.terms)),      # above the exact cap
        lambda: gml_b200.moments(FactorGraph(2, 4097, "spin", gm.terms), B200Gibbs(), 10),
        lambda: gml_b200.moments(FactorGraph(2, 3, "spin", {}), B200Gibbs(), 10),   # no terms, no keys
        lambda: gml_b200.empirical_moments(data, "all"),
        lambda: gml_b200.empirical_moments(np.array([1, 1, 1])),              # not a K x (N+1) matrix
        lambda: gml_b200.log_likelihood(FactorGraph(2, 4, "spin", gm.terms), data),
    ]
    bad_keys = [[], [()], [(1, 1)], [(0,)], [(4,)], [(1, 2, 3, 1)], [tuple(range(1, 10))], "diagonal"]
    for keys in bad_keys:
        value_errors.append(lambda k=keys: gml_b200.moments(gm, keys=k))
        value_errors.append(lambda k=keys: gml_b200.moments(gm, B200Gibbs(), 10, keys=k))
        value_errors.append(lambda k=keys: gml_b200.empirical_moments(data, k))
    for call in value_errors:
        with pytest.raises(ValueError):
            call()
    for sampler in (gml_b200.GMLSampler(), "B200Gibbs", 0):
        with pytest.raises(TypeError):
            gml_b200.moments(gm, sampler, 10)
    with pytest.raises(NotImplementedError):
        gml_b200.moments(gm, gml_b200.Gibbs(), 10)


def test_moments_fail_loudly_without_device(request):
    lib = _lib.load()
    if lib.gml_b200_device_count() > 0:
        rerun_without_device(request)
        return
    idx = np.array([[0, 1], [2, -1]], dtype=np.int32)
    keys = np.array([[0, 2], [1, -1]], dtype=np.int32)
    mean, err, rhat, swap = np.zeros(64), np.zeros(64), np.zeros(2), np.zeros(31)

    def mcmc(N=3, order=2, ti=idx, w=(0.3, -0.1), n_rungs=1, betas=None, n=100, chains=0, burn_in=10, thin=1, key_order=2,
             n_keys=2, ki=keys, out=mean):
        wts = np.array(w, dtype=np.float64)
        return lib.gml_b200_moments_mcmc(0, N, order, len(wts), ti.ctypes.data, wts.ctypes.data, n_rungs,
                                         None if betas is None else betas.ctypes.data, n, chains, burn_in, thin, 0, key_order,
                                         n_keys, None if ki is None else ki.ctypes.data, None if out is None else out.ctypes.data,
                                         err.ctypes.data, rhat.ctypes.data, swap.ctypes.data, None)

    def exact(N=3, order=2, ti=idx, w=(0.3, -0.1), key_order=2, n_keys=2, ki=keys, out=mean):
        wts = np.array(w, dtype=np.float64)
        return lib.gml_b200_moments_exact(0, N, order, len(wts), ti.ctypes.data, wts.ctypes.data, key_order, n_keys,
                                          None if ki is None else ki.ctypes.data, None if out is None else out.ctypes.data, None)

    # valid calls reach the device
    assert mcmc() == _lib.ECUDA
    assert mcmc(n_keys=_lib.KEYS_PAIRWISE, ki=None) == _lib.ECUDA
    assert mcmc(n_rungs=0) == _lib.ECUDA                                  # the default tempering ladder
    assert mcmc(n_rungs=4, betas=np.array([1.0, 0.5, 0.25, 0.0])) == _lib.ECUDA
    assert exact() == _lib.ECUDA
    assert exact(n_keys=_lib.KEYS_PAIRWISE, ki=None) == _lib.ECUDA
    # bad input is found before the device is touched
    bad_keys = [dict(n_keys=0), dict(n_keys=-2), dict(ki=None), dict(key_order=0), dict(key_order=9, n_keys=1,
                ki=np.arange(9, dtype=np.int32)[None, :] % 3), dict(ki=np.array([[0, 3], [1, -1]], dtype=np.int32)),
                dict(ki=np.array([[0, 0], [1, -1]], dtype=np.int32)), dict(ki=np.array([[-1, -1], [1, -1]], dtype=np.int32)),
                dict(ki=np.array([[0, -2], [1, -1]], dtype=np.int32)), dict(n_keys=_lib.KEYS_PAIRWISE), dict(out=None)]
    for kw in bad_keys:
        assert mcmc(**kw) == _lib.EINVAL, kw
        assert exact(**kw) == _lib.EINVAL, kw
    bad_mcmc = [dict(N=0), dict(N=4097), dict(N=2), dict(w=(float("nan"), 0.1)), dict(n=0), dict(chains=-1),
                dict(chains=2 ** 31 + 1), dict(burn_in=-1), dict(thin=0), dict(n_rungs=1, betas=np.array([1.0])),
                dict(n_rungs=3, betas=np.array([1.0, 0.5, 0.1])), dict(n_rungs=2, betas=np.array([0.5, 0.1])),
                dict(n_rungs=2, betas=None), dict(N=4096, n=2 ** 50, chains=1)]
    for kw in bad_mcmc:
        assert mcmc(**kw) == _lib.EINVAL, kw
    for kw in (dict(N=0), dict(N=41), dict(N=2), dict(w=(float("inf"), 0.1)),
               dict(ti=np.array([[1, 1], [2, -1]], dtype=np.int32))):
        assert exact(**kw) == _lib.EINVAL, kw
    # a null handle, and keys checked like the model entries would need a resident histogram first
    assert lib.gml_b200_moments_histogram(None, 0, _lib.KEYS_PAIRWISE, None, mean.ctypes.data) == _lib.EINVAL
