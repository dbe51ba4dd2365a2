"""Host side of fit_likelihood: the Python refusals that need no device, the loud failure of the two C entry points
without a CUDA device (and EINVAL on bad input before the device is touched), and the float64 oracle mle_exact against
closed forms."""
import math

import numpy as np
import pytest

import gml_b200
import mle_oracle
from gml_b200 import B200Gibbs, B200Tempering, FactorGraph, _lib
from test_host_api import rerun_without_device


def test_host_refusals():
    gm = FactorGraph(2, 3, "spin", {(1, 2): 0.1, (3,): -0.2})
    data = np.array([[2, 1, -1, 1], [1, -1, -1, 1]])
    value_errors = [
        lambda: gml_b200.fit_likelihood(gm, data, B200Tempering()),
        lambda: gml_b200.fit_likelihood(FactorGraph(2, 3, "boolean", gm.terms), data),
        lambda: gml_b200.fit_likelihood(FactorGraph(2, 3, "spin", {}), data),
        lambda: gml_b200.fit_likelihood(FactorGraph(2, 41, "spin", gm.terms), np.ones((1, 42))),    # above the exact cap
        lambda: gml_b200.fit_likelihood(FactorGraph(2, 4097, "spin", gm.terms), np.ones((1, 4098)), B200Gibbs()),
        lambda: gml_b200.fit_likelihood(FactorGraph(2, 4, "spin", gm.terms), data),                  # N differs
        lambda: gml_b200.fit_likelihood(gm, np.array([1, 1, 1])),                                    # not K x (N+1)
        lambda: gml_b200.fit_likelihood(gm, np.array([[0, 1, 1, 1]])),                               # M = 0
        lambda: gml_b200.fit_likelihood(gm, np.array([[-1, 1, 1, 1], [2, 1, 1, 1]])),                # negative count
        lambda: gml_b200.fit_likelihood(gm, data, regularizer=-0.1),
        lambda: gml_b200.fit_likelihood(gm, data, regularizer=float("nan")),
        lambda: gml_b200.fit_likelihood(gm, data, B200Gibbs(), steps=0),
        lambda: gml_b200.fit_likelihood(gm, data, B200Gibbs(), step_size=-0.1),
        lambda: gml_b200.fit_likelihood(gm, data, B200Gibbs(), step_size=float("inf")),
        lambda: gml_b200.fit_likelihood(gm, data, B200Gibbs(chains=-1)),
        lambda: gml_b200.fit_likelihood(gm, data, B200Gibbs(burn_in=-1)),
        lambda: gml_b200.fit_likelihood(gm, data, B200Gibbs(thin=0)),
        lambda: gml_b200.fit_likelihood(gm, data, B200Gibbs(thin=2 ** 30), steps=2 ** 31),       # too many sweeps
        lambda: gml_b200.fit_likelihood(gm, data, tol=0.0),
        lambda: gml_b200.fit_likelihood(gm, data, tol=float("nan")),
        lambda: gml_b200.fit_likelihood(gm, data, max_iter=0),
        lambda: gml_b200.fit_likelihood(FactorGraph(9, 9, "spin", {tuple(range(1, 10)): 0.1}), np.ones((1, 10))),  # > 8 spins
    ]
    for call in value_errors:
        with pytest.raises(ValueError):
            call()
    for sampler in (gml_b200.GMLSampler(), "B200Gibbs", 0):
        with pytest.raises(TypeError):
            gml_b200.fit_likelihood(gm, data, sampler)
    with pytest.raises(NotImplementedError):
        gml_b200.fit_likelihood(gm, data, gml_b200.Gibbs())


def test_fit_entries_fail_loudly_without_device(request):
    lib = _lib.load()
    if lib.gml_b200_device_count() > 0:
        rerun_without_device(request)
        return
    idx = np.array([[0, 1], [2, -1]], dtype=np.int32)
    out, mm, trace, obj, iters = np.zeros(8), np.zeros(8), np.zeros(64), np.zeros(1), np.zeros(1, dtype=np.int32)

    def arrays(w, dm):
        return np.array(w, dtype=np.float64), np.array(dm, dtype=np.float64)

    def mcmc(N=3, order=2, ti=idx, w=(0.3, -0.1), dm=(0.2, -0.4), lam=0.0, chains=0, burn_in=10, thin=1, steps=20, eta=0.1,
             o=out, dm_null=False):
        wts, d = arrays(w, dm)
        return lib.gml_b200_fit_likelihood_mcmc(0, N, order, len(wts), ti.ctypes.data, wts.ctypes.data,
                                                None if dm_null else d.ctypes.data, lam, chains, burn_in, thin, steps, eta, 0,
                                                None if o is None else o.ctypes.data, mm.ctypes.data, trace.ctypes.data, None)

    def exact(N=3, order=2, ti=idx, w=(0.3, -0.1), dm=(0.2, -0.4), lam=0.0, tol=1e-10, max_iter=100, o=out, dm_null=False):
        wts, d = arrays(w, dm)
        return lib.gml_b200_fit_likelihood_exact(0, N, order, len(wts), ti.ctypes.data, wts.ctypes.data,
                                                 None if dm_null else d.ctypes.data, lam, tol, max_iter,
                                                 None if o is None else o.ctypes.data, obj.ctypes.data, iters.ctypes.data, None)

    # valid calls reach the device
    assert mcmc() == _lib.ECUDA
    assert mcmc(eta=0.0) == _lib.ECUDA                                    # step_size = 0 samples gm unchanged
    assert mcmc(dm=(1.0, -0.4), lam=0.01) == _lib.ECUDA                  # lambda bounds the pair
    assert exact() == _lib.ECUDA
    assert exact(dm=(-1.0, -0.4), lam=0.01) == _lib.ECUDA
    # bad input is found before the device is touched
    common = [dict(dm=(1.5, 0.0)), dict(dm=(0.2, -1.01)), dict(dm=(float("nan"), 0.0)), dict(dm=(0.2, float("inf"))),
              dict(dm=(1.0, 0.0)),                                         # the pair at lambda = 0: no finite maximum
              dict(dm=(0.2, -1.0), lam=0.5),                               # a field: lambda does not bound it
              dict(lam=-0.1), dict(lam=float("nan")), dict(lam=float("inf")), dict(dm_null=True), dict(o=None),
              dict(w=()), dict(N=0), dict(N=2), dict(w=(float("nan"), 0.1)),
              dict(ti=np.array([[1, 1], [2, -1]], dtype=np.int32))]
    for kw in common:
        assert mcmc(**kw) == _lib.EINVAL, kw
        assert exact(**kw) == _lib.EINVAL, kw
    for kw in (dict(N=4097), dict(steps=0), dict(eta=-0.1), dict(eta=float("nan")), dict(chains=-1),
               dict(chains=2 ** 31 + 1), dict(burn_in=-1), dict(thin=0), dict(N=4096, steps=2 ** 50, thin=1)):
        assert mcmc(**kw) == _lib.EINVAL, kw
    for kw in (dict(N=41), dict(tol=0.0), dict(tol=-1.0), dict(tol=float("nan")), dict(max_iter=0)):
        assert exact(**kw) == _lib.EINVAL, kw


def test_oracle_fields_closed_form():
    m = np.array([0.3, -0.5, 0.1, 0.0, 0.95])
    w = mle_oracle.mle_exact({(i + 1,): 0.0 for i in range(5)}, 5, m, 0.0)
    assert np.abs(w - np.arctanh(m)).max() <= 1e-12
    # with lambda, fields stay unpenalised
    w = mle_oracle.mle_exact({(i + 1,): 0.5 for i in range(5)}, 5, m, 0.3)
    assert np.abs(w - np.arctanh(m)).max() <= 1e-12


def test_oracle_pair_closed_form():
    for m1, m2, c in [(0.2, -0.3, 0.4), (0.0, 0.0, -0.7), (0.6, 0.5, 0.45)]:
        p = {(a, b): (1 + m1 * a + m2 * b + c * a * b) / 4 for a in (1, -1) for b in (1, -1)}
        J = 0.25 * math.log(p[1, 1] * p[-1, -1] / (p[1, -1] * p[-1, 1]))
        h1 = 0.25 * math.log(p[1, 1] * p[1, -1] / (p[-1, 1] * p[-1, -1]))
        h2 = 0.25 * math.log(p[1, 1] * p[-1, 1] / (p[1, -1] * p[-1, -1]))
        w = mle_oracle.mle_exact({(1,): 0.0, (2,): 0.0, (1, 2): 0.0}, 2, [m1, m2, c], 0.0)
        assert np.abs(w - [h1, h2, J]).max() <= 1e-12, (m1, m2, c)
