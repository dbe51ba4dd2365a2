"""Host side of log_partition(gm, sampler): the argument refusals that need no device, and the loud failure of the
partition-function C entry point without a CUDA device."""
import numpy as np
import pytest

import gml_b200
from gml_b200 import _lib
from test_host_api import rerun_without_device


def test_host_refusals():
    gm = gml_b200.FactorGraph(2, 3, "spin", {(1, 2): 0.1})
    T = gml_b200.B200Tempering
    value_errors = [lambda: gml_b200.log_partition(gm, gml_b200.B200Gibbs()),
                    lambda: gml_b200.log_partition(gml_b200.FactorGraph(2, 3, "boolean", gm.terms)),
                    lambda: gml_b200.log_partition(gml_b200.FactorGraph(2, 4097, "spin", gm.terms)),
                    lambda: gml_b200.log_partition(gml_b200.FactorGraph(2, 41, "spin", gm.terms), gml_b200.B200Exact()),
                    lambda: gml_b200.log_partition(gm, sweeps=0),
                    lambda: gml_b200.log_partition(gm, T(chains=1)),
                    lambda: gml_b200.log_partition(gm, T(chains=-1)),
                    lambda: gml_b200.log_partition(gm, T(burn_in=-1)),
                    lambda: gml_b200.log_partition(gml_b200.FactorGraph(2, 3, "spin", {(0, 1): 0.1}))]
    # ladders the sampler refuses, and ladders it takes that do not end at beta = 0 (the sampling default among them)
    for betas in ([1.0], [1.0, 0.5, 0.0], [1.0, 0.5], [0.5, 0.0], [1.0, 0.0, 0.5, 0.0], [1.0, -0.0, 0.0, -0.5],
                  list(np.geomspace(1.0, 0.1, 16)), [1.0, float("nan")]):
        value_errors.append(lambda b=betas: gml_b200.log_partition(gm, T(betas=b)))
    for call in value_errors:
        with pytest.raises(ValueError):
            call()
    for sampler in (gml_b200.Gibbs(), gml_b200.GMLSampler(), "B200Tempering", 0):
        with pytest.raises(TypeError):
            gml_b200.log_partition(gm, sampler)


def test_log_partition_fails_loudly_without_device(request):
    lib = _lib.load()
    if lib.gml_b200_device_count() > 0:
        rerun_without_device(request)
        return
    idx = np.array([[0, 1], [2, -1]], dtype=np.int32)
    log_z, stderr = np.zeros(1), np.zeros(1)

    def call(N=3, order=2, ti=idx, w=(0.3, -0.1), betas=np.array([1.0, 0.5, 0.25, 0.0]), n_rungs=None, chains=0, burn_in=10,
             sweeps=100, out=log_z, n_terms=2):
        n_rungs = (0 if betas is None else len(betas)) if n_rungs is None else n_rungs
        wts = np.array(w, dtype=np.float64)
        return lib.gml_b200_log_partition_tempering(0, N, order, n_terms, ti.ctypes.data, wts.ctypes.data, n_rungs,
                                                    None if betas is None else betas.ctypes.data, chains, burn_in, sweeps, 0,
                                                    None if out is None else out.ctypes.data, stderr.ctypes.data, None, None,
                                                    None)

    assert call() == _lib.ECUDA
    assert call(betas=None) == _lib.ECUDA               # the default ladder
    assert call(chains=2) == _lib.ECUDA
    assert call(n_terms=0) == _lib.ECUDA                # no terms: log Z = N log 2, still run on the device
    # input errors are found before the device is touched
    bad = [dict(N=0), dict(N=4097), dict(N=2),            # N = 2: spin index 2 outside [0, N)
           dict(order=0, ti=np.array([[0]], dtype=np.int32), w=(0.3,), n_terms=1),
           dict(order=9, ti=np.arange(9, dtype=np.int32)[None, :], w=(0.3,), n_terms=1),
           dict(ti=np.array([[0, -2], [2, -1]], dtype=np.int32)), dict(ti=np.array([[1, 1], [2, -1]], dtype=np.int32)),
           dict(w=(float("inf"), 0.1)), dict(w=(0.3, float("nan"))),
           dict(chains=1), dict(chains=-1), dict(chains=2 ** 31 + 1), dict(burn_in=-1), dict(sweeps=0), dict(out=None),
           dict(N=4096, sweeps=2 ** 50),                 # 4096 * 2^50 = 2^62 site steps
           dict(betas=np.array([1.0, 0.5])), dict(betas=np.geomspace(1.0, 0.1, 16)), dict(betas=np.array([1.0])),
           dict(betas=np.array([1.0, 0.5, 0.0])), dict(betas=None, n_rungs=2), dict(betas=np.array([1.0, 0.0]), n_rungs=0),
           dict(betas=np.array([0.5, 0.0])), dict(betas=np.array([1.0, 1.0, 0.5, 0.0])),
           dict(betas=np.array([1.0, 0.5, 0.7, 0.0])), dict(betas=np.array([1.0, 0.5, -0.5, 0.0])),
           dict(betas=np.array([1.0, np.nan, 0.5, 0.0])), dict(betas=np.linspace(1.0, 0.0, 64))]
    for kw in bad:
        assert call(**kw) == _lib.EINVAL, kw
