"""log_partition(gm, B200Tempering()) (gml_b200_log_partition_tempering, csrc/mcmc_sampler.cu with BRIDGE): log Z by
bridge sampling along a replica-exchange ladder that ends at beta = 0, against exact values -- N log 2 without terms,
closed forms for fields, periodic rings and the Curie-Weiss model up to N = 4096, and enumeration (log_partition with
B200Exact) for models up to N = 30 and order 8 -- plus a calibration of the standard error over 64 seeds, the output
contract, and the B200Tempering sampling output pinned to the bytes it had before the estimator existed.  Every seed is
fixed.

Bars: |estimate - exact| <= 5 stderr + sum_t |w_t - fl32(w_t)| (the chains sample the model with fp32-rounded weights),
and the stderr itself under a cap of about 3x the value measured on a B200, which stands next to each cap."""
import ctypes
import hashlib
import math

import numpy as np
import pytest
from scipy import special, stats

import gml_b200
from gml_b200 import B200Exact, B200Tempering, FactorGraph, _lib
from helpers import random_ising, three_body_model
from test_gpu_fullsize import lattice_model
from test_gpu_tempering_sampler import FERRO_4X5, ORDER3_N14, term_arrays

pytestmark = pytest.mark.gpu


def fp32_bound(gm):
    """sum_t |w_t - fl32(w_t)|: the most log Z of the fp32-rounded model can differ from log Z of gm"""
    w = np.array(list(gm.terms.values()), dtype=np.float64)
    return float(np.abs(w - w.astype(np.float32).astype(np.float64)).sum())


def check(name, gm, exact, cap, sampler, sweeps=1000):
    log_z, err, info = gml_b200.log_partition(gm, sampler, sweeps, return_info=True)
    bar = 5.0 * err + fp32_bound(gm)
    print(f"{name}: log Z {log_z:.6f} exact {exact:.6f} error {log_z - exact:+.2e} stderr {err:.2e} (cap {cap:.0e}) "
          f"min swap rate {min(info['swap_rate']):.3f}")
    assert abs(log_z - exact) <= bar
    assert 0.0 < err <= cap


def log_2cosh(x):
    x = np.abs(np.asarray(x, dtype=np.float64))
    return x + np.log1p(np.exp(-2.0 * x))


def ring(n, J):
    return FactorGraph(2, n, "spin", {(i, i + 1): J for i in range(1, n)} | {(1, n): J})


def curie_weiss(n, J):
    return FactorGraph(2, n, "spin", {(i, j): J / n for i in range(1, n + 1) for j in range(i + 1, n + 1)})


def curie_weiss_log_z(n, J):
    k = np.arange(n + 1)
    M = 2.0 * k - n
    t = special.gammaln(n + 1) - special.gammaln(k + 1) - special.gammaln(n - k + 1) + J * (M * M - n) / (2.0 * n)
    return float(special.logsumexp(t))


def order8_model(n=12, seed=8):
    """random terms of every order 1..8 on n spins, weights +-U[0.05, 0.3]"""
    rng = np.random.default_rng(seed)
    terms = {}
    for q in range(1, 9):
        for _ in range(4):
            terms[tuple(sorted(int(x) + 1 for x in rng.choice(n, q, replace=False)))] = float(rng.choice([-1, 1]) *
                                                                                                rng.uniform(0.05, 0.3))
    return FactorGraph(8, n, "spin", terms)


@pytest.mark.parametrize("n", [1, 64, 65, 4096])
def test_no_terms_is_n_log_2(n):
    """E = 0 on every rung: every bridge term is exactly 1, so log Z = N log 2 and the stderr is 0, bit for bit."""
    gm = FactorGraph(2, n, "spin", {})
    log_z, err, info = gml_b200.log_partition(gm, B200Tempering(chains=64, burn_in=2), 5, return_info=True)
    assert log_z == n * math.log(2.0) and err == 0.0
    assert info["log_ratio"] == [0.0] * 31 and info["log_ratio_stderr"] == [0.0] * 31


def test_fields_only():
    rng = np.random.default_rng(1)
    h = rng.integers(-64, 65, 4096) / 64.0                      # dyadic: exact in fp32
    gm = FactorGraph(1, 4096, "spin", {(i + 1,): float(v) for i, v in enumerate(h)})
    check("fields N=4096", gm, float(log_2cosh(h).sum()), 0.04,                # measured stderr 1.29e-2
          B200Tempering(seed=1, chains=512, burn_in=100), 400)


@pytest.mark.parametrize("n,J,cap", [(1000, 1.0, 0.045), (4096, 0.5, 0.04)])   # measured stderr 1.49e-2, 1.29e-2
def test_periodic_ring(n, J, cap):
    exact = float(n * log_2cosh(J) + np.log1p(np.tanh(J) ** n))
    check(f"ring N={n} J={J}", ring(n, J), exact, cap, B200Tempering(seed=2, chains=512, burn_in=100), 400)


@pytest.mark.parametrize("J,cap", [(0.5, 5e-4), (1.5, 0.025)])                  # measured stderr 1.60e-4, 8.15e-3
def test_curie_weiss(J, cap):
    """N = 256, every pair at J / N (dyadic); J = 1.5 is the ordered phase, where the ladder crosses the transition."""
    check(f"Curie-Weiss N=256 J={J}", curie_weiss(256, J), curie_weiss_log_z(256, J), cap,
          B200Tempering(seed=3, chains=1024, burn_in=100), 300)


@pytest.mark.parametrize("name,model,cap", [
    ("ferromagnet 4x5 J=1.5", lambda: FERRO_4X5, 4e-3),                              # measured stderr 1.31e-3
    ("order-3 N=14 x2", lambda: ORDER3_N14, 1.3e-3),                                  # 4.23e-4
    ("random_ising(30, 30)", lambda: FactorGraph.from_matrix(random_ising(30, 30)), 1.3e-3),   # 4.33e-4
    ("order-8 N=12", order8_model, 3e-4),                                             # 9.07e-5
])
def test_against_enumeration(name, model, cap):
    gm = model()
    exact, err0 = gml_b200.log_partition(gm, B200Exact())
    assert err0 == 0.0
    check(name, gm, exact, cap, B200Tempering(seed=4))


def test_stderr_is_calibrated():
    """64 seeds of a short run on ORDER3_N14 against log Z of its fp32-rounded weights (what the chains sample): the
    z-scores have mean 0 within the normal bound and variance 1 within the chi^2(63) bounds, both at rate 1e-6."""
    gm32 = FactorGraph(3, 14, "spin", {k: float(np.float32(v)) for k, v in ORDER3_N14.terms.items()})
    exact = gml_b200.log_partition(gm32, B200Exact())[0]
    z = []
    for seed in range(64):
        log_z, err = gml_b200.log_partition(ORDER3_N14, B200Tempering(seed=100 + seed, chains=256, burn_in=50), 100)
        z.append((log_z - exact) / err)
    z = np.array(z)
    mean_bound = stats.norm.isf(0.5e-6) / math.sqrt(len(z))
    lo, hi = stats.chi2.ppf(0.5e-6, len(z) - 1) / (len(z) - 1), stats.chi2.isf(0.5e-6, len(z) - 1) / (len(z) - 1)
    print(f"calibration: mean z {z.mean():+.3f} (bound {mean_bound:.3f}), var z {z.var(ddof=1):.3f} (bounds {lo:.3f}, {hi:.3f})")
    assert abs(z.mean()) <= mean_bound
    assert lo <= z.var(ddof=1) <= hi


def test_output_contract():
    gm = FactorGraph.from_matrix(random_ising(30, 30))
    make = lambda seed=5: B200Tempering(seed=seed, chains=128, burn_in=50, betas=list(np.linspace(1.0, 0.0, 16)))  # noqa: E731
    log_z, err, info = gml_b200.log_partition(gm, make(), 200, return_info=True)
    assert len(info["log_ratio"]) == len(info["log_ratio_stderr"]) == len(info["swap_rate"]) == 15
    assert info["betas"] == list(np.linspace(1.0, 0.0, 16)) and info["ladders"] == 128 and info["sweeps"] == 200
    assert log_z - 30 * math.log(2.0) == pytest.approx(sum(info["log_ratio"]), rel=1e-12, abs=1e-12)
    assert all(0.0 < r <= 1.0 for r in info["swap_rate"]) and all(e > 0.0 for e in info["log_ratio_stderr"])
    assert err > 0.0
    # bit-identical for the same arguments, different for another seed; None is the default B200Tempering()
    assert gml_b200.log_partition(gm, make(), 200, return_info=True) == (log_z, err, info)
    assert gml_b200.log_partition(gm, make(6), 200) != (log_z, err)
    d = gml_b200.log_partition(gm, None, 20, return_info=True)
    assert d[:2] == gml_b200.log_partition(gm, B200Tempering(), 20)
    assert len(d[2]["betas"]) == _lib.LOG_Z_DEFAULT_RUNGS and d[2]["betas"][-1] == 0.0 and d[2]["ladders"] == 4096
    # thin is ignored; B200Exact gives stderr 0
    assert gml_b200.log_partition(gm, B200Tempering(seed=5, chains=128, burn_in=50, thin=7,
                                                    betas=list(np.linspace(1.0, 0.0, 16))), 200) == (log_z, err)
    small = FactorGraph.from_matrix(random_ising(10, 10))
    assert gml_b200.log_partition(small, B200Exact(), return_info=True)[1:] == (0.0, {})
    # the C entry with null optional outputs writes the same log Z
    order, idx, wts = term_arrays(gm)
    betas = np.linspace(1.0, 0.0, 16)
    out = ctypes.c_double(0.0)
    rc = _lib.load().gml_b200_log_partition_tempering(0, 30, order, len(wts), idx.ctypes.data, wts.ctypes.data, 16,
                                                       betas.ctypes.data, 128, 50, 200, 5, ctypes.byref(out), None, None,
                                                       None, None)
    assert rc == _lib.OK and out.value == log_z


# ---- B200Tempering sampling output, pinned to the bytes of the sampler before the estimator existed ----------------
def tempering_digest(lib, gm, n, reps, seed, chains, burn_in, thin, betas):
    """sha256 prefix of the counts, spins, R-hat and swap rates that gml_b200_sample_tempering_device writes into host
    buffers.  `lib` is any build of the library, so the same digest can be taken from an older one."""
    c = ctypes
    lib.gml_b200_sample_tempering_device.argtypes = [c.c_int32, c.c_int32, c.c_int32, c.c_int32, c.c_void_p, c.c_void_p,
                                                     c.c_int32, c.c_void_p, c.c_int64, c.c_int32, c.c_int64, c.c_int32,
                                                     c.c_int32, c.c_uint64, c.c_void_p, c.c_void_p, c.c_void_p, c.c_void_p,
                                                     c.c_void_p, c.c_int64, c.c_void_p]
    order, idx, wts = term_arrays(gm)
    N = gm.varible_count
    b = None if betas is None else np.asarray(betas, dtype=np.float64)
    R = _lib.TEMPERING_DEFAULT_RUNGS if b is None else len(b)
    ld = reps * min(n, 1 << N)
    K, rhat, swap = np.zeros(reps, dtype=np.int64), np.zeros((reps, 2)), np.zeros((reps, R - 1))
    counts, spins = np.zeros(ld), np.zeros((N, ld), dtype=np.int8)
    rc = lib.gml_b200_sample_tempering_device(0, N, order, len(wts), idx.ctypes.data, wts.ctypes.data,
                                              0 if b is None else R, None if b is None else b.ctypes.data, n, reps, chains,
                                              burn_in, thin, seed, K.ctypes.data, rhat.ctypes.data, swap.ctypes.data,
                                              counts.ctypes.data, spins.ctypes.data, ld, None)
    assert rc == 0
    rows = int(K.sum())
    return hashlib.sha256(K.tobytes() + counts[:rows].tobytes() + np.ascontiguousarray(spins[:, :rows]).tobytes() +
                          rhat.tobytes() + swap.tobytes()).hexdigest()[:16]


PINNED_TEMPERING = [  # (name, model, n, replicates, seed, chains, burn_in, thin, betas, sha256 prefix)
    ("order-3 N=14", lambda: FactorGraph(3, 14, "spin", three_body_model(14, 14)), 50_000, 2, 11, 0, 50, 2,
     [1.0, 0.6, 0.3, 0.1], "112bfe06ec790887"),
    ("pairwise N=20", lambda: FactorGraph.from_matrix(random_ising(20, 20)), 100_000, 2, 7, 1000, 100, 3, None, "98852821da3a6ab8"),
    ("C2 N=100", lambda: FactorGraph.from_matrix(lattice_model()[0]), 20_000, 2, 3, 256, 30, 1,
     [1.0, 0.8, 0.6, 0.5, 0.4, 0.3, 0.2, 0.1], "ca577b28025b1992"),
]


def test_tempering_output_is_pinned():
    """B200Tempering writes, for these fixed seeds, the bytes the sampler wrote before the log Z estimator shared its
    kernel: counts, spins, R-hat and swap rates, as sha256 prefixes taken on a B200 at that commit."""
    lib = _lib.load()
    for name, model, n, reps, seed, chains, burn_in, thin, betas, digest in PINNED_TEMPERING:
        assert tempering_digest(lib, model(), n, reps, seed, chains, burn_in, thin, betas) == digest, name
