"""moments / empirical_moments / log_likelihood on the B200: exact moments against numpy enumeration and against central
differences of log Z, MCMC moments against the sampler's own draws bit for bit, against exact values and closed forms
(fields, periodic ring, Curie-Weiss), a 64-seed calibration of the standard error, the data side against numpy, and the
output contract.  Every seed is fixed.

Bars for MCMC estimates: |estimate - exact| <= k stderr + (e^{2 delta} - 1) per entry, with k = norm.isf(0.5e-6 /
n_entries) (family-wise rate 1e-6) and delta = sum_t |w_t - fl32(w_t)| (the chains sample fp32-rounded weights); each
stderr cap sits at about 3x the largest stderr measured on a B200, which stands next to it."""
import math

import numpy as np
import pytest
from scipy import special, stats

import gml_b200
from gml_b200 import B200Exact, B200Gibbs, B200Tempering, FactorGraph
from helpers import random_ising
from test_gpu_log_partition import curie_weiss, fp32_bound, order8_model, ring
from test_gpu_tempering_sampler import FERRO_4X5, ORDER3_N14

pytestmark = pytest.mark.gpu


def enumerate_model(gm):
    """all 2^N configurations S [2^N x N] (spin_i = 2 bit_i - 1) and their probabilities, in fp64"""
    N = gm.varible_count
    c = np.arange(2 ** N, dtype=np.int64)
    S = (((c[:, None] >> np.arange(N)) & 1) * 2 - 1).astype(np.float64)
    E = np.zeros(len(c))
    for k, w in gm.terms.items():
        E += w * np.prod(S[:, np.asarray(k) - 1], axis=1)
    p = np.exp(E - E.max())
    return S, p / p.sum(), E


def brute_keys(S, p, keys):
    return np.array([p @ np.prod(S[:, np.asarray(k) - 1], axis=1) for k in keys])


def brute_pairwise(S, p):
    C = S.T @ (S * p[:, None])
    np.fill_diagonal(C, p @ S)
    return C


def values(fg):
    return np.array(list(fg.terms.values()))


def k_bar(n_entries):
    return stats.norm.isf(0.5e-6 / n_entries)


def pairwise_keys(N):
    return [(i,) for i in range(1, N + 1)] + [(i, j) for i in range(1, N + 1) for j in range(i + 1, N + 1)]


# ---- 1-2: exact -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,model", [("order-8 N=12", order8_model), ("order-3 N=14", lambda: ORDER3_N14)])
def test_exact_against_enumeration(name, model):
    gm = model()
    S, p, _ = enumerate_model(gm)
    mean, err = gml_b200.moments(gm)
    assert list(mean.terms) == list(gm.terms) and not values(err).any()
    d = np.abs(values(mean) - brute_keys(S, p, gm.terms)).max()
    C, Cerr = gml_b200.moments(gm, keys="pairwise")
    d2 = np.abs(C - brute_pairwise(S, p)).max()
    print(f"{name}: gm keys {d:.1e}, pairwise {d2:.1e}")
    assert d <= 1e-12 and d2 <= 1e-12 and not Cerr.any()


def test_exact_is_derivative_of_log_z():
    gm = FactorGraph.from_matrix(random_ising(20, 20))
    keys = list(gm.terms)[:10]
    mean = values(gml_b200.moments(gm, keys=keys)[0])
    h = 1e-4
    for key, m in zip(keys, mean):
        lz = []
        for s in (1, -1):
            t = dict(gm.terms)
            t[key] += s * h
            lz.append(gml_b200.log_partition(FactorGraph(2, 20, "spin", t), B200Exact())[0])
        assert abs((lz[0] - lz[1]) / (2 * h) - m) <= 1e-7, key


# ---- 3: MCMC against the sampler's own draws ------------------------------------------------------------------------
MCMC_CASES = [  # (name, model, n, sampler fields)
    ("Gibbs N=20 (histogram rows)", lambda: FactorGraph.from_matrix(random_ising(20, 20)), 12_345,
     dict(cls=B200Gibbs, seed=3, chains=1000, burn_in=50, thin=2)),
    ("Gibbs N=100 (draw rows)", lambda: ring(100, 0.4), 5_000, dict(cls=B200Gibbs, seed=4, chains=256, burn_in=20, thin=1)),
    ("Tempering order-3 N=14", lambda: ORDER3_N14, 3_001,
     dict(cls=B200Tempering, seed=5, chains=64, burn_in=30, thin=1, betas=[1.0, 0.6, 0.3, 0.1])),
]


def make(fields):
    f = dict(fields)
    return f.pop("cls")(**f)


@pytest.mark.parametrize("name,model,n,fields", MCMC_CASES)
def test_mcmc_equals_own_draws(name, model, n, fields):
    gm = model()
    N = gm.varible_count
    S1, S2 = make(fields), make(fields)
    mean, err = gml_b200.moments(gm, S1, n)
    draws = gml_b200.sample(gm, n, 1, S2)
    assert draws[:, 0].sum() == n
    emp = gml_b200.empirical_moments(draws, list(gm.terms))
    assert np.array_equal(values(mean), values(emp)), name
    assert np.array_equal(S1.last_rhat, S2.last_rhat, equal_nan=True)
    if isinstance(S1, B200Tempering):
        assert S1.last_swap_rate == S2.last_swap_rate
    assert np.isfinite(values(err)).all() and (values(err) >= 0).all()
    # pairwise against the key list of every field and pair, mean and stderr bit for bit
    keys = pairwise_keys(N)
    km, ke = gml_b200.moments(gm, make(fields), n, keys=keys)
    C, Ce = gml_b200.moments(gm, make(fields), n, keys="pairwise")
    for (k, m), e in zip(km.terms.items(), ke.terms.values()):
        i, j = (k[0] - 1, k[-1] - 1)
        assert C[i, j] == m and C[j, i] == m and Ce[i, j] == e and Ce[j, i] == e, k
    Cemp = values(gml_b200.empirical_moments(draws, keys))
    assert np.array_equal(values(km), Cemp)


# ---- 4: MCMC against exact values -----------------------------------------------------------------------------------
@pytest.mark.parametrize("name,model,sampler,n,cap", [
    ("ferromagnet 4x5 J=1.5", lambda: FERRO_4X5, B200Tempering(seed=6), 200_000, 6.5e-3),          # measured 2.16e-3
    ("order-3 N=14 x2", lambda: ORDER3_N14, B200Gibbs(seed=7), 500_000, 6e-3),                          # 1.95e-3
    ("random_ising(30, 30)", lambda: FactorGraph.from_matrix(random_ising(30, 30)), B200Gibbs(seed=8), 500_000, 6.5e-3),   # 2.16e-3
    ("order-8 N=12", order8_model, B200Gibbs(seed=9), 500_000, 5e-3),                                   # 1.70e-3
])
def test_mcmc_against_exact(name, model, sampler, n, cap):
    gm = model()
    exact = values(gml_b200.moments(gm)[0])
    mean, err = (values(x) for x in gml_b200.moments(gm, sampler, n))
    bar = k_bar(len(exact)) * err + math.expm1(2 * fp32_bound(gm))
    print(f"{name}: max |error| {np.abs(mean - exact).max():.2e}, max stderr {err.max():.2e} (cap {cap:.0e})")
    assert (np.abs(mean - exact) <= bar).all()
    assert err.max() <= cap


# ---- 5: closed forms beyond enumeration -----------------------------------------------------------------------------
def test_fields_only():
    rng = np.random.default_rng(1)
    h = rng.integers(-64, 65, 4096) / 64.0                      # dyadic: exact in fp32
    gm = FactorGraph(1, 4096, "spin", {(i + 1,): float(v) for i, v in enumerate(h)})
    mean, err = (values(x) for x in gml_b200.moments(gm, B200Gibbs(seed=1, chains=4096, burn_in=5, thin=1), 100_000))
    print(f"fields N=4096: max |error| {np.abs(mean - np.tanh(h)).max():.2e}, max stderr {err.max():.2e}")
    assert (np.abs(mean - np.tanh(h)) <= k_bar(4096) * err).all()
    assert err.max() <= 0.015                                  # measured 5.01e-3


def test_periodic_ring_pairwise():
    N, J = 1000, 0.5
    t = math.tanh(J)
    d = np.abs(np.arange(N)[:, None] - np.arange(N)[None, :])
    exact = (t ** d + t ** (N - d)) / (1 + t ** N)
    np.fill_diagonal(exact, 0.0)
    C, Ce = gml_b200.moments(ring(N, J), B200Gibbs(seed=2, chains=8192, burn_in=50, thin=2), 200_000, keys="pairwise")
    print(f"ring N=1000: max |error| {np.abs(C - exact).max():.2e}, max stderr {Ce.max():.2e}")
    assert (np.abs(C - exact) <= k_bar(N * N) * Ce).all()
    assert Ce.max() <= 0.012                                   # measured 3.84e-3


@pytest.mark.parametrize("J,cap", [(0.5, 0.015), (1.5, 0.032)])           # measured stderr 4.88e-3, 1.06e-2
def test_curie_weiss(J, cap):
    """N = 256, every pair at J / N (dyadic); J = 1.5 is the ordered phase, where only the ladder flips the magnetisation."""
    n = 256
    k = np.arange(n + 1)
    M = 2.0 * k - n
    logw = special.gammaln(n + 1) - special.gammaln(k + 1) - special.gammaln(n - k + 1) + J * (M * M - n) / (2.0 * n)
    w = np.exp(logw - logw.max())
    pair = ((w @ (M * M)) / w.sum() - n) / (n * (n - 1))
    exact = np.full((n, n), pair)
    np.fill_diagonal(exact, 0.0)
    C, Ce = gml_b200.moments(curie_weiss(n, J), B200Tempering(seed=3, chains=1024, burn_in=100), 100_000, keys="pairwise")
    print(f"Curie-Weiss J={J}: <s_i s_j> exact {pair:.4f}, max |error| {np.abs(C - exact).max():.2e}, max stderr {Ce.max():.2e}")
    assert (np.abs(C - exact) <= k_bar(n * n) * Ce).all()
    assert Ce.max() <= cap


# ---- 6: stderr calibration ------------------------------------------------------------------------------------------
def test_stderr_is_calibrated():
    gm32 = FactorGraph(3, 14, "spin", {k: float(np.float32(v)) for k, v in ORDER3_N14.terms.items()})
    keys = [(1, 2), (3,)]
    exact = values(gml_b200.moments(gm32, keys=keys)[0])
    z = []
    for seed in range(64):
        mean, err = (values(x) for x in gml_b200.moments(ORDER3_N14, B200Gibbs(seed=200 + seed, chains=2048, burn_in=100,
                                                                                  thin=2), 20_000, keys=keys))
        z.append((mean - exact) / err)
    z = np.array(z)
    mean_bound = stats.norm.isf(0.5e-6 / 2) / math.sqrt(len(z))
    lo, hi = stats.chi2.ppf(0.25e-6, len(z) - 1) / (len(z) - 1), stats.chi2.isf(0.25e-6, len(z) - 1) / (len(z) - 1)
    print(f"calibration: mean z {z.mean(axis=0)}, var z {z.var(axis=0, ddof=1)} (bounds {lo:.3f}, {hi:.3f})")
    assert (np.abs(z.mean(axis=0)) <= mean_bound).all()
    assert ((lo <= z.var(axis=0, ddof=1)) & (z.var(axis=0, ddof=1) <= hi)).all()


# ---- 7: data side ---------------------------------------------------------------------------------------------------
def random_histogram(N, K, seed, integer=True):
    rng = np.random.default_rng(seed)
    spins = rng.choice([-1, 1], size=(K, N))
    counts = rng.integers(1, 5, K).astype(np.float64) if integer else rng.uniform(0.1, 3.0, K)
    return np.concatenate([counts[:, None], spins], axis=1)


def test_data_key_lists_non_integer_counts():
    data = random_histogram(20, 3000, 11, integer=False)
    rng = np.random.default_rng(12)
    keys = [tuple(sorted(int(x) + 1 for x in rng.choice(20, q, replace=False))) for q in range(1, 9) for _ in range(5)]
    keys = list(dict.fromkeys(keys))
    got = values(gml_b200.empirical_moments(data, keys))
    w = data[:, 0] / data[:, 0].sum()
    ref = np.array([w @ np.prod(data[:, np.asarray(k)], axis=1) for k in keys])
    assert np.abs(got - ref).max() <= 1e-13


@pytest.mark.parametrize("N", [300, 1000])
def test_data_pairwise(N):
    data = random_histogram(N, 20_000, N)
    C = gml_b200.empirical_moments(data)
    w = data[:, 0] / data[:, 0].sum()
    S = data[:, 1:]
    ref = S.T @ (S * w[:, None])
    np.fill_diagonal(ref, w @ S)
    print(f"data pairwise N={N}: max |error| {np.abs(C - ref).max():.2e}")
    assert np.abs(C - ref).max() <= 1e-7 and np.array_equal(C, C.T)
    sess = gml_b200.Session().upload(np.ascontiguousarray(data[:, 0]), np.ascontiguousarray(S.T.astype(np.int8)))
    assert np.array_equal(sess.moments(), C)
    keys = [(1,), (2, 5), (3, 4, 7)]
    assert sess.moments(keys) == gml_b200.empirical_moments(data, keys)


# ---- 8: log_likelihood ----------------------------------------------------------------------------------------------
def test_log_likelihood():
    gm = FactorGraph.from_matrix(random_ising(20, 20))
    data = gml_b200.sample(gm, 20_000, 1, B200Exact(seed=5))
    S, p, E = enumerate_model(gm)
    log_z = special.logsumexp(E)
    w = data[:, 0] / data[:, 0].sum()
    e_data = 0.0
    for k, v in gm.terms.items():
        e_data += v * (w @ np.prod(data[:, np.asarray(k)], axis=1))
    exact = e_data - log_z
    value, err = gml_b200.log_likelihood(gm, data, B200Exact())
    assert abs(value - exact) <= 1e-9 and err == 0.0
    value, err = gml_b200.log_likelihood(gm, data, B200Tempering(seed=6))
    print(f"log_likelihood tempering: error {value - exact:+.2e}, stderr {err:.2e}")
    assert abs(value - exact) <= 5 * err + fp32_bound(gm)


# ---- 9: output contract ---------------------------------------------------------------------------------------------
def test_output_contract():
    gm = FactorGraph.from_matrix(random_ising(30, 30))
    a = gml_b200.moments(gm, B200Gibbs(seed=1, chains=512), 20_000)
    assert gml_b200.moments(gm, B200Gibbs(seed=1, chains=512), 20_000) == a
    assert gml_b200.moments(gm, B200Gibbs(seed=2, chains=512), 20_000)[0] != a[0]
    t = gml_b200.moments(gm, B200Tempering(seed=1, chains=128), 5_000, keys="pairwise")
    t2 = gml_b200.moments(gm, B200Tempering(seed=1, chains=128), 5_000, keys="pairwise")
    assert np.array_equal(t[0], t2[0]) and np.array_equal(t[1], t2[1])
    small = FactorGraph.from_matrix(random_ising(12, 12))
    e = gml_b200.moments(small, None, keys="pairwise")
    assert np.array_equal(e[0], gml_b200.moments(small, B200Exact(), keys="pairwise")[0]) and not e[1].any()
    # fewer than two groups of warps: no standard error
    one = gml_b200.moments(gm, B200Gibbs(seed=1, chains=32), 1_000)[1]
    assert np.isnan(values(one)).all()
