"""fit_likelihood on the B200: the exact path against the float64 oracle (weights, zeros and the KKT conditions), the
persistent chains against the sampler bit for bit, the MCMC path against the exact path over 8 seeds, a refit of
RISE fits at the C2 and C3 scales of bench.py, and the output contract.  Every seed is fixed; measured values stand
next to the bars."""
import math

import numpy as np
import pytest
from scipy import stats

import gml_b200
import mle_oracle
from bench import c2_model, c3_model
from gml_b200 import RISE, B200Exact, B200Gibbs, FactorGraph
from helpers import random_ising
from test_gpu_tempering_sampler import ORDER3_N14

pytestmark = pytest.mark.gpu


def values(fg):
    return np.array(list(fg.terms.values()))


def widened(gm):
    """gm's keys plus every field and pair of its spins, all at weight 0 (a support wider than the truth)"""
    N = gm.varible_count
    keys = [(i,) for i in range(1, N + 1)] + [(i, j) for i in range(1, N + 1) for j in range(i + 1, N + 1)]
    keys += [k for k in gm.terms if len(k) > 2]
    return FactorGraph(gm.order, N, "spin", {k: 0.0 for k in keys})


def max_abs(x):
    return float(np.abs(x).max()) if x.size else 0.0


def fp32_delta(fg):
    w = values(fg)
    return float(np.abs(w - w.astype(np.float32).astype(np.float64)).sum())


EXACT_MODELS = {"pairwise N=12": lambda: FactorGraph.from_matrix(random_ising(12, 12)),
                "pairwise N=16": lambda: FactorGraph.from_matrix(random_ising(16, 16)),
                "order-3 N=14": lambda: ORDER3_N14}


# ---- 1: exact path against the oracle ------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(EXACT_MODELS))
@pytest.mark.parametrize("regularizer", [0.0, 1.0])
def test_exact_against_oracle(name, regularizer):
    truth = EXACT_MODELS[name]()
    N = truth.varible_count
    data = gml_b200.sample(truth, 100_000, 1, B200Exact(seed=7))
    start = widened(truth) if regularizer else FactorGraph(truth.order, N, "spin", {k: 0.0 for k in truth.terms})
    fg, info = gml_b200.fit_likelihood(start, data, regularizer=regularizer, return_info=True)
    assert list(fg.terms) == list(start.terms)
    lam, dm = info["lambda"], np.array(info["data_moments"])
    w = values(fg)
    w_or = mle_oracle.mle_exact(start.terms, N, dm, lam)
    err = np.abs(w - w_or).max()
    m = values(gml_b200.moments(fg)[0])
    pen = np.array([len(k) >= 2 for k in fg.terms])
    r = dm - m
    free = max_abs(r[~pen])
    nz = pen & (w != 0)
    on = max_abs(r[nz] - lam * np.sign(w[nz]))
    zero = max_abs(r[pen & (w == 0)]) - lam
    print(f"{name} lambda={lam:.2e}: |w - oracle| {err:.1e}, {int((w_or == 0).sum())} oracle zeros, {int((w == 0).sum())} "
          f"zeros, KKT free {free:.1e} nonzero {on:.1e} zero-excess {zero:.1e}, {info['iterations']} iterations")
    assert err <= 1e-8                                    # measured <= 1.5e-9
    assert (w[w_or == 0] == 0).all()
    if regularizer:
        assert (w_or == 0).any()                          # the lambda zeroes some couplings
    assert free <= 1e-9 and on <= 1e-9 and zero <= 1e-9   # measured <= 1.0e-10, 9.3e-11 and -2.9e-5


# ---- 2: persistent chains are exactly the sampler ------------------------------------------------------------------
@pytest.mark.parametrize("N,chains", [(12, 100), (80, 96), (80, 4100)])
def test_persistence_is_the_sampler(N, chains):
    gm = FactorGraph.from_matrix(random_ising(N, N + 1))
    data = gml_b200.sample(gm, 20_000, 1, B200Gibbs(seed=3, chains=1024))
    b, k, steps, seed = 7, 3, 9, 11
    fg, info = gml_b200.fit_likelihood(gm, data, B200Gibbs(seed=seed, chains=chains, burn_in=b, thin=k), steps=steps,
                                       step_size=0.0, return_info=True)
    h = steps // 2
    ref = gml_b200.moments(gm, B200Gibbs(seed=seed, chains=chains, burn_in=b + h * k, thin=k), (steps - h) * chains)[0]
    assert np.array_equal(np.array(info["model_moments"]), values(ref))
    assert np.array_equal(values(fg), values(gm)) and list(fg.terms) == list(gm.terms)


# ---- 3: MCMC against the exact path --------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["pairwise N=16", "order-3 N=14"])
def test_mcmc_against_exact(name):
    truth = EXACT_MODELS[name]()
    data = gml_b200.sample(truth, 100_000, 1, B200Exact(seed=8))
    start = FactorGraph(truth.order, truth.varible_count, "spin", {k: 0.0 for k in truth.terms})
    w_exact = values(gml_b200.fit_likelihood(start, data))
    errs, fits = [], []
    for seed in range(8):
        fg, info = gml_b200.fit_likelihood(start, data, B200Gibbs(seed=seed, thin=1), return_info=True)
        errs.append(np.abs(values(fg) - w_exact).max())
        fits.append((fg, info))
    print(f"{name}: |w_mcmc - w_exact| over 8 seeds: " + " ".join(f"{e:.1e}" for e in errs))
    assert max(errs) <= W_BAR
    fg, info = fits[0]
    dm = np.array(info["data_moments"])
    n = 1_000_000
    mean, err = gml_b200.moments(fg, B200Gibbs(seed=100, thin=1), n)
    delta = float(np.abs(values(fg) - w_exact).sum()) + fp32_delta(fg)
    tol = stats.norm.isf(0.5e-6 / len(dm)) * values(err) + math.expm1(2 * delta) + 1e-9
    dev = np.abs(values(mean) - dm)
    print(f"{name}: moment residual {dev.max():.1e}, bound {tol.min():.1e}..{tol.max():.1e}, max stderr {values(err).max():.1e}")
    assert (dev <= tol).all()          # measured residual 3.2e-3 (pairwise) and 2.7e-3 (order-3), bounds >= 1.2e-2


# |w_mcmc - w_exact| bar.  The averaged iterate pools 1000 steps of 2^17 chains; its stochastic-approximation error is
# ~ sqrt(tau / (2^17 * 1000)) / (smallest curvature) with tau the chains' autocorrelation in steps (1e-4 to 1e-3 for
# these models), and the fp32 weights move the fixed point by at most ~ 2^-24 |w| / curvature (< 1e-6 here).  Measured
# on a B200 over seeds 0..7: 2.1e-4..3.4e-4 (pairwise N=16) and 2.5e-3..3.4e-3 (order-3 N=14, whose triplet weights
# are the least constrained); the bar is 3x the largest.
W_BAR = 1e-2


# ---- 4: a refit improves a RISE fit at scale -----------------------------------------------------------------------
def rise_support(J, N, tau):
    keys = {(i + 1,): float(J[i, i]) for i in range(N)}
    keys.update({(i + 1, j + 1): float(J[i, j]) for i in range(N) for j in range(i + 1, N) if abs(J[i, j]) > tau})
    return FactorGraph(2, N, "spin", keys)


def coupling_error(fg, truth):
    return max(abs(v - truth[k[0] - 1, k[1] - 1]) for k, v in fg.terms.items() if len(k) == 2)


@pytest.mark.parametrize("config", ["C2", "C3"])
def test_refit_improves_rise(config):
    truth = c2_model() if config == "C2" else c3_model(1000)[3]
    N = truth.shape[0]
    gm = FactorGraph.from_matrix(truth)
    M = 1_000_000 if config == "C2" else 200_000
    data = gml_b200.sample(gm, M, 1, B200Gibbs(seed=21)).astype(np.int8)
    rise = rise_support(gml_b200.learn(data, RISE()), N, 0.1)
    refit, info = gml_b200.fit_likelihood(rise, data, B200Gibbs(seed=22, thin=1), return_info=True)
    dm = np.array(info["data_moments"])
    check = B200Gibbs(seed=23, thin=1)
    res_rise = np.abs(values(gml_b200.moments(rise, check, 1_000_000)[0]) - dm).max()
    res_refit = np.abs(values(gml_b200.moments(refit, check, 1_000_000)[0]) - dm).max()
    e_rise, e_refit = coupling_error(rise, truth), coupling_error(refit, truth)
    msg = (f"{config}: {len(rise.terms)} terms, moment residual RISE {res_rise:.2e} refit {res_refit:.2e}; coupling error "
           f"RISE {e_rise:.2e} refit {e_refit:.2e}")
    if config == "C2":
        ll_rise, s_rise = gml_b200.log_likelihood(rise, data)
        ll_refit, s_refit = gml_b200.log_likelihood(refit, data)
        msg += f"; log-likelihood RISE {ll_rise:.5f} +- {s_rise:.1e}, refit {ll_refit:.5f} +- {s_refit:.1e}"
        assert ll_refit >= ll_rise - 3 * s_refit     # measured -55.24068 against -55.24069, stderr 5.2e-4
    print(msg)
    assert res_refit < res_rise               # measured C2 3.46e-3 < 5.59e-3, C3 5.80e-3 < 1.03e-2
    assert e_refit <= e_rise + COUPLING_BAR   # measured C2 2.92e-3 vs 5.22e-3, C3 7.22e-3 vs 1.47e-2


# The refit's coupling error may exceed RISE's by at most the statistical error of a coupling at these sample sizes
# (~ 1 / sqrt(M (1 - m^2)) ~ 3e-3 at M = 1e6).
COUPLING_BAR = 1e-2


# ---- 5: contract ---------------------------------------------------------------------------------------------------
def test_contract():
    truth = FactorGraph.from_matrix(random_ising(16, 5))
    data = gml_b200.sample(truth, 50_000, 1, B200Exact(seed=1))
    start = FactorGraph(2, 16, "spin", {k: 0.0 for k in reversed(list(truth.terms))})
    sampler = B200Gibbs(seed=4, chains=4096, burn_in=20, thin=1)
    a, ia = gml_b200.fit_likelihood(start, data, sampler, steps=400, return_info=True)
    b, ib = gml_b200.fit_likelihood(start, data, sampler, steps=400, return_info=True)
    assert list(a.terms) == list(start.terms)
    assert np.array_equal(values(a), values(b)) and ia["trace"] == ib["trace"] and ia["model_moments"] == ib["model_moments"]
    trace = np.array(ia["trace"])
    assert len(trace) == 400 and len(ia["step_sizes"]) == 400
    print(f"trace: first 10 % mean {trace[:40].mean():.2e}, last 10 % mean {trace[-40:].mean():.2e}")
    assert trace[-40:].mean() < trace[:40].mean()      # measured 3.45e-2 < 1.40e-1
    e1 = gml_b200.fit_likelihood(start, data, return_info=True)
    e2 = gml_b200.fit_likelihood(start, data, return_info=True)
    assert np.array_equal(values(e1[0]), values(e2[0])) and e1[1]["objective"] == e2[1]["objective"]
