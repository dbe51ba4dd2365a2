"""The multi-sample Gibbs sampler (csrc/mcmc_sampler.cu, sample(gm, n, replicates, B200Gibbs())): moments against exact
enumeration with error bars from independent replicates, the output contract, sample -> learn at N = 100 and on an
order-3 model, the split-R-hat diagnostic, and input refusals.  Every seed is fixed."""
import ctypes

import numpy as np
import pytest
from scipy import stats

import gml_b200
from gml_b200 import B200, B200Gibbs, FactorGraph, RISE, RPLE, Session, _lib, multiRISE
from helpers import random_ising, three_body_model
from test_gpu_exact_sampler import config_index, log_weights, logsumexp
from test_gpu_fullsize import lattice_model

pytestmark = pytest.mark.gpu


def term_arrays(gm):
    order = max(len(k) for k in gm.terms)
    idx = -np.ones((len(gm.terms), order), dtype=np.int32)
    for t, k in enumerate(gm.terms):
        idx[t, :len(k)] = np.array(k) - 1
    return order, idx, np.array(list(gm.terms.values()), dtype=np.float64)


def mcmc_call(gm, n, reps, sampler, counts=None, spins=None, ld=0):
    """gml_b200_sample_mcmc_device with raw buffers (None = count-only); returns (rc, K, rhat)."""
    order, idx, wts = term_arrays(gm)
    K, rhat = np.zeros(reps, dtype=np.int64), np.zeros((reps, 2))
    rc = _lib.load().gml_b200_sample_mcmc_device(0, gm.varible_count, order, len(wts), idx.ctypes.data, wts.ctypes.data, n,
                                                 reps, sampler.chains, sampler.burn_in, sampler.thin, sampler.seed,
                                                 K.ctypes.data, rhat.ctypes.data, counts, spins, ld, None)
    return rc, K, rhat


def c2_graph():
    truth = lattice_model()[0]
    return truth, FactorGraph.from_matrix(truth)


@pytest.mark.parametrize("name,gm", [("pairwise N=20", FactorGraph.from_matrix(random_ising(20, 20))),
                                     ("order-3 N=14", FactorGraph(3, 14, "spin", three_body_model(14, 14)))])
def test_moments_match_enumeration(name, gm):
    """Magnetisations and pair correlations of R = 32 independent replicates against exact enumeration.  MCMC draws are
    correlated, so the error bar of each quantity is the spread of its replicate values; the threshold is the Student-t
    (R - 1 degrees of freedom) quantile that keeps the family-wise false-alarm rate over all quantities at 1e-6
    (Bonferroni, two-sided)."""
    n_spins, draws, R = gm.varible_count, 200_000, 32
    e = log_weights(gm.terms, n_spins)
    p = np.exp(e - logsumexp(e))
    conf = ((np.arange(2 ** n_spins)[:, None] >> np.arange(n_spins)) & 1) * 2.0 - 1.0
    iu = np.triu_indices(n_spins, 1)
    exact = np.concatenate([p @ conf, ((conf * p[:, None]).T @ conf)[iu]])
    reps = gml_b200.sample(gm, draws, R, B200Gibbs(seed=7))
    vals = []
    for h in reps:
        w = h[:, 0] / draws
        s = h[:, 1:].astype(np.float64)
        vals.append(np.concatenate([w @ s, ((s * w[:, None]).T @ s)[iu]]))
    vals = np.array(vals)
    t = np.abs(vals.mean(axis=0) - exact) / (vals.std(axis=0, ddof=1) / np.sqrt(R))
    thr = stats.t.isf(1e-6 / (2 * len(exact)), R - 1)
    print(f"{name}: max |t| {t.max():.2f} over {len(exact)} quantities (threshold {thr:.2f})")
    assert t.max() <= thr


def test_output_contract():
    gm = FactorGraph(3, 14, "spin", three_body_model(14, 14))
    sampler = B200Gibbs(seed=11, burn_in=50, thin=2)
    reps = gml_b200.sample(gm, 50_000, 3, sampler)
    reps_rhat = np.array(sampler.last_rhat)
    assert len(reps) == 3 and reps_rhat.shape == (3, 2)
    for h in reps:
        assert h.dtype == np.int64 and h.shape[1] == 15
        assert h[:, 0].sum() == 50_000 and (h[:, 0] > 0).all()
        assert set(np.unique(h[:, 1:])) <= {-1, 1}
        assert (np.diff(config_index(h[:, 1:].T).astype(np.int64)) > 0).all()
    assert not np.array_equal(reps[0], reps[1])
    # bit-identical for the same arguments, different for another seed; replicate 0 is the single-replicate call
    again = gml_b200.sample(gm, 50_000, 3, B200Gibbs(seed=11, burn_in=50, thin=2))
    assert all(np.array_equal(x, y) for x, y in zip(reps, again))
    assert np.array_equal(reps[0], gml_b200.sample(gm, 50_000, sampler=B200Gibbs(seed=11, burn_in=50, thin=2)))
    assert not np.array_equal(reps[0], gml_b200.sample(gm, 50_000, sampler=B200Gibbs(seed=12, burn_in=50, thin=2)))
    # the device form holds the same rows
    counts, spins = gml_b200.sample_device(gm, 50_000, sampler=sampler)
    assert np.array_equal(counts.cpu().numpy(), reps[0][:, 0]) and np.array_equal(spins.cpu().numpy(), reps[0][:, 1:].T)
    # count-only and host-buffer calls agree with the device-buffer call; a too-small ld is refused with out_K filled
    rc, K, rhat = mcmc_call(gm, 50_000, 3, sampler)
    assert rc == _lib.OK and K.tolist() == [h.shape[0] for h in reps]
    assert np.array_equal(rhat, reps_rhat, equal_nan=True)
    rows = int(K.sum())
    hc, hs = np.zeros(rows), np.zeros((14, rows), dtype=np.int8)
    rc, _, _ = mcmc_call(gm, 50_000, 3, sampler, hc.ctypes.data, hs.ctypes.data, rows)
    assert rc == _lib.OK
    assert np.array_equal(np.concatenate([h[:, 0] for h in reps]), hc)
    assert np.array_equal(np.concatenate([h[:, 1:] for h in reps]).T, hs)
    rc, K2, _ = mcmc_call(gm, 50_000, 3, sampler, hc.ctypes.data, hs.ctypes.data, rows - 1)
    assert rc == _lib.EINVAL and np.array_equal(K, K2)


def test_output_contract_beyond_64_spins():
    """N = 100: one row of count 1 per draw, in draw order."""
    import torch
    _, gm = c2_graph()
    sampler = B200Gibbs(seed=3, burn_in=20, thin=1, chains=1024)
    n = 5000                                         # 4 full record steps of 1024 chains and a partial fifth
    h = gml_b200.sample(gm, n, sampler=sampler)
    assert h.shape == (n, 101) and (h[:, 0] == 1).all() and set(np.unique(h[:, 1:])) <= {-1, 1}
    two = gml_b200.sample(gm, n, 2, sampler)
    assert isinstance(two, list) and np.array_equal(two[0], h) and not np.array_equal(two[0], two[1])
    assert np.array_equal(h, gml_b200.sample(gm, n, sampler=B200Gibbs(seed=3, burn_in=20, thin=1, chains=1024)))
    assert not np.array_equal(h, gml_b200.sample(gm, n, sampler=B200Gibbs(seed=4, burn_in=20, thin=1, chains=1024)))
    counts, spins = gml_b200.sample_device(gm, n, sampler=sampler)
    assert counts.numel() == n and np.array_equal(spins.cpu().numpy(), h[:, 1:].T)
    rc, K, _ = mcmc_call(gm, n, 2, sampler)
    assert rc == _lib.OK and K.tolist() == [n, n]
    hc, hs = np.zeros(2 * n), np.zeros((100, 2 * n), dtype=np.int8)
    assert mcmc_call(gm, n, 2, sampler, hc.ctypes.data, hs.ctypes.data, 2 * n)[0] == _lib.OK
    assert (hc == 1).all() and np.array_equal(hs[:, :n], h[:, 1:].T) and np.array_equal(hs[:, n:], two[1][:, 1:].T)
    small_c = torch.empty(2 * n - 1, dtype=torch.float64, device="cuda:0")
    small_s = torch.empty((100, 2 * n - 1), dtype=torch.int8, device="cuda:0")
    rc, K2, _ = mcmc_call(gm, n, 2, sampler, small_c.data_ptr(), small_s.data_ptr(), 2 * n - 1)
    assert rc == _lib.EINVAL and K2.tolist() == [n, n]


@pytest.fixture(scope="module")
def c2_sample():
    truth, gm = c2_graph()
    sampler = B200Gibbs(seed=1)
    counts, spins = gml_b200.sample_device(gm, 1_000_000, sampler=sampler)
    return truth, counts, spins, sampler.last_rhat[0]


@pytest.mark.parametrize("form_cls,c", [(RISE, 0.4), (RPLE, 0.2)])
def test_c2_sample_learns_back(c2_sample, form_cls, c):
    """1e6 draws of the C2 lattice (N = 100) with the default settings: couplings and fields within 0.02, the bar the
    old sampler's input meets in test_gpu_fullsize."""
    truth, counts, spins, _ = c2_sample
    assert counts.numel() == 1_000_000
    sess = Session(0).attach_device(counts.data_ptr(), spins.data_ptr(), counts.numel(), 100, spins.stride(0))
    theta = sess.solve_pairwise(form_cls(c, False), B200())
    off = theta - np.diag(np.diag(theta))
    print(f"{form_cls.__name__}: max coupling error {np.abs(off - truth).max():.4f}, max field {np.abs(np.diag(theta)).max():.4f}")
    assert np.abs(off - truth).max() <= 0.02
    assert np.abs(np.diag(theta)).max() <= 0.02


def test_rhat_of_a_mixed_c2_sample(c2_sample):
    rhat = c2_sample[3]
    print(f"C2 R-hat (energy, magnetisation): {rhat}")
    assert max(rhat) <= 1.01


def test_rhat_flags_an_unmixed_ferromagnet():
    """A 32 x 32 open ferromagnet at J = 1 (far below the critical temperature, J_c ~ 0.44) from random starts with 10
    burn-in sweeps: the chains sit in different domain patterns, and R-hat must say so."""
    side = 32
    m = np.zeros((side * side, side * side))
    for r in range(side):
        for c in range(side):
            i = r * side + c
            for j in ([i + 1] if c + 1 < side else []) + ([i + side] if r + 1 < side else []):
                m[i, j] = m[j, i] = 1.0
    sampler = B200Gibbs(seed=5, chains=4096, burn_in=10, thin=1)
    gml_b200.sample_device(FactorGraph.from_matrix(m), 8 * 4096, sampler=sampler)
    print(f"ferromagnet R-hat (energy, magnetisation): {sampler.last_rhat[0]}")
    assert max(sampler.last_rhat[0]) > 1.1


def test_rhat_is_nan_below_two_records_per_half():
    gm = FactorGraph(3, 14, "spin", three_body_model(14, 14))
    sampler = B200Gibbs(seed=1, chains=1024, burn_in=10, thin=1)
    gml_b200.sample(gm, 3 * 1024, sampler=sampler)
    assert np.isnan(sampler.last_rhat[0]).all()
    gml_b200.sample(gm, 4 * 1024, sampler=sampler)
    assert np.isfinite(sampler.last_rhat[0]).all()


def test_order3_sample_learns_back():
    """three_body_model(30, 30) (ring couplings +-0.3, triples +-0.4), 1e6 draws, multiRISE(order 3).  Every one of the
    30 + 435 + 4060 coefficients within 0.05: the L1 shrinkage at lambda = 0.4 sqrt(log(N^2 / 0.05) / M) ~ 1.3e-3 and the
    statistical spread at 1e6 draws are a few 1e-3 (a B200 run measured a max error of 0.0065), so 0.05 leaves a 10x margin
    for other seeds while staying far below the smallest true coefficient (0.3): a sampler that drew from the wrong
    distribution fails it."""
    n = 30
    truth = three_body_model(n, 30)
    hist = gml_b200.sample(FactorGraph(3, n, "spin", truth), 1_000_000, sampler=B200Gibbs(seed=2))
    learned = gml_b200.learn(hist, multiRISE(0.4, True, 3), B200())
    err = max(abs(v - truth.get(k, 0.0)) for k, v in learned.terms.items())
    print(f"order-3 N=30: max coefficient error {err:.4f} over {len(learned.terms)} coefficients")
    assert len(learned.terms) == 30 + 435 + 4060 and err <= 0.05


def test_refusals():
    gm = FactorGraph.from_matrix(random_ising(10, 10))
    lib = _lib.load()
    idx = np.array([[0, 1]], dtype=np.int32)
    K, rhat = np.zeros(2, dtype=np.int64), np.zeros((2, 2))

    def call(N=10, order=2, ti=idx, w=0.1, n=10, reps=1, chains=0, burn_in=10, thin=1):
        wts = np.array([w])
        return lib.gml_b200_sample_mcmc_device(0, N, order, 1, ti.ctypes.data, wts.ctypes.data, n, reps, chains, burn_in,
                                               thin, 0, K.ctypes.data, rhat.ctypes.data, None, None, 0, None)

    assert call() == _lib.OK
    bad = [dict(N=0), dict(N=4097), dict(order=0, ti=np.array([[0]], dtype=np.int32)),
           dict(order=9, ti=np.arange(9, dtype=np.int32)[None, :]), dict(ti=np.array([[0, 10]], dtype=np.int32)),
           dict(ti=np.array([[0, -2]], dtype=np.int32)), dict(ti=np.array([[3, 3]], dtype=np.int32)), dict(w=float("inf")),
           dict(w=float("nan")), dict(n=0), dict(reps=0), dict(chains=-1), dict(burn_in=-1), dict(thin=0),
           dict(N=64, n=2 ** 31)]
    for kw in bad:
        assert call(**kw) == _lib.EINVAL, kw
    for terms in ({(1, 11): 0.1}, {(1, 2): float("nan")}, {(2, 2): 0.1}):
        with pytest.raises(gml_b200.GMLB200Error) as e:
            gml_b200.sample(FactorGraph(2, 10, "spin", terms), 10, sampler=B200Gibbs())
        assert e.value.code == _lib.EINVAL, terms
    with pytest.raises(ValueError):
        gml_b200.sample(gm, 10, sampler=B200Gibbs(), return_log_z=True)


@pytest.mark.parametrize("chains", [32, 160, 2000])
def test_chain_counts_that_leave_warps_of_the_last_block_empty(chains):
    """Chain counts that are not a multiple of a block's 128 chains (the last block has warps without chains) and that
    give every half-chain at least 2 records: a full histogram, the same rows again, and finite R-hat that the count-only
    call reproduces."""
    gm = FactorGraph(3, 14, "spin", three_body_model(14, 14))
    n = 8 * chains + 5
    sampler = B200Gibbs(seed=9, chains=chains, burn_in=50, thin=2)
    h = gml_b200.sample(gm, n, sampler=sampler)
    rhat = np.array(sampler.last_rhat)
    assert h[:, 0].sum() == n and (h[:, 0] > 0).all() and set(np.unique(h[:, 1:])) <= {-1, 1}
    assert (np.diff(config_index(h[:, 1:].T).astype(np.int64)) > 0).all()
    assert np.isfinite(rhat).all() and (rhat > 0.5).all() and (rhat < 2.0).all(), rhat
    assert np.array_equal(h, gml_b200.sample(gm, n, sampler=B200Gibbs(seed=9, chains=chains, burn_in=50, thin=2)))
    rc, K, rhat2 = mcmc_call(gm, n, 1, sampler)
    assert rc == _lib.OK and K.tolist() == [h.shape[0]] and np.array_equal(rhat, rhat2)
    # beyond 64 spins: one row per draw, all of them written
    _, big = c2_graph()
    counts, spins = gml_b200.sample_device(big, 4 * chains + 3, sampler=B200Gibbs(seed=9, chains=chains, burn_in=20, thin=1))
    assert (counts.cpu().numpy() == 1).all() and set(np.unique(spins.cpu().numpy())) <= {-1, 1}


def test_rhat_of_statistics_that_never_change():
    """W = 0: a constant statistic has R-hat 1, chains frozen at different values have R-hat +inf."""
    sampler = B200Gibbs(seed=2, chains=256, burn_in=5, thin=1)
    gml_b200.sample(FactorGraph(2, 10, "spin", {}), 1024, sampler=sampler)         # no terms: the energy is always 0
    assert sampler.last_rhat[0][0] == 1.0 and np.isfinite(sampler.last_rhat[0][1])
    gml_b200.sample(FactorGraph(2, 1, "spin", {(1,): 20.0}), 1024, sampler=sampler)  # one spin pinned up
    assert sampler.last_rhat[0] == (1.0, 1.0)
    gml_b200.sample(FactorGraph(2, 2, "spin", {(1, 2): 20.0}), 1024, sampler=sampler)  # aligned pair, frozen at ++ or --
    assert sampler.last_rhat[0][0] == 1.0 and sampler.last_rhat[0][1] == float("inf")


def test_term_sampler_output_is_pinned():
    """The one-draw-per-chain term sampler (gml_b200_sample_gibbs_terms_device) builds its incidence lists with the helper
    the MCMC sampler shares; its output for these fixed seeds is pinned to the bytes it produced before that helper
    existed (sha256 prefixes of the int8 spin block)."""
    import hashlib
    for terms, n, digest in ((three_body_model(30, 30), 30, "165576566771b00f"),
                             (FactorGraph.from_matrix(lattice_model()[0]).terms, 100, "06066ec417a74dba"),
                             (FactorGraph.from_matrix(random_ising(20, 3)).terms, 20, "56b1993b51ea03fa")):
        spins = gml_b200.sample_terms_device(terms, n, 200_000, sweeps=60, seed=1)
        assert hashlib.sha256(spins.cpu().numpy().tobytes()).hexdigest()[:16] == digest, n
