"""The replica-exchange sampler (csrc/mcmc_sampler.cu with R > 1 rungs, sample(gm, n, replicates, B200Tempering())):
moments against exact enumeration on a ferromagnet that B200Gibbs cannot mix, swap rates against their exact expectation,
R-hat on an 8 x 8 ferromagnet, the output contract, sample -> learn at N = 100, refusals, and the B200Gibbs output pinned
to the bytes of the sampler before the ladder existed.  Every seed is fixed."""
import ctypes
import hashlib

import numpy as np
import pytest
from scipy import stats

import gml_b200
from gml_b200 import B200, B200Gibbs, B200Tempering, FactorGraph, RISE, Session, _lib
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


def tempering_call(gm, n, reps, sampler, counts=None, spins=None, ld=0):
    """gml_b200_sample_tempering_device with raw buffers (None = count-only); returns (rc, K, rhat, swap_rate)."""
    order, idx, wts = term_arrays(gm)
    betas = None if sampler.betas is None else np.asarray(sampler.betas, dtype=np.float64)
    R = _lib.TEMPERING_DEFAULT_RUNGS if betas is None else len(betas)
    K, rhat, swap = np.zeros(reps, dtype=np.int64), np.zeros((reps, 2)), np.zeros((reps, R - 1))
    rc = _lib.load().gml_b200_sample_tempering_device(
        0, gm.varible_count, order, len(wts), idx.ctypes.data, wts.ctypes.data, 0 if betas is None else R,
        None if betas is None else betas.ctypes.data, n, reps, sampler.chains, sampler.burn_in, sampler.thin, sampler.seed,
        K.ctypes.data, rhat.ctypes.data, swap.ctypes.data, counts, spins, ld, None)
    return rc, K, rhat, swap


def open_ferromagnet(rows, cols, J, h=0.0):
    m = np.zeros((rows * cols, rows * cols))
    for r in range(rows):
        for c in range(cols):
            i = r * cols + c
            m[i, i] = h
            for j in ([i + 1] if c + 1 < cols else []) + ([i + cols] if r + 1 < rows else []):
                m[i, j] = m[j, i] = J
    return FactorGraph.from_matrix(m)


FERRO_4X5 = open_ferromagnet(4, 5, 1.5, 0.05)          # exact P(m > 0) = 0.881
ORDER3_N14 = FactorGraph(3, 14, "spin", {k: 2.0 * v for k, v in three_body_model(14, 14).items()})


def moments_t(gm, sampler, draws=200_000, R=32):
    """max |t| of the magnetisations and pair correlations of R replicates against enumeration, and the Student-t /
    Bonferroni threshold at family-wise rate 1e-6 (as in test_gpu_mcmc_sampler.test_moments_match_enumeration)."""
    n_spins = gm.varible_count
    e = log_weights(gm.terms, n_spins)
    p = np.exp(e - logsumexp(e))
    conf = ((np.arange(2 ** n_spins)[:, None] >> np.arange(n_spins)) & 1) * 2.0 - 1.0
    iu = np.triu_indices(n_spins, 1)
    exact = np.concatenate([p @ conf, ((conf * p[:, None]).T @ conf)[iu]])
    vals = []
    for h in gml_b200.sample(gm, draws, R, sampler):
        w = h[:, 0] / draws
        s = h[:, 1:].astype(np.float64)
        vals.append(np.concatenate([w @ s, ((s * w[:, None]).T @ s)[iu]]))
    vals = np.array(vals)
    t = np.abs(vals.mean(axis=0) - exact) / (vals.std(axis=0, ddof=1) / np.sqrt(R))
    return t.max(), stats.t.isf(1e-6 / (2 * len(exact)), R - 1)


@pytest.mark.parametrize("name,gm,gibbs_fails", [("ferromagnet 4x5 J=1.5", FERRO_4X5, True),
                                                 ("order-3 N=14 x2", ORDER3_N14, False)])
def test_moments_match_enumeration(name, gm, gibbs_fails):
    """B200Tempering (default ladder) passes; on the ferromagnet B200Gibbs with the same draws and seed fails the same
    check, so the swaps are what does the work."""
    t, thr = moments_t(gm, B200Tempering(seed=7))
    print(f"{name}: B200Tempering max |t| {t:.2f} (threshold {thr:.2f})")
    assert t <= thr
    if gibbs_fails:
        t_gibbs, _ = moments_t(gm, B200Gibbs(seed=7))
        print(f"{name}: B200Gibbs max |t| {t_gibbs:.2f}")
        assert t_gibbs > thr


def test_swap_rates_match_enumeration():
    """In equilibrium the rungs are independent, so pair (a, b) accepts with probability
    sum_x sum_y p_a(x) p_b(y) min(1, exp((beta_a - beta_b) (E(y) - E(x)))); 16 replicates against it with the Student-t
    bound.  A wrong sign, rung lookup or energy would show here even where the beta = 1 moments look right."""
    gm = FactorGraph.from_matrix(2.0 * random_ising(10, 10))
    betas = [1.0, 0.7, 0.4, 0.1]
    e = log_weights(gm.terms, 10)
    p = [np.exp(b * e - logsumexp(b * e)) for b in betas]
    expected = np.array([p[k] @ np.minimum(1.0, np.exp((betas[k] - betas[k + 1]) * (e[None, :] - e[:, None]))) @ p[k + 1]
                         for k in range(3)])
    sampler = B200Tempering(seed=4, betas=betas)
    R = 16
    gml_b200.sample_device(gm, 100_000, R, sampler)
    rates = np.array(sampler.last_swap_rate)
    assert rates.shape == (R, 3)
    t = np.abs(rates.mean(axis=0) - expected) / (rates.std(axis=0, ddof=1) / np.sqrt(R))
    thr = stats.t.isf(1e-6 / (2 * 3), R - 1)
    print(f"swap rates {rates.mean(axis=0)} expected {expected}, max |t| {t.max():.2f} (threshold {thr:.2f})")
    assert t.max() <= thr


def test_rhat_on_a_ferromagnet_gibbs_cannot_mix():
    """8 x 8 open ferromagnet at J = 1 (N = 64, the last size on the key path), 1024 chains, 40 records each at the
    default burn_in and thin.  On a B200 the magnetisation R-hat was 50.5 for B200Gibbs, 1.077 for B200Tempering's default
    ladder and 1.038 for 32 rungs geometric from 1 to 0.1, the ladder used here: the bound 1.1 leaves a margin of 0.06 above
    it and sits far below Gibbs' value."""
    gm = open_ferromagnet(8, 8, 1.0)
    n = 40 * 1024
    gibbs = B200Gibbs(seed=5, chains=1024)
    gml_b200.sample_device(gm, n, sampler=gibbs)
    temper = B200Tempering(seed=5, chains=1024, betas=np.geomspace(1.0, 0.1, 32).tolist())
    gml_b200.sample_device(gm, n, sampler=temper)
    print(f"8x8 ferromagnet R-hat (energy, magnetisation): B200Gibbs {gibbs.last_rhat[0]}, B200Tempering "
          f"{temper.last_rhat[0]}, swap rates {np.round(temper.last_swap_rate[0], 3).tolist()}")
    assert gibbs.last_rhat[0][1] > 1.1
    assert temper.last_rhat[0][1] <= 1.1


def test_output_contract():
    gm = FactorGraph(3, 14, "spin", three_body_model(14, 14))

    def make(seed=11):
        return B200Tempering(seed=seed, burn_in=50, thin=2, betas=[1.0, 0.6, 0.3, 0.1])

    sampler = make()
    reps = gml_b200.sample(gm, 50_000, 3, sampler)
    reps_rhat, reps_swap = np.array(sampler.last_rhat), np.array(sampler.last_swap_rate)
    assert len(reps) == 3 and reps_rhat.shape == (3, 2) and reps_swap.shape == (3, 3)
    assert ((reps_swap > 0) & (reps_swap <= 1)).all()
    for h in reps:
        assert h.dtype == np.int64 and h.shape[1] == 15
        assert h[:, 0].sum() == 50_000 and (h[:, 0] > 0).all()
        assert set(np.unique(h[:, 1:])) <= {-1, 1}
        assert (np.diff(config_index(h[:, 1:].T).astype(np.int64)) > 0).all()
    assert not np.array_equal(reps[0], reps[1])
    # bit-identical for the same arguments, different for another seed; replicate 0 is the single-replicate call
    again = make()
    assert all(np.array_equal(x, y) for x, y in zip(reps, gml_b200.sample(gm, 50_000, 3, again)))
    assert np.array_equal(np.array(again.last_swap_rate), reps_swap)
    one = make()
    assert np.array_equal(reps[0], gml_b200.sample(gm, 50_000, sampler=one))
    assert one.last_swap_rate == [reps_swap[0].tolist()]
    assert not np.array_equal(reps[0], gml_b200.sample(gm, 50_000, sampler=make(12)))
    # the device form holds the same rows
    counts, spins = gml_b200.sample_device(gm, 50_000, sampler=sampler)
    assert np.array_equal(counts.cpu().numpy(), reps[0][:, 0]) and np.array_equal(spins.cpu().numpy(), reps[0][:, 1:].T)
    # count-only and host-buffer calls agree with the device-buffer call; a too-small ld is refused with out_K filled
    rc, K, rhat, swap = tempering_call(gm, 50_000, 3, sampler)
    assert rc == _lib.OK and K.tolist() == [h.shape[0] for h in reps]
    assert np.array_equal(rhat, reps_rhat, equal_nan=True) and np.array_equal(swap, reps_swap)
    rows = int(K.sum())
    hc, hs = np.zeros(rows), np.zeros((14, rows), dtype=np.int8)
    rc, _, rhat, swap = tempering_call(gm, 50_000, 3, sampler, hc.ctypes.data, hs.ctypes.data, rows)
    assert rc == _lib.OK
    assert np.array_equal(rhat, reps_rhat, equal_nan=True) and np.array_equal(swap, reps_swap)
    assert np.array_equal(np.concatenate([h[:, 0] for h in reps]), hc)
    assert np.array_equal(np.concatenate([h[:, 1:] for h in reps]).T, hs)
    rc, K2, _, _ = tempering_call(gm, 50_000, 3, sampler, hc.ctypes.data, hs.ctypes.data, rows - 1)
    assert rc == _lib.EINVAL and np.array_equal(K, K2)
    # the default ladder: 15 swap rates per replicate
    default = B200Tempering(seed=11, burn_in=50, thin=2)
    gml_b200.sample(gm, 10_000, 2, default)
    assert np.array(default.last_swap_rate).shape == (2, _lib.TEMPERING_DEFAULT_RUNGS - 1)


def test_output_contract_beyond_64_spins():
    """N = 100: one row of count 1 per draw, in draw order."""
    import torch
    gm = FactorGraph.from_matrix(lattice_model()[0])

    def make(seed=3):
        return B200Tempering(seed=seed, burn_in=20, thin=1, chains=256, betas=[1.0, 0.8, 0.6, 0.5, 0.4, 0.3, 0.2, 0.1])

    sampler = make()
    n = 5 * 256 + 100                                # 5 full record steps of 256 ladders and a partial sixth
    h = gml_b200.sample(gm, n, sampler=sampler)
    assert h.shape == (n, 101) and (h[:, 0] == 1).all() and set(np.unique(h[:, 1:])) <= {-1, 1}
    swap = np.array(sampler.last_swap_rate)
    two = gml_b200.sample(gm, n, 2, sampler)
    assert isinstance(two, list) and np.array_equal(two[0], h) and not np.array_equal(two[0], two[1])
    assert np.array_equal(np.array(sampler.last_swap_rate)[0], swap[0])
    assert np.array_equal(h, gml_b200.sample(gm, n, sampler=make()))
    assert not np.array_equal(h, gml_b200.sample(gm, n, sampler=make(4)))
    counts, spins = gml_b200.sample_device(gm, n, sampler=sampler)
    assert counts.numel() == n and np.array_equal(spins.cpu().numpy(), h[:, 1:].T)
    rc, K, _, swap2 = tempering_call(gm, n, 2, sampler)
    assert rc == _lib.OK and K.tolist() == [n, n] and np.array_equal(swap2[0], swap[0])
    hc, hs = np.zeros(2 * n), np.zeros((100, 2 * n), dtype=np.int8)
    assert tempering_call(gm, n, 2, sampler, hc.ctypes.data, hs.ctypes.data, 2 * n)[0] == _lib.OK
    assert (hc == 1).all() and np.array_equal(hs[:, :n], h[:, 1:].T) and np.array_equal(hs[:, n:], two[1][:, 1:].T)
    small_c = torch.empty(2 * n - 1, dtype=torch.float64, device="cuda:0")
    small_s = torch.empty((100, 2 * n - 1), dtype=torch.int8, device="cuda:0")
    rc, K2, _, _ = tempering_call(gm, n, 2, sampler, small_c.data_ptr(), small_s.data_ptr(), 2 * n - 1)
    assert rc == _lib.EINVAL and K2.tolist() == [n, n]


@pytest.mark.parametrize("rungs,chains", [(2, 48), (8, 20), (32, 5), (16, 3)])
def test_chain_counts_that_leave_warps_of_the_last_block_empty(rungs, chains):
    """Ladder counts whose last block has warps without ladders (and, for 8 and 16 rungs, a partly filled warp), with
    every half-chain holding at least 2 records: a full histogram, the same rows again, finite R-hat and swap rates in
    (0, 1] that the count-only call reproduces, and all rows written beyond 64 spins."""
    gm = FactorGraph(3, 14, "spin", three_body_model(14, 14))
    betas = list(np.geomspace(1.0, 0.2, rungs))
    n = 8 * chains + 5
    sampler = B200Tempering(seed=9, chains=chains, burn_in=50, thin=2, betas=betas)
    h = gml_b200.sample(gm, n, sampler=sampler)
    rhat, swap = np.array(sampler.last_rhat), np.array(sampler.last_swap_rate)
    assert h[:, 0].sum() == n and (h[:, 0] > 0).all() and set(np.unique(h[:, 1:])) <= {-1, 1}
    assert (np.diff(config_index(h[:, 1:].T).astype(np.int64)) > 0).all()
    assert np.isfinite(rhat).all() and (rhat > 0.5).all() and (rhat < 3.0).all(), rhat
    assert swap.shape == (1, rungs - 1) and ((swap > 0) & (swap <= 1)).all(), swap
    assert np.array_equal(h, gml_b200.sample(gm, n, sampler=B200Tempering(seed=9, chains=chains, burn_in=50, thin=2,
                                                                          betas=betas)))
    rc, K, rhat2, swap2 = tempering_call(gm, n, 1, sampler)
    assert rc == _lib.OK and K.tolist() == [h.shape[0]] and np.array_equal(rhat, rhat2) and np.array_equal(swap, swap2)
    big = FactorGraph.from_matrix(lattice_model()[0])
    counts, spins = gml_b200.sample_device(big, 4 * chains + 3, sampler=B200Tempering(seed=9, chains=chains, burn_in=20,
                                                                                      thin=1, betas=betas))
    assert (counts.cpu().numpy() == 1).all() and set(np.unique(spins.cpu().numpy())) <= {-1, 1}


def test_c2_sample_learns_back():
    """1e6 draws of the C2 lattice (N = 100, the row path) at the defaults: RISE couplings and fields within 0.02 (the bar
    of the B200Gibbs test) and both R-hats at most 1.01."""
    truth = lattice_model()[0]
    sampler = B200Tempering(seed=1)
    counts, spins = gml_b200.sample_device(FactorGraph.from_matrix(truth), 1_000_000, sampler=sampler)
    assert counts.numel() == 1_000_000
    sess = Session(0).attach_device(counts.data_ptr(), spins.data_ptr(), counts.numel(), 100, spins.stride(0))
    theta = sess.solve_pairwise(RISE(0.4, False), B200())
    off = theta - np.diag(np.diag(theta))
    print(f"C2: max coupling error {np.abs(off - truth).max():.4f}, max field {np.abs(np.diag(theta)).max():.4f}, "
          f"R-hat {sampler.last_rhat[0]}")
    assert np.abs(off - truth).max() <= 0.02
    assert np.abs(np.diag(theta)).max() <= 0.02
    assert max(sampler.last_rhat[0]) <= 1.01


def test_refusals():
    gm = FactorGraph.from_matrix(random_ising(10, 10))
    lib = _lib.load()
    idx = np.array([[0, 1]], dtype=np.int32)
    K, rhat, swap = np.zeros(2, dtype=np.int64), np.zeros((2, 2)), np.zeros((2, 31))

    def call(N=10, order=2, ti=idx, w=0.1, n=10, reps=1, chains=0, burn_in=10, thin=1, betas=(1.0, 0.5), n_rungs=None):
        wts = np.array([w])
        b = None if betas is None else np.array(betas, dtype=np.float64)
        n_rungs = (0 if b is None else len(b)) if n_rungs is None else n_rungs
        return lib.gml_b200_sample_tempering_device(0, N, order, 1, ti.ctypes.data, wts.ctypes.data, n_rungs,
                                                    None if b is None else b.ctypes.data, n, reps, chains, burn_in, thin, 0,
                                                    K.ctypes.data, rhat.ctypes.data, swap.ctypes.data, None, None, 0, None)

    assert call() == _lib.OK and call(betas=None) == _lib.OK
    bad = [dict(N=0), dict(N=4097), dict(order=0, ti=np.array([[0]], dtype=np.int32)),
           dict(order=9, ti=np.arange(9, dtype=np.int32)[None, :]), dict(ti=np.array([[0, 10]], dtype=np.int32)),
           dict(ti=np.array([[0, -2]], dtype=np.int32)), dict(ti=np.array([[3, 3]], dtype=np.int32)), dict(w=float("inf")),
           dict(w=float("nan")), dict(n=0), dict(reps=0), dict(chains=-1), dict(burn_in=-1), dict(thin=0),
           dict(N=64, n=2 ** 31),
           dict(betas=(1.0,)), dict(betas=(1.0, 0.5, 0.2)), dict(betas=tuple(np.geomspace(1, 0.1, 64))),
           dict(betas=None, n_rungs=2), dict(betas=(1.0, 0.5), n_rungs=0), dict(betas=(0.9, 0.5)),
           dict(betas=(1.0, 1.0)), dict(betas=(1.0, 0.5, 0.6, 0.1)), dict(betas=(1.0, -0.5)), dict(betas=(1.0, float("nan"))),
           dict(betas=(1.0, float("-inf")))]
    for kw in bad:
        assert call(**kw) == _lib.EINVAL, kw
    for terms in ({(1, 11): 0.1}, {(1, 2): float("nan")}, {(2, 2): 0.1}):
        with pytest.raises(gml_b200.GMLB200Error) as e:
            gml_b200.sample(FactorGraph(2, 10, "spin", terms), 10, sampler=B200Tempering())
        assert e.value.code == _lib.EINVAL, terms
    for kw in (dict(return_log_z=True),):
        with pytest.raises(ValueError):
            gml_b200.sample(gm, 10, sampler=B200Tempering(), **kw)
    with pytest.raises(ValueError):
        gml_b200.sample(gm, 10, sampler=B200Tempering(betas=[1.0, 0.5, 0.1]))


# ---- B200Gibbs output, pinned to the bytes of the sampler before the ladder existed -------------------------------
def gibbs_digest(lib, gm, n, reps, seed, chains, burn_in, thin):
    """sha256 prefix of the counts and spins that gml_b200_sample_mcmc_device writes into host buffers, and of its R-hat.
    `lib` is any build of the library, so the same digest can be taken from an older one."""
    c = ctypes
    lib.gml_b200_sample_mcmc_device.argtypes = [c.c_int32, c.c_int32, c.c_int32, c.c_int32, c.c_void_p, c.c_void_p,
                                                c.c_int64, c.c_int32, c.c_int64, c.c_int32, c.c_int32, c.c_uint64, c.c_void_p,
                                                c.c_void_p, c.c_void_p, c.c_void_p, c.c_int64, c.c_void_p]
    order, idx, wts = term_arrays(gm)
    N = gm.varible_count
    ld = reps * min(n, 1 << N)
    K, rhat = np.zeros(reps, dtype=np.int64), np.zeros((reps, 2))
    counts, spins = np.zeros(ld), np.zeros((N, ld), dtype=np.int8)
    rc = lib.gml_b200_sample_mcmc_device(0, N, order, len(wts), idx.ctypes.data, wts.ctypes.data, n, reps, chains, burn_in,
                                         thin, seed, K.ctypes.data, rhat.ctypes.data, counts.ctypes.data, spins.ctypes.data,
                                         ld, None)
    assert rc == 0
    rows = int(K.sum())
    return hashlib.sha256(K.tobytes() + counts[:rows].tobytes() + np.ascontiguousarray(spins[:, :rows]).tobytes() +
                          rhat.tobytes()).hexdigest()[:16]


PINNED_GIBBS = [  # (name, model, n, replicates, seed, chains, burn_in, thin, sha256 prefix)
    ("order-3 N=14", lambda: FactorGraph(3, 14, "spin", three_body_model(14, 14)), 50_000, 2, 11, 0, 50, 2, "a9500f18636728a9"),
    ("pairwise N=20", lambda: FactorGraph.from_matrix(random_ising(20, 20)), 100_000, 2, 7, 1000, 100, 3, "314e68c110c5449c"),
    ("C2 N=100", lambda: FactorGraph.from_matrix(lattice_model()[0]), 20_000, 2, 3, 0, 30, 1, "451e8f1681ea538f"),
]


def test_gibbs_output_is_pinned():
    """B200Gibbs (R = 1 of the shared kernel) writes, for these fixed seeds, the bytes the sampler wrote before it gained
    the ladder: counts, spins and R-hat, as sha256 prefixes taken on a B200 at that commit."""
    lib = _lib.load()
    for name, model, n, reps, seed, chains, burn_in, thin, digest in PINNED_GIBBS:
        assert gibbs_digest(lib, model(), n, reps, seed, chains, burn_in, thin) == digest, name
