"""The Swendsen-Wang sampler (cluster_kernel in csrc/mcmc_sampler.cu, sample(gm, n, replicates, B200SwendsenWang())):
moments against enumeration on a ferromagnet that B200Gibbs cannot mix, an antiferromagnet, a frustrated model, fields
only and no terms; closed forms beyond 64 spins (periodic ring, Curie-Weiss, disconnected blocks); moments equal to the
sampler's own draws bit for bit; R-hat on lattices that B200Gibbs and B200Tempering do not mix; sample -> learn at C2;
and the output contract.  Every seed is fixed.

The chains sample the model with weights w' whose bond probabilities are exact to 64 bits: |w'_t - w_t| <= 2^-52 +
2^-64 e^{2|w_t|} (DESIGN 4.9), so the moments of w' differ from those of w by at most e^{2 delta} - 1, delta = sum_t of
that bound; the bars below add it, as test_gpu_moments adds the fp32 rounding of the Gibbs chains."""
import math

import numpy as np
import pytest

import gml_b200
from gml_b200 import B200, B200SwendsenWang, FactorGraph, RISE, Session, _lib
from helpers import random_ising
from test_gpu_exact_sampler import config_index, log_weights, logsumexp
from test_gpu_fullsize import lattice_model
from test_gpu_log_partition import curie_weiss, ring
from test_gpu_moments import k_bar, pairwise_keys, values
from test_gpu_tempering_sampler import FERRO_4X5, moments_t, open_ferromagnet

pytestmark = pytest.mark.gpu


def sw_bound(gm):
    """e^{2 delta} - 1 with delta = sum_t (2^-52 + 2^-64 e^{2|w_t|}): the most a moment of the sampled model can differ"""
    w = np.abs(np.array(list(gm.terms.values()), dtype=np.float64))
    return math.expm1(2.0 * float(np.sum(2.0 ** -52 + 2.0 ** -64 * np.exp(2.0 * w))))


def exact_pairwise(gm):
    """<s_i> on the diagonal and <s_i s_j> off it, by enumeration"""
    n = gm.varible_count
    e = log_weights(gm.terms, n)
    p = np.exp(e - logsumexp(e))
    S = ((np.arange(2 ** n)[:, None] >> np.arange(n)) & 1) * 2.0 - 1.0
    C = S.T @ (S * p[:, None])
    np.fill_diagonal(C, p @ S)
    return C


# ---- against enumeration --------------------------------------------------------------------------------------------
ENUMERATED = [  # (name, model, burn_in); max |t| measured on a B200 in the comment (thresholds 7.5-8.0)
    ("ferromagnet 4x5 J=1.5 h=0.05", FERRO_4X5, 200),                                          # 3.16
    ("antiferromagnet 4x5 J=-1.5", open_ferromagnet(4, 5, -1.5), 200),                         # 2.53
    # frustrated: cluster moves mix slower than Gibbs here; burn_in 200 measured max |t| 92.4, 2000 gives 2.44
    ("2 random_ising(16, 16)", FactorGraph.from_matrix(2.0 * random_ising(16, 16)), 2000),    # 2.44
    ("fields only N=12", FactorGraph(1, 12, "spin", {(i + 1,): 0.25 * (i - 6) for i in range(12)}), 200),   # 2.62
    ("no terms N=10", FactorGraph(2, 10, "spin", {}), 200),                                     # 2.59
]


@pytest.mark.parametrize("name,gm,burn_in", ENUMERATED, ids=[e[0] for e in ENUMERATED])
def test_moments_match_enumeration(name, gm, burn_in):
    """32 replicates of 2e5 draws against enumeration, Student-t / Bonferroni at family-wise rate 1e-6 (B200Gibbs fails
    the same check on the ferromagnet, max |t| 1283)."""
    assert sw_bound(gm) < 1e-12
    t, thr = moments_t(gm, B200SwendsenWang(seed=7, burn_in=burn_in))
    print(f"{name}: B200SwendsenWang max |t| {t:.2f} (threshold {thr:.2f})")
    assert t <= thr


# ---- closed forms beyond 64 spins -----------------------------------------------------------------------------------
def test_periodic_ring_pairwise():
    """N = 1000, J = 2: <s_i s_j> = (t^d + t^(N-d)) / (1 + t^N), t = tanh J, on the draw-row path"""
    N, J = 1000, 2.0
    t = math.tanh(J)
    d = np.abs(np.arange(N)[:, None] - np.arange(N)[None, :])
    exact = (t ** d + t ** (N - d)) / (1 + t ** N)
    np.fill_diagonal(exact, 0.0)
    gm = ring(N, J)
    C, Ce = gml_b200.moments(gm, B200SwendsenWang(seed=2, chains=8192, burn_in=50, thin=2), 200_000, keys="pairwise")
    print(f"ring N=1000 J=2: max |error| {np.abs(C - exact).max():.2e}, max stderr {Ce.max():.2e}")
    assert (np.abs(C - exact) <= k_bar(N * N) * Ce + sw_bound(gm)).all()


def test_curie_weiss_ordered_phase():
    """N = 256, every pair at J / N with J = 1.5 (the ordered phase): the formula of test_gpu_moments.test_curie_weiss"""
    from scipy import special
    n, J = 256, 1.5
    k = np.arange(n + 1)
    M = 2.0 * k - n
    logw = special.gammaln(n + 1) - special.gammaln(k + 1) - special.gammaln(n - k + 1) + J * (M * M - n) / (2.0 * n)
    w = np.exp(logw - logw.max())
    pair = ((w @ (M * M)) / w.sum() - n) / (n * (n - 1))
    exact = np.full((n, n), pair)
    np.fill_diagonal(exact, 0.0)
    gm = curie_weiss(n, J)
    C, Ce = gml_b200.moments(gm, B200SwendsenWang(seed=3, chains=1024, burn_in=100), 100_000, keys="pairwise")
    print(f"Curie-Weiss J={J}: <s_i s_j> exact {pair:.4f}, max |error| {np.abs(C - exact).max():.2e}, max stderr {Ce.max():.2e}")
    assert (np.abs(C - exact) <= k_bar(n * n) * Ce + sw_bound(gm)).all()


def test_disconnected_blocks_factorise():
    """Five disconnected copies of FERRO_4X5 (N = 100): each block's fields and pairs against enumeration of one block,
    and the pairs across blocks against the products of the exact fields."""
    B, nb = 5, 20
    terms = {tuple(i + b * nb for i in key): v for b in range(B) for key, v in FERRO_4X5.terms.items()}
    gm = FactorGraph(2, B * nb, "spin", terms)
    one = exact_pairwise(FERRO_4X5)
    field = np.tile(np.diag(one), B)
    exact = np.outer(field, field)
    for b in range(B):
        exact[b * nb:(b + 1) * nb, b * nb:(b + 1) * nb] = one
    n = 200_000
    C, Ce = gml_b200.moments(gm, B200SwendsenWang(seed=4, chains=4096), n, keys="pairwise")
    # a corner pair has <s_i s_j> = 0.99995: about 5 of the draws disagree, and a sample where none does has a group
    # stderr of 0, so the stderr is floored at the iid value sqrt((1 - m^2) / n), which correlated draws only exceed
    err = np.maximum(Ce, np.sqrt((1.0 - exact ** 2) / n))
    print(f"5 x FERRO_4X5: max |error| {np.abs(C - exact).max():.2e}, max stderr {Ce.max():.2e}, "
          f"max |error| / stderr {(np.abs(C - exact) / err).max():.2f} (bar {k_bar(C.size):.2f})")
    assert (np.abs(C - exact) <= k_bar(C.size) * err + sw_bound(gm)).all()


# ---- moments equal the sampler's own draws --------------------------------------------------------------------------
@pytest.mark.parametrize("name,model,n,chains", [
    ("N=20 (histogram rows)", lambda: FactorGraph.from_matrix(random_ising(20, 20)), 12_345, 1000),
    ("N=100 (draw rows)", lambda: FactorGraph.from_matrix(lattice_model()[0]), 5_000, 256),
])
def test_moments_equal_own_draws(name, model, n, chains):
    gm = model()
    N = gm.varible_count

    def make():
        return B200SwendsenWang(seed=3, chains=chains, burn_in=30, thin=2)

    S1, S2 = make(), make()
    mean, err = gml_b200.moments(gm, S1, n)
    draws = gml_b200.sample(gm, n, 1, S2)
    assert draws[:, 0].sum() == n
    assert np.array_equal(values(mean), values(gml_b200.empirical_moments(draws, list(gm.terms)))), name
    assert np.array_equal(S1.last_rhat, S2.last_rhat, equal_nan=True)
    assert np.isfinite(values(err)).all() and (values(err) >= 0).all()
    keys = pairwise_keys(N)
    km, ke = gml_b200.moments(gm, make(), n, keys=keys)
    C, Ce = gml_b200.moments(gm, make(), n, keys="pairwise")
    for (k, m), e in zip(km.terms.items(), ke.terms.values()):
        i, j = (k[0] - 1, k[-1] - 1)
        assert C[i, j] == m and C[j, i] == m and Ce[i, j] == e and Ce[j, i] == e, k
    assert np.array_equal(values(km), values(gml_b200.empirical_moments(draws, keys)))


# ---- mixing ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("side,J", [(32, 1.0), (64, 0.44)])
def test_rhat_on_lattices_gibbs_cannot_mix(side, J):
    """1024 chains of 40 records at the defaults.  On the 32 x 32 J = 1 lattice B200Gibbs measured a magnetisation R-hat
    of 16.0 and 32-rung B200Tempering 1.099 (DESIGN 4.5)."""
    sampler = B200SwendsenWang(seed=5, chains=1024)
    gml_b200.sample_device(open_ferromagnet(side, side, J), 40 * 1024, sampler=sampler)
    print(f"{side}x{side} J={J}: R-hat (energy, magnetisation) {sampler.last_rhat[0]}")
    assert max(sampler.last_rhat[0]) <= 1.01


# ---- learning back --------------------------------------------------------------------------------------------------
def test_c2_sample_learns_back():
    """1e6 draws of the C2 lattice (N = 100) at the defaults: RISE couplings and fields within 0.02, the bar of the
    B200Gibbs and B200Tempering tests."""
    truth = lattice_model()[0]
    sampler = B200SwendsenWang(seed=1)
    counts, spins = gml_b200.sample_device(FactorGraph.from_matrix(truth), 1_000_000, sampler=sampler)
    sess = Session(0).attach_device(counts.data_ptr(), spins.data_ptr(), counts.numel(), 100, spins.stride(0))
    theta = sess.solve_pairwise(RISE(0.4, False), B200())
    off = theta - np.diag(np.diag(theta))
    print(f"C2: max coupling error {np.abs(off - truth).max():.4f}, max field {np.abs(np.diag(theta)).max():.4f}, "
          f"R-hat {sampler.last_rhat[0]}")
    assert np.abs(off - truth).max() <= 0.02
    assert np.abs(np.diag(theta)).max() <= 0.02
    assert max(sampler.last_rhat[0]) <= 1.01


# ---- output contract ------------------------------------------------------------------------------------------------
def cluster_call(gm, n, reps, sampler, counts=None, spins=None, ld=0):
    """gml_b200_sample_cluster_device with raw buffers (None = count-only); returns (rc, K, rhat)."""
    order, idx, wts = gml_b200.api._term_arrays(gm)
    K, rhat = np.zeros(reps, dtype=np.int64), np.zeros((reps, 2))
    rc = _lib.load().gml_b200_sample_cluster_device(0, gm.varible_count, order, len(gm.terms), idx.ctypes.data,
                                                    wts.ctypes.data, n, reps, sampler.chains, sampler.burn_in, sampler.thin,
                                                    sampler.seed, K.ctypes.data, rhat.ctypes.data, counts, spins, ld, None)
    return rc, K, rhat


def test_output_contract():
    gm = FactorGraph.from_matrix(random_ising(14, 14))

    def make(seed=11):
        return B200SwendsenWang(seed=seed, burn_in=50, thin=2)

    sampler = make()
    reps = gml_b200.sample(gm, 50_000, 3, sampler)
    reps_rhat = np.array(sampler.last_rhat)
    assert len(reps) == 3 and reps_rhat.shape == (3, 2)
    for h in reps:
        assert h.dtype == np.int64 and h.shape[1] == 15
        assert h[:, 0].sum() == 50_000 and (h[:, 0] > 0).all()
        assert set(np.unique(h[:, 1:])) <= {-1, 1}
        assert (np.diff(config_index(h[:, 1:].T).astype(np.int64)) > 0).all()     # sorted, deduplicated
    assert not np.array_equal(reps[0], reps[1])
    again = make()
    assert all(np.array_equal(x, y) for x, y in zip(reps, gml_b200.sample(gm, 50_000, 3, again)))
    assert np.array_equal(np.array(again.last_rhat), reps_rhat, equal_nan=True)
    assert np.array_equal(reps[0], gml_b200.sample(gm, 50_000, sampler=make()))
    assert not np.array_equal(reps[0], gml_b200.sample(gm, 50_000, sampler=make(12)))
    counts, spins = gml_b200.sample_device(gm, 50_000, sampler=sampler)
    assert np.array_equal(counts.cpu().numpy(), reps[0][:, 0]) and np.array_equal(spins.cpu().numpy(), reps[0][:, 1:].T)
    # count-only and host-buffer calls agree with the device-buffer call; a too-small ld is refused with out_K filled
    rc, K, rhat = cluster_call(gm, 50_000, 3, sampler)
    assert rc == _lib.OK and K.tolist() == [h.shape[0] for h in reps]
    assert np.array_equal(rhat, reps_rhat, equal_nan=True)
    rows = int(K.sum())
    hc, hs = np.zeros(rows), np.zeros((14, rows), dtype=np.int8)
    rc, _, _ = cluster_call(gm, 50_000, 3, sampler, hc.ctypes.data, hs.ctypes.data, rows)
    assert rc == _lib.OK
    assert np.array_equal(np.concatenate([h[:, 0] for h in reps]), hc)
    assert np.array_equal(np.concatenate([h[:, 1:] for h in reps]).T, hs)
    rc, K2, _ = cluster_call(gm, 50_000, 3, sampler, hc.ctypes.data, hs.ctypes.data, rows - 1)
    assert rc == _lib.EINVAL and np.array_equal(K, K2)


def test_output_contract_beyond_64_spins():
    """N = 100: one row of count 1 per draw, in draw order; replicate 0 is the single-replicate call; host buffers"""
    gm = FactorGraph.from_matrix(lattice_model()[0])

    def make(seed=3):
        return B200SwendsenWang(seed=seed, burn_in=20, thin=1, chains=256)

    n = 5 * 256 + 100
    h = gml_b200.sample(gm, n, sampler=make())
    assert h.shape == (n, 101) and (h[:, 0] == 1).all() and set(np.unique(h[:, 1:])) <= {-1, 1}
    two = gml_b200.sample(gm, n, 2, make())
    assert np.array_equal(two[0], h) and not np.array_equal(two[0], two[1])
    assert np.array_equal(h, gml_b200.sample(gm, n, sampler=make()))
    hc, hs = np.zeros(2 * n), np.zeros((100, 2 * n), dtype=np.int8)
    assert cluster_call(gm, n, 2, make(), hc.ctypes.data, hs.ctypes.data, 2 * n)[0] == _lib.OK
    assert (hc == 1).all() and np.array_equal(hs[:, :n], h[:, 1:].T) and np.array_equal(hs[:, n:], two[1][:, 1:].T)


@pytest.mark.parametrize("chains", [3, 20, 48, 33])
def test_chain_counts_that_leave_warps_empty(chains):
    """Chain counts whose last block has a warp without chains (two warps per block) or a partly filled warp, with every
    half-chain holding at least 2 records: a full histogram, the same rows again, finite R-hat, all rows beyond 64 spins."""
    gm = FactorGraph.from_matrix(random_ising(14, 14))
    n = 8 * chains + 5
    sampler = B200SwendsenWang(seed=9, chains=chains, burn_in=50, thin=2)
    h = gml_b200.sample(gm, n, sampler=sampler)
    rhat = np.array(sampler.last_rhat)
    assert h[:, 0].sum() == n and (h[:, 0] > 0).all() and set(np.unique(h[:, 1:])) <= {-1, 1}
    assert (np.diff(config_index(h[:, 1:].T).astype(np.int64)) > 0).all()
    assert np.isfinite(rhat).all() and (rhat > 0.5).all() and (rhat < 3.0).all(), rhat
    assert np.array_equal(h, gml_b200.sample(gm, n, sampler=B200SwendsenWang(seed=9, chains=chains, burn_in=50, thin=2)))
    big = FactorGraph.from_matrix(lattice_model()[0])
    counts, spins = gml_b200.sample_device(big, 4 * chains + 3, sampler=B200SwendsenWang(seed=9, chains=chains, burn_in=20,
                                                                                          thin=1))
    assert counts.numel() == 4 * chains + 3
    assert (counts.cpu().numpy() == 1).all() and set(np.unique(spins.cpu().numpy())) <= {-1, 1}

