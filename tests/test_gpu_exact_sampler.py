"""The exact device sampler (csrc/exact_sampler.cu) against enumeration of all 2^N weights: log Z, the multinomial law of
the counts, the output contract, sample -> learn end to end, and input refusals.  Every seed is fixed."""
import ctypes

import numpy as np
import pytest
from scipy import stats

import gml_b200
from gml_b200 import B200, B200Exact, FactorGraph, RISE, RPLE, Session, _lib, logRISE
from helpers import MODELS, random_ising, three_body_model

pytestmark = pytest.mark.gpu
FORMS = {"RISE": RISE, "logRISE": logRISE, "RPLE": RPLE}


def log_weights(terms, n):
    """sum_t w_t prod_{i in t} s_i for every configuration c (spin_i = 2*bit_i(c) - 1, bit 0 = spin 1), float64."""
    c = np.arange(2 ** n, dtype=np.uint64)
    e = np.zeros(2 ** n)
    for k, w in terms.items():
        mask = np.uint64(sum(1 << (i - 1) for i in k))
        e += np.where(np.bitwise_count(mask & ~c) & 1, -w, w)
    return e


def logsumexp(e):
    m = e.max()
    return m + np.log(np.exp(e - m).sum())


def config_index(spins):
    """configuration index of every row of an N x K int8 spin block"""
    bits = (np.asarray(spins) > 0).astype(np.uint64)
    return (bits << np.arange(bits.shape[0], dtype=np.uint64)[:, None]).sum(axis=0)


def pairwise(n, seed):
    return FactorGraph.from_matrix(random_ising(n, seed))


def full_counts(hist, n):
    """the histogram of sample() as counts over all 2^n configurations"""
    out = np.zeros(2 ** n, dtype=np.int64)
    out[config_index(hist[:, 1:].T)] = hist[:, 0]
    return out


@pytest.mark.parametrize("name,gm", [("pairwise N=12", pairwise(12, 12)),
                                     ("order-3 N=10", FactorGraph(3, 10, "spin", three_body_model(10, 10))),
                                     ("pairwise N=24", pairwise(24, 24))])
def test_log_z_matches_enumeration(name, gm):
    _, log_z = gml_b200.sample(gm, 1000, return_log_z=True)
    ref = logsumexp(log_weights(gm.terms, gm.varible_count))
    assert abs(log_z - ref) <= 1e-12 * abs(ref), (name, log_z, ref)


def test_counts_follow_the_multinomial_law():
    n, draws = 10, 10_000_000
    gm = pairwise(n, 10)
    e = log_weights(gm.terms, n)
    p = np.exp(e - logsumexp(e))
    got = full_counts(gml_b200.sample(gm, draws, sampler=B200Exact(seed=3)), n)
    mean = draws * p
    z = np.abs(got - mean) / np.sqrt(mean * (1 - p))
    chi2 = ((got - mean) ** 2 / mean).sum()
    print(f"max z {z.max():.2f}, chi2 {chi2:.1f} over {2 ** n} cells")
    assert z.max() <= 5.0
    assert chi2 <= stats.chi2.isf(1e-6, 2 ** n - 1)


def test_moments_match_enumeration_n20():
    n, draws = 20, 2_000_000
    gm = pairwise(n, 20)
    e = log_weights(gm.terms, n)
    p = np.exp(e - logsumexp(e))
    conf = ((np.arange(2 ** n)[:, None] >> np.arange(n)) & 1) * 2.0 - 1.0
    exact_c = (conf * p[:, None]).T @ conf
    exact_m = p @ conf
    hist = gml_b200.sample(gm, draws, sampler=B200Exact(seed=5)).astype(np.float64)
    w = hist[:, 0] / draws
    s = hist[:, 1:]
    corr = (s * w[:, None]).T @ s
    mag = w @ s
    zc = np.abs(corr - exact_c) / np.sqrt(np.maximum(1.0 - exact_c ** 2, 1e-3) / draws)
    zm = np.abs(mag - exact_m) / np.sqrt(np.maximum(1.0 - exact_m ** 2, 1e-3) / draws)
    print(f"max z corr {zc.max():.2f}, max z mag {zm.max():.2f}")
    assert zc.max() <= 5.0 and zm.max() <= 5.0


def test_output_contract():
    gm = FactorGraph(3, 14, "spin", three_body_model(14, 14))
    for n_draws in (1, 7, 50_000):
        reps = gml_b200.sample(gm, n_draws, 3, B200Exact(seed=11))
        assert len(reps) == 3
        for h in reps:
            assert h.dtype == np.int64 and h.shape[1] == 15
            assert h[:, 0].sum() == n_draws and (h[:, 0] > 0).all()
            assert h.shape[0] <= min(n_draws, 2 ** 14)
            assert set(np.unique(h[:, 1:])) <= {-1, 1}
            assert (np.diff(config_index(h[:, 1:].T).astype(np.int64)) > 0).all()
        if n_draws > 1:
            assert not np.array_equal(reps[0], reps[1]) and not np.array_equal(reps[1], reps[2])
    # bit-identical for the same seed, different for another; replicate 0 is the single-replicate draw
    a, b = gml_b200.sample(gm, 50_000, 2, B200Exact(seed=11)), gml_b200.sample(gm, 50_000, 2, B200Exact(seed=11))
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    assert np.array_equal(a[0], gml_b200.sample(gm, 50_000, sampler=B200Exact(seed=11)))
    assert not np.array_equal(a[0], gml_b200.sample(gm, 50_000, sampler=B200Exact(seed=12)))
    # the device form holds the same rows
    (counts, spins), log_z = gml_b200.sample_device(gm, 50_000, sampler=B200Exact(seed=11), return_log_z=True)
    assert np.array_equal(counts.cpu().numpy(), a[0][:, 0]) and np.array_equal(spins.cpu().numpy(), a[0][:, 1:].T)
    # a count-only call (no buffers) gives the same sizes and log Z; buffers that are too small are refused
    lib = _lib.load()
    idx = -np.ones((len(gm.terms), 3), dtype=np.int32)
    for t, k in enumerate(gm.terms):
        idx[t, :len(k)] = np.array(k) - 1
    wts = np.array(list(gm.terms.values()), dtype=np.float64)
    K = np.zeros(2, dtype=np.int64)
    lz = ctypes.c_double()
    _lib.check(lib.gml_b200_sample_exact_device(0, 14, 3, len(wts), idx.ctypes.data, wts.ctypes.data, 50_000, 2, 11,
                                                K.ctypes.data, ctypes.byref(lz), None, None, 0, None))
    assert K.tolist() == [x.shape[0] for x in a] and lz.value == log_z
    # host buffers (the Julia shim's path) receive the same rows
    rows = int(K.sum()) + 3
    hc, hs = np.zeros(rows), np.zeros((14, rows), dtype=np.int8)
    _lib.check(lib.gml_b200_sample_exact_device(0, 14, 3, len(wts), idx.ctypes.data, wts.ctypes.data, 50_000, 2, 11,
                                                K.ctypes.data, None, hc.ctypes.data, hs.ctypes.data, rows, None))
    k0 = int(K[0])
    assert np.array_equal(hc[:k0], a[0][:, 0]) and np.array_equal(hs[:, :k0], a[0][:, 1:].T)
    assert np.array_equal(hc[k0:k0 + K[1]], a[1][:, 0]) and np.array_equal(hs[:, k0:k0 + K[1]], a[1][:, 1:].T)
    import torch
    small_c = torch.empty(int(K.sum()) - 1, dtype=torch.float64, device="cuda:0")
    small_s = torch.empty((14, int(K.sum()) - 1), dtype=torch.int8, device="cuda:0")
    K2 = np.zeros(2, dtype=np.int64)
    rc = lib.gml_b200_sample_exact_device(0, 14, 3, len(wts), idx.ctypes.data, wts.ctypes.data, 50_000, 2, 11, K2.ctypes.data,
                                          None, small_c.data_ptr(), small_s.data_ptr(), small_c.numel(), None)
    assert rc == _lib.EINVAL and np.array_equal(K, K2)


def test_docs_example_end_to_end():
    """test/runtests.jl:188-196 with the device sampler: learn(sample(gm, 100000), RISE(), B200())."""
    m = MODELS["a"]
    learned = gml_b200.learn(gml_b200.sample(FactorGraph.from_matrix(m), 100_000), RISE(), B200())
    assert np.abs(m - learned).max() <= 0.01


@pytest.mark.parametrize("form", list(FORMS))
def test_learned_model_accuracy_end_to_end(form):
    """test/runtests.jl:105-127 at 10000 samples drawn by the device sampler."""
    for name, m in MODELS.items():
        hist = gml_b200.sample(FactorGraph.from_matrix(m), 10_000, sampler=B200Exact(seed=1))
        learned = gml_b200.learn(hist, FORMS[form](), B200())
        assert np.abs(m - learned).max() <= 0.05, name


def test_device_resident_sample_learns_n24():
    """A random N = 24 model: sampled on the device, attached to a Session without a host copy, learned within 0.05."""
    m = random_ising(24, 124)
    counts, spins = gml_b200.sample_device(FactorGraph.from_matrix(m), 1_000_000, sampler=B200Exact(seed=2))
    assert counts.is_cuda and spins.is_cuda
    sess = Session().attach_device(counts.data_ptr(), spins.data_ptr(), counts.numel(), 24, spins.stride(0))
    assert sess.num_samples == 1_000_000
    learned = sess.solve_pairwise(RISE(), B200())
    assert np.abs(m - learned).max() <= 0.05


def test_refusals():
    gm = pairwise(10, 10)
    with pytest.raises(ValueError):
        gml_b200.sample(FactorGraph(2, 41, "spin", {(1, 2): 0.1}), 10)
    with pytest.raises(ValueError):
        gml_b200.sample(gm, 0)
    with pytest.raises(ValueError):
        gml_b200.sample(FactorGraph(gm.order, gm.varible_count, "boolean", gm.terms), 10)
    for terms in ({(1, 11): 0.1}, {(1, 2): float("inf")}, {(1, 2): float("nan")}, {(2, 2): 0.1}):
        with pytest.raises(gml_b200.GMLB200Error) as e:
            gml_b200.sample(FactorGraph(2, 10, "spin", terms), 10)
        assert e.value.code == _lib.EINVAL, terms
    lib = _lib.load()
    idx = np.array([[0, 1]], dtype=np.int32)
    wts = np.array([0.1])
    K = np.zeros(1, dtype=np.int64)
    for n_spins, n_draws, reps in ((41, 10, 1), (0, 10, 1), (10, 0, 1), (10, 10, 0)):
        rc = lib.gml_b200_sample_exact_device(0, n_spins, 2, 1, idx.ctypes.data, wts.ctypes.data, n_draws, reps, 0,
                                              K.ctypes.data, None, None, None, 0, None)
        assert rc == _lib.EINVAL, (n_spins, n_draws, reps)
