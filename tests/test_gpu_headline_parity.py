"""Oracle-pinned parity on the SHAPES the headline benchmark runs on (everything through the C ABI):

  * objective / gradient passes of the tensor-core backend with several 128-feature chunks accumulated in TMEM and
    several 64-node tiles (N = 300 / 1000: Fp = 384 / 1024, CTA-pair kernel and the single-CTA streaming kernel;
    N = 1100: Fp = 1152, streaming kernel only), on the coarse AND the fine precision level, all three formulations,
    against the float64 restatement of src/GraphicalModelLearning.jl:170 / 279 / 317 (oracle/gml_oracle.c,
    gml_oracle_eval_pairwise);
  * full fista_tc solves (level switch, parking, active-set compaction) against the oracle's exact L1 minimiser on
    node subsets of an N = 200 problem and of the C2 fixture (N = 100 lattice, 1e6 samples), RISE / logRISE / RPLE;
  * multiRISE order 3 at the C4 shape (N = 30: 436 keys per node, Fp = 512) against the oracle on two nodes;
  * the out-of-range fallback (an optimum beyond the fixed-point range |x| < 7.9), the mean-field warm start, and the
    device samplers against exact enumeration.

Tolerances: north_star asks max |dtheta| <= 1e-4 and objectives to 1e-6 relative; the bars below are tighter.
"""
import ctypes
import functools

import numpy as np
import pytest

import c_oracle as c
import gml_b200
import gml_oracle as o
from gml_b200 import B200, RISE, RPLE, _lib, logRISE, multiRISE
from helpers import (TC_F_REL, random_ising, tc_f_err, tc_grad_bar, tc_level_nr, tc_pass_terms, tc_residual_limbs,
                     three_body_model)

pytestmark = pytest.mark.gpu
FORMS = {"RISE": RISE, "logRISE": logRISE, "RPLE": RPLE}


def rel(a, b, form="RISE"):
    """relative objective error; logRISE's objective is the LOG of a RISE-type sum (src/GraphicalModelLearning.jl:279), so
    its relative error is measured on exp(objective) -- the value itself passes through 0"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    if form == "logRISE":
        a, b = np.exp(a), np.exp(b)
    return float(np.max(np.abs(a - b) / np.abs(b)))


# ------------------------------------------------------------------------------------------------
# (a) objective / gradient passes at headline shapes
# ------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def eval_case(n):
    rng = np.random.default_rng(1000 + n)
    k = 30_001                                                    # ragged: not a multiple of 128 (nor of 256)
    spins = rng.choice(np.array([-1, 1], dtype=np.int8), size=(n, k))
    counts = rng.integers(1, 5, size=k).astype(np.float64)
    nnz = 40.0 / n                                                # ~40 nonzeros per row, |x_u|_1 ~ 2
    x = rng.normal(size=(n, n + 1)) * 0.06 * (rng.random((n, n + 1)) < nnz)
    x = np.clip(np.round(x * 2 ** 13) / 2 ** 13, -0.9, 0.9)       # on the rough lattice (hence also on the coarse and fine ones)
    x[np.arange(n), np.arange(n)] = 0.0
    return counts, spins, x


@functools.lru_cache(maxsize=None)
def eval_oracle(n, form):
    counts, spins, x = eval_case(n)
    return c.eval_pairwise(counts, spins, form, x)


@functools.lru_cache(maxsize=None)
def eval_terms(n):
    counts, spins, x = eval_case(n)
    return tc_pass_terms(counts, spins, x, np.arange(n))


@functools.lru_cache(maxsize=None)
def eval_session(n):
    counts, spins, _ = eval_case(n)
    return gml_b200.Session().upload(counts, np.ascontiguousarray(spins))


@pytest.mark.parametrize("form", list(FORMS))
@pytest.mark.parametrize("level", ["coarse", "fine"])
@pytest.mark.parametrize("n,kernel", [(300, "pair"), (300, "streaming"), (1000, "pair"), (1000, "streaming"), (1100, "streaming")])
def test_passes_at_headline_shapes(monkeypatch, n, kernel, level, form):
    """Objective to TC_F_REL relative and every gradient component within the error model's bar (tests/helpers.py:
    residual rounding on the level's digit grid plus the fp32 error of the exponentials), on all nodes."""
    if kernel == "streaming":
        monkeypatch.setenv("GML_B200_NO_PAIR", "1")               # read when the backend is created (every eval call)
    else:
        monkeypatch.delenv("GML_B200_NO_PAIR", raising=False)
    counts, _, x = eval_case(n)
    fr, gr = eval_oracle(n, form)
    f, g = eval_session(n).eval_pairwise(FORMS[form](), x, "fista_tc", coarse={"rough": "rough", "coarse": True, "fine": False}[level])
    nr = tc_level_nr(level, tc_residual_limbs(counts))
    ferr = tc_f_err(f, fr, form).max()
    ratio = (np.abs(g - gr) / tc_grad_bar(eval_terms(n), form, nr, gr)).max()
    print(f"N={n} {kernel} {level} nr={nr} {form}: f err {ferr:.2e}, worst g err / bar {ratio:.3f}")
    assert ferr <= TC_F_REL
    assert ratio <= 1.0


def test_rough_level_is_refused_for_strongly_weighted_histograms():
    _, _, x = eval_case(300)
    sess = eval_session(300)
    with pytest.raises(gml_b200.GMLB200Error):
        sess.eval_pairwise(RISE(), x, "fista_tc", coarse="rough")
    # bench_passes takes the same levels as eval_pairwise: a refused one is an error, not a timing of the fine level
    with pytest.raises(gml_b200.GMLB200Error):
        sess.bench_passes(RISE(), "fista_tc", reps=1, coarse="rough")
    with pytest.raises(gml_b200.GMLB200Error) as e:
        sess.bench_passes(RISE(), "fista_cc", reps=1, coarse=True)      # the CUDA-core backend has no coarse level
    assert e.value.code == 1
    opts, out = B200(solver="fista_tc")._opts(), np.zeros(4)
    assert _lib.load().gml_b200_bench_passes(sess._h, 7, ctypes.byref(opts), 1, ctypes.c_void_p(out.ctypes.data)) == 1   # unknown formulation id
    ms = sess.bench_passes(RISE(), "fista_tc", reps=1, coarse=True)
    assert len(ms) == 4 and all(np.isfinite(v) and v >= 0.0 for v in ms.values()) and ms["full_pass_wall"] > 0.0


@pytest.mark.parametrize("kernel", ["pair", "streaming"])
def test_rough_level_kernels_vs_oracle(monkeypatch, kernel):
    """The opt-in rough level (2-limb iterate on 2^-14, ONE 8-bit residual plane; needs sqrt(K) wmax <= 2e-3, i.e. >= 250 000
    uniformly weighted rows): exact energies, objective to fp32 accuracy, gradient within the error model's bar for the
    8-bit residual grid."""
    if kernel == "streaming":
        monkeypatch.setenv("GML_B200_NO_PAIR", "1")
    else:
        monkeypatch.delenv("GML_B200_NO_PAIR", raising=False)
    rng = np.random.default_rng(77)
    n, k = 300, 262_145
    spins = rng.choice(np.array([-1, 1], dtype=np.int8), size=(n, k))
    counts = np.ones(k)
    x = rng.normal(size=(n, n + 1)) * 0.06 * (rng.random((n, n + 1)) < 40.0 / n)
    x = np.clip(np.round(x * 2 ** 13) / 2 ** 13, -0.9, 0.9)
    x[np.arange(n), np.arange(n)] = 0.0
    sess = gml_b200.Session().upload(counts, spins)
    bars = tc_pass_terms(counts, spins, x, np.arange(n))
    for form in FORMS:
        fr, gr = c.eval_pairwise(counts, spins, form, x)
        f, g = sess.eval_pairwise(FORMS[form](), x, "fista_tc", coarse="rough")
        ferr = tc_f_err(f, fr, form).max()
        ratio = (np.abs(g - gr) / tc_grad_bar(bars, form, 1, gr)).max()
        print(f"rough {kernel} {form}: f err {ferr:.2e}, worst g err / bar {ratio:.3f}")
        assert ferr <= TC_F_REL and ratio <= 1.0


def test_eval_rejects_points_outside_the_fixed_point_range():
    n = 70
    counts, spins = np.ones(1000), np.random.default_rng(0).choice(np.array([-1, 1], dtype=np.int8), size=(n, 1000))
    sess = gml_b200.Session().upload(counts, spins)
    x = np.zeros((n, n + 1)); x[3, 5] = 8.5
    with pytest.raises(gml_b200.GMLB200Error) as e:
        sess.eval_pairwise(RISE(), x, "fista_tc")
    assert e.value.code == 1
    x[3, 5] = 2.5
    with pytest.raises(gml_b200.GMLB200Error):
        sess.eval_pairwise(RISE(), x, "fista_tc", coarse=True)
    f, _ = sess.eval_pairwise(RISE(), x, "fista_tc")                # fine level holds it
    f2, _ = sess.eval_pairwise(RISE(), x, "fista_cc")
    assert np.allclose(f, f2, rtol=1e-5)


# ------------------------------------------------------------------------------------------------
# (b) full solves against the oracle's exact minimiser
# ------------------------------------------------------------------------------------------------
def sparse_model(n, seed, jlo=0.3, jhi=0.6, hmax=0.2):
    """degree-4 graph (ring + chord of length 7), couplings +-U[jlo, jhi], fields U[-hmax, hmax] on the diagonal"""
    rng = np.random.default_rng(seed)
    m = np.zeros((n, n))
    for i in range(n):
        for j in ((i + 1) % n, (i + 7) % n):
            m[i, j] = m[j, i] = rng.choice([-1.0, 1.0]) * rng.uniform(jlo, jhi)
        m[i, i] = rng.uniform(-hmax, hmax)
    return m


def gibbs_pairwise(model, n_samples, sweeps, seed):
    import torch
    n = model.shape[0]
    row_ptr = np.zeros(n + 1, dtype=np.int32); col, val = [], []
    for i in range(n):
        nz = [j for j in range(n) if j != i and model[i, j] != 0.0]
        row_ptr[i + 1] = row_ptr[i] + len(nz); col += nz; val += [model[i, j] for j in nz]
    col, val = np.array(col, dtype=np.int32), np.array(val, dtype=np.float32)
    field = np.ascontiguousarray(np.diag(model), dtype=np.float32)
    out = torch.empty((n, n_samples), dtype=torch.int8, device="cuda")
    _lib.check(_lib.load().gml_b200_sample_gibbs_device(0, n, row_ptr.ctypes.data, col.ctypes.data, val.ctypes.data, field.ctypes.data,
                                                        n_samples, sweeps, seed, ctypes.c_void_p(out.data_ptr()), n_samples, None))
    torch.cuda.synchronize()
    return out


@pytest.fixture(scope="module")
def n200():
    model = sparse_model(200, 7)
    spins = gibbs_pairwise(model, 50_000, 50, 11).cpu().numpy()
    counts = np.ones(spins.shape[1])
    return model, counts, spins, gml_b200.Session().upload(counts, spins)


@pytest.mark.parametrize("form,creg", [("RISE", 0.4), ("logRISE", 0.8), ("RPLE", 0.2)])
def test_fista_tc_solve_vs_oracle_n200(n200, form, creg):
    """N = 200: Fp = 256 (2 feature chunks), 4 node tiles; default two-level solve with parking and compaction."""
    model, counts, spins, sess = n200
    m = B200(solver="fista_tc", tol=1e-7)
    got, info = sess.solve_pairwise(FORMS[form](creg, False), m, return_info=True)
    assert info["n_unconverged"] == 0 and info["solver_used"] == 3
    lam = info["lambda"]
    worst, worst_obj = 0.0, 0.0
    for b, e in ((0, 1), (63, 65), (199, 200)):                   # first node, a tile boundary, last node
        ref, rinfo = c.learn_pairwise_packed(counts, spins, form, lam, False, nodes=(b, e), return_info=True)
        worst = max(worst, np.abs(got[b:e] - ref[b:e]).max())
        worst_obj = max(worst_obj, rel(info["objective"][b:e], rinfo["objective"][b:e], form))
    print(f"N=200 {form}: max |dtheta| {worst:.2e}, objective rel {worst_obj:.2e}, rounds {info['iterations']}")
    assert worst <= 1e-5 and worst_obj <= 1e-6


@pytest.mark.parametrize("form,creg", [("RISE", 0.4), ("logRISE", 0.8), ("RPLE", 0.2)])
def test_default_settings_solve_vs_oracle_n200(n200, form, creg):
    """The path a plain learn(samples, formulation, B200()) takes at this size: default tol 1e-6, mean-field start,
    retirement on the coarse level (exact prox-gradient mapping <= tol), fine level only for what is left."""
    model, counts, spins, sess = n200
    m = B200()
    got, info = sess.solve_pairwise(FORMS[form](creg, False), m, return_info=True)
    assert info["n_unconverged"] == 0 and info["solver_used"] == 3 and info["max_residual"] <= 1e-6 and info["n_stalled"] == 0
    worst = 0.0
    for b, e in ((0, 1), (63, 65), (199, 200)):
        ref = c.learn_pairwise_packed(counts, spins, form, info["lambda"], False, nodes=(b, e))
        worst = max(worst, np.abs(got[b:e] - ref[b:e]).max())
    print(f"N=200 {form} default settings: max |dtheta| {worst:.2e}, rounds {info['iterations']}, passes {info['n_fg_passes']}")
    assert worst <= 1e-5


@pytest.fixture(scope="module")
def c2():
    from test_gpu_fullsize import lattice_model
    import torch
    truth, row_ptr, col, val = lattice_model()
    n, k = 100, 1_000_000
    spins = torch.empty((n, k), dtype=torch.int8, device="cuda")
    counts = torch.ones(k, dtype=torch.float64, device="cuda")
    _lib.check(_lib.load().gml_b200_sample_gibbs_device(0, n, row_ptr.ctypes.data, col.ctypes.data, val.ctypes.data, None,
                                                        k, 60, 100, ctypes.c_void_p(spins.data_ptr()), k, None))
    torch.cuda.synchronize()
    sess = gml_b200.Session(0).attach_device(counts.data_ptr(), spins.data_ptr(), k, n, k)
    return sess, spins.cpu().numpy(), spins


@pytest.mark.parametrize("form,creg,nodes", [("RISE", 0.4, (0, 55)), ("logRISE", 0.8, (37,)), ("RPLE", 0.2, (99,))])
def test_c2_fixture_nodes_vs_oracle(c2, form, creg, nodes):
    """BASELINE config C2 (N = 100 lattice spin glass, 1e6 samples) on a node subset, all three formulations."""
    sess, host_spins, _ = c2
    counts = np.ones(host_spins.shape[1])
    got, info = sess.solve_pairwise(FORMS[form](creg, False), B200(tol=1e-7), return_info=True)
    assert info["n_unconverged"] == 0 and info["solver_used"] == 3
    worst, worst_obj = 0.0, 0.0
    for u in nodes:
        ref, rinfo = c.learn_pairwise_packed(counts, host_spins, form, info["lambda"], False, nodes=(u, u + 1), return_info=True)
        worst = max(worst, np.abs(got[u] - ref[u]).max())
        worst_obj = max(worst_obj, rel(info["objective"][u], rinfo["objective"][u], form))
    print(f"C2 {form}: max |dtheta| {worst:.2e}, objective rel {worst_obj:.2e}, rounds {info['iterations']}")
    assert worst <= 1e-5 and worst_obj <= 1e-6


def test_warm_start_changes_the_path_not_the_answer(c2):
    sess, _, _ = c2
    cold = B200(tol=1e-7, warm_start=False)
    warm = B200(tol=1e-7, warm_start=True)
    a = sess.solve_pairwise(RISE(0.4, False), cold)
    b = sess.solve_pairwise(RISE(0.4, False), warm)
    print("rounds cold", cold.last_stats["iterations"], "warm", warm.last_stats["iterations"])
    assert np.abs(a - b).max() <= 2e-6


# ------------------------------------------------------------------------------------------------
# (c) multiRISE order 3 at the C4 shape
# ------------------------------------------------------------------------------------------------
def test_multirise_c4_shape_vs_oracle():
    """BASELINE config C4 at reduced sample count: N = 30, ring of pair couplings +-0.3 plus 30 random triples +-0.4,
    6e4 Gibbs samples from the device term sampler; order 3 -> 436 keys per node, 466 base features (Fp = 512) through
    the tensor-core FISTA path; two node problems against the oracle (src/GraphicalModelLearning.jl:83-133)."""
    n, k = 30, 60_000
    terms = three_body_model(n, 30)
    spins = gml_b200.sample_terms_device(terms, n, k, sweeps=80, seed=30).cpu().numpy()
    counts = np.ones(k)
    lam = gml_b200.regularizer_lambda(0.4, n, float(k))
    m = B200(tol=1e-7)
    got, info = gml_b200.learn_packed(counts, spins, multiRISE(0.4, False, 3), m, return_info=True)
    assert info["solver_used"] == 3 and info["n_unconverged"] == 0
    worst = 0.0
    for u in (0, 29):
        ref = c.learn_multibody_packed(counts, spins, lam, False, 3, nodes=(u, u + 1))
        assert len(ref) == 436
        worst = max(worst, max(abs(got[key] - v) for key, v in ref.items()))
    print(f"C4 shape: max |dtheta| over 2 x 436 keys {worst:.2e}, rounds {info['iterations']}")
    assert worst <= 1e-5
    # the generating three-body terms are recovered (statistical, 1e5 samples)
    sym = gml_b200.learn_packed(counts, spins, multiRISE(0.4, True, 3), B200())
    for key, v in terms.items():
        assert abs(sym[key] - v) <= 0.06


# ------------------------------------------------------------------------------------------------
# (d) optimum beyond the fixed-point range of the tensor-core backend
# ------------------------------------------------------------------------------------------------
def test_out_of_range_node_is_resolved_not_clamped():
    """Two perfectly correlated spins and M = 1e9 samples: the RISE coupling is ~ log(1/lambda) ~ 9 > 7.9.  The
    fixed-point backend must not return the clamp: the node is re-solved by the CUDA-core backend."""
    rng = np.random.default_rng(2)
    n, k = 70, 4096
    spins = rng.choice(np.array([-1, 1], dtype=np.int8), size=(n, k))
    spins[1] = spins[0]
    counts = np.full(k, 1e9 / k)
    lam = gml_b200.regularizer_lambda(0.4, n, counts.sum())
    m = B200(solver="fista_tc", tol=1e-6, max_iter=20000)
    try:
        got = gml_b200.learn_packed(counts, spins, RISE(0.4, False), m, lam=lam)
    except gml_b200.GMLB200Error as err:          # loud failure is acceptable, a silently clamped answer is not
        assert err.code == 3
        return
    ref = c.learn_pairwise_packed(counts, spins, "RISE", lam, False, nodes=(0, 2))
    assert abs(ref[0, 1]) > 7.9
    assert np.abs(got[:2] - ref[:2]).max() <= 1e-3 * abs(ref[0, 1])


# ------------------------------------------------------------------------------------------------
# (e) device samplers against the exact distribution
# ------------------------------------------------------------------------------------------------
def test_device_samplers_match_exact_enumeration():
    """Pair correlations and magnetisations of the device Gibbs samplers (pairwise kernel and term-list kernel) at
    N = 16 against exact enumeration of the 2^16 weights (the reference's own sampler, src/sampling.jl:26-47), 5 sigma."""
    n, m_samples = 16, 2_000_000
    model = random_ising(n, 16)
    terms = o.matrix_to_terms(model)
    conf = ((np.arange(2 ** n)[:, None] >> np.arange(n)) & 1) * 2.0 - 1.0
    logw = 0.5 * np.einsum("ki,ij,kj->k", conf, model - np.diag(np.diag(model)), conf) + conf @ np.diag(model)
    p = np.exp(logw - logw.max()); p /= p.sum()
    exact_c = (conf * p[:, None]).T @ conf
    exact_m = p @ conf
    for name, sampler in (("pairwise", lambda: gibbs_pairwise(model, m_samples, 200, 3)),
                          ("terms", lambda: gml_b200.sample_terms_device(terms, n, m_samples, sweeps=200, seed=3))):
        s = sampler().float()
        corr = (s @ s.T / m_samples).cpu().numpy()
        mag = s.mean(dim=1).cpu().numpy()
        sig_c = np.sqrt(np.maximum(1.0 - exact_c ** 2, 1e-3) / m_samples)
        sig_m = np.sqrt(np.maximum(1.0 - exact_m ** 2, 1e-3) / m_samples)
        zc = np.abs(corr - exact_c) / sig_c
        zm = np.abs(mag - exact_m) / sig_m
        print(f"{name}: max z corr {zc.max():.2f}, max z mag {zm.max():.2f}")
        assert zc.max() <= 5.0 and zm.max() <= 5.0


def test_device_multirise_symmetrisation_and_threshold(golden):
    """SURVEY 8f-3: the mean over the per-node estimates of every sorted key (src/GraphicalModelLearning.jl:135-149) computed on
    the device equals the host Dict grouping of the same solve; thresholding zeroes small off-diagonal entries."""
    s = golden("c_samples.csv")
    counts, spins = gml_b200.pack_histogram(s)
    sess = gml_b200.Session().upload(counts, spins)
    for order in (2, 3, 4):
        host = gml_b200.learn(s, multiRISE(0.2, True, order), B200())
        dev = sess.solve_multibody_sym(multiRISE(0.2, True, order), B200())
        assert dev.terms.keys() == host.terms.keys()
        assert max(abs(dev[k] - host[k]) for k in host.terms) <= 1e-12
    n = 30
    terms = three_body_model(n, 30)
    sp = gml_b200.sample_terms_device(terms, n, 50_000, sweeps=60, seed=1).cpu().numpy()
    cn = np.ones(sp.shape[1])
    s2 = gml_b200.Session().upload(cn, sp)
    host = gml_b200.learn_packed(cn, sp, multiRISE(0.4, True, 3), B200(tol=1e-7))
    dev = s2.solve_multibody_sym(multiRISE(0.4, True, 3), B200(tol=1e-7))
    assert len(dev.terms) == 30 + 435 + 4060 and dev.terms.keys() == host.terms.keys()
    assert max(abs(dev[k] - host[k]) for k in host.terms) <= 1e-12
    theta = gml_b200.learn(s, RISE(), B200())
    cut, nnz = sess.threshold(theta, 0.15)
    expect = np.where((np.abs(theta) < 0.15) & ~np.eye(4, dtype=bool), 0.0, theta)
    assert np.array_equal(cut, expect) and nnz == int(np.count_nonzero(expect - np.diag(np.diag(expect))))


# ------------------------------------------------------------------------------------------------
# (f) second-order finishes beyond 64 features: barrier point up to 128 features, support polish for any size
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def n100():
    from test_gpu_fullsize import lattice_model
    truth, _, _, _ = lattice_model()
    spins = gibbs_pairwise(truth, 10_000, 60, 100).cpu().numpy()
    return np.ones(spins.shape[1]), spins


def test_barrier_point_n100_passes_the_reference_isapprox(n100):
    """B200(barrier_mu=1e-9) at N = 100 (101 features per node: the fp64 Newton solver with the dense 101 x 101 Hessian)
    against the oracle's barrier point -- the criterion of the reference's own known-answer tests
    (test/runtests.jl:77,89,95,101: isapprox, relative Frobenius <= sqrt(eps))."""
    counts, spins = n100
    lam = gml_b200.regularizer_lambda(0.4, 100, counts.sum())
    got, info = gml_b200.learn_packed(counts, spins, RISE(0.4, False), B200(barrier_mu=1e-9), lam=lam, return_info=True)
    assert info["solver_used"] == 1
    ref = c.learn_pairwise_packed(counts, spins, "RISE", lam, False, mode="barrier", mu=1e-9)
    assert np.linalg.norm(got - ref) <= np.sqrt(np.finfo(float).eps) * np.linalg.norm(ref)
    assert np.abs(got - ref).max() <= 1e-8
    for form, creg in (("logRISE", 0.8), ("RPLE", 0.2)):
        lam = gml_b200.regularizer_lambda(creg, 100, counts.sum())
        got = gml_b200.learn_packed(counts, spins, FORMS[form](creg, False), B200(barrier_mu=1e-9), lam=lam)
        ref = c.learn_pairwise_packed(counts, spins, form, lam, False, mode="barrier", mu=1e-9, nodes=(40, 48))
        assert np.linalg.norm(got[40:48] - ref[40:48]) <= np.sqrt(np.finfo(float).eps) * np.linalg.norm(ref[40:48])
    with pytest.raises(gml_b200.GMLB200Error):                     # beyond 128 features the barrier point is refused, loudly
        gml_b200.learn_packed(np.ones(500), np.ones((130, 500), dtype=np.int8), RISE(), B200(barrier_mu=1e-9))


@pytest.mark.parametrize("form,creg", [("RISE", 0.4), ("logRISE", 0.8), ("RPLE", 0.2)])
def test_support_polish_reaches_the_exact_minimiser(n200, form, creg):
    """FISTA to 1e-5, then fp64 Newton on each node's identified support (csrc/polish.cu): the oracle's exact L1 minimiser
    to 1e-9 at N = 200 (201 features per node, supports of a few dozen)."""
    _, counts, spins, sess = n200
    m = B200(solver="fista_tc", tol=1e-5, polish=True)
    got, info = sess.solve_pairwise(FORMS[form](creg, False), m, return_info=True)
    assert info["n_unconverged"] == 0
    worst, worst_obj = 0.0, 0.0
    for b, e in ((0, 2), (64, 65), (198, 200)):
        ref, rinfo = c.learn_pairwise_packed(counts, spins, form, info["lambda"], False, nodes=(b, e), return_info=True)
        worst = max(worst, np.abs(got[b:e] - ref[b:e]).max())
        worst_obj = max(worst_obj, rel(info["objective"][b:e], rinfo["objective"][b:e], form))
    print(f"polish N=200 {form}: max |dtheta| {worst:.2e}, objective rel {worst_obj:.2e}")
    assert worst <= 1e-9 and worst_obj <= 1e-11
