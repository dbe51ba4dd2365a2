"""Parity of the CUDA path (through the C ABI) against the oracle and the reference's golden fixtures.
Tolerances: north_star asks max|dtheta| <= 1e-4 and objectives to 1e-6 relative; the small-problem
solver is held to far tighter bars (it is fp64 Newton)."""
import numpy as np
import pytest

import c_oracle as c
import gml_b200
import gml_oracle as o
from gml_b200 import B200, RISE, RPLE, logRISE, multiRISE
from helpers import DEFAULT_C, MODELS, histogram_c1, three_body_model

pytestmark = pytest.mark.gpu
FORMS = {"RISE": RISE, "logRISE": logRISE, "RPLE": RPLE}


@pytest.mark.parametrize("name", ["a", "b", "c"])
@pytest.mark.parametrize("form", list(FORMS))
def test_goldens_abc(golden, name, form):
    """test/runtests.jl:68-80 -- default formulations, symmetrised; barrier_mu=1e-9 reproduces the stored
    Ipopt output to the reference's own isapprox tolerance."""
    s = golden(f"{name}_samples.csv")
    gold = golden(f"{name}_{form}_learned.csv")
    got, info = gml_b200.learn(s, FORMS[form](), B200(barrier_mu=1e-9), return_info=True)
    assert info["solver_used"] == 1
    assert np.abs(got - gold).max() <= 2e-9
    assert np.linalg.norm(got - gold) <= np.sqrt(np.finfo(float).eps) * np.linalg.norm(gold)
    exact = gml_b200.learn(s, FORMS[form](), B200())
    assert np.abs(exact - gold).max() <= 2e-8
    assert np.abs(exact - c.learn_pairwise(s, form)).max() <= 1e-10


@pytest.mark.parametrize("form", list(FORMS))
def test_goldens_mvt(golden, form):
    """test/runtests.jl:83-101 -- (0.2, false), lambda = 5.4e-5."""
    s = golden("mvt_samples.csv")
    gold = golden(f"mvt_{form}_learned.csv")
    got, info = gml_b200.learn(s, FORMS[form](0.2, False), B200(barrier_mu=1e-9), return_info=True)
    assert np.abs(got - gold).max() <= 1e-4                      # north-star bar vs the real Ipopt output
    ref, rinfo = c.learn_pairwise(s, form, 0.2, False, mode="barrier", mu=1e-9, return_info=True)
    assert np.abs(got - ref).max() <= 1e-8
    exact, einfo = gml_b200.learn(s, FORMS[form](0.2, False), B200(), return_info=True)
    oexact, oinfo = c.learn_pairwise(s, form, 0.2, False, return_info=True)
    assert np.abs(exact - oexact).max() <= 1e-9
    assert np.allclose(einfo["objective"], oinfo["objective"], rtol=1e-9, atol=0)


@pytest.mark.parametrize("form", list(FORMS))
@pytest.mark.parametrize("solver", ["newton", "fista_cc", "fista_tc"])
def test_c1_random_ising(form, solver):
    """BASELINE config C1: N=16 random Ising, 1e5 exact samples."""
    _, hist = histogram_c1()
    ref, rinfo = c.learn_pairwise(hist, form, return_info=True)
    # FISTA: default tol 1e-6 for the CUDA-core backend (fp32 gradient noise floor ~2e-6), 1e-7 for the
    # fixed-point tensor-core backend
    tol = {"newton": 0.0, "fista_cc": 0.0, "fista_tc": 1e-7}[solver]
    got, info = gml_b200.learn(hist, FORMS[form](), B200(solver=solver, tol=tol), return_info=True)
    bar = {"newton": 1e-9, "fista_cc": 5e-5, "fista_tc": 2e-6}[solver]
    assert np.abs(got - ref).max() <= bar
    assert np.allclose(info["objective"], rinfo["objective"], rtol=1e-9 if solver == "newton" else 1e-6, atol=0)


@pytest.mark.parametrize("solver", ["fista_cc", "fista_tc"])
def test_unsymmetrised_and_rows(solver):
    _, hist = histogram_c1(n=12, m_samples=20000, seed=5)
    ref = c.learn_pairwise(hist, "RISE", 0.3, False)
    got = gml_b200.learn(hist, RISE(0.3, False), B200(solver=solver))
    assert np.abs(got - ref).max() <= 5e-5
    assert not np.allclose(got, got.T)


@pytest.mark.parametrize("name", ["a", "b", "c", "mvt"])
def test_multirise_order2_equals_rise(golden, name):
    """test/runtests.jl:132-158."""
    s = golden(f"{name}_samples.csv")
    r = gml_b200.matrix_to_dict(gml_b200.learn(s, RISE(0.2, False), B200(barrier_mu=1e-9)))
    m = gml_b200.learn(s, multiRISE(0.2, False, 2), B200(barrier_mu=1e-9))
    assert m.order == 2 and len(r) == len(m.terms)
    for k, v in r.items():
        assert abs(m[k] - v) <= 1e-7


@pytest.mark.parametrize("sym", [False, True])
def test_multirise_order3_vs_oracle(golden, sym):
    s = golden("c_samples.csv")
    ref = c.learn_multibody(s, 0.2, sym, 3)
    got = gml_b200.learn(s, multiRISE(0.2, sym, 3), B200())
    assert got.terms.keys() == ref.keys()
    assert max(abs(got[k] - ref[k]) for k in ref) <= 1e-9


def test_multirise_order4_recovers_truth():
    """test/runtests.jl:161-172: order-4 relabelled models, 10000 samples, lambda = 0, atol 0.15."""
    rng = np.random.default_rng(0)
    for m in MODELS.values():
        terms = o.matrix_to_terms(m)
        hist = o.sample_exact(terms, m.shape[0], 10000, rng)
        got = gml_b200.learn(hist, multiRISE(0.0, False, min(4, m.shape[0])), B200())
        for k, v in terms.items():
            assert abs(got[k] - v) <= 0.15


def test_multirise_order3_larger_fista():
    """C4-style (reduced): N=10 three-body model, order 3, F=46 base features -> Newton; and the FISTA
    backends agree with it."""
    n = 10
    terms = three_body_model(n, 30)
    hist = o.sample_exact(terms, n, 200_000, np.random.default_rng(31))
    base = gml_b200.learn(hist, multiRISE(0.4, False, 3), B200(solver="newton"))
    for solver in ("fista_cc", "fista_tc"):
        got = gml_b200.learn(hist, multiRISE(0.4, False, 3), B200(solver=solver))
        assert max(abs(got[k] - base[k]) for k in base.terms) <= 5e-5


def test_multirise_c4_reduced_tensor_path():
    """BASELINE config C4 reduced to N=12 (exactly samplable): order 3 -> 79 base features, beyond the Newton
    solver's 64, so the auto solver takes the tensor-core FISTA path; checked against the oracle key by key."""
    n = 12
    terms = three_body_model(n, 30)
    hist = o.sample_exact(terms, n, 200_000, np.random.default_rng(32))
    ref = c.learn_multibody(hist, 0.4, True, 3)
    m = B200()
    got, info = gml_b200.learn(hist, multiRISE(0.4, True, 3), m, return_info=True)
    assert info["solver_used"] == 3
    assert got.terms.keys() == ref.keys()
    assert max(abs(got[k] - ref[k]) for k in ref) <= 1e-5
    # the strongest learned three-body terms are the true ones
    triples = {k: v for k, v in got.terms.items() if len(k) == 3}
    top = sorted(triples, key=lambda k: -abs(triples[k]))[:6]
    assert all(k in terms for k in top)


def test_multilevel_continuation_agrees():
    """Opt-in strided-subsample warm starts must land on the same optimum."""
    _, hist = histogram_c1(n=16, m_samples=400_000, seed=16)
    big = np.repeat(hist.astype(np.float64), 64, axis=0)   # 64 copies of every configuration: K ~ 1e6 rows ...
    big[:, 0] /= 64.0                                      # ... with the counts split, so M, lambda and the optimum are unchanged
    big = big[np.random.default_rng(0).permutation(big.shape[0])]
    a = gml_b200.learn(big, RISE(), B200(solver="fista_tc", multilevel=True))
    b = gml_b200.learn(hist, RISE(), B200(solver="newton"))
    assert np.abs(a - b).max() <= 1e-5


@pytest.mark.parametrize("n_samples,thr", [(1000, 0.15), (10000, 0.05)])
@pytest.mark.parametrize("form", list(FORMS))
def test_learned_model_accuracy(form, n_samples, thr):
    """test/runtests.jl:105-127."""
    rng = np.random.default_rng(0)
    for m in MODELS.values():
        hist = o.sample_exact(o.matrix_to_terms(m), m.shape[0], n_samples, rng)
        learned = gml_b200.learn(hist, FORMS[form]())
        assert np.abs(m - learned).max() <= thr


def test_docs_example():
    """test/runtests.jl:188-196 / README quick start."""
    m = MODELS["a"]
    hist = o.sample_exact(o.matrix_to_terms(m), 3, 100_000, np.random.default_rng(0))
    learned = gml_b200.learn(hist)
    assert np.abs(m - learned).max() <= 0.01


def test_edge_cases(golden):
    s = golden("a_samples.csv")
    # single configuration repeated: K = 1 (degenerate but valid shape) must not crash the pack path
    counts, spins = gml_b200.pack_histogram(s)
    # leading dimension larger than K
    wide = np.ones((3, s.shape[0] + 5), dtype=np.int8)
    wide[:, :s.shape[0]] = spins
    got = gml_b200.learn_packed(counts, wide[:, :s.shape[0]], RISE(), B200())
    assert np.abs(got - gml_b200.learn(s)).max() == 0.0
    # invalid spins / counts are rejected on device with EINVAL
    bad = spins.copy(); bad[1, 2] = 3
    with pytest.raises(gml_b200.GMLB200Error) as e:
        gml_b200.learn_packed(counts, bad, RISE(), B200())
    assert e.value.code == 1
    badc = counts.copy(); badc[0] = 0.0
    with pytest.raises(gml_b200.GMLB200Error) as e:
        gml_b200.learn_packed(badc, spins, RISE(), B200())
    assert e.value.code == 1
    # barrier mode is refused outside the Newton solver
    with pytest.raises(gml_b200.GMLB200Error):
        gml_b200.learn(s, RISE(), B200(solver="fista_cc", barrier_mu=1e-9))
    # max_iter too small -> ENOTCONV, like the reference's @assert LOCALLY_SOLVED
    _, hist = histogram_c1(n=8, m_samples=5000, seed=3)
    with pytest.raises(gml_b200.GMLB200Error) as e:
        gml_b200.learn(hist, RISE(), B200(solver="fista_cc", max_iter=2))
    assert e.value.code == 3
    # the pairwise Session methods refuse multiRISE like learn() refuses a formulation it cannot run
    sess = gml_b200.Session().upload(counts, spins)
    for call in (lambda f: sess.solve_pairwise(f, B200()), lambda f: sess.solve_pairwise_device(f, B200(), 0, 0, 3),
                 lambda f: sess.eval_pairwise(f, np.zeros((3, 4))), lambda f: sess.bench_passes(f),
                 lambda f: sess.solve_path(f, B200(), [0.2])):
        with pytest.raises(NotImplementedError):
            call(multiRISE())


@pytest.mark.parametrize("form", list(FORMS))
@pytest.mark.parametrize("backend", ["fista_cc", "fista_tc"])
def test_contraction_kernels_vs_oracle_gradient(form, backend):
    """Objective and gradient passes (K2/K3) at a dense random point against the float64 restatement of
    src/GraphicalModelLearning.jl:170/279/317 (N=40: 41 features -> one 128-wide feature block, ragged node tile)."""
    n = 40
    rng = np.random.default_rng(3)
    spins = rng.choice(np.array([-1, 1], dtype=np.int8), size=(n, 30_001))       # K not a multiple of 128
    counts = rng.integers(1, 5, size=30_001).astype(np.float64)
    hist = np.concatenate([counts[:, None], spins.T.astype(np.float64)], axis=1)
    w = counts / counts.sum()
    x = rng.normal(size=(n, n + 1)) * 0.1 * (rng.random((n, n + 1)) < 0.3)
    x = np.round(x * 2 ** 24) / 2 ** 24
    x[np.arange(n), np.arange(n)] = 0.0
    sess = gml_b200.Session().upload(counts, np.ascontiguousarray(spins))
    f, g = sess.eval_pairwise(FORMS[form](), x, backend)
    fr = np.zeros(n); gr = np.zeros((n, n + 1))
    for u in range(n):
        stat = o.nodal_stat_pairwise(hist, u)
        xv = x[u, :n].copy(); xv[u] = x[u, n]
        fu, gu, _ = o.smooth_parts(form, xv, stat, w, hess=False)
        fr[u] = fu; gr[u, :n] = gu; gr[u, n] = gu[u]; gr[u, u] = 0.0
    assert np.abs(f - fr).max() <= 2e-6 * max(1.0, np.abs(fr).max())
    assert np.abs(g - gr).max() <= 2e-5 * max(1.0, np.abs(gr).max())
