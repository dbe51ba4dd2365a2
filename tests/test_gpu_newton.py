"""The fp64 Newton solver (csrc/newton.cu) against the float64 oracle (oracle/gml_oracle.c) at every accumulator
instantiation, in both launch forms, through the C ABI.

solve_newton picks its kernels from the feature count F and the padded row count Kp = round_up(K, 128):
  * the one-launch form newton_small_kernel<NE> when F <= 32, Kp <= 2048 and GML_B200_NO_FUSED_NEWTON is unset, with
    NE = max(1, ceil((F + F(F+1)/2) / 256)) in {1, 2, 3};
  * otherwise the chunked form, whose f / g / H pass is newton_accum_kernel<NE> with NE the smallest of
    {1, 2, 3, 5, 9, 17, 33} >= ceil((F + F(F+1)/2) / 256), over min(ceil(Kp / 1024), max(1, 1184 / Nn)) chunks of
    whole 128-row tiles (the third cap, 2^24 / (Nn (1 + F + F(F+1)/2)), is above 1184 / Nn for every F <= 128).
Gradient entries sit in slot i = 0 of every thread (F <= 128 < 256); the slots i >= 1 of the larger instantiations hold
only Hessian entries.  A wrong Hessian still converges to the right point, only more slowly, so every case also pins the
number of Newton iterations per node against the oracle's count.

Histograms: spins from a vectorised numpy Gibbs sampler over many chains of random_ising(N, N) (so the L1 optimum has a
real support), integer counts 1..4: K = 127 (one partial tile), 2048 (the fused limit), 2049 (chunked: 3 chunks of 768
rows, the last one 640), 30 000 at N = 63 (Kp = 30 080: 30 chunks wanted, the cap 1184 / 63 = 18 binds; rounded to whole
tiles that is 17 chunks of 1792 rows, the last one 1408), 4096 with one row carrying half
of the weight, 20 000 at N = 127 (the barrier point at F = 128: 9 chunks, the last one partial).
"""
import ctypes
import functools
import math
import re

import numpy as np
import pytest

import c_oracle as c
import gml_b200
from gml_b200 import B200, RISE, RPLE, _lib, logRISE, multiRISE
from gml_oracle import multirise_keys, regularizer_lambda
from helpers import DEFAULT_C, compiled_kernel_names, profiled_kernel_names, random_ising

pytestmark = pytest.mark.gpu
FORMS = {"RISE": RISE, "logRISE": logRISE, "RPLE": RPLE}
FORM_ID = {"RISE": _lib.RISE_ID, "logRISE": _lib.LOGRISE_ID, "RPLE": _lib.RPLE_ID}
ACCUM_NE = (1, 2, 3, 5, 9, 17, 33)
# Bars, measured on one NVIDIA B200 (power limit 1000 W): worst max |dtheta| 3.7e-14 (exact), 1.1e-14 (barrier), 6.1e-16
# (multiRISE); worst objective error 2.7e-14.  The bars leave about two orders of magnitude above that.
THETA_BAR = 5e-12                            # max |dtheta| against the oracle, exact minimiser and barrier point
OBJ_BAR = 2e-12                              # objective, relative (logRISE: the relative error of its sum, |expm1(df)|)
ITER_MARGIN = 1                              # Newton iterations allowed above the oracle's count, per node (measured: +1)
MU = 1e-9


# ------------------------------------------------------------------------------------------------
# which kernels the selection rules give, and which ran
# ------------------------------------------------------------------------------------------------
def n_entries(F):
    return F + F * (F + 1) // 2                   # gradient + lower-triangle Hessian entries


def kp_of(k):
    return -(-k // 128) * 128


def is_fused(F, k, no_fused=False):
    return F <= 32 and kp_of(k) <= 2048 and not no_fused


def expected_kernel(F, k, no_fused=False):
    need = -(-n_entries(F) // 256)
    if is_fused(F, k, no_fused):
        return ("newton_small_kernel", max(1, need))
    return ("newton_accum_kernel", min(ne for ne in ACCUM_NE if ne >= need))


KERNEL_RE = re.compile(r"(newton_accum_kernel|newton_small_kernel)<(\d+)>")
MANGLED_RE = re.compile(r"(newton_accum_kernel|newton_small_kernel)ILi(\d+)EE")


def newton_kernels(names):
    out = set()
    for name in names:
        out |= {(k, int(ne)) for k, ne in KERNEL_RE.findall(name)}
        out |= {(k, int(ne)) for k, ne in MANGLED_RE.findall(name)}
    return out


def profiled(fn):
    """fn()'s result and the Newton f / g / H kernels it launched.  Every solve launches at least one of them, so an empty
    capture is a profiler session that recorded no kernels (seen once, late in a long run): the solve, which is bitwise
    repeatable, is then profiled once more."""
    for _ in range(2):
        out, names = profiled_kernel_names(fn)
        ran = newton_kernels(names)
        if ran:
            break
    return out, ran


def compiled_kernels():
    """the Newton f / g / H instantiations in the in-tree library, or None without cuobjdump"""
    names = compiled_kernel_names(_lib.LIB_PATH)
    return None if names is None else newton_kernels(names)


def use_form(monkeypatch, launch):
    if launch == "chunked":
        monkeypatch.setenv("GML_B200_NO_FUSED_NEWTON", "1")      # read by every solve
    else:
        monkeypatch.delenv("GML_B200_NO_FUSED_NEWTON", raising=False)


# ------------------------------------------------------------------------------------------------
# inputs (seeded)
# ------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def gibbs(n, chains, sweeps=12):
    """[chains x n] +-1 configurations of random_ising(n, n) after `sweeps` systematic Gibbs sweeps of every chain"""
    model = random_ising(n, n)
    J = model - np.diag(np.diag(model))
    h = np.diag(model)
    rng = np.random.default_rng(1000 + n)
    s = rng.choice(np.array([-1.0, 1.0]), size=(chains, n))
    for _ in range(sweeps):
        for i in range(n):
            field = s @ J[:, i] + h[i]
            s[:, i] = np.where(rng.random(chains) < 1.0 / (1.0 + np.exp(-2.0 * field)), 1.0, -1.0)
    return s.astype(np.int8)


HISTS = {"K127": 127, "K2048": 2048, "K2049": 2049, "heavy": 4096, "K20000": 20_000, "K30000": 30_000}


@functools.lru_cache(maxsize=None)
def histogram(n, hist):
    """counts f64[K] and spins int8 [n x K] of a pairwise case"""
    k = HISTS[hist]
    spins = np.ascontiguousarray(gibbs(n, k).T)
    rng = np.random.default_rng([n, k])
    counts = rng.integers(1, 5, size=k).astype(np.float64)
    if hist == "heavy":
        counts[k // 3] = counts.sum() - counts[k // 3]            # one row carries half of M
    return counts, spins


@functools.lru_cache(maxsize=None)
def session(n, hist):
    counts, spins = histogram(n, hist)
    return gml_b200.Session().upload(counts, spins)


def check_nodes(n):
    """the first, second, last two and four (N >= 90: two) seeded random nodes"""
    extra = np.random.default_rng(n).choice(n, 4 if n < 90 else 2, replace=False).tolist()
    return sorted({0, 1, n - 2, n - 1, *extra})


def lam_of(n, hist, form):
    counts, _ = histogram(n, hist)
    return regularizer_lambda(DEFAULT_C[form], n, counts.sum())


@functools.lru_cache(maxsize=None)
def oracle_node(n, hist, form, lam, mode, u):
    """(row u of theta, objective, Newton iterations) of the oracle's solve of node u.  Its count of f / g / H evaluations
    is one per Newton iteration, plus the barrier warm start's evaluation when the barrier phase runs."""
    counts, spins = histogram(n, hist)
    th, info = c.learn_pairwise_packed(counts, spins, form, lam, False, mode, MU, nodes=(u, u + 1), return_info=True)
    return th[u], info["objective"][u], info["n_fgh"] - (mode == "barrier" and lam > 0.0)


def obj_err(f, f_ref, form):
    if form == "logRISE":
        return np.abs(np.expm1(f - f_ref))
    return np.abs(f - f_ref) / np.abs(f_ref)


# ------------------------------------------------------------------------------------------------
# the solver through the C ABI
# ------------------------------------------------------------------------------------------------
def solve(sess, form, lam, method, nb=0, ne=0):
    """gml_b200_solve_pairwise, unsymmetrised, over nodes [nb, ne): (rc, theta [N x N], objective [N], stats)"""
    n = sess.N
    theta, obj, st = np.zeros((n, n), order="F"), np.zeros(n), _lib.Stats()
    opts = method._opts(nb, ne)
    rc = _lib.load().gml_b200_solve_pairwise(sess._h, FORM_ID[form], lam, 0, ctypes.byref(opts),
                                             ctypes.c_void_p(theta.ctypes.data), ctypes.c_void_p(obj.ctypes.data),
                                             ctypes.byref(st))
    return rc, np.ascontiguousarray(theta), obj, st.as_dict()


def solved(sess, form, lam, method, nb=0, ne=0):
    rc, theta, obj, st = solve(sess, form, lam, method, nb, ne)
    _lib.check(rc)
    return theta, obj, st


def check_case(monkeypatch, n, hist, form, launch, mode, solver="auto", lam=None):
    """One pairwise case: the kernels the full solve launched; theta and the objective on the checked nodes against the
    oracle; per checked node, the device's iteration count (a one-node solve) against the oracle's, and a solve capped at
    that bound converges.  Returns (theta, objective, launched kernels) of the full solve."""
    use_form(monkeypatch, launch)
    counts, _ = histogram(n, hist)
    F, k = n + 1, len(counts)
    lam = lam_of(n, hist, form) if lam is None else lam
    method = B200(solver=solver, barrier_mu=MU if mode == "barrier" else 0.0)
    sess = session(n, hist)
    (theta, obj, st), ran = profiled(lambda: solved(sess, form, lam, method))
    assert st["solver_used"] == _lib.SOLVER_NEWTON and st["n_unconverged"] == 0
    assert ran == {expected_kernel(F, k, launch == "chunked")}, ran

    nodes = check_nodes(n)
    refs = [oracle_node(n, hist, form, lam, mode, u) for u in nodes]
    th_ref = np.array([r[0] for r in refs])
    ob_ref = np.array([r[1] for r in refs])
    dth = np.abs(theta[nodes] - th_ref).max()
    dob = obj_err(obj[nodes], ob_ref, form).max()
    worst_ratio, worst_excess, d_one = 0.0, -99, 0.0
    for u, (_, _, n_ref) in zip(nodes, refs):
        one = solved(sess, form, lam, method, u, u + 1)[2]
        assert one["iterations"] <= n_ref + ITER_MARGIN, \
            f"node {u}: {one['iterations']} Newton iterations, the oracle needs {n_ref}"
        worst_ratio = max(worst_ratio, one["iterations"] / n_ref)
        worst_excess = max(worst_excess, one["iterations"] - n_ref)
        capped = B200(solver=solver, barrier_mu=method.barrier_mu, max_iter=n_ref + ITER_MARGIN)
        rc, th_cap, _, _ = solve(sess, form, lam, capped, u, u + 1)
        assert rc == _lib.OK, f"node {u}: not converged within {n_ref + ITER_MARGIN} iterations"
        d_one = max(d_one, np.abs(th_cap[u] - theta[u]).max())
    print(f"NEWTON N={n} {hist} {launch} {mode} {form} {sorted(ran)}: max|dtheta| {dth:.2e}, obj rel {dob:.2e}, "
          f"iterations / oracle <= {worst_ratio:.2f} (excess {worst_excess:+d}), one-node vs full {d_one:.1e}, "
          f"full solve {st['iterations']} iterations, {st['n_stalled']} node(s) stalled at the rounding floor")
    assert d_one <= 1e-11
    assert dth <= THETA_BAR and dob <= OBJ_BAR
    if mode == "barrier":       # the reference's own isapprox
        assert np.linalg.norm(theta[nodes] - th_ref) <= np.sqrt(np.finfo(float).eps) * np.linalg.norm(th_ref)
    return theta, obj, ran


# ------------------------------------------------------------------------------------------------
# the matrix
# ------------------------------------------------------------------------------------------------
FUSED_CASES = [(20, "K127"), (20, "K2048"), (21, "K2048"), (29, "K2048"), (30, "K2048"), (31, "K2048")]
CHUNKED_CASES = [(21, "K2049"), (31, "K2049"), (36, "K2049"), (37, "K2049"), (48, "K2049"), (49, "heavy"), (63, "K30000")]
EXACT_CASES = [(n, h, launch) for n, h in FUSED_CASES for launch in ("fused", "chunked")]
EXACT_CASES += [(n, h, "chunked") for n, h in CHUNKED_CASES]


@pytest.mark.parametrize("form", list(FORMS))
@pytest.mark.parametrize("n,hist,launch", EXACT_CASES)
def test_exact_vs_oracle(monkeypatch, n, hist, launch, form):
    """AUTO, exact L1: N = 20 … 63 on both sides of every accumulator boundary and of the fused limit (F = 32, Kp = 2048)"""
    check_case(monkeypatch, n, hist, form, launch, "exact")


@pytest.mark.parametrize("form", list(FORMS))
@pytest.mark.parametrize("n", [66, 90])
def test_explicit_newton_vs_oracle(monkeypatch, n, form):
    """solver="newton" beyond the AUTO limit: accum<17> (F = 67 and 91) in the exact phase"""
    check_case(monkeypatch, n, "K2049", form, "chunked", "exact", solver="newton")


BARRIER_CASES = [(30, "K2048", "fused"), (30, "K2048", "chunked"), (49, "K2049", "chunked"), (66, "K2049", "chunked"),
                 (90, "K2049", "chunked"), (91, "K2049", "chunked"), (127, "K20000", "chunked")]


@pytest.mark.parametrize("form", list(FORMS))
@pytest.mark.parametrize("n,hist,launch", BARRIER_CASES)
def test_barrier_vs_oracle(monkeypatch, n, hist, launch, form):
    """barrier_mu = 1e-9 (the point Ipopt returns): accum<3>, <9>, <17> at both ends, <33> at F = 92 and F = 128 (the
    direction kernel's 128 x 128 Hessian: 135 KB of dynamic shared memory)"""
    check_case(monkeypatch, n, hist, form, launch, "barrier")


def test_auto_switch_and_feature_limit():
    """AUTO hands 64 features to Newton and 65 to the tensor-core FISTA solver; the barrier point is refused beyond 128"""
    for n, used in ((63, _lib.SOLVER_NEWTON), (64, _lib.SOLVER_FISTA_TC)):
        rc, _, _, st = solve(session(n, "K2049"), "RISE", lam_of(n, "K2049", "RISE"), B200())
        assert rc == _lib.OK and st["solver_used"] == used
    counts, spins = histogram(127, "K20000")
    wide = np.ascontiguousarray(np.concatenate([spins, spins[:1]]))
    with pytest.raises(gml_b200.GMLB200Error) as e:
        gml_b200.learn_packed(counts, wide, RISE(), B200(barrier_mu=MU))
    assert e.value.code == _lib.EINVAL


@pytest.mark.parametrize("form", list(FORMS))
@pytest.mark.parametrize("launch", ["fused", "chunked"])
@pytest.mark.parametrize("mode", ["exact", "barrier"])
@pytest.mark.parametrize("edge", ["no_l1", "all_zero"])
def test_regulariser_edges(monkeypatch, edge, mode, launch, form):
    """lambda = 0 (no penalty: the barrier phase is skipped) and lambda = 5 > max |grad f| (every coupling is exactly zero
    at the exact minimiser: the barrier warm start, direction mode 2, starts from an all-zero point)"""
    lam = 0.0 if edge == "no_l1" else 5.0
    theta, _, _ = check_case(monkeypatch, 30, "K2048", form, launch, mode, lam=lam)
    off = theta[:, :30][~np.eye(30, dtype=bool)]
    if edge == "all_zero" and mode == "exact":
        assert not off.any()
    else:
        assert np.count_nonzero(off) == off.size


# ------------------------------------------------------------------------------------------------
# multiRISE through Newton
# ------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def multibody_histogram(n):
    """the distinct configurations of 20 000 Gibbs chains and their multiplicities"""
    rows, counts = np.unique(gibbs(n, 20_000), axis=0, return_counts=True)
    return counts.astype(np.float64), np.ascontiguousarray(rows.T)


@pytest.mark.parametrize("n,order", [(6, 3), (7, 3), (8, 3), (9, 3), (10, 3), (6, 4), (7, 4)])
def test_multirise_vs_oracle(monkeypatch, n, order):
    """multiRISE (RISE on products of spins) with F = sum_{q < order} C(N, q) = 22, 29, 37, 46, 56 (order 3) and 42, 64
    (order 4) base features: small<2> fused (F = 22, 29), accum<3>, <5>, <9>; checked key by key on every node"""
    monkeypatch.delenv("GML_B200_NO_FUSED_NEWTON", raising=False)
    counts, spins = multibody_histogram(n)
    F = sum(math.comb(n, q) for q in range(order))
    lam = regularizer_lambda(0.4, n, counts.sum())
    sess = gml_b200.Session().upload(counts, spins)
    (vals, info), ran = profiled(lambda: sess.solve_multibody(multiRISE(0.4, False, order), B200(), lam, return_info=True))
    assert info["solver_used"] == _lib.SOLVER_NEWTON
    assert ran == {expected_kernel(F, len(counts))}, ran
    worst = 0.0
    for u in range(n):
        ref = c.learn_multibody_packed(counts, spins, lam, False, order, nodes=(u, u + 1))
        keys = multirise_keys(n, u + 1, order)
        worst = max(worst, max(abs(vals[u, f] - ref[key]) for f, key in enumerate(keys)))
    print(f"NEWTON multiRISE N={n} order {order} F={F} K={len(counts)} {sorted(ran)}: max|dtheta| {worst:.2e}")
    assert worst <= THETA_BAR


# ------------------------------------------------------------------------------------------------
# exact invariants
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("form", list(FORMS))
def test_repeat_node_range_and_launch_forms(monkeypatch, form):
    """A repeated solve is bitwise equal (no floating-point atomics).  A node-range solve (nodes 5..40 of N = 48) returns
    bitwise the rows of the full solve when both use the same chunk count (K = 2049: 3 chunks either way), and agrees to
    1e-12 when they do not (N = 63, K = 30 000: 30 chunks for 36 nodes, 17 for 63).  The fused and the chunked form of
    the same problem agree to 1e-11."""
    use_form(monkeypatch, "chunked")
    for n, hist, bitwise in ((48, "K2049", True), (63, "K30000", False)):
        sess, lam = session(n, hist), lam_of(n, hist, form)
        theta, obj, _ = solved(sess, form, lam, B200())
        again, obj2, _ = solved(sess, form, lam, B200())
        assert np.array_equal(theta, again) and np.array_equal(obj, obj2)
        part, pobj, _ = solved(sess, form, lam, B200(), 5, 41)
        if bitwise:
            assert np.array_equal(part[5:41], theta[5:41]) and np.array_equal(pobj[5:41], obj[5:41])
        else:
            assert np.abs(part[5:41] - theta[5:41]).max() <= 1e-12
    sess, lam = session(30, "K2048"), lam_of(30, "K2048", form)
    for mu in (0.0, MU):
        chunked = solved(sess, form, lam, B200(barrier_mu=mu))[0]
        use_form(monkeypatch, "fused")
        fused = solved(sess, form, lam, B200(barrier_mu=mu))[0]
        assert np.array_equal(fused, solved(sess, form, lam, B200(barrier_mu=mu))[0])
        use_form(monkeypatch, "chunked")
        assert np.abs(fused - chunked).max() <= 1e-11


@pytest.mark.parametrize("launch", ["fused", "chunked"])
@pytest.mark.parametrize("mode", ["exact", "barrier"])
def test_max_iter_exhaustion(monkeypatch, launch, mode):
    """max_iter = 1 leaves the solve unconverged: ENOTCONV (code 3), in both launch forms"""
    use_form(monkeypatch, launch)
    sess, lam = session(30, "K2048"), lam_of(30, "K2048", "RISE")
    rc, _, _, st = solve(sess, "RISE", lam, B200(max_iter=1, barrier_mu=MU if mode == "barrier" else 0.0))
    assert rc == _lib.ENOTCONV and st["n_unconverged"] > 0


def test_every_compiled_newton_kernel_is_launched(monkeypatch):
    """The union of the f / g / H kernels a compact set of solves launches equals the set of newton_accum_kernel /
    newton_small_kernel instantiations compiled into the library: no instantiation is unreachable"""
    plan = [(20, "K2048", "fused"), (21, "K2048", "fused"), (31, "K2048", "fused"), (20, "K2049", "chunked"),
            (21, "K2049", "chunked"), (31, "K2049", "chunked"), (37, "K2049", "chunked"), (49, "K2049", "chunked"),
            (66, "K2049", "chunked"), (91, "K2049", "chunked")]
    launched = set()
    for n, hist, launch in plan:
        use_form(monkeypatch, launch)
        counts, spins = histogram(n, hist)
        _, ran = profiled(lambda: gml_b200.learn_packed(counts, spins, RISE(0.4, False), B200(solver="newton")))
        assert ran == {expected_kernel(n + 1, len(counts), launch == "chunked")}, (n, hist, ran)
        launched |= ran
    assert launched == {("newton_accum_kernel", ne) for ne in ACCUM_NE} | {("newton_small_kernel", ne) for ne in (1, 2, 3)}
    compiled = compiled_kernels()
    if compiled is None:
        pytest.skip("cuobjdump not available: the launched set is not compared with the compiled set")
    assert launched == compiled, f"compiled, never launched: {sorted(compiled - launched)}; launched, not found: {sorted(launched - compiled)}"
