"""Every objective / gradient pass variant of the tensor-core backend (csrc/eval_tc.cu) against the float64 oracle
(oracle/gml_oracle.c, gml_oracle_eval_pairwise), through the C ABI, with bars from the error model in tests/helpers.py.

BackendTC picks its kernels from the histogram and the problem size:
  * residual digit planes: the fine level has nR = 3 when sqrt(K) w_max <= 2e-3, else 4; the coarse level nr =
    max(2, nR - 1), the rough level nr = 1 (and is refused unless nR = 3);
  * tc_energy_pair_kernel when Fp <= 1024, there are >= 2 sample blocks and GML_B200_NO_PAIR is unset, else
    tc_energy_kernel; objective-only passes (want_grad = False) run the GRAD = false instantiation of their level;
  * tc_grad_kernel<nr, FT> with FT = 256 when nr <= 2 and Fp % 256 == 0, else 128.
Each case runs under torch.profiler and asserts that the instantiations it expects from these rules launched, so a
change of the selection fails here instead of silently testing another kernel.

Histograms:
  U  uniform counts, K = 262 145 (nR = 3, the precision the C3 headline runs at; 2049 sample blocks, so the pair
     kernel gets a half-empty last pair), the leading rows of one N = 1100 spin array as the N = 1100 / 1000 / 200 /
     128 / 127 / 65 problems (Fp = 1152 / 1024 / 256 / 256 / 128 / 128): streaming-only Fp, the C3 shape, FT = 256 and
     128, a second feature chunk with one real feature, no padding column, a one-node trailing energy tile;
  W  weighted counts 1..4 at N = 200 with K = 1, 127, 128 (one sample block: the streaming kernel even where the pair
     kernel is eligible), 129 and 257 (a half-filled pair block), and K = 30 001 with one row carrying half of M
     (w_max = 0.5); nR = 4.
"""
import ctypes
import functools
import re

import numpy as np
import pytest

import c_oracle as c
import gml_b200
from gml_b200 import B200, RISE, RPLE, _lib, logRISE
from helpers import (TC_F_REL, compiled_kernel_names, profiled_kernel_names, random_spins, tc_f_err, tc_grad_bar, tc_level_nr,
                     tc_pass_terms, tc_residual_limbs)

pytestmark = pytest.mark.gpu
FORMS = {"RISE": RISE, "logRISE": logRISE, "RPLE": RPLE}
LEVEL_ARG = {"rough": "rough", "coarse": True, "fine": False}        # Session.eval_pairwise(coarse=...)
LEVEL_ID = {"fine": 0, "coarse": 1, "rough": 2}                      # opts.reserved[5]
LATTICE = {"rough": 2.0 ** -14, "coarse": 2.0 ** -22, "fine": 2.0 ** -24}
X_RANGE = {"rough": 1.95, "coarse": 1.95, "fine": 7.9}
XL = {"rough": 2, "coarse": 3, "fine": 4}                            # iterate limbs
U_K = 262_145
W_HISTS = ("W1", "W127", "W128", "W129", "W257", "Wheavy")


def fp_of(n):
    return -(-(n + 1) // 128) * 128


# ------------------------------------------------------------------------------------------------
# inputs (seeded) and the oracle, cached per (histogram, N, form)
# ------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def histogram(name):
    """counts and the full spin array of a histogram (problems use its leading rows)"""
    if name == "U":
        return np.ones(U_K), random_spins(1100, U_K, np.random.default_rng(1100))
    if name == "Wheavy":
        k = 30_001
        counts = np.ones(k)
        counts[k // 2] = k - 1                                   # half of M on one row: w_max = 0.5
        return counts, random_spins(200, k, np.random.default_rng(30_001))
    k = int(name[1:])
    rng = np.random.default_rng(k)
    return rng.integers(1, 5, size=k).astype(np.float64), random_spins(200, k, rng)


@functools.lru_cache(maxsize=None)
def point(hist, n):
    """about 40 nonzeros per row on the rough lattice 2^-14 (hence on every level's), |x| <= 0.9, zero self entries"""
    rng = np.random.default_rng([n, sum(map(ord, hist))])
    x = rng.normal(size=(n, n + 1)) * 0.06 * (rng.random((n, n + 1)) < min(1.0, 40.0 / n))
    x = np.clip(np.round(x * 2 ** 14) / 2 ** 14, -0.9, 0.9)
    x[np.arange(n), np.arange(n)] = 0.0
    return x


@functools.lru_cache(maxsize=None)
def check_nodes(n):
    """tile and chunk edges (0, 1, 63, 64, 127, 128, N-2, N-1) and four seeded random nodes"""
    extra = np.random.default_rng(n).choice(n, 4, replace=False).tolist()
    return np.array(sorted({u for u in [0, 1, 63, 64, 127, 128, n - 2, n - 1] + extra if 0 <= u < n}), dtype=np.int32)


@functools.lru_cache(maxsize=None)
def oracle(hist, n, form):
    counts, spins = histogram(hist)
    nodes = check_nodes(n)
    return c.eval_pairwise(counts, spins[:n], form, point(hist, n)[nodes], nodes)


@functools.lru_cache(maxsize=None)
def terms(hist, n):
    counts, spins = histogram(hist)
    nodes = check_nodes(n)
    return tc_pass_terms(counts, spins[:n], point(hist, n)[nodes], nodes)


@functools.lru_cache(maxsize=None)
def session(hist, n):
    counts, spins = histogram(hist)
    return gml_b200.Session().upload(counts, spins[:n])         # a row-slice view: ld = K of the full array


# ------------------------------------------------------------------------------------------------
# which kernels ran
# ------------------------------------------------------------------------------------------------
KERNEL_RE = re.compile(r"(tc_energy_pair_kernel|tc_energy_kernel|tc_grad_kernel)<([^>]*)>")
MANGLED_RE = re.compile(r"(tc_energy_pair_kernel|tc_energy_kernel|tc_grad_kernel)I((?:L[a-z]\d+E)+)E")


def tc_kernels(names):
    """{(kernel, template arguments as ints)} of the tensor-core pass kernels among demangled or mangled names"""
    out = set()
    for name in names:
        for k, args in KERNEL_RE.findall(name):
            vals = (re.sub(r"\(\w+\)", "", a).strip() for a in args.split(","))
            out.add((k, tuple(int({"true": "1", "false": "0"}.get(v, v)) for v in vals)))
        for k, args in MANGLED_RE.findall(name):
            out.add((k, tuple(int(v) for v in re.findall(r"L[a-z](\d+)E", args))))
    return out


def profiled(fn):
    """fn()'s result and the tensor-core kernels it launched"""
    out, names = profiled_kernel_names(fn)
    return out, tc_kernels(names)


def expected_kernels(counts, n, level, form, want_grad, pair_allowed):
    """the instantiations the selection rules of BackendTC give for one pass"""
    nr = tc_level_nr(level, tc_residual_limbs(counts))
    fp, blocks = fp_of(n), -(-len(counts) // 128)
    pair = pair_allowed and fp <= 1024 and blocks >= 2
    kform = 2 if form == "RPLE" else 0                           # logRISE runs the RISE kernels
    e_nr = nr if want_grad else (1 if XL[level] == 2 else 2)     # one objective-only kernel per iterate width
    out = {("tc_energy_pair_kernel" if pair else "tc_energy_kernel", (kform, int(want_grad), XL[level], e_nr))}
    if want_grad:
        out.add(("tc_grad_kernel", (nr, 256 if nr <= 2 and fp % 256 == 0 else 128)))
    return out


def use_kernel(monkeypatch, kernel):
    if kernel == "streaming":
        monkeypatch.setenv("GML_B200_NO_PAIR", "1")              # read when the backend is created (every eval call)
    else:
        monkeypatch.delenv("GML_B200_NO_PAIR", raising=False)


def compiled_kernels():
    """the tensor-core pass instantiations in the in-tree library, or None without cuobjdump"""
    names = compiled_kernel_names(_lib.LIB_PATH)
    return None if names is None else tc_kernels(names)


# ------------------------------------------------------------------------------------------------
# the matrix
# ------------------------------------------------------------------------------------------------
CASES = [("U", n, kernel) for n in (1100, 1000, 200, 128, 127, 65) for kernel in ("pair", "streaming") if kernel == "streaming" or fp_of(n) <= 1024]
CASES += [(h, 200, kernel) for h in W_HISTS for kernel in ("pair", "streaming")]


@pytest.mark.parametrize("form", list(FORMS))
@pytest.mark.parametrize("level", ["rough", "coarse", "fine"])
@pytest.mark.parametrize("hist,n,kernel", CASES)
def test_pass_vs_oracle(monkeypatch, hist, n, kernel, level, form):
    """One pass against the oracle on the checked nodes (objective to TC_F_REL, gradient to the error model's bar), and
    on all nodes the exact invariants: a repeated eval, and the pair kernel against the streaming kernel, give bitwise
    equal gradients (the same residual bytes, summed exactly in int64); the objective-only pass gives the same objective
    up to the order of the fp64 atomics.  (logRISE runs the RISE kernels and divides their gradient by the objective sum,
    whose fp64 atomics and fp32 partial sums are not ordered: its gradients are compared bitwise as RISE's.)"""
    use_kernel(monkeypatch, kernel)
    counts, _ = histogram(hist)
    sess, x, ev = session(hist, n), point(hist, n), FORMS[form]()
    if level == "rough" and tc_residual_limbs(counts) == 4:
        with pytest.raises(gml_b200.GMLB200Error) as e:
            sess.eval_pairwise(ev, x, "fista_tc", coarse="rough")
        assert e.value.code == _lib.EINVAL
        return
    (f, g), ran = profiled(lambda: sess.eval_pairwise(ev, x, "fista_tc", coarse=LEVEL_ARG[level]))
    assert ran == expected_kernels(counts, n, level, form, True, kernel == "pair")
    (f0, g0), ran0 = profiled(lambda: sess.eval_pairwise(ev, x, "fista_tc", want_grad=False, coarse=LEVEL_ARG[level]))
    assert g0 is None and ran0 == expected_kernels(counts, n, level, form, False, kernel == "pair")

    # exact invariants, all nodes
    f_obj_err = tc_f_err(f0, f, form).max()
    assert f_obj_err <= 1e-12, f"objective-only pass differs from the full pass by {f_obj_err:.2e}"
    if form != "logRISE":
        assert np.array_equal(sess.eval_pairwise(ev, x, "fista_tc", coarse=LEVEL_ARG[level])[1], g)
        if kernel == "pair":
            use_kernel(monkeypatch, "streaming")
            assert np.array_equal(sess.eval_pairwise(ev, x, "fista_tc", coarse=LEVEL_ARG[level])[1], g)

    # against the oracle, checked nodes
    nodes = check_nodes(n)
    fr, gr = oracle(hist, n, form)
    nr = tc_level_nr(level, tc_residual_limbs(counts))
    ferr = tc_f_err(f[nodes], fr, form).max()
    ratio = (np.abs(g[nodes] - gr) / tc_grad_bar(terms(hist, n), form, nr, gr)).max()
    print(f"TCPASS {hist} N={n} {kernel} {level} nr={nr} {form}: f err {ferr:.2e}, worst g err / bar {ratio:.3f}")
    assert ferr <= TC_F_REL
    assert ratio <= 1.0


@pytest.mark.parametrize("level", ["rough", "coarse", "fine"])
@pytest.mark.parametrize("begin", [37, 64])
def test_node_range_eval_returns_the_rows_of_the_full_eval(monkeypatch, level, begin):
    """gml_b200_eval_pairwise over opts.node_begin..N returns bitwise the gradient rows of the full eval.  begin = 37 puts
    the shard's first spin row off a 16-byte boundary, which selects the scalar spin loads of the energy epilogue;
    begin = 64 keeps the vector loads (U, N = 1000, pair kernel)."""
    monkeypatch.delenv("GML_B200_NO_PAIR", raising=False)
    n = 1000
    sess, x = session("U", n), point("U", n)
    _, g = sess.eval_pairwise(RISE(), x, "fista_tc", coarse=LEVEL_ARG[level])
    opts = B200(solver="fista_tc")._opts(begin, n)
    opts.reserved[5] = LEVEL_ID[level]
    xs = np.ascontiguousarray(x[begin:])
    fs, gs = np.zeros(n - begin), np.zeros_like(xs)
    _lib.check(_lib.load().gml_b200_eval_pairwise(sess._h, _lib.RISE_ID, ctypes.byref(opts), ctypes.c_void_p(xs.ctypes.data),
                                                  ctypes.c_void_p(fs.ctypes.data), ctypes.c_void_p(gs.ctypes.data)))
    assert np.array_equal(gs, g[begin:])


def test_every_compiled_pass_kernel_is_launched(monkeypatch):
    """The union of the kernels a compact set of passes launches (U at N = 200 and 65, W257; every level, both kernels,
    RISE and RPLE, with and without gradient) equals the set of tc_energy_kernel / tc_energy_pair_kernel / tc_grad_kernel
    instantiations compiled into the library: no instantiation is unreachable."""
    plan = [("U", 200, kernel, level, form, grad) for kernel in ("pair", "streaming") for level in ("rough", "coarse", "fine")
            for form in ("RISE", "RPLE") for grad in (True, False)]
    plan += [("U", 65, "pair", level, "RISE", True) for level in ("rough", "coarse")]           # FT = 128 at nr <= 2
    plan += [("W257", 200, kernel, level, form, grad) for kernel in ("pair", "streaming") for level in ("coarse", "fine")
             for form in ("RISE", "RPLE") for grad in (True, False)]
    launched = set()
    for hist, n, kernel, level, form, grad in plan:
        use_kernel(monkeypatch, kernel)
        sess, x = session(hist, n), point(hist, n)
        _, ran = profiled(lambda: sess.eval_pairwise(FORMS[form](), x, "fista_tc", want_grad=grad, coarse=LEVEL_ARG[level]))
        assert ran == expected_kernels(histogram(hist)[0], n, level, form, grad, kernel == "pair")
        launched |= ran
    compiled = compiled_kernels()
    if compiled is None:
        pytest.skip("cuobjdump not available: the launched set is not compared with the compiled set")
    assert launched == compiled, f"compiled, never launched: {sorted(compiled - launched)}; launched, not found: {sorted(launched - compiled)}"


# ------------------------------------------------------------------------------------------------
# iterate limbs at their digit boundaries
# ------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def limb_histogram():
    """N = 300, K = 4097 uniform (nR = 4); spin rows 150 + i repeat rows i, so +a on feature i and -a on 150 + i cancel
    in every energy: |x_u|_1 can sit near the coarse level's limit while the energies stay small"""
    top = random_spins(150, 4097, np.random.default_rng(4097))
    return np.ones(4097), np.concatenate([top, top])


@functools.lru_cache(maxsize=None)
def limb_point(level):
    lat, n = LATTICE[level], 300
    vals = [s * k * lat for k in (127, 128, 129, 256 * 128, 2 ** 23 - 1) for s in (1, -1) if k * lat <= X_RANGE[level]]
    rng = np.random.default_rng(300)
    x = np.zeros((n, n + 1))
    for u in range(1, 9):                 # every boundary value on three features of nodes 1..8
        f = rng.choice(np.delete(np.arange(n + 1), u), 3 * len(vals), replace=False)
        x[u, f] = np.tile(vals, 3)
    a = np.round(1.65 * 2 ** 14) / 2 ** 14
    d = np.round(rng.uniform(0.0, 0.02, 149) * 2 ** 14) / 2 ** 14
    x[0, 1:150] = a                       # node 0: |x_0|_1 ~ 492, just below the 3-limb guard |x_u|_1 < 500
    x[0, 151:300] = -(a - d)
    x[0, 300] = 0.25
    return x


@pytest.mark.parametrize("form", list(FORMS))
@pytest.mark.parametrize("level", ["coarse", "fine"])
def test_limb_boundaries_vs_oracle(monkeypatch, level, form):
    """Iterate entries at balanced base-256 digit boundaries, k * lattice for k = +-127, +-128, +-129, +-256*128 and
    +-(2^23 - 1) where the level's range allows, and one node with |x_u|_1 just below the 3-limb guard (500).  An error in
    any limb above the lowest shifts the coefficient x_j the kernel uses by >= 256 lattice units (>= 1.5e-5 on the fine
    level).  The gradient check catches it: component j moves by about that shift times S = sum_k w_k psi_k (the
    Hessian's diagonal), against a bar near 1e-8.  The objective moves only by the shift times g_j, which for a feature
    uncorrelated with the data is ~f / sqrt(K) and can stay below TC_F_REL.  An error in the lowest limb is a few lattice
    units, at or below the fp32 resolution of the energy once |t| >= 1; this test does not claim to see it.  (Node 0's
    RISE residual grid is set by e^{min(B, 80)}: its RISE gradient check is vacuous; its RPLE gradient is not.)"""
    monkeypatch.delenv("GML_B200_NO_PAIR", raising=False)
    counts, spins = limb_histogram()
    x = limb_point(level)
    nodes = np.arange(9, dtype=np.int32)
    assert 490.0 < np.abs(x[0]).sum() < 500.0
    sess = gml_b200.Session().upload(counts, spins)
    (f, g), ran = profiled(lambda: sess.eval_pairwise(FORMS[form](), x, "fista_tc", coarse=LEVEL_ARG[level]))
    assert ran == expected_kernels(counts, 300, level, form, True, True)
    if form != "logRISE":
        use_kernel(monkeypatch, "streaming")
        assert np.array_equal(sess.eval_pairwise(FORMS[form](), x, "fista_tc", coarse=LEVEL_ARG[level])[1], g)
    fr, gr = c.eval_pairwise(counts, spins, form, x[nodes], nodes)
    nr = tc_level_nr(level, tc_residual_limbs(counts))
    ferr = tc_f_err(f[nodes], fr, form)
    ratio = np.abs(g[nodes] - gr) / tc_grad_bar(tc_pass_terms(counts, spins, x[nodes], nodes), form, nr, gr)
    print(f"TCPASS limbs {level} nr={nr} {form}: f err {ferr.max():.2e}, worst g err / bar {ratio.max():.3f}")
    assert ferr.max() <= TC_F_REL
    assert ratio.max() <= 1.0
