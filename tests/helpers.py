"""Seeded synthetic inputs shared by the tests (BASELINE.json configs, reduced where noted)."""
import re
import shutil
import subprocess

import numpy as np

import gml_oracle as o

# test/common.jl:15-32
MODEL_A = np.array([[0.0, 0.1, 0.2], [0.1, 0.0, 0.3], [0.2, 0.3, 0.0]])
MODEL_B = np.array([[0.3, 0.1, 0.2], [0.1, 0.2, 0.3], [0.2, 0.3, 0.1]])
MODEL_C = np.array([[0.0, 0.1, 0.2, 0.3], [0.1, 0.0, 0.2, 0.3], [0.2, 0.2, 0.0, 0.3], [0.3, 0.3, 0.3, 0.0]])
MODELS = {"a": MODEL_A, "b": MODEL_B, "c": MODEL_C}
DEFAULT_C = {"RISE": 0.4, "logRISE": 0.8, "RPLE": 0.2}


def random_ising(n, seed, p_edge=0.25, jlo=0.2, jhi=0.6, hmax=0.2):
    """C1: Erdos-Renyi couplings +-U[jlo,jhi], fields U[-hmax,hmax] (SURVEY 8d)."""
    rng = np.random.default_rng(seed)
    m = np.zeros((n, n))
    for i in range(n):
        for j in range(i + 1, n):
            if rng.random() < p_edge:
                m[i, j] = m[j, i] = rng.choice([-1.0, 1.0]) * rng.uniform(jlo, jhi)
        m[i, i] = rng.uniform(-hmax, hmax)
    return m


def histogram_c1(n=16, m_samples=100_000, seed=16):
    model = random_ising(n, seed)
    rng = np.random.default_rng(seed + 1)
    return model, o.sample_exact(o.matrix_to_terms(model), n, m_samples, rng)


def random_spins(n, k, rng):
    """n x k array of independent uniform +-1 spins (int8, spin-major)"""
    return (rng.integers(0, 2, size=(n, k), dtype=np.int8) * 2 - 1).astype(np.int8)


# ---- error model of the tensor-core objective / gradient passes (csrc/eval_tc.cu) ---------------------------------
# The energies are exact integers.  The objective terms pass through fp32 (ex2.approx: 2 ulp; partial sums of <= 32
# terms: 31 * 2^-24), so the objective is bounded by TC_F_REL relative.  The gradient is an exact int64 sum of residual
# digits; its error is the rounding of each residual r_k = s_u w_k psi_k to the node's grid delta = top / qmax(nr) plus
# the fp32 error of psi_k itself.
TC_F_REL = 2e-6
TC_R_QMAX = {1: 120, 2: 32_000, 3: 4_000_000, 4: 1_000_000_000}     # r_qmax(nr)
TC_APPROX_REL = 2.0 ** -22                                         # ex2.approx.ftz.f32 and div.approx.f32: 2 ulp each
# approximate instructions in a residual: RISE / logRISE ex2; RPLE ex2 and the division of 2 w sigma(-2t)
TC_N_APPROX = {"RISE": 1, "RPLE": 2}


def tc_residual_limbs(counts):
    """residual digit planes of the fine level: 3 when sqrt(K) w_max <= 2e-3 (near-uniform counts), else 4"""
    counts = np.asarray(counts, dtype=np.float64)
    return 3 if np.sqrt(len(counts)) * counts.max() / counts.sum() <= 2e-3 else 4


def tc_level_nr(level, n_limbs):
    """residual digit planes of a pass on `level` (BackendTC::level_nr)"""
    return {"rough": 1, "coarse": max(2, n_limbs - 1), "fine": n_limbs}[level]


def tc_pass_terms(counts, spins, x_rows, nodes):
    """The float64 per-node sums the error model needs, at x_rows [len(nodes) x (N+1)] (couplings, then the field).
    Per node u and residual kind ("RISE": psi = e^{-t}, also logRISE; "RPLE": 2 sigma(-2t) = 1 - tanh t), with
    g_k = w_k psi_k the residual magnitude of row k:
      S   = sum_k g_k                     (the RISE sum, which normalises the logRISE gradient)
      se  = sqrt(sum_k (g_k eps_k)^2)     eps_k = 2^-22 per approximate instruction + |t_k| 2^-23 (fp32 rounding of the
                                          energy and of the exponent's argument): the fp32 error of the residuals, as a
                                          standard deviation
      det = sum_k |w32_k - w_k| psi_k     the fp32 rounding of the weights, which can be the same for every row
    plus B = |x_u|_1 (the bound on |t| that sets the residual grid), K (rows) and w_max."""
    counts = np.asarray(counts, dtype=np.float64)
    w = counts / counts.sum()
    dw = np.abs(w.astype(np.float32).astype(np.float64) - w)
    n = spins.shape[0]
    out = {"K": int(np.count_nonzero(counts)), "wmax": float(w.max()), "B": np.zeros(len(nodes)),
           "RISE": {k: np.zeros(len(nodes)) for k in ("S", "se", "det")},
           "RPLE": {k: np.zeros(len(nodes)) for k in ("S", "se", "det")}}
    for q, u in enumerate(nodes):
        xu = np.asarray(x_rows[q], dtype=np.float64)
        nz = np.flatnonzero(xu[:n])
        nz = nz[nz != u]
        t = spins[u] * (xu[n] + xu[nz] @ spins[nz].astype(np.float64))
        out["B"][q] = np.abs(xu[nz]).sum() + abs(xu[n])
        for kind, psi in (("RISE", np.exp(-t)), ("RPLE", 1.0 - np.tanh(t))):
            eps = TC_N_APPROX[kind] * TC_APPROX_REL + np.abs(t) * 2.0 ** -23
            o = out[kind]
            o["S"][q] = w @ psi
            o["se"][q] = np.sqrt(np.sum((w * psi * eps) ** 2))
            o["det"][q] = dw @ psi
    return out


def tc_grad_bar(terms, form, nr, g_ref):
    """Per-component bar on |g - g_ref| for the nodes of `terms` (g_ref [len(nodes) x (N+1)]: the float64 gradient).
    Every row's residual is rounded on the same grid delta (set by w_max, whatever the row's own weight), so the
    rounding noise of a component is sqrt(K) delta / sqrt(12); the bar is 6 standard deviations of rounding and fp32
    noise together, plus the weight rounding.  The approximate instructions can also be biased: that part of their error
    adds coherently over the rows, i.e. up to their relative bound times |g|.  logRISE divides the RISE gradient by S,
    which carries the same errors."""
    kind = "RPLE" if form == "RPLE" else "RISE"
    o = terms[kind]
    top = 2.0 * terms["wmax"] if form == "RPLE" else terms["wmax"] * np.exp(np.minimum(terms["B"], 80.0))
    sq = np.sqrt(terms["K"]) * top / (TC_R_QMAX[nr] * np.sqrt(12.0))
    base = (6.0 * np.hypot(sq, o["se"]) + o["det"])[:, None]
    g_ref = np.abs(np.asarray(g_ref, dtype=np.float64))
    bias = TC_N_APPROX[kind] * TC_APPROX_REL * g_ref
    if form == "logRISE":          # g = G / S: the errors of G and of S both enter
        return (base + g_ref * (6.0 * o["se"] + o["det"])[:, None]) / o["S"][:, None] + 2.0 * bias
    return base + bias


def tc_f_err(f, f_ref, form):
    """relative objective error per node; logRISE's objective is the log of a RISE sum, so its error is that of the sum"""
    f, f_ref = np.asarray(f, dtype=np.float64), np.asarray(f_ref, dtype=np.float64)
    if form == "logRISE":
        return np.abs(np.expm1(f - f_ref))
    return np.abs(f - f_ref) / np.abs(f_ref)


def three_body_model(n, seed, n_triples=None):
    """C4-style: ring of pair couplings +-0.3 plus random triples +-0.4."""
    rng = np.random.default_rng(seed)
    terms = {}
    for i in range(n):
        terms[(i + 1, (i + 1) % n + 1) if i + 1 < (i + 1) % n + 1 else ((i + 1) % n + 1, i + 1)] = \
            float(rng.choice([-0.3, 0.3]))
    for _ in range(n_triples or n):
        t = tuple(sorted(int(x) + 1 for x in rng.choice(n, 3, replace=False)))
        terms[t] = float(rng.choice([-0.4, 0.4]))
    return terms


# ---- which kernels ran, which are compiled ------------------------------------------------------------------------------
def profiled_kernel_names(fn):
    """fn()'s result and the names of the CUDA kernels it launched (torch.profiler)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, [ev.key for ev in prof.key_averages()]


def compiled_kernel_names(lib_path):
    """the (mangled) names of the kernels compiled into the library at lib_path, read with cuobjdump; None without it"""
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not shutil.which(tool):
        return None
    out = subprocess.run([tool, "-sass", str(lib_path)], capture_output=True, text=True, check=True).stdout
    return re.findall(r"Function : (\S+)", out)
