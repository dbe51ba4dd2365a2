"""Host-side mirror of the reference's operator interface for the learn() hot path.

Same names, argument meaning and error behaviour as lanl-ansi/GraphicalModelLearning.jl:
  RISE / logRISE / RPLE / multiRISE      src/GraphicalModelLearning.jl:20-56
  GMLMethod / NLP                        src/GraphicalModelLearning.jl:59-65
  learn(samples, formulation, method)    src/GraphicalModelLearning.jl:69-73, 83-336
  data_info                              src/GraphicalModelLearning.jl:76-81
  FactorGraph (container + conversions)  src/models.jl:8-20, 105-154
The new method type is `B200` -- the sibling of `NLP` that the Julia shim
(julia/GMLB200.jl) adds; `learn` dispatches to libgml_b200.so through the C ABI.  There is no
CPU code path here: `NLP` (JuMP + Ipopt) is not available in this image and raises.
"""
from __future__ import annotations

import ctypes
import math
from dataclasses import dataclass, field
from typing import Dict, Optional, Tuple

import numpy as np

from . import _lib


# ---- formulations (src/GraphicalModelLearning.jl:20-56) ------------------------------------
class GMLFormulation:
    pass


@dataclass
class multiRISE(GMLFormulation):
    regularizer: float = 0.4
    symmetrization: bool = True
    interaction_order: int = 2


@dataclass
class RISE(GMLFormulation):
    regularizer: float = 0.4
    symmetrization: bool = True


@dataclass
class RISEA(GMLFormulation):   # dead code in the reference (removed JuMP API), kept for the name only
    regularizer: float = 0.4
    symmetrization: bool = True


@dataclass
class logRISE(GMLFormulation):
    regularizer: float = 0.8
    symmetrization: bool = True


@dataclass
class RPLE(GMLFormulation):
    regularizer: float = 0.2
    symmetrization: bool = True


# ---- methods (src/GraphicalModelLearning.jl:59-65) -----------------------------------------
class GMLMethod:
    pass


@dataclass
class NLP(GMLMethod):
    solver: object = None


@dataclass
class B200(GMLMethod):
    """Batched GPU solver.  tol: stopping tolerance (prox-gradient mapping max-norm for FISTA,
    Newton step for the small-problem solver; 0 = solver default 1e-6 / 1e-12).  barrier_mu > 0
    returns the log-barrier point Ipopt stops at (use 1e-9 to reproduce the reference's stored
    fixtures to ~1e-9) instead of the exact L1 minimiser; it needs the Newton solver (at most 128
    features per node).  polish=True finishes a FISTA solve with fp64 Newton on each node's support."""
    tol: float = 0.0
    max_iter: int = 0
    solver: str = "auto"          # auto | newton | fista_cc | fista_tc
    barrier_mu: float = 0.0
    device: int = 0
    verbose: int = 0
    profile: bool = False         # time the contraction kernels with CUDA events (stats energy_*_ms / grad_ms)
    multilevel: bool = False      # FISTA: solve on strided sample subsets first (warm starts); opt-in
    sample_sharded: bool = False  # histogram rows split over ranks, NCCL all-reduce per pass (Session.comm_init)
    coarse_level: object = True   # fista_tc: 3-limb iterate / one residual limb less while far from convergence ("rough": also the
                                  # experimental 2-limb / 8-bit level first)
    devices: int = 1              # one-shot learn(): shard the nodes over this many GPUs from this process
    compaction: bool = True       # FISTA: restrict the passes to the nodes that are still active (parked / converged ones drop out)
    warm_start: Optional[bool] = None   # FISTA, cold solves of all nodes: start from the mean-field couplings (None = the
                                        # library default: on for 128 <= N <= 2048; True forces it on, False switches it off)
    polish: bool = False          # FISTA solvers: finish every node with fp64 Newton on its identified support (exact L1 minimiser to ~1e-12)
    last_stats: dict = field(default_factory=dict, repr=False, compare=False)

    def _opts(self, node_begin: int = 0, node_end: int = 0, stream: int = 0) -> _lib.Opts:
        o = _lib.default_opts()
        o.tol = float(self.tol)
        o.max_iter = int(self.max_iter)
        o.solver = {"auto": 0, "newton": 1, "fista_cc": 2, "fista_tc": 3}[self.solver]
        o.barrier_mu = float(self.barrier_mu)
        o.device = int(self.device)
        o.verbose = int(self.verbose)
        o.node_begin, o.node_end = int(node_begin), int(node_end)
        o.stream = ctypes.c_void_p(stream) if stream else None
        o.reserved[0] = 1 if self.profile else 0
        o.reserved[1] = 1 if self.multilevel else 0
        o.reserved[2] = 1 if self.sample_sharded else 0
        o.reserved[3] = 2 if self.coarse_level == "rough" else (0 if self.coarse_level else 1)
        o.reserved[4] = int(self.devices)
        o.reserved[6] = 0 if self.compaction else 1
        o.reserved[7] = (1 if self.warm_start else 0) | (2 if self.polish else 0) | (4 if self.warm_start is False else 0)
        return o


# ---- FactorGraph (src/models.jl) ------------------------------------------------------------
@dataclass
class FactorGraph:
    order: int
    varible_count: int            # sic -- the reference's spelling (src/models.jl:10)
    alphabet: str
    terms: Dict[Tuple[int, ...], float]
    variable_names: Optional[list] = None

    def __getitem__(self, key):
        return self.terms[tuple(key)]

    def __iter__(self):
        return iter(self.terms.items())

    def keys(self):
        return self.terms.keys()

    @staticmethod
    def from_matrix(m) -> "FactorGraph":
        """FactorGraph(matrix): diagonal -> (i,), upper triangle -> (i,j); zeros dropped
        (src/models.jl:105-135).  Keys are 1-based like the reference's."""
        m = np.asarray(m, dtype=np.float64)
        assert m.shape[0] == m.shape[1]
        n = m.shape[0]
        terms = {}
        for i in range(n):
            if not math.isclose(m[i, i], 0.0, abs_tol=0.0):
                terms[(i + 1,)] = float(m[i, i])
        for i in range(n):
            for j in range(i + 1, n):
                if not math.isclose(m[i, j], 0.0, abs_tol=0.0):
                    terms[(i + 1, j + 1)] = float(m[i, j])
        return FactorGraph(2, n, "spin", terms)

    def to_matrix(self) -> np.ndarray:
        """convert(Array{T,2}, gm) (src/models.jl:137-154)."""
        if self.order != 2:
            raise ValueError(f"cannot convert a FactorGraph of order {self.order} to a matrix")
        m = np.zeros((self.varible_count, self.varible_count))
        for k, v in self.terms.items():
            if len(k) == 1:
                m[k[0] - 1, k[0] - 1] = v
            else:
                m[k[0] - 1, k[1] - 1] = v
                m[k[1] - 1, k[0] - 1] = v
        return m


def matrix_to_dict(m) -> Dict[Tuple[int, ...], float]:
    """convert(Dict, matrix): all ordered pairs + diagonal (src/models.jl:157-182)."""
    m = np.asarray(m)
    n = m.shape[0]
    out = {}
    for i in range(n):
        if m[i, i] != 0.0:
            out[(i + 1,)] = float(m[i, i])
    for i in range(n):
        for j in range(n):
            if i != j and m[i, j] != 0.0:
                out[(i + 1, j + 1)] = float(m[i, j])
    return out


# ---- learn ------------------------------------------------------------------------------------
def data_info(samples):
    """(num_conf, num_spins, num_samples) -- src/GraphicalModelLearning.jl:76-81."""
    num_conf, num_row = samples.shape
    return num_conf, num_row - 1, samples[:, 0].sum()


def regularizer_lambda(c: float, num_spins: int, num_samples: float) -> float:
    """src/GraphicalModelLearning.jl:157."""
    return c * math.sqrt(math.log((num_spins ** 2) / 0.05) / num_samples)


def _pairwise_id(formulation) -> int:
    """Formulation id of the C ABI for RISE / logRISE / RPLE."""
    form_id = {RISE: _lib.RISE_ID, logRISE: _lib.LOGRISE_ID, RPLE: _lib.RPLE_ID}.get(type(formulation))
    if form_id is None:
        raise NotImplementedError(f"{type(formulation).__name__} is not on the B200 hot path")
    return form_id


# precision level of Session.eval_pairwise / bench_passes (opts.reserved[5]): fine, coarse, rough
_LEVELS = {False: 0, True: 1, "rough": 2}


def pack_histogram(samples):
    """[count, s_1..s_N] (any real dtype, any memory order -- the Adjoint shim of :73 is a no-op
    here) -> counts float64[K], spins int8 spin-major [N x K]."""
    samples = np.asarray(samples)
    if samples.ndim != 2 or samples.shape[1] < 2 or samples.shape[0] < 1:
        raise ValueError("samples must be a K x (N+1) matrix [count, s_1..s_N]")
    counts = np.ascontiguousarray(samples[:, 0], dtype=np.float64)
    body = samples[:, 1:]
    spins = np.ascontiguousarray(body.T.astype(np.int8))
    if not np.array_equal(spins, body.T):
        raise ValueError("spin columns must be exactly -1 or +1")
    return counts, spins


def multirise_keys(num_spins: int, u: int, inter_order: int):
    """Keys of node u in the reference's order (src/GraphicalModelLearning.jl:94-104 with
    permutations() of src/models.jl:228-246 = ascending combinations), 1-based."""
    import itertools
    neighbours = [i for i in range(1, num_spins + 1) if i != u]
    keys = [(u,)]
    for p in range(2, inter_order + 1):
        keys.extend((u,) + c for c in itertools.combinations(neighbours, p - 1))
    return keys


def _ptr(a: np.ndarray) -> ctypes.c_void_p:
    return ctypes.c_void_p(a.ctypes.data)


def learn_packed(counts: np.ndarray, spins: np.ndarray, formulation: GMLFormulation, method: B200,
                 lam: Optional[float] = None, return_info: bool = False):
    """learn() on a pre-packed histogram (counts f64[K], spins int8 [N x K] spin-major)."""
    lib = _lib.load()
    N, K = spins.shape
    assert counts.dtype == np.float64 and spins.dtype == np.int8 and counts.shape == (K,)
    assert spins.strides[1] == 1
    ld = spins.strides[0]
    if lam is None:
        lam = regularizer_lambda(formulation.regularizer, N, float(counts.sum()))
    return _learn_one_shot(lib.gml_b200_learn_multibody, lib.gml_b200_learn_pairwise, (_ptr(counts), _ptr(spins), K, N, ld),
                           lam, N, formulation, method, return_info, {"lambda": lam})


MATRIX_DTYPES = {np.dtype(np.float64): 0, np.dtype(np.int64): 1, np.dtype(np.float32): 2, np.dtype(np.int32): 3,
                 np.dtype(np.int8): 4}


def _learn_one_shot(learn_multibody, learn_pairwise, source: tuple, lam: float, N: int, formulation, method: B200,
                    return_info: bool, info: dict):
    """The C call and result of learn_packed / learn_matrix.  learn_multibody / learn_pairwise: their C entry points;
    source: the leading arguments that locate the histogram; lam: the lambda (packed) or regularizer (matrix) argument;
    info: what return_info reports besides the objective and the stats."""
    stats = _lib.Stats()
    obj = np.zeros(N)
    opts = method._opts()
    if isinstance(formulation, multiRISE):
        order = int(formulation.interaction_order)
        vals = np.zeros((N, int(_lib.load().gml_b200_multibody_num_keys(N, order))))
        rc = learn_multibody(*source, order, lam, ctypes.byref(opts), _ptr(vals), _ptr(obj), ctypes.byref(stats))
    else:
        form_id = _pairwise_id(formulation)
        theta = np.zeros((N, N), order="F")                              # Julia-native column-major
        rc = learn_pairwise(*source, form_id, lam, int(bool(formulation.symmetrization)), ctypes.byref(opts),
                            _ptr(theta), _ptr(obj), ctypes.byref(stats))
    method.last_stats = stats.as_dict()
    _lib.check(rc)
    result = _multirise_result(vals, N, formulation) if isinstance(formulation, multiRISE) else np.ascontiguousarray(theta)
    if return_info:
        return result, {**info, "objective": obj, **method.last_stats}
    return result


def _multirise_result(vals: np.ndarray, N: int, formulation) -> "FactorGraph":
    order = int(formulation.interaction_order)
    recon = {}
    for u in range(1, N + 1):
        for f, key in enumerate(multirise_keys(N, u, order)):
            recon[key] = float(vals[u - 1, f])                      # :129-132
    if formulation.symmetrization:                                   # :135-149
        groups: Dict[Tuple[int, ...], list] = {}
        for k, v in recon.items():
            groups.setdefault(tuple(sorted(k)), []).append(v)
        recon = {k: float(np.mean(v)) for k, v in groups.items()}
    return FactorGraph(order, N, "spin", recon)                      # :151


def learn_matrix(samples: np.ndarray, formulation: GMLFormulation, method: B200, return_info: bool = False):
    """learn() straight from the reference's input type: a COLUMN-major (Fortran-order, i.e. Julia-native) K x (N+1) matrix
    [count, s_1..s_N] of float64 / int64 / float32 / int32 / int8.  The library narrows the spins on the host while it
    streams them to the device and computes num_samples and lambda itself (src/GraphicalModelLearning.jl:76-81, :157)."""
    lib = _lib.load()
    if samples.ndim != 2 or samples.shape[1] < 2 or samples.shape[0] < 1:
        raise ValueError("samples must be a K x (N+1) matrix [count, s_1..s_N]")
    K, N = samples.shape[0], samples.shape[1] - 1
    col_major = samples.strides[0] == samples.itemsize and samples.strides[1] >= K * samples.itemsize and \
        samples.strides[1] % samples.itemsize == 0
    if not col_major or samples.dtype not in MATRIX_DTYPES:
        raise ValueError("learn_matrix needs a column-major (Fortran-ordered) matrix of float64 / int64 / float32 / int32 / int8")
    ld = samples.strides[1] // samples.itemsize          # leading dimension >= K (a row range of a taller matrix is fine)
    return _learn_one_shot(lib.gml_b200_learn_multibody_matrix, lib.gml_b200_learn_pairwise_matrix,
                           (_ptr(samples), MATRIX_DTYPES[samples.dtype], K, N, ld), float(formulation.regularizer), N,
                           formulation, method, return_info, {})


def learn(samples, formulation: Optional[GMLFormulation] = None, method: Optional[GMLMethod] = None,
          return_info: bool = False):
    """learn(samples[, formulation[, method]]) -- src/GraphicalModelLearning.jl:69-73.
    Pairwise formulations return the N x N matrix (row u = node u, diagonal = fields, :181-188);
    multiRISE returns a FactorGraph (:151).  Raises on solver failure like the reference's
    @assert (:180)."""
    formulation = RISE() if formulation is None else formulation
    method = B200() if method is None else method
    if isinstance(method, NLP):
        raise NotImplementedError("NLP (JuMP + Ipopt) is the reference's CPU method and is not available here; "
                                  "pass B200() as the method")
    if not isinstance(method, B200):
        raise TypeError("method must be a GMLMethod")
    samples = np.asarray(samples)
    if samples.ndim == 2 and samples.flags.f_contiguous and samples.dtype in MATRIX_DTYPES and samples.shape[0] > 1:
        return learn_matrix(samples, formulation, method, return_info=return_info)      # Julia-native layout: no host copy
    counts, spins = pack_histogram(samples)
    return learn_packed(counts, spins, formulation, method, return_info=return_info)


def sample_terms_device(terms: Dict[Tuple[int, ...], float], num_spins: int, n_samples: int, sweeps: int = 60,
                        seed: int = 0, device: int = 0):
    """Device multi-chain Gibbs sampler (csrc/sampler.cu) for a +-1 model given as a FactorGraph-style term dict
    {(i, ...): weight} with 1-based spin labels (keys of length 1 are fields) -- the distribution the reference's
    `sample` draws from by enumerating all 2^N configurations (src/sampling.jl:58-88), which stops at N ~ 25.
    One sample per chain after `sweeps` sweeps from a random start.  Returns a torch int8 tensor [N x n_samples]
    (spin-major, the layout the solver uploads) on `device`."""
    import torch
    lib = _lib.load()
    order = max((len(k) for k in terms), default=1)
    idx = -np.ones((max(len(terms), 1), order), dtype=np.int32)
    wts = np.zeros(max(len(terms), 1), dtype=np.float32)
    for t, (k, v) in enumerate(terms.items()):
        idx[t, :len(k)] = np.asarray(k, dtype=np.int32) - 1
        wts[t] = v
    out = torch.empty((num_spins, n_samples), dtype=torch.int8, device=f"cuda:{device}")
    _lib.check(lib.gml_b200_sample_gibbs_terms_device(device, num_spins, order, len(terms), _ptr(idx), _ptr(wts),
                                                      n_samples, sweeps, seed, ctypes.c_void_p(out.data_ptr()),
                                                      n_samples, None))
    return out


# ---- samplers (src/sampling.jl:1-3, 90-106) ---------------------------------------------------
class GMLSampler:
    pass


@dataclass
class Gibbs(GMLSampler):
    """The reference's CPU sampler (enumeration of all 2^N configurations on one thread); not available here."""


@dataclass
class B200Exact(GMLSampler):
    """Exact iid sampler on the device (csrc/exact_sampler.cu): the reference's distribution, drawn by enumerating all
    2^N configurations in blocks, for N <= 40.  The draws depend only on (model, number_sample, replicates, seed)."""
    seed: int = 0
    device: int = 0


@dataclass
class B200Gibbs(GMLSampler):
    """Multi-sample Gibbs sampler on the device (csrc/mcmc_sampler.cu) for N <= 4096 spins and terms of order <= 8.  Each
    of `chains` chains (0 = min(round_up(number_sample, 32), 2^17)) runs `burn_in` systematic-scan sweeps from a random
    start, then records its configuration after every `thin`-th sweep.  The draws depend only on (model, number_sample,
    replicates, seed, chains, burn_in, thin).  The draws are correlated and only as good as the chains' mixing:
    last_rhat holds, per replicate of the last call, the split-R-hat (energy, magnetisation) over the chains' halves."""
    seed: int = 0
    device: int = 0
    chains: int = 0
    burn_in: int = 200
    thin: int = 10
    last_rhat: list = field(default_factory=list, repr=False, compare=False)


@dataclass
class B200Tempering(GMLSampler):
    """Replica-exchange (parallel tempering) sampler on the device (csrc/mcmc_sampler.cu) for models whose B200Gibbs chains
    do not mix, such as ferromagnets below T_c and low-temperature spin glasses; N <= 4096, terms of order <= 8.  Each
    chain is a ladder of replicas at the inverse temperatures `betas` (betas[0] = 1, strictly decreasing, non-negative, 2,
    4, 8, 16 or 32 rungs; None = the library's default, 16 rungs geometric from 1 to 0.1) that exchange states between
    adjacent rungs after every sweep; only the beta = 1 replica records.  chains = 0 picks min(round_up(number_sample,
    32/R), 2^17/R) ladders of R rungs.  A draw costs about R times a B200Gibbs draw at the same thin.  The draws depend only
    on (model, number_sample, replicates, seed, chains, burn_in, thin, betas).  last_rhat holds, per replicate of the last
    call, the split-R-hat (energy, magnetisation) of the recorded chains; last_swap_rate the fraction of accepted swaps of
    each adjacent pair of rungs after burn_in (R - 1 floats)."""
    seed: int = 0
    device: int = 0
    chains: int = 0
    burn_in: int = 200
    thin: int = 10
    betas: Optional[list] = None
    last_rhat: list = field(default_factory=list, repr=False, compare=False)
    last_swap_rate: list = field(default_factory=list, repr=False, compare=False)


@dataclass
class B200SwendsenWang(GMLSampler):
    """Swendsen-Wang cluster sampler on the device (csrc/mcmc_sampler.cu) for pairwise models (terms of one or two spins)
    with N <= 4096, such as ferromagnets at or below the critical coupling, where B200Gibbs chains do not mix.  Each
    update bonds the satisfied terms with probability 1 - e^{-2|w_t|} (fields bond to a ghost spin fixed at +1) and flips
    every cluster without the ghost with probability 1/2; it is valid for any signs, but frustrated models gain nothing
    over B200Gibbs.  Fields and schedule as B200Gibbs, one update per "sweep": `chains` chains (0 = min(round_up(
    number_sample, 32), 2^17)) run `burn_in` updates from a random start, then record after every `thin`-th.  The draws
    depend only on (model, number_sample, replicates, seed, chains, burn_in, thin).  The chains sample the fp64 weights to
    within |dw_t| <= 2^-52 + 2^-64 e^{2|w_t|}.  last_rhat holds, per replicate of the last call, the split-R-hat (energy,
    magnetisation) over the chains' halves."""
    seed: int = 0
    device: int = 0
    chains: int = 0
    burn_in: int = 200
    thin: int = 10
    last_rhat: list = field(default_factory=list, repr=False, compare=False)


def _ladder(sampler: B200Tempering) -> np.ndarray:
    """The betas of a B200Tempering as float64 (empty: the library default); ValueError for a ladder the library refuses."""
    if sampler.betas is None:
        return np.zeros(0)
    b = np.asarray(sampler.betas, dtype=np.float64).ravel()
    if len(b) not in (2, 4, 8, 16, 32):
        raise ValueError(f"B200Tempering needs 2, 4, 8, 16 or 32 betas, got {len(b)}")
    if b[0] != 1.0 or not np.isfinite(b).all() or (b < 0).any() or (np.diff(b) >= 0).any():
        raise ValueError("B200Tempering betas must start at 1 and be finite, non-negative and strictly decreasing")
    return b


def _term_arrays(gm: FactorGraph):
    """The term lists of the sampler entry points: (order, term_idx int32 [n_terms x order] 0-based, -1 padded,
    term_weight float64 [n_terms])."""
    order = max((len(k) for k in gm.terms), default=1)
    idx = -np.ones((max(len(gm.terms), 1), order), dtype=np.int32)
    wts = np.zeros(max(len(gm.terms), 1), dtype=np.float64)
    for t, (k, v) in enumerate(gm.terms.items()):
        if min(k, default=1) < 1:
            raise ValueError(f"FactorGraph keys are 1-based spin labels, got {k}")
        idx[t, :len(k)] = np.asarray(k, dtype=np.int64) - 1                     # the library refuses labels > N
        wts[t] = v
    return order, idx, wts


def _pairwise_only(gm: FactorGraph) -> None:
    """ValueError for a term of three or more spins, which B200SwendsenWang does not take"""
    big = next((k for k in gm.terms if len(k) > 2), None)
    if big is not None:
        raise ValueError(f"B200SwendsenWang samples pairwise models only (terms of one or two spins), got the term {big}")


def _sample_call(gm: FactorGraph, number_sample: int, replicates: int, sampler, return_log_z: bool):
    """Validates the arguments of sample / sample_device and runs the sampler's C entry point into device buffers sized
    for the largest possible result (min(n, 2^N) rows per replicate).  Returns (counts, spins, K, log_z); log_z is None
    for the MCMC samplers, which record their R-hat in sampler.last_rhat (B200Tempering: also last_swap_rate)."""
    import torch
    sampler = B200Exact() if sampler is None else sampler
    if isinstance(sampler, Gibbs):
        raise NotImplementedError("Gibbs is the reference's CPU sampler and is not available here; pass B200Exact() "
                                  "(N <= 40) or B200Gibbs() (MCMC) as the sampler")
    if not isinstance(sampler, (B200Exact, B200Gibbs, B200Tempering, B200SwendsenWang)):
        raise TypeError("sampler must be a GMLSampler")
    mcmc = isinstance(sampler, (B200Gibbs, B200Tempering, B200SwendsenWang))
    tempering = isinstance(sampler, B200Tempering)
    name = type(sampler).__name__
    if mcmc:
        sampler.last_rhat = []
        if tempering:
            sampler.last_swap_rate = []
        if return_log_z:
            raise ValueError(f"{name} is an MCMC sampler and has no partition function: return_log_z needs B200Exact")
    if gm.alphabet != "spin":                                                    # src/sampling.jl:95-97
        raise ValueError(f"sampling of a FactorGraph is only supported for the spin alphabet, not {gm.alphabet!r}")
    N, n, reps = int(gm.varible_count), int(number_sample), int(replicates)
    cap = _lib.MCMC_MAX_N if mcmc else _lib.EXACT_MAX_N
    if not 1 <= N <= cap:
        raise ValueError(f"the {name} sampler supports 1 <= N <= {cap} spins, got {N}")
    if n < 1 or reps < 1:
        raise ValueError("number_sample and replicates must be >= 1")
    if mcmc:
        if sampler.chains < 0 or sampler.burn_in < 0 or sampler.thin < 1:
            raise ValueError(f"{name} needs chains >= 0, burn_in >= 0 and thin >= 1")
        if N <= 64 and n >= 2 ** 31:
            raise ValueError(f"{name} builds the histogram of N <= 64 spins from fewer than 2^31 draws per replicate")
    betas = _ladder(sampler) if tempering else None
    order, idx, wts = _term_arrays(gm)
    if isinstance(sampler, B200SwendsenWang):
        _pairwise_only(gm)
    ld = reps * min(n, 1 << N)
    dev = f"cuda:{int(sampler.device)}"
    counts = torch.empty(ld, dtype=torch.float64, device=dev)
    spins = torch.empty((N, ld), dtype=torch.int8, device=dev)
    K = np.zeros(reps, dtype=np.int64)
    lib = _lib.load()
    head = (int(sampler.device), N, order, len(gm.terms), _ptr(idx), _ptr(wts), n, reps)
    tail = (ctypes.c_void_p(counts.data_ptr()), ctypes.c_void_p(spins.data_ptr()), ld, None)
    if not mcmc:
        log_z = ctypes.c_double(0.0)
        _lib.check(lib.gml_b200_sample_exact_device(*head, int(sampler.seed) & (2 ** 64 - 1), _ptr(K), ctypes.byref(log_z), *tail))
        return counts, spins, K, log_z.value
    rhat = np.zeros((reps, 2))
    run = (int(sampler.chains), int(sampler.burn_in), int(sampler.thin), int(sampler.seed) & (2 ** 64 - 1), _ptr(K), _ptr(rhat))
    if tempering:
        swap = np.zeros((reps, (len(betas) or _lib.TEMPERING_DEFAULT_RUNGS) - 1))
        _lib.check(lib.gml_b200_sample_tempering_device(*head[:6], len(betas), _ptr(betas) if len(betas) else None, *head[6:],
                                                        *run, _ptr(swap), *tail))
        sampler.last_swap_rate = swap.tolist()
    elif isinstance(sampler, B200SwendsenWang):
        _lib.check(lib.gml_b200_sample_cluster_device(*head, *run, *tail))
    else:
        _lib.check(lib.gml_b200_sample_mcmc_device(*head, *run, *tail))
    sampler.last_rhat = [tuple(r) for r in rhat.tolist()]
    return counts, spins, K, None


def sample_device(gm: FactorGraph, number_sample: int, replicates: int = 1, sampler: Optional[GMLSampler] = None,
                  return_log_z: bool = False):
    """Device-resident form of `sample`: the packed histogram (counts float64[K], spins int8 [N x K] spin-major, a view with
    leading dimension spins.stride(0)) as torch tensors on the sampler's device.  Session.attach_device(counts.data_ptr(),
    spins.data_ptr(), K, N, spins.stride(0)) takes it without a host copy.  A list of (counts, spins) when replicates > 1;
    with return_log_z (B200Exact only), also log Z (natural log of the partition function)."""
    counts, spins, K, log_z = _sample_call(gm, number_sample, replicates, sampler, return_log_z)
    ends = np.cumsum(K)
    hists = [(counts[e - k:e], spins[:, e - k:e]) for k, e in zip(K.tolist(), ends.tolist())]
    out = hists[0] if replicates == 1 else hists
    return (out, log_z) if return_log_z else out


def sample(gm: FactorGraph, number_sample: int, replicates: int = 1, sampler: Optional[GMLSampler] = None,
           return_log_z: bool = False):
    """sample(gm, number_sample[, replicates[, sampler]]) -- src/sampling.jl:90-106.  Returns the reference's int64
    K x (N+1) matrix [count, s_1..s_N] (spin_i = 2*bit_i - 1), or a list of them when replicates > 1; learn() takes it as it
    is.  Rows are in increasing configuration index, except for B200Gibbs, B200Tempering and B200SwendsenWang beyond 64
    spins, whose rows are the draws in order with count 1.  The default sampler is B200Exact(seed=0, device=0)."""
    counts, spins, K, log_z = _sample_call(gm, number_sample, replicates, sampler, return_log_z)
    rows = int(K.sum())
    c = counts[:rows].cpu().numpy().astype(np.int64)
    s = spins[:, :rows].cpu().numpy().astype(np.int64)
    ends = np.cumsum(K)
    hists = [np.concatenate([c[e - k:e, None], s[:, e - k:e].T], axis=1) for k, e in zip(K.tolist(), ends.tolist())]
    out = hists[0] if replicates == 1 else hists
    return (out, log_z) if return_log_z else out


def log_partition(gm: FactorGraph, sampler: Optional[GMLSampler] = None, sweeps: int = 1000, return_info: bool = False):
    """(log Z, stderr): the natural log of the partition function Z = sum_s exp(sum_t w_t prod s) of a spin model and its
    standard error.  The held-out log-likelihood of a model is then the mean over rows of E(s) = sum_t w_t prod s, minus
    log Z.

    - None or B200Tempering: bridge sampling along a replica-exchange ladder that ends at beta = 0, where log Z = N log 2
      (gml_b200_log_partition_tempering, N <= 4096, terms of order <= 8).  Uses the sampler's seed, device, chains (0 =
      2^17 / R ladders), burn_in and betas (None = the log Z default: 32 rungs evenly spaced from 1 to 0; a given ladder
      must end at 0); thin is ignored.  Each ladder runs burn_in + `sweeps` sweeps; the standard error is the delta-method
      error over the independent ladders.  The estimate is of the model with fp32-rounded weights, which the chains sample:
      it differs from log Z of the fp64 weights by at most sum_t |w_t - fl32(w_t)|.  The result depends only on (model,
      betas, chains, burn_in, sweeps, seed).
    - B200Exact: enumeration (N <= 40); stderr 0.0.
    - return_info (B200Tempering) adds a dict: log_ratio and log_ratio_stderr (log Z_k - log Z_{k+1} per adjacent pair of
      rungs and its standard error), swap_rate (per pair), betas, ladders and sweeps.  A ladder too coarse for the model
      shows there as small swap rates and large per-pair errors.  With B200Exact the dict is empty."""
    sampler = B200Tempering() if sampler is None else sampler
    if isinstance(sampler, B200Gibbs):
        raise ValueError("B200Gibbs has no temperature ladder to bridge: log_partition needs B200Tempering or B200Exact")
    if not isinstance(sampler, (B200Exact, B200Tempering)):
        raise TypeError("log_partition needs a B200Tempering or B200Exact sampler")
    if gm.alphabet != "spin":
        raise ValueError(f"log_partition is only supported for the spin alphabet, not {gm.alphabet!r}")
    exact = isinstance(sampler, B200Exact)
    N = int(gm.varible_count)
    cap = _lib.EXACT_MAX_N if exact else _lib.MCMC_MAX_N
    name = type(sampler).__name__
    if not 1 <= N <= cap:
        raise ValueError(f"log_partition with {name} supports 1 <= N <= {cap} spins, got {N}")
    order, idx, wts = _term_arrays(gm)
    lib = _lib.load()
    seed = int(sampler.seed) & (2 ** 64 - 1)
    log_z = ctypes.c_double(0.0)
    if exact:
        K = np.zeros(1, dtype=np.int64)
        _lib.check(lib.gml_b200_sample_exact_device(int(sampler.device), N, order, len(gm.terms), _ptr(idx), _ptr(wts), 1, 1,
                                                    seed, _ptr(K), ctypes.byref(log_z), None, None, 0, None))
        return (log_z.value, 0.0, {}) if return_info else (log_z.value, 0.0)
    betas = _ladder(sampler)
    if len(betas) and betas[-1] != 0.0:
        raise ValueError("log_partition needs a ladder whose last rung is beta = 0")
    sweeps = int(sweeps)
    if sweeps < 1 or sampler.chains < 0 or sampler.chains == 1 or sampler.burn_in < 0:
        raise ValueError("log_partition needs sweeps >= 1, burn_in >= 0 and chains = 0 or >= 2 (the standard error is "
                         "taken over the ladders)")
    R = len(betas) or _lib.LOG_Z_DEFAULT_RUNGS
    stderr = ctypes.c_double(0.0)
    ratio, swap = np.zeros((R - 1, 2)), np.zeros(R - 1)
    _lib.check(lib.gml_b200_log_partition_tempering(int(sampler.device), N, order, len(gm.terms), _ptr(idx), _ptr(wts),
                                                    len(betas), _ptr(betas) if len(betas) else None, int(sampler.chains),
                                                    int(sampler.burn_in), sweeps, seed, ctypes.byref(log_z),
                                                    ctypes.byref(stderr), _ptr(ratio), _ptr(swap), None))
    if not return_info:
        return log_z.value, stderr.value
    info = {"log_ratio": ratio[:, 0].tolist(), "log_ratio_stderr": ratio[:, 1].tolist(), "swap_rate": swap.tolist(),
            "betas": betas.tolist() if len(betas) else [1.0 - k / (R - 1) for k in range(R)],
            "ladders": int(sampler.chains) or (1 << 17) // R, "sweeps": sweeps}
    return log_z.value, stderr.value, info


def _key_arrays(keys, N: int):
    """A list of 1-based keys (tuples of 1..8 distinct spin labels in [1, N]) as the C ABI's key list: (key_order, key_idx
    int32 [n_keys x key_order] 0-based, -1 padded, the keys as tuples)."""
    keys = [tuple(int(i) for i in k) for k in keys]
    if not keys:
        raise ValueError("moments need at least one key")
    for k in keys:
        if not 1 <= len(k) <= 8 or len(set(k)) != len(k) or min(k) < 1 or max(k) > N:
            raise ValueError(f"a key is a tuple of 1..8 distinct 1-based spin labels in [1, {N}], got {k}")
    order = max(len(k) for k in keys)
    idx = -np.ones((len(keys), order), dtype=np.int32)
    for t, k in enumerate(keys):
        idx[t, :len(k)] = np.asarray(k) - 1
    return order, idx, keys


def _keys_call(keys, N: int):
    """((key_order, n_keys, key_idx pointer), key tuples or None, output shape, the key_idx array the pointer refers to)
    of the C moments entries; keys is a key list or "pairwise" (the N x N output)."""
    if isinstance(keys, str):
        if keys != "pairwise":
            raise ValueError(f'keys must be a list of tuples or "pairwise", got {keys!r}')
        return (0, _lib.KEYS_PAIRWISE, None), None, (N, N), None
    order, idx, tuples = _key_arrays(keys, N)
    return (order, len(tuples), _ptr(idx)), tuples, (len(tuples),), idx


def _moments_result(values, tuples, N: int):
    """An N x N array (pairwise) as it is, or a FactorGraph over the key tuples"""
    if tuples is None:
        return values
    return FactorGraph(max(len(k) for k in tuples), N, "spin", dict(zip(tuples, values.tolist())))


def moments(gm: FactorGraph, sampler: Optional[GMLSampler] = None, number_sample: Optional[int] = None, keys=None):
    """(mean, stderr): the model's moments <prod_{i in t} s_i> of keys t, the derivatives d log Z / d w_t.

    - keys: None = gm's own keys in gm's order; a list of 1-based tuples (1..8 distinct spins each); both return two
      FactorGraphs over those keys.  "pairwise" returns two N x N arrays laid out like learn()'s matrix: <s_i> on the
      diagonal, <s_i s_j> off it.
    - None or B200Exact: enumeration (N <= 40, gml_b200_moments_exact), exact in fp64, stderr all zeros; number_sample must
      be None.  Cost ~2^N * (n_terms + n_keys): pairwise has N(N+1)/2 keys, ~5e11 operations at N = 30, ~9e14 at N = 40.
    - B200Gibbs / B200Tempering (N <= 4096, gml_b200_moments_mcmc) and B200SwendsenWang (gml_b200_moments_cluster) need
      number_sample: the mean is over exactly the draws that sample(gm, number_sample, 1, sampler) returns with the same
      sampler fields, bit for bit, without writing them; stderr comes from G = min(32, warps) groups of chains (NaN with
      fewer than 2).  Sets last_rhat (and last_swap_rate) as sample does.  The Gibbs chains sample fp32-rounded weights:
      the moments of gm differ by at most e^{2 delta} - 1, delta = sum_t |w_t - fl32(w_t)|."""
    sampler = B200Exact() if sampler is None else sampler
    if isinstance(sampler, Gibbs):
        raise NotImplementedError("Gibbs is the reference's CPU sampler and is not available here; pass B200Exact(), "
                                  "B200Gibbs() or B200Tempering()")
    if not isinstance(sampler, (B200Exact, B200Gibbs, B200Tempering, B200SwendsenWang)):
        raise TypeError("sampler must be a GMLSampler")
    mcmc = not isinstance(sampler, B200Exact)
    name = type(sampler).__name__
    if gm.alphabet != "spin":
        raise ValueError(f"moments are only supported for the spin alphabet, not {gm.alphabet!r}")
    N = int(gm.varible_count)
    cap = _lib.MCMC_MAX_N if mcmc else _lib.EXACT_MAX_N
    if not 1 <= N <= cap:
        raise ValueError(f"moments with {name} support 1 <= N <= {cap} spins, got {N}")
    if mcmc and number_sample is None:
        raise ValueError(f"{name} needs number_sample")
    if not mcmc and number_sample is not None:
        raise ValueError("B200Exact moments are exact: number_sample must be None")
    if mcmc and (int(number_sample) < 1 or sampler.chains < 0 or sampler.burn_in < 0 or sampler.thin < 1):
        raise ValueError(f"{name} needs number_sample >= 1, chains >= 0, burn_in >= 0 and thin >= 1")
    betas = _ladder(sampler) if isinstance(sampler, B200Tempering) else None
    if isinstance(sampler, B200SwendsenWang):
        _pairwise_only(gm)
    key_args, tuples, shape, _keep = _keys_call(list(gm.terms) if keys is None else keys, N)
    order, idx, wts = _term_arrays(gm)
    lib = _lib.load()
    seed = int(sampler.seed) & (2 ** 64 - 1)
    mean, err = np.zeros(shape), np.zeros(shape)
    model = (int(sampler.device), N, order, len(gm.terms), _ptr(idx), _ptr(wts))
    if not mcmc:
        _lib.check(lib.gml_b200_moments_exact(*model, *key_args, _ptr(mean), None))
    elif isinstance(sampler, B200SwendsenWang):
        sampler.last_rhat = []
        rhat = np.zeros(2)
        _lib.check(lib.gml_b200_moments_cluster(*model, int(number_sample), int(sampler.chains), int(sampler.burn_in),
                                                int(sampler.thin), seed, *key_args, _ptr(mean), _ptr(err), _ptr(rhat), None))
        sampler.last_rhat = [tuple(rhat.tolist())]
    else:
        sampler.last_rhat = []
        rhat = np.zeros(2)
        if betas is None:
            ladder, swap = (1, None), None
        else:
            ladder = (len(betas), _ptr(betas) if len(betas) else None)
            swap = np.zeros((1, (len(betas) or _lib.TEMPERING_DEFAULT_RUNGS) - 1))
            sampler.last_swap_rate = []
        _lib.check(lib.gml_b200_moments_mcmc(*model, *ladder, int(number_sample), int(sampler.chains), int(sampler.burn_in),
                                             int(sampler.thin), seed, *key_args, _ptr(mean), _ptr(err), _ptr(rhat),
                                             None if swap is None else _ptr(swap), None))
        sampler.last_rhat = [tuple(rhat.tolist())]
        if swap is not None:
            sampler.last_swap_rate = swap.tolist()
    return _moments_result(mean, tuples, N), _moments_result(err, tuples, N)


def empirical_moments(samples, keys="pairwise", device: int = 0):
    """The data's moments sum_k c_k prod_{i in t} s_ki / M of a histogram (any `samples` learn() takes), on the device.
    keys: "pairwise" (an N x N array laid out like learn()'s matrix: <s_i> on the diagonal, <s_i s_j> off it; the
    tensor-core gradient pass at x = 0) or a list of 1-based tuples (a FactorGraph over them; raw counts summed in fp64, so
    integer counts give exactly the MCMC moments of the same draws).  Session.moments does the same for a resident
    histogram."""
    counts, spins = pack_histogram(samples)
    _keys_call(keys, spins.shape[0])                      # refuse bad keys before a device is needed
    return Session(device).upload(counts, spins).moments(keys)


def log_likelihood(gm: FactorGraph, samples, sampler: Optional[GMLSampler] = None, sweeps: int = 1000):
    """(value, stderr): the mean log-likelihood of the rows of `samples` under gm, sum_t w_t <prod_{i in t} s_i>_data -
    log Z.  The data term uses gm's fp64 weights and empirical_moments over gm's keys; log Z and the stderr come from
    log_partition(gm, sampler, sweeps) with its samplers and defaults (None = B200Tempering(); B200Exact for N <= 40)."""
    if not gm.terms:
        raise ValueError("log_likelihood needs a model with at least one term")
    counts, spins = pack_histogram(samples)
    if spins.shape[0] != int(gm.varible_count):
        raise ValueError(f"samples have {spins.shape[0]} spins, the model {gm.varible_count}")
    keys = list(gm.terms)
    _keys_call(keys, spins.shape[0])
    log_z, err = log_partition(gm, sampler, sweeps)
    device = 0 if sampler is None else int(sampler.device)
    data = Session(device).upload(counts, spins).moments(keys)
    energy = float(sum(w * m for w, m in zip(gm.terms.values(), data.terms.values())))
    return energy - log_z, err


def fit_likelihood(gm: FactorGraph, samples, sampler: Optional[GMLSampler] = None, regularizer: float = 0.0,
                   steps: int = 2000, step_size: Optional[float] = None, tol: float = 1e-10, max_iter: int = 100000,
                   return_info: bool = False):
    """Maximum-likelihood refit of gm's weights on gm's own terms: a FactorGraph with gm's keys in gm's order whose weights
    maximise  l(w) = sum_t w_t m^_t - log Z(w) - lambda sum_{|t| >= 2} |w_t|,  starting from gm's weights.  m^_t are the
    data moments of `samples` (any input learn() takes) over gm's keys (terms of at most 8 spins), lambda =
    regularizer_lambda(regularizer, N, M) (fields are not penalised; the default 0 refits on the given support).  Keys
    whose weight in gm is 0 are fitted too.  At the maximum the model's moments equal m^ on every unpenalised term, which
    removes the shrinkage of an L1-penalised RISE / RPLE fit: select the support with learn(), refit it here.

    - None or B200Exact: FISTA with backtracking on the exact objective (gml_b200_fit_likelihood_exact, N <= 40; each
      iteration enumerates 2^N configurations once or twice, so it is practical to about N = 28).  Stops when the max-norm
      of the prox-gradient mapping is <= tol; GMLB200Error (code ENOTCONV) after max_iter iterations.
    - B200Gibbs: stochastic maximum likelihood with persistent chains (gml_b200_fit_likelihood_mcmc, N <= 4096).  The
      sampler's seed, device, chains (0 = 2^17), burn_in and thin (sweeps per step) describe the chains.  `steps`
      preconditioned proximal steps of size step_size (1 + s / 100)^-0.6 (None = the library default, 0.1) run on the
      device; the result is the mean of the weights over the second half of the steps.  The chains sample fl32(w).
    - B200Tempering is refused: persistent replica-exchange ladders are not built.
    - return_info adds a dict: lambda and data_moments (m^ in gm's key order); for B200Gibbs also model_moments (the
      chains' mean moments over the averaged steps), trace (max_t |m^_t - m_t| of every step) and step_sizes; for
      B200Exact the objective l at the result and the iterations run."""
    sampler = B200Exact() if sampler is None else sampler
    if isinstance(sampler, Gibbs):
        raise NotImplementedError("Gibbs is the reference's CPU sampler and is not available here; pass B200Exact() or "
                                  "B200Gibbs()")
    if isinstance(sampler, B200Tempering):
        raise ValueError("fit_likelihood does not take B200Tempering: persistent replica-exchange ladders are not built; "
                         "pass B200Gibbs() or B200Exact()")
    if not isinstance(sampler, (B200Exact, B200Gibbs)):
        raise TypeError("sampler must be B200Exact or B200Gibbs")
    mcmc = isinstance(sampler, B200Gibbs)
    name = type(sampler).__name__
    if gm.alphabet != "spin":
        raise ValueError(f"fit_likelihood is only supported for the spin alphabet, not {gm.alphabet!r}")
    if not gm.terms:
        raise ValueError("fit_likelihood needs a model with at least one term")
    N = int(gm.varible_count)
    cap = _lib.MCMC_MAX_N if mcmc else _lib.EXACT_MAX_N
    if not 1 <= N <= cap:
        raise ValueError(f"fit_likelihood with {name} supports 1 <= N <= {cap} spins, got {N}")
    counts, spins = pack_histogram(samples)
    if spins.shape[0] != N:
        raise ValueError(f"samples have {spins.shape[0]} spins, the model {N}")
    M = float(counts.sum())
    if not (math.isfinite(M) and M > 0 and (counts >= 0).all()):
        raise ValueError("sample counts must be non-negative with a positive finite total")
    regularizer = float(regularizer)
    if not (math.isfinite(regularizer) and regularizer >= 0):
        raise ValueError("regularizer must be finite and >= 0")
    lam = regularizer_lambda(regularizer, N, M)
    steps, max_iter = int(steps), int(max_iter)
    eta0 = _lib.FIT_STEP_SIZE if step_size is None else float(step_size)
    if mcmc:
        if steps < 1 or not (math.isfinite(eta0) and eta0 >= 0):
            raise ValueError("B200Gibbs fits need steps >= 1 and a finite step_size >= 0")
        if sampler.chains < 0 or sampler.chains > 2 ** 31 or sampler.burn_in < 0 or sampler.thin < 1:
            raise ValueError("B200Gibbs needs 0 <= chains <= 2^31, burn_in >= 0 and thin >= 1")
        if sampler.burn_in >= 2 ** 31 or sampler.thin >= 2 ** 31 or (sampler.burn_in + steps * sampler.thin) * N >= 2 ** 62:
            raise ValueError("too many sweeps")
    elif not (math.isfinite(float(tol)) and tol > 0 and 1 <= max_iter < 2 ** 31):
        raise ValueError("B200Exact fits need a finite tol > 0 and 1 <= max_iter < 2^31")
    keys = list(gm.terms)
    _keys_call(keys, N)
    order, idx, wts = _term_arrays(gm)
    data = np.array(list(Session(int(sampler.device)).upload(counts, spins).moments(keys).terms.values()), dtype=np.float64)
    sizes = np.array([len(k) for k in keys])
    if not (np.isfinite(data).all() and (np.abs(data) <= 1).all()):
        raise ValueError("the data moments are not in [-1, 1]")
    unbounded = (np.abs(data) == 1) & ~((sizes >= 2) & (lam > 0))
    if unbounded.any():
        k = keys[int(np.argmax(unbounded))]
        raise ValueError(f"the data moment of {k} is +-1 and lambda does not bound its weight: the likelihood has no "
                         "finite maximum")
    lib = _lib.load()
    out = np.zeros(len(keys))
    model = (int(sampler.device), N, order, len(keys), _ptr(idx), _ptr(wts), _ptr(data), lam)
    info = {"lambda": lam, "data_moments": data.tolist()}
    if mcmc:
        mm, trace = np.zeros(len(keys)), np.zeros(steps)
        _lib.check(lib.gml_b200_fit_likelihood_mcmc(*model, int(sampler.chains), int(sampler.burn_in), int(sampler.thin), steps,
                                                    eta0, int(sampler.seed) & (2 ** 64 - 1), _ptr(out), _ptr(mm), _ptr(trace),
                                                    None))
        info.update(model_moments=mm.tolist(), trace=trace.tolist(),
                    step_sizes=[eta0 * (1.0 + s / _lib.FIT_STEP_S0) ** -0.6 for s in range(steps)])
    else:
        obj, iters = ctypes.c_double(0.0), ctypes.c_int32(0)
        _lib.check(lib.gml_b200_fit_likelihood_exact(*model, float(tol), max_iter, _ptr(out), ctypes.byref(obj),
                                                     ctypes.byref(iters), None))
        info.update(objective=obj.value, iterations=iters.value)
    fg = FactorGraph(gm.order, N, "spin", dict(zip(keys, out.tolist())))
    return (fg, info) if return_info else fg


class Session:
    """Handle API (include/gml_b200.h): keeps the histogram resident in HBM across calls."""

    def __init__(self, device: int = 0):
        self._lib = _lib.load()
        self._h = ctypes.c_void_p()
        _lib.check(self._lib.gml_b200_create(ctypes.byref(self._h), device))
        self.device = device
        self.N = self.K = 0
        self.upload_stats: dict = {}

    def close(self):
        if self._h:
            self._lib.gml_b200_destroy(self._h)
            self._h = ctypes.c_void_p()

    __del__ = close

    def upload(self, counts: np.ndarray, spins: np.ndarray):
        N, K = spins.shape
        assert counts.dtype == np.float64 and spins.dtype == np.int8 and spins.strides[1] == 1
        st = _lib.Stats()
        _lib.check(self._lib.gml_b200_upload_histogram(self._h, _ptr(counts), _ptr(spins), K, N,
                                                       spins.strides[0], ctypes.byref(st)))
        self.N, self.K, self.upload_stats = N, K, st.as_dict()
        return self

    def attach_device(self, d_counts_ptr: int, d_spins_ptr: int, K: int, N: int, ld: int):
        st = _lib.Stats()
        _lib.check(self._lib.gml_b200_attach_histogram_device(self._h, ctypes.c_void_p(d_counts_ptr),
                                                              ctypes.c_void_p(d_spins_ptr), K, N, ld, ctypes.byref(st)))
        self.N, self.K, self.upload_stats = N, K, st.as_dict()
        return self

    @property
    def num_samples(self) -> float:
        return float(self._lib.gml_b200_num_samples(self._h))

    def moments(self, keys="pairwise"):
        """The resident histogram's moments, as empirical_moments: an N x N array for "pairwise", else a FactorGraph over
        the 1-based key tuples."""
        key_args, tuples, shape, _keep = _keys_call(keys, self.N)
        mean = np.zeros(shape)
        _lib.check(self._lib.gml_b200_moments_histogram(self._h, *key_args, _ptr(mean)))
        return _moments_result(mean, tuples, self.N)

    def _lam(self, formulation, lam: Optional[float]) -> float:
        """lam, by default the reference's lambda (:157) of the resident histogram"""
        return regularizer_lambda(formulation.regularizer, self.N, self.num_samples) if lam is None else lam

    def solve_pairwise(self, formulation, method: B200, lam: Optional[float] = None, return_info=False):
        N = self.N
        form_id = _pairwise_id(formulation)
        lam = self._lam(formulation, lam)
        theta = np.zeros((N, N), order="F")
        obj = np.zeros(N)
        st = _lib.Stats()
        opts = method._opts()
        rc = self._lib.gml_b200_solve_pairwise(self._h, form_id, lam, int(bool(formulation.symmetrization)),
                                               ctypes.byref(opts), _ptr(theta), _ptr(obj), ctypes.byref(st))
        method.last_stats = st.as_dict()
        _lib.check(rc)
        out = np.ascontiguousarray(theta)
        return (out, {"lambda": lam, "objective": obj, **method.last_stats}) if return_info else out

    def solve_pairwise_device(self, formulation, method: B200, d_rows_ptr: int, node_begin: int, node_end: int,
                              lam: Optional[float] = None, stream: int = 0, d_obj_ptr: int = 0):
        form_id = _pairwise_id(formulation)
        lam = self._lam(formulation, lam)
        st = _lib.Stats()
        opts = method._opts(node_begin, node_end, stream)
        rc = self._lib.gml_b200_solve_pairwise_device(self._h, form_id, lam, ctypes.byref(opts),
                                                      ctypes.c_void_p(d_rows_ptr),
                                                      ctypes.c_void_p(d_obj_ptr) if d_obj_ptr else None, ctypes.byref(st))
        method.last_stats = st.as_dict()
        _lib.check(rc)
        return method.last_stats

    def solve_multibody(self, formulation, method: B200, lam: Optional[float] = None, return_info=False):
        """multiRISE on the resident histogram: the raw per-node values [N x n_keys] in the reference's key order
        (src/GraphicalModelLearning.jl:94-104); Dict assembly / mean-symmetrisation: learn_packed."""
        N = self.N
        order = int(formulation.interaction_order)
        lam = self._lam(formulation, lam)
        n_keys = int(self._lib.gml_b200_multibody_num_keys(N, order))
        vals, obj = np.zeros((N, n_keys)), np.zeros(N)
        st = _lib.Stats()
        opts = method._opts()
        rc = self._lib.gml_b200_solve_multibody(self._h, order, lam, ctypes.byref(opts), _ptr(vals), _ptr(obj), ctypes.byref(st))
        method.last_stats = st.as_dict()
        _lib.check(rc)
        return (vals, {"lambda": lam, "objective": obj, **method.last_stats}) if return_info else vals

    def solve_multibody_sym(self, formulation, method: B200, lam: Optional[float] = None, return_info=False):
        """multiRISE with the mean-symmetrisation of :135-149 done on the device: returns the FactorGraph over SORTED
        keys (values zipped with the canonical enumeration: by size, then lexicographic = permutations(1:N, q))."""
        import itertools
        N = self.N
        order = int(formulation.interaction_order)
        lam = self._lam(formulation, lam)
        n_sym = int(self._lib.gml_b200_multibody_num_sym_keys(N, order))
        vals, obj = np.zeros(n_sym), np.zeros(N)
        st = _lib.Stats()
        opts = method._opts()
        rc = self._lib.gml_b200_solve_multibody_sym(self._h, order, lam, ctypes.byref(opts), _ptr(vals), _ptr(obj), ctypes.byref(st))
        method.last_stats = st.as_dict()
        _lib.check(rc)
        keys = itertools.chain.from_iterable(itertools.combinations(range(1, N + 1), q) for q in range(1, order + 1))
        fg = FactorGraph(order, N, "spin", dict(zip(keys, vals.tolist())))
        return (fg, {"lambda": lam, "objective": obj, **method.last_stats}) if return_info else fg

    def threshold(self, theta: np.ndarray, tau: float):
        """Post-hoc support selection on the device: zero the off-diagonal |theta| < tau; returns (theta, nnz)."""
        import torch
        t = torch.from_numpy(np.ascontiguousarray(theta, dtype=np.float64)).to(f"cuda:{self.device}")
        nnz = ctypes.c_int64(0)
        _lib.check(self._lib.gml_b200_threshold_device(ctypes.c_void_p(t.data_ptr()), theta.shape[0], float(tau), ctypes.byref(nnz), None))
        return t.cpu().numpy(), int(nnz.value)

    def eval_pairwise(self, formulation, x: np.ndarray, backend: str = "fista_tc", want_grad: bool = True,
                      coarse: bool = False):
        """f_u and grad f_u at rows x [N x (N+1)] (couplings then field).  coarse=True evaluates on the tensor-core
        backend's coarse precision level (iterate lattice 2^-22, |x| < 1.95, 16-bit residual digits); "rough": the opt-in
        rough level (lattice 2^-14, one 8-bit residual plane)."""
        form_id = _pairwise_id(formulation)
        x = np.ascontiguousarray(x, dtype=np.float64)
        assert x.shape == (self.N, self.N + 1)
        f = np.zeros(self.N)
        g = np.zeros_like(x) if want_grad else None
        opts = B200(solver=backend)._opts()
        opts.reserved[5] = _LEVELS[coarse]
        _lib.check(self._lib.gml_b200_eval_pairwise(self._h, form_id, ctypes.byref(opts), _ptr(x), _ptr(f),
                                                    _ptr(g) if want_grad else None))
        return f, g

    def bench_passes(self, formulation, backend: str = "fista_tc", reps: int = 5, node_begin: int = 0, node_end: int = 0,
                     coarse: bool = False):
        """Mean device ms of the contraction kernels: dict(energy_full, grad, energy_obj, full_pass_wall)."""
        form_id = _pairwise_id(formulation)
        out = np.zeros(4)
        opts = B200(solver=backend)._opts(node_begin, node_end)
        opts.reserved[5] = _LEVELS[coarse]
        _lib.check(self._lib.gml_b200_bench_passes(self._h, form_id, ctypes.byref(opts), reps, _ptr(out)))
        return dict(zip(("energy_full", "grad", "energy_obj", "full_pass_wall"), out.tolist()))

    # ---- sample-sharded mode -------------------------------------------------------------------------
    _comm_owners: dict = {}        # (device, id(group)) -> Session that owns the process's communicator for that group

    def comm_init(self, group=None, reuse: bool = True):
        """Join the library's NCCL communicator over the ranks of a torch.distributed group, then make the resident
        histogram slice global.  The communicator is created ONCE per (device, group) and process -- the 128-byte unique
        id travels through torch.distributed -- and later sessions attach to it (gml_b200_comm_attach): like a process
        group, it is set-up cost, not part of a learn() call."""
        import torch
        import torch.distributed as dist
        key = (self.device, id(group))
        owner = Session._comm_owners.get(key) if reuse else None
        if owner is not None and owner._h:
            if owner is not self:
                _lib.check(self._lib.gml_b200_comm_attach(self._h, owner._h))
            _lib.check(self._lib.gml_b200_comm_globalize_histogram(self._h))
            return self
        if reuse:
            owner = self if not self.N else Session(self.device)      # a data-less handle keeps the communicator alive
        else:
            owner = self
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        ident = (ctypes.c_uint8 * 128)()
        if rank == 0:
            _lib.check(self._lib.gml_b200_comm_unique_id(ident))
        dev = f"cuda:{self.device}" if dist.get_backend(group) == "nccl" else "cpu"
        t = torch.tensor(list(ident), dtype=torch.uint8, device=dev)
        dist.broadcast(t, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        ident = (ctypes.c_uint8 * 128)(*t.cpu().tolist())
        _lib.check(self._lib.gml_b200_comm_init(owner._h, ident, rank, world))
        if reuse:
            Session._comm_owners[key] = owner
        if owner is not self:
            _lib.check(self._lib.gml_b200_comm_attach(self._h, owner._h))
        _lib.check(self._lib.gml_b200_comm_globalize_histogram(self._h))
        return self

    def solve_path(self, formulation, method: B200, regularizers):
        """Regularisation path: one solve per regulariser c (lambda = c*sqrt(log(N^2/0.05)/M), :157), each warm
        started from the previous one.  Returns an array [len(regularizers), N, N]."""
        N = self.N
        form_id = _pairwise_id(formulation)
        lams = np.array([regularizer_lambda(c, N, self.num_samples) for c in regularizers], dtype=np.float64)
        out = np.zeros((len(lams), N, N))
        st = _lib.Stats()
        opts = method._opts()
        rc = self._lib.gml_b200_solve_pairwise_path(self._h, form_id, _ptr(lams), len(lams),
                                                    int(bool(formulation.symmetrization)), ctypes.byref(opts), _ptr(out),
                                                    ctypes.byref(st))
        method.last_stats = st.as_dict()
        _lib.check(rc)
        return np.ascontiguousarray(out.transpose(0, 2, 1))      # column-major slices -> row-major numpy
