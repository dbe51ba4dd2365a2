"""ctypes binding of libgml_b200.so (include/gml_b200.h).  No CPU fallback: if the CUDA library is
missing and cannot be built, importing the compute entry points fails loudly."""
from __future__ import annotations

import ctypes
import pathlib

_HERE = pathlib.Path(__file__).resolve().parent
import os

# GML_B200_LIB_PATH selects an experimental build variant (developer A/B runs); default = the in-tree product
LIB_PATH = pathlib.Path(os.environ.get("GML_B200_LIB_PATH", str(_HERE / "libgml_b200.so")))

OK, EINVAL, ECUDA, ENOTCONV = 0, 1, 2, 3
RISE_ID, LOGRISE_ID, RPLE_ID = 0, 1, 2
EXACT_MAX_N = 40   # GML_B200_EXACT_MAX_N
MCMC_MAX_N = 4096  # GML_B200_MCMC_MAX_N
TEMPERING_DEFAULT_RUNGS = 16  # GML_B200_TEMPERING_DEFAULT_RUNGS
LOG_Z_DEFAULT_RUNGS = 32  # GML_B200_LOG_Z_DEFAULT_RUNGS
KEYS_PAIRWISE = -1  # GML_B200_KEYS_PAIRWISE
FIT_STEP_SIZE = 0.1  # default eta_0 of fit_likelihood with B200Gibbs
FIT_STEP_S0 = 100.0  # eta_s = eta_0 (1 + s / FIT_STEP_S0)^-0.6 (FIT_STEP_S0 in csrc/common.cuh)
SOLVER_AUTO, SOLVER_NEWTON, SOLVER_FISTA_CC, SOLVER_FISTA_TC = 0, 1, 2, 3

# every symbol include/gml_b200.h declares
EXPORTS = (
    "gml_b200_version", "gml_b200_last_error", "gml_b200_device_count", "gml_b200_opts_default",
    "gml_b200_learn_pairwise", "gml_b200_learn_multibody", "gml_b200_multibody_num_keys",
    "gml_b200_learn_pairwise_matrix", "gml_b200_learn_multibody_matrix", "gml_b200_upload_matrix",
    "gml_b200_create", "gml_b200_destroy", "gml_b200_upload_histogram",
    "gml_b200_attach_histogram_device", "gml_b200_num_samples", "gml_b200_solve_pairwise",
    "gml_b200_solve_pairwise_device", "gml_b200_solve_pairwise_path", "gml_b200_solve_multibody", "gml_b200_solve_multibody_sym",
    "gml_b200_multibody_num_sym_keys", "gml_b200_threshold_device", "gml_b200_eval_pairwise", "gml_b200_bench_passes",
    "gml_b200_symmetrize_device",
    "gml_b200_sample_gibbs_device", "gml_b200_sample_gibbs_terms_device", "gml_b200_sample_exact_device",
    "gml_b200_sample_mcmc_device", "gml_b200_sample_tempering_device", "gml_b200_log_partition_tempering",
    "gml_b200_sample_cluster_device", "gml_b200_moments_cluster",
    "gml_b200_moments_mcmc", "gml_b200_moments_exact", "gml_b200_moments_histogram",
    "gml_b200_fit_likelihood_mcmc", "gml_b200_fit_likelihood_exact",
    "gml_b200_build_histogram_device",
    "gml_b200_comm_unique_id", "gml_b200_comm_init", "gml_b200_comm_globalize_histogram", "gml_b200_comm_attach",
)


class Opts(ctypes.Structure):
    _fields_ = [("tol", ctypes.c_double), ("barrier_mu", ctypes.c_double), ("max_iter", ctypes.c_int32),
                ("solver", ctypes.c_int32), ("device", ctypes.c_int32), ("node_begin", ctypes.c_int32),
                ("node_end", ctypes.c_int32), ("verbose", ctypes.c_int32), ("stream", ctypes.c_void_p),
                ("reserved", ctypes.c_int32 * 8)]


class Stats(ctypes.Structure):
    _fields_ = [("solver_used", ctypes.c_int32), ("iterations", ctypes.c_int32),
                ("n_fg_passes", ctypes.c_int32), ("n_f_passes", ctypes.c_int32),
                ("n_unconverged", ctypes.c_int32), ("n_stalled", ctypes.c_int32),
                ("kernel_launches", ctypes.c_int64), ("evals", ctypes.c_double),
                ("pack_ms", ctypes.c_double), ("h2d_ms", ctypes.c_double), ("solve_ms", ctypes.c_double),
                ("d2h_ms", ctypes.c_double), ("total_ms", ctypes.c_double),
                ("max_residual", ctypes.c_double), ("reserved_d", ctypes.c_double * 4)]

    def as_dict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_ if not k.startswith("reserved")}
        d["energy_fg_ms"], d["grad_ms"], d["energy_f_ms"] = self.reserved_d[0], self.reserved_d[1], self.reserved_d[2]
        d["timed_full_passes"] = int(self.reserved_d[3])
        return d


class GMLB200Error(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"gml_b200 error {code}: {message}")
        self.code = code


_lib = None


def load(build_if_missing: bool = True) -> ctypes.CDLL:
    """Load libgml_b200.so; build it in-tree with nvcc if absent.  Raises if neither works."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        if not build_if_missing:
            raise GMLB200Error(ECUDA, f"{LIB_PATH} is missing (run graphicalmodellearning.jl_b200/build.py)")
        from . import build as _build
        _build.build()
    lib = ctypes.CDLL(str(LIB_PATH))
    c = ctypes
    dp, i8p, vp = c.POINTER(c.c_double), c.POINTER(c.c_int8), c.c_void_p
    op, sp = c.POINTER(Opts), c.POINTER(Stats)
    lib.gml_b200_version.restype = c.c_char_p
    lib.gml_b200_last_error.restype = c.c_char_p
    lib.gml_b200_device_count.restype = c.c_int
    lib.gml_b200_opts_default.argtypes = [op]
    lib.gml_b200_opts_default.restype = None
    lib.gml_b200_learn_pairwise.argtypes = [vp, vp, c.c_int64, c.c_int32, c.c_int64, c.c_int32, c.c_double,
                                            c.c_int32, op, vp, vp, sp]
    lib.gml_b200_learn_multibody.argtypes = [vp, vp, c.c_int64, c.c_int32, c.c_int64, c.c_int32, c.c_double,
                                             op, vp, vp, sp]
    lib.gml_b200_learn_pairwise_matrix.argtypes = [vp, c.c_int32, c.c_int64, c.c_int32, c.c_int64, c.c_int32, c.c_double,
                                                   c.c_int32, op, vp, vp, sp]
    lib.gml_b200_learn_multibody_matrix.argtypes = [vp, c.c_int32, c.c_int64, c.c_int32, c.c_int64, c.c_int32, c.c_double,
                                                    op, vp, vp, sp]
    lib.gml_b200_upload_matrix.argtypes = [vp, vp, c.c_int32, c.c_int64, c.c_int64, c.c_int32, c.c_int64, sp]
    lib.gml_b200_multibody_num_keys.argtypes = [c.c_int32, c.c_int32]
    lib.gml_b200_multibody_num_keys.restype = c.c_int64
    lib.gml_b200_create.argtypes = [c.POINTER(vp), c.c_int32]
    lib.gml_b200_destroy.argtypes = [vp]
    lib.gml_b200_destroy.restype = None
    lib.gml_b200_upload_histogram.argtypes = [vp, vp, vp, c.c_int64, c.c_int32, c.c_int64, sp]
    lib.gml_b200_attach_histogram_device.argtypes = [vp, vp, vp, c.c_int64, c.c_int32, c.c_int64, sp]
    lib.gml_b200_num_samples.argtypes = [vp]
    lib.gml_b200_num_samples.restype = c.c_double
    lib.gml_b200_solve_pairwise.argtypes = [vp, c.c_int32, c.c_double, c.c_int32, op, vp, vp, sp]
    lib.gml_b200_solve_pairwise_device.argtypes = [vp, c.c_int32, c.c_double, op, vp, vp, sp]
    lib.gml_b200_solve_pairwise_path.argtypes = [vp, c.c_int32, vp, c.c_int32, c.c_int32, op, vp, sp]
    lib.gml_b200_solve_multibody.argtypes = [vp, c.c_int32, c.c_double, op, vp, vp, sp]
    lib.gml_b200_solve_multibody_sym.argtypes = [vp, c.c_int32, c.c_double, op, vp, vp, sp]
    lib.gml_b200_multibody_num_sym_keys.argtypes = [c.c_int32, c.c_int32]
    lib.gml_b200_multibody_num_sym_keys.restype = c.c_int64
    lib.gml_b200_threshold_device.argtypes = [vp, c.c_int32, c.c_double, c.POINTER(c.c_int64), vp]
    lib.gml_b200_eval_pairwise.argtypes = [vp, c.c_int32, op, vp, vp, vp]
    lib.gml_b200_bench_passes.argtypes = [vp, c.c_int32, op, c.c_int32, vp]
    lib.gml_b200_symmetrize_device.argtypes = [vp, c.c_int32, vp]
    lib.gml_b200_sample_gibbs_device.argtypes = [c.c_int32, c.c_int32, vp, vp, vp, vp, c.c_int64, c.c_int32,
                                                 c.c_uint64, vp, c.c_int64, vp]
    lib.gml_b200_sample_gibbs_terms_device.argtypes = [c.c_int32, c.c_int32, c.c_int32, c.c_int32, vp, vp, c.c_int64, c.c_int32,
                                                       c.c_uint64, vp, c.c_int64, vp]
    lib.gml_b200_sample_exact_device.argtypes = [c.c_int32, c.c_int32, c.c_int32, c.c_int32, vp, vp, c.c_int64, c.c_int32,
                                                 c.c_uint64, vp, vp, vp, vp, c.c_int64, vp]
    lib.gml_b200_sample_mcmc_device.argtypes = [c.c_int32, c.c_int32, c.c_int32, c.c_int32, vp, vp, c.c_int64, c.c_int32,
                                                c.c_int64, c.c_int32, c.c_int32, c.c_uint64, vp, vp, vp, vp, c.c_int64, vp]
    lib.gml_b200_sample_cluster_device.argtypes = lib.gml_b200_sample_mcmc_device.argtypes
    lib.gml_b200_moments_cluster.argtypes = [c.c_int32, c.c_int32, c.c_int32, c.c_int32, vp, vp, c.c_int64, c.c_int64, c.c_int32,
                                             c.c_int32, c.c_uint64, c.c_int32, c.c_int32, vp, vp, vp, vp, vp]
    lib.gml_b200_sample_tempering_device.argtypes = [c.c_int32, c.c_int32, c.c_int32, c.c_int32, vp, vp, c.c_int32, vp,
                                                     c.c_int64, c.c_int32, c.c_int64, c.c_int32, c.c_int32, c.c_uint64, vp, vp,
                                                     vp, vp, vp, c.c_int64, vp]
    lib.gml_b200_log_partition_tempering.argtypes = [c.c_int32, c.c_int32, c.c_int32, c.c_int32, vp, vp, c.c_int32, vp,
                                                     c.c_int64, c.c_int32, c.c_int64, c.c_uint64, vp, vp, vp, vp, vp]
    lib.gml_b200_moments_mcmc.argtypes = [c.c_int32, c.c_int32, c.c_int32, c.c_int32, vp, vp, c.c_int32, vp, c.c_int64, c.c_int64,
                                          c.c_int32, c.c_int32, c.c_uint64, c.c_int32, c.c_int32, vp, vp, vp, vp, vp, vp]
    lib.gml_b200_moments_exact.argtypes = [c.c_int32, c.c_int32, c.c_int32, c.c_int32, vp, vp, c.c_int32, c.c_int32, vp, vp, vp]
    lib.gml_b200_moments_histogram.argtypes = [vp, c.c_int32, c.c_int32, vp, vp]
    lib.gml_b200_fit_likelihood_mcmc.argtypes = [c.c_int32, c.c_int32, c.c_int32, c.c_int32, vp, vp, vp, c.c_double, c.c_int64,
                                                 c.c_int32, c.c_int32, c.c_int64, c.c_double, c.c_uint64, vp, vp, vp, vp]
    lib.gml_b200_fit_likelihood_exact.argtypes = [c.c_int32, c.c_int32, c.c_int32, c.c_int32, vp, vp, vp, c.c_double, c.c_double,
                                                  c.c_int32, vp, vp, vp, vp]
    lib.gml_b200_build_histogram_device.argtypes = [c.c_int32, vp, c.c_int64, c.c_int32, c.c_int64, vp, c.c_int64, vp,
                                                    c.POINTER(c.c_int64), vp]
    lib.gml_b200_comm_unique_id.argtypes = [vp]
    lib.gml_b200_comm_init.argtypes = [vp, vp, c.c_int32, c.c_int32]
    lib.gml_b200_comm_globalize_histogram.argtypes = [vp]
    lib.gml_b200_comm_attach.argtypes = [vp, vp]
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc == OK:
        return
    raise GMLB200Error(rc, load().gml_b200_last_error().decode())


def default_opts() -> Opts:
    o = Opts()
    load().gml_b200_opts_default(ctypes.byref(o))
    return o
