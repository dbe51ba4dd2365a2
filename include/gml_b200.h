/*
 * gml_b200.h -- C ABI of libgml_b200.so, the B200-native replacement for the per-node convex fits
 * behind `learn(samples, formulation, method)` of lanl-ansi/GraphicalModelLearning.jl (v0.2.2).
 *
 * The reference has no FFI of its own: the hot path is Julia code that hands each node's problem to
 * JuMP/Ipopt (src/GraphicalModelLearning.jl:83-152, 154-189, 263-298, 301-336).  The entry points
 * below are what a new `GMLMethod` subtype binds with `ccall` (see INTEGRATION.md and
 * graphicalmodellearning.jl_b200/julia/GMLB200.jl); each one cites the reference lines it replaces.
 *
 * Conventions
 *   - plain C types only, no exceptions cross the boundary; every function returns a status code and
 *     `gml_b200_last_error()` holds a thread-local message for the last non-zero status.
 *   - the caller owns every host buffer; the library owns all device memory behind a handle.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point returns
 *     GML_B200_ECUDA.
 *
 * Histogram layout (the reference's `samples` matrix, src/GraphicalModelLearning.jl:76-81):
 *   counts[k]            = samples[k,1]                      (double, > 0)
 *   spins[i*ld + k]      = samples[k,1+i]  in {-1,+1}         (int8, spin-major, ld >= K)
 * which is exactly the memory of Julia's column-major `Int8.(samples[:,2:end])`.
 */
#ifndef GML_B200_H
#define GML_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GML_B200_OK 0
#define GML_B200_EINVAL 1   /* invalid input (shape, spin not +-1, count <= 0, unsupported option) */
#define GML_B200_ECUDA 2    /* CUDA runtime / driver error, or no device */
#define GML_B200_ENOTCONV 3 /* a node did not reach `tol` within `max_iter`; mirrors the reference's
                               @assert termination_status == LOCALLY_SOLVED (:127,180,289,327) */

/* formulation ids: RISE (:154), logRISE (:263), RPLE (:301) */
#define GML_B200_RISE 0
#define GML_B200_LOGRISE 1
#define GML_B200_RPLE 2

/* solver selection */
#define GML_B200_SOLVER_AUTO 0
#define GML_B200_SOLVER_NEWTON 1   /* fp64 proximal-Newton / barrier-Newton, features <= 128 (AUTO: <= 64) */
#define GML_B200_SOLVER_FISTA_CC 2 /* batched FISTA, CUDA-core fp32 contractions                   */
#define GML_B200_SOLVER_FISTA_TC 3 /* batched FISTA, tcgen05 (int8 limb) tensor-core contractions.  The iterate is a
                                      fixed-point number with |x| < 7.9; a node whose optimum lies beyond that range is
                                      detected and re-solved by the FISTA_CC backend inside the same call            */

typedef struct gml_b200_opts {
    double tol;         /* stopping tolerance (max-norm of prox-gradient mapping / Newton step); default 1e-6 FISTA, 1e-12 Newton.
                           FISTA accepts a node that stalls at the gradient noise floor within 10*tol: see gml_b200_stats.n_stalled */
    double barrier_mu;  /* 0 = exact L1 minimiser; > 0 = Ipopt-compatible log-barrier point at this mu (Newton solver: at most
                           128 features per node; AUTO selects it) */
    int32_t max_iter;   /* default 5000 */
    int32_t solver;     /* GML_B200_SOLVER_* */
    int32_t device;     /* CUDA device ordinal */
    int32_t node_begin; /* node shard [node_begin, node_end); node_end <= 0 means N */
    int32_t node_end;
    int32_t verbose;
    void* stream;       /* cudaStream_t to launch on; NULL = the handle's own stream */
    int32_t reserved[8]; /* reserved[0] != 0: time the contraction kernels with CUDA events (stats.reserved_d);
                            reserved[1] != 0: enable the multilevel (sample-subset) continuation of the FISTA solvers;
                            reserved[2] == 1: sample-sharded solve (see gml_b200_comm_init); == 2: force node shards in the
                            multi-device one-shot calls;
                            reserved[3] == 1: disable the lower precision levels of the tensor-core FISTA solver; == 2: also run
                            the experimental rough level first (measured slower: see DESIGN.md);
                            reserved[4] > 1: the one-shot calls split the work over that many devices (device, device+1, ...)
                            from this one process, one host thread per device: histogram rows when every device keeps
                            >= 65536 of them (sample-sharded solve), node shards otherwise;
                            reserved[5]: gml_b200_eval_pairwise / gml_b200_bench_passes run on the coarse (1) or rough (2)
                            precision level;
                            reserved[6] != 0: disable the active-set compaction of the FISTA passes;
                            reserved[7]: bit 0 force the mean-field warm start of cold full pairwise FISTA solves (default: on
                            for 128 <= N <= 2048), bit 2 switch it off, bit 1 finish every node with fp64 Newton on its
                            identified support (exact L1 minimiser to ~1e-10 for any number of features; a node whose support
                            exceeds 128 coordinates keeps its first-order solution -- reported with verbose > 0) */
} gml_b200_opts;

typedef struct gml_b200_stats {
    int32_t solver_used;
    int32_t iterations;       /* outer iterations (max over nodes) */
    int32_t n_fg_passes;      /* full objective+gradient passes over the histogram */
    int32_t n_f_passes;       /* objective-only passes */
    int32_t n_unconverged;    /* nodes that missed tol (the call then returns GML_B200_ENOTCONV) */
    int32_t n_stalled;        /* FISTA: nodes whose gradient mapping stopped improving at the backend's gradient noise floor
                                 with tol < residual <= 10*tol; they are ACCEPTED (not counted in n_unconverged) and their
                                 residual is part of max_residual -- callers that need tol strictly check n_stalled == 0.
                                 Newton, barrier_mu > 0: nodes whose barrier Newton step stayed between 1e-15 (the stop) and
                                 1e-13 with a flat merit for 4 iterations (the fp64 rounding floor); also accepted */
    int64_t kernel_launches;  /* kernels of this library launched by the call */
    double evals;             /* node*sample evals = nodes*K*(fg + 0.5*f), passes weighted by the fraction of
                                 the histogram they swept (coarse continuation levels count 1/stride)  (SURVEY 8d) */
    double pack_ms;           /* device: validate + layout build */
    double h2d_ms;            /* host->device copies */
    double solve_ms;          /* device-timed solver (CUDA events on the launch stream) */
    double d2h_ms;
    double total_ms;          /* host wall clock of the whole call */
    double max_residual;      /* largest final stopping residual over nodes */
    double reserved_d[4];     /* profiling: [0] energy kernel ms in full passes, [1] gradient kernel ms,
                                 [2] energy kernel ms in objective-only passes, [3] number of timed full passes
                                 (only launches over the whole histogram are timed) */
} gml_b200_stats;

typedef struct gml_b200_handle gml_b200_handle;

const char* gml_b200_version(void);
const char* gml_b200_last_error(void);
int gml_b200_device_count(void);
void gml_b200_opts_default(gml_b200_opts* opts);

/* ---- one-shot entry points (host buffers in, host buffers out) ------------------------------- */

/* Replaces learn(samples, ::RISE/::logRISE/::RPLE, ::NLP)  (src/GraphicalModelLearning.jl:154-189,
 * 263-298, 301-336).  `lambda` is the reference's regularizer*sqrt(log(N^2/0.05)/M) (:157), computed
 * by the caller.  out_theta is N x N COLUMN-major (Julia native): out_theta[u + N*i] = x_u[i], the
 * diagonal holds the fields (:181); symmetrised as 0.5*(R+R') iff symmetrize != 0 (:184-186). */
int gml_b200_learn_pairwise(const double* counts, const int8_t* spins, int64_t K, int32_t N, int64_t ld,
                            int32_t formulation, double lambda, int32_t symmetrize,
                            const gml_b200_opts* opts, double* out_theta, double* out_objective /* N, nullable */,
                            gml_b200_stats* stats /* nullable */);

/* Replaces the per-node core of learn(samples, ::multiRISE, ::NLP) (src/GraphicalModelLearning.jl:83-133).
 * out_vals[u*n_keys + f] is node u's value for its f-th key in the reference's own key order:
 * (u,), then (u,j) j ascending, then (u,j<k) lexicographic, ... (src/GraphicalModelLearning.jl:94-104,
 * src/models.jl:228-246).  n_keys = gml_b200_multibody_num_keys(N, order).  Symmetrisation by key
 * (:135-149) is Dict work and stays with the caller. */
int gml_b200_learn_multibody(const double* counts, const int8_t* spins, int64_t K, int32_t N, int64_t ld,
                             int32_t interaction_order, double lambda, const gml_b200_opts* opts,
                             double* out_vals, double* out_objective /* N, nullable */, gml_b200_stats* stats);

int64_t gml_b200_multibody_num_keys(int32_t N, int32_t interaction_order);

/* ---- the reference's own input type ---------------------------------------------------------------
 * `samples` as learn() receives it (src/GraphicalModelLearning.jl:69-81): a COLUMN-major K x (N+1) matrix with leading
 * dimension ld (in elements), column 0 = counts, column 1+i = spin i in {-1,+1}; element type Float64 (readdlm) or Int64
 * (`sample`, src/sampling.jl:54), also Float32 / Int32 / Int8.  The library narrows the spins to bytes on the host with a
 * thread pool (validating +-1) while streaming them to the device, computes num_samples (:79) and
 * lambda = regularizer*sqrt(log(N^2/0.05)/num_samples) (:157) itself, and then does what gml_b200_learn_pairwise does.
 * With opts->reserved[4] = n > 1 the histogram rows are split over n devices (sample-sharded solve). */
#define GML_B200_DTYPE_F64 0
#define GML_B200_DTYPE_I64 1
#define GML_B200_DTYPE_F32 2
#define GML_B200_DTYPE_I32 3
#define GML_B200_DTYPE_I8 4
int gml_b200_learn_pairwise_matrix(const void* samples, int32_t dtype, int64_t K, int32_t N, int64_t ld,
                                   int32_t formulation, double regularizer, int32_t symmetrize,
                                   const gml_b200_opts* opts, double* out_theta, double* out_objective /* N, nullable */,
                                   gml_b200_stats* stats /* nullable */);
int gml_b200_learn_multibody_matrix(const void* samples, int32_t dtype, int64_t K, int32_t N, int64_t ld,
                                    int32_t interaction_order, double regularizer, const gml_b200_opts* opts,
                                    double* out_vals, double* out_objective /* N, nullable */, gml_b200_stats* stats);

/* ---- handle API: keep the histogram resident in HBM across solves ----------------------------- */

int gml_b200_create(gml_b200_handle** h, int32_t device);
void gml_b200_destroy(gml_b200_handle* h);

/* data_info (src/GraphicalModelLearning.jl:76-81) + device layout build.  Host pointers. */
int gml_b200_upload_histogram(gml_b200_handle* h, const double* counts, const int8_t* spins,
                              int64_t K, int32_t N, int64_t ld, gml_b200_stats* stats);
/* Same from the reference's K x (N+1) matrix (see gml_b200_learn_pairwise_matrix); rows [row_begin, row_begin + K) of a
 * matrix with leading dimension ld are ingested.  stats->h2d_ms covers narrowing + transfer (they overlap). */
int gml_b200_upload_matrix(gml_b200_handle* h, const void* samples, int32_t dtype, int64_t row_begin, int64_t K, int32_t N,
                           int64_t ld, gml_b200_stats* stats);
/* Same, but counts/spins already live in device memory of h's device (no host copies). */
int gml_b200_attach_histogram_device(gml_b200_handle* h, const double* d_counts, const int8_t* d_spins,
                                     int64_t K, int32_t N, int64_t ld, gml_b200_stats* stats);
/* sum of counts of the resident histogram (num_samples of data_info) */
double gml_b200_num_samples(const gml_b200_handle* h);

/* Solve on the resident histogram, result to host (same layout as gml_b200_learn_pairwise). */
int gml_b200_solve_pairwise(gml_b200_handle* h, int32_t formulation, double lambda, int32_t symmetrize,
                            const gml_b200_opts* opts, double* out_theta, double* out_objective,
                            gml_b200_stats* stats);
/* Solve the node shard [opts->node_begin, opts->node_end) and leave the rows in device memory:
 * d_out_rows is (node_end-node_begin) x N ROW-major (row u contiguous) so that shards of several
 * GPUs concatenate with one all-gather.  No symmetrisation here. */
int gml_b200_solve_pairwise_device(gml_b200_handle* h, int32_t formulation, double lambda,
                                   const gml_b200_opts* opts, double* d_out_rows, double* d_out_objective /* nullable */,
                                   gml_b200_stats* stats);
/* Regularisation path (SURVEY 8f-3): solves the same histogram for n_lambda values of lambda, each solve warm
 * started from the previous solution (pass the lambdas in decreasing order).  out_thetas holds n_lambda
 * consecutive N x N column-major matrices.  FISTA solvers only (opts->solver = FISTA_TC / FISTA_CC, or AUTO with
 * more than 64 features). */
int gml_b200_solve_pairwise_path(gml_b200_handle* h, int32_t formulation, const double* lambdas, int32_t n_lambda,
                                 int32_t symmetrize, const gml_b200_opts* opts, double* out_thetas, gml_b200_stats* stats);
int gml_b200_solve_multibody(gml_b200_handle* h, int32_t interaction_order, double lambda,
                             const gml_b200_opts* opts, double* out_vals, double* out_objective,
                             gml_b200_stats* stats);

/* multiRISE with the symmetrisation of src/GraphicalModelLearning.jl:135-149 done on the device: out_sym_vals[i] is the
 * MEAN of the per-node estimates of the i-th sorted key, sorted keys enumerated by size (1..interaction_order) and then
 * lexicographically -- the order of the reference's permutations(1:N, q) (src/models.jl:228-246), so the caller zips the
 * values with that enumeration instead of grouping 13 080 boxed Dict entries.  n = gml_b200_multibody_num_sym_keys. */
int gml_b200_solve_multibody_sym(gml_b200_handle* h, int32_t interaction_order, double lambda,
                                 const gml_b200_opts* opts, double* out_sym_vals, double* out_objective,
                                 gml_b200_stats* stats);
int64_t gml_b200_multibody_num_sym_keys(int32_t N, int32_t interaction_order);

/* Post-hoc support selection (SURVEY 8f-3): zero the off-diagonal entries of a ROW-major N x N device matrix with
 * |theta| < tau; *out_nnz (nullable) receives the number of surviving off-diagonal entries. */
int gml_b200_threshold_device(double* d_theta, int32_t N, double tau, int64_t* out_nnz, void* stream);

/* Objective and gradient of the smooth part f_u (src/GraphicalModelLearning.jl:170 / 279 / 317) for all nodes of
 * the shard at a caller-supplied point.  x, g_out: (node_end-node_begin) x (N+1) row-major host arrays, feature
 * order = couplings to spins 0..N-1 (the self entry is ignored / returns 0), then the local field.  `solver`
 * selects the contraction backend (GML_B200_SOLVER_FISTA_CC or _TC; the TC backend rounds x to the lattice of the
 * precision level chosen by opts->reserved[5]: 2^-24 fine, 2^-22 coarse, 2^-14 rough; a coefficient outside the level's
 * range (|x| < 7.9 fine, < 1.95 below) is GML_B200_EINVAL, never clamped). */
int gml_b200_eval_pairwise(gml_b200_handle* h, int32_t formulation, const gml_b200_opts* opts, const double* x,
                           double* f_out, double* g_out /* nullable */);

/* Times `reps` full objective+gradient passes and `reps` objective-only passes of the contraction backend
 * selected by opts->solver over the shard, with CUDA events around each kernel.  out_ms[0] = mean energy-kernel ms
 * in a full pass, out_ms[1] = mean gradient-kernel ms, out_ms[2] = mean energy-kernel ms in an objective-only
 * pass, out_ms[3] = mean wall ms of a full pass (all kernels of the pass). */
int gml_b200_bench_passes(gml_b200_handle* h, int32_t formulation, const gml_b200_opts* opts, int32_t reps,
                          double* out_ms);

/* 0.5*(R + R') in place on a ROW-major N x N device matrix (src/GraphicalModelLearning.jl:184-186). */
int gml_b200_symmetrize_device(double* d_theta, int32_t N, void* stream);

/* ---- input generator (SURVEY 8f-2): multi-chain Gibbs sampler for pairwise +-1 models ----------
 * Fills d_spins (int8, spin-major, ld >= n_samples) with one sample per chain after `sweeps` full
 * sweeps from a random start.  Neighbour lists in CSR form on the host.  Deterministic in `seed`. */
int gml_b200_sample_gibbs_device(int32_t device, int32_t N, const int32_t* row_ptr, const int32_t* col_idx,
                                 const float* coupling, const float* field, int64_t n_samples,
                                 int32_t sweeps, uint64_t seed, int8_t* d_spins, int64_t ld, void* stream);

/* Same for general +-1 models p(s) ~ exp(sum_t w_t prod_{i in t} s_i) -- the distribution the reference's `sample`
 * enumerates for order > 2 (src/sampling.jl:58-88); generates the 3-body inputs of the multiRISE benchmark config.
 * term_idx: n_terms x order 0-based spin ids, -1 padded (a term of length 1 is a field); term_weight[n_terms]. */
int gml_b200_sample_gibbs_terms_device(int32_t device, int32_t N, int32_t order, int32_t n_terms, const int32_t* term_idx,
                                       const float* term_weight, int64_t n_samples, int32_t sweeps, uint64_t seed,
                                       int8_t* d_spins, int64_t ld, void* stream);

/* Exact iid sampler: the reference's `sample(gm, number_sample, replicates)` (src/sampling.jl:58-106) on the device, for the
 * same term lists as gml_b200_sample_gibbs_terms_device but with fp64 weights.  p(s) ~ exp(sum_t w_t prod_{i in t} s_i),
 * drawn exactly by enumerating all 2^N configurations (never stored: they are recomputed in blocks of 2^12).
 * Configuration c has spin_i = 2*bit_i(c) - 1 (bit 0 = spin 1, src/sampling.jl:11-14).  Replicate r is the histogram of
 * draws [r*n_samples, (r+1)*n_samples) of one counter-based stream; its rows are the configurations drawn at least once,
 * in increasing c.  The output depends only on (terms, n_samples, replicates, seed).
 *   - out_K[replicates] receives the rows of every replicate, *out_log_z (nullable) the natural log of the partition
 *     function.  With d_counts == NULL nothing else is written; with buffers (the histogram layout above, ld >= sum of
 *     out_K, e.g. replicates * min(n_samples, 2^N)), replicate r's rows follow those of replicate r-1.  The buffers are
 *     device memory of `device` (written in place) or host memory (staged on the device and copied back).
 *     A count-only call costs as much as a full one: callers that can afford the bound should pass buffers at once.
 *   - N <= 40 (GML_B200_EXACT_MAX_N).  Cost ~ 2^N * n_terms fp64 sign+add (plus the same again for the blocks that
 *     receive draws); device memory ~ 40 * 2^(N-12) bytes + 10 bytes per draw.
 *   - GML_B200_EINVAL: N outside [1, 40], an index outside [-1, N) or repeated in a term, a non-finite weight (or sum of
 *     |weights|), n_samples < 1, replicates < 1, or ld smaller than the rows (out_K is then filled). */
#define GML_B200_EXACT_MAX_N 40
int gml_b200_sample_exact_device(int32_t device, int32_t N, int32_t order, int32_t n_terms, const int32_t* term_idx,
                                 const double* term_weight, int64_t n_samples, int32_t replicates, uint64_t seed,
                                 int64_t* out_K /* [replicates] */, double* out_log_z /* nullable */,
                                 double* d_counts, int8_t* d_spins, int64_t ld, void* stream);

/* Multi-sample Gibbs sampler: `sample(gm, number_sample, replicates)` by MCMC for models beyond the exact sampler's cap, on
 * the term lists of gml_b200_sample_exact_device (fp64 weights, rounded once to fp32 on the device).  Systematic-scan
 * single-site Gibbs; one warp advances 32 chains with their spins in shared memory.  Each chain runs burn_in sweeps from a
 * random start, then records its configuration at the end of every thin-th sweep; draw d = r*chains + c is chain c's r-th
 * record and the first n_samples draws form a replicate.  Replicate r runs chains [r*chains, (r+1)*chains) of one
 * counter-based stream, so replicates are independent and replicate 0 equals a single-replicate call.  chains = 0 picks
 * min(round_up(n_samples, 32), 2^17).  The output depends only on (terms, n_samples, replicates, chains, burn_in, thin,
 * seed).
 *   - N <= 64: each replicate is a deduplicated histogram, rows in increasing configuration index (the layout of
 *     gml_b200_sample_exact_device).  N > 64: each replicate is n_samples rows of count 1, draw order; repeated
 *     configurations are not merged (learn() weighs a repeated row exactly like one row with the summed count).
 *   - out_K[replicates] receives the rows of every replicate; out_rhat (nullable) [replicates][2] the split-R-hat of the
 *     energy sum_t w_t prod s and of the magnetisation sum_i s_i over the 2*chains half-chains of the floor(n_samples /
 *     chains) records every chain holds (NaN when a half holds fewer than 2; when no half-chain varies, 1 if they all
 *     hold the same value and +inf if not).  Buffers as gml_b200_sample_exact_device:
 *     d_counts == NULL is a count-only call, device buffers are written in place, host buffers are staged on the device.
 *   - GML_B200_EINVAL: N outside [1, GML_B200_MCMC_MAX_N], order outside [1, 8], an index outside [-1, N) or repeated in a
 *     term, a non-finite weight, n_samples < 1, replicates < 1, chains < 0, burn_in < 0, thin < 1, N <= 64 with
 *     n_samples >= 2^31, or ld smaller than the rows (out_K is then filled). */
#define GML_B200_MCMC_MAX_N 4096
int gml_b200_sample_mcmc_device(int32_t device, int32_t N, int32_t order, int32_t n_terms, const int32_t* term_idx,
                                const double* term_weight, int64_t n_samples, int32_t replicates, int64_t chains,
                                int32_t burn_in, int32_t thin, uint64_t seed, int64_t* out_K /* [replicates] */,
                                double* out_rhat /* nullable, [replicates][2]: energy, magnetisation */, double* d_counts,
                                int8_t* d_spins, int64_t ld, void* stream);

/* Replica-exchange (parallel tempering) sampler: gml_b200_sample_mcmc_device for models whose single-site Gibbs chains do
 * not mix (strong ferromagnets, low-temperature glasses).  A chain is a ladder of n_rungs replicas of the model at the
 * inverse temperatures betas[0] = 1 > betas[1] > ... >= 0 (replica k draws from p(s)^betas[k]); after every sweep the
 * adjacent pairs (k, k+1) with k = sweep (mod 2) propose to exchange their states (deterministic even-odd scheme), accepted
 * with probability min(1, exp((beta_k - beta_{k+1}) (E_{k+1} - E_k))), E = sum_t w_t prod s.  Only the beta = 1 replica
 * records: draw d = r*chains + c is ladder c's r-th record.  n_rungs = 0 with betas = NULL selects the default ladder:
 * 16 rungs geometric from 1 to 0.1 (beta_k = 0.1^(k/15)).  chains = 0 picks min(round_up(n_samples, 32/R), 2^17/R) ladders
 * of R rungs.  Each ladder yields one draw per record step, so a draw costs about R times a gml_b200_sample_mcmc_device
 * draw at the same thin.  The output depends only on (terms, n_samples, replicates, chains, burn_in, thin, betas, seed).
 *   - Output layout, out_K, out_rhat (of the beta = 1 records) and the buffers as gml_b200_sample_mcmc_device.
 *   - out_swap_rate (nullable) [replicates][n_rungs - 1] (default ladder: GML_B200_TEMPERING_DEFAULT_RUNGS - 1): per
 *     adjacent pair, the fraction of the swaps proposed after burn_in that were accepted (NaN when none was proposed).
 *   - GML_B200_EINVAL: everything gml_b200_sample_mcmc_device refuses, n_rungs not in {0, 2, 4, 8, 16, 32}, exactly one of
 *     n_rungs == 0 and betas == NULL, betas[0] != 1, betas not strictly decreasing, or a negative or non-finite beta. */
#define GML_B200_TEMPERING_MAX_RUNGS 32
#define GML_B200_TEMPERING_DEFAULT_RUNGS 16
int gml_b200_sample_tempering_device(int32_t device, int32_t N, int32_t order, int32_t n_terms, const int32_t* term_idx,
                                     const double* term_weight, int32_t n_rungs, const double* betas /* [n_rungs] */,
                                     int64_t n_samples, int32_t replicates, int64_t chains, int32_t burn_in, int32_t thin,
                                     uint64_t seed, int64_t* out_K /* [replicates] */,
                                     double* out_rhat /* nullable [replicates][2] */,
                                     double* out_swap_rate /* nullable [replicates][n_rungs - 1] */, double* d_counts,
                                     int8_t* d_spins, int64_t ld, void* stream);

/* Swendsen-Wang cluster sampler: gml_b200_sample_mcmc_device for pairwise models whose single-site Gibbs chains do not
 * mix, such as ferromagnets at or below the critical coupling.  Edwards-Sokal form with a ghost spin fixed at +1 that
 * carries the fields: each update bonds every term t = (i, j) or (i,) with w_t s_i s_j > 0 (s_ghost = +1) with probability
 * 1 - e^{-2|w_t|} (unsatisfied terms never bond; bonds are per term, so repeated keys stay correct) and flips every
 * cluster without the ghost with probability 1/2.  One update counts as one sweep for burn_in and thin.  Valid for any
 * signs; on frustrated models it samples correctly without the speed-up.
 *   - Arguments, output layout, out_K, out_rhat, the buffers and chains = 0 (min(round_up(n_samples, 32), 2^17)) as
 *     gml_b200_sample_mcmc_device; the output depends only on (terms, n_samples, replicates, chains, burn_in, thin, seed).
 *   - Accuracy: "no bond" is drawn when a 64-bit uniform lies below q_t = e^{-2|w_t|}, computed on the host in fp64
 *     from the fp64 weights, so the chains sample the model with w'_t = -1/2 log q'_t, |w'_t - w_t| <= 2^-52 +
 *     2^-64 e^{2|w_t|} (while that is <= 1/2).  Unlike the Gibbs samplers, no weight is rounded to fp32.
 *   - GML_B200_EINVAL: everything gml_b200_sample_mcmc_device refuses, a term of three or more spins, or
 *     (burn_in + ceil(n_samples / chains) * thin) * (n_terms + N + 1) >= 2^62 counters. */
int gml_b200_sample_cluster_device(int32_t device, int32_t N, int32_t order, int32_t n_terms, const int32_t* term_idx,
                                   const double* term_weight, int64_t n_samples, int32_t replicates, int64_t chains,
                                   int32_t burn_in, int32_t thin, uint64_t seed, int64_t* out_K /* [replicates] */,
                                   double* out_rhat /* nullable, [replicates][2]: energy, magnetisation */,
                                   double* d_counts, int8_t* d_spins, int64_t ld, void* stream);

/* Partition function by replica exchange: *out_log_z = log Z, Z = sum_s exp(sum_t w_t prod s), for the models of
 * gml_b200_sample_tempering_device (N <= 4096, order <= 8) by bridge sampling between the adjacent rungs of ladders
 * betas[0] = 1 > betas[1] > ... > betas[R-1] = 0; log Z(0) = N log 2 ties the chain of ratios to a known value.
 *   - Each of `chains` ladders runs the replica-exchange kernel of gml_b200_sample_tempering_device (the same RNG streams
 *     and swaps, no draws) for burn_in + sweeps sweeps.  On each of the last `sweeps` sweeps, before the swap, pair k
 *     (dbeta_k = beta_k - beta_{k+1}) adds the fp64 energies E_{k+1} of rung k+1 and E_k of rung k to
 *     a_{c,k} = log mean exp(+dbeta_k E_{k+1} / 2) and b_{c,k} = log mean exp(-dbeta_k E_k / 2) (running log-sum-exps).
 *     Over the L ladders a_k = logsumexp_c a_{c,k} - log L, b_k likewise, and the geometric bridge (Meng & Wong 1996) gives
 *     log Z_k - log Z_{k+1} = a_k - b_k and log Z = N log 2 + sum_k (a_k - b_k).
 *   - *out_stderr (nullable): the delta-method standard error over the independent ladders, std_c(sum_k u_{c,k}) / sqrt(L)
 *     with ddof = 1, u_{c,k} = exp(a_{c,k} - a_k) - exp(b_{c,k} - b_k).  out_log_ratio (nullable) [n_rungs-1][2]: per pair
 *     the estimate a_k - b_k and its standard error (the same formula without the sum over k); the estimates sum to
 *     log Z - N log 2.  out_swap_rate (nullable) [n_rungs-1]: the swap rates as gml_b200_sample_tempering_device.  The
 *     reduction runs in ladder order: the result depends only on (terms, betas, chains, burn_in, sweeps, seed).
 *   - n_rungs = 0 with betas = NULL selects GML_B200_LOG_Z_DEFAULT_RUNGS rungs evenly spaced, beta_k = 1 - k/31.
 *     chains = 0 picks 2^17 / R ladders (4096 for 32 rungs).  Cost ~ chains * R * (burn_in + sweeps) site updates.
 *   - Accuracy: the estimate is of the model with fp32-rounded weights, the model the chains sample; |log Z(w) -
 *     log Z(fl32(w))| <= sum_t |w_t - fl32(w_t)|.  Each bridge is accurate while dbeta_k * (spread of E at rungs k, k+1)
 *     stays of order 1; a ladder too coarse for the model shows as small swap rates and large per-pair standard errors,
 *     and nothing is clamped.  At most 32 rungs.
 *   - GML_B200_EINVAL: everything gml_b200_sample_tempering_device refuses that applies here (N, order, terms, weights,
 *     the ladder), betas[n_rungs-1] != 0, chains < 0, chains == 1 (no standard error), burn_in < 0, sweeps < 1,
 *     out_log_z == NULL, or (burn_in + sweeps) * N >= 2^62 site steps. */
#define GML_B200_LOG_Z_DEFAULT_RUNGS 32
int gml_b200_log_partition_tempering(int32_t device, int32_t N, int32_t order, int32_t n_terms, const int32_t* term_idx,
                                     const double* term_weight, int32_t n_rungs, const double* betas /* [n_rungs] */,
                                     int64_t chains, int32_t burn_in, int64_t sweeps, uint64_t seed, double* out_log_z,
                                     double* out_stderr /* nullable */,
                                     double* out_log_ratio /* nullable [n_rungs-1][2]: estimate, stderr */,
                                     double* out_swap_rate /* nullable [n_rungs-1] */, void* stream);

/* ---- moments <prod_{i in t} s_i> of keys t: the model's (MCMC or exact) and the data's (resident histogram) --------
 * Keys: n_keys >= 1 rows of key_idx [n_keys x key_order], key_order <= 8, each row 1..8 distinct 0-based spins in
 * [0, N) padded with -1 (the layout of term_idx); out_mean [n_keys].  n_keys = GML_B200_KEYS_PAIRWISE with key_idx =
 * NULL selects all <s_i> and <s_i s_j>: out_mean [N x N] row-major, <s_i> on the diagonal, symmetric.
 *
 * gml_b200_moments_mcmc: the mean of prod_{i in t} s_i over exactly the n_samples draws that
 * gml_b200_sample_mcmc_device (n_rungs = 1, betas = NULL) or gml_b200_sample_tempering_device (otherwise, the same
 * ladder rules) with replicates = 1 and the same sizes and seed returns: the same chains, RNG streams, records and swaps.
 *   - The kernel copies each warp's N state words and a mask of the lanes whose record is a draw to a record buffer of
 *     records * warps * (N + 1) * 4 bytes, one bit per spin and chain record (R bits per draw with R rungs), and
 *     integer popcount reductions sum it: the sums are exact, so the mean is the draws' mean bit for bit.
 *   - out_stderr (nullable): the warps are split into G = min(32, warps) contiguous groups of whole warps with sums S_g
 *     over n_g draws; stderr = sqrt(G/(G-1) sum_g (S_g - mean n_g)^2) / sum n_g, NaN when G < 2.
 *   - out_rhat (nullable) [2] and out_swap_rate (nullable) [n_rungs-1]: as the sampler reports them.
 *   - Pairwise cost: an XNOR-popcount bit-GEMM of N^2/2 * records * warps 32-bit popcounts and G * N^2 * 8 bytes of sums.
 *   - The chains sample fp32-rounded weights: |<f>(w) - <f>(fl32(w))| <= e^{2 delta} - 1, delta = sum_t |w_t - fl32(w_t)|.
 *   - GML_B200_EINVAL: what the sampler entry points refuse, bad keys, n_samples < 1, out_mean == NULL.
 * gml_b200_moments_exact: sum_c e^{E_c} prod s / Z by enumeration for the models of gml_b200_sample_exact_device
 *   (N <= 40), in fp64; the result depends only on (terms, keys).  Cost ~2^N * (n_terms + n_keys) sign+add: pairwise
 *   has N(N+1)/2 keys, ~5e11 operations at N = 30 and ~9e14 at N = 40.
 * gml_b200_moments_histogram: sum_k c_k prod s_k / M over the resident histogram.  Key lists sum the raw counts in fp64
 *   (exact for integer counts below 2^53 in total, so equal to the MCMC mean of the same draws bit for bit); pairwise is the
 *   tensor-core gradient pass at x = 0 (the mean-field warm start's), symmetrised as 0.5 (C + C').  Not for a
 *   sample-sharded histogram. */
#define GML_B200_KEYS_PAIRWISE (-1)
int gml_b200_moments_mcmc(int32_t device, int32_t N, int32_t order, int32_t n_terms, const int32_t* term_idx,
                          const double* term_weight, int32_t n_rungs, const double* betas /* [n_rungs] */, int64_t n_samples,
                          int64_t chains, int32_t burn_in, int32_t thin, uint64_t seed, int32_t key_order, int32_t n_keys,
                          const int32_t* key_idx, double* out_mean, double* out_stderr /* nullable */,
                          double* out_rhat /* nullable [2] */, double* out_swap_rate /* nullable [n_rungs-1] */, void* stream);
/* gml_b200_moments_cluster: gml_b200_moments_mcmc for gml_b200_sample_cluster_device, without a ladder: the mean over
 * exactly the n_samples draws that gml_b200_sample_cluster_device with replicates = 1 and the same sizes and seed returns,
 * with the same group standard errors and out_rhat.  GML_B200_EINVAL: what gml_b200_sample_cluster_device refuses, bad
 * keys, n_samples < 1, out_mean == NULL. */
int gml_b200_moments_cluster(int32_t device, int32_t N, int32_t order, int32_t n_terms, const int32_t* term_idx,
                             const double* term_weight, int64_t n_samples, int64_t chains, int32_t burn_in, int32_t thin,
                             uint64_t seed, int32_t key_order, int32_t n_keys, const int32_t* key_idx, double* out_mean,
                             double* out_stderr /* nullable */, double* out_rhat /* nullable [2] */, void* stream);
int gml_b200_moments_exact(int32_t device, int32_t N, int32_t order, int32_t n_terms, const int32_t* term_idx,
                           const double* term_weight, int32_t key_order, int32_t n_keys, const int32_t* key_idx, double* out_mean,
                           void* stream);
int gml_b200_moments_histogram(gml_b200_handle* h, int32_t key_order, int32_t n_keys, const int32_t* key_idx, double* out_mean);

/* ---- maximum-likelihood refit of a model's weights on its own terms -----------------------------------------------
 * Both entries maximise l(w) = sum_t w_t data_mean[t] - log Z(w) - lambda sum_{|t| >= 2} |w_t| over the weights of the
 * n_terms terms of term_idx (the layout of gml_b200_sample_mcmc_device), starting at init_weight, and write the
 * maximiser to out_weight [n_terms].  data_mean [n_terms] are the data moments <prod_{i in t} s_i> (for example from
 * gml_b200_moments_histogram over the same keys).  Fields (terms of one spin) are not penalised.  At the maximum the
 * model's moments equal data_mean on every unpenalised term.
 *
 * gml_b200_fit_likelihood_mcmc: stochastic maximum likelihood with persistent Gibbs chains, N <= 4096, order <= 8.
 *   - `chains` chains (0 = 2^17) run burn_in sweeps at init_weight.  Then each of `steps` steps s advances them by `thin`
 *     sweeps of one long run (the RNG streams of gml_b200_sample_mcmc_device with the same seed and chains), reduces their
 *     final states to the model moments m_t over gm's terms, and updates every weight on the device:
 *     w_t <- w_t + eta_s g_t / d_t, g_t = data_mean[t] - m_t, d_t = max(1 - data_mean[t]^2, 0.01), soft-thresholded by
 *     eta_s lambda / d_t on terms of >= 2 spins, eta_s = step_size (1 + s / 100)^-0.6.  The chains sample fl32(w).
 *   - out_weight is the mean of w over the steps s >= floor(steps / 2) (Polyak-Ruppert averaging).
 *     out_model_moments (nullable) [n_terms] is the chains' mean moment over the draws of the same steps, sum S / sum n
 *     of integer sums: with step_size = 0 it equals gml_b200_moments_mcmc with burn_in + floor(steps/2) * thin burn-in
 *     sweeps, the same thin, chains and seed, and n_samples = (steps - floor(steps/2)) * chains, bit for bit.
 *     out_trace (nullable) [steps] holds max_t |g_t| of every step.
 *   - No host synchronisation between steps, and no atomics: the result depends only on the arguments.
 * gml_b200_fit_likelihood_exact: FISTA with backtracking on -l with exact log Z and moments by enumeration (the models
 *   of gml_b200_sample_exact_device, N <= 40; each iteration costs one or two passes of ~2^N * 2 n_terms sign+add).  It
 *   stops when the max-norm of the prox-gradient mapping is <= tol; *out_objective (nullable) = l(out_weight),
 *   *out_iterations (nullable) = the iterations run.  GML_B200_ENOTCONV (out_weight holds the last iterate) after max_iter.
 *
 * GML_B200_EINVAL: what gml_b200_moments_mcmc / gml_b200_moments_exact refuse for the model and sizes, n_terms < 1, a null
 * data_mean or out_weight, a data_mean entry outside [-1, 1] or not finite, |data_mean[t]| = 1 on a term that lambda
 * does not bound (a field, or lambda = 0: no finite maximum), lambda < 0 or not finite, steps < 1, step_size < 0 or not
 * finite (step_size = 0 samples init_weight unchanged), (burn_in + steps * thin) * N >= 2^62, tol <= 0, max_iter < 1. */
int gml_b200_fit_likelihood_mcmc(int32_t device, int32_t N, int32_t order, int32_t n_terms, const int32_t* term_idx,
                                 const double* init_weight, const double* data_mean, double lambda, int64_t chains, int32_t burn_in,
                                 int32_t thin, int64_t steps, double step_size, uint64_t seed, double* out_weight,
                                 double* out_model_moments /* nullable [n_terms] */, double* out_trace /* nullable [steps] */,
                                 void* stream);
int gml_b200_fit_likelihood_exact(int32_t device, int32_t N, int32_t order, int32_t n_terms, const int32_t* term_idx,
                                  const double* init_weight, const double* data_mean, double lambda, double tol, int32_t max_iter,
                                  double* out_weight, double* out_objective /* nullable */,
                                  int32_t* out_iterations /* nullable */, void* stream);

/* ---- sample-sharded mode (SURVEY 8e): histogram rows split over ranks, every rank solves all nodes; per pass
 * the int64 gradient sums and fp64 objective sums are combined with NCCL all-reduces on the solve stream.
 *   rank 0: gml_b200_comm_unique_id(id) -> broadcast the 128 bytes with any transport -> every rank:
 *   gml_b200_comm_init(h, id, rank, world); upload the rank's slice; gml_b200_comm_globalize_histogram(h)
 *   (global M and weights); then solve with opts->reserved[2] = 1.  lambda must be computed from the GLOBAL
 *   sample count (gml_b200_num_samples after the globalize call). */
int gml_b200_comm_unique_id(uint8_t* out128);
int gml_b200_comm_init(gml_b200_handle* h, const uint8_t* id128, int32_t rank, int32_t world);
int gml_b200_comm_globalize_histogram(gml_b200_handle* h);
/* Borrow the communicator of `owner` (same device, same process; `owner` must outlive h's last solve): creating an NCCL
 * communicator costs 0.1-1 s, a process makes ONE and every later histogram / learn() call attaches to it. */
int gml_b200_comm_attach(gml_b200_handle* h, gml_b200_handle* owner);

/* ---- histogram builder (SURVEY 8f-1): replaces the host `countmap` of src/sampling.jl:52-54 -----------------
 * d_samples: M raw samples, int8 spin-major [N x ld] in device memory, N <= 64.  Writes the K distinct
 * configurations to d_out_spins (int8 spin-major, leading dimension ld_out >= K) and their multiplicities to
 * d_out_counts; *out_K receives K.  Rows come out sorted by the bit-packed configuration (bit i = spin i+1 up). */
int gml_b200_build_histogram_device(int32_t device, const int8_t* d_samples, int64_t M, int32_t N, int64_t ld,
                                    int8_t* d_out_spins, int64_t ld_out, double* d_out_counts, int64_t* out_K,
                                    void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GML_B200_H */
