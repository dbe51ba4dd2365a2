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
                                 residual is part of max_residual -- callers that need tol strictly check n_stalled == 0 */
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
