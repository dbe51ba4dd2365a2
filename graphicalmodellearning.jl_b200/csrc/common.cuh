// Shared declarations of libgml_b200: device problem description, error plumbing, launch counting.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <memory>
#include <string>
#include <vector>

#include "../../include/gml_b200.h"

namespace gml {

// ---------------------------------------------------------------------------------------------
// error plumbing (no exceptions across the C ABI: everything funnels into a thread-local string)
// ---------------------------------------------------------------------------------------------
void set_error(const std::string& msg);
struct CudaError { int code; };

#define GML_CUDA(expr)                                                                         \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            ::gml::set_error(std::string(#expr) + " failed: " + cudaGetErrorString(_e) +       \
                             " (" __FILE__ ":" + std::to_string(__LINE__) + ")");              \
            throw ::gml::CudaError{GML_B200_ECUDA};                                            \
        }                                                                                      \
    } while (0)

#define GML_REQUIRE(cond, msg)                                                                 \
    do {                                                                                       \
        if (!(cond)) {                                                                         \
            ::gml::set_error(std::string(msg));                                                \
            throw ::gml::CudaError{GML_B200_EINVAL};                                           \
        }                                                                                      \
    } while (0)

extern thread_local int64_t g_launches;   // kernels launched by the current call
#define GML_LAUNCHED()                                                                         \
    do { ++::gml::g_launches; GML_CUDA(cudaGetLastError()); } while (0)

// Device buffers come from the device's stream-ordered memory pool (retention threshold raised once per device
// by pool_init): after the first solve the multi-GB work buffers of a solve are re-used instead of being mapped
// and unmapped by cudaMalloc / cudaFree on every call.  Frees are issued only after the solve stream has been
// synchronised (all entry points synchronise before their buffers go out of scope).
void pool_init();
template <class T> struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    void alloc(size_t count) {
        if (count <= n && p) return;
        release();
        pool_init();
        GML_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&p), count * sizeof(T), cudaStreamLegacy));
        GML_CUDA(cudaStreamSynchronize(cudaStreamLegacy));
        n = count;
    }
    void release() { if (p) cudaFreeAsync(p, cudaStreamLegacy); p = nullptr; n = 0; }
    ~DevBuf() { release(); }
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
};

static inline int64_t round_up(int64_t a, int64_t b) { return (a + b - 1) / b * b; }
static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// penalty classes of a (node, feature) coordinate
enum : uint8_t { PEN_FREE = 0, PEN_L1 = 1, PEN_ZERO = 2 };

constexpr int KPAD = 128;   // sample padding (rows of the histogram)
constexpr int FPAD = 128;   // feature padding

// ---------------------------------------------------------------------------------------------
// Resident histogram.
//   base  : int8 [Fb x Kp], feature-major (sample-contiguous), Fb = round_up(N+1, FPAD).
//           Row i < N is spin i (the reference's samples[:,1+i]), row N is the constant 1 (its
//           coefficient is the local field), rows > N are 0.  Padded samples (k >= K) hold +1 and
//           carry weight 0.  This is the pairwise feature matrix [S | 1] itself.
//   mb    : int8 [mb_Fp x Kp] multibody base-feature matrix (products of spins), built on demand.
//   P     : int8 [Kp x Fp] sample-major (feature-contiguous) copy of the active feature matrix,
//           built on demand for the tensor path.
// ---------------------------------------------------------------------------------------------
struct Histogram {
    int64_t K = 0, Kp = 0;
    int32_t N = 0;           // spins
    int32_t Fb = 0;          // padded rows of `base`
    double M = 0.0;          // sum of counts (num_samples of data_info); global after comm_globalize_histogram
    double M_local = 0.0;    // this rank's share in sample-sharded mode (0 = not sharded)
    double K_total = 0.0;    // histogram rows over all ranks (= K unless sample-sharded)
    double wmax = 0.0;       // max_k c_k / M
    DevBuf<int8_t> base;
    DevBuf<double> counts;   // [K] c_k as uploaded (the data moments sum them exactly)
    DevBuf<double> w64;      // [Kp] c_k / M
    DevBuf<float> w32;       // [Kp]
    int32_t mb_order = 0, mb_F = 0, mb_Fp = 0;
    DevBuf<int8_t> mb;
    DevBuf<int8_t> P;        // transposed copy of whichever feature matrix was last requested
    const int8_t* P_of = nullptr;
    DevBuf<int8_t> Qb;       // sample-blocked copy [Kp/128][Fp][128] of the same matrix (tile-contiguous for TMA)
    const int8_t* Qb_of = nullptr;
};

// One batched solve: Nn node problems over a shared +-1 feature matrix Q [Fp x Kp].
//   minimise over x_u:  sum_k w_k g( s_u[k] * sum_f Q[f,k] x_u[f] ) + lambda * sum_{pen==L1} |x_u[f]|
struct Comm;

struct NodeProblem {
    Histogram* hist = nullptr;
    Comm* comm = nullptr;           // sample-sharded mode: partial sums are all-reduced over this communicator
    const int8_t* Q = nullptr;      // feature matrix (hist->base or hist->mb)
    int32_t F = 0, Fp = 0;
    int32_t form = 0;
    double lambda = 0.0;
    int32_t Nn = 0;                 // nodes in this shard
    DevBuf<int32_t> spin_row;       // [Nn] row of hist->base that holds s_u
    DevBuf<uint8_t> pen;            // [Nn x Fp] penalty class per coordinate (padded features = PEN_ZERO)
    const double* x0 = nullptr;     // optional warm start [Nn x Fp] (e.g. the previous point of a lambda path)
    // Reduced-space problems (support polish): node u's feature f is row feat[u * Fp + f] of Q instead of row f
    // (Newton solver only; nullptr = the shared feature order).
    const int32_t* feat = nullptr;
};

struct SolveResult {
    double profile[4] = {0, 0, 0, 0};
    double fg_units = -1.0, f_units = -1.0;   // passes weighted by the fraction of the histogram they swept (< 0: use n_fg / n_f)
    DevBuf<double> x;         // [Nn x Fp]
    DevBuf<double> objective; // [Nn]  f_u(x) + lambda*|x_pen|_1
    int iterations = 0, n_fg = 0, n_f = 0, n_unconverged = 0;
    int n_stalled = 0;        // nodes accepted at the gradient noise floor with tol < residual <= 10 tol
    int n_out_of_range = 0;   // nodes re-solved by the CUDA-core backend because they left the fixed-point range
    int n_unpolished = 0;     // support polish: nodes whose support exceeded the reduced solver's NEWTON_MAX_F = 128 features (FISTA point kept)
    DevBuf<double> grad;      // [Nn x Fp] gradient of the smooth part at x (filled by solve_fista when want_grad_at_x)
    bool want_grad_at_x = false;
    bool want_objective = true;   // false: the FISTA driver skips the final objective pass (`objective` is then not filled)
    double max_residual = 0.0;
};

// --- pack.cu
void hist_from_device(Histogram& h, const double* d_counts, const int8_t* d_spins, int64_t K, int32_t N,
                      int64_t ld, cudaStream_t st);
// multibody base features: all subsets of size <= order-1 of the N spins (subset {} = constant).
// h_subsets: [F x (order-1)] 0-based spin ids, -1 padded.
void build_multibody_features(Histogram& h, int order, const std::vector<int32_t>& h_subsets, int F,
                              cudaStream_t st);
// sample-major copy [Kp x Fp] of Q [Fp x Kp] (cached in h.P)
const int8_t* ensure_P(Histogram& h, const int8_t* Q, int Fp, cudaStream_t st);
// sample-blocked copy [Kp/128][Fp][128] of Q [Fp x Kp] (cached in h.Qb): every 128-sample tile is contiguous
const int8_t* ensure_Qb(Histogram& h, const int8_t* Q, int Fp, cudaStream_t st);
// sum of w over the samples of every `stride`-th 128-sample block
double subsample_weight(const Histogram& h, int64_t stride, cudaStream_t st);
void launch_block_copy(const int8_t* Q, int8_t* Qb, int Fp, int64_t Kp, cudaStream_t st);

// --- ingest.cu : K x (N+1) matrix of Real (the reference's `samples`) -> device rows, narrowed on the host by a thread pool
void ingest_matrix(const void* samples, int dtype, int64_t ld, int64_t k0, int64_t K, int32_t N, int8_t* d_base, int64_t Kp,
                   double* d_counts, int n_threads, double* out_host_ms);

// --- newton.cu : fp64 proximal-Newton / barrier-Newton for small feature counts
constexpr int NEWTON_MAX_F = 128;    // feature limit of the fp64 Newton solver (dense F x F Hessian per node in shared memory)
constexpr int NEWTON_AUTO_F = 64;    // solver = AUTO takes the Newton solver up to this many features, FISTA beyond
void solve_newton(const NodeProblem& p, const gml_b200_opts& o, SolveResult& r, cudaStream_t st);

// --- polish.cu : reduced-space Newton polish of a FISTA solution on its identified support (exact or barrier point)
void polish_on_support(const NodeProblem& p, const gml_b200_opts& o, SolveResult& r, cudaStream_t st);

// --- fista.cu : batched FISTA driver over an evaluation backend
void solve_fista(const NodeProblem& p, const gml_b200_opts& o, int backend, SolveResult& r, cudaStream_t st);

// --- warmstart.cu : mean-field starting point of a full pairwise solve from its first-pass gradient (opt-in)
bool meanfield_start(const double* G0, int N, int Fp, const uint8_t* pen, double xmax, double lattice, double* x0, cudaStream_t st);

// --- evaluation backends (objective / gradient passes over the histogram)
struct EvalBackend {
    virtual ~EvalBackend() {}
    // Evaluate at point x [Nn x Fp] (double).  f_out[Nn] receives the smooth objective, g_out
    // [Nn x Fp] its gradient when want_grad.  lattice() > 0 means x must lie on that grid.
    virtual void eval(const double* x, bool want_grad, double* f_out, double* g_out, cudaStream_t st) = 0;
    virtual double lattice() const { return 0.0; }
    // largest |x| the backend can represent at the current precision level (0 = unbounded)
    virtual double x_range() const { return 0.0; }
    // precision level of the following passes: 0 = coarse (cheaper, coarser lattice), 1 = fine.  Returns
    // whether the requested level was taken (backends without levels always run fine).
    virtual bool set_level(int lv, cudaStream_t) { return lv == 1; }
    // device word whose bit 1 is raised when the coarse level's range overflowed (nullptr: no such condition);
    // the driver reads it together with its own per-round counters to keep ONE host sync per round
    virtual const int* device_flags() const { return nullptr; }
    virtual void note_coarse_overflow() {}
    // estimated absolute noise of one gradient component at the current precision level (per unit weight mass)
    virtual double grad_noise() const { return 5e-6; }
    // optional per-kernel device timing (opts.reserved[0] != 0): out[0] = energy-kernel ms (full passes),
    // out[1] = gradient-kernel ms, out[2] = energy-kernel ms (objective-only passes), out[3] = number of timed full passes
    // (only launches that sweep the whole histogram are timed)
    // Restrict the passes to every `stride`-th block of 128 samples; returns the weight mass rho of the
    // subset (sum of w over the used samples), or a negative value when the backend cannot subsample.
    virtual double set_subsample(int64_t /*stride*/, cudaStream_t) { return -1.0; }
    // Restrict the following passes to the nodes d_idx[0..n) (device array, entries < 0 = empty slot); nullptr = the
    // whole shard.  Outputs of nodes outside the list are left untouched.  Returns false when the backend always
    // evaluates every node (the call is then a no-op).
    virtual bool set_active(const int* /*d_idx*/, int /*n*/, cudaStream_t) { return false; }
    virtual void set_profiling(bool) {}
    virtual void collect_profile(double* /*out4*/) {}
};
EvalBackend* make_backend_cc(const NodeProblem& p, cudaStream_t st);
EvalBackend* make_backend_tc(const NodeProblem& p, cudaStream_t st);

// --- histogram.cu : raw samples -> deduplicated histogram (returns the number of distinct configurations)
int64_t build_histogram(const int8_t* d_samples, int64_t M, int N, int64_t ld, int8_t* d_out_spins, int64_t ld_out,
                        double* d_out_counts, cudaStream_t st);
// The tail of build_histogram, for callers that produce the 64-bit configuration keys (bit i = spin i+1 up) themselves:
// sort_key_runs sorts M < 2^31 keys of N bits and run-length encodes them (runs.K distinct keys, increasing);
// unpack_key_runs writes the runs as histogram rows [counts, spins] at rows [0, runs.K) of the output.
struct KeyRuns {
    DevBuf<unsigned long long> uniq;
    DevBuf<int> run_len;
    int64_t K = 0;
};
void sort_key_runs(const unsigned long long* d_keys, int64_t M, int N, KeyRuns& runs, cudaStream_t st);
void unpack_key_runs(const KeyRuns& runs, int N, int8_t* d_out_spins, int64_t ld_out, double* d_out_counts, cudaStream_t st);

// --- comm.cu : NCCL plumbing of the sample-sharded mode
void comm_unique_id(uint8_t* out128);
Comm* comm_create(const uint8_t* id128, int rank, int world);
void comm_destroy(Comm* c);
void comm_group_start(Comm* c);
void comm_group_end(Comm* c);
void comm_allreduce_sum_i64(Comm* c, long long* buf, size_t n, cudaStream_t st);
void comm_allreduce_sum_f64(Comm* c, double* buf, size_t n, cudaStream_t st);
void comm_allreduce_max_f64(Comm* c, double* buf, size_t n, cudaStream_t st);
void comm_globalize_histogram(Comm* c, Histogram& h, cudaStream_t st);
int comm_agree_max(Comm* c, int value, cudaStream_t st);

// --- sampler.cu
void sample_gibbs(int N, const int32_t* d_row_ptr, const int32_t* d_col, const float* d_J, const float* d_h,
                  int max_deg, int64_t n_samples, int sweeps, uint64_t seed, int8_t* d_spins, int64_t ld,
                  cudaStream_t st);

void sample_gibbs_terms(int N, int width, const int32_t* d_row_ptr, const int32_t* d_others, const float* d_weight,
                        int64_t n_samples, int sweeps, uint64_t seed, int8_t* d_spins, int64_t ld, cudaStream_t st);

// Per-site incidence lists (CSR) of a term list term_idx [n_terms x order] (0-based spin ids, negative = padding):
// entry q in [row_ptr[i], row_ptr[i+1]) of site i is term term[q], with its width = max(1, order-1) other members in
// others[q*width ..] (-1 padded).  Refuses an index >= N or a spin repeated in a term.  With no entries, one padding
// entry (term -1) keeps the arrays non-empty.
struct Incidence {
    int width = 1;
    std::vector<int32_t> row_ptr, others, term;
};
Incidence build_incidence(int N, int order, int n_terms, const int32_t* term_idx);

// --- mcmc_sampler.cu : multi-sample Gibbs sampler (one warp = 32 chains, state in shared memory) and its replica-exchange
// form (betas.size() = R > 1 rungs: a ladder of R lanes per chain, only rung 0 = betas[0] = 1 records); fills out_K and
// out_rhat (nullable, [replicates][2]: split-R-hat of the energy and of the magnetisation), out_swap_rate (nullable, R > 1,
// [replicates][R-1]: accepted / proposed swaps of each adjacent pair after burn_in) and, when d_counts is set, the
// replicates' rows at consecutive rows: N <= 64 deduplicated histograms, N > 64 one row per draw.
// N <= GML_B200_MCMC_MAX_N; term weights are rounded once to fp32.
constexpr int64_t MCMC_AUTO_CHAINS = 1 << 17;
constexpr int TEMPERING_MAX_RUNGS = GML_B200_TEMPERING_MAX_RUNGS;
int64_t mcmc_auto_chains(int64_t n_samples, int rungs);
// The bond list of the Swendsen-Wang sampler (cluster_kernel): per term of one or two spins with a nonzero weight, its
// nodes (node 0 = the ghost spin, node i + 1 = spin i) and sign, and q_t = e^{-2|w_t|} in units of 2^-64.  Refuses a term
// of three or more spins.
struct ClusterBonds {
    std::vector<uint32_t> ends;
    std::vector<unsigned long long> q;
};
ClusterBonds cluster_bonds(int order, const std::vector<int32_t>& term_idx, const std::vector<double>& term_weight);
// bonds != nullptr (betas = {1}): Swendsen-Wang updates instead of Gibbs sweeps, with the same records and outputs
void sample_mcmc(int N, int order, const std::vector<int32_t>& term_idx, const std::vector<double>& term_weight,
                 const Incidence& inc, const std::vector<double>& betas, int64_t n_samples, int replicates, int64_t chains,
                 int64_t burn_in, int64_t thin, uint64_t seed, int64_t* out_K, double* out_rhat, double* out_swap_rate,
                 double* d_counts, int8_t* d_spins, int64_t ld, cudaStream_t st, const ClusterBonds* bonds = nullptr);
// log Z of the model by bridge sampling along a replica-exchange ladder betas[0] = 1 > ... > betas[R-1] = 0 (R > 1):
// `chains` ladders, burn_in sweeps, then `sweeps` sweeps that feed the bridge sums; fills *out_log_z and the nullable
// out_stderr, out_log_ratio [R-1][2] (estimate, stderr of log Z_k - log Z_{k+1}) and out_swap_rate [R-1].  chains >= 2.
void log_partition_tempering(int N, int order, const std::vector<int32_t>& term_idx, const std::vector<double>& term_weight,
                             const Incidence& inc, const std::vector<double>& betas, int64_t chains, int64_t burn_in,
                             int64_t sweeps, uint64_t seed, double* out_log_z, double* out_stderr, double* out_log_ratio,
                             double* out_swap_rate, cudaStream_t st);

// Persistent Gibbs chains (PERSIST instantiation of mcmc_kernel, fit_likelihood): `chains` chains of the model with
// fp32 weights in the device buffers term_w [n_terms] and weight [incidence entries], which a caller may rewrite between
// launches.  run(sweep0, k) advances every chain by sweeps sweep0 + 1 .. sweep0 + k of one long run (sweep0 = 0: from the
// random start of sweep 0) and leaves the final state in `record`, a record buffer [(N+1) x warps] of one record (the
// layout reduce_records reads, the live lanes as draws); it is also the state the next launch resumes from.
struct PersistentChains {
    struct Impl;
    std::unique_ptr<Impl> impl;
    int64_t warps = 0;
    const uint32_t* record = nullptr;
    float* term_w = nullptr;
    float* weight = nullptr;
    PersistentChains(int N, int order, const std::vector<int32_t>& term_idx, const std::vector<double>& term_weight,
                     const Incidence& inc, int64_t chains, uint64_t seed, cudaStream_t st);
    ~PersistentChains();
    void run(int64_t sweep0, int64_t sweeps, cudaStream_t st);
};

// --- moments.cu : moments <prod_{i in t} s_i> of keys t.  pairwise: all <s_i> (diagonal) and <s_i s_j> as an N x N
// row-major matrix; otherwise n_keys keys of `order` 0-based spins, -1 padded ([n_keys x order]).
struct MomentKeys {
    bool pairwise = false;
    int order = 0, n_keys = 0;
    std::vector<int32_t> idx;
};
int64_t moment_outputs(const MomentKeys& keys, int N);
// mean and stderr (nullable) of the keys over the draws of a record buffer of mcmc_kernel's RECORD mode
void reduce_records(const uint32_t* rec, int N, int64_t records, int64_t warps, const MomentKeys& keys, double* out_mean,
                    double* out_stderr, cudaStream_t st);
// the integer sums behind reduce_records' key-list means, left on the device: n_g [G] draws and S [G x n_keys] key sums
// of the G = record_groups(warps) groups of warps (d_key_idx [n_keys x order] on the device)
int record_groups(int64_t warps);
void record_key_sums(const uint32_t* rec, int N, int64_t records, int64_t warps, int order, int n_keys, const int32_t* d_key_idx,
                     long long* d_n_g, long long* d_S, cudaStream_t st);
// key-list moments of a resident histogram: sum_k c_k prod s / M
void moments_histogram_keys(const Histogram& hist, const MomentKeys& keys, double* out_mean, cudaStream_t st);
// The moments over exactly the n_samples draws that sample_mcmc(..., replicates = 1, ...) returns with the same arguments,
// with their standard errors over G = min(32, warps) groups of warps, out_rhat [2] and out_swap_rate [R-1] as sample_mcmc.
void moments_mcmc(int N, int order, const std::vector<int32_t>& term_idx, const std::vector<double>& term_weight,
                  const Incidence& inc, const std::vector<double>& betas, int64_t n_samples, int64_t chains, int64_t burn_in,
                  int64_t thin, uint64_t seed, const MomentKeys& keys, double* out_mean, double* out_stderr, double* out_rhat,
                  double* out_swap_rate, cudaStream_t st, const ClusterBonds* bonds = nullptr);

// --- likelihood.cu : maximum-likelihood refit of the weights of a term list from data moments data_mean (fit_likelihood).
// penalised[t] = 1 marks the terms of >= 2 spins, which carry lambda |w_t|.
constexpr double FISHER_FLOOR = 1e-2;    // floor of the diagonal preconditioner 1 - m^_t^2 of the MCMC steps
constexpr double FIT_STEP_S0 = 100.0;    // eta_s = eta_0 (1 + s / FIT_STEP_S0)^-0.6
double fit_step_size(double eta0, int64_t s);
// persistent-chain stochastic maximum likelihood; out_weight [n_terms] = the Polyak-Ruppert mean over steps >= steps / 2,
// out_model_moments (nullable) [n_terms] = the chains' mean moments over the same steps, out_trace (nullable) [steps]
void fit_likelihood_mcmc(int N, int order, const std::vector<int32_t>& term_idx, const std::vector<double>& init_weight,
                         const Incidence& inc, const std::vector<double>& data_mean, const std::vector<uint8_t>& penalised,
                         double lambda, int64_t chains, int64_t burn_in, int64_t thin, int64_t steps, double eta0, uint64_t seed,
                         double* out_weight, double* out_model_moments, double* out_trace, cudaStream_t st);
// FISTA on the exact objective (term t = spins of masks[t]); false when the prox-gradient mapping did not reach tol
bool fit_likelihood_exact(int N, const std::vector<uint64_t>& masks, const std::vector<double>& init_weight,
                          const std::vector<double>& data_mean, const std::vector<uint8_t>& penalised, double lambda, double tol,
                          int max_iter, double* out_weight, double* out_objective, int* out_iterations, cudaStream_t st);

// --- exact_sampler.cu : iid draws from the exact distribution by enumeration (term t = spins of masks[t]); fills
// out_K[replicates] and, when d_counts is set, the histograms at consecutive rows; returns log Z.  N <= GML_B200_EXACT_MAX_N.
double sample_exact(int N, const std::vector<uint64_t>& masks, const std::vector<double>& weights, int64_t n_samples,
                    int replicates, uint64_t seed, int64_t* out_K, double* d_counts, int8_t* d_spins, int64_t ld,
                    cudaStream_t st);
// exact moments of the keys (masks over spins 0..N-1; out_mean[keys]) by enumeration, N <= GML_B200_EXACT_MAX_N, and
// (nullable out_log_z) log Z from the same pass
void moments_exact(int N, const std::vector<uint64_t>& masks, const std::vector<double>& weights,
                   const std::vector<uint64_t>& key_masks, double* out_mean, cudaStream_t st, double* out_log_z = nullptr);

}  // namespace gml
