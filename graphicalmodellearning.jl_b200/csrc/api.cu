// C ABI of libgml_b200 (see include/gml_b200.h): handle management, problem set-up, solver dispatch,
// row placement / symmetrisation (src/GraphicalModelLearning.jl:181-186) and result transfer.
#include "common.cuh"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <thread>
#include <tuple>

namespace gml {

thread_local std::string g_error;
thread_local int64_t g_launches = 0;
void set_error(const std::string& msg) { g_error = msg; }

void pool_init() {
    static thread_local int done_for = -1;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev == done_for) return;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        unsigned long long keep = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    done_for = dev;
}

namespace {

double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

struct EventTimer {
    cudaEvent_t a = nullptr, b = nullptr;
    cudaStream_t st;
    explicit EventTimer(cudaStream_t s) : st(s) {
        GML_CUDA(cudaEventCreate(&a)); GML_CUDA(cudaEventCreate(&b));
        GML_CUDA(cudaEventRecord(a, st));
    }
    double stop() {
        float ms = 0.f;
        GML_CUDA(cudaEventRecord(b, st));
        GML_CUDA(cudaEventSynchronize(b));
        GML_CUDA(cudaEventElapsedTime(&ms, a, b));
        return ms;
    }
    ~EventTimer() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
};

// pairwise penalty classes (:171): coupling to itself does not exist, the field is free
__global__ void pairwise_setup_kernel(int N, int Fp, int node_begin, int Nn, int32_t* spin_row, uint8_t* pen) {
    const int u = blockIdx.x;
    if (threadIdx.x == 0) spin_row[u] = node_begin + u;
    for (int f = threadIdx.x; f < Fp; f += blockDim.x) {
        uint8_t c = PEN_ZERO;
        if (f < N) c = (f == node_begin + u) ? PEN_ZERO : PEN_L1;
        else if (f == N) c = PEN_FREE;
        pen[(int64_t)u * Fp + f] = c;
    }
}

// reconstruction[u, 1:N] = value.(x) (:181): coupling columns, field on the diagonal
__global__ void pairwise_rows_kernel(const double* __restrict__ x, int N, int Fp, int node_begin, double* __restrict__ rows) {
    const int u = blockIdx.x;
    for (int i = threadIdx.x; i < N; i += blockDim.x)
        rows[(int64_t)u * N + i] = (i == node_begin + u) ? x[(int64_t)u * Fp + N] : x[(int64_t)u * Fp + i];
}

__global__ void symmetrize_kernel(double* __restrict__ m, int N) {
    const int i = blockIdx.y * blockDim.y + threadIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N && j < N && j > i) {
        const double v = 0.5 * (m[(int64_t)i * N + j] + m[(int64_t)j * N + i]);   // 0.5*(R + R') (:185)
        m[(int64_t)i * N + j] = v; m[(int64_t)j * N + i] = v;
    }
}

__global__ void multibody_setup_kernel(int Fp, int n_keys, const int32_t* __restrict__ key_map, int32_t* spin_row, uint8_t* pen) {
    const int u = blockIdx.x;
    if (threadIdx.x == 0) spin_row[u] = u;
    for (int f = threadIdx.x; f < Fp; f += blockDim.x) pen[(int64_t)u * Fp + f] = PEN_ZERO;
    __syncthreads();
    for (int f = threadIdx.x; f < n_keys; f += blockDim.x)
        pen[(int64_t)u * Fp + key_map[(int64_t)u * n_keys + f]] = (f == 0) ? PEN_FREE : PEN_L1;   // length-1 key is free (:118)
}

__global__ void multibody_gather_kernel(const double* __restrict__ x, int Fp, int n_keys, const int32_t* __restrict__ key_map,
                                        double* __restrict__ vals) {
    const int u = blockIdx.x;
    for (int f = threadIdx.x; f < n_keys; f += blockDim.x)
        vals[(int64_t)u * n_keys + f] = x[(int64_t)u * Fp + key_map[(int64_t)u * n_keys + f]];
}

// multiRISE symmetrisation on the device (src/GraphicalModelLearning.jl:135-149): thread i owns the i-th SORTED key S
// (subsets of [N] of size 1..order, by size then lexicographic) and averages the |S| per-node estimates -- node u in S
// holds its value for (u, S \ {u}) at base feature index(S \ {u}) of row u (base features are the subsets of size
// <= order-1 in the same enumeration).  binom: (N+1) x (order+1) table; size_off[q] = first key / feature of size q.
__device__ __forceinline__ long long comb_rank(const int* c, int r, int N, const long long* binom, int W) {
    long long rank = 0;
    int prev = -1;
    for (int i = 0; i < r; ++i) {
        for (int v = prev + 1; v < c[i]; ++v) rank += binom[(N - 1 - v) * W + (r - 1 - i)];
        prev = c[i];
    }
    return rank;
}
__global__ void multibody_symmetrize_kernel(const double* __restrict__ x, int N, int Fp, int order, const long long* __restrict__ binom,
                                            const long long* __restrict__ key_off /* [order+2] by key size */,
                                            const long long* __restrict__ feat_off /* [order+1] by feature size */,
                                            long long n_sym, double* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_sym) return;
    const int W = order + 1;
    int q = 1;
    while (q < order && i >= key_off[q + 1]) ++q;
    long long rem = i - key_off[q];
    int mem[8];
    int v = 0;
    for (int j = 0; j < q; ++j) {             // unrank the combination
        for (;; ++v) {
            const long long cnt = binom[(N - 1 - v) * W + (q - 1 - j)];
            if (rem < cnt) break;
            rem -= cnt;
        }
        mem[j] = v++;
    }
    double acc = 0.0;
    for (int j = 0; j < q; ++j) {
        int t[8];
        int r = 0;
        for (int m = 0; m < q; ++m) if (m != j) t[r++] = mem[m];
        const long long f = feat_off[q - 1] + comb_rank(t, q - 1, N, binom, W);
        acc += x[(long long)mem[j] * Fp + f];
    }
    out[i] = acc / q;
}

int64_t binom(int n, int k) {
    if (k < 0 || k > n) return 0;
    long double r = 1;
    for (int i = 1; i <= k; ++i) r = r * (n - k + i) / i;
    return (int64_t)llround((double)r);
}

void fill_opts(gml_b200_opts& o, const gml_b200_opts* in) {
    gml_b200_opts_default(&o);
    if (in) o = *in;
}

int pick_solver(const gml_b200_opts& o, int F) {
    int s = o.solver;
    // AUTO: the fp64 Newton solver for small problems; the Ipopt-compatible barrier point needs it (up to 128 features)
    if (s == GML_B200_SOLVER_AUTO)
        s = (F <= NEWTON_AUTO_F || (o.barrier_mu > 0.0 && F <= NEWTON_MAX_F)) ? GML_B200_SOLVER_NEWTON : GML_B200_SOLVER_FISTA_TC;
    GML_REQUIRE(s >= GML_B200_SOLVER_NEWTON && s <= GML_B200_SOLVER_FISTA_TC, "unknown solver id");
    GML_REQUIRE(s != GML_B200_SOLVER_NEWTON || F <= NEWTON_MAX_F, "Newton solver needs <= 128 features per node");
    GML_REQUIRE(o.barrier_mu == 0.0 || s == GML_B200_SOLVER_NEWTON,
                "barrier_mu (Ipopt-compatible mode) is only available with the Newton solver (<= 128 features per node); "
                "beyond that use the exact minimiser, optionally with the support polish (opts.reserved[7] & 2)");
    return s;
}

void run_solver(const NodeProblem& p, const gml_b200_opts& o, SolveResult& r, int& solver_used, cudaStream_t st) {
    solver_used = pick_solver(o, p.F);
    if (solver_used == GML_B200_SOLVER_NEWTON) { solve_newton(p, o, r, st); return; }
    const bool polish = (o.reserved[7] & 2) != 0;       // FISTA to tol, then reduced-space Newton on the support
    r.want_grad_at_x = polish;
    solve_fista(p, o, solver_used, r, st);
    if (polish && r.n_unconverged == 0) polish_on_support(p, o, r, st);
}

}  // namespace
}  // namespace gml

using namespace gml;

struct gml_b200_handle {
    int device = 0;
    cudaStream_t own_stream = nullptr;
    Histogram hist;
    bool has_hist = false;
    Comm* comm = nullptr;      // sample-sharded mode
    bool owns_comm = false;    // false: borrowed from another handle (gml_b200_comm_attach)
};

namespace {

cudaStream_t stream_of(gml_b200_handle* h, const gml_b200_opts& o) {
    return o.stream ? (cudaStream_t)o.stream : h->own_stream;
}

template <class Fn> int guarded(Fn&& fn) {
    try {
        fn();
        return GML_B200_OK;
    } catch (const CudaError& e) {
        return e.code;
    } catch (const std::exception& e) {
        set_error(std::string("internal error: ") + e.what());
        return GML_B200_ECUDA;
    }
}

void finish_stats(gml_b200_stats* stats, const SolveResult& r, int solver_used, int Nn, int64_t K, double solve_ms,
                  double d2h_ms, double t0) {
    if (!stats) return;
    stats->solver_used = solver_used;
    stats->iterations = r.iterations;
    stats->n_fg_passes = r.n_fg;
    stats->n_f_passes = r.n_f;
    stats->n_unconverged = r.n_unconverged;
    stats->n_stalled = r.n_stalled;
    stats->kernel_launches = g_launches;
    const double fg = r.fg_units >= 0.0 ? r.fg_units : r.n_fg, fo = r.f_units >= 0.0 ? r.f_units : r.n_f;
    stats->evals = (double)Nn * (double)K * (fg + 0.5 * fo);
    stats->solve_ms = solve_ms;
    stats->d2h_ms = d2h_ms;
    stats->total_ms += now_ms() - t0;
    stats->max_residual = r.max_residual;
    for (int i = 0; i < 4; ++i) stats->reserved_d[i] = r.profile[i];
}

// Runs fill(counts, spins) on the output buffers of a sampler entry point: device buffers as they are; host buffers through
// device staging buffers, of which the first sum(out_K) rows are copied back; null buffers (a count-only call) as null.
template <class Fill> void into_sample_buffers(double* d_counts, int8_t* d_spins, int64_t ld, int N, int replicates,
                                               const int64_t* out_K, cudaStream_t st, Fill&& fill) {
    cudaPointerAttributes attr{};
    const bool on_host = d_counts && (cudaPointerGetAttributes(&attr, d_counts) != cudaSuccess ||
                                      (attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged));
    cudaGetLastError();   // an unregistered host pointer may leave an error behind
    DevBuf<double> stage_c;
    DevBuf<int8_t> stage_s;
    if (on_host) { stage_c.alloc(ld); stage_s.alloc((size_t)N * ld); }
    fill(on_host ? stage_c.p : d_counts, on_host ? stage_s.p : d_spins);
    if (on_host) {
        int64_t rows = 0;
        for (int r = 0; r < replicates; ++r) rows += out_K[r];
        GML_CUDA(cudaMemcpyAsync(d_counts, stage_c.p, sizeof(double) * rows, cudaMemcpyDeviceToHost, st));
        GML_CUDA(cudaMemcpy2DAsync(d_spins, ld, stage_s.p, ld, rows, N, cudaMemcpyDeviceToHost, st));
        GML_CUDA(cudaStreamSynchronize(st));
    }
}

// The MCMC entry points (betas = {1}: gml_b200_sample_mcmc_device; R > 1 rungs: gml_b200_sample_tempering_device, whose
// ladder the caller has checked): argument checks, then the sampler into the caller's buffers.
void run_mcmc(int32_t device, int32_t N, int32_t order, int32_t n_terms, const int32_t* term_idx, const double* term_weight,
              const std::vector<double>& betas, int64_t n_samples, int32_t replicates, int64_t chains, int32_t burn_in,
              int32_t thin, uint64_t seed, int64_t* out_K, double* out_rhat, double* out_swap_rate, double* d_counts,
              int8_t* d_spins, int64_t ld, void* stream) {
    GML_REQUIRE(N >= 1 && N <= GML_B200_MCMC_MAX_N, "MCMC sampler needs 1 <= N <= " + std::to_string(GML_B200_MCMC_MAX_N));
    GML_REQUIRE(order >= 1 && order <= 8 && n_terms >= 0 && (n_terms == 0 || (term_idx && term_weight)) && out_K,
                "bad sampler argument");
    GML_REQUIRE(n_samples >= 1 && replicates >= 1 && chains >= 0 && chains <= (INT64_C(1) << 31) && burn_in >= 0 && thin >= 1,
                "bad sampler sizes");
    GML_REQUIRE(N > 64 || n_samples < (INT64_C(1) << 31), "the histogram of N <= 64 spins takes fewer than 2^31 draws per replicate");
    GML_REQUIRE(!d_counts || (d_spins && ld >= 1), "d_counts needs d_spins and ld >= 1");
    const int rungs = (int)betas.size();
    if (chains == 0) chains = mcmc_auto_chains(n_samples, rungs);
    const double steps = ((double)burn_in + (double)thin * (double)ceil_div(n_samples, chains)) * N;
    GML_REQUIRE(steps * replicates < 0x1.0p62, "too many sweeps");
    std::vector<int32_t> idx(term_idx, term_idx + (size_t)n_terms * order);
    std::vector<double> weights(term_weight, term_weight + n_terms);
    for (int t = 0; t < n_terms; ++t) {
        for (int m = 0; m < order; ++m) GML_REQUIRE(idx[(size_t)t * order + m] >= -1, "sampler term refers to a spin outside [0, N)");
        GML_REQUIRE(std::isfinite(weights[t]), "sampler term weight is not finite");
    }
    const Incidence inc = build_incidence(N, order, n_terms, idx.data());
    if (N > 64 && d_counts && ld < n_samples * replicates) {
        for (int r = 0; r < replicates; ++r) out_K[r] = n_samples;
        GML_REQUIRE(false, "ld = " + std::to_string(ld) + " is smaller than the " + std::to_string(n_samples * replicates) +
                           " rows of the replicates (out_K holds their sizes)");
    }
    GML_CUDA(cudaSetDevice(device));
    cudaStream_t st = (cudaStream_t)stream;
    into_sample_buffers(d_counts, d_spins, ld, N, replicates, out_K, st, [&](double* c, int8_t* sp) {
        sample_mcmc(N, order, idx, weights, inc, betas, n_samples, replicates, chains, burn_in, thin, seed, out_K, out_rhat,
                    out_swap_rate, c, sp, ld, st);
    });
}

void throw_if_unconverged(int n_unconverged) {
    if (n_unconverged == 0) return;
    set_error("solver did not reach tol within max_iter for " + std::to_string(n_unconverged) + " node(s)");
    throw CudaError{GML_B200_ENOTCONV};
}

// 0.5 (R + R') (:185) of the N x N matrix m in place (symmetric in (i, j): row- or column-major alike)
void launch_symmetrize(double* m, int N, cudaStream_t st) {
    dim3 b(32, 8), g((unsigned)ceil_div(N, 32), (unsigned)ceil_div(N, 8));
    symmetrize_kernel<<<g, b, 0, st>>>(m, N);
    GML_LAUNCHED();
}

// rows [Nn x N] of the nodes nb.. into the column-major (Julia-native) N x N matrix `out`
void scatter_rows(const double* rows, int Nn, int N, int nb, double* out) {
    for (int u = 0; u < Nn; ++u)
        for (int i = 0; i < N; ++i) out[(size_t)(nb + u) + (size_t)N * i] = rows[(size_t)u * N + i];
}

// the nodes [nb, ne) a call covers (opts->node_begin / node_end; ne <= 0 = through the last of the N nodes)
std::pair<int, int> node_range(int nb, int ne, int N) {
    if (ne <= 0) ne = N;
    GML_REQUIRE(nb >= 0 && ne <= N && nb < ne, "node shard out of range");
    return {nb, ne};
}

// Node problems [nb, ne) of a pairwise formulation over the resident feature matrix [S | 1] (hist.base), with their
// penalty classes set up on the device.
void pairwise_problem(NodeProblem& p, Histogram& hist, int formulation, double lambda, int nb, int ne, cudaStream_t st) {
    GML_REQUIRE(formulation >= GML_B200_RISE && formulation <= GML_B200_RPLE, "unknown formulation id");
    std::tie(nb, ne) = node_range(nb, ne, hist.N);
    p.hist = &hist; p.Q = hist.base.p; p.F = hist.N + 1; p.Fp = hist.Fb;
    p.form = formulation; p.lambda = lambda; p.Nn = ne - nb;
    p.spin_row.alloc(p.Nn); p.pen.alloc((size_t)p.Nn * p.Fp);
    pairwise_setup_kernel<<<p.Nn, 128, 0, st>>>(hist.N, p.Fp, nb, p.Nn, p.spin_row.p, p.pen.p);
    GML_LAUNCHED();
}

void solve_pairwise_rows_one(gml_b200_handle* h, int formulation, double lambda, const gml_b200_opts& o, int nb, int ne,
                             double* d_rows, double* d_obj, gml_b200_stats* stats, cudaStream_t st, double t0,
                             DevBuf<double>* warm = nullptr /* in: start point (if allocated), out: solution [Nn x Fp] */) {
    Histogram& hist = h->hist;
    const int N = hist.N;
    NodeProblem p;
    if (o.reserved[2] == 1) {
        GML_REQUIRE(h->comm != nullptr, "sample-sharded solve needs gml_b200_comm_init first");
        GML_REQUIRE(hist.M_local > 0.0, "sample-sharded solve needs gml_b200_comm_globalize_histogram after the upload");
        GML_REQUIRE(o.solver == GML_B200_SOLVER_FISTA_TC || (o.solver == GML_B200_SOLVER_AUTO && N + 1 > NEWTON_AUTO_F),
                    "sample-sharded mode is implemented for the tensor-core FISTA solver");
        p.comm = h->comm;
    }
    EventTimer timer(st);
    pairwise_problem(p, hist, formulation, lambda, nb, ne, st);
    SolveResult r;
    // The objective at the returned point costs one more pass over the histogram: only when somebody asked for it.  In a
    // sample-sharded solve that pass contains an all-reduce, so EVERY rank must make the same choice (the callers pass the
    // same arguments on all ranks; the single-process form hands the other devices a scratch buffer when device 0 asks).
    r.want_objective = d_obj != nullptr;
    int solver_used = 0;
    if (warm && warm->p) p.x0 = warm->p;
    run_solver(p, o, r, solver_used, st);
    pairwise_rows_kernel<<<p.Nn, 128, 0, st>>>(r.x.p, N, p.Fp, nb, d_rows);
    GML_LAUNCHED();
    if (d_obj) GML_CUDA(cudaMemcpyAsync(d_obj, r.objective.p, sizeof(double) * p.Nn, cudaMemcpyDeviceToDevice, st));
    if (warm) {
        warm->alloc((size_t)p.Nn * p.Fp);
        GML_CUDA(cudaMemcpyAsync(warm->p, r.x.p, sizeof(double) * p.Nn * p.Fp, cudaMemcpyDeviceToDevice, st));
    }
    const double solve_ms = timer.stop();
    finish_stats(stats, r, solver_used, p.Nn, hist.K, solve_ms, 0.0, t0);
    throw_if_unconverged(r.n_unconverged);
}

// Memory-aware front end: the residual limbs of the tensor-core path take nR * nodes * Kp bytes (31 GB at C3 on one
// GPU).  When a shard would not fit next to the resident histogram copies, its nodes are solved in consecutive
// chunks (node problems are independent, src/GraphicalModelLearning.jl:161) instead of failing with out-of-memory.
void solve_pairwise_rows(gml_b200_handle* h, int formulation, double lambda, const gml_b200_opts& o, int node_begin,
                         int node_end, double* d_rows, double* d_obj, gml_b200_stats* stats, cudaStream_t st, double t0,
                         DevBuf<double>* warm = nullptr) {
    GML_REQUIRE(h->has_hist, "no histogram resident: call gml_b200_upload_histogram first");
    GML_REQUIRE(lambda >= 0.0 && std::isfinite(lambda), "lambda must be finite and >= 0");
    const Histogram& hist = h->hist;
    const int N = hist.N;
    const auto [nb, ne] = node_range(node_begin, node_end, N);
    const int F = N + 1;
    int solver = pick_solver(o, F);
    int chunk = ne - nb;
    if (solver == GML_B200_SOLVER_FISTA_TC && !warm && o.reserved[2] != 1) {
        size_t free_b = 0, total_b = 0;
        GML_CUDA(cudaMemGetInfo(&free_b, &total_b));
        const double Kp = (double)hist.Kp, Fp = (double)hist.Fb;
        const double resident = 3.0 * Kp * Fp + 12.0 * Kp;                        // base, P, Qb, weights
        double budget = 0.88 * (double)total_b - resident;
        if (const char* env = std::getenv("GML_B200_MEM_BUDGET_GB")) budget = std::atof(env) * 1e9;   // test hook
        auto need = [&](int nn) {                                                 // per-solve buffers for nn nodes
            const double np2 = (double)round_up(nn, 128);
            return 4.0 * np2 * Kp + 8.0 * 8.0 * np2 * Fp + 7.0 * np2 * Fp;         // R (<= 4 limbs), fp64 state + G64, limb tiles
        };
        if (need(chunk) > budget) {
            chunk = (int)((budget - 0.0) / (need(128) / 128.0)) / 128 * 128;
            GML_REQUIRE(chunk >= 128, "histogram too large for one GPU even with node chunking: use more GPUs (node shards) or "
                                      "the sample-sharded mode");
        }
    }
    if (chunk >= ne - nb) {
        solve_pairwise_rows_one(h, formulation, lambda, o, nb, ne, d_rows, d_obj, stats, st, t0, warm);
        return;
    }
    gml_b200_stats acc{}, cur{};
    int unconverged = 0;
    for (int b = nb; b < ne; b += chunk) {
        const int e = std::min(ne, b + chunk);
        std::memset(&cur, 0, sizeof(cur));
        try {
            solve_pairwise_rows_one(h, formulation, lambda, o, b, e, d_rows + (size_t)(b - nb) * N, d_obj ? d_obj + (b - nb) : nullptr,
                                    &cur, st, now_ms());
        } catch (const CudaError& err) {
            if (err.code != GML_B200_ENOTCONV) throw;
        }
        unconverged += cur.n_unconverged;
        acc.n_stalled += cur.n_stalled;
        acc.solver_used = cur.solver_used;
        acc.iterations = std::max(acc.iterations, cur.iterations);
        acc.n_fg_passes += cur.n_fg_passes; acc.n_f_passes += cur.n_f_passes;
        acc.evals += cur.evals; acc.solve_ms += cur.solve_ms;
        acc.max_residual = std::max(acc.max_residual, cur.max_residual);
        for (int i = 0; i < 4; ++i) acc.reserved_d[i] += cur.reserved_d[i];
    }
    acc.n_unconverged = unconverged;
    acc.kernel_launches = g_launches;
    acc.total_ms = now_ms() - t0;
    if (stats) *stats = acc;
    throw_if_unconverged(unconverged);
}

// base features of multiRISE order p: all subsets of [N] of size <= p-1, by size then lexicographic
struct MultibodyLayout {
    int F = 0, n_keys = 0, width = 0;
    std::vector<int32_t> subsets;   // [F x width]
    std::vector<int32_t> key_map;   // [N x n_keys] base-feature index of node u's f-th key
};

MultibodyLayout multibody_layout(int N, int order) {
    MultibodyLayout L;
    L.width = std::max(1, order - 1);
    std::map<std::vector<int>, int> index;
    std::vector<std::vector<int>> all;
    for (int q = 0; q <= order - 1 && q <= N; ++q) {
        std::vector<int> c(q);
        for (int i = 0; i < q; ++i) c[i] = i;
        for (;;) {
            index[c] = (int)all.size();
            all.push_back(c);
            int i = q - 1;
            while (i >= 0 && c[i] == N - q + i) --i;
            if (i < 0) break;
            ++c[i];
            for (int j = i + 1; j < q; ++j) c[j] = c[j - 1] + 1;
        }
    }
    L.F = (int)all.size();
    L.subsets.assign((size_t)L.F * L.width, -1);
    for (int f = 0; f < L.F; ++f)
        for (size_t j = 0; j < all[f].size(); ++j) L.subsets[(size_t)f * L.width + j] = all[f][j];
    // node keys in the reference's order (:94-104): (u,), (u, comb of neighbours of size 1), size 2, ...
    for (int u = 0; u < N; ++u) {
        int count = 0;
        for (int q = 0; q <= order - 1 && q <= N - 1; ++q) {
            std::vector<int> c(q);   // combination over the N-1 neighbours, mapped to spin ids
            for (int i = 0; i < q; ++i) c[i] = i;
            for (;;) {
                std::vector<int> ids(q);
                for (int i = 0; i < q; ++i) ids[i] = c[i] < u ? c[i] : c[i] + 1;
                L.key_map.push_back(index[ids]);
                ++count;
                int i = q - 1;
                while (i >= 0 && c[i] == (N - 1) - q + i) --i;
                if (i < 0) break;
                ++c[i];
                for (int j = i + 1; j < q; ++j) c[j] = c[j - 1] + 1;
            }
        }
        L.n_keys = count;
    }
    return L;
}

// The eval / bench entry points: node problems opts->node_begin..node_end and the evaluation backend opts->solver
// names, on the precision level opts->reserved[5] asks for.
std::unique_ptr<EvalBackend> eval_backend(gml_b200_handle* h, int formulation, const gml_b200_opts& o, NodeProblem& p,
                                          cudaStream_t st) {
    GML_REQUIRE(o.solver == GML_B200_SOLVER_FISTA_CC || o.solver == GML_B200_SOLVER_FISTA_TC,
                "eval and bench need solver = FISTA_CC or FISTA_TC");
    pairwise_problem(p, h->hist, formulation, 0.0, o.node_begin, o.node_end, st);
    std::unique_ptr<EvalBackend> be(o.solver == GML_B200_SOLVER_FISTA_TC ? make_backend_tc(p, st) : make_backend_cc(p, st));
    if (o.reserved[5] == 1)      // the coarse precision level (lattice 2^-22, |x| < 1.95)
        GML_REQUIRE(be->set_level(0, st), "this backend has no coarse precision level");
    if (o.reserved[5] == 2)      // the rough level (lattice 2^-14, |x| < 1.95, one residual digit plane)
        GML_REQUIRE(be->set_level(-1, st), "the rough precision level is not available for this backend / histogram (it needs near-uniform counts)");
    return be;
}

// Host upload of a K-row histogram: fill(d_counts, d_base, Kp) writes the counts and the spin rows of `base` (pitch Kp)
// and returns its host-side time (stats->h2d_ms); validation and padding then run in place.  The handle holds no
// histogram until that has succeeded.
template <class Fill> void upload_histogram_with(gml_b200_handle* h, int64_t K, int32_t N, gml_b200_stats* stats, Fill&& fill) {
    const double t0 = now_ms();
    GML_CUDA(cudaSetDevice(h->device));
    DevBuf<double> dc;
    dc.alloc(K);
    Histogram& hist = h->hist;
    const int64_t Kp = round_up(K, KPAD);
    h->has_hist = false;
    hist.base.alloc((size_t)round_up(N + 1, FPAD) * Kp);
    const double h2d = fill(dc.p, hist.base.p, Kp);
    gml_b200_stats tmp;
    const int rc = gml_b200_attach_histogram_device(h, dc.p, hist.base.p, K, N, Kp, &tmp);
    if (rc != GML_B200_OK) throw CudaError{rc};
    if (stats) {
        *stats = tmp;
        stats->h2d_ms = h2d;
        stats->total_ms = now_ms() - t0;
    }
}

// where the histogram of a one-shot call comes from: packed (counts + int8 spins) or the reference's K x (N+1) matrix
struct HostSource {
    const double* counts = nullptr; const int8_t* spins = nullptr;     // packed form
    const void* matrix = nullptr; int dtype = 0;                       // matrix form
    int64_t ld = 0;
    double regularizer = -1.0;      // >= 0: lambda = regularizer*sqrt(log(N^2/0.05)/M) (:157) from the global sample count
    int upload(gml_b200_handle* h, int64_t k0, int64_t k1, int32_t N, gml_b200_stats* up) const {
        if (matrix) return gml_b200_upload_matrix(h, matrix, dtype, k0, k1 - k0, N, ld, up);
        return gml_b200_upload_histogram(h, counts + k0, spins + k0, k1 - k0, N, ld, up);
    }
    double lambda_for(double lambda, int32_t N, double M) const {
        return regularizer >= 0.0 ? regularizer * std::sqrt(std::log(((double)N * (double)N) / 0.05) / M) : lambda;
    }
};

// One-shot call on one device: its own handle, the upload of all K rows of `src`, then solve(handle, lambda, stats);
// the stats add the upload's to the solve's.
template <class Solve> int learn_one_device(int device, const HostSource& src, int64_t K, int32_t N, double lambda,
                                            gml_b200_stats* stats, Solve&& solve) {
    gml_b200_handle* h = nullptr;
    int rc = gml_b200_create(&h, device);
    if (rc != GML_B200_OK) return rc;
    gml_b200_stats up{}, so{};
    rc = src.upload(h, 0, K, N, &up);
    if (rc == GML_B200_OK) rc = solve(h, src.lambda_for(lambda, N, gml_b200_num_samples(h)), &so);
    if (stats) {
        *stats = so;
        stats->pack_ms = up.pack_ms; stats->h2d_ms = up.h2d_ms;
        stats->kernel_launches += up.kernel_launches;
        stats->total_ms += up.total_ms;
    }
    gml_b200_destroy(h);
    return rc;
}

// Runs body(r) -> status for the devices first_device + r, r < n_dev, on one host thread each.  The combined status is
// the first failure other than ENOTCONV, else ENOTCONV if a device did not converge; the error names the device.
template <class Body> int on_each_device(int first_device, int n_dev, Body&& body) {
    std::vector<int> rcs(n_dev, GML_B200_OK);
    std::vector<std::string> errs(n_dev);
    std::vector<std::thread> threads;
    for (int r = 0; r < n_dev; ++r)
        threads.emplace_back([&, r] {
            rcs[r] = body(r);
            if (rcs[r] != GML_B200_OK) errs[r] = gml_b200_last_error();
        });
    for (auto& t : threads) t.join();
    int rc = GML_B200_OK;
    for (int r = 0; r < n_dev; ++r)
        if (rcs[r] != GML_B200_OK && (rc == GML_B200_OK || rc == GML_B200_ENOTCONV)) { rc = rcs[r]; set_error("device " + std::to_string(first_device + r) + ": " + errs[r]); }
    return rc;
}

// devices of a one-shot call: opts->reserved[4] from opts->device on, as far as they exist
int one_shot_devices(const gml_b200_opts* opts) {
    if (!opts || opts->reserved[4] <= 1) return 1;
    return std::min<int>(opts->reserved[4], std::max(1, gml_b200_device_count() - opts->device));
}

// Partition (SURVEY 8e): sample slices when the tensor-core solver runs and every device still gets a GPU-filling
// number of rows -- each device then streams K/n rows per pass instead of all K.
bool use_sample_slices(const gml_b200_opts* opts, int64_t K, int32_t N, int n_dev) {
    if (n_dev <= 1) return false;
    const bool tc = (opts->solver == GML_B200_SOLVER_AUTO && N + 1 > NEWTON_AUTO_F) || opts->solver == GML_B200_SOLVER_FISTA_TC;
    return tc && K / n_dev >= 65536 && opts->barrier_mu == 0.0;
}

}  // namespace

extern "C" {

const char* gml_b200_version(void) { return "gml_b200 0.2.0 (sm_100a)"; }
const char* gml_b200_last_error(void) { return g_error.c_str(); }

int gml_b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

void gml_b200_opts_default(gml_b200_opts* o) {
    if (!o) return;
    std::memset(o, 0, sizeof(*o));
    o->tol = 0.0;           // 0 = solver default (1e-6 FISTA, 1e-12 Newton)
    o->barrier_mu = 0.0;
    o->max_iter = 0;        // 0 = solver default
    o->solver = GML_B200_SOLVER_AUTO;
    o->device = 0;
    o->node_begin = 0; o->node_end = 0;
}

int64_t gml_b200_multibody_num_keys(int32_t N, int32_t order) {
    int64_t n = 0;
    for (int q = 0; q <= order - 1; ++q) n += binom(N - 1, q);
    return n;
}

int gml_b200_create(gml_b200_handle** out, int32_t device) {
    return guarded([&] {
        GML_REQUIRE(out != nullptr, "null handle pointer");
        int n = 0;
        if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
            cudaGetLastError();
            set_error("no CUDA device available: libgml_b200 has no CPU fallback");
            throw CudaError{GML_B200_ECUDA};
        }
        GML_REQUIRE(device >= 0 && device < n, "device ordinal out of range");
        GML_CUDA(cudaSetDevice(device));
        auto* h = new gml_b200_handle();
        h->device = device;
        GML_CUDA(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
        *out = h;
    });
}

void gml_b200_destroy(gml_b200_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->owns_comm) comm_destroy(h->comm);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    delete h;
}

double gml_b200_num_samples(const gml_b200_handle* h) { return h ? h->hist.M : 0.0; }

int gml_b200_attach_histogram_device(gml_b200_handle* h, const double* d_counts, const int8_t* d_spins, int64_t K,
                                     int32_t N, int64_t ld, gml_b200_stats* stats) {
    return guarded([&] {
        GML_REQUIRE(h && d_counts && d_spins, "null argument");
        const double t0 = now_ms();
        g_launches = 0;
        GML_CUDA(cudaSetDevice(h->device));
        cudaStream_t st = h->own_stream;
        EventTimer timer(st);
        h->has_hist = false;
        hist_from_device(h->hist, d_counts, d_spins, K, N, ld, st);
        h->has_hist = true;
        if (stats) {
            std::memset(stats, 0, sizeof(*stats));
            stats->pack_ms = timer.stop();
            stats->kernel_launches = g_launches;
            stats->total_ms = now_ms() - t0;
        }
    });
}

int gml_b200_upload_histogram(gml_b200_handle* h, const double* counts, const int8_t* spins, int64_t K, int32_t N,
                              int64_t ld, gml_b200_stats* stats) {
    return guarded([&] {
        GML_REQUIRE(h && counts && spins, "null argument");
        GML_REQUIRE(K >= 1 && N >= 1 && ld >= K, "histogram needs K >= 1, N >= 1, ld >= K");
        // the spins land directly in their final place (rows of `base`, pitch Kp); validation and padding
        // then run in place -- no staging copy of the histogram on the device
        upload_histogram_with(h, K, N, stats, [&](double* d_counts, int8_t* d_base, int64_t Kp) {
            cudaStream_t st = h->own_stream;
            EventTimer timer(st);
            GML_CUDA(cudaMemcpyAsync(d_counts, counts, sizeof(double) * K, cudaMemcpyHostToDevice, st));
            GML_CUDA(cudaMemcpy2DAsync(d_base, Kp, spins, ld, K, N, cudaMemcpyHostToDevice, st));
            return timer.stop();
        });
    });
}

int gml_b200_upload_matrix(gml_b200_handle* h, const void* samples, int32_t dtype, int64_t row_begin, int64_t K, int32_t N,
                           int64_t ld, gml_b200_stats* stats) {
    return guarded([&] {
        GML_REQUIRE(h && samples, "null argument");
        GML_REQUIRE(K >= 1 && N >= 1 && row_begin >= 0 && ld >= row_begin + K, "samples matrix needs K >= 1, N >= 1, ld >= row_begin + K");
        upload_histogram_with(h, K, N, stats, [&](double* d_counts, int8_t* d_base, int64_t Kp) {
            double host_ms = 0.0;
            ingest_matrix(samples, dtype, ld, row_begin, K, N, d_base, Kp, d_counts, 0, &host_ms);
            return host_ms;
        });
    });
}

int gml_b200_solve_pairwise_device(gml_b200_handle* h, int32_t formulation, double lambda, const gml_b200_opts* opts,
                                   double* d_out_rows, double* d_out_objective, gml_b200_stats* stats) {
    return guarded([&] {
        GML_REQUIRE(h && d_out_rows, "null argument");
        const double t0 = now_ms();
        g_launches = 0;
        gml_b200_opts o; fill_opts(o, opts);
        GML_CUDA(cudaSetDevice(h->device));
        if (stats) std::memset(stats, 0, sizeof(*stats));
        solve_pairwise_rows(h, formulation, lambda, o, o.node_begin, o.node_end, d_out_rows, d_out_objective, stats,
                            stream_of(h, o), t0);
    });
}

int gml_b200_solve_pairwise(gml_b200_handle* h, int32_t formulation, double lambda, int32_t symmetrize,
                            const gml_b200_opts* opts, double* out_theta, double* out_objective, gml_b200_stats* stats) {
    return guarded([&] {
        GML_REQUIRE(h && out_theta, "null argument");
        GML_REQUIRE(h->has_hist, "no histogram resident: call gml_b200_upload_histogram first");
        const double t0 = now_ms();
        g_launches = 0;
        gml_b200_opts o; fill_opts(o, opts);
        GML_CUDA(cudaSetDevice(h->device));
        cudaStream_t st = stream_of(h, o);
        if (stats) std::memset(stats, 0, sizeof(*stats));
        const int N = h->hist.N;
        const auto [nb, ne] = node_range(o.node_begin, o.node_end, N);
        const int Nn = ne - nb;
        DevBuf<double> rows, obj;
        rows.alloc((size_t)Nn * N); obj.alloc(Nn);
        int rc = GML_B200_OK;
        try {
            solve_pairwise_rows(h, formulation, lambda, o, nb, ne, rows.p, out_objective ? obj.p : nullptr, stats, st, t0);
        } catch (const CudaError& e) {
            if (e.code != GML_B200_ENOTCONV) throw;
            rc = e.code;   // still hand back the best iterate, then report
        }
        EventTimer timer(st);
        if (symmetrize && Nn == N) launch_symmetrize(rows.p, N, st);
        std::vector<double> hrows((size_t)Nn * N);
        GML_CUDA(cudaMemcpyAsync(hrows.data(), rows.p, sizeof(double) * Nn * N, cudaMemcpyDeviceToHost, st));
        if (out_objective) GML_CUDA(cudaMemcpyAsync(out_objective + nb, obj.p, sizeof(double) * Nn, cudaMemcpyDeviceToHost, st));
        const double d2h = timer.stop();
        scatter_rows(hrows.data(), Nn, N, nb, out_theta);
        if (stats) { stats->d2h_ms = d2h; stats->kernel_launches = g_launches; stats->total_ms = now_ms() - t0; }
        if (rc != GML_B200_OK) throw CudaError{rc};
    });
}

int gml_b200_solve_pairwise_path(gml_b200_handle* h, int32_t formulation, const double* lambdas, int32_t n_lambda,
                                 int32_t symmetrize, const gml_b200_opts* opts, double* out_thetas, gml_b200_stats* stats) {
    return guarded([&] {
        GML_REQUIRE(h && lambdas && out_thetas && n_lambda >= 1, "bad argument");
        GML_REQUIRE(h->has_hist, "no histogram resident: call gml_b200_upload_histogram first");
        const double t0 = now_ms();
        g_launches = 0;
        gml_b200_opts o; fill_opts(o, opts);
        GML_CUDA(cudaSetDevice(h->device));
        cudaStream_t st = stream_of(h, o);
        const int N = h->hist.N;
        GML_REQUIRE(pick_solver(o, N + 1) != GML_B200_SOLVER_NEWTON, "the regularisation path uses the FISTA solvers (set opts->solver)");
        DevBuf<double> rows, warm;
        rows.alloc((size_t)N * N);
        std::vector<double> hrows((size_t)N * N);
        gml_b200_stats acc{}, cur{};
        for (int li = 0; li < n_lambda; ++li) {
            std::memset(&cur, 0, sizeof(cur));
            solve_pairwise_rows(h, formulation, lambdas[li], o, 0, N, rows.p, nullptr, &cur, st, now_ms(), &warm);   // warm start
            if (symmetrize) launch_symmetrize(rows.p, N, st);
            GML_CUDA(cudaMemcpyAsync(hrows.data(), rows.p, sizeof(double) * N * N, cudaMemcpyDeviceToHost, st));
            GML_CUDA(cudaStreamSynchronize(st));
            scatter_rows(hrows.data(), N, N, 0, out_thetas + (size_t)li * N * N);
            acc.iterations += cur.iterations; acc.n_fg_passes += cur.n_fg_passes; acc.n_f_passes += cur.n_f_passes;
            acc.evals += cur.evals; acc.solve_ms += cur.solve_ms; acc.solver_used = cur.solver_used;
            acc.max_residual = std::max(acc.max_residual, cur.max_residual);
        }
        acc.kernel_launches = g_launches;
        acc.total_ms = now_ms() - t0;
        if (stats) *stats = acc;
    });
}

static int solve_multibody_impl(gml_b200_handle* h, int32_t order, double lambda, const gml_b200_opts* opts,
                                double* out_vals, double* out_sym, double* out_objective, gml_b200_stats* stats) {
    return guarded([&] {
        GML_REQUIRE(h && (out_vals || out_sym), "null argument");
        GML_REQUIRE(h->has_hist, "no histogram resident: call gml_b200_upload_histogram first");
        GML_REQUIRE(order >= 1, "interaction_order must be >= 1");
        GML_REQUIRE(lambda >= 0.0 && std::isfinite(lambda), "lambda must be finite and >= 0");
        const double t0 = now_ms();
        g_launches = 0;
        gml_b200_opts o; fill_opts(o, opts);
        GML_CUDA(cudaSetDevice(h->device));
        cudaStream_t st = stream_of(h, o);
        if (stats) std::memset(stats, 0, sizeof(*stats));
        Histogram& hist = h->hist;
        const int N = hist.N;
        int64_t nf = 0;
        for (int q = 0; q <= order - 1; ++q) nf += binom(N, q);
        GML_REQUIRE(nf <= (1 << 16), "multiRISE feature count exceeds 65536: reduce interaction_order");
        MultibodyLayout L = multibody_layout(N, order);
        EventTimer timer(st);
        build_multibody_features(hist, order, L.subsets, L.F, st);
        NodeProblem p;
        p.hist = &hist; p.Q = hist.mb.p; p.F = L.F; p.Fp = hist.mb_Fp;
        p.form = GML_B200_RISE; p.lambda = lambda; p.Nn = N;
        p.spin_row.alloc(N); p.pen.alloc((size_t)N * p.Fp);
        DevBuf<int32_t> key_map;
        key_map.alloc(L.key_map.size());
        GML_CUDA(cudaMemcpyAsync(key_map.p, L.key_map.data(), sizeof(int32_t) * L.key_map.size(), cudaMemcpyHostToDevice, st));
        multibody_setup_kernel<<<N, 128, 0, st>>>(p.Fp, L.n_keys, key_map.p, p.spin_row.p, p.pen.p);
        GML_LAUNCHED();
        SolveResult r;
        int solver_used = 0;
        run_solver(p, o, r, solver_used, st);
        DevBuf<double> vals, sym;
        DevBuf<long long> tab;
        int64_t n_sym = 0;
        if (out_vals) {
            vals.alloc((size_t)N * L.n_keys);
            multibody_gather_kernel<<<N, 128, 0, st>>>(r.x.p, p.Fp, L.n_keys, key_map.p, vals.p);
            GML_LAUNCHED();
        }
        if (out_sym) {
            GML_REQUIRE(order <= 8, "device symmetrisation supports interaction_order <= 8");
            const int W = order + 1;
            std::vector<long long> ht((size_t)(N + 1) * W + (order + 2) + (order + 1), 0);
            for (int n = 0; n <= N; ++n)
                for (int k = 0; k <= order; ++k) ht[(size_t)n * W + k] = binom(n, k);
            long long* key_off = ht.data() + (size_t)(N + 1) * W;        // by key size q = 1..order
            long long* feat_off = key_off + (order + 2);                  // by feature size q = 0..order-1
            for (int q = 1; q <= order; ++q) key_off[q + 1] = key_off[q] + binom(N, q);
            for (int q = 0; q < order; ++q) feat_off[q + 1] = feat_off[q] + binom(N, q);
            n_sym = key_off[order + 1];
            tab.alloc(ht.size()); sym.alloc((size_t)n_sym);
            GML_CUDA(cudaMemcpyAsync(tab.p, ht.data(), sizeof(long long) * ht.size(), cudaMemcpyHostToDevice, st));
            multibody_symmetrize_kernel<<<(unsigned)ceil_div(n_sym, 128), 128, 0, st>>>(r.x.p, N, p.Fp, order, tab.p, tab.p + (size_t)(N + 1) * W,
                                                                                   tab.p + (size_t)(N + 1) * W + (order + 2), n_sym, sym.p);
            GML_LAUNCHED();
            GML_CUDA(cudaStreamSynchronize(st));      // `ht` is read by the copy above
        }
        const double solve_ms = timer.stop();
        EventTimer t2(st);
        if (out_vals) GML_CUDA(cudaMemcpyAsync(out_vals, vals.p, sizeof(double) * N * L.n_keys, cudaMemcpyDeviceToHost, st));
        if (out_sym) GML_CUDA(cudaMemcpyAsync(out_sym, sym.p, sizeof(double) * n_sym, cudaMemcpyDeviceToHost, st));
        if (out_objective) GML_CUDA(cudaMemcpyAsync(out_objective, r.objective.p, sizeof(double) * N, cudaMemcpyDeviceToHost, st));
        const double d2h = t2.stop();
        finish_stats(stats, r, solver_used, N, hist.K, solve_ms, d2h, t0);
        throw_if_unconverged(r.n_unconverged);
    });
}

int gml_b200_solve_multibody(gml_b200_handle* h, int32_t order, double lambda, const gml_b200_opts* opts,
                             double* out_vals, double* out_objective, gml_b200_stats* stats) {
    if (!out_vals) { set_error("null argument"); return GML_B200_EINVAL; }
    return solve_multibody_impl(h, order, lambda, opts, out_vals, nullptr, out_objective, stats);
}

int gml_b200_solve_multibody_sym(gml_b200_handle* h, int32_t order, double lambda, const gml_b200_opts* opts,
                                 double* out_sym_vals, double* out_objective, gml_b200_stats* stats) {
    if (!out_sym_vals) { set_error("null argument"); return GML_B200_EINVAL; }
    return solve_multibody_impl(h, order, lambda, opts, nullptr, out_sym_vals, out_objective, stats);
}

int64_t gml_b200_multibody_num_sym_keys(int32_t N, int32_t order) {
    int64_t n = 0;
    for (int q = 1; q <= order; ++q) n += binom(N, q);
    return n;
}

// |theta| < tau -> 0 off the diagonal (post-hoc support selection, SURVEY 8f-3); counts the surviving off-diagonal entries
__global__ void threshold_kernel(double* __restrict__ m, int N, double tau, unsigned long long* __restrict__ nnz) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)N * N) return;
    const int r = (int)(i / N), c = (int)(i % N);
    if (r == c) return;
    if (fabs(m[i]) < tau) m[i] = 0.0;
    else atomicAdd(nnz, 1ull);
}

int gml_b200_threshold_device(double* d_theta, int32_t N, double tau, int64_t* out_nnz, void* stream) {
    return guarded([&] {
        GML_REQUIRE(d_theta && N >= 1 && tau >= 0.0, "bad argument");
        cudaStream_t st = (cudaStream_t)stream;
        DevBuf<unsigned long long> cnt;
        cnt.alloc(1);
        GML_CUDA(cudaMemsetAsync(cnt.p, 0, sizeof(unsigned long long), st));
        threshold_kernel<<<(unsigned)ceil_div((int64_t)N * N, 256), 256, 0, st>>>(d_theta, N, tau, cnt.p);
        GML_LAUNCHED();
        unsigned long long hc = 0;
        GML_CUDA(cudaMemcpyAsync(&hc, cnt.p, sizeof(hc), cudaMemcpyDeviceToHost, st));
        GML_CUDA(cudaStreamSynchronize(st));
        if (out_nnz) *out_nnz = (int64_t)hc;
    });
}

int gml_b200_eval_pairwise(gml_b200_handle* h, int32_t formulation, const gml_b200_opts* opts, const double* x,
                           double* f_out, double* g_out) {
    return guarded([&] {
        GML_REQUIRE(h && x && f_out, "null argument");
        GML_REQUIRE(h->has_hist, "no histogram resident: call gml_b200_upload_histogram first");
        g_launches = 0;
        gml_b200_opts o; fill_opts(o, opts);
        GML_CUDA(cudaSetDevice(h->device));
        cudaStream_t st = stream_of(h, o);
        NodeProblem p;
        const std::unique_ptr<EvalBackend> be = eval_backend(h, formulation, o, p, st);
        const int nb = o.node_begin, F = p.F;
        std::vector<double> hx((size_t)p.Nn * p.Fp, 0.0);
        const double lat = be->lattice(), xmax = be->x_range();
        for (int u = 0; u < p.Nn; ++u)
            for (int f = 0; f < F; ++f) {
                double v = (f == nb + u) ? 0.0 : x[(size_t)u * F + f];
                GML_REQUIRE(std::isfinite(v) && (xmax <= 0.0 || std::fabs(v) <= xmax),
                            "eval: a coefficient lies outside the fixed-point range of the tensor-core backend "
                            "(|x| < 7.9 on the fine level, < 1.95 on the coarse one); use solver = FISTA_CC");
                if (lat > 0.0) v = std::nearbyint(v / lat) * lat;
                hx[(size_t)u * p.Fp + f] = v;
            }
        DevBuf<double> dx, df, dg;
        dx.alloc(hx.size()); df.alloc(p.Nn); dg.alloc(hx.size());
        GML_CUDA(cudaMemcpyAsync(dx.p, hx.data(), sizeof(double) * hx.size(), cudaMemcpyHostToDevice, st));
        be->eval(dx.p, g_out != nullptr, df.p, dg.p, st);
        GML_CUDA(cudaMemcpyAsync(f_out, df.p, sizeof(double) * p.Nn, cudaMemcpyDeviceToHost, st));
        if (g_out) {
            GML_CUDA(cudaMemcpyAsync(hx.data(), dg.p, sizeof(double) * hx.size(), cudaMemcpyDeviceToHost, st));
            GML_CUDA(cudaStreamSynchronize(st));
            for (int u = 0; u < p.Nn; ++u)
                for (int f = 0; f < F; ++f) g_out[(size_t)u * F + f] = (f == nb + u) ? 0.0 : hx[(size_t)u * p.Fp + f];
        }
        GML_CUDA(cudaStreamSynchronize(st));
    });
}

int gml_b200_bench_passes(gml_b200_handle* h, int32_t formulation, const gml_b200_opts* opts, int32_t reps,
                          double* out_ms) {
    return guarded([&] {
        GML_REQUIRE(h && out_ms && reps >= 1, "bad argument");
        GML_REQUIRE(h->has_hist, "no histogram resident: call gml_b200_upload_histogram first");
        g_launches = 0;
        gml_b200_opts o; fill_opts(o, opts);
        GML_CUDA(cudaSetDevice(h->device));
        cudaStream_t st = stream_of(h, o);
        NodeProblem p;
        const std::unique_ptr<EvalBackend> be = eval_backend(h, formulation, o, p, st);
        DevBuf<double> dx, df, dg;
        const size_t nx = (size_t)p.Nn * p.Fp;
        dx.alloc(nx); df.alloc(p.Nn); dg.alloc(nx);
        GML_CUDA(cudaMemsetAsync(dx.p, 0, sizeof(double) * nx, st));
        be->eval(dx.p, true, df.p, dg.p, st);    // warm-up
        be->eval(dx.p, false, df.p, nullptr, st);
        be->set_profiling(true);
        EventTimer wall(st);
        for (int i = 0; i < reps; ++i) be->eval(dx.p, true, df.p, dg.p, st);
        const double wall_ms = wall.stop();
        for (int i = 0; i < reps; ++i) be->eval(dx.p, false, df.p, nullptr, st);
        GML_CUDA(cudaStreamSynchronize(st));
        double prof[4] = {0, 0, 0, 0};
        be->collect_profile(prof);
        out_ms[0] = prof[0] / reps; out_ms[1] = prof[1] / reps; out_ms[2] = prof[2] / reps; out_ms[3] = wall_ms / reps;
    });
}

int gml_b200_symmetrize_device(double* d_theta, int32_t N, void* stream) {
    return guarded([&] {
        GML_REQUIRE(d_theta && N >= 1, "bad argument");
        launch_symmetrize(d_theta, N, (cudaStream_t)stream);
    });
}

// Single-process multi-GPU form of the one-shot call (opts->reserved[4] = number of devices): one host thread per
// device, each with its own handle, the histogram replicated, node shards with 16-aligned cuts; every thread writes
// its rows straight into the caller's matrix, the symmetrisation of the N x N result runs on the host.  This is what a
// single Julia process uses; multi-process launches (torchrun) use gml_b200_solve_pairwise_device + an all-gather.
static int learn_pairwise_multi_device(const HostSource& src, int64_t K, int32_t N, int32_t formulation, double lambda,
                                       int32_t symmetrize, const gml_b200_opts& base, int n_dev, double* out_theta,
                                       double* out_objective, gml_b200_stats* stats) {
    const double t0 = now_ms();
    std::vector<gml_b200_stats> sts(n_dev);
    auto cut = [&](int r) {            // same rule as distributed.shard_bounds
        const int per = N / n_dev, extra = N % n_dev;
        int b = r * per + std::min(r, extra), e = b + per + (r < extra ? 1 : 0);
        if (per >= 64) {
            auto up = [&](int v) { return std::min(N, (v + 15) / 16 * 16); };
            b = r == 0 ? 0 : up(b); e = r == n_dev - 1 ? N : up(e);
        }
        return std::make_pair(b, e);
    };
    int rc = on_each_device(base.device, n_dev, [&](int r) {
        gml_b200_handle* h = nullptr;
        gml_b200_opts o = base;
        o.device = base.device + r;
        const auto be = cut(r);
        o.node_begin = be.first; o.node_end = be.second; o.stream = nullptr;
        int rc = gml_b200_create(&h, o.device);
        gml_b200_stats up{};
        if (rc == GML_B200_OK && be.first < be.second) {
            rc = src.upload(h, 0, K, N, &up);
            if (rc == GML_B200_OK)
                rc = gml_b200_solve_pairwise(h, formulation, lambda, 0, &o, out_theta, out_objective, &sts[r]);
            sts[r].pack_ms = up.pack_ms; sts[r].h2d_ms = up.h2d_ms; sts[r].kernel_launches += up.kernel_launches;
        }
        gml_b200_destroy(h);
        return rc;
    });
    if (symmetrize && (rc == GML_B200_OK || rc == GML_B200_ENOTCONV)) {
        // on the first device: the rows of all shards are already in the caller's matrix
        const int rs = guarded([&] {
            GML_CUDA(cudaSetDevice(base.device));
            DevBuf<double> m;
            m.alloc((size_t)N * N);
            GML_CUDA(cudaMemcpy(m.p, out_theta, sizeof(double) * N * N, cudaMemcpyHostToDevice));
            launch_symmetrize(m.p, N, 0);
            GML_CUDA(cudaMemcpy(out_theta, m.p, sizeof(double) * N * N, cudaMemcpyDeviceToHost));
        });
        if (rs != GML_B200_OK) rc = rs;
    }
    if (stats) {
        std::memset(stats, 0, sizeof(*stats));
        for (int r = 0; r < n_dev; ++r) {
            stats->solver_used = sts[r].solver_used;
            stats->iterations = std::max(stats->iterations, sts[r].iterations);
            stats->n_fg_passes = std::max(stats->n_fg_passes, sts[r].n_fg_passes);
            stats->n_f_passes = std::max(stats->n_f_passes, sts[r].n_f_passes);
            stats->n_unconverged += sts[r].n_unconverged;
            stats->kernel_launches += sts[r].kernel_launches;
            stats->evals += sts[r].evals;
            stats->solve_ms = std::max(stats->solve_ms, sts[r].solve_ms);
            stats->h2d_ms = std::max(stats->h2d_ms, sts[r].h2d_ms);
            stats->pack_ms = std::max(stats->pack_ms, sts[r].pack_ms);
            stats->max_residual = std::max(stats->max_residual, sts[r].max_residual);
        }
        stats->total_ms = now_ms() - t0;
    }
    return rc;
}

// Single-process multi-GPU, sample-sharded form: one host thread per device, each uploads ITS slice of the histogram
// rows (one pass over the host link per byte, no replication), the threads join one NCCL communicator and advance all
// node problems in lockstep (all-reduce of the exact int64 gradient sums per pass, csrc/comm.cu).  Every device ends
// with the full solution; device `base.device` symmetrises it on the device (:184-186) and writes the caller's matrix.
static int learn_pairwise_multi_device_samples(const HostSource& src, int64_t K, int32_t N,
                                               int32_t formulation, double lambda, int32_t symmetrize, const gml_b200_opts& base,
                                               int n_dev, double* out_theta, double* out_objective, gml_b200_stats* stats) {
    const double t0 = now_ms();
    // One communicator per (first device, device count) and process: ncclCommInitRank costs 0.1-1 s, a learn() call ~1 s.
    // The per-rank communicators are created by the first call and reused by the host threads of every later call.
    static std::mutex cache_mutex;
    static std::map<std::pair<int, int>, std::vector<Comm*>> comm_cache;
    std::lock_guard<std::mutex> cache_lock(cache_mutex);      // also serialises concurrent multi-device calls on these devices
    std::vector<Comm*>& cached = comm_cache[std::make_pair((int)base.device, n_dev)];
    const bool have_comm = (int)cached.size() == n_dev;
    uint8_t ident[128];
    if (!have_comm && gml_b200_comm_unique_id(ident) != GML_B200_OK) { comm_cache.erase(std::make_pair((int)base.device, n_dev)); return -1; }   // no NCCL: node shards
    if (!have_comm) cached.assign(n_dev, nullptr);
    std::vector<gml_b200_stats> sts(n_dev);
    const int64_t per = round_up(ceil_div(K, n_dev), 256);
    const int rc = on_each_device(base.device, n_dev, [&](int r) {
        gml_b200_handle* h = nullptr;
        gml_b200_opts o = base;
        o.device = base.device + r; o.stream = nullptr;
        o.node_begin = 0; o.node_end = 0; o.reserved[2] = 1; o.reserved[4] = 0;
        o.solver = GML_B200_SOLVER_FISTA_TC;
        const int64_t k0 = std::min<int64_t>(K, r * per), k1 = std::min<int64_t>(K, (r + 1) * per);
        gml_b200_stats up{};
        int rc = gml_b200_create(&h, o.device);
        if (rc == GML_B200_OK) rc = src.upload(h, k0, k1, N, &up);
        // every thread must reach the communicator set-up, also after a failed upload (the others would wait for ever)
        int rc_comm = GML_B200_ECUDA;
        if (h && have_comm) { h->comm = cached[r]; h->owns_comm = false; rc_comm = GML_B200_OK; }
        else if (h) {
            rc_comm = gml_b200_comm_init(h, ident, r, n_dev);
            if (rc_comm == GML_B200_OK) { cached[r] = h->comm; h->owns_comm = false; }      // the cache owns it from now on
        }
        if (rc == GML_B200_OK) rc = rc_comm;
        if (rc_comm == GML_B200_OK) {       // leave together if any device failed so far
            int agreed = rc;
            if (guarded([&] { agreed = comm_agree_max(h->comm, rc, h->own_stream); }) == GML_B200_OK && agreed != GML_B200_OK && rc == GML_B200_OK) {
                rc = agreed; set_error("another device of the multi-device solve failed");
            }
        }
        if (rc == GML_B200_OK) rc = gml_b200_comm_globalize_histogram(h);
        if (rc == GML_B200_OK) {
            const double lam = src.lambda_for(lambda, N, gml_b200_num_samples(h));     // global M after the globalize step
            if (r == 0) rc = gml_b200_solve_pairwise(h, formulation, lam, symmetrize, &o, out_theta, out_objective, &sts[r]);
            else {
                DevBuf<double> rows, obj_scratch;
                try { rows.alloc((size_t)N * N); if (out_objective) obj_scratch.alloc(N); } catch (const CudaError& e) { rc = e.code; }
                if (rc == GML_B200_OK)      // same passes as device 0: the objective pass is a collective
                    rc = gml_b200_solve_pairwise_device(h, formulation, lam, &o, rows.p, out_objective ? obj_scratch.p : nullptr, &sts[r]);
                cudaStreamSynchronize(h->own_stream);
            }
            sts[r].pack_ms = up.pack_ms; sts[r].h2d_ms = up.h2d_ms; sts[r].kernel_launches += up.kernel_launches;
        }
        gml_b200_destroy(h);
        return rc;
    });
    if (!have_comm)
        for (int r = 0; r < n_dev; ++r)
            if (!cached[r]) { comm_cache.erase(std::make_pair((int)base.device, n_dev)); break; }      // set-up failed on some device: retry next call
    if (stats) {
        *stats = sts[0];
        for (int r = 1; r < n_dev; ++r) {
            stats->kernel_launches += sts[r].kernel_launches;
            stats->evals += sts[r].evals;
            stats->solve_ms = std::max(stats->solve_ms, sts[r].solve_ms);
            stats->h2d_ms = std::max(stats->h2d_ms, sts[r].h2d_ms);
            stats->pack_ms = std::max(stats->pack_ms, sts[r].pack_ms);
        }
        stats->total_ms = now_ms() - t0;
    }
    return rc;
}

int gml_b200_learn_pairwise(const double* counts, const int8_t* spins, int64_t K, int32_t N, int64_t ld,
                            int32_t formulation, double lambda, int32_t symmetrize, const gml_b200_opts* opts,
                            double* out_theta, double* out_objective, gml_b200_stats* stats) {
    HostSource src;
    src.counts = counts; src.spins = spins; src.ld = ld;
    const int n_dev = one_shot_devices(opts);
    // else node shards with the histogram replicated; opts->reserved[2] = 2 forces them
    if (use_sample_slices(opts, K, N, n_dev) && opts->reserved[2] != 2) {
        const int rc = learn_pairwise_multi_device_samples(src, K, N, formulation, lambda, symmetrize, *opts,
                                                           n_dev, out_theta, out_objective, stats);
        if (rc >= 0) return rc;
    }
    if (n_dev > 1 && N >= 2 * n_dev)
        return learn_pairwise_multi_device(src, K, N, formulation, lambda, symmetrize, *opts, n_dev, out_theta,
                                           out_objective, stats);
    return learn_one_device(opts ? opts->device : 0, src, K, N, lambda, stats, [&](gml_b200_handle* h, double lam, gml_b200_stats* so) {
        return gml_b200_solve_pairwise(h, formulation, lam, symmetrize, opts, out_theta, out_objective, so);
    });
}

int gml_b200_learn_multibody(const double* counts, const int8_t* spins, int64_t K, int32_t N, int64_t ld,
                             int32_t order, double lambda, const gml_b200_opts* opts, double* out_vals,
                             double* out_objective, gml_b200_stats* stats) {
    HostSource src;
    src.counts = counts; src.spins = spins; src.ld = ld;
    return learn_one_device(opts ? opts->device : 0, src, K, N, lambda, stats, [&](gml_b200_handle* h, double lam, gml_b200_stats* so) {
        return gml_b200_solve_multibody(h, order, lam, opts, out_vals, out_objective, so);
    });
}

int gml_b200_learn_pairwise_matrix(const void* samples, int32_t dtype, int64_t K, int32_t N, int64_t ld,
                                   int32_t formulation, double regularizer, int32_t symmetrize, const gml_b200_opts* opts,
                                   double* out_theta, double* out_objective, gml_b200_stats* stats) {
    if (!(regularizer >= 0.0) || !std::isfinite(regularizer)) { set_error("regularizer must be finite and >= 0"); return GML_B200_EINVAL; }
    HostSource src;
    src.matrix = samples; src.dtype = dtype; src.ld = ld; src.regularizer = regularizer;
    const int n_dev = one_shot_devices(opts);
    if (use_sample_slices(opts, K, N, n_dev)) {
        const int rc = learn_pairwise_multi_device_samples(src, K, N, formulation, 0.0, symmetrize, *opts, n_dev, out_theta,
                                                           out_objective, stats);
        if (rc >= 0) return rc;
    }
    return learn_one_device(opts ? opts->device : 0, src, K, N, 0.0, stats, [&](gml_b200_handle* h, double lam, gml_b200_stats* so) {
        return gml_b200_solve_pairwise(h, formulation, lam, symmetrize, opts, out_theta, out_objective, so);
    });
}

int gml_b200_learn_multibody_matrix(const void* samples, int32_t dtype, int64_t K, int32_t N, int64_t ld, int32_t order,
                                    double regularizer, const gml_b200_opts* opts, double* out_vals, double* out_objective,
                                    gml_b200_stats* stats) {
    if (!(regularizer >= 0.0) || !std::isfinite(regularizer)) { set_error("regularizer must be finite and >= 0"); return GML_B200_EINVAL; }
    HostSource src;
    src.matrix = samples; src.dtype = dtype; src.ld = ld; src.regularizer = regularizer;
    return learn_one_device(opts ? opts->device : 0, src, K, N, 0.0, stats, [&](gml_b200_handle* h, double lam, gml_b200_stats* so) {
        return gml_b200_solve_multibody(h, order, lam, opts, out_vals, out_objective, so);
    });
}

int gml_b200_sample_gibbs_device(int32_t device, int32_t N, const int32_t* row_ptr, const int32_t* col_idx,
                                 const float* coupling, const float* field, int64_t n_samples, int32_t sweeps,
                                 uint64_t seed, int8_t* d_spins, int64_t ld, void* stream) {
    return guarded([&] {
        GML_REQUIRE(N >= 1 && N <= 4096 && row_ptr && col_idx && coupling && d_spins, "bad sampler argument");
        GML_REQUIRE(n_samples >= 1 && ld >= n_samples && sweeps >= 1, "bad sampler sizes");
        GML_CUDA(cudaSetDevice(device));
        cudaStream_t st = (cudaStream_t)stream;
        const int nnz = row_ptr[N];
        int max_deg = 0;
        for (int i = 0; i < N; ++i) max_deg = std::max(max_deg, row_ptr[i + 1] - row_ptr[i]);
        DevBuf<int32_t> rp, ci;
        DevBuf<float> jj, hh;
        rp.alloc(N + 1); ci.alloc(std::max(nnz, 1)); jj.alloc(std::max(nnz, 1)); hh.alloc(N);
        std::vector<float> hz(N, 0.f);
        GML_CUDA(cudaMemcpyAsync(rp.p, row_ptr, sizeof(int32_t) * (N + 1), cudaMemcpyHostToDevice, st));
        GML_CUDA(cudaMemcpyAsync(ci.p, col_idx, sizeof(int32_t) * nnz, cudaMemcpyHostToDevice, st));
        GML_CUDA(cudaMemcpyAsync(jj.p, coupling, sizeof(float) * nnz, cudaMemcpyHostToDevice, st));
        GML_CUDA(cudaMemcpyAsync(hh.p, field ? field : hz.data(), sizeof(float) * N, cudaMemcpyHostToDevice, st));
        sample_gibbs(N, rp.p, ci.p, jj.p, hh.p, max_deg, n_samples, sweeps, seed, d_spins, ld, st);
        GML_CUDA(cudaStreamSynchronize(st));
    });
}

int gml_b200_sample_gibbs_terms_device(int32_t device, int32_t N, int32_t order, int32_t n_terms, const int32_t* term_idx,
                                       const float* term_weight, int64_t n_samples, int32_t sweeps, uint64_t seed,
                                       int8_t* d_spins, int64_t ld, void* stream) {
    return guarded([&] {
        GML_REQUIRE(N >= 1 && N <= 4096 && order >= 1 && order <= 8 && n_terms >= 0 && term_idx && term_weight && d_spins,
                    "bad sampler argument");
        GML_REQUIRE(n_samples >= 1 && ld >= n_samples && sweeps >= 1, "bad sampler sizes");
        GML_CUDA(cudaSetDevice(device));
        cudaStream_t st = (cudaStream_t)stream;
        const Incidence inc = build_incidence(N, order, n_terms, term_idx);
        std::vector<float> weight(inc.term.size(), 0.f);
        for (size_t q = 0; q < inc.term.size(); ++q)
            if (inc.term[q] >= 0) weight[q] = term_weight[inc.term[q]];
        DevBuf<int32_t> rp, ot;
        DevBuf<float> ww;
        rp.alloc(N + 1); ot.alloc(inc.others.size()); ww.alloc(weight.size());
        GML_CUDA(cudaMemcpyAsync(rp.p, inc.row_ptr.data(), sizeof(int32_t) * (N + 1), cudaMemcpyHostToDevice, st));
        GML_CUDA(cudaMemcpyAsync(ot.p, inc.others.data(), sizeof(int32_t) * inc.others.size(), cudaMemcpyHostToDevice, st));
        GML_CUDA(cudaMemcpyAsync(ww.p, weight.data(), sizeof(float) * weight.size(), cudaMemcpyHostToDevice, st));
        sample_gibbs_terms(N, inc.width, rp.p, ot.p, ww.p, n_samples, sweeps, seed, d_spins, ld, st);
        GML_CUDA(cudaStreamSynchronize(st));
    });
}

int gml_b200_sample_exact_device(int32_t device, int32_t N, int32_t order, int32_t n_terms, const int32_t* term_idx,
                                 const double* term_weight, int64_t n_samples, int32_t replicates, uint64_t seed,
                                 int64_t* out_K, double* out_log_z, double* d_counts, int8_t* d_spins, int64_t ld,
                                 void* stream) {
    return guarded([&] {
        GML_REQUIRE(N >= 1 && N <= GML_B200_EXACT_MAX_N, "exact sampler needs 1 <= N <= " + std::to_string(GML_B200_EXACT_MAX_N));
        GML_REQUIRE(order >= 1 && order <= GML_B200_EXACT_MAX_N && n_terms >= 0 && (n_terms == 0 || (term_idx && term_weight)) && out_K,
                    "bad sampler argument");
        GML_REQUIRE(n_samples >= 1 && replicates >= 1 && n_samples <= (INT64_C(1) << 62) / replicates, "bad sampler sizes");
        GML_REQUIRE(!d_counts || (d_spins && ld >= 1), "d_counts needs d_spins and ld >= 1");
        std::vector<uint64_t> masks(n_terms, 0);
        std::vector<double> weights(term_weight, term_weight + n_terms);
        double abs_sum = 0.0;
        for (int t = 0; t < n_terms; ++t) {
            for (int m = 0; m < order; ++m) {
                const int i = term_idx[(size_t)t * order + m];
                if (i == -1) continue;
                GML_REQUIRE(i >= 0 && i < N, "sampler term refers to a spin outside [0, N)");
                GML_REQUIRE(!((masks[t] >> i) & 1ull), "sampler term repeats a spin");
                masks[t] |= 1ull << i;
            }
            GML_REQUIRE(std::isfinite(weights[t]), "sampler term weight is not finite");
            abs_sum += std::fabs(weights[t]);
        }
        GML_REQUIRE(std::isfinite(abs_sum), "sum of |term weights| is not finite");
        GML_CUDA(cudaSetDevice(device));
        cudaStream_t st = (cudaStream_t)stream;
        double log_z = 0.0;
        into_sample_buffers(d_counts, d_spins, ld, N, replicates, out_K, st, [&](double* c, int8_t* sp) {
            log_z = sample_exact(N, masks, weights, n_samples, replicates, seed, out_K, c, sp, ld, st);
        });
        if (out_log_z) *out_log_z = log_z;
    });
}

int gml_b200_sample_mcmc_device(int32_t device, int32_t N, int32_t order, int32_t n_terms, const int32_t* term_idx,
                                const double* term_weight, int64_t n_samples, int32_t replicates, int64_t chains, int32_t burn_in,
                                int32_t thin, uint64_t seed, int64_t* out_K, double* out_rhat, double* d_counts, int8_t* d_spins,
                                int64_t ld, void* stream) {
    return guarded([&] {
        run_mcmc(device, N, order, n_terms, term_idx, term_weight, {1.0}, n_samples, replicates, chains, burn_in, thin, seed,
                 out_K, out_rhat, nullptr, d_counts, d_spins, ld, stream);
    });
}

int gml_b200_sample_tempering_device(int32_t device, int32_t N, int32_t order, int32_t n_terms, const int32_t* term_idx,
                                     const double* term_weight, int32_t n_rungs, const double* betas, int64_t n_samples,
                                     int32_t replicates, int64_t chains, int32_t burn_in, int32_t thin, uint64_t seed,
                                     int64_t* out_K, double* out_rhat, double* out_swap_rate, double* d_counts, int8_t* d_spins,
                                     int64_t ld, void* stream) {
    return guarded([&] {
        GML_REQUIRE(n_rungs == 0 || n_rungs == 2 || n_rungs == 4 || n_rungs == 8 || n_rungs == 16 || n_rungs == 32,
                    "n_rungs must be 0 (the default ladder) or one of 2, 4, 8, 16, 32");
        GML_REQUIRE((n_rungs == 0) == (betas == nullptr), "n_rungs = 0 goes with betas = NULL (the default ladder) and only with it");
        std::vector<double> ladder;
        if (n_rungs == 0) {                          // the default ladder: geometric from 1 to 0.1
            constexpr int R = GML_B200_TEMPERING_DEFAULT_RUNGS;
            for (int k = 0; k < R; ++k) ladder.push_back(std::pow(0.1, (double)k / (R - 1)));
        } else {
            ladder.assign(betas, betas + n_rungs);
            GML_REQUIRE(ladder[0] == 1.0, "betas[0] must be 1 (the rung that records)");
            for (int k = 1; k < n_rungs; ++k)
                GML_REQUIRE(std::isfinite(ladder[k]) && ladder[k] >= 0.0 && ladder[k] < ladder[k - 1],
                            "betas must be finite, non-negative and strictly decreasing");
        }
        run_mcmc(device, N, order, n_terms, term_idx, term_weight, ladder, n_samples, replicates, chains, burn_in, thin, seed,
                 out_K, out_rhat, out_swap_rate, d_counts, d_spins, ld, stream);
    });
}

int gml_b200_build_histogram_device(int32_t device, const int8_t* d_samples, int64_t M, int32_t N, int64_t ld,
                                    int8_t* d_out_spins, int64_t ld_out, double* d_out_counts, int64_t* out_K,
                                    void* stream) {
    return guarded([&] {
        GML_REQUIRE(d_samples && d_out_spins && d_out_counts && out_K, "null argument");
        GML_REQUIRE(ld >= M, "ld must be >= M");
        GML_CUDA(cudaSetDevice(device));
        *out_K = build_histogram(d_samples, M, N, ld, d_out_spins, ld_out, d_out_counts, (cudaStream_t)stream);
    });
}

int gml_b200_comm_unique_id(uint8_t* out128) {
    return guarded([&] {
        GML_REQUIRE(out128 != nullptr, "null argument");
        comm_unique_id(out128);
    });
}

int gml_b200_comm_init(gml_b200_handle* h, const uint8_t* id128, int32_t rank, int32_t world) {
    return guarded([&] {
        GML_REQUIRE(h && id128, "null argument");
        GML_CUDA(cudaSetDevice(h->device));
        if (h->owns_comm) comm_destroy(h->comm);
        h->comm = nullptr; h->owns_comm = false;
        h->comm = comm_create(id128, rank, world);
        h->owns_comm = true;
    });
}

int gml_b200_comm_attach(gml_b200_handle* h, gml_b200_handle* owner) {
    return guarded([&] {
        GML_REQUIRE(h && owner && owner->comm, "needs a handle and an owner handle with a communicator");
        GML_REQUIRE(h->device == owner->device, "the two handles must live on the same device");
        if (h->owns_comm) comm_destroy(h->comm);
        h->comm = owner->comm; h->owns_comm = false;
    });
}

int gml_b200_comm_globalize_histogram(gml_b200_handle* h) {
    return guarded([&] {
        GML_REQUIRE(h && h->has_hist && h->comm, "needs a resident histogram and gml_b200_comm_init");
        GML_CUDA(cudaSetDevice(h->device));
        comm_globalize_histogram(h->comm, h->hist, h->own_stream);
        GML_CUDA(cudaStreamSynchronize(h->own_stream));
    });
}

}  // extern "C"
