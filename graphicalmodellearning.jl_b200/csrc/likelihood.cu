// Maximum-likelihood refit of a model's weights on its own terms (fit_likelihood): maximise
//   l(w) = sum_t w_t m^_t - log Z(w) - lambda sum_{|t| >= 2} |w_t|
// from the data moments m^_t, starting at gm's weights.  Its stationarity condition is <phi_t>_model = m^_t on every
// unpenalised term.
//   - MCMC (B200Gibbs): stochastic maximum likelihood with persistent chains (Younes 1989; Tieleman 2008).  burn_in
//     sweeps at the initial weights, then per step s, with no host synchronisation: (1) the PERSIST kernel advances every
//     chain by `thin` sweeps of one long run; (2) record_key_sums reduces the chains' final states to integer sums S_g, n_g
//     over gm's terms; (3) update_kernel (one CTA) forms g_t = m^_t - sum S / sum n, takes the diagonally preconditioned
//     proximal step w_t <- prox(w_t + eta_s g_t / d_t), d_t = max(1 - m^_t^2, FISHER_FLOOR), soft threshold eta_s lambda /
//     d_t on |t| >= 2, keeps the Polyak-Ruppert running mean of w over steps s >= h = floor(steps / 2) together with the
//     int64 totals of the sums, writes fl32(w) to the chains' term weights and trace[s] = max_t |g_t|; (4)
//     refresh_kernel copies the term weights to the incidence entries.  eta_s = eta_0 (1 + s / S0)^-0.6.  Every sum is an
//     integer or is taken per term in step order, so the result depends only on (model, data moments, lambda, chains,
//     burn_in, thin, steps, eta_0, seed); there are no atomics.
//   - Exact (B200Exact, N <= 40): FISTA with backtracking and gradient-based adaptive restart on -l; each evaluation is one
//     enumeration pass that returns log Z and the moments of gm's terms (moments_exact).
#include <cmath>

#include "common.cuh"

namespace gml {
namespace {

constexpr int UPDATE_THREADS = 1024;

// w, avg, S_tot, n_tot, term_w and trace: see the top.  One CTA; thread t owns terms t, t + 1024, ...
__global__ void __launch_bounds__(UPDATE_THREADS) update_kernel(int n_terms, int G, const long long* __restrict__ S,
                                                                const long long* __restrict__ n_g, const double* __restrict__ data_mean,
                                                                const uint8_t* __restrict__ penalised, double eta, double lambda,
                                                                int64_t s, int64_t h, double* __restrict__ w, double* __restrict__ avg,
                                                                long long* __restrict__ S_tot, long long* __restrict__ n_tot,
                                                                float* __restrict__ term_w, double* __restrict__ trace) {
    __shared__ double red[UPDATE_THREADS / 32];
    long long n = 0;
    for (int g = 0; g < G; ++g) n += n_g[g];
    const bool window = s >= h;
    double gmax = 0.0;
    for (int t = threadIdx.x; t < n_terms; t += UPDATE_THREADS) {
        long long sum = 0;
        for (int g = 0; g < G; ++g) sum += S[(int64_t)g * n_terms + t];
        const double m = data_mean[t];
        const double grad = m - (double)sum / (double)n;
        const double d = fmax(1.0 - m * m, FISHER_FLOOR);
        double x = w[t] + eta * grad / d;
        if (penalised[t]) x = copysign(fmax(fabs(x) - eta * lambda / d, 0.0), x);
        w[t] = x;
        if (window) {
            avg[t] += (x - avg[t]) / (double)(s - h + 1);     // exact while x stays the same
            S_tot[t] += sum;
        }
        term_w[t] = (float)x;
        gmax = fmax(gmax, fabs(grad));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) gmax = fmax(gmax, __shfl_xor_sync(0xffffffffu, gmax, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = gmax;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < UPDATE_THREADS / 32; ++k) gmax = fmax(gmax, red[k]);
        trace[s] = gmax;
        if (window) *n_tot += n;
    }
}

// weight[q] = term_w[term[q]] for every incidence entry (term -1: padding, weight 0)
__global__ void refresh_kernel(int64_t nnz, const int32_t* __restrict__ term, const float* __restrict__ term_w,
                               float* __restrict__ weight) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q < nnz) weight[q] = term[q] >= 0 ? term_w[term[q]] : 0.f;
}

}  // namespace

double fit_step_size(double eta0, int64_t s) { return eta0 * std::pow(1.0 + (double)s / FIT_STEP_S0, -0.6); }

void fit_likelihood_mcmc(int N, int order, const std::vector<int32_t>& term_idx, const std::vector<double>& init_weight,
                         const Incidence& inc, const std::vector<double>& data_mean, const std::vector<uint8_t>& penalised,
                         double lambda, int64_t chains, int64_t burn_in, int64_t thin, int64_t steps, double eta0, uint64_t seed,
                         double* out_weight, double* out_model_moments, double* out_trace, cudaStream_t st) {
    const int n_terms = (int)init_weight.size();
    PersistentChains chains_(N, order, term_idx, init_weight, inc, chains, seed, st);
    const int G = record_groups(chains_.warps);
    DevBuf<int32_t> d_idx, d_term;
    DevBuf<long long> n_g, S, S_tot, n_tot;
    DevBuf<double> dm, w, avg, trace;
    DevBuf<uint8_t> pen;
    d_idx.alloc(term_idx.size()); d_term.alloc(inc.term.size());
    n_g.alloc(G); S.alloc((size_t)G * n_terms); S_tot.alloc(n_terms); n_tot.alloc(1);
    dm.alloc(n_terms); w.alloc(n_terms); avg.alloc(n_terms); trace.alloc(steps); pen.alloc(n_terms);
    GML_CUDA(cudaMemcpyAsync(d_idx.p, term_idx.data(), sizeof(int32_t) * term_idx.size(), cudaMemcpyHostToDevice, st));
    GML_CUDA(cudaMemcpyAsync(d_term.p, inc.term.data(), sizeof(int32_t) * inc.term.size(), cudaMemcpyHostToDevice, st));
    GML_CUDA(cudaMemcpyAsync(dm.p, data_mean.data(), sizeof(double) * n_terms, cudaMemcpyHostToDevice, st));
    GML_CUDA(cudaMemcpyAsync(w.p, init_weight.data(), sizeof(double) * n_terms, cudaMemcpyHostToDevice, st));
    GML_CUDA(cudaMemcpyAsync(pen.p, penalised.data(), n_terms, cudaMemcpyHostToDevice, st));
    GML_CUDA(cudaMemsetAsync(avg.p, 0, sizeof(double) * n_terms, st));
    GML_CUDA(cudaMemsetAsync(S_tot.p, 0, sizeof(long long) * n_terms, st));
    GML_CUDA(cudaMemsetAsync(n_tot.p, 0, sizeof(long long), st));

    const int64_t h = steps / 2, nnz = (int64_t)inc.term.size();
    if (burn_in > 0) chains_.run(0, burn_in, st);
    for (int64_t s = 0; s < steps; ++s) {
        chains_.run(burn_in + s * thin, thin, st);
        record_key_sums(chains_.record, N, 1, chains_.warps, order, n_terms, d_idx.p, n_g.p, S.p, st);
        update_kernel<<<1, UPDATE_THREADS, 0, st>>>(n_terms, G, S.p, n_g.p, dm.p, pen.p, fit_step_size(eta0, s), lambda, s, h,
                                                    w.p, avg.p, S_tot.p, n_tot.p, chains_.term_w, trace.p);
        GML_LAUNCHED();
        refresh_kernel<<<(unsigned)ceil_div(nnz, 256), 256, 0, st>>>(nnz, d_term.p, chains_.term_w, chains_.weight);
        GML_LAUNCHED();
    }
    std::vector<long long> s_tot(n_terms);
    long long total = 0;
    GML_CUDA(cudaMemcpyAsync(out_weight, avg.p, sizeof(double) * n_terms, cudaMemcpyDeviceToHost, st));
    GML_CUDA(cudaMemcpyAsync(s_tot.data(), S_tot.p, sizeof(long long) * n_terms, cudaMemcpyDeviceToHost, st));
    GML_CUDA(cudaMemcpyAsync(&total, n_tot.p, sizeof(long long), cudaMemcpyDeviceToHost, st));
    if (out_trace) GML_CUDA(cudaMemcpyAsync(out_trace, trace.p, sizeof(double) * steps, cudaMemcpyDeviceToHost, st));
    GML_CUDA(cudaStreamSynchronize(st));
    if (out_model_moments)                                   // divided as moments.cu's finalize_kernel divides
        for (int t = 0; t < n_terms; ++t) out_model_moments[t] = (double)s_tot[t] / (double)total;
}

bool fit_likelihood_exact(int N, const std::vector<uint64_t>& masks, const std::vector<double>& init_weight,
                          const std::vector<double>& data_mean, const std::vector<uint8_t>& penalised, double lambda, double tol,
                          int max_iter, double* out_weight, double* out_objective, int* out_iterations, cudaStream_t st) {
    const size_t n = init_weight.size();
    // f(w) = log Z(w) - sum_t w_t m^_t and its gradient m(w) - m^ from one enumeration pass
    auto eval = [&](const std::vector<double>& w, std::vector<double>& grad) {
        double log_z = 0.0;
        moments_exact(N, masks, w, masks, grad.data(), st, &log_z);
        double f = log_z;
        for (size_t t = 0; t < n; ++t) { f -= w[t] * data_mean[t]; grad[t] -= data_mean[t]; }
        return f;
    };
    auto penalty = [&](const std::vector<double>& w) {
        double p = 0.0;
        for (size_t t = 0; t < n; ++t) if (penalised[t]) p += std::fabs(w[t]);
        return lambda * p;
    };
    std::vector<double> x = init_weight, y = x, x_new(n), g_y(n), g_x(n);
    double f_y = eval(y, g_y), L = 1.0, t_k = 1.0, f_x = 0.0;
    bool converged = false;
    int it = 0;
    while (it < max_iter) {
        ++it;
        double mapping = 0.0;
        for (;;) {                                           // backtracking on the quadratic upper bound at y
            for (size_t t = 0; t < n; ++t) {
                const double z = y[t] - g_y[t] / L;
                x_new[t] = penalised[t] ? std::copysign(std::fmax(std::fabs(z) - lambda / L, 0.0), z) : z;
            }
            f_x = eval(x_new, g_x);
            double lin = 0.0, sq = 0.0;
            mapping = 0.0;
            for (size_t t = 0; t < n; ++t) {
                const double d = x_new[t] - y[t];
                lin += g_y[t] * d; sq += d * d;
                mapping = std::fmax(mapping, std::fabs(d));
            }
            // the slack absorbs the rounding of the two log Z values, which dominates once the steps are tiny
            if (f_x <= f_y + lin + 0.5 * L * sq + 64.0 * 2.2e-16 * (std::fabs(f_y) + 1.0)) break;
            L *= 2.0;
        }
        mapping *= L;                                        // max-norm of the prox-gradient mapping L (y - x_new)
        if (mapping <= tol) { x = x_new; converged = true; break; }
        double restart = 0.0;                                // gradient scheme of O'Donoghue & Candes (2015)
        for (size_t t = 0; t < n; ++t) restart += (y[t] - x_new[t]) * (x_new[t] - x[t]);
        if (restart > 0.0) {
            t_k = 1.0;
            x = x_new; y = x_new; f_y = f_x; g_y = g_x;
            continue;
        }
        const double t_next = 0.5 * (1.0 + std::sqrt(1.0 + 4.0 * t_k * t_k));
        for (size_t t = 0; t < n; ++t) y[t] = x_new[t] + (t_k - 1.0) / t_next * (x_new[t] - x[t]);
        x = x_new; t_k = t_next;
        f_y = eval(y, g_y);
    }
    std::copy(x.begin(), x.end(), out_weight);
    if (out_objective) *out_objective = -(f_x + penalty(x));
    if (out_iterations) *out_iterations = it;
    return converged;
}

}  // namespace gml
