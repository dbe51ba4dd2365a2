// K5: small-problem solver.  fp64 proximal Newton (exact L1 minimiser) and damped barrier Newton
// (the log-barrier point Ipopt returns) for node problems with at most NEWTON_MAX_F (128) features.
//
// This is the device counterpart of what the reference asks Ipopt to do per node
// (src/GraphicalModelLearning.jl:164-181): every outer iteration evaluates f, grad f and the dense
// Hessian over the whole histogram -- here for ALL nodes at once, sample-parallel, in float64.
// Objectives follow :170 (RISE), :279 (logRISE), :317 (RPLE); the L1 term covers the coordinates
// whose penalty class is PEN_L1 (j != current_spin, :171; keys of length > 1, :118).
#include "common.cuh"

namespace gml {
namespace {

constexpr int TS = 128;        // samples per staged tile
constexpr int NT = 256;        // threads per accumulation CTA
constexpr int NALPHA = 12;     // step sizes 1, 1/2, ..., 2^-11 tried per line-search pass
// Barrier phase stall rule.  The phase stops at a Newton step below 1e-15, but at some nodes rounding keeps the step at a
// few 1e-15 (the direction is computed from fp64 sums over K rows) and the merit stops moving.  A node whose step stays
// below STALL_STEP with a merit change within the line search's summation slack for STALL_ITERS consecutive iterations
// is converged at the rounding floor: accepted and counted in stats.n_stalled, not run out to max_iter.
constexpr double STALL_STEP = 1e-13;
constexpr int STALL_ITERS = 4;

struct NewtonParams {
    const int8_t* Q;           // [Fp x Kp]
    const int8_t* base;        // spins live in rows of hist->base
    const double* w;           // [Kp]
    const int32_t* spin_row;   // [Nn]
    const uint8_t* pen;        // [Nn x Fp]
    const int32_t* feat;       // [Nn x Fp] per-node feature rows (reduced-space problems) or nullptr
    int64_t Kp;
    int F, Fp, Nn, chunks;
    int64_t chunk_len;         // multiple of TS
    double lambda, mu, tol;
    int barrier;               // 0 exact phase, 1 barrier phase
    double* x;                 // [Nn x Fp]
    double* d;                 // [Nn x Fp]
    double* part;              // [Nn x chunks x P]   P = 1 + F + F(F+1)/2
    double* part_ls;           // [Nn x chunks x NALPHA]
    double* fcur;              // [Nn] merit at x (smooth + penalty)
    double* slope;             // [Nn] model decrease / directional derivative
    double* obj;               // [Nn]
    double* resid;             // [Nn] last step size
    int* conv;                 // [Nn]
    int* idle;                 // [Nn] consecutive barrier iterations at the rounding floor (STALL_ITERS: stalled)
    int* n_active;             // [1]
};

__device__ __forceinline__ void sample_terms(int form, double t, double w, double& fterm, double& gw, double& hw) {
    if (form == GML_B200_RPLE) {
        const double a = -2.0 * t;
        fterm = w * (fmax(a, 0.0) + log1p(exp(-fabs(a))));
        const double sig = 1.0 / (1.0 + exp(2.0 * t));
        gw = 2.0 * w * sig;
        hw = 4.0 * w * sig * (1.0 - sig);
    } else {   // RISE and (unnormalised) logRISE
        const double e = w * exp(-t);
        fterm = e; gw = e; hw = e;
    }
}

__device__ __forceinline__ double sample_value(int form, double t, double w) {
    if (form == GML_B200_RPLE) {
        const double a = -2.0 * t;
        return w * (fmax(a, 0.0) + log1p(exp(-fabs(a))));
    }
    return w * exp(-t);
}

// f, g, H partial sums of one (chunk, node).  NE = owned accumulator entries per thread.
template <int NE>
__device__ __forceinline__ void newton_accum_body(const NewtonParams& p, int form, int u, int c) {
    const int F = p.F;
    const int P = 1 + F + F * (F + 1) / 2;
    __shared__ int8_t stat[TS][NEWTON_MAX_F];
    __shared__ double s_gw[TS], s_hw[TS];
    __shared__ double s_x[NEWTON_MAX_F];
    __shared__ double s_red[NT / 32];
    const int tid = threadIdx.x;
    __shared__ int s_feat[NEWTON_MAX_F];
    if (tid < F) {
        s_x[tid] = p.x[(int64_t)u * p.Fp + tid];
        s_feat[tid] = p.feat ? p.feat[(int64_t)u * p.Fp + tid] : tid;
    }

    // owned entries: e in [0,F) gradient, e >= F Hessian pair (a >= b)
    int ea[NE], eb[NE];
    double acc[NE];
#pragma unroll
    for (int i = 0; i < NE; ++i) {
        const int e = tid + i * NT;
        acc[i] = 0.0;
        ea[i] = -1; eb[i] = 0;
        if (e < F) { ea[i] = e; eb[i] = -1; }
        else if (e < P - 1) {
            const int q = e - F;
            int a = (int)((sqrt(8.0 * q + 1.0) - 1.0) * 0.5);
            while ((a + 1) * (a + 2) / 2 <= q) ++a;
            while (a * (a + 1) / 2 > q) --a;
            ea[i] = a; eb[i] = q - a * (a + 1) / 2;
        }
    }
    double fsum = 0.0;
    const int8_t* srow = p.base + (int64_t)p.spin_row[u] * p.Kp;
    const int64_t k_begin = (int64_t)c * p.chunk_len;
    const int64_t k_end = min(k_begin + p.chunk_len, p.Kp);
    __syncthreads();
    for (int64_t k0 = k_begin; k0 < k_end; k0 += TS) {
        if (tid < TS) {
            const int64_t k = k0 + tid;
            const int su = srow[k];
            double m = 0.0;
            for (int f = 0; f < F; ++f) {
                const int q = p.Q[(int64_t)s_feat[f] * p.Kp + k];
                stat[tid][f] = (int8_t)(su * q);
                m += s_x[f] * (double)q;
            }
            double ft, gw, hw;
            sample_terms(form, su * m, p.w[k], ft, gw, hw);
            fsum += ft;
            s_gw[tid] = gw; s_hw[tid] = hw;
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < NE; ++i) {
            if (ea[i] < 0) continue;
            double a = acc[i];
            if (eb[i] < 0) {
                for (int k = 0; k < TS; ++k) a -= s_gw[k] * (double)stat[k][ea[i]];
            } else {
                for (int k = 0; k < TS; ++k) a += s_hw[k] * (double)(stat[k][ea[i]] * stat[k][eb[i]]);
            }
            acc[i] = a;
        }
        __syncthreads();
    }
    for (int o = 16; o; o >>= 1) fsum += __shfl_xor_sync(0xffffffffu, fsum, o);
    if ((tid & 31) == 0) s_red[tid >> 5] = fsum;
    __syncthreads();
    double* out = p.part + ((int64_t)u * p.chunks + c) * P;
    if (tid == 0) {
        double s = 0.0;
        for (int i = 0; i < NT / 32; ++i) s += s_red[i];
        out[0] = s;
    }
#pragma unroll
    for (int i = 0; i < NE; ++i) {
        const int e = tid + i * NT;
        if (e < P - 1) out[1 + e] = acc[i];
    }
}
template <int NE>
__global__ void __launch_bounds__(NT) newton_accum_kernel(NewtonParams p, int form) {
    const int u = blockIdx.y, c = blockIdx.x;
    if (p.conv[u]) return;
    newton_accum_body<NE>(p, form, u, c);
}

__device__ __forceinline__ double barrier_phi(double x, double lam, double mu) {
    const double eps = mu / lam, r = sqrt(eps * eps + x * x), z = eps + r;
    return lam * z - mu * log(2.0 * eps * z);
}

// One CTA (128 threads >= NEWTON_MAX_F) per node: reduce partials, form the direction.
// mode 0: exact (coordinate descent on the L1 quadratic model)
// mode 1: barrier Newton (Cholesky)
// mode 2: barrier warm start (moves exact zeros to their first-order barrier value), no direction
// mode 3: objective only (obj[u] = f + lambda*|x_pen|_1)
constexpr int ND = 128;        // threads of the direction kernel: one per feature (F <= NEWTON_MAX_F = 128)
static_assert(ND >= NEWTON_MAX_F, "the direction kernel initialises one feature per thread");
// (runs with any block size >= F: strides follow blockDim.x -- 128 threads as a kernel of its own, 256 inside the fused one)
__device__ __forceinline__ void newton_direction_body(const NewtonParams& p, int form, int mode, int u) {
    const int F = p.F, tid = threadIdx.x;
    const int nthr = blockDim.x;
    const int P = 1 + F + F * (F + 1) / 2;
    extern __shared__ double sm[];
    double* H = sm;                       // F x F
    double* g = H + F * F;                // F
    double* x = g + F;                    // F
    double* d = x + F;                    // F
    double* Hd = d + F;                   // F
    __shared__ double s_f;
    __shared__ uint8_t s_pen[NEWTON_MAX_F];
    const double lam = p.lambda;

    for (int e = tid; e < P; e += nthr) {
        double s = 0.0;
        const double* src = p.part + (int64_t)u * p.chunks * P + e;
        for (int c = 0; c < p.chunks; ++c) s += src[(int64_t)c * P];
        if (e == 0) s_f = s;
        else if (e <= F) g[e - 1] = s;
        else {
            const int q = e - 1 - F;
            int a = (int)((sqrt(8.0 * q + 1.0) - 1.0) * 0.5);
            while ((a + 1) * (a + 2) / 2 <= q) ++a;
            while (a * (a + 1) / 2 > q) --a;
            const int b = q - a * (a + 1) / 2;
            H[a * F + b] = s; H[b * F + a] = s;
        }
    }
    if (tid < F) {
        x[tid] = p.x[(int64_t)u * p.Fp + tid];
        s_pen[tid] = p.pen[(int64_t)u * p.Fp + tid];
        d[tid] = 0.0; Hd[tid] = 0.0;
    }
    __syncthreads();
    double fval = s_f;
    if (form == GML_B200_LOGRISE) {
        const double Z = s_f;
        fval = log(Z);
        __syncthreads();
        if (tid < F) g[tid] /= Z;
        __syncthreads();
        for (int e = tid; e < F * F; e += nthr) H[e] = H[e] / Z - g[e / F] * g[e % F];
        __syncthreads();
    }
    // fixed-zero coordinates drop out of the model
    for (int e = tid; e < F * F; e += nthr) {
        const int a = e / F, b = e % F;
        if (s_pen[a] == PEN_ZERO || s_pen[b] == PEN_ZERO) H[e] = (a == b) ? 1.0 : 0.0;
    }
    if (tid < F && s_pen[tid] == PEN_ZERO) g[tid] = 0.0;
    __syncthreads();

    if (mode == 3) {
        if (tid == 0) {
            double l1 = 0.0;
            for (int j = 0; j < F; ++j) if (s_pen[j] == PEN_L1) l1 += fabs(x[j]);
            p.obj[u] = fval + lam * l1;
        }
        return;
    }
    if (mode == 2) {
        if (tid < F && s_pen[tid] == PEN_L1 && x[tid] == 0.0) {
            const double den = fmax(lam * lam - g[tid] * g[tid], 1e-300);
            p.x[(int64_t)u * p.Fp + tid] = -2.0 * p.mu * g[tid] / den;
        }
        return;
    }

    if (mode == 0) {
        // ---- cyclic coordinate descent, executed by warp 0 (lanes own rows lane, lane+32 of Hd)
        if (tid < 32) {
            const double cd_tol = 1e-16 + 1e-3 * p.tol;
            for (int sweep = 0; sweep < 10000; ++sweep) {
                double maxchg = 0.0;
                for (int j = 0; j < F; ++j) {
                    if (s_pen[j] == PEN_ZERO) continue;
                    const double a = fmax(H[j * F + j], 1e-300);
                    const double cur = x[j] + d[j];
                    double v = cur - (g[j] + Hd[j]) / a;
                    if (s_pen[j] == PEN_L1) {
                        const double av = fabs(v) - lam / a;
                        v = av > 0.0 ? copysign(av, v) : 0.0;
                    }
                    const double delta = v - cur;
                    __syncwarp();
                    if (delta != 0.0) {
                        if (tid == 0) d[j] += delta;
                        for (int i = tid; i < F; i += 32) Hd[i] += H[i * F + j] * delta;
                        maxchg = fmax(maxchg, fabs(delta));
                    }
                    __syncwarp();
                }
                if (maxchg < cd_tol) break;
            }
        }
        __syncthreads();
        if (tid == 0) {
            double step = 0.0, gd = 0.0, l1n = 0.0, l1o = 0.0;
            for (int j = 0; j < F; ++j) {
                step = fmax(step, fabs(d[j]));
                gd += g[j] * d[j];
                if (s_pen[j] == PEN_L1) { l1n += fabs(x[j] + d[j]); l1o += fabs(x[j]); }
            }
            p.fcur[u] = fval + lam * l1o;
            p.slope[u] = gd + lam * (l1n - l1o);
            p.resid[u] = step;
            if (step < p.tol) p.conv[u] = 2;   // final step is applied by the update kernel
        }
        __syncthreads();
        if (tid < F) p.d[(int64_t)u * p.Fp + tid] = d[tid];
        return;
    }

    // ---- mode 1: barrier Newton.  grad = g + phi', Hm = H + diag(phi''), solve Hm d = -grad
    const double eps = p.mu / lam;
    if (tid < F && s_pen[tid] == PEN_L1) {
        const double r = sqrt(eps * eps + x[tid] * x[tid]), z = eps + r;
        g[tid] += lam * x[tid] / z;
        H[tid * F + tid] += lam * (z - x[tid] * x[tid] / r) / (z * z);
    }
    __syncthreads();
    // Cholesky (lower) in place, column by column
    for (int j = 0; j < F; ++j) {
        if (tid == 0) {
            double s = H[j * F + j];
            for (int k = 0; k < j; ++k) s -= H[j * F + k] * H[j * F + k];
            H[j * F + j] = sqrt(fmax(s, 1e-300));
        }
        __syncthreads();
        const double l = H[j * F + j];
        for (int i = j + 1 + tid; i < F; i += nthr) {
            double t = H[i * F + j];
            for (int k = 0; k < j; ++k) t -= H[i * F + k] * H[j * F + k];
            H[i * F + j] = t / l;
        }
        __syncthreads();
    }
    if (tid == 0) {
        for (int i = 0; i < F; ++i) {
            double t = -g[i];
            for (int k = 0; k < i; ++k) t -= H[i * F + k] * d[k];
            d[i] = t / H[i * F + i];
        }
        for (int i = F - 1; i >= 0; --i) {
            double t = d[i];
            for (int k = i + 1; k < F; ++k) t -= H[k * F + i] * d[k];
            d[i] = t / H[i * F + i];
        }
        double slope = 0.0, pen = 0.0;
        for (int j = 0; j < F; ++j) {
            slope += g[j] * d[j];
            if (s_pen[j] == PEN_L1) pen += barrier_phi(x[j], lam, p.mu);
        }
        p.fcur[u] = fval + pen;
        p.slope[u] = slope;
    }
    __syncthreads();
    if (tid < F) p.d[(int64_t)u * p.Fp + tid] = d[tid];
}
__global__ void __launch_bounds__(ND) newton_direction_kernel(NewtonParams p, int form, int mode) {
    const int u = blockIdx.x;
    if (p.conv[u] && mode < 2) return;
    newton_direction_body(p, form, mode, u);
}

// smooth objective along x + alpha_i d for all alpha_i at once (energies are linear in x)
__device__ __forceinline__ void newton_linesearch_body(const NewtonParams& p, int form, int n_alpha, int u, int c) {
    const int F = p.F, tid = threadIdx.x;
    __shared__ double s_x[NEWTON_MAX_F], s_d[NEWTON_MAX_F];
    __shared__ double s_red[NT / 32][NALPHA];
    __shared__ int s_feat[NEWTON_MAX_F];
    if (tid < F) {
        s_x[tid] = p.x[(int64_t)u * p.Fp + tid]; s_d[tid] = p.d[(int64_t)u * p.Fp + tid];
        s_feat[tid] = p.feat ? p.feat[(int64_t)u * p.Fp + tid] : tid;
    }
    __syncthreads();
    double acc[NALPHA];
#pragma unroll
    for (int i = 0; i < NALPHA; ++i) acc[i] = 0.0;
    const int8_t* srow = p.base + (int64_t)p.spin_row[u] * p.Kp;
    const int64_t k_begin = (int64_t)c * p.chunk_len;
    const int64_t k_end = min(k_begin + p.chunk_len, p.Kp);
    for (int64_t k = k_begin + tid; k < k_end; k += NT) {
        const double su = srow[k];
        double mx = 0.0, md = 0.0;
        for (int f = 0; f < F; ++f) {
            const double q = p.Q[(int64_t)s_feat[f] * p.Kp + k];
            mx += s_x[f] * q; md += s_d[f] * q;
        }
        const double w = p.w[k];
        double alpha = 1.0;
#pragma unroll
        for (int i = 0; i < NALPHA; ++i) {
            if (i < n_alpha) acc[i] += sample_value(form, su * (mx + alpha * md), w);
            alpha *= 0.5;
        }
    }
#pragma unroll
    for (int i = 0; i < NALPHA; ++i) {
        double v = acc[i];
        for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((tid & 31) == 0) s_red[tid >> 5][i] = v;
    }
    __syncthreads();
    if (tid < NALPHA) {
        double s = 0.0;
        for (int i = 0; i < NT / 32; ++i) s += s_red[i][tid];
        p.part_ls[((int64_t)u * p.chunks + c) * NALPHA + tid] = s;
    }
}
__global__ void __launch_bounds__(NT) newton_linesearch_kernel(NewtonParams p, int form, int n_alpha) {
    const int u = blockIdx.y, c = blockIdx.x;
    if (p.conv[u] == 1) return;
    newton_linesearch_body(p, form, n_alpha, u, c);
}

// one warp per node: pick the first alpha that passes Armijo, update x, flag convergence
__device__ __forceinline__ void newton_update_body(const NewtonParams& p, int form, int n_alpha, int u, int lane) {
    if (p.conv[u] == 1) return;
    const int F = p.F;
    const double lam = p.lambda;
    double* x = p.x + (int64_t)u * p.Fp;
    const double* d = p.d + (int64_t)u * p.Fp;
    const uint8_t* pen = p.pen + (int64_t)u * p.Fp;
    if (p.conv[u] == 2) {   // converged this iteration: apply the last (tiny) step
        for (int j = lane; j < F; j += 32) x[j] += d[j];
        __syncwarp();
        if (lane == 0) p.conv[u] = 1;
        return;
    }
    double chosen = 0.0, last_merit = 0.0, last_alpha = 0.0;
    bool found = false;
    double alpha = 1.0;
    for (int i = 0; i < n_alpha && !found; ++i) {
        double s = 0.0;
        for (int c = lane; c < p.chunks; c += 32) s += p.part_ls[((int64_t)u * p.chunks + c) * NALPHA + i];
        double penv = 0.0;
        for (int j = lane; j < F; j += 32) if (pen[j] == PEN_L1) {
            const double xn = x[j] + alpha * d[j];
            penv += p.barrier ? barrier_phi(xn, lam, p.mu) : lam * fabs(xn);
        }
        for (int o = 16; o; o >>= 1) {
            s += __shfl_xor_sync(0xffffffffu, s, o);
            penv += __shfl_xor_sync(0xffffffffu, penv, o);
        }
        const double fv = (form == GML_B200_LOGRISE) ? log(s) : s;
        const double merit = fv + penv;
        const double f0 = p.fcur[u];
        // fp64 summation noise of the two passes (different reduction orders) is ~1e-14 |f|
        const double slack = 1e-13 * fmax(fabs(f0), 1.0);
        last_merit = merit; last_alpha = alpha;
        if (merit <= f0 + 1e-4 * alpha * p.slope[u] + slack) { found = true; chosen = alpha; }
        else alpha *= 0.5;
    }
    if (!found) {
        // Armijo failed down to 2^-(n_alpha-1): keep descending if the smallest step still lowers the
        // merit, otherwise the iterate is numerically stationary.
        if (last_merit < p.fcur[u]) chosen = last_alpha;
        else { if (lane == 0) p.conv[u] = 1; return; }
    }
    double step = 0.0;
    for (int j = lane; j < F; j += 32) {
        const double dx = chosen * d[j];
        x[j] += dx;
        step = fmax(step, fabs(dx));
    }
    for (int o = 16; o; o >>= 1) step = fmax(step, __shfl_xor_sync(0xffffffffu, step, o));
    if (lane == 0) {
        p.resid[u] = step;
        bool done = false;
        if (p.barrier) {
            const double f0 = p.fcur[u];
            const bool flat = step >= p.tol && step < STALL_STEP && fabs(f0 - last_merit) <= 1e-13 * fmax(fabs(f0), 1.0);
            p.idle[u] = flat ? p.idle[u] + 1 : 0;
            done = step < p.tol || p.idle[u] >= STALL_ITERS;
        }
        if (done) p.conv[u] = 1;
        else atomicAdd(p.n_active, 1);
    }
}

__global__ void newton_update_kernel(NewtonParams p, int form, int n_alpha) {
    const int u = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
    if (u >= p.Nn) return;
    newton_update_body(p, form, n_alpha, u, threadIdx.x & 31);
}

// K5, single-launch form (SURVEY 7.3-7): for tiny problems -- a handful of nodes, a histogram of at most 2048 rows (the
// README example, the reference's test fixtures), <= 32 features -- the four kernels of a Newton iteration and the host
// read between iterations cost more than the arithmetic.  One CTA per node runs the WHOLE solve: exact phase, optional barrier warm start + barrier phase, final
// objective; the stages are the same device functions as above (one chunk = the whole histogram), separated by block
// barriers, exchanging their partial sums through the same global scratch.  info[2u] = iterations, info[2u+1] = 1 when a
// phase ran out of iterations.
template <int NE>
__global__ void __launch_bounds__(NT) newton_small_kernel(NewtonParams p, int form, int max_iter, double tol_exact, int* __restrict__ info) {
    const int u = blockIdx.x, tid = threadIdx.x;
    int iters = 0, unconv = 0;
    for (int phase = 0; phase < 2; ++phase) {
        if (phase == 1) {
            if (!(p.mu > 0.0 && p.lambda > 0.0)) break;
            // exact zeros -> their first-order barrier value (direction mode 2), then damped Newton on f + sum phi_mu
            if (tid == 0) p.conv[u] = 0;
            __syncthreads();
            newton_accum_body<NE>(p, form, u, 0);
            __syncthreads();
            newton_direction_body(p, form, 2, u);
            __syncthreads();
        }
        p.barrier = phase;
        p.tol = phase ? 1e-15 : tol_exact;
        int it = 0;
        for (; it < max_iter; ++it) {
            newton_accum_body<NE>(p, form, u, 0);
            __syncthreads();
            newton_direction_body(p, form, phase, u);
            __syncthreads();
            newton_linesearch_body(p, form, NALPHA, u, 0);
            __syncthreads();
            if (tid < 32) newton_update_body(p, form, NALPHA, u, tid);
            __syncthreads();
            if (p.conv[u] == 1) { ++it; break; }
        }
        iters += it;
        if (p.conv[u] != 1) unconv = 1;
        __syncthreads();
    }
    // objective at the returned point
    if (tid == 0) p.conv[u] = 0;
    __syncthreads();
    newton_accum_body<NE>(p, form, u, 0);
    __syncthreads();
    newton_direction_body(p, form, 3, u);
    if (tid == 0) { info[2 * u] = iters; info[2 * u + 1] = unconv; }
}

void launch_accum(const NewtonParams& P, int form, cudaStream_t st) {
    const int Ptot = P.F + P.F * (P.F + 1) / 2;
    const int ne = (int)ceil_div(Ptot, NT);
    dim3 grid(P.chunks, P.Nn);
    if (ne <= 1) newton_accum_kernel<1><<<grid, NT, 0, st>>>(P, form);
    else if (ne <= 2) newton_accum_kernel<2><<<grid, NT, 0, st>>>(P, form);
    else if (ne <= 3) newton_accum_kernel<3><<<grid, NT, 0, st>>>(P, form);
    else if (ne <= 5) newton_accum_kernel<5><<<grid, NT, 0, st>>>(P, form);
    else if (ne <= 9) newton_accum_kernel<9><<<grid, NT, 0, st>>>(P, form);
    else if (ne <= 17) newton_accum_kernel<17><<<grid, NT, 0, st>>>(P, form);
    else newton_accum_kernel<33><<<grid, NT, 0, st>>>(P, form);      // F <= 128: F + F(F+1)/2 <= 33 * 256
    GML_LAUNCHED();
}

// nodes whose barrier phase stopped at the rounding floor (synchronises the stream)
int count_stalled(const int* d_idle, int Nn, cudaStream_t st) {
    std::vector<int> h(Nn);
    GML_CUDA(cudaMemcpyAsync(h.data(), d_idle, sizeof(int) * Nn, cudaMemcpyDeviceToHost, st));
    GML_CUDA(cudaStreamSynchronize(st));
    int n = 0;
    for (int v : h) n += v >= STALL_ITERS;
    return n;
}

}  // namespace

void solve_newton(const NodeProblem& prob, const gml_b200_opts& o, SolveResult& r, cudaStream_t st) {
    const Histogram& h = *prob.hist;
    const int F = prob.F, Fp = prob.Fp, Nn = prob.Nn;
    GML_REQUIRE(F <= NEWTON_MAX_F, "Newton solver supports at most 128 features per node");
    const int Ptot = 1 + F + F * (F + 1) / 2;
    // tiny problems: the whole solve in ONE launch, one CTA per node (newton_small_kernel).  Measured: C0 (K = 8) 0.41 -> 0.29 ms
    // per learn(); at C1 size (K = 18 700) one CTA per node sweeping the histogram alone is 5x SLOWER than the chunked
    // kernels (9.7 against 1.9 ms), hence the small row limit.
    const bool fused = F <= 32 && h.Kp <= 2048 && !std::getenv("GML_B200_NO_FUSED_NEWTON");
    int64_t chunks = ceil_div(h.Kp, 1024);
    chunks = std::min<int64_t>(chunks, std::max<int64_t>(1, 1184 / Nn));
    chunks = std::min<int64_t>(chunks, std::max<int64_t>(1, (int64_t)(1 << 24) / ((int64_t)Nn * Ptot)));
    if (fused) chunks = 1;
    const int64_t chunk_len = round_up(ceil_div(h.Kp, chunks), TS);
    chunks = ceil_div(h.Kp, chunk_len);

    DevBuf<double> d, part, part_ls, fcur, slope, resid;
    DevBuf<int> conv, idle, n_active;
    r.x.alloc((size_t)Nn * Fp);
    r.objective.alloc(Nn);
    d.alloc((size_t)Nn * Fp);
    part.alloc((size_t)Nn * chunks * Ptot);
    part_ls.alloc((size_t)Nn * chunks * NALPHA);
    fcur.alloc(Nn); slope.alloc(Nn); resid.alloc(Nn);
    conv.alloc(Nn); idle.alloc(Nn); n_active.alloc(1);
    if (prob.x0) GML_CUDA(cudaMemcpyAsync(r.x.p, prob.x0, sizeof(double) * Nn * Fp, cudaMemcpyDeviceToDevice, st));
    else GML_CUDA(cudaMemsetAsync(r.x.p, 0, sizeof(double) * Nn * Fp, st));
    GML_CUDA(cudaMemsetAsync(d.p, 0, sizeof(double) * Nn * Fp, st));
    GML_CUDA(cudaMemsetAsync(conv.p, 0, sizeof(int) * Nn, st));
    GML_CUDA(cudaMemsetAsync(idle.p, 0, sizeof(int) * Nn, st));
    GML_CUDA(cudaMemsetAsync(resid.p, 0, sizeof(double) * Nn, st));

    NewtonParams P{};
    P.Q = prob.Q; P.base = h.base.p; P.w = h.w64.p; P.spin_row = prob.spin_row.p; P.pen = prob.pen.p; P.feat = prob.feat;
    P.Kp = h.Kp; P.F = F; P.Fp = Fp; P.Nn = Nn; P.chunks = (int)chunks; P.chunk_len = chunk_len;
    P.lambda = prob.lambda; P.mu = o.barrier_mu;
    P.x = r.x.p; P.d = d.p; P.part = part.p; P.part_ls = part_ls.p; P.fcur = fcur.p; P.slope = slope.p;
    P.obj = r.objective.p; P.resid = resid.p; P.conv = conv.p; P.idle = idle.p; P.n_active = n_active.p;

    const size_t dir_smem = sizeof(double) * ((size_t)F * F + 4 * F);
    const int form = prob.form;
    const int max_iter = o.max_iter > 0 ? o.max_iter : 200;
    int total_iter = 0, n_fg = 0, n_f = 0, active = Nn;

    auto run_phase = [&](int barrier, double tol) {
        P.barrier = barrier; P.tol = tol;
        for (int it = 0; it < max_iter; ++it) {
            ++total_iter;
            launch_accum(P, form, st); ++n_fg;
            newton_direction_kernel<<<Nn, ND, dir_smem, st>>>(P, form, barrier ? 1 : 0);
            GML_LAUNCHED();
            newton_linesearch_kernel<<<dim3(P.chunks, Nn), NT, 0, st>>>(P, form, NALPHA);
            GML_LAUNCHED(); ++n_f;
            GML_CUDA(cudaMemsetAsync(n_active.p, 0, sizeof(int), st));
            newton_update_kernel<<<(unsigned)ceil_div(Nn, 4), 128, 0, st>>>(P, form, NALPHA);
            GML_LAUNCHED();
            GML_CUDA(cudaMemcpyAsync(&active, n_active.p, sizeof(int), cudaMemcpyDeviceToHost, st));
            GML_CUDA(cudaStreamSynchronize(st));
            if (active == 0) break;
        }
    };

    if (dir_smem > 48 * 1024)
        GML_CUDA(cudaFuncSetAttribute(newton_direction_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dir_smem));

    const double tol_exact = o.tol > 0 ? o.tol : 1e-12;
    if (fused) {
        DevBuf<int> info;
        info.alloc((size_t)2 * Nn);
        const int ne = (int)ceil_div(Ptot - 1, NT);
        if (ne <= 1) newton_small_kernel<1><<<Nn, NT, dir_smem, st>>>(P, form, max_iter, tol_exact, info.p);
        else if (ne <= 2) newton_small_kernel<2><<<Nn, NT, dir_smem, st>>>(P, form, max_iter, tol_exact, info.p);
        else newton_small_kernel<3><<<Nn, NT, dir_smem, st>>>(P, form, max_iter, tol_exact, info.p);
        GML_LAUNCHED();
        std::vector<int> hinfo((size_t)2 * Nn);
        std::vector<double> hres(Nn);
        GML_CUDA(cudaMemcpyAsync(hinfo.data(), info.p, sizeof(int) * 2 * Nn, cudaMemcpyDeviceToHost, st));
        GML_CUDA(cudaMemcpyAsync(hres.data(), resid.p, sizeof(double) * Nn, cudaMemcpyDeviceToHost, st));
        const int stalled = count_stalled(idle.p, Nn, st);
        int unconv = 0, iters = 0;
        double mr = 0.0;
        for (int u = 0; u < Nn; ++u) { iters = std::max(iters, hinfo[2 * u]); unconv += hinfo[2 * u + 1]; mr = std::max(mr, hres[u]); }
        const bool two_phase = o.barrier_mu > 0.0 && prob.lambda > 0.0;
        r.iterations = iters; r.n_fg = iters + (two_phase ? 2 : 1); r.n_f = iters; r.n_unconverged = unconv; r.max_residual = mr;
        r.n_stalled = stalled;
        return;
    }
    run_phase(0, tol_exact);
    int unconverged = active;
    if (o.barrier_mu > 0.0 && prob.lambda > 0.0) {
        GML_CUDA(cudaMemsetAsync(conv.p, 0, sizeof(int) * Nn, st));
        launch_accum(P, form, st); ++n_fg;
        newton_direction_kernel<<<Nn, ND, dir_smem, st>>>(P, form, 2);
        GML_LAUNCHED();
        run_phase(1, 1e-15);
        unconverged += active;
    }
    // final objective at the returned point
    GML_CUDA(cudaMemsetAsync(conv.p, 0, sizeof(int) * Nn, st));
    launch_accum(P, form, st); ++n_fg;
    newton_direction_kernel<<<Nn, ND, dir_smem, st>>>(P, form, 3);
    GML_LAUNCHED();

    std::vector<double> hres(Nn);
    GML_CUDA(cudaMemcpyAsync(hres.data(), resid.p, sizeof(double) * Nn, cudaMemcpyDeviceToHost, st));
    const int stalled = count_stalled(idle.p, Nn, st);
    double mr = 0.0;
    for (double v : hres) mr = std::max(mr, v);
    r.iterations = total_iter; r.n_fg = n_fg; r.n_f = n_f; r.n_unconverged = unconverged; r.max_residual = mr;
    r.n_stalled = stalled;
}

}  // namespace gml
