// Input generator (SURVEY 8f-2): multi-chain single-site Gibbs sampler for +-1 models, pairwise
//   p(s) ~ exp( sum_{i<j} J_ij s_i s_j + sum_i h_i s_i )
// and general term lists (3-body and higher: gibbs_terms_kernel below, the C4 input generator)
// The reference's `sample` enumerates all 2^N configurations (src/sampling.jl:34-57) and cannot
// produce the N = 100 / N = 1000 benchmark inputs; here every chain is one thread, its spins are
// bit-packed in thread-local words, and one sample per chain is emitted after `sweeps` sweeps from
// a random start.  Counter-based RNG: results depend only on (seed, chain, sweep, site).
#include <algorithm>

#include "common.cuh"

namespace gml {
namespace {

__device__ __forceinline__ uint32_t mix32(uint64_t x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL;
    x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL;
    x ^= x >> 33;
    return (uint32_t)(x >> 16);
}

template <int NW>
__global__ void __launch_bounds__(128) gibbs_kernel(int N, const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col,
                                                   const float* __restrict__ J, const float* __restrict__ hfield,
                                                   int64_t n_samples, int sweeps, uint64_t seed,
                                                   int8_t* __restrict__ out, int64_t ld) {
    const int64_t chain = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (chain >= n_samples) return;
    uint32_t s[NW];
    const uint64_t key = seed * 0x9E3779B97F4A7C15ULL + (uint64_t)chain * 0xD1B54A32D192ED03ULL;
#pragma unroll
    for (int w = 0; w < NW; ++w) s[w] = mix32(key + 0x1234567ULL * (w + 1)) ^ (mix32(key ^ (0xABCDEFULL * (w + 7))) << 16);
    for (int sw = 0; sw < sweeps; ++sw) {
        for (int i = 0; i < N; ++i) {
            float field = hfield[i];
            const int b = row_ptr[i], e = row_ptr[i + 1];
            for (int q = b; q < e; ++q) {
                const int j = col[q];
                const float sj = ((s[j >> 5] >> (j & 31)) & 1u) ? 1.f : -1.f;
                field = fmaf(J[q], sj, field);
            }
            const float p_up = 1.f / (1.f + __expf(-2.f * field));
            const uint32_t r = mix32(key + ((uint64_t)(sw * (int64_t)N + i + 1) << 20));
            const uint32_t bit = (r * 2.3283064365386963e-10f < p_up) ? 1u : 0u;
            s[i >> 5] = (s[i >> 5] & ~(1u << (i & 31))) | (bit << (i & 31));
        }
    }
    for (int i = 0; i < N; ++i) out[(int64_t)i * ld + chain] = ((s[i >> 5] >> (i & 31)) & 1u) ? 1 : -1;
}

// General +-1 models  p(s) ~ exp( sum_t w_t prod_{i in t} s_i )  (the reference's weigh_proba, src/sampling.jl:58-65):
// site i sees the local field  sum_{t containing i} w_t prod_{j in t, j != i} s_j.  Per-site incidence lists in CSR
// form: entry q of site i holds the weight and the (width) other members of one term (-1 padded).
template <int NW>
__global__ void __launch_bounds__(128) gibbs_terms_kernel(int N, int width, const int32_t* __restrict__ row_ptr,
                                                         const int32_t* __restrict__ others, const float* __restrict__ weight,
                                                         int64_t n_samples, int sweeps, uint64_t seed,
                                                         int8_t* __restrict__ out, int64_t ld) {
    const int64_t chain = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (chain >= n_samples) return;
    uint32_t s[NW];
    const uint64_t key = seed * 0x9E3779B97F4A7C15ULL + (uint64_t)chain * 0xD1B54A32D192ED03ULL;
#pragma unroll
    for (int w = 0; w < NW; ++w) s[w] = mix32(key + 0x1234567ULL * (w + 1)) ^ (mix32(key ^ (0xABCDEFULL * (w + 7))) << 16);
    for (int sw = 0; sw < sweeps; ++sw) {
        for (int i = 0; i < N; ++i) {
            float field = 0.f;
            const int b = row_ptr[i], e = row_ptr[i + 1];
            for (int q = b; q < e; ++q) {
                uint32_t neg = 0;                       // parity of the number of down spins among the other members
                for (int m = 0; m < width; ++m) {
                    const int j = others[(int64_t)q * width + m];
                    if (j >= 0) neg ^= ~(s[j >> 5] >> (j & 31)) & 1u;
                }
                field += neg ? -weight[q] : weight[q];
            }
            const float p_up = 1.f / (1.f + __expf(-2.f * field));
            const uint32_t r = mix32(key + ((uint64_t)(sw * (int64_t)N + i + 1) << 20));
            const uint32_t bit = (r * 2.3283064365386963e-10f < p_up) ? 1u : 0u;
            s[i >> 5] = (s[i >> 5] & ~(1u << (i & 31))) | (bit << (i & 31));
        }
    }
    for (int i = 0; i < N; ++i) out[(int64_t)i * ld + chain] = ((s[i >> 5] >> (i & 31)) & 1u) ? 1 : -1;
}

}  // namespace

Incidence build_incidence(int N, int order, int n_terms, const int32_t* term_idx) {
    Incidence inc;
    inc.width = std::max(1, order - 1);
    const int width = inc.width;
    inc.row_ptr.assign(N + 1, 0);
    for (int t = 0; t < n_terms; ++t)
        for (int m = 0; m < order; ++m) {
            const int i = term_idx[(size_t)t * order + m];
            if (i < 0) continue;
            GML_REQUIRE(i < N, "sampler term refers to a spin >= N");
            for (int m2 = 0; m2 < m; ++m2) GML_REQUIRE(term_idx[(size_t)t * order + m2] != i, "sampler term repeats a spin");
            ++inc.row_ptr[i + 1];
        }
    for (int i = 0; i < N; ++i) inc.row_ptr[i + 1] += inc.row_ptr[i];
    const int nnz = inc.row_ptr[N];
    inc.others.assign((size_t)std::max(nnz, 1) * width, -1);
    inc.term.assign(std::max(nnz, 1), -1);
    std::vector<int32_t> fill(inc.row_ptr.begin(), inc.row_ptr.end() - 1);
    for (int t = 0; t < n_terms; ++t)
        for (int m = 0; m < order; ++m) {
            const int i = term_idx[(size_t)t * order + m];
            if (i < 0) continue;
            const int q = fill[i]++;
            inc.term[q] = t;
            int w = 0;
            for (int m2 = 0; m2 < order; ++m2) {
                const int j = term_idx[(size_t)t * order + m2];
                if (j >= 0 && m2 != m) inc.others[(size_t)q * width + w++] = j;
            }
        }
    return inc;
}

void sample_gibbs_terms(int N, int width, const int32_t* d_row_ptr, const int32_t* d_others, const float* d_weight,
                        int64_t n_samples, int sweeps, uint64_t seed, int8_t* d_spins, int64_t ld, cudaStream_t st) {
    const unsigned grid = (unsigned)ceil_div(n_samples, 128);
    const int nw = (N + 31) / 32;
#define GML_GIBBS_T(NW) gibbs_terms_kernel<NW><<<grid, 128, 0, st>>>(N, width, d_row_ptr, d_others, d_weight, n_samples, sweeps, seed, d_spins, ld)
    if (nw <= 1) GML_GIBBS_T(1);
    else if (nw <= 4) GML_GIBBS_T(4);
    else if (nw <= 32) GML_GIBBS_T(32);
    else GML_GIBBS_T(128);
#undef GML_GIBBS_T
    GML_LAUNCHED();
}

void sample_gibbs(int N, const int32_t* d_row_ptr, const int32_t* d_col, const float* d_J, const float* d_h,
                  int /*max_deg*/, int64_t n_samples, int sweeps, uint64_t seed, int8_t* d_spins, int64_t ld,
                  cudaStream_t st) {
    const unsigned grid = (unsigned)ceil_div(n_samples, 128);
    const int nw = (N + 31) / 32;
#define GML_GIBBS(NW) gibbs_kernel<NW><<<grid, 128, 0, st>>>(N, d_row_ptr, d_col, d_J, d_h, n_samples, sweeps, seed, d_spins, ld)
    if (nw <= 1) GML_GIBBS(1);
    else if (nw <= 4) GML_GIBBS(4);
    else if (nw <= 32) GML_GIBBS(32);
    else GML_GIBBS(128);
#undef GML_GIBBS
    GML_LAUNCHED();
}

}  // namespace gml
