// K1: histogram validation + device layout build.
// Replaces data_info (src/GraphicalModelLearning.jl:76-81), the weights samples[k,1]/num_samples
// (:170) and the per-node nodal_stat allocations (:162, :94-108) of the reference: the +-1 feature
// matrix is built ONCE, shared by all nodes, and the node sign s_u is applied inside the kernels.
#include "common.cuh"

namespace gml {

namespace {

// flags: bit0 = spin not +-1, bit1 = count <= 0 or non-finite
__global__ void pack_spins_kernel(const int8_t* __restrict__ in, int64_t ld, int64_t K, int64_t Kp, int N,
                                  int Fb, int8_t* __restrict__ base, int* __restrict__ flags) {
    const int row = blockIdx.y;
    int8_t* dst = base + (int64_t)row * Kp;
    const int64_t k0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 16;
    if (k0 >= Kp) return;
    int8_t v[16];
    if (row < N) {
        const int8_t* src = in + (int64_t)row * ld;
        bool bad = false;
        if (k0 + 16 <= K && ((reinterpret_cast<uintptr_t>(src + k0) & 15) == 0)) {
            int4 q = *reinterpret_cast<const int4*>(src + k0);
            memcpy(v, &q, 16);
#pragma unroll
            for (int j = 0; j < 16; ++j) bad |= (v[j] != 1 && v[j] != -1);
        } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                if (k0 + j < K) { v[j] = src[k0 + j]; bad |= (v[j] != 1 && v[j] != -1); }
                else v[j] = 1;
            }
        }
        if (bad) atomicOr(flags, 1);
    } else {
        const int8_t fill = (row == N) ? 1 : 0;
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = fill;
    }
    int4 q;
    memcpy(&q, v, 16);
    *reinterpret_cast<int4*>(dst + k0) = q;
}

__global__ void count_stats_kernel(const double* __restrict__ counts, int64_t K, double* __restrict__ sum,
                                   double* __restrict__ cmax, int* __restrict__ flags) {
    double s = 0.0, m = 0.0;
    bool bad = false;
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < K; k += (int64_t)gridDim.x * blockDim.x) {
        double c = counts[k];
        bad |= !(c > 0.0) || !isfinite(c);
        s += c;
        m = fmax(m, c);
    }
    for (int o = 16; o; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(sum, s);
        // counts are positive: ordering of the bit patterns equals ordering of the values
        atomicMax(reinterpret_cast<unsigned long long*>(cmax), (unsigned long long)__double_as_longlong(m));
    }
    if (bad) atomicOr(flags, 2);
}

__global__ void weights_kernel(const double* __restrict__ counts, int64_t K, int64_t Kp,
                               const double* __restrict__ sum, double* __restrict__ w64, float* __restrict__ w32) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= Kp) return;
    const double w = (k < K) ? counts[k] / *sum : 0.0;
    w64[k] = w;
    w32[k] = (float)w;
}

// Q [Fp x Kp] -> P [Kp x Fp], 64x64 byte tiles through shared memory
__global__ void transpose_i8_kernel(const int8_t* __restrict__ Q, int8_t* __restrict__ P, int Fp, int64_t Kp) {
    __shared__ int8_t tile[64][64 + 4];
    const int64_t k0 = (int64_t)blockIdx.x * 64;
    const int f0 = blockIdx.y * 64;
    // load: 64 feature rows x 64 samples; thread (ty, tx): row ty+16*i, 4 bytes at tx*4
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;   // 256 threads: 16 x 16
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = ty + 16 * i;
        const char4 v = *reinterpret_cast<const char4*>(Q + (int64_t)(f0 + r) * Kp + k0 + tx * 4);
        tile[r][tx * 4 + 0] = v.x; tile[r][tx * 4 + 1] = v.y; tile[r][tx * 4 + 2] = v.z; tile[r][tx * 4 + 3] = v.w;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = ty + 16 * i;   // sample within tile
        char4 v;
        v.x = tile[tx * 4 + 0][r]; v.y = tile[tx * 4 + 1][r]; v.z = tile[tx * 4 + 2][r]; v.w = tile[tx * 4 + 3][r];
        *reinterpret_cast<char4*>(P + (k0 + r) * Fp + f0 + tx * 4) = v;
    }
}

// Q [Fp x Kp] -> Qb [Kp/128][Fp][128]: 16 bytes per thread, both sides coalesced in 128 B segments
__global__ void block_i8_kernel(const int8_t* __restrict__ Q, int8_t* __restrict__ Qb, int Fp, int64_t Kp) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // 16-byte chunk index
    const int64_t chunks_per_row = Kp / 16;
    if (i >= chunks_per_row * Fp) return;
    const int64_t f = i / chunks_per_row, c = i % chunks_per_row;       // chunk c of feature row f
    const int64_t sb = c / 8, within = c % 8;
    const int4 v = *reinterpret_cast<const int4*>(Q + f * Kp + c * 16);
    *reinterpret_cast<int4*>(Qb + ((sb * Fp + f) * 128) + within * 16) = v;
}

__global__ void subsample_weight_kernel(const double* __restrict__ w, int64_t blocks, int64_t stride, double* __restrict__ out) {
    double s = 0.0;
    for (int64_t b = blockIdx.x; b * stride < blocks; b += gridDim.x) s += w[b * stride * 128 + threadIdx.x];
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(out, s);
}

// multibody base features: row f = product of the spins listed in subsets[f*(order-1) ...]
__global__ void multibody_features_kernel(const int8_t* __restrict__ base, int64_t Kp, const int32_t* __restrict__ subsets,
                                          int width, int F, int8_t* __restrict__ out) {
    const int f = blockIdx.y;
    const int64_t k0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 16;
    if (k0 >= Kp) return;
    int8_t v[16];
    if (f < F) {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = 1;
        for (int q = 0; q < width; ++q) {
            const int s = subsets[f * width + q];
            if (s < 0) break;
            int4 t = *reinterpret_cast<const int4*>(base + (int64_t)s * Kp + k0);
            int8_t u[16];
            memcpy(u, &t, 16);
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = (int8_t)(v[j] * u[j]);
        }
    } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = 0;
    }
    int4 t;
    memcpy(&t, v, 16);
    *reinterpret_cast<int4*>(out + (int64_t)f * Kp + k0) = t;
}

}  // namespace

void hist_from_device(Histogram& h, const double* d_counts, const int8_t* d_spins, int64_t K, int32_t N,
                      int64_t ld, cudaStream_t st) {
    GML_REQUIRE(K >= 1 && N >= 1 && ld >= K, "histogram needs K >= 1, N >= 1, ld >= K");
    h.K = K; h.N = N;
    h.Kp = round_up(K, KPAD);
    h.Fb = (int32_t)round_up(N + 1, FPAD);
    h.base.alloc((size_t)h.Fb * h.Kp);
    h.counts.alloc(K);
    h.w64.alloc(h.Kp);
    h.w32.alloc(h.Kp);
    h.mb_order = 0; h.P_of = nullptr; h.Qb_of = nullptr;

    DevBuf<double> scal;   // [0] sum, [1] max
    DevBuf<int> flags;
    scal.alloc(2); flags.alloc(1);
    GML_CUDA(cudaMemsetAsync(scal.p, 0, 2 * sizeof(double), st));
    GML_CUDA(cudaMemsetAsync(flags.p, 0, sizeof(int), st));

    dim3 grid((unsigned)ceil_div(h.Kp, 16 * 256), h.Fb);
    pack_spins_kernel<<<grid, 256, 0, st>>>(d_spins, ld, K, h.Kp, N, h.Fb, h.base.p, flags.p);
    GML_LAUNCHED();
    GML_CUDA(cudaMemcpyAsync(h.counts.p, d_counts, sizeof(double) * K, cudaMemcpyDeviceToDevice, st));
    const int nb = (int)std::min<int64_t>(ceil_div(K, 256), 148 * 8);
    count_stats_kernel<<<nb, 256, 0, st>>>(d_counts, K, scal.p, scal.p + 1, flags.p);
    GML_LAUNCHED();
    weights_kernel<<<(unsigned)ceil_div(h.Kp, 256), 256, 0, st>>>(d_counts, K, h.Kp, scal.p, h.w64.p, h.w32.p);
    GML_LAUNCHED();

    double hs[2]; int hf = 0;
    GML_CUDA(cudaMemcpyAsync(hs, scal.p, sizeof(hs), cudaMemcpyDeviceToHost, st));
    GML_CUDA(cudaMemcpyAsync(&hf, flags.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    GML_CUDA(cudaStreamSynchronize(st));
    GML_REQUIRE((hf & 1) == 0, "histogram spins must be exactly -1 or +1");
    GML_REQUIRE((hf & 2) == 0, "histogram counts must be positive and finite");
    h.M = hs[0];
    h.wmax = hs[1] / hs[0];
    h.M_local = 0.0;
    h.K_total = (double)K;
}

void build_multibody_features(Histogram& h, int order, const std::vector<int32_t>& h_subsets, int F,
                              cudaStream_t st) {
    const int width = order - 1;
    h.mb_F = F;
    h.mb_Fp = (int32_t)round_up(F, FPAD);
    h.mb_order = order;
    h.mb.alloc((size_t)h.mb_Fp * h.Kp);
    DevBuf<int32_t> sub;
    sub.alloc(h_subsets.size());
    GML_CUDA(cudaMemcpyAsync(sub.p, h_subsets.data(), h_subsets.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    dim3 grid((unsigned)ceil_div(h.Kp, 16 * 256), h.mb_Fp);
    multibody_features_kernel<<<grid, 256, 0, st>>>(h.base.p, h.Kp, sub.p, width, F, h.mb.p);
    GML_LAUNCHED();
    GML_CUDA(cudaStreamSynchronize(st));   // `sub` is freed on return
    if (h.P_of == h.mb.p) h.P_of = nullptr;
    if (h.Qb_of == h.mb.p) h.Qb_of = nullptr;
}

const int8_t* ensure_P(Histogram& h, const int8_t* Q, int Fp, cudaStream_t st) {
    if (h.P_of == Q && h.P.p) return h.P.p;
    h.P.alloc((size_t)h.Kp * Fp);
    dim3 grid((unsigned)(h.Kp / 64), Fp / 64);
    transpose_i8_kernel<<<grid, 256, 0, st>>>(Q, h.P.p, Fp, h.Kp);
    GML_LAUNCHED();
    h.P_of = Q;
    return h.P.p;
}

double subsample_weight(const Histogram& h, int64_t stride, cudaStream_t st) {
    if (stride <= 1) return 1.0;
    DevBuf<double> acc;
    acc.alloc(1);
    GML_CUDA(cudaMemsetAsync(acc.p, 0, sizeof(double), st));
    subsample_weight_kernel<<<592, 128, 0, st>>>(h.w64.p, h.Kp / 128, stride, acc.p);
    GML_LAUNCHED();
    double rho = 0.0;
    GML_CUDA(cudaMemcpyAsync(&rho, acc.p, sizeof(double), cudaMemcpyDeviceToHost, st));
    GML_CUDA(cudaStreamSynchronize(st));
    return rho;
}

void launch_block_copy(const int8_t* Q, int8_t* Qb, int Fp, int64_t Kp, cudaStream_t st) {
    const int64_t chunks = Kp / 16 * Fp;
    block_i8_kernel<<<(unsigned)ceil_div(chunks, 256), 256, 0, st>>>(Q, Qb, Fp, Kp);
    GML_LAUNCHED();
}

const int8_t* ensure_Qb(Histogram& h, const int8_t* Q, int Fp, cudaStream_t st) {
    if (h.Qb_of == Q && h.Qb.p) return h.Qb.p;
    h.Qb.alloc((size_t)h.Kp * Fp);
    launch_block_copy(Q, h.Qb.p, Fp, h.Kp, st);
    h.Qb_of = Q;
    return h.Qb.p;
}

}  // namespace gml
