// Exact iid sampler for +-1 models  p(s) ~ exp( sum_t w_t prod_{i in t} s_i )  over s in {-1,+1}^N: the distribution
// the reference's `sample` draws from by enumerating all 2^N weights on one CPU thread (src/sampling.jl:58-88).
// Configuration c in [0, 2^N) has spin_i = 2*bit_i(c) - 1 (src/sampling.jl:11-14); term t flips sign with the parity
// of its down spins, (-1)^popc(mask_t & ~c).  The 2^N weights are never stored; they are recomputed:
//   1. partition: blocks of 2^12 configurations; per block the max energy and sum exp(E - max), fp64.
//   2. normalise: global max, rescaled block sums, fp64 inclusive scan over blocks -> block CDF; log Z from its last entry.
//   3. draw: counter-based fp64 uniforms (draw d of one stream per seed), block by binary search over the block CDF,
//      bucketed by block (count, scan, scatter) together with the uniform's residual position inside the block.
//   4. resolve: every block with draws recomputes its 2^12 energies into a shared-memory CDF and places its draws by
//      binary search; the non-zero configurations are emitted in index order at offsets from a scan over blocks.
// Every reduction and scan has a fixed shape that depends on N only, so the output depends on (model, n, replicates,
// seed) and not on the grid, the block scheduling or the device.  Cost: ~2^N * n_terms sign+add in fp64 for pass 1 (the
// resolve pass only recomputes blocks that received draws); memory: 40 bytes per block plus 10 bytes per draw.
#include <cmath>
#include <cstring>

#include "common.cuh"

namespace gml {
namespace {

constexpr int BLOCK_BITS = 12;                      // configurations per enumeration block: 2^12
constexpr int BLOCK_CFG = 1 << BLOCK_BITS;
constexpr int THREADS = 256;
constexpr int PER_THREAD = BLOCK_CFG / THREADS;     // 16 consecutive configurations per thread: its low 4 bits
constexpr int TERM_CHUNK = 512;                     // terms staged in shared memory at a time
constexpr int SCAN_TILE = 1024;                     // elements per tile of the block scans (4 per thread)

typedef unsigned long long ull;

__device__ __forceinline__ int popc(uint32_t x) { return __popc(x); }
__device__ __forceinline__ int popc(uint64_t x) { return __popcll(x); }

// Butterfly reductions leave the same value in every lane; the per-warp results are then combined in warp order.
template <class T, class Op> __device__ __forceinline__ T block_reduce(T v, T* red, Op op) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, o));
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    T r = red[0];
    for (int w = 1; w < THREADS / 32; ++w) r = op(r, red[w]);
    return r;
}

// Exclusive prefix of v over the threads of the block (thread order).
template <class T> __device__ __forceinline__ T block_exclusive_scan(T v, T* red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    T incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T u = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += u;
    }
    __syncthreads();
    if (lane == 31) red[warp] = incl;
    __syncthreads();
    T base = 0;
    for (int w = 0; w < warp; ++w) base += red[w];
    return base + incl - v;
}

// Energies of the thread's 16 configurations cfg0 + k.  A term's mask splits into its low 4 bits, whose sign pattern
// over k is precomputed (bit k of par = parity of popc(mask & 0xF & ~k)), and its high bits, which are the same for all
// 16 configurations: one popc per term and thread, then a sign flip per configuration.
template <class MaskT>
__device__ __forceinline__ void thread_energies(uint64_t cfg0, int n_terms, const uint64_t* __restrict__ hi,
                                                const double* __restrict__ w, const uint32_t* __restrict__ par,
                                                MaskT* s_hi, double* s_w, uint32_t* s_par, double (&e)[PER_THREAD]) {
#pragma unroll
    for (int k = 0; k < PER_THREAD; ++k) e[k] = 0.0;
    const MaskT down = ~(MaskT)cfg0;
    for (int t0 = 0; t0 < n_terms; t0 += TERM_CHUNK) {
        const int nt = min(TERM_CHUNK, n_terms - t0);
        __syncthreads();
        for (int t = threadIdx.x; t < nt; t += THREADS) {
            s_hi[t] = (MaskT)hi[t0 + t]; s_w[t] = w[t0 + t]; s_par[t] = par[t0 + t];
        }
        __syncthreads();
        for (int t = 0; t < nt; ++t) {
            const uint32_t flip = s_par[t] ^ (0u - (uint32_t)(popc((MaskT)(s_hi[t] & down)) & 1));
            const int whi = __double2hiint(s_w[t]), wlo = __double2loint(s_w[t]);
#pragma unroll
            for (int k = 0; k < PER_THREAD; ++k)
                e[k] += __hiloint2double(whi ^ (int)((flip << (31 - k)) & 0x80000000u), wlo);
        }
    }
}

// Valid configurations get their energy, the padding of a model with N < 12 gets -inf (weight 0); returns the max.
__device__ __forceinline__ double mask_padding(uint64_t cfg0, int N, double (&e)[PER_THREAD]) {
    double m = -INFINITY;
#pragma unroll
    for (int k = 0; k < PER_THREAD; ++k) {
        if (((cfg0 + k) >> N) != 0) e[k] = -INFINITY;
        m = fmax(m, e[k]);
    }
    return m;
}

struct MaxOp { __device__ double operator()(double a, double b) const { return fmax(a, b); } };
struct AddOp { template <class T> __device__ T operator()(T a, T b) const { return a + b; } };

template <class MaskT>
__global__ void __launch_bounds__(THREADS) exact_partition_kernel(int N, int n_terms, const uint64_t* __restrict__ hi,
                                                                  const double* __restrict__ w, const uint32_t* __restrict__ par,
                                                                  double* __restrict__ bmax, double* __restrict__ bsum) {
    __shared__ MaskT s_hi[TERM_CHUNK];
    __shared__ double s_w[TERM_CHUNK];
    __shared__ uint32_t s_par[TERM_CHUNK];
    __shared__ double red[THREADS / 32];
    const uint64_t cfg0 = ((uint64_t)blockIdx.x << BLOCK_BITS) + (uint64_t)PER_THREAD * threadIdx.x;
    double e[PER_THREAD];
    thread_energies<MaskT>(cfg0, n_terms, hi, w, par, s_hi, s_w, s_par, e);
    const double m = block_reduce(mask_padding(cfg0, N, e), red, MaxOp());
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < PER_THREAD; ++k) s += exp(e[k] - m);
    s = block_reduce(s, red, AddOp());
    if (threadIdx.x == 0) { bmax[blockIdx.x] = m; bsum[blockIdx.x] = s; }
}

// order-preserving map of doubles to unsigned keys (for atomicMax)
__device__ __forceinline__ ull order_key(double x) {
    const ull b = (ull)__double_as_longlong(x);
    return (b >> 63) ? ~b : (b | (1ull << 63));
}
__device__ __forceinline__ double from_order_key(ull k) {
    return __longlong_as_double((long long)((k >> 63) ? (k & ~(1ull << 63)) : ~k));
}

__global__ void __launch_bounds__(THREADS) max_kernel(const double* __restrict__ a, int64_t n, ull* __restrict__ key) {
    __shared__ double red[THREADS / 32];
    double m = -INFINITY;
    for (int64_t i = (int64_t)blockIdx.x * THREADS + threadIdx.x; i < n; i += (int64_t)gridDim.x * THREADS) m = fmax(m, a[i]);
    m = block_reduce(m, red, MaxOp());
    if (threadIdx.x == 0) atomicMax(key, order_key(m));
}

__global__ void rescale_kernel(const double* __restrict__ bmax, double* __restrict__ bsum, int64_t n, const ull* __restrict__ key) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) bsum[i] *= exp(bmax[i] - from_order_key(*key));
}

// In-place inclusive scan of one tile of SCAN_TILE elements; tile_tot[tile] receives its total.
template <class T> __global__ void __launch_bounds__(THREADS) tile_scan_kernel(T* __restrict__ a, int64_t n, T* __restrict__ tile_tot) {
    __shared__ T red[THREADS / 32];
    const int64_t i0 = (int64_t)blockIdx.x * SCAN_TILE + 4 * threadIdx.x;
    T v[4], run = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) { v[k] = (i0 + k < n) ? a[i0 + k] : T(0); run += v[k]; v[k] = run; }
    const T base = block_exclusive_scan(run, red);
#pragma unroll
    for (int k = 0; k < 4; ++k) if (i0 + k < n) a[i0 + k] = base + v[k];
    if (tile_tot && threadIdx.x == THREADS - 1) tile_tot[blockIdx.x] = base + run;
}

template <class T> __global__ void __launch_bounds__(THREADS) tile_add_kernel(T* __restrict__ a, int64_t n, const T* __restrict__ tile_incl) {
    const T add = tile_incl[blockIdx.x];             // block j adds the inclusive total of tiles 0..j to tile j+1
    const int64_t i0 = (int64_t)(blockIdx.x + 1) * SCAN_TILE;
    for (int k = threadIdx.x; k < SCAN_TILE; k += THREADS)
        if (i0 + k < n) a[i0 + k] += add;
}

template <class T> int64_t scan_scratch(int64_t n) {
    int64_t s = 0;
    for (int64_t t = ceil_div(n, SCAN_TILE); n > SCAN_TILE; n = t, t = ceil_div(n, SCAN_TILE)) s += t;
    return std::max<int64_t>(s, 1);
}

// In-place inclusive scan with a fixed tile tree (the summation order depends on n only).
template <class T> void scan_inclusive(T* a, int64_t n, T* scratch, cudaStream_t st) {
    const int64_t tiles = ceil_div(n, SCAN_TILE);
    tile_scan_kernel<T><<<(unsigned)tiles, THREADS, 0, st>>>(a, n, tiles > 1 ? scratch : nullptr);
    GML_LAUNCHED();
    if (tiles == 1) return;
    scan_inclusive(scratch, tiles, scratch + tiles, st);
    tile_add_kernel<T><<<(unsigned)(tiles - 1), THREADS, 0, st>>>(a, n, scratch);
    GML_LAUNCHED();
}

// Draw d of the stream of `seed`: a uniform in [0, 1) with 53 random bits.
__device__ __forceinline__ double uniform01(uint64_t seed, uint64_t d) {
    uint64_t x = seed * 0x9E3779B97F4A7C15ULL + (d + 1) * 0xD1B54A32D192ED03ULL;
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL;
    x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL;
    x ^= x >> 33;
    return (double)(x >> 11) * 0x1.0p-53;
}

// Block of draw d (first b with cdf[b] > u * total; never a block of weight 0) and the draw's position inside it.
__device__ __forceinline__ int64_t locate(const double* __restrict__ cdf, int64_t nb, uint64_t seed, uint64_t d, double* resid) {
    const double total = cdf[nb - 1];
    const double x = fmin(uniform01(seed, d) * total, nextafter(total, 0.0));
    int64_t lo = 0, hi = nb - 1;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (cdf[mid] > x) hi = mid; else lo = mid + 1;
    }
    const double below = lo ? cdf[lo - 1] : 0.0;
    *resid = fmin(fmax((x - below) / (cdf[lo] - below), 0.0), nextafter(1.0, 0.0));
    return lo;
}

__global__ void count_draws_kernel(const double* __restrict__ cdf, int64_t nb, uint64_t seed, int64_t d0, int64_t n, ull* __restrict__ cnt) {
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += (int64_t)gridDim.x * blockDim.x) {
        double r;
        atomicAdd(&cnt[locate(cdf, nb, seed, (uint64_t)(d0 + q), &r)], 1ull);
    }
}

// cur[b] enters as the inclusive end of bucket b and leaves as its start.  The order of draws inside a bucket is not
// deterministic, but only the per-configuration counts of a bucket are ever read.
__global__ void scatter_draws_kernel(const double* __restrict__ cdf, int64_t nb, uint64_t seed, int64_t d0, int64_t n,
                                     ull* __restrict__ cur, double* __restrict__ resid) {
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += (int64_t)gridDim.x * blockDim.x) {
        double r;
        const int64_t b = locate(cdf, nb, seed, (uint64_t)(d0 + q), &r);
        resid[atomicAdd(&cur[b], ~0ull) - 1] = r;
    }
}

// Places the draws of one block on its configurations (cfg receives the low 12 bits) and counts the configurations hit.
template <class MaskT>
__global__ void __launch_bounds__(THREADS) exact_resolve_kernel(int N, int n_terms, const uint64_t* __restrict__ hi,
                                                                const double* __restrict__ w, const uint32_t* __restrict__ par,
                                                                const ull* __restrict__ cnt, const ull* __restrict__ start,
                                                                const double* __restrict__ resid, uint16_t* __restrict__ cfg,
                                                                ull* __restrict__ nz) {
    __shared__ MaskT s_hi[TERM_CHUNK];
    __shared__ double s_w[TERM_CHUNK];
    __shared__ uint32_t s_par[TERM_CHUNK];
    __shared__ double red[THREADS / 32];
    __shared__ ull red_u[THREADS / 32];
    __shared__ double cdf[BLOCK_CFG];
    __shared__ uint8_t hit[BLOCK_CFG];
    const ull c = cnt[blockIdx.x];
    if (c == 0) {
        if (threadIdx.x == 0) nz[blockIdx.x] = 0;
        return;
    }
    const uint64_t cfg0 = ((uint64_t)blockIdx.x << BLOCK_BITS) + (uint64_t)PER_THREAD * threadIdx.x;
    double e[PER_THREAD];
    thread_energies<MaskT>(cfg0, n_terms, hi, w, par, s_hi, s_w, s_par, e);
    const double m = block_reduce(mask_padding(cfg0, N, e), red, MaxOp());
    double run = 0.0;
#pragma unroll
    for (int k = 0; k < PER_THREAD; ++k) { run += exp(e[k] - m); e[k] = run; }
    const double base = block_exclusive_scan(run, red);
#pragma unroll
    for (int k = 0; k < PER_THREAD; ++k) { cdf[PER_THREAD * threadIdx.x + k] = base + e[k]; hit[PER_THREAD * threadIdx.x + k] = 0; }
    __syncthreads();
    const double total = cdf[BLOCK_CFG - 1], top = nextafter(total, 0.0);
    const ull s = start[blockIdx.x];
    for (ull q = threadIdx.x; q < c; q += THREADS) {
        const double x = fmin(resid[s + q] * total, top);
        int lo = 0, hi_ = BLOCK_CFG - 1;
        while (lo < hi_) {
            const int mid = (lo + hi_) >> 1;
            if (cdf[mid] > x) hi_ = mid; else lo = mid + 1;
        }
        cfg[s + q] = (uint16_t)lo;
        hit[lo] = 1;
    }
    __syncthreads();
    ull mine = 0;
#pragma unroll
    for (int k = 0; k < PER_THREAD; ++k) mine += hit[PER_THREAD * threadIdx.x + k];
    mine = block_reduce(mine, red_u, AddOp());
    if (threadIdx.x == 0) nz[blockIdx.x] = mine;
}

// Counts the draws of one block per configuration and writes its non-zero configurations in index order at row
// out0 + (rows of the blocks before it).
__global__ void __launch_bounds__(THREADS) exact_emit_kernel(int N, const ull* __restrict__ cnt, const ull* __restrict__ start,
                                                             const uint16_t* __restrict__ cfg, const ull* __restrict__ nz_incl,
                                                             int64_t out0, double* __restrict__ counts, int8_t* __restrict__ spins,
                                                             int64_t ld) {
    __shared__ ull per_cfg[BLOCK_CFG];
    __shared__ ull red[THREADS / 32];
    const ull c = cnt[blockIdx.x];
    if (c == 0) return;
    for (int j = threadIdx.x; j < BLOCK_CFG; j += THREADS) per_cfg[j] = 0;
    __syncthreads();
    const ull s = start[blockIdx.x];
    for (ull q = threadIdx.x; q < c; q += THREADS) atomicAdd(&per_cfg[cfg[s + q]], 1ull);
    __syncthreads();
    ull mine = 0;
#pragma unroll
    for (int k = 0; k < PER_THREAD; ++k) mine += per_cfg[PER_THREAD * threadIdx.x + k] != 0;
    int64_t row = out0 + (int64_t)(blockIdx.x ? nz_incl[blockIdx.x - 1] : 0) + (int64_t)block_exclusive_scan(mine, red);
    for (int k = 0; k < PER_THREAD; ++k) {
        const int j = PER_THREAD * threadIdx.x + k;
        if (per_cfg[j] == 0) continue;
        const uint64_t conf = ((uint64_t)blockIdx.x << BLOCK_BITS) + j;
        counts[row] = (double)per_cfg[j];
        for (int i = 0; i < N; ++i) spins[(int64_t)i * ld + row] = ((conf >> i) & 1ull) ? 1 : -1;
        ++row;
    }
}

}  // namespace

double sample_exact(int N, const std::vector<uint64_t>& masks, const std::vector<double>& weights, int64_t n_samples,
                    int replicates, uint64_t seed, int64_t* out_K, double* d_counts, int8_t* d_spins, int64_t ld,
                    cudaStream_t st) {
    const int n_terms = (int)masks.size();
    const int64_t nb = N > BLOCK_BITS ? (int64_t)1 << (N - BLOCK_BITS) : 1;
    std::vector<uint64_t> hi(std::max(n_terms, 1), 0);
    std::vector<uint32_t> par(std::max(n_terms, 1), 0);
    for (int t = 0; t < n_terms; ++t) {
        hi[t] = masks[t] & ~0xFull;
        for (int k = 0; k < PER_THREAD; ++k) par[t] |= (uint32_t)(__builtin_popcountll(masks[t] & 0xFull & ~(uint64_t)k) & 1) << k;
    }
    DevBuf<uint64_t> d_hi;
    DevBuf<uint32_t> d_par;
    DevBuf<double> d_w, bmax, cdf, dscan, resid;
    DevBuf<ull> key, cnt, cur, nz, uscan;
    DevBuf<uint16_t> cfg;
    d_hi.alloc(hi.size()); d_par.alloc(par.size()); d_w.alloc(std::max(n_terms, 1));
    bmax.alloc(nb); cdf.alloc(nb); key.alloc(1); cnt.alloc(nb); cur.alloc(nb); nz.alloc(nb);
    dscan.alloc(scan_scratch<double>(nb)); uscan.alloc(scan_scratch<ull>(nb));
    resid.alloc(n_samples); cfg.alloc(n_samples);
    GML_CUDA(cudaMemcpyAsync(d_hi.p, hi.data(), sizeof(uint64_t) * hi.size(), cudaMemcpyHostToDevice, st));
    GML_CUDA(cudaMemcpyAsync(d_par.p, par.data(), sizeof(uint32_t) * par.size(), cudaMemcpyHostToDevice, st));
    if (n_terms) GML_CUDA(cudaMemcpyAsync(d_w.p, weights.data(), sizeof(double) * n_terms, cudaMemcpyHostToDevice, st));

    // 1-2: block partition sums, global max, block CDF
    if (N <= 32) exact_partition_kernel<uint32_t><<<(unsigned)nb, THREADS, 0, st>>>(N, n_terms, d_hi.p, d_w.p, d_par.p, bmax.p, cdf.p);
    else exact_partition_kernel<uint64_t><<<(unsigned)nb, THREADS, 0, st>>>(N, n_terms, d_hi.p, d_w.p, d_par.p, bmax.p, cdf.p);
    GML_LAUNCHED();
    GML_CUDA(cudaMemsetAsync(key.p, 0, sizeof(ull), st));
    max_kernel<<<(unsigned)std::min<int64_t>(ceil_div(nb, THREADS), 1024), THREADS, 0, st>>>(bmax.p, nb, key.p);
    GML_LAUNCHED();
    rescale_kernel<<<(unsigned)ceil_div(nb, THREADS), THREADS, 0, st>>>(bmax.p, cdf.p, nb, key.p);
    GML_LAUNCHED();
    scan_inclusive(cdf.p, nb, dscan.p, st);
    double total = 0.0, gmax = 0.0;
    ull hkey = 0;
    GML_CUDA(cudaMemcpyAsync(&total, cdf.p + nb - 1, sizeof(double), cudaMemcpyDeviceToHost, st));
    GML_CUDA(cudaMemcpyAsync(&hkey, key.p, sizeof(ull), cudaMemcpyDeviceToHost, st));
    GML_CUDA(cudaStreamSynchronize(st));
    { const uint64_t b = (hkey >> 63) ? (hkey & ~(1ull << 63)) : ~hkey; std::memcpy(&gmax, &b, sizeof(double)); }
    const double log_z = gmax + std::log(total);

    // 3-4 per replicate: draws [r*n, (r+1)*n) of the stream
    const unsigned draw_grid = (unsigned)std::min<int64_t>(ceil_div(n_samples, THREADS), 148 * 16);
    int64_t rows = 0;
    bool fits = true;
    for (int r = 0; r < replicates; ++r) {
        const int64_t d0 = (int64_t)r * n_samples;
        GML_CUDA(cudaMemsetAsync(cnt.p, 0, sizeof(ull) * nb, st));
        count_draws_kernel<<<draw_grid, THREADS, 0, st>>>(cdf.p, nb, seed, d0, n_samples, cnt.p);
        GML_LAUNCHED();
        GML_CUDA(cudaMemcpyAsync(cur.p, cnt.p, sizeof(ull) * nb, cudaMemcpyDeviceToDevice, st));
        scan_inclusive(cur.p, nb, uscan.p, st);
        scatter_draws_kernel<<<draw_grid, THREADS, 0, st>>>(cdf.p, nb, seed, d0, n_samples, cur.p, resid.p);
        GML_LAUNCHED();
        if (N <= 32) exact_resolve_kernel<uint32_t><<<(unsigned)nb, THREADS, 0, st>>>(N, n_terms, d_hi.p, d_w.p, d_par.p, cnt.p, cur.p, resid.p, cfg.p, nz.p);
        else exact_resolve_kernel<uint64_t><<<(unsigned)nb, THREADS, 0, st>>>(N, n_terms, d_hi.p, d_w.p, d_par.p, cnt.p, cur.p, resid.p, cfg.p, nz.p);
        GML_LAUNCHED();
        scan_inclusive(nz.p, nb, uscan.p, st);
        ull K = 0;
        GML_CUDA(cudaMemcpyAsync(&K, nz.p + nb - 1, sizeof(ull), cudaMemcpyDeviceToHost, st));
        GML_CUDA(cudaStreamSynchronize(st));
        out_K[r] = (int64_t)K;
        fits = fits && rows + (int64_t)K <= ld;
        if (d_counts && fits) {
            exact_emit_kernel<<<(unsigned)nb, THREADS, 0, st>>>(N, cnt.p, cur.p, cfg.p, nz.p, rows, d_counts, d_spins, ld);
            GML_LAUNCHED();
        }
        rows += (int64_t)K;
    }
    GML_CUDA(cudaStreamSynchronize(st));
    GML_REQUIRE(!d_counts || fits, "ld = " + std::to_string(ld) + " is smaller than the " + std::to_string(rows) +
                                   " rows of the replicates (out_K holds their sizes)");
    return log_z;
}

}  // namespace gml
