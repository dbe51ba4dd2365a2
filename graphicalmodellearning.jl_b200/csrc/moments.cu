// Moments <prod_{i in t} s_i> from the record buffer of mcmc_kernel's RECORD mode (model side) and from a resident
// histogram (data side).
//   - Record buffer: spin-major [(N+1) x ld], ld = records * warps, column r * warps + w = warp w's r-th record: bit c of
//     row i is spin i of lane c, row N the mask of the lanes whose record is a draw.  The warps are split into
//     G = min(32, warps) contiguous groups of whole warps (warps are independent); every reduction keeps one sum per group.
//   - Key lists: a key of q <= 8 spins has, per record word, odd = XOR_m ~w[i_m] (the lanes with an odd number of down
//     spins, the rule of down_parity); the record adds popc(mask) - 2 popc(odd & mask).  One warp per (key, group).
//   - Pairwise: C_ij = sum (2 popc(~(w_i ^ w_j) & mask) - popc(mask)) by a tiled XNOR-popcount bit-GEMM, 64 x 64 spin
//     tiles of the upper triangle per CTA and group, the group's record columns staged 32 at a time in shared memory;
//     <s_i> from the key-list kernel with the N singleton keys.
//   - All sums are integers (int64), so they do not depend on the grid or the order of the atomics-free reductions.  Per
//     entry, in group order: mean = sum S_g / sum n_g, stderr = sqrt(G/(G-1) sum_g (S_g - mean n_g)^2) / sum n_g (NaN for
//     G < 2).
//   - Histogram key lists: sum_k c_k prod s_ki over the int8 rows of hist.base with the raw counts in fp64 (exact for
//     integer counts below 2^53 in total), per-chunk partials over a fixed number of row chunks that depends on K only,
//     summed in chunk order and divided by M once.
#include <cmath>

#include "common.cuh"

namespace gml {
namespace {

constexpr uint32_t FULL = 0xffffffffu;
constexpr int MAX_GROUPS = 32;
constexpr int TILE = 64;          // spins per side of a bit-GEMM tile
constexpr int CHUNK = 32;         // record columns staged per step of the bit-GEMM
constexpr int HIST_CHUNKS = 512;  // row chunks of the histogram key-list kernel (at most)

__device__ __forceinline__ int64_t group_begin(int g, int G, int64_t warps) { return (int64_t)g * warps / G; }

// column of the t-th record of a group of nw warps from warp wb on (records in order, warps in order within a record)
__device__ __forceinline__ int64_t group_column(int64_t t, int64_t nw, int64_t wb, int64_t warps) {
    const int64_t r = t / nw;
    return r * warps + wb + (t - r * nw);
}

__device__ __forceinline__ long long warp_sum_i64(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

// n_g: draws of group g (blockIdx.x), one warp
__global__ void group_draws_kernel(const uint32_t* __restrict__ rec, int N, int64_t records, int64_t warps, int64_t ld, int G,
                                   long long* __restrict__ n_g) {
    const int g = blockIdx.x, lane = threadIdx.x;
    const int64_t wb = group_begin(g, G, warps), we = group_begin(g + 1, G, warps);
    const uint32_t* masks = rec + (int64_t)N * ld;
    const int64_t nw = we - wb, total = records * nw;
    long long acc = 0;
    for (int64_t t = lane; t < total; t += 32) acc += __popc(masks[group_column(t, nw, wb, warps)]);
    acc = warp_sum_i64(acc);
    if (lane == 0) n_g[g] = acc;
}

// S[g][k] = sum over the records of group g of (popc(mask) - 2 popc(odd & mask)); one warp per key, grid (keys / 4, G)
__global__ void __launch_bounds__(128) key_sums_kernel(const uint32_t* __restrict__ rec, int N, int64_t records, int64_t warps,
                                                       int64_t ld, int G, int order, int n_keys, const int32_t* __restrict__ key_idx,
                                                       long long* __restrict__ S) {
    const int lane = threadIdx.x & 31;
    const int k = blockIdx.x * 4 + (threadIdx.x >> 5), g = blockIdx.y;
    if (k >= n_keys) return;
    int32_t mem[8];
    int q = 0;
    for (int m = 0; m < order; ++m) {
        const int32_t i = key_idx[(int64_t)k * order + m];
        if (i >= 0) mem[q++] = i;
    }
    const int64_t wb = group_begin(g, G, warps), we = group_begin(g + 1, G, warps);
    const uint32_t* masks = rec + (int64_t)N * ld;
    const int64_t nw = we - wb, total = records * nw;
    long long acc = 0;
    for (int64_t t = lane; t < total; t += 32) {
        const int64_t col = group_column(t, nw, wb, warps);
        uint32_t odd = 0;
        for (int m = 0; m < q; ++m) odd ^= ~__ldg(rec + (int64_t)mem[m] * ld + col);
        const uint32_t mask = __ldg(masks + col);
        acc += __popc(mask) - 2 * __popc(odd & mask);
    }
    acc = warp_sum_i64(acc);
    if (lane == 0) S[(int64_t)g * n_keys + k] = acc;
}

// A[g][i][j] = sum over the records of group g of popc(~(w_i ^ w_j) & mask) for the 64 x 64 tile (blockIdx.y, blockIdx.x)
// of the upper triangle of tiles (i <= j within a diagonal tile is what the caller reads).  Thread (ty, tx) owns spins
// i0 + 4 ty + a and j0 + 4 tx + b.
__global__ void __launch_bounds__(256) pair_sums_kernel(const uint32_t* __restrict__ rec, int N, int64_t records, int64_t warps,
                                                        int64_t ld, int G, unsigned long long* __restrict__ A) {
    const int bi = blockIdx.y, bj = blockIdx.x, g = blockIdx.z;
    if (bj < bi) return;
    __shared__ __align__(16) uint32_t si[CHUNK][TILE], sj[CHUNK][TILE];
    __shared__ uint32_t sm[CHUNK];
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    const int i0 = bi * TILE, j0 = bj * TILE;
    const int64_t wb = group_begin(g, G, warps), we = group_begin(g + 1, G, warps);
    const uint32_t* masks = rec + (int64_t)N * ld;
    const int64_t nw = we - wb, total = records * nw;
    const int c_own = tid % CHUNK, row0 = tid / CHUNK;       // every thread stages one column: coalesced rows
    unsigned long long acc[4][4] = {};
    for (int64_t t0 = 0; t0 < total; t0 += CHUNK) {
        __syncthreads();
        const bool in = t0 + c_own < total;
        const int64_t col = in ? group_column(t0 + c_own, nw, wb, warps) : 0;
        for (int row = row0; row < TILE; row += 256 / CHUNK) {
            si[c_own][row] = (in && i0 + row < N) ? __ldg(rec + (int64_t)(i0 + row) * ld + col) : 0u;
            sj[c_own][row] = (in && j0 + row < N) ? __ldg(rec + (int64_t)(j0 + row) * ld + col) : 0u;
        }
        if (row0 == 0) sm[c_own] = in ? __ldg(masks + col) : 0u;   // padding: mask 0
        __syncthreads();
#pragma unroll 4
        for (int c = 0; c < CHUNK; ++c) {
            const uint4 a = *reinterpret_cast<const uint4*>(&si[c][4 * ty]);
            const uint4 b = *reinterpret_cast<const uint4*>(&sj[c][4 * tx]);
            const uint32_t m = sm[c];
            const uint32_t wi[4] = {a.x, a.y, a.z, a.w}, wj[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int x = 0; x < 4; ++x)
#pragma unroll
                for (int y = 0; y < 4; ++y) acc[x][y] += __popc(~(wi[x] ^ wj[y]) & m);
        }
    }
    const int64_t NN = (int64_t)N * N;
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) {
            const int i = i0 + 4 * ty + x, j = j0 + 4 * tx + y;
            if (i < N && j < N) A[g * NN + (int64_t)i * N + j] = acc[x][y];
        }
}

// mean and stderr of entry e from the per-group sums, in group order.  Pairwise (A != nullptr): entry (i, j) of the
// N x N output, S_g = 2 A[g][min][max] - n_g off the diagonal and the singleton-key sum S[g][i] on it.
__global__ void finalize_kernel(const long long* __restrict__ S, const unsigned long long* __restrict__ A, int N, int64_t n_out,
                                const long long* __restrict__ n_g, int G, double* __restrict__ mean, double* __restrict__ stderr_) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_out) return;
    auto sum_of = [&](int g) -> long long {
        if (!A) return S[(int64_t)g * n_out + e];
        const int i = (int)(e / N), j = (int)(e % N);
        if (i == j) return S[(int64_t)g * N + i];
        const int lo = min(i, j), hi = max(i, j);
        return 2 * (long long)A[(int64_t)g * N * N + (int64_t)lo * N + hi] - n_g[g];
    };
    long long s = 0, n = 0;
    for (int g = 0; g < G; ++g) { s += sum_of(g); n += n_g[g]; }
    const double m = (double)s / (double)n;
    double q = 0.0;
    for (int g = 0; g < G; ++g) {
        const double d = (double)sum_of(g) - m * (double)n_g[g];
        q += d * d;
    }
    mean[e] = m;
    if (stderr_) stderr_[e] = G < 2 ? NAN : sqrt((double)G / (G - 1) * q) / (double)n;
}

// partial[c][k] = sum over the rows of chunk c of counts[r] prod_{i in key k} s_i[r]; one warp per key, grid (keys / 4, chunks)
__global__ void __launch_bounds__(128) hist_key_sums_kernel(const int8_t* __restrict__ base, int64_t Kp, const double* __restrict__ counts,
                                                            int64_t K, int64_t rows_per_chunk, int order, int n_keys,
                                                            const int32_t* __restrict__ key_idx, double* __restrict__ partial) {
    const int lane = threadIdx.x & 31;
    const int k = blockIdx.x * 4 + (threadIdx.x >> 5), c = blockIdx.y;
    if (k >= n_keys) return;
    int32_t mem[8];
    int q = 0;
    for (int m = 0; m < order; ++m) {
        const int32_t i = key_idx[(int64_t)k * order + m];
        if (i >= 0) mem[q++] = i;
    }
    const int64_t r0 = (int64_t)c * rows_per_chunk, r1 = min(K, r0 + rows_per_chunk);
    double acc = 0.0;
    for (int64_t r = r0 + lane; r < r1; r += 32) {
        int neg = 0;
        for (int m = 0; m < q; ++m) neg ^= __ldg(base + (int64_t)mem[m] * Kp + r) < 0;
        const double cnt = __ldg(counts + r);
        acc += neg ? -cnt : cnt;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(FULL, acc, o);
    if (lane == 0) partial[(int64_t)c * n_keys + k] = acc;
}

__global__ void hist_finalize_kernel(const double* __restrict__ partial, int chunks, int n_keys, double M, double* __restrict__ mean) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_keys) return;
    double s = 0.0;
    for (int c = 0; c < chunks; ++c) s += partial[(int64_t)c * n_keys + k];
    mean[k] = s / M;
}

// the singleton keys 0..N-1
std::vector<int32_t> singletons(int N) {
    std::vector<int32_t> idx(N);
    for (int i = 0; i < N; ++i) idx[i] = i;
    return idx;
}

}  // namespace

int64_t moment_outputs(const MomentKeys& keys, int N) { return keys.pairwise ? (int64_t)N * N : keys.n_keys; }

int record_groups(int64_t warps) { return (int)std::min<int64_t>(MAX_GROUPS, warps); }

void record_key_sums(const uint32_t* rec, int N, int64_t records, int64_t warps, int order, int n_keys, const int32_t* d_key_idx,
                     long long* d_n_g, long long* d_S, cudaStream_t st) {
    const int G = record_groups(warps);
    const int64_t ld = records * warps;
    group_draws_kernel<<<G, 32, 0, st>>>(rec, N, records, warps, ld, G, d_n_g);
    GML_LAUNCHED();
    key_sums_kernel<<<dim3((unsigned)ceil_div(n_keys, 4), G), 128, 0, st>>>(rec, N, records, warps, ld, G, order, n_keys, d_key_idx, d_S);
    GML_LAUNCHED();
}

void reduce_records(const uint32_t* rec, int N, int64_t records, int64_t warps, const MomentKeys& keys, double* out_mean,
                    double* out_stderr, cudaStream_t st) {
    const int G = record_groups(warps);
    const int64_t ld = records * warps, n_out = moment_outputs(keys, N);
    const std::vector<int32_t> idx = keys.pairwise ? singletons(N) : keys.idx;
    const int order = keys.pairwise ? 1 : keys.order, n_keys = keys.pairwise ? N : keys.n_keys;
    DevBuf<long long> n_g, S;
    DevBuf<int32_t> d_idx;
    DevBuf<unsigned long long> A;
    DevBuf<double> mean, err;
    n_g.alloc(G); S.alloc((size_t)G * n_keys); d_idx.alloc(idx.size());
    mean.alloc(n_out); err.alloc(n_out);
    GML_CUDA(cudaMemcpyAsync(d_idx.p, idx.data(), sizeof(int32_t) * idx.size(), cudaMemcpyHostToDevice, st));
    record_key_sums(rec, N, records, warps, order, n_keys, d_idx.p, n_g.p, S.p, st);
    if (keys.pairwise) {
        A.alloc((size_t)G * N * N);
        const unsigned t = (unsigned)ceil_div(N, TILE);
        pair_sums_kernel<<<dim3(t, t, G), 256, 0, st>>>(rec, N, records, warps, ld, G, A.p);
        GML_LAUNCHED();
    }
    finalize_kernel<<<(unsigned)ceil_div(n_out, 256), 256, 0, st>>>(S.p, keys.pairwise ? A.p : nullptr, N, n_out, n_g.p, G,
                                                                     mean.p, err.p);
    GML_LAUNCHED();
    GML_CUDA(cudaMemcpyAsync(out_mean, mean.p, sizeof(double) * n_out, cudaMemcpyDeviceToHost, st));
    if (out_stderr) GML_CUDA(cudaMemcpyAsync(out_stderr, err.p, sizeof(double) * n_out, cudaMemcpyDeviceToHost, st));
    GML_CUDA(cudaStreamSynchronize(st));
}

void moments_histogram_keys(const Histogram& hist, const MomentKeys& keys, double* out_mean, cudaStream_t st) {
    const int64_t K = hist.K;
    const int chunks = (int)std::min<int64_t>(HIST_CHUNKS, ceil_div(K, 1024));
    const int64_t per = ceil_div(K, chunks);
    DevBuf<int32_t> d_idx;
    DevBuf<double> partial, mean;
    d_idx.alloc(keys.idx.size()); partial.alloc((size_t)chunks * keys.n_keys); mean.alloc(keys.n_keys);
    GML_CUDA(cudaMemcpyAsync(d_idx.p, keys.idx.data(), sizeof(int32_t) * keys.idx.size(), cudaMemcpyHostToDevice, st));
    hist_key_sums_kernel<<<dim3((unsigned)ceil_div(keys.n_keys, 4), chunks), 128, 0, st>>>(hist.base.p, hist.Kp, hist.counts.p, K, per,
                                                                                           keys.order, keys.n_keys, d_idx.p, partial.p);
    GML_LAUNCHED();
    hist_finalize_kernel<<<(unsigned)ceil_div(keys.n_keys, 256), 256, 0, st>>>(partial.p, chunks, keys.n_keys, hist.M, mean.p);
    GML_LAUNCHED();
    GML_CUDA(cudaMemcpyAsync(out_mean, mean.p, sizeof(double) * keys.n_keys, cudaMemcpyDeviceToHost, st));
    GML_CUDA(cudaStreamSynchronize(st));
}

}  // namespace gml
