// Device histogram builder (SURVEY 8f-1): raw sample stream -> deduplicated [count, s_1..s_N] histogram.
// The reference collapses duplicate configurations with `countmap` on the host (src/sampling.jl:52-54); here each
// sample is bit-packed into a 64-bit key (N <= 64), keys are radix-sorted and run-length encoded on the device
// (CUB primitives), and the unique keys are unpacked back to spin-major int8 rows.  For N <= ~40 this shrinks K by
// orders of magnitude before the solve; for N > 64 every sample is distinct with overwhelming probability and the
// stream is used as is.
#include <cub/cub.cuh>

#include "common.cuh"

namespace gml {
namespace {

__global__ void pack_keys_kernel(const int8_t* __restrict__ samples, int64_t ld, int64_t M, int N, unsigned long long* __restrict__ keys,
                                 int* __restrict__ flags) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= M) return;
    unsigned long long key = 0;
    bool bad = false;
    for (int i = 0; i < N; ++i) {
        const int8_t s = samples[(int64_t)i * ld + k];
        bad |= (s != 1 && s != -1);
        key |= (unsigned long long)(s > 0) << i;          // bit i = spin i+1 up, like int_to_spin (src/sampling.jl:11-14)
    }
    keys[k] = key;
    if (bad) atomicOr(flags, 1);
}

__global__ void unpack_keys_kernel(const unsigned long long* __restrict__ keys, const int* __restrict__ run_len, int64_t K, int N,
                                   int64_t ld_out, int8_t* __restrict__ spins, double* __restrict__ counts) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    const unsigned long long key = keys[k];
    for (int i = 0; i < N; ++i) spins[(int64_t)i * ld_out + k] = ((key >> i) & 1ull) ? 1 : -1;
    counts[k] = (double)run_len[k];
}

}  // namespace

void sort_key_runs(const unsigned long long* d_keys, int64_t M, int N, KeyRuns& runs, cudaStream_t st) {
    DevBuf<unsigned long long> keys_sorted;
    DevBuf<int> n_runs;
    keys_sorted.alloc(M); runs.uniq.alloc(M); runs.run_len.alloc(M); n_runs.alloc(1);
    size_t tmp_bytes = 0, tmp2 = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, d_keys, keys_sorted.p, (int)M, 0, N, st);
    cub::DeviceRunLengthEncode::Encode(nullptr, tmp2, keys_sorted.p, runs.uniq.p, runs.run_len.p, n_runs.p, (int)M, st);
    DevBuf<uint8_t> tmp;
    tmp.alloc(std::max(tmp_bytes, tmp2));
    GML_CUDA(cub::DeviceRadixSort::SortKeys(tmp.p, tmp_bytes, d_keys, keys_sorted.p, (int)M, 0, N, st));
    ++g_launches;
    GML_CUDA(cub::DeviceRunLengthEncode::Encode(tmp.p, tmp2, keys_sorted.p, runs.uniq.p, runs.run_len.p, n_runs.p, (int)M, st));
    ++g_launches;
    int hk = 0;
    GML_CUDA(cudaMemcpyAsync(&hk, n_runs.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    GML_CUDA(cudaStreamSynchronize(st));
    runs.K = hk;
}

void unpack_key_runs(const KeyRuns& runs, int N, int8_t* d_out_spins, int64_t ld_out, double* d_out_counts, cudaStream_t st) {
    unpack_keys_kernel<<<(unsigned)ceil_div(runs.K, 256), 256, 0, st>>>(runs.uniq.p, runs.run_len.p, runs.K, N, ld_out,
                                                                        d_out_spins, d_out_counts);
    GML_LAUNCHED();
}

int64_t build_histogram(const int8_t* d_samples, int64_t M, int N, int64_t ld, int8_t* d_out_spins, int64_t ld_out,
                        double* d_out_counts, cudaStream_t st) {
    GML_REQUIRE(N >= 1 && N <= 64, "device histogram builder supports 1 <= N <= 64 spins (64-bit keys)");
    GML_REQUIRE(M >= 1 && M < (1ll << 31), "device histogram builder supports up to 2^31-1 samples per call");
    DevBuf<unsigned long long> keys;
    DevBuf<int> flags;
    keys.alloc(M); flags.alloc(1);
    GML_CUDA(cudaMemsetAsync(flags.p, 0, sizeof(int), st));
    pack_keys_kernel<<<(unsigned)ceil_div(M, 256), 256, 0, st>>>(d_samples, ld, M, N, keys.p, flags.p);
    GML_LAUNCHED();
    KeyRuns runs;
    sort_key_runs(keys.p, M, N, runs, st);
    int hf = 0;
    GML_CUDA(cudaMemcpyAsync(&hf, flags.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    GML_CUDA(cudaStreamSynchronize(st));
    GML_REQUIRE(hf == 0, "samples must be exactly -1 or +1");
    GML_REQUIRE(ld_out >= runs.K, "output leading dimension smaller than the number of distinct configurations");
    unpack_key_runs(runs, N, d_out_spins, ld_out, d_out_counts, st);
    GML_CUDA(cudaStreamSynchronize(st));
    return runs.K;
}

}  // namespace gml
