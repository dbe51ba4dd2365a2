// Multi-sample Gibbs sampler for +-1 models  p(s) ~ exp( sum_t w_t prod_{i in t} s_i ),  N <= GML_B200_MCMC_MAX_N,
// term order <= 8: the sampler behind sample(gm, n, replicates, B200Gibbs()) for models beyond the exact sampler's cap.
//   - One warp advances 32 chains, one lane per chain.  The warp's state is N 32-bit words in shared memory: bit c of
//     word i is spin i of chain c.  Site i is updated for all 32 chains at once: every lane reads the same neighbour
//     words (a broadcast), computes its local field from the per-site incidence list (weight and other members of each
//     term containing i), draws its bit, and __ballot_sync assembles word i.  Control flow is warp-uniform and no chain
//     state lives in local memory.
//   - Schedule: burn_in systematic-scan sweeps from a random start, then the configuration at the end of every thin-th
//     sweep is recorded.  Draw d = r * chains + c is chain c's r-th record; the first n draws form the sample.
//   - Counter-based RNG on (seed, global chain, sweep, site) with global chain = replicate * chains + c: the output depends
//     on (model, n, seed, chains, burn_in, thin) and the replicate only, not on the grid or the device.
//   - Arithmetic: fp32 local fields from weights rounded once to fp32; a 24-bit uniform u draws +1 when
//     u < p_up = 1 / (1 + exp(-2h)), evaluated as u * (1 + exp(-2h)) < 1.
//   - Records: N <= 64: the chain's 64-bit key (bit i = spin i+1 up), built during the recording sweep, then sorted and
//     run-length encoded into a histogram (histogram.cu).  N > 64: int8 spin-major rows written during the recording sweep
//     (one 32-byte store per site and warp), count 1 each.
//   - Mixing diagnostic: per chain and half of its full record steps, fp64 sums and sums of squares of the energy
//     E(s) = sum_t w_t prod s (a warp-uniform pass over the term list after each recording sweep) and the magnetisation
//     sum_i s_i; folded into split-R-hat per replicate on the host.
//   - Replica exchange (R > 1 rungs, B200Tempering): a ladder is R consecutive lanes of a warp, so "chains" are ladders
//     (32/R per warp).  Each lane runs the model at its rung's inverse temperature beta (p_up = 1 / (1 + exp(-2 beta h)));
//     a swap exchanges the rung labels of two lanes and moves no spin words.  After sweep sw the pairs (k, k+1) with
//     k = sw (mod 2) are proposed (deterministic even-odd scheme) and accepted with probability
//     min(1, exp((beta_k - beta_{k+1}) (E_{k+1} - E_k))), E from an fp64 term-list pass after every sweep.  Only the lane
//     at rung 0 (beta = 1) records: draw d = r * ladders + ladder.  Order within a sweep: sweep, record, swap.
#include <cmath>
#include <type_traits>

#include "common.cuh"

namespace gml {
namespace {

constexpr int WARPS = 4;              // warps (groups of 32 chains) per block
#ifdef GML_MCMC_NO_ENERGY             // measurement build (build.py -DGML_MCMC_NO_ENERGY): without the energy pass
constexpr bool ENERGY_PASS = false;
#else
constexpr bool ENERGY_PASS = true;
#endif
constexpr uint32_t FULL = 0xffffffffu;

__device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL;
    x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL;
    x ^= x >> 33;
    return x;
}

// 32 random bits of step `ctr` (= sweep * N + site; sweep 0 is the random start) of the chain with key `chain_key`
__device__ __forceinline__ uint32_t rand32(uint64_t chain_key, uint64_t ctr) {
    return (uint32_t)(mix64(chain_key + (ctr + 1) * 0x9E3779B97F4A7C15ULL) >> 32);
}

constexpr uint64_t SWAP_CTR = 1ull << 63;   // swap counters: disjoint from the site counters sweep * N + site < 2^62

struct McmcParams {
    int N, order, width, n_terms;
    const int32_t* row_ptr;    // [N+1] per-site incidence lists
    const int32_t* others;     // [nnz x width] other members of the term of each entry, -1 padded
    const float* weight;       // [nnz]
    const int32_t* term_idx;   // [n_terms x order] members of each term, -1 padded (energy pass)
    const float* term_w;       // [n_terms]
    int64_t chains, chain0;    // chains per replicate; global id of this replicate's chain 0
    int64_t n;                 // draws of the replicate
    int64_t burn_in, thin, records;
    int64_t full_records;      // records of every chain (floor(n / chains)): the ones the diagnostic uses
    double inv_h, inv_h1;      // 1/h and 1/(h-1) for the half length h = full_records / 2
    uint64_t seed;
    unsigned long long* keys;  // N <= 64: [n] configuration keys
    int8_t* spins;             // N > 64: [N x ld] rows of the replicate (nullptr: count-only call)
    double* counts;
    int64_t ld;
    double* warp_stats;        // [warps x 6]: per statistic (energy, magnetisation) sum of half-chain means, of their
                               // squares and of the half-chain variances over the warp's chains
    unsigned long long* swap_acc;   // R > 1: [warps x (R-1)] swaps of pair (k, k+1) accepted after burn_in
    double beta[TEMPERING_MAX_RUNGS];  // R > 1: inverse temperature of each rung, beta[0] = 1
};

// parity (1 = odd) of the down spins of lane `lane` among the members m of a list (entries < 0 are padding)
__device__ __forceinline__ uint32_t down_parity(const uint32_t* __restrict__ s, const int32_t* __restrict__ members, int count,
                                                int lane) {
    uint32_t neg = 0;
    for (int m = 0; m < count; ++m) {
        const int j = __ldg(members + m);
        if (j >= 0) neg ^= ~(s[j] >> lane) & 1u;
    }
    return neg;
}

// Adds one record's value x to the sums of the half it belongs to (records [0, h) and [full - h, full), h = full / 2).
// The values are offsets from the chain's first record, so a statistic that stays constant sums to exactly 0.
__device__ __forceinline__ void add_half(int64_t r, int64_t h, int64_t full, double x, double& s0, double& q0, double& s1,
                                         double& q1) {
    if (r < h) { s0 += x; q0 += x * x; }
    else if (r >= full - h) { s1 += x; q1 += x * x; }
}

// mean and unbiased variance of a half-chain of h values from the sum and sum of squares of their offsets from x0
// (inv_h = 1/h, inv_h1 = 1/(h-1))
__device__ __forceinline__ void half_moments(double x0, double s, double q, double inv_h, double inv_h1, double& mean,
                                             double& var) {
    const double d = s * inv_h;
    mean = x0 + d;
    var = fmax(q - s * d, 0.0) * inv_h1;
}

// E(s) = sum_t w_t prod s of lane `lane`'s configuration, accumulated in T (a warp-uniform pass over the term list)
template <class T>
__device__ __forceinline__ T term_energy(const uint32_t* __restrict__ s, const McmcParams& p, int n_terms, int lane) {
    T energy = 0;
    for (int t = 0; t < n_terms; ++t) {
        const float w = __ldg(p.term_w + t);
        energy += down_parity(s, p.term_idx + (size_t)t * p.order, p.order, lane) ? -w : w;
    }
    return energy;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

// R = 1: multi-sample Gibbs, one chain per lane.  R > 1: one ladder of R rungs per R consecutive lanes (see the top).
template <bool KEYS, int R>
__global__ void __launch_bounds__(WARPS * 32) mcmc_kernel(McmcParams p) {
    using Energy = typename std::conditional<R == 1, float, double>::type;
    constexpr int LADDERS = 32 / R;                           // ladders (chains) per warp
    extern __shared__ uint32_t smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int slot = lane % R;                                // this lane's position in its ladder
    const int64_t warp = (int64_t)blockIdx.x * WARPS + wib;
    const int64_t c = warp * LADDERS + lane / R;             // chain (ladder) within the replicate
    if (warp * LADDERS >= p.chains) return;                  // a warp of the last block without chains: nothing to do
    const bool live = c < p.chains;
    uint32_t* s = smem + (size_t)wib * p.N;
    const int N = p.N;
    const uint64_t key = mix64(p.seed * 0xD1B54A32D192ED03ULL + mix64((uint64_t)((p.chain0 + c) * R + slot) + 1));
    // R > 1: rung = this lane's rung; who = the slot of the lane at rung `slot`; the ladder's swap stream is the key of
    // its slot-0 lane at counters SWAP_CTR + sw * R + k
    int rung = slot, who = slot;
    float beta = 1.f;
    uint64_t ladder_key = 0;
    unsigned long long n_acc = 0;                             // accepted swaps of pair (slot, slot + 1) after burn_in
    if constexpr (R > 1) {
        ladder_key = __shfl_sync(FULL, (unsigned long long)key, 0, R);
        beta = (float)p.beta[slot];
    }

    for (int i = 0; i < N; ++i) {                             // random start (sweep 0)
        const uint32_t w = __ballot_sync(FULL, rand32(key, (uint64_t)i) >> 31);
        if (lane == 0) s[i] = w;
    }
    __syncwarp();

    const int64_t h = p.full_records / 2;
    double es0 = 0, eq0 = 0, es1 = 0, eq1 = 0, ms0 = 0, mq0 = 0, ms1 = 0, mq1 = 0;
    Energy e_first = 0;                                       // the statistics of the chain's first record
    int m_first = 0;
    const int64_t sweeps = p.burn_in + p.records * p.thin;
    int64_t next_rec = p.burn_in + p.thin, r = -1;           // the sweep that ends with the next record, its index
    for (int64_t sw = 1; sw <= sweeps; ++sw) {
        const bool rec = sw == next_rec;                      // warp-uniform
        if (rec) { ++r; next_rec += p.thin; }
        const int64_t d = r * p.chains + c;
        const bool out = rec && live && d < p.n && rung == 0;
        unsigned long long cfg = 0;
        int ups = 0;
        const uint64_t ctr0 = (uint64_t)sw * (uint64_t)N;
        for (int i = 0; i < N; ++i) {
            float field = 0.f;
            const int b = __ldg(p.row_ptr + i), e = __ldg(p.row_ptr + i + 1);
            for (int q = b; q < e; ++q) {
                const float w = __ldg(p.weight + q);
                field += down_parity(s, p.others + (size_t)q * p.width, p.width, lane) ? -w : w;
            }
            if constexpr (R > 1) field *= beta;               // beta = 1 leaves the field exact
            // u < p_up = 1 / (1 + exp(-2h)), tested as u * (1 + exp(-2h)) < 1: no division (whose slow path costs a stack frame)
            const float u = (float)(rand32(key, ctr0 + i) >> 8) * 0x1.0p-24f;
            const uint32_t bit = u * (1.f + expf(-2.f * field)) < 1.f ? 1u : 0u;
            const uint32_t word = __ballot_sync(FULL, bit);
            if (lane == 0) s[i] = word;
            __syncwarp();
            if (rec) {
                ups += bit;
                if (KEYS) cfg |= (unsigned long long)bit << i;
                else if (out && p.spins) p.spins[(int64_t)i * p.ld + d] = bit ? 1 : -1;
            }
        }
        double energy_now = 0;                                // R > 1: the energy of every lane, for the swap test
        if constexpr (R > 1) energy_now = term_energy<double>(s, p, p.n_terms, lane);
        if (rec) {
            if (out) {
                if (KEYS) p.keys[d] = cfg;
                else if (p.counts) p.counts[d] = 1.0;
            }
            if (r < p.full_records && h >= 2) {
                Energy energy;
                int mag;
                if constexpr (R == 1) {
                    energy = term_energy<float>(s, p, ENERGY_PASS ? p.n_terms : 0, lane);
                    mag = 2 * ups - N;
                } else {                                      // the rung-0 lane's statistics, kept in every lane
                    const int at0 = __shfl_sync(FULL, who, 0, R);
                    energy = __shfl_sync(FULL, energy_now, at0, R);
                    mag = 2 * __shfl_sync(FULL, ups, at0, R) - N;
                }
                if (r == 0) { e_first = energy; m_first = mag; }
                add_half(r, h, p.full_records, (double)energy - (double)e_first, es0, eq0, es1, eq1);
                add_half(r, h, p.full_records, (double)(mag - m_first), ms0, mq0, ms1, mq1);
            }
        }
        if constexpr (R > 1) {                                // swap: slot k decides the pair (rung k, rung k + 1)
            const double e_k = __shfl_sync(FULL, energy_now, who, R);
            const double e_k1 = __shfl_down_sync(FULL, e_k, 1, R);
            const int who_up = __shfl_down_sync(FULL, who, 1, R), who_down = __shfl_up_sync(FULL, who, 1, R);
            bool acc = false;
            if (((slot ^ (int)sw) & 1) == 0 && slot + 1 < R) {
                const double x = (p.beta[slot] - p.beta[slot + 1]) * (e_k1 - e_k);
                const double u = (double)rand32(ladder_key, SWAP_CTR + (uint64_t)sw * R + slot) * 0x1.0p-32;
                acc = x >= 0.0 || u < exp(x);
                if (acc && live && sw > p.burn_in) ++n_acc;
            }
            const bool acc_below = __shfl_up_sync(FULL, (int)acc, 1, R) && slot > 0;   // pair (slot - 1, slot) swapped
            const int delta = acc ? 1 : acc_below ? -1 : 0;
            who = acc ? who_up : acc_below ? who_down : who;
            rung += __shfl_sync(FULL, delta, rung, R);
            beta = (float)p.beta[rung];
        }
    }

    if constexpr (R > 1) {                                    // per pair, the sum over the warp's ladders
#pragma unroll
        for (int o = R; o < 32; o <<= 1) n_acc += __shfl_xor_sync(FULL, n_acc, o);
        if (lane < R - 1) p.swap_acc[warp * (R - 1) + lane] = n_acc;
    }
    if (h < 2) return;
    double em = 0, em2 = 0, ev = 0, mm = 0, mm2 = 0, mv = 0;
    if (live && slot == 0) {
        double m0, v0, m1, v1;
        half_moments(e_first, es0, eq0, p.inv_h, p.inv_h1, m0, v0); half_moments(e_first, es1, eq1, p.inv_h, p.inv_h1, m1, v1);
        em = m0 + m1; em2 = m0 * m0 + m1 * m1; ev = v0 + v1;
        half_moments(m_first, ms0, mq0, p.inv_h, p.inv_h1, m0, v0); half_moments(m_first, ms1, mq1, p.inv_h, p.inv_h1, m1, v1);
        mm = m0 + m1; mm2 = m0 * m0 + m1 * m1; mv = v0 + v1;
    }
    em = warp_sum(em); em2 = warp_sum(em2); ev = warp_sum(ev);
    mm = warp_sum(mm); mm2 = warp_sum(mm2); mv = warp_sum(mv);
    if (lane == 0) {
        double* o = p.warp_stats + warp * 6;
        o[0] = em; o[1] = em2; o[2] = ev; o[3] = mm; o[4] = mm2; o[5] = mv;
    }
}

// split-R-hat of one statistic from the sums over M half-chains of h records each (Gelman et al., BDA3 sec. 11.4).
// W = 0 means every half-chain held one value throughout: R-hat is then 1 when all half-chains held the same value (a
// constant statistic has nothing to diagnose; the 1e-12 relative slack only absorbs the rounding of the sums) and +inf
// when they held different values (chains frozen apart).
double split_rhat(double sum_mean, double sum_mean2, double sum_var, double M, double h) {
    const double W = sum_var / M;
    const double mbar = sum_mean / M;
    const double B_over_h = std::max(sum_mean2 - M * mbar * mbar, 0.0) / (M - 1.0);
    if (W == 0.0) return B_over_h <= 1e-12 * mbar * mbar ? 1.0 : INFINITY;
    return std::sqrt(((h - 1.0) / h * W + B_over_h) / W);
}

}  // namespace

int64_t mcmc_auto_chains(int64_t n, int rungs) {
    return std::min<int64_t>(round_up(n, 32 / rungs), MCMC_AUTO_CHAINS / rungs);
}

namespace {
template <bool KEYS> void (*ladder_kernel(int rungs))(McmcParams) {
    switch (rungs) {
        case 1: return mcmc_kernel<KEYS, 1>;
        case 2: return mcmc_kernel<KEYS, 2>;
        case 4: return mcmc_kernel<KEYS, 4>;
        case 8: return mcmc_kernel<KEYS, 8>;
        case 16: return mcmc_kernel<KEYS, 16>;
        default: return mcmc_kernel<KEYS, 32>;
    }
}
}  // namespace

void sample_mcmc(int N, int order, const std::vector<int32_t>& term_idx, const std::vector<double>& term_weight,
                 const Incidence& inc, const std::vector<double>& betas, int64_t n_samples, int replicates, int64_t chains,
                 int64_t burn_in, int64_t thin, uint64_t seed, int64_t* out_K, double* out_rhat, double* out_swap_rate,
                 double* d_counts, int8_t* d_spins, int64_t ld, cudaStream_t st) {
    const bool keys_path = N <= 64;
    const int n_terms = (int)term_weight.size();
    const int rungs = (int)betas.size();
    const int64_t warps = ceil_div(chains, 32 / rungs), blocks = ceil_div(warps, WARPS);
    const size_t smem = sizeof(uint32_t) * (size_t)N * WARPS;
    std::vector<float> w32(term_weight.begin(), term_weight.end());
    std::vector<float> inc_w(inc.term.size());
    for (size_t q = 0; q < inc.term.size(); ++q) inc_w[q] = inc.term[q] >= 0 ? (float)term_weight[inc.term[q]] : 0.f;

    DevBuf<int32_t> rp, ot, ti;
    DevBuf<float> ww, tw;
    DevBuf<double> wstats;
    DevBuf<unsigned long long> keys, swaps;
    rp.alloc(inc.row_ptr.size()); ot.alloc(inc.others.size()); ww.alloc(inc_w.size());
    ti.alloc(std::max<size_t>(term_idx.size(), 1)); tw.alloc(std::max<size_t>(w32.size(), 1));
    wstats.alloc(warps * 6);
    if (rungs > 1) swaps.alloc(warps * (rungs - 1));
    if (keys_path) keys.alloc(n_samples);
    GML_CUDA(cudaMemcpyAsync(rp.p, inc.row_ptr.data(), sizeof(int32_t) * inc.row_ptr.size(), cudaMemcpyHostToDevice, st));
    GML_CUDA(cudaMemcpyAsync(ot.p, inc.others.data(), sizeof(int32_t) * inc.others.size(), cudaMemcpyHostToDevice, st));
    GML_CUDA(cudaMemcpyAsync(ww.p, inc_w.data(), sizeof(float) * inc_w.size(), cudaMemcpyHostToDevice, st));
    if (n_terms) {
        GML_CUDA(cudaMemcpyAsync(ti.p, term_idx.data(), sizeof(int32_t) * term_idx.size(), cudaMemcpyHostToDevice, st));
        GML_CUDA(cudaMemcpyAsync(tw.p, w32.data(), sizeof(float) * n_terms, cudaMemcpyHostToDevice, st));
    }
    auto kernel = keys_path ? ladder_kernel<true>(rungs) : ladder_kernel<false>(rungs);
    GML_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));

    McmcParams p{};
    p.N = N; p.order = order; p.width = inc.width; p.n_terms = n_terms;
    p.row_ptr = rp.p; p.others = ot.p; p.weight = ww.p; p.term_idx = ti.p; p.term_w = tw.p;
    p.chains = chains; p.n = n_samples; p.burn_in = burn_in; p.thin = thin;
    p.records = ceil_div(n_samples, chains); p.full_records = n_samples / chains;
    p.seed = seed; p.keys = keys.p; p.warp_stats = wstats.p; p.swap_acc = swaps.p;
    for (int k = 0; k < rungs; ++k) p.beta[k] = betas[k];
    const int64_t h = p.full_records / 2;
    p.inv_h = 1.0 / (double)h;
    p.inv_h1 = 1.0 / (double)(h - 1);
    const int64_t sweeps = burn_in + p.records * thin;
    std::vector<double> hs(warps * 6);
    std::vector<unsigned long long> accepted(rungs > 1 ? warps * (rungs - 1) : 0);
    auto with_parity = [](int64_t x, int par) { return par ? (x + 1) / 2 : x / 2; };   // sw in [1, x] with sw = par (mod 2)
    int64_t rows = 0;
    bool fits = true;
    for (int rep = 0; rep < replicates; ++rep) {
        p.chain0 = (int64_t)rep * chains;
        const bool write = d_counts && !keys_path && rows + n_samples <= ld;
        p.spins = write ? d_spins + rows : nullptr;
        p.counts = write ? d_counts + rows : nullptr;
        p.ld = ld;
        kernel<<<(unsigned)blocks, WARPS * 32, smem, st>>>(p);
        GML_LAUNCHED();
        int64_t K = n_samples;
        if (keys_path) {
            KeyRuns runs;
            sort_key_runs(keys.p, n_samples, N, runs, st);
            K = runs.K;
            if (d_counts && rows + K <= ld) unpack_key_runs(runs, N, d_spins + rows, ld, d_counts + rows, st);
            GML_CUDA(cudaStreamSynchronize(st));         // before the runs' buffers are released
        }
        out_K[rep] = K;
        fits = fits && rows + K <= ld;
        rows += K;
        if (out_rhat) {
            double* rh = out_rhat + 2 * rep;
            rh[0] = rh[1] = NAN;
            if (h >= 2) {
                GML_CUDA(cudaMemcpyAsync(hs.data(), wstats.p, sizeof(double) * hs.size(), cudaMemcpyDeviceToHost, st));
                GML_CUDA(cudaStreamSynchronize(st));
                double acc[6] = {0, 0, 0, 0, 0, 0};
                for (int64_t w = 0; w < warps; ++w)
                    for (int k = 0; k < 6; ++k) acc[k] += hs[w * 6 + k];
                rh[0] = split_rhat(acc[0], acc[1], acc[2], 2.0 * chains, (double)h);
                rh[1] = split_rhat(acc[3], acc[4], acc[5], 2.0 * chains, (double)h);
            }
        }
        if (out_swap_rate && rungs > 1) {                    // accepted / proposed swaps after burn_in, per pair
            GML_CUDA(cudaMemcpyAsync(accepted.data(), swaps.p, sizeof(unsigned long long) * accepted.size(), cudaMemcpyDeviceToHost,
                                     st));
            GML_CUDA(cudaStreamSynchronize(st));
            for (int k = 0; k + 1 < rungs; ++k) {
                unsigned long long a = 0;
                for (int64_t w = 0; w < warps; ++w) a += accepted[w * (rungs - 1) + k];
                // the sweeps sw in (burn_in, sweeps] with sw = k (mod 2) propose pair k in every ladder
                const int64_t proposals = with_parity(sweeps, k % 2) - with_parity(burn_in, k % 2);
                out_swap_rate[(size_t)rep * (rungs - 1) + k] = proposals > 0 ? (double)a / ((double)proposals * chains) : NAN;
            }
        }
    }
    GML_CUDA(cudaStreamSynchronize(st));
    GML_REQUIRE(!d_counts || fits, "ld = " + std::to_string(ld) + " is smaller than the " + std::to_string(rows) +
                                   " rows of the replicates (out_K holds their sizes)");
}

}  // namespace gml
