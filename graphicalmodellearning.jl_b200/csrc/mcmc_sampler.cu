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
//   - Partition function (R > 1, BRIDGE, log_partition(gm, B200Tempering())): on every sweep after burn_in,
//     before the swap, the lane at slot k < R-1 adds x = +dbeta_k E_{k+1} / 2 and y = -dbeta_k E_k / 2 (dbeta_k = beta_k -
//     beta_{k+1}) to two running log-sum-exps (running maximum, so nothing overflows) and finally writes their log-means:
//     the two halves of the geometric bridge log Z_k - log Z_{k+1} = log E_{k+1}[e^x] - log E_k[e^y] (Meng & Wong 1996).
//     The RNG streams and the swap decisions are those of the sampler.
//   - Moments (RECORD, moments(gm, sampler)): after every recording sweep each warp copies its N state words and a 32-bit
//     mask of the lanes whose record is a draw (live && d < n && rung == 0) to column r * warps + warp of a spin-major
//     record buffer [(N+1) x records * warps] (row N = the masks); nothing else is written.  moments.cu reduces it.
//   - Persistent chains (PERSIST, R = 1, fit_likelihood(gm, samples, B200Gibbs())): a launch runs sweeps sweep0 + 1 ..
//     sweep0 + thin of the chains of one long run, so the site counters sweep * N + site continue across launches while
//     the caller rewrites the weights between them.  The state lives in a record buffer [(N+1) x warps]: a launch with
//     sweep0 > 0 loads its warp's column, and every launch stores its final state words and the mask of its live lanes
//     there (one record per launch, column = warp).  No draws, energies or R-hat sums.
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
    double* bridge;            // BRIDGE: [chains x (R-1) x 2] per ladder and pair k the log-means of e^x and e^y
    uint32_t* record;          // RECORD: [(N+1) x ld_rec] state words and draw masks, column r * rec_warps + warp
    int64_t rec_warps, ld_rec; // RECORD: warps of the grid, records * rec_warps
    int64_t sweep0;            // PERSIST: the sweeps of this launch are sweep0 + 1 .. sweep0 + thin
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

// adds x to the running log-sum-exp  m + log(sum).  One exp on either side of the maximum (m = -inf: e = 0), in fp32:
// e is in (0, 1], its relative error ~1e-7 moves the log-sum by as little, and an fp64 exp's constants would take the
// registers of the sweep loop.
__device__ __forceinline__ void log_sum_exp_add(double x, double& m, double& sum) {
    const double e = expf((float)-fabs(x - m));
    sum = x > m ? fma(sum, e, 1.0) : sum + e;
    m = fmax(m, x);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

// R = 1: multi-sample Gibbs, one chain per lane.  R > 1: one ladder of R rungs per R consecutive lanes (see the top);
// BRIDGE adds the sums of the log Z estimator, RECORD the record buffer of the moments, PERSIST (R = 1) the persistent
// chains of fit_likelihood (separate instantiations: the sampler's registers stay as they are).
template <bool KEYS, int R, bool BRIDGE = false, bool RECORD = false, bool PERSIST = false>
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
    double a_max = -INFINITY, a_sum = 0, b_max = -INFINITY, b_sum = 0;   // the bridge sums of pair (slot, slot + 1)
    if constexpr (R > 1) {
        ladder_key = __shfl_sync(FULL, (unsigned long long)key, 0, R);
        beta = (float)p.beta[slot];
    }

    if (PERSIST && p.sweep0 > 0) {                            // resume from the state the previous launch stored
        const uint32_t* src = p.record + warp;
#pragma unroll 1
        for (int i = lane; i < N; i += 32) s[i] = src[(int64_t)i * p.ld_rec];
    } else {
        for (int i = 0; i < N; ++i) {                         // random start (sweep 0)
            const uint32_t w = __ballot_sync(FULL, rand32(key, (uint64_t)i) >> 31);
            if (lane == 0) s[i] = w;
        }
    }
    __syncwarp();

    const int64_t h = p.full_records / 2;
    double es0 = 0, eq0 = 0, es1 = 0, eq1 = 0, ms0 = 0, mq0 = 0, ms1 = 0, mq1 = 0;
    Energy e_first = 0;                                       // the statistics of the chain's first record
    int m_first = 0;
    const int64_t sweeps = PERSIST ? p.sweep0 + p.thin : p.burn_in + p.records * p.thin;
    int64_t next_rec = p.burn_in + p.thin, r = -1;           // the sweep that ends with the next record, its index
    for (int64_t sw = PERSIST ? p.sweep0 + 1 : 1; sw <= sweeps; ++sw) {
        const bool rec = !PERSIST && sw == next_rec;          // warp-uniform
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
        if (RECORD && rec) {
            const uint32_t draws = __ballot_sync(FULL, out);
            uint32_t* dst = p.record + r * p.rec_warps + warp + lane * p.ld_rec;
#pragma unroll 1
            for (int i = lane; i < N; i += 32, dst += 32 * p.ld_rec) *dst = s[i];
            if (lane == 0) p.record[N * p.ld_rec + r * p.rec_warps + warp] = draws;
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
            if (BRIDGE && sw > p.burn_in && slot + 1 < R) {
                const double half = 0.5 * (p.beta[slot] - p.beta[slot + 1]);
                log_sum_exp_add(half * e_k1, a_max, a_sum);
                log_sum_exp_add(-half * e_k, b_max, b_sum);
            }
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

    if constexpr (PERSIST) {                                  // the final state and the mask of the live lanes
        const uint32_t live_mask = __ballot_sync(FULL, live);
        uint32_t* dst = p.record + warp + lane * p.ld_rec;
#pragma unroll 1
        for (int i = lane; i < N; i += 32, dst += 32 * p.ld_rec) *dst = s[i];
        if (lane == 0) p.record[N * p.ld_rec + warp] = live_mask;
        return;
    }
    if constexpr (R > 1) {                                    // per pair, the sum over the warp's ladders
#pragma unroll
        for (int o = R; o < 32; o <<= 1) n_acc += __shfl_xor_sync(FULL, n_acc, o);
        if (lane < R - 1) p.swap_acc[warp * (R - 1) + lane] = n_acc;
        if (BRIDGE && live && slot + 1 < R) {               // log-means over the records * thin sweeps after burn_in
            const double log_s = log((double)(p.records * p.thin));
            double* o = p.bridge + (c * (R - 1) + slot) * 2;
            o[0] = a_max + log(a_sum) - log_s;
            o[1] = b_max + log(b_sum) - log_s;
        }
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

// --- Swendsen-Wang cluster sampler (B200SwendsenWang) for pairwise models, Edwards-Sokal form with a ghost spin -----
// Node 0 is a ghost spin fixed at +1 and node i + 1 is spin i, so a field (i,) is a bond between i + 1 and the ghost.
// One update (a "sweep" for burn_in and thin): term t = (a, b) with w_t s_a s_b > 0 bonds unless u_t < q_t =
// e^{-2|w_t|} (u_t a 64-bit uniform, q_t = bond_q[t] / 2^64 from fp64 on the host); every cluster without the ghost
// flips with probability 1/2.  The warp keeps mcmc_kernel's state words and updates its 32 chains one after another,
// lanes striding over terms and sites: the union-find hooks the larger root under the smaller, so every root is the least
// node of its cluster and the labels do not depend on the order of the hooks.  Counters per sweep: bond t at sw * S + t,
// the flip of root r at sw * S + n_bonds + r, S = n_bonds + N + 1; sweep 0 is mcmc_kernel's random start.
constexpr int CLUSTER_WARPS = 2;      // 24.6 KB of shared memory per warp at N = 4096: 4 blocks (8 warps) per SM

struct ClusterParams {
    McmcParams m;                      // the model's term list (energy pass), the run and the outputs, as for mcmc_kernel
    int n_bonds;
    const uint32_t* bond_ends;         // [n_bonds] node a | node b << 16 | (w_t < 0) << 31, a in [1, N], b in [0, N]
    const unsigned long long* bond_q;  // [n_bonds] round(e^{-2|w_t|} 2^64)
};

// 64 random bits of step `ctr` of the chain with key `chain_key` (rand32 is their upper half)
__device__ __forceinline__ uint64_t rand64(uint64_t chain_key, uint64_t ctr) {
    return mix64(chain_key + (ctr + 1) * 0x9E3779B97F4A7C15ULL);
}

// the root of x; volatile: other lanes hook roots while this lane walks
__device__ __forceinline__ int uf_find(const volatile uint16_t* par, int x) {
    int p = par[x];
    while (p != x) { x = p; p = par[x]; }
    return x;
}

// joins the clusters of a and b: hooks the larger root under the smaller with a CAS, retrying when another lane moved it
__device__ __forceinline__ void uf_union(uint16_t* par, int a, int b) {
    while (true) {
        a = uf_find(par, a);
        b = uf_find(par, b);
        if (a == b) return;
        if (a < b) { const int t = a; a = b; b = t; }
        if (atomicCAS(reinterpret_cast<unsigned short*>(par + a), (unsigned short)a, (unsigned short)b) == a) return;
    }
}

template <bool KEYS, bool RECORD>
__global__ void __launch_bounds__(CLUSTER_WARPS * 32, 1) cluster_kernel(ClusterParams cp) {
    const McmcParams& p = cp.m;
    extern __shared__ uint32_t smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t warp = (int64_t)blockIdx.x * CLUSTER_WARPS + wib;
    const int64_t c = warp * 32 + lane;
    if (warp * 32 >= p.chains) return;
    const bool live = c < p.chains;
    const int N = p.N, n_bonds = cp.n_bonds;
    uint32_t* s = smem + (size_t)wib * N;
    uint16_t* par = reinterpret_cast<uint16_t*>(smem + (size_t)CLUSTER_WARPS * N) + (size_t)wib * (N + 1);
    const int chains_here = p.chains - warp * 32 < 32 ? (int)(p.chains - warp * 32) : 32;   // live chains of the warp
    const uint64_t key = mix64(p.seed * 0xD1B54A32D192ED03ULL + mix64((uint64_t)(p.chain0 + c) + 1));
    for (int i = 0; i < N; ++i) {                             // random start (sweep 0), as mcmc_kernel's
        const uint32_t w = __ballot_sync(FULL, rand32(key, (uint64_t)i) >> 31);
        if (lane == 0) s[i] = w;
    }
    __syncwarp();

    const int64_t h = p.full_records / 2;
    double es0 = 0, eq0 = 0, es1 = 0, eq1 = 0, ms0 = 0, mq0 = 0, ms1 = 0, mq1 = 0;
    float e_first = 0;
    int m_first = 0;
    const uint64_t stride = (uint64_t)n_bonds + N + 1;
    const int64_t sweeps = p.burn_in + p.records * p.thin;
    int64_t next_rec = p.burn_in + p.thin, r = -1;
    for (int64_t sw = 1; sw <= sweeps; ++sw) {
        const uint64_t ctr0 = (uint64_t)sw * stride;
#pragma unroll 1
        for (int cc = 0; cc < chains_here; ++cc) {
            const uint64_t ck = __shfl_sync(FULL, (unsigned long long)key, cc);
            for (int i = lane; i <= N; i += 32) par[i] = (uint16_t)i;
            __syncwarp();
            for (int t = lane; t < n_bonds; t += 32) {        // bonds of the satisfied terms
                const uint32_t ends = __ldg(cp.bond_ends + t);
                const int a = ends & 0xffff, b = (ends >> 16) & 0x7fff;
                const uint32_t sa = (s[a - 1] >> cc) & 1u, sb = b ? (s[b - 1] >> cc) & 1u : 1u;
                if ((sa ^ sb) != (ends >> 31)) continue;      // w_t s_a s_b < 0: never bonds
                if (rand64(ck, ctr0 + t) < __ldg(cp.bond_q + t)) continue;   // u_t < q_t: no bond
                uf_union(par, a, b);
            }
            __syncwarp();
            for (int i = lane; i <= N; i += 32) par[i] = (uint16_t)uf_find(par, i);
            __syncwarp();
            for (int i = lane; i < N; i += 32) {              // flip the clusters whose root drew 1, never the ghost's
                const int root = par[i + 1];
                if (root != 0 && rand32(ck, ctr0 + n_bonds + root) >> 31) s[i] ^= 1u << cc;
            }
            __syncwarp();
        }
        if (sw != next_rec) continue;
        ++r;
        next_rec += p.thin;
        const int64_t d = r * p.chains + c;
        const bool out = live && d < p.n;
        unsigned long long cfg = 0;
        int ups = 0;
        for (int i = 0; i < N; ++i) {
            const uint32_t bit = (s[i] >> lane) & 1u;
            ups += bit;
            if (KEYS) cfg |= (unsigned long long)bit << i;
            else if (out && p.spins) p.spins[(int64_t)i * p.ld + d] = bit ? 1 : -1;
        }
        if (RECORD) {
            const uint32_t draws = __ballot_sync(FULL, out);
            uint32_t* dst = p.record + r * p.rec_warps + warp + lane * p.ld_rec;
#pragma unroll 1
            for (int i = lane; i < N; i += 32, dst += 32 * p.ld_rec) *dst = s[i];
            if (lane == 0) p.record[N * p.ld_rec + r * p.rec_warps + warp] = draws;
        }
        if (out) {
            if (KEYS) p.keys[d] = cfg;
            else if (p.counts) p.counts[d] = 1.0;
        }
        if (r < p.full_records && h >= 2) {
            const float energy = term_energy<float>(s, p, p.n_terms, lane);
            const int mag = 2 * ups - N;
            if (r == 0) { e_first = energy; m_first = mag; }
            add_half(r, h, p.full_records, (double)energy - (double)e_first, es0, eq0, es1, eq1);
            add_half(r, h, p.full_records, (double)(mag - m_first), ms0, mq0, ms1, mq1);
        }
    }

    if (h < 2) return;
    double em = 0, em2 = 0, ev = 0, mm = 0, mm2 = 0, mv = 0;
    if (live) {
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

void (*bridge_kernel(int rungs))(McmcParams) {
    switch (rungs) {
        case 2: return mcmc_kernel<false, 2, true>;
        case 4: return mcmc_kernel<false, 4, true>;
        case 8: return mcmc_kernel<false, 8, true>;
        case 16: return mcmc_kernel<false, 16, true>;
        default: return mcmc_kernel<false, 32, true>;
    }
}

void (*record_kernel(int rungs))(McmcParams) {
    switch (rungs) {
        case 1: return mcmc_kernel<false, 1, false, true>;
        case 2: return mcmc_kernel<false, 2, false, true>;
        case 4: return mcmc_kernel<false, 4, false, true>;
        case 8: return mcmc_kernel<false, 8, false, true>;
        case 16: return mcmc_kernel<false, 16, false, true>;
        default: return mcmc_kernel<false, 32, false, true>;
    }
}

// The bond list of a cluster run on the device, and its launches
struct ClusterRun {
    DevBuf<uint32_t> ends;
    DevBuf<unsigned long long> q;
    int n_bonds;

    ClusterRun(const ClusterBonds& b, cudaStream_t st) : n_bonds((int)b.ends.size()) {
        ends.alloc(std::max<size_t>(b.ends.size(), 1)); q.alloc(std::max<size_t>(b.q.size(), 1));
        if (n_bonds) {
            GML_CUDA(cudaMemcpyAsync(ends.p, b.ends.data(), sizeof(uint32_t) * n_bonds, cudaMemcpyHostToDevice, st));
            GML_CUDA(cudaMemcpyAsync(q.p, b.q.data(), sizeof(unsigned long long) * n_bonds, cudaMemcpyHostToDevice, st));
        }
    }

    template <bool KEYS, bool RECORD> void launch(const McmcParams& p, int64_t warps, cudaStream_t st) const {
        // per warp: N state words and N + 1 16-bit parents
        const size_t smem = CLUSTER_WARPS * (sizeof(uint32_t) * (size_t)p.N + sizeof(uint16_t) * (size_t)(p.N + 1));
        GML_CUDA(cudaFuncSetAttribute(cluster_kernel<KEYS, RECORD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cluster_kernel<KEYS, RECORD><<<(unsigned)ceil_div(warps, CLUSTER_WARPS), CLUSTER_WARPS * 32, smem, st>>>(
            ClusterParams{p, n_bonds, ends.p, q.p});
        GML_LAUNCHED();
    }
};

// A model on the device for mcmc_kernel: the incidence lists and the term list with weights rounded once to fp32, and the
// parameters that describe the model and the ladder.  The caller fills in the run.
struct DeviceModel {
    DevBuf<int32_t> rp, ot, ti;
    DevBuf<float> ww, tw;
    std::vector<float> w32, inc_w;                    // the host sources of the fp32 weights
    McmcParams p{};

    DeviceModel(int N, int order, const std::vector<int32_t>& term_idx, const std::vector<double>& term_weight,
                const Incidence& inc, const std::vector<double>& betas, cudaStream_t st)
        : w32(term_weight.begin(), term_weight.end()), inc_w(inc.term.size()) {
        const int n_terms = (int)term_weight.size();
        for (size_t q = 0; q < inc.term.size(); ++q) inc_w[q] = inc.term[q] >= 0 ? (float)term_weight[inc.term[q]] : 0.f;
        rp.alloc(inc.row_ptr.size()); ot.alloc(inc.others.size()); ww.alloc(inc_w.size());
        ti.alloc(std::max<size_t>(term_idx.size(), 1)); tw.alloc(std::max<size_t>(w32.size(), 1));
        GML_CUDA(cudaMemcpyAsync(rp.p, inc.row_ptr.data(), sizeof(int32_t) * inc.row_ptr.size(), cudaMemcpyHostToDevice, st));
        GML_CUDA(cudaMemcpyAsync(ot.p, inc.others.data(), sizeof(int32_t) * inc.others.size(), cudaMemcpyHostToDevice, st));
        GML_CUDA(cudaMemcpyAsync(ww.p, inc_w.data(), sizeof(float) * inc_w.size(), cudaMemcpyHostToDevice, st));
        if (n_terms) {
            GML_CUDA(cudaMemcpyAsync(ti.p, term_idx.data(), sizeof(int32_t) * term_idx.size(), cudaMemcpyHostToDevice, st));
            GML_CUDA(cudaMemcpyAsync(tw.p, w32.data(), sizeof(float) * n_terms, cudaMemcpyHostToDevice, st));
        }
        p.N = N; p.order = order; p.width = inc.width; p.n_terms = n_terms;
        p.row_ptr = rp.p; p.others = ot.p; p.weight = ww.p; p.term_idx = ti.p; p.term_w = tw.p;
        for (size_t k = 0; k < betas.size(); ++k) p.beta[k] = betas[k];
    }
};

// split-R-hat (energy, magnetisation) into rh[2] from the per-warp sums of warp_stats over half-chains of h records
void rhat_of(const double* warp_stats, int64_t warps, int64_t chains, int64_t h, double* rh, cudaStream_t st) {
    rh[0] = rh[1] = NAN;
    if (h < 2) return;
    std::vector<double> hs(warps * 6);
    GML_CUDA(cudaMemcpyAsync(hs.data(), warp_stats, sizeof(double) * hs.size(), cudaMemcpyDeviceToHost, st));
    GML_CUDA(cudaStreamSynchronize(st));
    double acc[6] = {0, 0, 0, 0, 0, 0};
    for (int64_t w = 0; w < warps; ++w)
        for (int k = 0; k < 6; ++k) acc[k] += hs[w * 6 + k];
    rh[0] = split_rhat(acc[0], acc[1], acc[2], 2.0 * chains, (double)h);
    rh[1] = split_rhat(acc[3], acc[4], acc[5], 2.0 * chains, (double)h);
}

// per adjacent pair, accepted / proposed swaps after burn_in from the per-warp counts of swap_acc
void swap_rates(const unsigned long long* swap_acc, int64_t warps, int rungs, int64_t chains, int64_t burn_in, int64_t sweeps,
                double* out, cudaStream_t st) {
    std::vector<unsigned long long> accepted(warps * (rungs - 1));
    GML_CUDA(cudaMemcpyAsync(accepted.data(), swap_acc, sizeof(unsigned long long) * accepted.size(), cudaMemcpyDeviceToHost, st));
    GML_CUDA(cudaStreamSynchronize(st));
    auto with_parity = [](int64_t x, int par) { return par ? (x + 1) / 2 : x / 2; };   // sw in [1, x] with sw = par (mod 2)
    for (int k = 0; k + 1 < rungs; ++k) {
        unsigned long long a = 0;
        for (int64_t w = 0; w < warps; ++w) a += accepted[w * (rungs - 1) + k];
        // the sweeps sw in (burn_in, sweeps] with sw = k (mod 2) propose pair k in every ladder
        const int64_t proposals = with_parity(sweeps, k % 2) - with_parity(burn_in, k % 2);
        out[k] = proposals > 0 ? (double)a / ((double)proposals * chains) : NAN;
    }
}
}  // namespace

ClusterBonds cluster_bonds(int order, const std::vector<int32_t>& term_idx, const std::vector<double>& term_weight) {
    ClusterBonds b;
    for (size_t t = 0; t < term_weight.size(); ++t) {
        int node[2] = {0, 0}, k = 0;
        for (int m = 0; m < order; ++m) {
            const int i = term_idx[t * order + m];
            if (i < 0) continue;
            GML_REQUIRE(k < 2, "the Swendsen-Wang sampler takes terms of one or two spins only");
            node[k++] = i + 1;
        }
        const double q = std::exp(-2.0 * std::fabs(term_weight[t]));
        if (k == 0 || q == 1.0) continue;                      // a constant, or |w| < 2^-54: never bonds
        const uint32_t a = std::max(node[0], node[1]), c = std::min(node[0], node[1]);   // c = 0: the ghost
        b.ends.push_back(a | c << 16 | (term_weight[t] < 0.0 ? 1u << 31 : 0u));
        b.q.push_back((unsigned long long)(q * 0x1p64));       // rounded down: exact for q >= 2^-11, within 2^-64 below
    }
    return b;
}

void sample_mcmc(int N, int order, const std::vector<int32_t>& term_idx, const std::vector<double>& term_weight,
                 const Incidence& inc, const std::vector<double>& betas, int64_t n_samples, int replicates, int64_t chains,
                 int64_t burn_in, int64_t thin, uint64_t seed, int64_t* out_K, double* out_rhat, double* out_swap_rate,
                 double* d_counts, int8_t* d_spins, int64_t ld, cudaStream_t st, const ClusterBonds* bonds) {
    const bool keys_path = N <= 64;
    const int rungs = (int)betas.size();
    const int64_t warps = ceil_div(chains, 32 / rungs), blocks = ceil_div(warps, WARPS);
    const size_t smem = sizeof(uint32_t) * (size_t)N * WARPS;

    DeviceModel model(N, order, term_idx, term_weight, inc, betas, st);
    std::unique_ptr<ClusterRun> cluster(bonds ? new ClusterRun(*bonds, st) : nullptr);
    DevBuf<double> wstats;
    DevBuf<unsigned long long> keys, swaps;
    wstats.alloc(warps * 6);
    if (rungs > 1) swaps.alloc(warps * (rungs - 1));
    if (keys_path) keys.alloc(n_samples);
    auto kernel = keys_path ? ladder_kernel<true>(rungs) : ladder_kernel<false>(rungs);
    GML_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));

    McmcParams& p = model.p;
    p.chains = chains; p.n = n_samples; p.burn_in = burn_in; p.thin = thin;
    p.records = ceil_div(n_samples, chains); p.full_records = n_samples / chains;
    p.seed = seed; p.keys = keys.p; p.warp_stats = wstats.p; p.swap_acc = swaps.p;
    const int64_t h = p.full_records / 2;
    p.inv_h = 1.0 / (double)h;
    p.inv_h1 = 1.0 / (double)(h - 1);
    const int64_t sweeps = burn_in + p.records * thin;
    int64_t rows = 0;
    bool fits = true;
    for (int rep = 0; rep < replicates; ++rep) {
        p.chain0 = (int64_t)rep * chains;
        const bool write = d_counts && !keys_path && rows + n_samples <= ld;
        p.spins = write ? d_spins + rows : nullptr;
        p.counts = write ? d_counts + rows : nullptr;
        p.ld = ld;
        if (!cluster) {
            kernel<<<(unsigned)blocks, WARPS * 32, smem, st>>>(p);
            GML_LAUNCHED();
        } else if (keys_path) {
            cluster->launch<true, false>(p, warps, st);
        } else {
            cluster->launch<false, false>(p, warps, st);
        }
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
        if (out_rhat) rhat_of(wstats.p, warps, chains, h, out_rhat + 2 * rep, st);
        if (out_swap_rate && rungs > 1)
            swap_rates(swaps.p, warps, rungs, chains, burn_in, sweeps, out_swap_rate + (size_t)rep * (rungs - 1), st);
    }
    GML_CUDA(cudaStreamSynchronize(st));
    GML_REQUIRE(!d_counts || fits, "ld = " + std::to_string(ld) + " is smaller than the " + std::to_string(rows) +
                                   " rows of the replicates (out_K holds their sizes)");
}

void moments_mcmc(int N, int order, const std::vector<int32_t>& term_idx, const std::vector<double>& term_weight,
                  const Incidence& inc, const std::vector<double>& betas, int64_t n_samples, int64_t chains, int64_t burn_in,
                  int64_t thin, uint64_t seed, const MomentKeys& keys, double* out_mean, double* out_stderr, double* out_rhat,
                  double* out_swap_rate, cudaStream_t st, const ClusterBonds* bonds) {
    const int rungs = (int)betas.size();
    const int64_t warps = ceil_div(chains, 32 / rungs), blocks = ceil_div(warps, WARPS);
    const size_t smem = sizeof(uint32_t) * (size_t)N * WARPS;

    DeviceModel model(N, order, term_idx, term_weight, inc, betas, st);
    DevBuf<double> wstats;
    DevBuf<unsigned long long> swaps;
    DevBuf<uint32_t> record;
    McmcParams& p = model.p;
    p.chains = chains; p.chain0 = 0; p.n = n_samples; p.burn_in = burn_in; p.thin = thin;
    p.records = ceil_div(n_samples, chains); p.full_records = n_samples / chains;
    const int64_t h = p.full_records / 2;
    p.inv_h = 1.0 / (double)h;
    p.inv_h1 = 1.0 / (double)(h - 1);
    p.rec_warps = warps; p.ld_rec = p.records * warps;
    wstats.alloc(warps * 6);
    if (rungs > 1) swaps.alloc(warps * (rungs - 1));
    record.alloc((size_t)(N + 1) * p.ld_rec);
    p.seed = seed; p.warp_stats = wstats.p; p.swap_acc = swaps.p; p.record = record.p;
    std::unique_ptr<ClusterRun> cluster(bonds ? new ClusterRun(*bonds, st) : nullptr);
    if (cluster) {
        cluster->launch<false, true>(p, warps, st);
    } else {
        auto kernel = record_kernel(rungs);
        GML_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kernel<<<(unsigned)blocks, WARPS * 32, smem, st>>>(p);
        GML_LAUNCHED();
    }
    if (out_rhat) rhat_of(wstats.p, warps, chains, h, out_rhat, st);
    if (out_swap_rate && rungs > 1)
        swap_rates(swaps.p, warps, rungs, chains, burn_in, burn_in + p.records * thin, out_swap_rate, st);
    reduce_records(record.p, N, p.records, warps, keys, out_mean, out_stderr, st);
}

struct PersistentChains::Impl {
    DeviceModel model;
    DevBuf<uint32_t> record;
    Impl(int N, int order, const std::vector<int32_t>& term_idx, const std::vector<double>& term_weight, const Incidence& inc,
         cudaStream_t st)
        : model(N, order, term_idx, term_weight, inc, {1.0}, st) {}
};

PersistentChains::PersistentChains(int N, int order, const std::vector<int32_t>& term_idx,
                                   const std::vector<double>& term_weight, const Incidence& inc, int64_t chains, uint64_t seed,
                                   cudaStream_t st)
    : impl(new Impl(N, order, term_idx, term_weight, inc, st)), warps(ceil_div(chains, 32)) {
    McmcParams& p = impl->model.p;
    p.chains = chains; p.chain0 = 0; p.seed = seed; p.records = 1;
    p.rec_warps = warps; p.ld_rec = warps;
    impl->record.alloc((size_t)(N + 1) * warps);
    p.record = impl->record.p;
    record = impl->record.p; term_w = impl->model.tw.p; weight = impl->model.ww.p;
    const size_t smem = sizeof(uint32_t) * (size_t)N * WARPS;
    GML_CUDA(cudaFuncSetAttribute(mcmc_kernel<false, 1, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
}

PersistentChains::~PersistentChains() = default;

void PersistentChains::run(int64_t sweep0, int64_t sweeps, cudaStream_t st) {
    McmcParams p = impl->model.p;
    p.sweep0 = sweep0; p.thin = sweeps;
    const size_t smem = sizeof(uint32_t) * (size_t)p.N * WARPS;
    mcmc_kernel<false, 1, false, true, true><<<(unsigned)ceil_div(warps, WARPS), WARPS * 32, smem, st>>>(p);
    GML_LAUNCHED();
}

void log_partition_tempering(int N, int order, const std::vector<int32_t>& term_idx, const std::vector<double>& term_weight,
                             const Incidence& inc, const std::vector<double>& betas, int64_t chains, int64_t burn_in,
                             int64_t sweeps, uint64_t seed, double* out_log_z, double* out_stderr, double* out_log_ratio,
                             double* out_swap_rate, cudaStream_t st) {
    const int rungs = (int)betas.size(), pairs = rungs - 1;
    const int64_t warps = ceil_div(chains, 32 / rungs), blocks = ceil_div(warps, WARPS);
    const size_t smem = sizeof(uint32_t) * (size_t)N * WARPS;

    DeviceModel model(N, order, term_idx, term_weight, inc, betas, st);
    DevBuf<double> wstats, bridge;
    DevBuf<unsigned long long> swaps;
    wstats.alloc(warps * 6);
    swaps.alloc(warps * pairs);
    bridge.alloc(chains * pairs * 2);
    auto kernel = bridge_kernel(rungs);
    GML_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));

    McmcParams& p = model.p;                          // no draws: every sweep after burn_in feeds the bridge sums
    p.chains = chains; p.chain0 = 0; p.n = 0; p.burn_in = burn_in; p.thin = 1; p.records = sweeps; p.full_records = 0;
    p.seed = seed; p.warp_stats = wstats.p; p.swap_acc = swaps.p; p.bridge = bridge.p;
    kernel<<<(unsigned)blocks, WARPS * 32, smem, st>>>(p);
    GML_LAUNCHED();
    std::vector<double> ab(chains * pairs * 2);
    GML_CUDA(cudaMemcpyAsync(ab.data(), bridge.p, sizeof(double) * ab.size(), cudaMemcpyDeviceToHost, st));
    GML_CUDA(cudaStreamSynchronize(st));
    if (out_swap_rate) swap_rates(swaps.p, warps, rungs, chains, burn_in, burn_in + sweeps, out_swap_rate, st);

    // Over the L ladders, in ladder order: mean_k = logsumexp_c v_{c,k} - log L for v = a, b; log Z_k - log Z_{k+1} =
    // mean_a - mean_b.  Delta method: u_{c,k} = e^{a_{c,k} - mean_a} - e^{b_{c,k} - mean_b}, stderr = std_c(u) / sqrt(L).
    const double L = (double)chains, log_L = std::log(L);
    std::vector<double> mean(pairs * 2), u_total(chains, 0.0), u(chains);
    auto at = [&](int64_t c, int k, int ab_) { return ab[(c * pairs + k) * 2 + ab_]; };
    auto stderr_of = [&](const std::vector<double>& x) {
        double m = 0, q = 0;
        for (double v : x) m += v;
        m /= L;
        for (double v : x) q += (v - m) * (v - m);
        return std::sqrt(q / (L - 1.0) / L);
    };
    double log_z = N * std::log(2.0);
    for (int k = 0; k < pairs; ++k) {
        for (int h = 0; h < 2; ++h) {
            double mx = -INFINITY, sum = 0;
            for (int64_t c = 0; c < chains; ++c) mx = std::max(mx, at(c, k, h));
            for (int64_t c = 0; c < chains; ++c) sum += std::exp(at(c, k, h) - mx);
            mean[k * 2 + h] = mx + std::log(sum) - log_L;
        }
        for (int64_t c = 0; c < chains; ++c) {
            u[c] = std::exp(at(c, k, 0) - mean[k * 2]) - std::exp(at(c, k, 1) - mean[k * 2 + 1]);
            u_total[c] += u[c];
        }
        const double ratio = mean[k * 2] - mean[k * 2 + 1];
        log_z += ratio;
        if (out_log_ratio) { out_log_ratio[k * 2] = ratio; out_log_ratio[k * 2 + 1] = stderr_of(u); }
    }
    *out_log_z = log_z;
    if (out_stderr) *out_stderr = stderr_of(u_total);
}

}  // namespace gml
