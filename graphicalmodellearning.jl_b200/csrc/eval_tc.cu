// K2/K3, tensor-core backend: the two dense contractions of an objective/gradient pass run on the
// sm_100a 5th-generation tensor cores (tcgen05.mma kind::i8, accumulators in TMEM, operands staged
// by TMA into 128B-swizzled shared memory), in EXACT fixed-point arithmetic:
//
//   * the iterate lives on the lattice 2^-24 (the FISTA driver snaps to it), so x = q * 2^-24 with
//     |q| < 2^27, split into 4 balanced base-256 int8 limbs (digits in [-128, 127]).  The energy contraction
//         E[k,u] = sum_f S[k,f] * x_u[f]            (S = +-1 features, int8)
//     is then four int8 GEMM column groups with int32 accumulation -- no rounding at all.
//   * the epilogue turns E into t = s_u E, psi = exp(-t) (or the RPLE logistic terms) in fp32, and
//     quantises  r = s_u w psi  with a per-node scale derived from the bound |t| <= |x_u|_1 to the integer
//     q + BIAS >= 0, stored as nR UNSIGNED base-256 digits (one byte plane per digit, written straight from
//     the epilogue registers to global memory); the objective terms are summed in fp32 per thread over
//     <= 32 sample blocks and then in fp64.
//   * the gradient contraction  G[u,f] = -sum_k r[u,k] S[k,f]  is again an int8 GEMM (u8 digits x s8 spins),
//     split over sample ranges; the BIAS is removed exactly through the column sums of S (the accumulators
//     start at -BIAS * colsum[f]); partial tiles are combined with int64 atomics, so the result is
//     independent of the reduction order (bitwise reproducible).
//   * precision levels (set_level): the fine level above, and the coarse working level (lattice 2^-22, 3 iterate
//     limbs, |x| < 1.95, 16-bit residuals) on which every node runs and -- at the default tolerance -- retires;
//     an opt-in rough level (2 limbs, one residual plane) is kept as a documented negative result.
//   * active-set compaction (set_active): the passes can be restricted to a list of nodes (slot -> node
//     indirection in the quantiser / finaliser, spins of the listed nodes gathered into P_act).
//
// Warp roles: warp 0 issues TMA, warp 1 issues tcgen05.mma, the remaining warps (16 in the energy
// kernels, 4 in the gradient kernel) run the TMEM epilogues; the energy kernels double-buffer their
// 2 x 256 TMEM columns so the MMA of sample block b+1 overlaps the epilogue of block b.  The energy GEMM
// runs on CTA pairs (tc_energy_pair_kernel: cta_group::2, the limb tile resident in shared memory) whenever
// a half limb tile fits (Fp <= 1024); tc_energy_kernel is the single-CTA form that streams the limb tile.
//
// Replaces the per-node JuMP expression evaluation of src/GraphicalModelLearning.jl:162-172 (and
// :271-281, :309-319, :106-119) for all nodes at once.
#include <cuda.h>

#include <cmath>
#include <cstdlib>

#include "common.cuh"

namespace gml {
namespace {

// ------------------------------------------------------------------------------------------
// PTX wrappers (sm_100a)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}"
        ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- single-issuer roles, warp-converged ---------------------------------------------------------
// The TMA / MMA roles run with all 32 lanes converged and warp-uniform operands; only the elected lane's
// instruction takes effect (predicate inside the asm).  Issuing from `if (lane == 0)` instead makes every
// operand a per-thread value, and ptxas then wraps each UTMALDG / UTCIMMA / UTCBAR in an
// ELECT + R2UR.BROADCAST + BRA.U.ANY waterfall (~20 instructions per MMA): measured, that instruction
// stream -- not the tensor pipe, TMA or the epilogue -- bounded these kernels at 60-78 % tensor activity.
__device__ __forceinline__ uint32_t elect_one_pred() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
    return pred;
}
__device__ __forceinline__ void mbar_expect_tx_if(uint64_t* bar, uint32_t bytes, uint32_t pred) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t"
                 "@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t}" ::"r"(smem_u32(bar)), "r"(bytes), "r"(pred) : "memory");
}
__device__ __forceinline__ void tma_load_2d_if(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, uint32_t pred) {
    asm volatile(
        "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %5, 0;\n\t"
        "@q cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n\t}"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(pred) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], int8 x int8 -> int32, M = 128, K = 32 per instruction
__device__ __forceinline__ void umma_i8_if(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate, uint32_t pred) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\tsetp.ne.b32 p, %4, 0;\n\tsetp.ne.b32 q, %5, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(pred) : "memory");
}
// all previously issued MMAs of the issuing thread arrive on `bar` when complete (implies fence::before_thread_sync)
__device__ __forceinline__ void umma_commit_if(uint64_t* bar, uint32_t pred) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %1, 0;\n\t"
                 "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar)), "r"(pred) : "memory");
}
// ---- CTA pairs (cta_group::2): two CTAs of a cluster on one TPC run ONE M = 256 MMA; each CTA stages its own 128
// rows of A and HALF of B, keeps its own 128 accumulator rows in its own TMEM; the MMA is issued by the leader (rank 0)
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same shared-memory location in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_rank(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    // default .release.cta semantics: a cluster-scope release costs a MEMBAR per arrive (measured: the top stall
    // reason of the epilogue warps); what is ordered here are TMEM reads, by tcgen05.wait::ld + fence::before_thread_sync
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load into this CTA's shared memory whose bytes are accounted on a barrier of the pair's leader CTA
__device__ __forceinline__ void tma_load_2d_pair_if(void* dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1, uint32_t pred) {
    asm volatile(
        "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %5, 0;\n\t"
        "@q cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n\t}"
        ::"r"(smem_u32(dst)), "l"(map), "r"(leader_bar), "r"(c0), "r"(c1), "r"(pred) : "memory");
}
// D[tmem, both CTAs] (+)= A * B, M = 256 (128 rows per CTA), K = 32 per instruction
__device__ __forceinline__ void umma_i8_pair_if(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate, uint32_t pred) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\tsetp.ne.b32 p, %4, 0;\n\tsetp.ne.b32 q, %5, 0;\n\t"
        "@q tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(pred) : "memory");
}
// all previously issued pair MMAs arrive on the barrier at this shared-memory offset in BOTH CTAs when complete
__device__ __forceinline__ void umma_commit_pair_if(uint64_t* bar, uint32_t pred) {
    asm volatile("{\n\t.reg .pred q;\n\t.reg .b16 m;\n\tsetp.ne.b32 q, %1, 0;\n\tmov.b16 m, 3;\n\t"
                 "@q tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], m;\n\t}"
                 ::"r"(smem_u32(bar)), "r"(pred) : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* slot, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t addr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, int32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, int32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr) : "memory");
}
// Wait for the outstanding TMEM loads; the registers pass through the statement so that no use of them can be
// scheduled above the wait (the loads are asynchronous: software-pipelined epilogues keep one chunk in flight).
__device__ __forceinline__ void tmem_ld_wait_on(int32_t (&v)[8]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]) :: "memory");
}
__device__ __forceinline__ void reg_fence(int32_t (&v)[8]) {
    asm volatile("" : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]) :: "memory");
}
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {     // non-blocking
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// K-major operand tile, rows of 128 bytes, 128B swizzle (what TMA SWIZZLE_128B writes):
// start address >> 4, LBO = 1 (ignored for swizzled K-major), SBO = 1024 B (8 rows), version 1, layout 2
__device__ __forceinline__ uint64_t make_kmajor_desc(uint32_t smem_addr) {
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) |
           ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// instruction descriptor, kind::i8: D = s32, A = s8 (or u8), B = s8, both K-major
__host__ __device__ constexpr uint32_t make_idesc_i8(int M, int N, bool a_unsigned = false) {
    return (2u << 4) | ((a_unsigned ? 0u : 1u) << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ------------------------------------------------------------------------------------------
// fixed-point helpers
// ------------------------------------------------------------------------------------------
// Two precision levels of the iterate:
//   fine   : lattice 2^-24, |x| < 7.9, 4 limbs                  -- tolerances below what the coarse lattice resolves, |x| >= 1.95
//   coarse : lattice 2^-22, |x| < 1.95, 3 limbs (24 bits)       -- the working level: the snapped iteration stops within half a
//            lattice unit of its fixed point, i.e. at a prox-gradient mapping of <= L * 2^-23 ~ 3e-7
//   rough  : lattice 2^-14, |x| < 1.95, 2 limbs (16 bits), ONE residual digit plane (8 bits) -- opt-in experiment (fista.cu)
// Digits are balanced base 256 ([-128, 127], the full int8 range; round 1 used base 128 and gave away one bit per limb:
// its 3-limb level had lattice 2^-20 over |x| < 1, too coarse for any node to meet tol = 1e-6 on it).
constexpr double X_LATTICE_FINE = 1.0 / 16777216.0, X_LATTICE_COARSE = 1.0 / 4194304.0, X_LATTICE_ROUGH = 1.0 / 16384.0;
constexpr int X_LIMBS_MAX = 4;
// representable range of the balanced base-256 limbs: 2 limbs hold |q| <= 32000 (x 2^-14), 3 limbs |q| <= 8300000 (x 2^-22);
// the 4-limb level keeps |q| <= 134000000 (x 2^-24: |x| < 7.99), far inside its 32 bits
constexpr double X_RANGE_COARSE = 1.95, X_RANGE_FINE = 7.9;
constexpr int NODE_TILE1 = 64;                   // nodes per energy tile (4 limbs -> N = 256)
constexpr int NODE_TILE2 = 128;                  // nodes per gradient tile (M = 128)

// residual grid: |q| <= r_qmax(nR), stored as q + r_bias(nR) in nR unsigned bytes (nR <= 3 round with the
// magic-number trick, which needs |q| < 2^22)
__host__ __device__ constexpr int r_qmax(int nR) { return nR == 1 ? 120 : (nR == 2 ? 32000 : (nR == 3 ? 4000000 : 1000000000)); }
// The biases of nR <= 3 are the ones the rounding constant provides for free: float_as_int(q + 1.5 * 2^23 [+ 2^15])
// holds q + 2^22 [+ 2^15] in its mantissa bits, so the stored bytes are plain byte extracts of that word.
__host__ __device__ constexpr unsigned r_bias(int nR) { return nR == 1 ? 0x80u : (nR == 2 ? 0x8000u : (nR == 3 ? 0x400000u : 0x80000000u)); }
__host__ __device__ constexpr float r_magic(int nR) { return nR == 1 ? 12582912.f + 128.f : (nR == 2 ? 12582912.f + 32768.f : 12582912.f); }

__device__ __forceinline__ int balanced_digit(int& q) {   // returns q mod 256 in [-128, 127], q <- (q - d) / 256
    const int d = ((q + 128) & 255) - 128;
    q = (q - d) >> 8;
    return d;
}
// Limb sums -> the integer energy, in wrap-around (unsigned) arithmetic: partial products may leave the int32 range, the
// energy itself (|E| <= |x_u|_1 / lattice) does not.
__device__ __forceinline__ int join2(int hi, int lo) { return (int)((unsigned)hi * 256u + (unsigned)lo); }


// x [Nn x Fp] (double, on the lattice) -> limb tiles X [(tile*xl + limb)*node_tile + i][Fp] and per-node residual scales
__global__ void __launch_bounds__(128) tc_quantize_x_kernel(const double* __restrict__ x, int Nn, int Fp, int form, double wmax,
                                                           int nR, int xl, int node_tile, double inv_lattice, int8_t* __restrict__ X,
                                                           float* __restrict__ inv_dr, double* __restrict__ delta /* [Nn_pad]: deltaR */,
                                                           int* __restrict__ flags, const int* __restrict__ act_idx /* slot -> node, or null */) {
    const int slot = blockIdx.x;
    const int tile = slot / node_tile, i = slot % node_tile;
    const int u = (slot < Nn) ? (act_idx ? act_idx[slot] : slot) : Nn;          // Nn here = number of slots in use; padding slots hold x = 0
    const bool live = slot < Nn && u >= 0;
    __shared__ double red[4];
    // largest |q| that xl balanced base-256 digits can hold (4 limbs: the |x| < 7.99 range of the fine level)
    const long long qcap = xl == 2 ? 32000LL : (xl == 3 ? 8300000LL : 134000000LL);
    double l1 = 0.0;
    for (int f = threadIdx.x; f < Fp; f += blockDim.x) {
        const double v = live ? x[(int64_t)u * Fp + f] : 0.0;
        l1 += fabs(v);
        long long ql = llrint(v * inv_lattice);
        if (ql > qcap || ql < -qcap) { atomicOr(flags, xl <= 3 ? 2 : 1); ql = ql > 0 ? qcap : -qcap; }
        int q = (int)ql;
        int d[X_LIMBS_MAX];
        for (int j = xl - 1; j > 0; --j) d[j] = balanced_digit(q);
        d[0] = q;
        const int64_t row = ((int64_t)tile * xl) * node_tile + i;
        for (int j = 0; j < xl; ++j) X[(row + (int64_t)j * node_tile) * Fp + f] = (int8_t)d[j];
    }
    for (int o = 16; o; o >>= 1) l1 += __shfl_xor_sync(0xffffffffu, l1, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = l1;
    __syncthreads();
    if (threadIdx.x == 0) {
        const double B = red[0] + red[1] + red[2] + red[3];   // |t| <= B for every sample
        // the 3-limb epilogue joins the limb sums in 32-bit arithmetic: |E| / lattice <= B * 2^22 must stay below 2^31
        if (xl == 3 && B >= 500.0) atomicOr(flags, 2);
        // residual bound: RISE/logRISE  w e^{-t} <= wmax e^B;  RPLE  2 w sigma(-2t) <= 2 wmax
        const double top = (form == GML_B200_RPLE) ? 2.0 * wmax : wmax * exp(fmin(B, 80.0));
        const float inv = (float)(r_qmax(nR) / (top * 1.000001));
        inv_dr[slot] = inv;
        delta[slot] = 1.0 / (double)inv;   // exact reciprocal of what the epilogue multiplies with
    }
}

// ------------------------------------------------------------------------------------------
// GEMM-1: energies + fused epilogue
// ------------------------------------------------------------------------------------------
struct EnergyParams {
    int Fp, Fspin, n_tiles, node_begin_row;        // node tile t covers spin rows node_begin_row + 64 t ... of each [Fspin x 128] block
    int spin_vec;                          // 1: the spin tile comes from P, sample-major [128 samples][64 nodes] (16 B per thread)
    int n_groups;                          // sample ranges; work item = (group, node tile)
    int n_waves, g_main;                   // CTA-pair kernel: wave-aligned item schedule (pair_schedule)
    int64_t sample_blocks;                 // sample blocks of this pass (Kp / 128 / block_stride)
    int64_t block_stride;                  // pass b uses histogram block b * block_stride (strided subsample)
    int64_t r_rows_per_limb;               // Nn_pad2
    float lattice;                         // value of one unit of the combined integer energy
    const float* w32;
    uint8_t* R;                            // residual digit planes [SB][nR][Nn_pad2][128]
    uint8_t* r_scratch;                    // [4][64][128] sink for the stores of a duplicated tail block
    const float* inv_dr;                   // [Nn_pad1] 1/deltaR
    double* fsum;                          // [Nn_pad1] objective sums
    int dbg;                               // ablation switches (only in -DGML_TC_ABLATE builds; see GML_DBG)
};

// Ablation switches for profiling (variant builds with -DGML_TC_ABLATE, env GML_B200_DBG): results are
// garbage, timings tell which stage of the pipeline bounds a kernel.  1: skip the epilogue math and the
// R store, 2: do not load the limb tile, 4: no operand loads at all (MMA on stale shared memory), 8: do not
// load the histogram tile (energy kernel), 16: issue no MMA (pair energy kernel: epilogue-only time), 32: epilogue
// stops after its TMEM reads, 64: no residual stores.
#ifdef GML_TC_ABLATE
#define GML_DBG(p, bit) (((p).dbg & (bit)) != 0)
#else
#define GML_DBG(p, bit) false
#endif

constexpr int E_STAGES = 4;
constexpr int E_EPI_WARPS = 16;     // 4 per TMEM lane quarter; measured: full pass 4.17 ms (8 warps) -> 3.50 ms (16 warps) at N=1000, K=1e6
constexpr int E_NPT = NODE_TILE1 / (E_EPI_WARPS / 4);   // nodes per epilogue thread: 16, i.e. four words of spin bytes
constexpr int E_THREADS = 64 + 32 * E_EPI_WARPS;
constexpr int E_A_BYTES = 128 * 128, E_B_BYTES = 256 * 128, E_STAGE_BYTES = E_A_BYTES + E_B_BYTES;
constexpr int E_S_BYTES = NODE_TILE1 * 128;          // spins tile of the node block
constexpr int E_SMEM = E_STAGES * E_STAGE_BYTES + 2 * E_S_BYTES + 1024 /*align*/ + 512 /*barriers, scales*/;
static_assert(E_SMEM <= 227 * 1024, "energy kernel exceeds the shared memory of an SM");

// explicit shared-space accesses (the carved-up dynamic smem pointer is generic to the compiler, which would
// otherwise emit generic LD/ST for every epilogue access)
__device__ __forceinline__ uint4 lds128(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds_u8(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ float lds_f32(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
    return v;
}

// a ^ (b & c) in one LOP3: flips the sign of float a when the spin byte shifted to the top of b is negative
__device__ __forceinline__ float flip_sign(float a, uint32_t b) {
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, 0x80000000, 0x78;" : "=r"(d) : "r"(__float_as_uint(a)), "r"(b));
    return __uint_as_float(d);
}
__device__ __forceinline__ float fast_ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float fast_lg2(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// Per-block epilogue math of one thread: NODES nodes of one sample (TMEM lane) whose XL limb sums are already in
// registers (a[limb][node]), sw = their spin bytes (0x01 / 0xFF; 0x00 for padding nodes), four to a word.  Recombines
// the limb sums exactly, applies the node sign, evaluates the objective / residual terms, accumulates the objective
// into facc and (GRAD) writes the NR residual digits (bytes of q + BIAS, most significant first) of every node straight
// to global memory at rgp[digit] + (node0 + node) * 128: a warp covers one full 32-byte sector per store, and no staging
// tile, proxy fence, block barrier or TMA store sits between the epilogue warps and the next block.
template <int FORM, bool GRAD, int XL, int NR, int NODES>
__device__ __forceinline__ void energy_epilogue(const EnergyParams& p, const int32_t (&a)[4][NODES], const uint32_t* sw, uint32_t scale_addr,
                                                uint8_t* const (&rgp)[4] /* per digit plane: address of this thread's byte of node 0 */,
                                                int node0, float wk, float* __restrict__ facc) {
    const float c_arg = -p.lattice * 1.4426950408889634f;      // exp(-t) = ex2(c_arg * s_u * E_int)
    constexpr unsigned R_BIAS = r_bias(NR);
    if (GML_DBG(p, 32)) { facc[0] += __int_as_float(a[0][0] ^ a[1][3] ^ (XL >= 3 ? a[2][7] : 0) ^ (XL == 4 ? a[3][5] : 0)); return; }   // ablation: TMEM reads only
#pragma unroll
    for (int i = 0; i < NODES; ++i) {
        const uint32_t w = sw[i >> 2];
        const uint32_t sb_top = (i & 3) == 3 ? w : (w << (24 - 8 * (i & 3)));      // spin byte in the top byte: its sign bit is that of s_u
        // recombine the limb sums: exact integers, at most one rounding
        float e;
        if (XL == 2) e = __int2float_rn(join2(a[0][i], a[1][i]));
        else if (XL == 3) e = __int2float_rn(join2(join2(a[0][i], a[1][i]), a[2][i]));       // exact in fp32 while |E| < 4
        else e = fmaf(__int2float_rn(join2(a[0][i], a[1][i])), 65536.f, __int2float_rn(join2(a[2][i], a[3][i])));
        const float es = flip_sign(e, sb_top);                  // s_u * E / lattice
        float gterm;
        if (FORM == GML_B200_RPLE) {
            const float t2 = -2.f * p.lattice * es;
            const float ex = fast_ex2(-fabsf(t2) * 1.4426950408889634f);
            facc[i] += wk * fmaf(fast_lg2(1.f + ex), 0.6931471805599453f, fmaxf(t2, 0.f));
            gterm = __fdividef(2.f * wk * (t2 > 0.f ? 1.f : ex), 1.f + ex);   // 2 w sigma(-2t)
        } else {
            // no clamp: |t| <= |x_u|_1 keeps the argument in range; an overflow for a wild trial point (|x_u|_1 > 80) gives
            // f = inf, which the driver's descent test rejects.  The objective term is one fma in every instantiation: with
            // a separately rounded product (the residual) the full passes and the objective-only passes of the line
            // search would differ by ~3e-9 relative
            const float ex = fast_ex2(es * c_arg);
            facc[i] = fmaf(wk, ex, facc[i]);
            gterm = wk * ex;
        }
        if (GRAD) {
            // r = s_u * gterm in units of the node's residual grid, rounded to nearest, plus the
            // bias that makes all balanced digits non-negative
            const float sscale = flip_sign(lds_f32(scale_addr + 4 * i), sb_top);      // s_u / deltaR
            unsigned qb;      // low NR bytes = q + BIAS
            if (NR == 4) qb = (unsigned)__float2int_rn(gterm * sscale) + R_BIAS;
            else qb = (unsigned)__float_as_int(fmaf(gterm, sscale, r_magic(NR)));   // round to nearest, |q| < 2^22; bias from the constant
            if (!GML_DBG(p, 64)) {
#pragma unroll
                for (int j = 0; j < NR; ++j) rgp[j][(node0 + i) * 128] = (uint8_t)(qb >> (8 * (NR - 1 - j)));      // plane 0 = most significant byte
            }
        }
    }
}
// TMEM loads of the XL limb sums of NODES (8 or 16) consecutive accumulator columns from tchunk on
template <int XL, int NODES>
__device__ __forceinline__ void epi_issue(uint32_t tchunk, int32_t (&a)[4][NODES]) {
    static_assert(NODES == 8 || NODES == 16, "TMEM loads come in x8 and x16 groups");
#pragma unroll
    for (int j = 0; j < XL; ++j) {
        if constexpr (NODES == 16) tmem_ld16(tchunk + j * NODE_TILE1, a[j]);
        else tmem_ld8(tchunk + j * NODE_TILE1, a[j]);
    }
}
template <int XL>
__device__ __forceinline__ void epi_wait(int32_t (&a)[4][8]) {
    tmem_ld_wait_on(a[0]);
#pragma unroll
    for (int j = 1; j < XL; ++j) reg_fence(a[j]);
}

// Producer side: the spin tile of node tile nt for histogram block sb, landing on `bar`.  From P itself (sample-major,
// box {64 nodes, 128 samples}) when the shard's first spin column is 16-byte aligned, else from the sample-blocked
// spin rows (node-major, box 64 rows).
__device__ __forceinline__ void load_spin_tile(const EnergyParams& p, void* dst, const CUtensorMap* tmS, const CUtensorMap* tmSv,
                                               uint64_t* bar, int nt, int64_t sb, uint32_t pred) {
    mbar_expect_tx_if(bar, E_S_BYTES, pred);
    if (p.spin_vec) tma_load_2d_if(dst, tmSv, bar, p.node_begin_row + nt * NODE_TILE1, (int)(sb * 128), pred);
    else tma_load_2d_if(dst, tmS, bar, 0, (int)(sb * p.Fspin) + p.node_begin_row + nt * NODE_TILE1, pred);
}
// Epilogue side: the spin bytes of the thread's E_NPT nodes from node0 on at sample `row` of the spin tile at `tile`, four
// to a word: 16 contiguous bytes of the sample-major tile [128 samples][64 nodes] (64B swizzle: 16-byte chunk index
// ^= (row >> 1) & 3), or one byte per node at column `row` of the node-major tile [64 nodes][128 samples].
__device__ __forceinline__ void spin_words(const EnergyParams& p, uint32_t tile, int row, int node0, uint32_t (&sw)[4]) {
    if (p.spin_vec) {
        const uint4 v = lds128(tile + row * NODE_TILE1 + (node0 ^ (((row >> 1) & 3) << 4)));
        sw[0] = v.x; sw[1] = v.y; sw[2] = v.z; sw[3] = v.w;
    } else {
        const uint32_t sa = tile + node0 * 128 + row;
#pragma unroll
        for (int w = 0; w < 4; ++w)
            sw[w] = lds_u8(sa + 4 * w * 128) | (lds_u8(sa + (4 * w + 1) * 128) << 8) | (lds_u8(sa + (4 * w + 2) * 128) << 16) | (lds_u8(sa + (4 * w + 3) * 128) << 24);
    }
}
// Per digit plane, the address of the thread's byte of node node0 of node tile nt in sample block sb:
// R[((sb * NR + digit) * rows + node) * 128 + sample].  A block that must not be stored (!valid) goes to a scratch tile.
template <int NR>
__device__ __forceinline__ void digit_planes(const EnergyParams& p, bool valid, int64_t sb, int nt, int node0, int row, uint8_t* (&rgp)[4]) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
        rgp[j] = valid ? p.R + (((sb * NR + j) * p.r_rows_per_limb + nt * NODE_TILE1 + node0) * 128 + row)
                       : p.r_scratch + ((j * NODE_TILE1 + node0) * 128 + row);
}

// Objective sums of one epilogue thread over one work item (its E_NPT nodes of node tile nt): fp32 per-thread partial
// sums over at most 32 sample blocks, then fp64 warp sums added to fsum.
struct ItemObjective {
    float facc[E_NPT];
    int since_flush;
    double* fsum;                             // objective sum of the thread's first node
    // start of an item; GRAD: also refill the node tile's residual scales
    template <bool GRAD>
    __device__ __forceinline__ void begin(const EnergyParams& p, int nt, int node0, float* s_scale) {
#pragma unroll
        for (int i = 0; i < E_NPT; ++i) facc[i] = 0.f;
        if (GRAD) {
            const int et = threadIdx.x - 64;
            named_bar_sync(1, 32 * E_EPI_WARPS);          // previous item's readers are done with s_scale
            if (et < NODE_TILE1) s_scale[et] = p.inv_dr[nt * NODE_TILE1 + et];
            named_bar_sync(1, 32 * E_EPI_WARPS);
        }
        since_flush = 0;
        fsum = p.fsum + (int64_t)nt * NODE_TILE1 + node0;
    }
    // before each sample block
    __device__ __forceinline__ void next_block() {
        if (since_flush >= 32) { flush(); since_flush = 0; }
        ++since_flush;
    }
    // after the item's last block
    __device__ __forceinline__ void flush() {
#pragma unroll
        for (int i = 0; i < E_NPT; ++i) {
            double v = (double)facc[i];
            for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if ((threadIdx.x & 31) == 0) atomicAdd(fsum + i, v);
            facc[i] = 0.f;
        }
    }
};

// Work decomposition: item = (sample range g, node tile nt), ordered group-major and dealt round-robin,
// so CTAs that run concurrently stream the SAME sample blocks for different node tiles (the P tiles are
// shared through L2 instead of being re-read from HBM once per node tile), while each CTA keeps one node
// tile for a whole sample range (objective partial sums stay in registers).
template <int FORM, bool GRAD, int XL, int NR>
__global__ void __launch_bounds__(E_THREADS, 1) tc_energy_kernel(const __grid_constant__ CUtensorMap tmA,   // P  [Kp x Fp]
                                                                const __grid_constant__ CUtensorMap tmB,   // X  [tiles*XL*64 x Fp], box XL*64 rows
                                                                const __grid_constant__ CUtensorMap tmS,   // spins, sample-blocked [SB*Fspin x 128], box 64 rows (row coordinates need no alignment)
                                                                const __grid_constant__ CUtensorMap tmSv,  // P, box {64 nodes, 128 samples}: used when the shard's first spin column is 16-byte aligned
                                                                EnergyParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* s_stage = smem;
    uint8_t* s_spin = smem + E_STAGES * E_STAGE_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_spin + 2 * E_S_BYTES);
    uint64_t* full = bars;                    // [E_STAGES]
    uint64_t* empty = bars + E_STAGES;        // [E_STAGES]
    uint64_t* tfull = bars + 2 * E_STAGES;    // [2]
    uint64_t* tempty = tfull + 2;             // [2]
    uint64_t* sfull = tempty + 2;             // [2]
    uint64_t* sempty = sfull + 2;             // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sempty + 2);
    float* s_scale = reinterpret_cast<float*>(tmem_slot + 2);   // [64] 1/deltaR of the node tile

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // warp index, uniform for the compiler
    const int kblocks = p.Fp / 128;
    const int n_items = p.n_tiles * p.n_groups;

    if (threadIdx.x == 0) {
        for (int i = 0; i < E_STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&tfull[i], 1); mbar_init(&tempty[i], E_EPI_WARPS);
            mbar_init(&sfull[i], 1); mbar_init(&sempty[i], E_EPI_WARPS);
        }
        fence_barrier_init();
        prefetch_tmap(&tmA); prefetch_tmap(&tmB); prefetch_tmap(&tmS); prefetch_tmap(&tmSv);
    }
    if (warp == 1) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

    auto item_range = [&](int item, int& nt, int64_t& b0, int64_t& b1) {
        const int g = item / p.n_tiles;
        nt = item % p.n_tiles;
        b0 = p.sample_blocks * g / p.n_groups;
        b1 = p.sample_blocks * (g + 1) / p.n_groups;
    };

    if (warp == 0) {
        // ================= TMA producer (whole warp converged, elected lane issues) =================
        const uint32_t leader = elect_one_pred();
        int stage = 0; uint32_t phase = 0;
        int slot = 0; uint32_t sphase = 0;
        for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
            int nt; int64_t b0, b1;
            item_range(item, nt, b0, b1);
            for (int64_t eb = b0; eb < b1; ++eb) {
                const int64_t sb = eb * p.block_stride;
                mbar_wait(&sempty[slot], sphase ^ 1);
                load_spin_tile(p, s_spin + slot * E_S_BYTES, &tmS, &tmSv, &sfull[slot], nt, sb, leader);
                if (++slot == 2) { slot = 0; sphase ^= 1; }
                for (int kb = 0; kb < kblocks; ++kb) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    const uint32_t ld_a = GML_DBG(p, 12) ? 0u : leader, ld_b = GML_DBG(p, 6) ? 0u : leader;
                    mbar_expect_tx_if(&full[stage], (ld_a ? E_A_BYTES : 0) + (ld_b ? XL * NODE_TILE1 * 128 : 0), leader);
                    uint8_t* a = s_stage + stage * E_STAGE_BYTES;
                    tma_load_2d_if(a, &tmA, &full[stage], kb * 128, (int)(sb * 128), ld_a);
                    tma_load_2d_if(a + E_A_BYTES, &tmB, &full[stage], kb * 128, nt * XL * NODE_TILE1, ld_b);
                    if (++stage == E_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer (whole warp converged, elected lane issues) =================
        const uint32_t leader = elect_one_pred();
        constexpr uint32_t idesc = make_idesc_i8(128, XL * NODE_TILE1);
        const uint32_t stage_base = smem_u32(s_stage);
        int stage = 0; uint32_t phase = 0;
        int as = 0; uint32_t aphase = 0;
        for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
            int nt; int64_t b0, b1;
            item_range(item, nt, b0, b1);
            for (int64_t sb = b0; sb < b1; ++sb) {
                mbar_wait(&tempty[as], aphase ^ 1);
                tc_fence_after();
                const uint32_t d = tmem_base + as * 256;
                for (int kb = 0; kb < kblocks; ++kb) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t a_addr = stage_base + stage * E_STAGE_BYTES;
                    const uint64_t da = make_kmajor_desc(a_addr), db = make_kmajor_desc(a_addr + E_A_BYTES);
#pragma unroll
                    for (int k = 0; k < 4; ++k) umma_i8_if(d, da + 2 * k, db + 2 * k, idesc, (kb | k) ? 1u : 0u, leader);
                    umma_commit_if(&empty[stage], leader);
                    if (++stage == E_STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit_if(&tfull[as], leader);
                if (++as == 2) { as = 0; aphase ^= 1; }
            }
        }
    } else {
        // ================= epilogue warps 2..17: TMEM lane quarter = warp % 4, node slice = (warp-2)/4 =========
        const int quarter = warp & 3;
        const int node0 = ((warp - 2) >> 2) * E_NPT;     // first node of the slice of the node tile this warp owns
        const int row = quarter * 32 + lane;            // sample within the block == TMEM lane
        ItemObjective obj;
        int as = 0; uint32_t aphase = 0;
        int slot = 0; uint32_t sphase = 0;
        for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
            int nt; int64_t b0, b1;
            item_range(item, nt, b0, b1);
            obj.begin<GRAD>(p, nt, node0, s_scale);
            for (int64_t eb = b0; eb < b1; ++eb) {
                const int64_t sb = eb * p.block_stride;
                obj.next_block();
                const float wk = p.w32[sb * 128 + row];
                mbar_wait(&sfull[slot], sphase);
                mbar_wait(&tfull[as], aphase);
                tc_fence_after();
                if (GML_DBG(p, 1)) {
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) { mbar_arrive(&tempty[as]); mbar_arrive(&sempty[slot]); }
                    if (++as == 2) { as = 0; aphase ^= 1; }
                    if (++slot == 2) { slot = 0; sphase ^= 1; }
                    continue;
                }
                uint8_t* rgp[4];
                digit_planes<NR>(p, true, sb, nt, node0, row, rgp);
                uint32_t sw[4];
                spin_words(p, smem_u32(s_spin) + slot * E_S_BYTES, row, node0, sw);
                int32_t a[4][E_NPT];
                epi_issue<XL>(tmem_base + ((uint32_t)(quarter * 32) << 16) + as * 256 + node0, a);
                tmem_ld_wait();
                tc_fence_before();                       // accumulator fully read: hand it back to the MMA warp
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty[as]);
                energy_epilogue<FORM, GRAD, XL, NR>(p, a, sw, smem_u32(s_scale) + 4 * node0, rgp, 0, wk, obj.facc);
                __syncwarp();
                if (lane == 0) mbar_arrive(&sempty[slot]);
                if (++as == 2) { as = 0; aphase ^= 1; }
                if (++slot == 2) { slot = 0; sphase ^= 1; }
            }
            obj.flush();
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------
// GEMM-1, CTA-pair form: the limb tile stays RESIDENT in shared memory
// ------------------------------------------------------------------------------------------
// The streaming kernel above re-loads the XL*64 x Fp limb tile (B operand) for every 128-sample block and
// therefore moves 96-107 bytes of L2 -> shared-memory traffic per SM clock at full tensor rate -- measured, that
// (not the tensor pipe, not the epilogue) bounds it (profiles/r1_ablation.txt).  Here two CTAs of a cluster pair
// up (tcgen05 cta_group::2, M = 256 = two 128-sample blocks): each CTA keeps HALF of the limb tile (XL*32 rows x
// Fp <= 128 KB) resident for a whole work item and streams only its own histogram tiles (16 KB per 128 features),
// 32-42 bytes per SM clock.  Same epilogue, same results (exact integer energies).
// Work item = (range of sample-block pairs, node tile); pair-step pb covers blocks 2 pb (rank 0) and 2 pb + 1 (rank 1).
constexpr int E2_MAX_FP = 1024;                          // resident limb half: XL*32 rows x Fp bytes
__host__ __device__ constexpr int e2_b_bytes(int xl) { return xl * 32 * E2_MAX_FP; }
__host__ __device__ constexpr int e2_fixed(int xl) { return e2_b_bytes(xl) + 2 * E_S_BYTES + 1024 + 512; }
__host__ __device__ constexpr int e2_stages(int xl) {
    const int room = 227 * 1024 - e2_fixed(xl);
    return room / E_A_BYTES > 6 ? 6 : room / E_A_BYTES;
}
__host__ __device__ constexpr int e2_smem(int xl) { return e2_fixed(xl) + e2_stages(xl) * E_A_BYTES; }

template <int FORM, bool GRAD, int XL, int NR>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(E_THREADS, 1)
tc_energy_pair_kernel(const __grid_constant__ CUtensorMap tmA,    // P  [Kp x Fp], box {128 features, 128 samples}
                      const __grid_constant__ CUtensorMap tmBh,   // X  [tiles*XL*64 x Fp], box {128 features, XL*32 rows}
                      const __grid_constant__ CUtensorMap tmS,    // spins, sample-blocked (see tc_energy_kernel)
                      const __grid_constant__ CUtensorMap tmSv,   // P, box {64 nodes, 128 samples}
                      EnergyParams p) {
    constexpr int STAGES = e2_stages(XL);
    constexpr int B_BYTES = e2_b_bytes(XL);
    constexpr int B_KB_BYTES = XL * 32 * 128;            // one 128-feature slab of the resident half
    static_assert(STAGES >= 3, "pair energy kernel: not enough shared memory for the histogram ring");
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* s_b = smem;
    uint8_t* s_a = s_b + B_BYTES;
    uint8_t* s_spin = s_a + STAGES * E_A_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_spin + 2 * E_S_BYTES);
    uint64_t* full = bars;                    // [STAGES]  leader: both CTAs' histogram tiles of the stage have landed
    uint64_t* empty = bars + STAGES;          // [STAGES]  per CTA: the pair MMAs that read the stage are complete
    uint64_t* tfull = bars + 2 * STAGES;      // [2]       per CTA: accumulator published
    uint64_t* tempty = tfull + 2;             // [2]       leader: both CTAs' epilogues have drained the accumulator
    uint64_t* sfull = tempty + 2;             // [2]       per CTA: spin tile landed
    uint64_t* sempty = sfull + 2;             // [2]
    uint64_t* bfull = sempty + 2;             // leader: both halves of the limb tile have landed
    uint64_t* bempty = bfull + 1;             // per CTA: all MMAs of the item are complete, the limb tile may be replaced
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bempty + 1);
    float* s_scale = reinterpret_cast<float*>(tmem_slot + 2);   // [64] 1/deltaR of the node tile

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
    const int kblocks = p.Fp / 128;
    const int n_items = p.n_tiles * p.n_groups;
    const int64_t pair_blocks = (p.sample_blocks + 1) / 2;

    if (threadIdx.x == 0) {
        for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 2 * E_EPI_WARPS);
            mbar_init(&sfull[i], 1); mbar_init(&sempty[i], E_EPI_WARPS);
        }
        mbar_init(bfull, 1); mbar_init(bempty, 1);
        fence_barrier_init();
        prefetch_tmap(&tmA); prefetch_tmap(&tmBh); prefetch_tmap(&tmS); prefetch_tmap(&tmSv);
    }
    if (warp == 1) tmem_alloc_pair(tmem_slot, 512);
    tc_fence_before();
    cluster_sync_all();                       // barriers of both CTAs initialised, TMEM allocated in both
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

    // Wave-aligned schedule: in every wave the first floor(n_pairs / n_tiles) * n_tiles pairs work on WHOLE sample ranges (one
    // pair per node tile of the range, started together, so the range's histogram tiles are fetched from HBM once and shared
    // through L2), the remaining pairs work through the leftover ranges tile by tile.  Plain round-robin over (range, tile)
    // items splits a range over two waves whenever n_pairs is not a multiple of n_tiles (74 pairs, 16 tiles: every wave),
    // and the split ranges were read twice (ncu: 21 GB for the 10 GB histogram).
    auto wave_item = [&](int w, int& nt, int64_t& b0, int64_t& b1) -> bool {
        const int T = p.n_tiles;
        const int main_pairs = (n_pairs / T) * T;
        int g;
        if (main_pairs == 0) {                       // more node tiles than pairs: round robin
            const int item = w * n_pairs + pair;
            if (item >= n_items) return false;
            g = item / T; nt = item % T;
        } else if (pair < main_pairs) {
            g = w * (main_pairs / T) + pair / T; nt = pair % T;
            if (g >= p.g_main) return false;
        } else {
            const int s = w * (n_pairs - main_pairs) + (pair - main_pairs);
            g = p.g_main + s / T; nt = s % T;
            if (g >= p.n_groups) return false;
        }
        b0 = pair_blocks * g / p.n_groups;
        b1 = pair_blocks * (g + 1) / p.n_groups;
        return true;
    };

    if (warp == 0) {
        // ================= TMA producer of this CTA (whole warp converged, elected lane issues) =================
        const uint32_t lane_leader = elect_one_pred();
        const uint32_t cta_leader = rank == 0 ? lane_leader : 0u;       // expect_tx is posted once, by the leader CTA
        const uint32_t bfull_leader = mapa_rank(smem_u32(bfull), 0);
        int stage = 0; uint32_t phase = 0;
        int slot = 0; uint32_t sphase = 0;
        uint32_t bphase = 0;
        for (int w = 0; w < p.n_waves; ++w) {
            int nt; int64_t b0, b1;
            if (!wave_item(w, nt, b0, b1)) continue;
            // ---- this CTA's half of the limb tile, resident for the whole item
            mbar_wait(bempty, bphase ^ 1);
            mbar_expect_tx_if(bfull, 2u * (uint32_t)(XL * 32) * (uint32_t)p.Fp, cta_leader);
            for (int kb = 0; kb < kblocks; ++kb)
                tma_load_2d_pair_if(s_b + kb * B_KB_BYTES, &tmBh, bfull_leader, kb * 128, nt * XL * NODE_TILE1 + (int)rank * XL * 32, lane_leader);
            bphase ^= 1;
            for (int64_t pb = b0; pb < b1; ++pb) {
                const int64_t eb = min(2 * pb + (int64_t)rank, p.sample_blocks - 1);    // an odd tail re-reads the last block (its epilogue is skipped)
                const int64_t sb = eb * p.block_stride;
                mbar_wait(&sempty[slot], sphase ^ 1);
                load_spin_tile(p, s_spin + slot * E_S_BYTES, &tmS, &tmSv, &sfull[slot], nt, sb, lane_leader);
                if (++slot == 2) { slot = 0; sphase ^= 1; }
                for (int kb = 0; kb < kblocks; ++kb) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    const bool no_a = GML_DBG(p, 4);
                    mbar_expect_tx_if(&full[stage], no_a ? 0 : 2 * E_A_BYTES, cta_leader);
                    tma_load_2d_pair_if(s_a + stage * E_A_BYTES, &tmA, mapa_rank(smem_u32(&full[stage]), 0), kb * 128, (int)(sb * 128), no_a ? 0u : lane_leader);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer: leader CTA only =================
        if (rank == 0) {
            const uint32_t lane_leader = elect_one_pred();
            constexpr uint32_t idesc = make_idesc_i8(256, XL * NODE_TILE1);
            const uint32_t a_base = smem_u32(s_a), b_base = smem_u32(s_b);
            int stage = 0; uint32_t phase = 0;
            int as = 0; uint32_t aphase = 0;
            uint32_t bphase = 0;
            for (int w = 0; w < p.n_waves; ++w) {
                int nt; int64_t b0, b1;
                if (!wave_item(w, nt, b0, b1)) continue;
                mbar_wait(bfull, bphase);
                tc_fence_after();
                for (int64_t pb = b0; pb < b1; ++pb) {
                    mbar_wait(&tempty[as], aphase ^ 1);
                    tc_fence_after();
                    const uint32_t d = tmem_base + as * 256;
                    for (int kb = 0; kb < kblocks; ++kb) {
                        mbar_wait(&full[stage], phase);
                        tc_fence_after();
                        const uint64_t da = make_kmajor_desc(a_base + stage * E_A_BYTES), db = make_kmajor_desc(b_base + kb * B_KB_BYTES);
#pragma unroll
                        for (int k = 0; k < 4; ++k) umma_i8_pair_if(d, da + 2 * k, db + 2 * k, idesc, (kb | k) ? 1u : 0u, GML_DBG(p, 16) ? 0u : lane_leader);
                        umma_commit_pair_if(&empty[stage], lane_leader);
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                    }
                    umma_commit_pair_if(&tfull[as], lane_leader);
                    if (++as == 2) { as = 0; aphase ^= 1; }
                }
                umma_commit_pair_if(bempty, lane_leader);
                bphase ^= 1;
            }
        }
    } else {
        // ================= epilogue warps of this CTA: its own 128 samples of every pair-step =================
        const int quarter = warp & 3;
        const int node0 = ((warp - 2) >> 2) * E_NPT;
        const int row = quarter * 32 + lane;
        ItemObjective obj;
        int as = 0; uint32_t aphase = 0;
        int slot = 0; uint32_t sphase = 0;
        const uint32_t tempty_leader0 = mapa_rank(smem_u32(&tempty[0]), 0), tempty_leader1 = mapa_rank(smem_u32(&tempty[1]), 0);
        const uint32_t tlane = tmem_base + ((uint32_t)(quarter * 32) << 16) + node0;
        const uint32_t scale_addr = smem_u32(s_scale) + 4 * node0;
        for (int w = 0; w < p.n_waves; ++w) {
            int nt; int64_t b0, b1;
            if (!wave_item(w, nt, b0, b1)) continue;
            obj.begin<GRAD>(p, nt, node0, s_scale);
            auto block_of = [&](int64_t pb) { return min(2 * pb + (int64_t)rank, p.sample_blocks - 1) * p.block_stride; };
            if (GML_DBG(p, 1)) {                        // ablation: no epilogue, only the barrier hand-shakes
                for (int64_t pb = b0; pb < b1; ++pb) {
                    mbar_wait(&sfull[slot], sphase);
                    mbar_wait(&tfull[as], aphase);
                    tc_fence_after();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) { mbar_arrive_cluster(as ? tempty_leader1 : tempty_leader0); mbar_arrive(&sempty[slot]); }
                    if (++as == 2) { as = 0; aphase ^= 1; }
                    if (++slot == 2) { slot = 0; sphase ^= 1; }
                }
                continue;
            }
            if (XL == 4) {
                // 4-limb passes: plain form (one x16 load group per block); the pipelined form below needs 2 x 32
                // accumulator registers there, spills, and measured slower (5.6 vs 5.0 ms at K = 2e6)
                float wk_next = b0 < b1 ? __ldg(p.w32 + block_of(b0) * 128 + row) : 0.f;
                for (int64_t pb = b0; pb < b1; ++pb) {
                    const bool valid = 2 * pb + (int64_t)rank < p.sample_blocks;
                    const int64_t sb = block_of(pb);
                    obj.next_block();
                    const float wk = wk_next;
                    if (pb + 1 < b1) wk_next = __ldg(p.w32 + block_of(pb + 1) * 128 + row);
                    mbar_wait(&sfull[slot], sphase);
                    mbar_wait(&tfull[as], aphase);
                    tc_fence_after();
                    const uint32_t tempty_leader = as ? tempty_leader1 : tempty_leader0;
                    if (!valid) {                           // the second block of an odd tail: hand everything back unused
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) { mbar_arrive_cluster(tempty_leader); mbar_arrive(&sempty[slot]); }
                    } else {
                        uint8_t* rgp[4];
                        digit_planes<NR>(p, true, sb, nt, node0, row, rgp);
                        uint32_t sw[4];
                        spin_words(p, smem_u32(s_spin) + slot * E_S_BYTES, row, node0, sw);
                        int32_t a[4][E_NPT];
                        epi_issue<XL>(tlane + as * 256, a);
                        tmem_ld_wait();
                        tc_fence_before();                   // accumulator fully read: hand it back to the MMA warp
                        __syncwarp();
                        if (lane == 0) mbar_arrive_cluster(tempty_leader);
                        energy_epilogue<FORM, GRAD, XL, NR>(p, a, sw, scale_addr, rgp, 0, wk, obj.facc);
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&sempty[slot]);
                    }
                    if (++as == 2) { as = 0; aphase ^= 1; }
                    if (++slot == 2) { slot = 0; sphase ^= 1; }
                }
                obj.flush();
                continue;
            }
            // Software pipeline over half-blocks (8 of the thread's 16 nodes): the TMEM loads of the next chunk are in
            // flight while the current chunk is evaluated -- also across block boundaries when the next accumulator is
            // already published -- so TMEM read latency / bandwidth overlaps the math instead of preceding it.
            int32_t ra[4][8], rb[4][8];
            float wk_next = b0 < b1 ? __ldg(p.w32 + block_of(b0) * 128 + row) : 0.f;
            if (b0 < b1) {
                mbar_wait(&sfull[slot], sphase);
                mbar_wait(&tfull[as], aphase);
                tc_fence_after();
                epi_issue<XL>(tlane + as * 256, ra);
            }
            for (int64_t pb = b0; pb < b1; ++pb) {
                const bool valid = 2 * pb + (int64_t)rank < p.sample_blocks;      // false: second block of an odd tail (nothing is stored or summed)
                const int64_t sb = block_of(pb);
                obj.next_block();
                const float wk = valid ? wk_next : 0.f;
                if (pb + 1 < b1) wk_next = __ldg(p.w32 + block_of(pb + 1) * 128 + row);
                uint8_t* rgp[4];
                digit_planes<NR>(p, valid, sb, nt, node0, row, rgp);
                uint32_t sw[4];
                spin_words(p, smem_u32(s_spin) + slot * E_S_BYTES, row, node0, sw);
                // The 16 spin bytes of this thread are in registers: hand the slot back NOW.  Releasing it only after the
                // block's math (as the first version did) chains the TMA producer -- which loads spin tile b+2 in order
                // with the histogram tiles of block b+2 -- to the END of epilogue b, and the MMA warp then starts every
                // block by waiting for histogram tiles (ncu: a third of its samples sat on full[stage] of k-block 0).
                __syncwarp();
                if (lane == 0) mbar_arrive(&sempty[slot]);
                // ---- nodes 0..7 (in ra); nodes 8..15 start loading
                epi_wait<XL>(ra);
                epi_issue<XL>(tlane + as * 256 + 8, rb);
                energy_epilogue<FORM, GRAD, XL, NR>(p, ra, sw, scale_addr, rgp, 0, wk, obj.facc);
                // ---- nodes 8..15 (in rb): the accumulator is now fully read
                epi_wait<XL>(rb);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(as ? tempty_leader1 : tempty_leader0);
                const int as_n = as ^ 1, slot_n = slot ^ 1;
                const uint32_t aphase_n = as ? aphase ^ 1 : aphase, sphase_n = slot ? sphase ^ 1 : sphase;
                bool pre = false;
                if (pb + 1 < b1) {
                    pre = __all_sync(0xffffffffu, mbar_test(&tfull[as_n], aphase_n) && mbar_test(&sfull[slot_n], sphase_n));
                    if (pre) { tc_fence_after(); epi_issue<XL>(tlane + as_n * 256, ra); }
                }
                energy_epilogue<FORM, GRAD, XL, NR>(p, rb, sw + 2, scale_addr + 32, rgp, 8, wk, obj.facc + 8);
                as = as_n; aphase = aphase_n; slot = slot_n; sphase = sphase_n;
                if (pb + 1 < b1 && !pre) {
                    mbar_wait(&sfull[slot], sphase);
                    mbar_wait(&tfull[as], aphase);
                    tc_fence_after();
                    epi_issue<XL>(tlane + as * 256, ra);
                }
            }
            obj.flush();
        }
    }
    tc_fence_before();
    cluster_sync_all();                       // the peer's shared memory and TMEM stay alive until both CTAs are done
    if (warp == 1) tmem_dealloc_pair(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------
// GEMM-2: gradient contraction, split over sample ranges
// ------------------------------------------------------------------------------------------
struct GradParams {
    int Fp, m_tiles, f_tiles;
    int64_t r_rows_per_limb;      // Nn_pad2
    int n_splits;                 // sample ranges; work item = (split, output tile)
    int64_t sample_blocks, block_stride;   // as in EnergyParams
    long long* G;                 // [Nn_pad2 x Fp] int64
    int dbg;                      // ablation switches (GML_DBG)
};

constexpr int G_TILE_BYTES = 128 * 128;
constexpr int64_t G_MAX_BLOCKS = 1 << 16;   // int32 accumulators: |acc| <= 255 * 128 * blocks < 2^31
// Output tile = 128 nodes x FT features per residual limb, all limbs resident in TMEM (NR * FT <= 512 columns).
// FT = 256 halves the shared-memory fill traffic per MAC of the R operand (the kernels sit at the L2 -> SM
// bandwidth, not at the tensor pipe, with 128-wide tiles: ablation in profiles/r1_ablation.txt); it fits for NR = 2.
__host__ __device__ constexpr int g_stage_bytes(int nr, int ft) { return nr * G_TILE_BYTES + ft * 128; }
__host__ __device__ constexpr int g_stages(int nr, int ft) { return (210 * 1024) / g_stage_bytes(nr, ft) >= 4 ? 4 : (210 * 1024) / g_stage_bytes(nr, ft); }

// Work decomposition: item = (sample split ks, output tile), split-major and dealt round-robin, one item
// per CTA when tiles * splits <= #SMs.  All CTAs of a split then sweep the SAME sample blocks in lockstep
// for different output tiles, so every R / Q operand tile is fetched from HBM once and shared through L2.
template <int NR, int FT>
__global__ void __launch_bounds__(192, 1) tc_grad_kernel(const __grid_constant__ CUtensorMap tmRa,   // R  [SB*nR*Nn_pad2 x 128], box 128 rows, SW128
                                                        const __grid_constant__ CUtensorMap tmQ,    // Qb [SB*Fp x 128], box FT rows, SW128
                                                        GradParams p) {
    static_assert(NR * FT <= 512, "the limb accumulators must fit the 512 TMEM columns");
    constexpr int STAGE_BYTES = g_stage_bytes(NR, FT);
    constexpr int G_STAGES = g_stages(NR, FT);
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + G_STAGES * STAGE_BYTES);
    uint64_t* full = bars;
    uint64_t* empty = bars + G_STAGES;
    uint64_t* tfull = bars + 2 * G_STAGES;
    uint64_t* tempty = tfull + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 1);
    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // warp index, uniform for the compiler

    const int tiles = p.m_tiles * p.f_tiles;
    const int n_items = tiles * p.n_splits;

    if (threadIdx.x == 0) {
        for (int i = 0; i < G_STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        mbar_init(tfull, 1); mbar_init(tempty, 4);
        fence_barrier_init();
        prefetch_tmap(&tmRa); prefetch_tmap(&tmQ);
    }
    if (warp == 1) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

    auto decode = [&](int item, int& mt, int& ft, int64_t& b0, int64_t& b1) {
        const int ks = item / tiles, r = item % tiles;
        mt = r / p.f_tiles; ft = r % p.f_tiles;
        b0 = p.sample_blocks * ks / p.n_splits;
        b1 = p.sample_blocks * (ks + 1) / p.n_splits;
    };

    if (warp == 0) {
        // ================= TMA producer (whole warp converged, elected lane issues) =================
        const uint32_t leader = elect_one_pred();
        int stage = 0; uint32_t phase = 0;
        for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
            int mt, ft; int64_t b0, b1;
            decode(item, mt, ft, b0, b1);
            for (int64_t eb = b0; eb < b1; ++eb) {
                const int64_t b = eb * p.block_stride;
                mbar_wait(&empty[stage], phase ^ 1);
                const uint32_t ld = GML_DBG(p, 4) ? 0u : leader;
                mbar_expect_tx_if(&full[stage], ld ? STAGE_BYTES : 0, leader);
                uint8_t* s = smem + stage * STAGE_BYTES;
#pragma unroll
                for (int j = 0; j < NR; ++j)
                    tma_load_2d_if(s + j * G_TILE_BYTES, &tmRa, &full[stage], 0, (int)((b * NR + j) * p.r_rows_per_limb) + mt * 128, ld);
                tma_load_2d_if(s + NR * G_TILE_BYTES, &tmQ, &full[stage], 0, (int)(b * p.Fp) + ft * FT, ld);
                if (++stage == G_STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer (whole warp converged, elected lane issues) =================
        const uint32_t leader = elect_one_pred();
        constexpr uint32_t idesc = make_idesc_i8(128, FT, /*a_unsigned=*/true);     // A = residual digit bytes (u8), B = spins (s8)
        const uint32_t s_base = smem_u32(smem);
        int stage = 0; uint32_t phase = 0, aphase = 0;
        for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
            int mt, ft; int64_t b0, b1;
            decode(item, mt, ft, b0, b1);
            for (int64_t c0 = b0; c0 < b1; c0 += G_MAX_BLOCKS) {       // sub-chunks bounded by the int32 range
                const int64_t c1 = min(c0 + G_MAX_BLOCKS, b1);
                mbar_wait(tempty, aphase ^ 1);
                tc_fence_after();
                for (int64_t b = c0; b < c1; ++b) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t s_addr = s_base + stage * STAGE_BYTES;
                    const uint64_t db = make_kmajor_desc(s_addr + NR * G_TILE_BYTES);
#pragma unroll
                    for (int j = 0; j < NR; ++j) {
                        const uint64_t da = make_kmajor_desc(s_addr + j * G_TILE_BYTES);
#pragma unroll
                        for (int k = 0; k < 4; ++k) umma_i8_if(tmem_base + j * FT, da + 2 * k, db + 2 * k, idesc, (b > c0 || k) ? 1u : 0u, leader);
                    }
                    umma_commit_if(&empty[stage], leader);
                    if (++stage == G_STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit_if(tfull, leader);
                aphase ^= 1;
            }
        }
    } else {
        const int quarter = warp & 3;
        const int row = quarter * 32 + lane;
        uint32_t aphase = 0;
        for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
            int mt, ft; int64_t b0, b1;
            decode(item, mt, ft, b0, b1);
            for (int64_t c0 = b0; c0 < b1; c0 += G_MAX_BLOCKS) {
                mbar_wait(tfull, aphase);
                tc_fence_after();
                const uint32_t tbase = tmem_base + ((uint32_t)(quarter * 32) << 16);
                long long* dst = p.G + ((int64_t)mt * 128 + row) * p.Fp + ft * FT;
#pragma unroll 1
                for (int c = 0; c < FT / 16; ++c) {
                    int32_t acc[NR][16];
#pragma unroll
                    for (int j = 0; j < NR; ++j) tmem_ld16(tbase + j * FT + c * 16, acc[j]);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        long long v = 0;
#pragma unroll
                        for (int j = 0; j < NR; ++j) v = v * 256 + (long long)acc[j][i];
                        if (v != 0) atomicAdd(reinterpret_cast<unsigned long long*>(dst + c * 16 + i), (unsigned long long)v);
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty);
                aphase ^= 1;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// Column sums of the +-1 feature matrix over the sample blocks of a pass (every `stride`-th block of the
// sample-blocked copy Qb [SB][Fp][128]): colsum[f] = sum_k S[k,f].  The residual digits hold q + BIAS, so
//     sum_k (q_k + BIAS) S[k,f] - BIAS * colsum[f] = sum_k q_k S[k,f]      exactly, in integers.
constexpr int CS_BLOCKS_PER_CTA = 64;
__global__ void __launch_bounds__(256) tc_colsum_kernel(const int8_t* __restrict__ Qb, int Fp, int64_t n_blocks, int64_t stride,
                                                      long long* __restrict__ colsum) {
    const int f = blockIdx.y * 256 + threadIdx.x;
    if (f >= Fp) return;
    const int64_t e0 = (int64_t)blockIdx.x * CS_BLOCKS_PER_CTA, e1 = min(e0 + CS_BLOCKS_PER_CTA, n_blocks);
    int acc = 0;
    for (int64_t e = e0; e < e1; ++e) {
        const int4* row = reinterpret_cast<const int4*>(Qb + ((e * stride) * Fp + f) * 128);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int4 v = __ldg(row + i);
            acc = __dp4a(v.x, 0x01010101, acc); acc = __dp4a(v.y, 0x01010101, acc);
            acc = __dp4a(v.z, 0x01010101, acc); acc = __dp4a(v.w, 0x01010101, acc);
        }
    }
    if (acc) atomicAdd(reinterpret_cast<unsigned long long*>(colsum + f), (unsigned long long)(long long)acc);
}
// gradient accumulators start at -BIAS * colsum[f] (see above)
__global__ void tc_grad_init_kernel(long long* __restrict__ G, const long long* __restrict__ colsum, long long bias, int64_t n, int Fp) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) G[i] = -bias * colsum[i % Fp];
}

// int64 sums -> double objective / gradient (and the logRISE normalisation, :279)
__global__ void tc_finalize_kernel(int form, int Fp, const double* __restrict__ fsum,
                                   const long long* __restrict__ G64, const double* __restrict__ delta,
                                   double* __restrict__ f_out, double* __restrict__ g_out, int want_grad,
                                   const int* __restrict__ act_idx /* slot -> node, or null */) {
    const int slot = blockIdx.x;
    const int u = act_idx ? act_idx[slot] : slot;
    if (u < 0) return;
    const double fs = fsum[slot];
    if (threadIdx.x == 0) f_out[u] = (form == GML_B200_LOGRISE) ? log(fs) : fs;
    if (!want_grad) return;
    const double sc = -delta[slot] / (form == GML_B200_LOGRISE ? fs : 1.0);
    for (int f = threadIdx.x; f < Fp; f += blockDim.x) g_out[(int64_t)u * Fp + f] = sc * (double)G64[(int64_t)slot * Fp + f];
}

// Active-set compaction: sample-major spin matrix of the active nodes only, P_act[k][slot] = s_{idx[slot]}[k]
// (columns >= n hold 0), the source of the epilogue's spin tiles while a compacted node list is in force.
__global__ void __launch_bounds__(256) tc_gather_spins_kernel(const int8_t* __restrict__ base, int64_t Kp, const int32_t* __restrict__ spin_row,
                                                            const int* __restrict__ act_idx, int n, int cap, int8_t* __restrict__ P_act) {
    __shared__ int8_t tile[64][128 + 16];
    const int64_t k0 = (int64_t)blockIdx.x * 128;
    const int j0 = blockIdx.y * 64;
    for (int r = threadIdx.x >> 3; r < 64; r += 32) {
        const int j = j0 + r;
        int4 v = make_int4(0, 0, 0, 0);
        if (j < n && act_idx[j] >= 0) v = *reinterpret_cast<const int4*>(base + (int64_t)spin_row[act_idx[j]] * Kp + k0 + (threadIdx.x & 7) * 16);
        *reinterpret_cast<int4*>(&tile[r][(threadIdx.x & 7) * 16]) = v;
    }
    __syncthreads();
    const int s = threadIdx.x >> 1, h = threadIdx.x & 1;
    uint32_t out[8];
#pragma unroll
    for (int w = 0; w < 8; ++w) {
        uint32_t v = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) v |= (uint32_t)(uint8_t)tile[h * 32 + w * 4 + b][s] << (8 * b);
        out[w] = v;
    }
    int4* dst = reinterpret_cast<int4*>(P_act + (k0 + s) * cap + j0 + h * 32);
    dst[0] = make_int4(out[0], out[1], out[2], out[3]);
    dst[1] = make_int4(out[4], out[5], out[6], out[7]);
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
CUtensorMap make_map_2d(const void* base, uint64_t inner, uint64_t outer, uint32_t box_inner, uint32_t box_outer,
                        CUtensorMapSwizzle swz) {
    CUtensorMap m;
    cuuint64_t dims[2] = {inner, outer};
    cuuint64_t strides[1] = {inner};   // bytes (int8 elements)
    cuuint32_t box[2] = {box_inner, box_outer};
    cuuint32_t estr[2] = {1, 1};
    // resolved through the runtime so that libgml_b200.so does not link libcuda (it must still load on a
    // box without a driver, where every compute entry point reports GML_B200_ECUDA)
    typedef CUresult (*encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static encode_fn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        GML_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        GML_REQUIRE(fn != nullptr && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available in this driver");
        encode = reinterpret_cast<encode_fn>(fn);
    }
    const CUresult rc = encode(&m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides, box, estr,
                                               CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (rc != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with code " + std::to_string((int)rc));
        throw CudaError{GML_B200_ECUDA};
    }
    return m;
}

// ---- the kernel instantiations, each named once; BackendTC::configure() and eval() both go through the lookups below
using EnergyKernel = void (*)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, EnergyParams);
using GradKernel = void (*)(CUtensorMap, CUtensorMap, GradParams);
template <class K> struct Launch { K kernel; int smem; };   // kernel and its dynamic shared memory

// form: RPLE, or RISE for both RISE and logRISE; xl = iterate limbs (4 fine, 3 coarse, 2 rough level); nr = residual
// digit planes, read by the gradient passes only.  The gradient kernels are the ones BackendTC::level_nr() can select:
// fine nr = nR in {3, 4}, coarse nr = max(2, nR - 1) in {2, 3}, rough nr = 1 (tests/test_gpu_tc_passes.py checks that
// every instantiation here is launched by some pass).
struct EnergyInstance { int form; bool grad; int xl, nr; EnergyKernel stream, pair; };
template <int FORM, bool GRAD, int XL, int NR>
EnergyInstance energy_instance() { return {FORM, GRAD, XL, NR, tc_energy_kernel<FORM, GRAD, XL, NR>, tc_energy_pair_kernel<FORM, GRAD, XL, NR>}; }
const EnergyInstance ENERGY_KERNELS[] = {
    energy_instance<GML_B200_RISE, false, 4, 2>(), energy_instance<GML_B200_RISE, true, 4, 3>(), energy_instance<GML_B200_RISE, true, 4, 4>(),
    energy_instance<GML_B200_RISE, false, 3, 2>(), energy_instance<GML_B200_RISE, true, 3, 2>(), energy_instance<GML_B200_RISE, true, 3, 3>(),
    energy_instance<GML_B200_RISE, false, 2, 1>(), energy_instance<GML_B200_RISE, true, 2, 1>(),
    energy_instance<GML_B200_RPLE, false, 4, 2>(), energy_instance<GML_B200_RPLE, true, 4, 3>(), energy_instance<GML_B200_RPLE, true, 4, 4>(),
    energy_instance<GML_B200_RPLE, false, 3, 2>(), energy_instance<GML_B200_RPLE, true, 3, 2>(), energy_instance<GML_B200_RPLE, true, 3, 3>(),
    energy_instance<GML_B200_RPLE, false, 2, 1>(), energy_instance<GML_B200_RPLE, true, 2, 1>()};
Launch<EnergyKernel> energy_kernel(int form, bool grad, int xl, int nr, bool pair) {
    const int kform = form == GML_B200_RPLE ? GML_B200_RPLE : GML_B200_RISE;
    for (const EnergyInstance& k : ENERGY_KERNELS)
        if (k.form == kform && k.grad == grad && k.xl == xl && (k.nr == nr || !grad))    // one objective-only kernel serves every nr
            return pair ? Launch<EnergyKernel>{k.pair, e2_smem(xl)} : Launch<EnergyKernel>{k.stream, E_SMEM};
    GML_REQUIRE(false, "no tensor-core energy kernel for this formulation and precision level");
    return {nullptr, 0};
}

// nr = residual digit planes, ft = feature-tile width
struct GradInstance { int nr, ft; GradKernel kernel; };
const GradInstance GRAD_KERNELS[] = {{1, 128, tc_grad_kernel<1, 128>}, {1, 256, tc_grad_kernel<1, 256>}, {2, 128, tc_grad_kernel<2, 128>},
                                     {2, 256, tc_grad_kernel<2, 256>}, {3, 128, tc_grad_kernel<3, 128>}, {4, 128, tc_grad_kernel<4, 128>}};
Launch<GradKernel> grad_kernel(int nr, int ft) {
    for (const GradInstance& k : GRAD_KERNELS)
        if (k.nr == nr && k.ft == ft) return {k.kernel, g_stages(nr, ft) * g_stage_bytes(nr, ft) + 1024 + 128};
    GML_REQUIRE(false, "no tensor-core gradient kernel for this residual width");
    return {nullptr, 0};
}

struct BackendTC : EvalBackend {
    const NodeProblem& p;
    int Nn_pad1, Nn_pad2, nR, n_sms;   // nR: residual limbs of the fine level
    int level = 1;                      // 0 = coarse (3-limb iterate, nR-1 residual limbs), 1 = fine
    int32_t first_row = 0;   // spin rows of this shard are contiguous in `base`: spin_row[u] = first_row + u
    DevBuf<int8_t> X, R;                // X: iterate limbs, room for 4; each pass's quantiser rewrites the rows its limb count uses
    DevBuf<float> inv_dr;
    DevBuf<double> delta;
    DevBuf<double> fsum;
    DevBuf<long long> G64;
    DevBuf<long long> colsum;           // [Fp] column sums of the feature matrix over the blocks of the current stride
    int64_t colsum_stride = 0;          // stride colsum was computed for (0 = not yet)
    DevBuf<int> flags;
    DevBuf<uint8_t> r_scratch;
    // active-set compaction (set_active): slot -> node list, spins of the listed nodes, their TMA map
    const int* act_idx = nullptr;
    int n_act = 0;
    DevBuf<int8_t> P_act;
    CUtensorMap tmSvAct;
    const int8_t* P;
    const int8_t* Qb;
    const int8_t* spin_blocked = nullptr;
    int Fspin = 0;
    DevBuf<int8_t> base_blocked;
    CUtensorMap tmB[3], tmBh[3];        // limb tile / half limb tile of xl = 2, 3, 4 iterate limbs, at [xl - 2]
    CUtensorMap tmA, tmS, tmSv, tmRa, tmQ, tmQ256;
    bool pair_ok = false;               // the CTA-pair energy kernel applies (limb half-tile fits: Fp <= E2_MAX_FP)
    bool spin_vec = false;

    BackendTC(const NodeProblem& prob, cudaStream_t st) : p(prob) {
        Histogram& h = *p.hist;
        // Residual limbs: the rounding noise of the gradient is ~0.3 sqrt(K) wmax e^B / qmax(nR).  3 limbs
        // (qmax 1e6) keep it below 1e-8 for near-uniform counts; strongly weighted histograms get 4.
        nR = (std::sqrt(h.K_total) * h.wmax > 2e-3) ? 4 : 3;
        Nn_pad1 = (int)round_up(p.Nn, NODE_TILE1);
        Nn_pad2 = (int)round_up(p.Nn, NODE_TILE2);
        int dev = 0;
        GML_CUDA(cudaGetDevice(&dev));
        GML_CUDA(cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, dev));
        P = ensure_P(h, p.Q, p.Fp, st);
        X.alloc((size_t)Nn_pad1 * X_LIMBS_MAX * p.Fp);
        R.alloc((size_t)nR * Nn_pad2 * h.Kp);
        inv_dr.alloc(Nn_pad1); delta.alloc(Nn_pad1);
        fsum.alloc(Nn_pad1);
        G64.alloc((size_t)Nn_pad2 * p.Fp);
        colsum.alloc(p.Fp);
        flags.alloc(1);
        r_scratch.alloc(4 * NODE_TILE1 * 128);
        GML_CUDA(cudaMemsetAsync(flags.p, 0, sizeof(int), st));
        // rows of R that belong to padding nodes are never written by GEMM-1 tiles beyond Nn_pad1: clear once
        GML_CUDA(cudaMemsetAsync(R.p, 0, (size_t)nR * Nn_pad2 * h.Kp, st));
        tmA = make_map_2d(P, p.Fp, h.Kp, 128, 128, CU_TENSOR_MAP_SWIZZLE_128B);
        for (int xl = 2; xl <= X_LIMBS_MAX; ++xl) {
            tmB[xl - 2] = make_map_2d(X.p, p.Fp, (uint64_t)Nn_pad1 * xl, 128, xl * NODE_TILE1, CU_TENSOR_MAP_SWIZZLE_128B);
            tmBh[xl - 2] = make_map_2d(X.p, p.Fp, (uint64_t)Nn_pad1 * xl, 128, xl * 32, CU_TENSOR_MAP_SWIZZLE_128B);
        }
        pair_ok = p.Fp <= E2_MAX_FP && !std::getenv("GML_B200_NO_PAIR");
        // Sample-blocked layouts: every TMA box is one contiguous 8/16 KB chunk (one 2 MB page) instead of
        // 64/128 rows that are Kp bytes apart.
        const uint64_t SB = (uint64_t)(h.Kp / 128);
        GML_REQUIRE(SB * nR * Nn_pad2 < (1ull << 31) && SB * p.Fp < (1ull << 31),
                    "problem too large for 32-bit TMA row coordinates: shard the nodes or the samples");
        Qb = ensure_Qb(h, p.Q, p.Fp, st);
        // spins of the shard's nodes: for pairwise problems they are rows of Q itself; multibody problems
        // read them from the blocked copy of `base` (built on demand)
        if (p.Q == h.base.p) { spin_blocked = Qb; Fspin = p.Fp; }
        else {
            base_blocked.alloc((size_t)h.Kp * h.Fb);
            launch_block_copy(h.base.p, base_blocked.p, h.Fb, h.Kp, st);
            spin_blocked = base_blocked.p; Fspin = h.Fb;
        }
        GML_REQUIRE(SB * Fspin < (1ull << 31), "problem too large for 32-bit TMA row coordinates: shard the samples");
        tmS = make_map_2d(spin_blocked, 128, SB * Fspin, 128, NODE_TILE1, CU_TENSOR_MAP_SWIZZLE_NONE);
        // 64B swizzle: 16-byte chunk index ^= (sample >> 1) & 3, so the epilogue's 16-byte loads (64-byte row pitch) are bank-conflict free
        tmSv = make_map_2d(P, p.Fp, h.Kp, NODE_TILE1, 128, CU_TENSOR_MAP_SWIZZLE_64B);
        tmRa = make_map_2d(R.p, 128, SB * nR * Nn_pad2, 128, 128, CU_TENSOR_MAP_SWIZZLE_128B);
        tmQ = make_map_2d(Qb, 128, SB * p.Fp, 128, 128, CU_TENSOR_MAP_SWIZZLE_128B);
        tmQ256 = make_map_2d(Qb, 128, SB * p.Fp, 128, 256, CU_TENSOR_MAP_SWIZZLE_128B);
        GML_CUDA(cudaMemcpyAsync(&first_row, p.spin_row.p, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        GML_CUDA(cudaStreamSynchronize(st));
        // vector spin loads need the shard's first spin column 16-byte aligned in P (TMA inner-dimension alignment)
        spin_vec = (p.Q == h.base.p) && (first_row % 16 == 0);
        configure();
    }

    template <class K> static void set_smem(Launch<K> k) {
        GML_CUDA(cudaFuncSetAttribute(k.kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, k.smem));
    }
    void configure() {
        for (const EnergyInstance& k : ENERGY_KERNELS) {
            set_smem(energy_kernel(k.form, k.grad, k.xl, k.nr, false));
            set_smem(energy_kernel(k.form, k.grad, k.xl, k.nr, true));
        }
        for (const GradInstance& k : GRAD_KERNELS) set_smem(grad_kernel(k.nr, k.ft));
    }
    // Number of sample ranges for `tiles` output tiles on n_sms persistent CTAs: the smallest count from one
    // wave upwards whose items fill the last wave to >= 96 % (items are dealt round-robin, range-major).
    static int balanced_splits(int tiles, int n_sms, int64_t max_splits) {
        const int s0 = std::max(1, n_sms / tiles);
        int best = s0; double best_eff = 0.0;
        for (int s = s0; s <= 8 * s0 + 8; ++s) {
            const int64_t items = (int64_t)tiles * s, waves = ceil_div(items, n_sms);
            const double eff = (double)items / (double)(waves * n_sms);
            if (eff > best_eff + 1e-9) { best = s; best_eff = eff; }
            if (eff >= 0.96) break;
        }
        return (int)std::max<int64_t>(1, std::min<int64_t>(best, max_splits));
    }

    // Sample ranges of the CTA-pair energy kernel.  The pairs that work on one range (one per node tile) share its
    // histogram tiles through L2 only while they stay within a few hundred blocks of each other; with one long range
    // per pair (the wave-balanced minimum) they drift apart over thousands of steps and every P tile is fetched from
    // HBM about twice (ncu: 20.1 GB read for a 10.2 GB histogram).  Ranges of at most ITEM_STEPS pair-steps bound the
    // drift; the limb-tile reload per item (96 KB against 256 KB of histogram tiles per step) stays below 0.2 %.
    static int pair_groups(int tiles, int n_pairs, int64_t pair_blocks) {
        constexpr int ITEM_STEPS = 256;
        const int64_t g_min = std::max<int64_t>(1, ceil_div(pair_blocks, ITEM_STEPS));
        const int wave = balanced_splits(tiles, n_pairs, pair_blocks);
        if (g_min <= wave) return wave;
        int64_t best = g_min; double best_eff = 0.0;
        for (int64_t g = g_min; g < g_min + 2 * n_pairs && g <= pair_blocks; ++g) {
            const int64_t items = (int64_t)tiles * g, waves = ceil_div(items, n_pairs);
            const double eff = (double)items / (double)(waves * n_pairs);
            if (eff > best_eff + 1e-9) { best = g; best_eff = eff; }
            if (eff >= 0.985) break;
        }
        return (int)std::min<int64_t>(best, pair_blocks);
    }

    double lattice() const override { return level < 0 ? X_LATTICE_ROUGH : (level == 0 ? X_LATTICE_COARSE : X_LATTICE_FINE); }
    double x_range() const override { return level <= 0 ? X_RANGE_COARSE : X_RANGE_FINE; }
    int level_xl() const { return level < 0 ? 2 : (level == 0 ? 3 : 4); }
    int level_nr() const { return level < 0 ? 1 : (level == 0 ? std::max(2, nR - 1) : nR); }
    // rounding noise of a gradient component: ~0.29 sqrt(K) wmax e^B / qmax(nr); e^B ~ 20 as a typical upper value
    double grad_noise() const override {
        const Histogram& h = *p.hist;
        return std::max(1e-9, 0.29 * std::sqrt(h.K_total) * h.wmax * 20.0 / r_qmax(level_nr()));
    }
    // level 0 needs |x| < 1 (checked by the quantiser: an overflow pins the backend to the fine level)
    bool coarse_overflow = false;
    // levels: -1 rough, 0 coarse, 1 fine.  The rough level's single 8-bit residual plane is only accurate enough for
    // near-uniform counts (the same condition that lets the fine level use 3 planes).
    bool set_level(int lv, cudaStream_t) override {
        int take = lv;
        if (take < 0 && nR != 3) take = 0;
        level = (take <= 0 && !coarse_overflow) ? take : 1;
        return level == lv;
    }
    const int* device_flags() const override { return flags.p; }
    void note_coarse_overflow() override { coarse_overflow = true; }

    // ---- strided sample subsets (multilevel continuation): a pass uses every `stride`-th 128-sample block
    int64_t stride = 1;
    double set_subsample(int64_t new_stride, cudaStream_t st) override {
        stride = std::max<int64_t>(1, new_stride);
        return subsample_weight(*p.hist, stride, st);
    }

    // ---- per-kernel timing with CUDA events on the launch stream
    bool profiling = false;
    struct Span { cudaEvent_t a, b; int kind; };
    std::vector<Span> spans;
    void set_profiling(bool on) override { profiling = on; }
    void span_begin(int kind, cudaStream_t st) {
        if (!profiling || stride != 1 || act_idx) return;   // only launches over the whole histogram and the whole shard are timed
        Span s; s.kind = kind;
        GML_CUDA(cudaEventCreate(&s.a)); GML_CUDA(cudaEventCreate(&s.b));
        GML_CUDA(cudaEventRecord(s.a, st));
        spans.push_back(s);
    }
    void span_end(cudaStream_t st) { if (profiling && stride == 1 && !act_idx) GML_CUDA(cudaEventRecord(spans.back().b, st)); }
    void collect_profile(double* out) override {
        for (auto& s : spans) {
            float ms = 0.f;
            GML_CUDA(cudaEventSynchronize(s.b));
            GML_CUDA(cudaEventElapsedTime(&ms, s.a, s.b));
            out[s.kind] += ms;
            if (s.kind == 0) out[3] += 1.0;      // number of timed full passes
            cudaEventDestroy(s.a); cudaEventDestroy(s.b);
        }
        spans.clear();
    }
    ~BackendTC() override { for (auto& s : spans) { cudaEventDestroy(s.a); cudaEventDestroy(s.b); } }

    // Restrict the following passes to the listed nodes (slot j evaluates node d_idx[j]; entries < 0 are empty
    // slots); nullptr restores the full shard.  The work of a pass scales with the padded list length.
    bool set_active(const int* d_idx, int n, cudaStream_t st) override {
        if (!d_idx || n <= 0 || n >= p.Nn) { act_idx = nullptr; n_act = 0; return true; }
        const Histogram& h = *p.hist;
        const int cap = (int)round_up(n, NODE_TILE2);
        P_act.alloc((size_t)h.Kp * cap);
        tc_gather_spins_kernel<<<dim3((unsigned)(h.Kp / 128), (unsigned)(cap / 64)), 256, 0, st>>>(h.base.p, h.Kp, p.spin_row.p, d_idx, n, cap, P_act.p);
        GML_LAUNCHED();
        tmSvAct = make_map_2d(P_act.p, cap, h.Kp, NODE_TILE1, 128, CU_TENSOR_MAP_SWIZZLE_64B);
        act_idx = d_idx; n_act = n;
        return true;
    }

    void eval(const double* x, bool want_grad, double* f_out, double* g_out, cudaStream_t st) override {
        const Histogram& h = *p.hist;
        const int xl = level_xl();
        const int nr = level_nr();                                  // residual digit planes of this pass
        const int n_nodes = act_idx ? n_act : p.Nn;                // slots of this pass
        const int pad1 = (int)round_up(n_nodes, NODE_TILE1), pad2 = (int)round_up(n_nodes, NODE_TILE2);
        tc_quantize_x_kernel<<<pad1, 128, 0, st>>>(x, n_nodes, p.Fp, p.form, h.wmax, nr, xl, NODE_TILE1, 1.0 / lattice(), X.p,
                                                   inv_dr.p, delta.p, flags.p, act_idx);
        GML_LAUNCHED();
        GML_CUDA(cudaMemsetAsync(fsum.p, 0, sizeof(double) * pad1, st));
        EnergyParams ep{};
        ep.Fp = p.Fp; ep.Fspin = Fspin; ep.n_tiles = pad1 / NODE_TILE1;
        ep.block_stride = stride; ep.sample_blocks = ceil_div(h.Kp / 128, stride); ep.r_rows_per_limb = Nn_pad2; ep.lattice = (float)lattice();
        ep.w32 = h.w32.p; ep.inv_dr = inv_dr.p; ep.fsum = fsum.p; ep.R = reinterpret_cast<uint8_t*>(R.p); ep.r_scratch = r_scratch.p;
        ep.node_begin_row = act_idx ? 0 : first_row; ep.spin_vec = (act_idx || spin_vec) ? 1 : 0;
        const CUtensorMap& tmSvUse = act_idx ? tmSvAct : tmSv;
        const char* dbg_env = std::getenv("GML_B200_DBG");
        ep.dbg = dbg_env ? std::atoi(dbg_env) : 0;

        const bool pair = pair_ok && ep.sample_blocks >= 2;
        const int n_pairs = n_sms / 2;
        ep.n_groups = pair ? pair_groups(ep.n_tiles, n_pairs, (ep.sample_blocks + 1) / 2) : balanced_splits(ep.n_tiles, n_sms, ep.sample_blocks);
        const int grid1 = pair ? 2 * std::min(n_pairs, ep.n_tiles * ep.n_groups) : std::min(n_sms, ep.n_tiles * ep.n_groups);
        if (pair) {                                   // wave-aligned schedule of the pair kernel (see wave_item)
            const int used = grid1 / 2, T = ep.n_tiles;
            ep.n_waves = (int)ceil_div((int64_t)T * ep.n_groups, used);
            const int m = used / T;                   // whole ranges per wave (0: more tiles than pairs -> round robin)
            ep.g_main = m ? std::min(ep.n_groups, ep.n_waves * m) : 0;
        }
        const Launch<EnergyKernel> ek = energy_kernel(p.form, want_grad, xl, nr, pair);
        span_begin(want_grad ? 0 : 2, st);
        ek.kernel<<<grid1, E_THREADS, ek.smem, st>>>(tmA, pair ? tmBh[xl - 2] : tmB[xl - 2], tmS, tmSvUse, ep);
        GML_LAUNCHED();
        span_end(st);
        if (want_grad) {
            if (colsum_stride != stride) {
                GML_CUDA(cudaMemsetAsync(colsum.p, 0, sizeof(long long) * p.Fp, st));
                const int64_t nb = ceil_div(h.Kp / 128, stride);
                tc_colsum_kernel<<<dim3((unsigned)ceil_div(nb, CS_BLOCKS_PER_CTA), (unsigned)ceil_div(p.Fp, 256)), 256, 0, st>>>(Qb, p.Fp, nb, stride, colsum.p);
                GML_LAUNCHED();
                colsum_stride = stride;
            }
            {
                const int64_t n = (int64_t)pad2 * p.Fp;
                tc_grad_init_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(G64.p, colsum.p, (long long)r_bias(nr), n, p.Fp);
                GML_LAUNCHED();
            }
            GradParams gp{};
            const int ft = (nr <= 2 && p.Fp % 256 == 0) ? 256 : 128;   // feature-tile width
            gp.Fp = p.Fp; gp.m_tiles = pad2 / 128; gp.f_tiles = p.Fp / ft;
            gp.r_rows_per_limb = Nn_pad2; gp.block_stride = stride; gp.sample_blocks = ceil_div(h.Kp / 128, stride); gp.G = G64.p;
            gp.dbg = ep.dbg;
            const int tiles = gp.m_tiles * gp.f_tiles;
            gp.n_splits = balanced_splits(tiles, n_sms, gp.sample_blocks);
            const int grid2 = std::min(n_sms, tiles * gp.n_splits);
            const Launch<GradKernel> gk = grad_kernel(nr, ft);
            span_begin(1, st);
            gk.kernel<<<grid2, 192, gk.smem, st>>>(tmRa, ft == 256 ? tmQ256 : tmQ, gp);
            GML_LAUNCHED();
            span_end(st);
        }
        if (p.comm) {   // sample-sharded: exact int64 gradient sums and fp64 objective sums across the ranks
            comm_group_start(p.comm);
            comm_allreduce_sum_f64(p.comm, fsum.p, pad1, st);
            if (want_grad) comm_allreduce_sum_i64(p.comm, G64.p, (size_t)pad2 * p.Fp, st);
            comm_group_end(p.comm);
        }
        tc_finalize_kernel<<<n_nodes, 128, 0, st>>>(p.form, p.Fp, fsum.p, G64.p, delta.p, f_out, g_out, want_grad ? 1 : 0, act_idx);
        GML_LAUNCHED();
    }
};

}  // namespace

EvalBackend* make_backend_tc(const NodeProblem& p, cudaStream_t st) { return new BackendTC(p, st); }

}  // namespace gml
