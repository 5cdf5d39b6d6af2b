// Split-integer ("Ozaki") emulation of the two FP64 X contractions on the 5th-generation tensor cores.
//
//   Y = X~ A^T      (linearcorex.py:247 / :210)      M = samples,   X~ K-major;   N = factors, A planes K-major
//   D = X~^T Y      (linearcorex.py:259 / :211)      M = variables, X~ MN-major;  N = factors, Y^T planes K-major
//
// tcgen05.mma has no f64 kind, but kind::i8 multiplies int8 digits exactly into int32 TMEM accumulators.
// Each fp64 operand is written as a fixed-point number with S signed int8 digits ("planes") in radix R = 254:
//     v = 2^E * sum_{k=1..S} d_k R^-k,   |d_k| <= 127
// with one exponent E for all of X~ (standardised data is bounded; chosen from max|X~|), one per factor
// row of A and one per factor column of Y.  The product is then
//     sum_i x_i a_i = 2^(Ex+Ea) * sum_{g=2..S+1} R^-g * P_g,   P_g = sum_{k+l=g} sum_i dx_k[i] da_l[i]
// where every P_g is an exact int32 dot product (|d d'| < 2^14; the host caps the contraction length seen by one
// accumulator at 2^31 / (127^2 S) through split-K).  Pairs with k+l > S+1 are dropped (they sit below the digits that were
// truncated anyway).  S = 6 keeps 48 bits below the row / column maximum -- truncation at the level of binary64
// rounding, the FP64-faithful mode (measured parity 1e-11 or better on full fits); S = 5 keeps 40 bits; S = 3 is the
// opt-in fast mode (24 bits: fp32-equivalent like 3xTF32, at 3 bytes per element and int8 rates); S = 7 keeps 56 bits.
//
// One CTA owns a 128 x bn output tile (bn = 64, 128 for S <= 4, or narrower for the last factor tile) and S accumulators
// of bn TMEM columns (group g at column bn g).  Warp 0 streams operand planes with TMA (cp.async.bulk.tensor, 64 B /
// 128 B swizzle; the X~ planes are multicast across the CTA pair that shares them) through a 2-4 stage mbarrier ring; warp 1
// issues the tcgen05.mma (digit k of A against digits 0..S-1-k of B as ONE wide instruction) and commits to the ring;
// warps 2-5 drain TMEM (tcgen05.ld), recombine the groups in fp64 (Horner from the smallest weight) and store.  The
// same row-major int8 image of X~ feeds both contractions as their M operand: K-major in the first, MN-major in the
// second (128 samples or 128 variables per tile: no padded rows either way), so X~ is stored once (S bytes per element,
// less than fp64).  The factor-side operand is K-major in both (A planes [S][m][n]; Y planes stored transposed,
// [S][m][N_local]), which is what lets its digit planes sit back to back in shared memory for the wide instructions.
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace lcx {
namespace oz {

constexpr int kRadix = 254;   // R: digits use the full int8 range (measured 100x tighter parity than the power of two 128)
constexpr int kBM = 128;      // output rows per CTA (UMMA M)
constexpr int kBK = 64;       // contraction depth per pipeline stage (two UMMA K=32 steps)
// Output columns per CTA (UMMA N per digit plane).  S group accumulators of bn columns must fit the 512 TMEM columns:
// 64 for S = 5, 6; 128 for S <= 4, where one CTA then owns all of m <= 128 factors and the X~ tile is delivered to one
// SM instead of two (the kernels are bound by operand delivery into the SMs, DESIGN.md 4).
__host__ __device__ constexpr int bn_max(int S) { return S <= 4 ? 128 : 64; }
// Pipeline depth: as many stages of S (8 KB + bn_max 64 B) planes as fit in 220 KB, at most 4.
__host__ __device__ constexpr int stages_for(int S) {
    return (220 * 1024) / (S * (kBM * kBK + bn_max(S) * kBK)) >= 4 ? 4 : (220 * 1024) / (S * (kBM * kBK + bn_max(S) * kBK));
}
constexpr int kThreads = 192; // warp 0 TMA, warp 1 MMA, warps 2..5 epilogue

// ---- PTX wrappers ----------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
            smem_u32(dst)),
        "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
// Multicast variant: the box lands at the same shared-memory offset in every CTA of `mask` and completes the same-offset
// mbarrier in each of them.
__device__ __forceinline__ void tma_load_3d_mc(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                               uint16_t mask) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%4, %5, %6}], "
        "[%2], %3;" ::"r"(smem_u32(dst)),
        "l"(map), "r"(smem_u32(bar)), "h"(mask), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                     smem_u32(bar)),
                 "h"(mask)
                 : "memory");
}
// One lane of a converged warp (elect.sync).  The MMA warp runs its loop with all 32 lanes converged and lets the elected
// lane issue: inside an `if (lane == 0)` region the compiler keeps the shared-memory descriptors in vector registers and
// wraps every tcgen05.mma in an ELECT / 4 x R2UR.BROADCAST / BRA.U.ANY waterfall (~17 instructions per MMA); with
// warp-uniform control flow they live in uniform registers and the instruction takes them directly.
__device__ __forceinline__ bool elect_one_sync() {
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols));
}
__device__ __forceinline__ void umma_i8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate));
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// Shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address >> 4 in [0,14), leading byte
// offset >> 4 in [16,30), stride byte offset >> 4 in [32,46), version = 1 in [46,48), layout type in [61,64)
// (2 = SWIZZLE_128B, 4 = SWIZZLE_64B).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)(layout & 7) << 61;
    return d;
}

// Instruction descriptor (cute::UMMA::InstrDescriptor) for kind::i8: c_format = S32 (2) at [4,6), a/b format =
// INT8 (1) at [7,10)/[10,13), a/b major at 15/16 (0 = K, 1 = MN), N >> 3 at [17,23), M >> 4 at [24,29).
__host__ __device__ constexpr uint32_t make_idesc_i8(int M, int N, int a_mn, int b_mn) {
    return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(N >> 3) << 17) |
           ((uint32_t)(M >> 4) << 24);
}

struct GemmParams {
    double* C;                   // fp64 output, row-major [rows][ldc] (+ z * c_split_stride)
    long long ldc;
    long long c_split_stride;
    const double* row_scale;     // optional per-output-row factor (2^(Ex + Ey_j) for D)
    const double* col_scale;     // optional per-output-col factor (2^(Ex + Ea_j) for Y)
    int rows, cols;              // valid output extent
    int k_total;                 // contraction length
    int k_chunk;                 // contraction range per blockIdx.z (multiple of kBK)
    double inv_radix;            // 1 / R: group g carries weight R^-(g+2)
    int n_tiles;                 // number of real N tiles of the product
    int n_groups, m_tiles, k_splits;  // work units of THIS launch: n_groups clusters' worth of N tiles x M tiles x K splits
    int n_tile0;                 // first N tile of this launch (a product may be split into launches of different cluster size)
    int m_tile0;                 // first M tile of this launch (the Gram product runs whole waves of full-K tiles, then a split tail)
    int bn;                      // width of EVERY N tile (multiple of 8, 16 <= bn <= bn_max(S)): the factors are split into
                                 // equal tiles (m = 100, S = 6 -> 56 + 56, not 64 + 48) so the CTAs that share an X~ tile by
                                 // multicast -- and therefore run in lock-step -- carry the same work
    int trans_out;               // 1: store C[col][row] (the second contraction writes (X~^T Y)^T factor-major)
    int debug;                   // experiments only (LCX_OZ_DEBUG): bit 0 skip the MMAs, bit 1 skip the M-side loads, bit 2 skip the
                                 // N-side loads -- results are garbage, timings isolate the operand feed from the tensor work
    const double* c_add;         // optional (with trans_out, no split): C = c_add + product, c_add laid out like C (may be C
                                 // itself: grad = G0 + H W, linearcorex.py:300; Qij = rinv + (ry - I) rinv, :266)
    // Two-level split (short contractions, e.g. 12 500 samples per rank): the uniform units fill whole rounds of the resident
    // clusters; the units that would start a mostly idle last round -- K chunk k_splits - 1 of the last tail_m_tiles M tiles --
    // are left out of the uniform walk (main_units of them remain) and run instead as tail_units finer units: that K chunk cut
    // tail_splits ways, partials in their own compact buffer (folded into the uniform layout by tail_fold_kernel).
    int main_units;              // 0: every uniform unit; else the uniform walk stops here
    int tail_units;              // n_groups * tail_m_tiles * tail_splits
    int tail_m_tile0, tail_m_tiles;
    int tail_kbase, tail_kchunk; // K range of tail split z: [tail_kbase + z * tail_kchunk, + tail_kchunk) clipped to k_total
    double* tail_C;              // indexed with ABSOLUTE rows / cols like C (+ z * tail_split_stride)
    long long tail_ldc, tail_split_stride;
};

// The N-side (factor) operand is always K-major: B tile = [64 rows][64 B of K] (SW64), tensor map (K, rows, slice),
// TMA coordinates (k0, n0, s).  The M-side operand is
// KMAJOR = true : A tile = [128 rows][64 B of K]   (SW64),  tensor map (K, rows, slice),      coordinates (k0, m0, s);
// KMAJOR = false: A tile = [64 K rows][128 B of M] (SW128), tensor map (M, K rows, slice),    coordinates (m0, k0, s).
// All MMAs of one 64-deep K block for a tile of compile-time width BN (multiple of 16, <= bn_max(S)).
// BN % 16 == 8 (equal-width tiles such as 56): N = BN c is a legal UMMA N only for even c.  An odd count is legal as N = BN c + 8
// in the instruction that closes a row of A: its last plane lands in the LAST group (g = S - 1), so the 8 extra columns fall
// into unused TMEM above the accumulators, and the 8 extra B rows it reads are whatever follows that plane in the stage.  A row
// therefore opens with the smallest even count that lets one instruction close it: bn = 56 issues 5 planes as 2 + 3 (N = 112,
// 176) and 3 planes as one N = 176, not 4 + 1 and 2 + 1 -- an N = 64 instruction occupies the tensor pipe for ~55 cycles while
// doing 28 cycles of work (profiles/r02_mma_mix_probe.txt), and S = 6 now needs 8 instructions per K step instead of 9.
template <int S, bool KMAJOR, int BN>
__device__ __forceinline__ void issue_kblock(uint32_t sa, uint32_t sb, uint32_t tmem_base, bool first_block) {
    constexpr int A_BYTES = kBM * kBK;
    constexpr int B_BYTES = BN * kBK;        // digit planes of B are packed at the tile's own width
    constexpr bool ODD8 = (BN % 16) != 0;
    constexpr int CMAX = ODD8 ? ((256 / BN) & ~1) : (256 / BN);  // digit planes of B per instruction (N <= 256)
    constexpr int CLAST = ODD8 ? (248 / BN) : CMAX;                // ... per row-closing instruction (N = BN c + 8 <= 256)
    static_assert(BN % 8 == 0 && BN >= 16 && CMAX >= 1 && CLAST >= 1, "tile width");
#pragma unroll
    for (int kk = 0; kk < kBK / 32; ++kk) {
#pragma unroll
        for (int ka = 0; ka < S; ++ka) {
            constexpr int kMaxInstr = S;     // upper bound on instructions per (kk, ka); the loop below exits on q0
            int q0 = 0;
#pragma unroll
            for (int it = 0; it < kMaxInstr; ++it) {
                const int left = S - ka - q0;
                if (left <= 0) break;
                int cnt;
                if (left <= CLAST) cnt = left;                       // closes the row
                else if (ODD8) cnt = min(CMAX, max(2, (left - CLAST + 1) & ~1));
                else cnt = CMAX;
                const int n = BN * cnt + ((ODD8 && (cnt & 1)) ? 8 : 0);  // (odd: spills 8 columns above group S - 1)
                const uint32_t idesc = make_idesc_i8(kBM, n, KMAJOR ? 0 : 1, 0);
                // K-major: rows at 64 B pitch, 8-row swizzle atoms of 512 B (SBO); a K step is +32 B inside the span; the
                // next B plane starts BN/8 atoms further, i.e. N simply continues.
                // MN-major A: K rows of 128 B (SW128, atoms of 8 rows = 1 KB); a K step is 32 rows = 4 KB.
                const uint64_t da = KMAJOR ? make_smem_desc(sa + ka * A_BYTES + kk * 32, 16, 512, 4)
                                           : make_smem_desc(sa + ka * A_BYTES + kk * 4096, 8192, 1024, 2);
                const uint64_t db = make_smem_desc(sb + q0 * B_BYTES + kk * 32, 16, 512, 4);
                const uint32_t acc = (!first_block || kk > 0 || ka > 0) ? 1u : 0u;
                umma_i8(tmem_base + (uint32_t)((ka + q0) * BN), da, db, idesc, acc);
                q0 += cnt;
            }
        }
    }
}

// CL = thread-block cluster size along the N tiles (1, 2 or 3).  The CL CTAs of a cluster share the M-side operand
// (the X~ planes, in both contractions): each CTA fetches S/CL of its digit planes and TMA
// multicasts them into every CTA of the cluster, which divides the L2 -> SM traffic of that operand by CL (the kernel
// ran at the L2 throughput cap without it: 18 GB per launch at config 3).  A stage is released to the producers only
// when every CTA of the cluster has finished reading it (multicast tcgen05.commit on all empty barriers).
// CADD: the epilogue adds p.c_add (transposed stores only).  Its values are fetched one 16-column chunk ahead -- the first
// chunk while the MMAs are still running -- so the global-load latency is not paid once per column by a single resident CTA.
//
// PERSISTENT: the grid is one cluster per CL SMs and every cluster walks the work units u = cluster, cluster + #clusters, ...
// of the launch (unit = one M tile x one K split x CL adjacent N tiles).  Barriers, tensor-map prefetch, the TMEM allocation
// and the cluster handshake are paid once per SM instead of once per tile, and the mbarrier ring simply keeps running across
// units: while warps 2-5 drain the accumulators of unit i, warp 0 is already filling the stages of unit i + 1 (the K loop
// is bound by shared-memory traffic -- operand fetch of the MMAs plus the TMA fill -- not by the tensor pipe, so what has
// to overlap with the drain is the fill).  The MMA warp waits for the drain (tmem_empty) before it touches TMEM again.
template <int S, bool KMAJOR, int CL, bool CADD = false>
__global__ void __launch_bounds__(kThreads, 1)
oz_gemm_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const GemmParams p) {
    constexpr int kBN = bn_max(S);
    constexpr int kStages = stages_for(S);
    constexpr int A_BYTES = kBM * kBK;          // 8 KB per slice either way
    constexpr int B_BYTES = kBN * kBK;          // 4 KB (8 KB) per slice (full-width tile)
    constexpr int STAGE_BYTES = S * (A_BYTES + B_BYTES);
    constexpr uint32_t TMEM_COLS = (S * kBN + 8 <= 128) ? 128 : (S * kBN + 8 <= 256 ? 256 : 512);  // (+ 8 spill columns)
    static_assert(S * kBN <= 512, "accumulators exceed TMEM");
    static_assert(kStages >= 2, "pipeline needs two stages");

    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    __shared__ __align__(8) uint64_t full_bar[kStages];
    __shared__ __align__(8) uint64_t empty_bar[kStages];
    __shared__ __align__(8) uint64_t tmem_full_bar;
    __shared__ __align__(8) uint64_t tmem_empty_bar;
    __shared__ uint32_t tmem_base_smem;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t crank = (CL > 1) ? cluster_ctarank() : 0u;
    constexpr uint16_t kMask = (uint16_t)((1u << CL) - 1u);
    // every N tile has the same width bn <= kBN (the factors are split evenly); digit planes of B are packed at bn * 64 bytes
    const int bn = p.bn;
    const int b_bytes = bn * kBK;
    // work units of this launch: u -> (N group, M tile, K split), N groups fastest
    const int cluster_id = (int)blockIdx.x / CL, n_clusters = (int)gridDim.x / CL;
    const int units_main = p.main_units > 0 ? p.main_units : p.n_groups * p.m_tiles * p.k_splits;
    const int units = units_main + p.tail_units;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&mapA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&mapB) : "memory");
        for (int i = 0; i < kStages; ++i) {
            mbar_init(&full_bar[i], 1);
            mbar_init(&empty_bar[i], CL);  // one arrival per CTA of the cluster (multicast commit)
        }
        mbar_init(&tmem_full_bar, 1);
        mbar_init(&tmem_empty_bar, 4);     // one arrival per epilogue warp
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(&tmem_base_smem, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    if (CL > 1) cluster_sync_all();  // peers may multicast into / arrive on this CTA's barriers only once they exist
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_smem;

    // decode of unit u for this CTA (its own N tile of the cluster's group)
    // (z < 0 encodes tail split -1 - z)
    auto unit_of = [&](int u, int& n_tile, int& m_tile, int& z, int& kbeg, int& num_kb) {
        int kend;
        if (u < units_main) {
            const int g = u % p.n_groups;
            const int r = u / p.n_groups;
            m_tile = p.m_tile0 + r % p.m_tiles;
            z = r / p.m_tiles;
            n_tile = p.n_tile0 + g * CL + (int)crank;
            kbeg = z * p.k_chunk;
            kend = min(p.k_total, kbeg + p.k_chunk);
        } else {
            const int v = u - units_main;
            const int g = v % p.n_groups;
            const int r = v / p.n_groups;
            m_tile = p.tail_m_tile0 + r % p.tail_m_tiles;
            const int zt = r / p.tail_m_tiles;
            z = -1 - zt;
            n_tile = p.n_tile0 + g * CL + (int)crank;
            kbeg = p.tail_kbase + zt * p.tail_kchunk;
            kend = min(p.k_total, kbeg + p.tail_kchunk);
        }
        num_kb = (kend > kbeg) ? (kend - kbeg + kBK - 1) / kBK : 0;
    };

    if (warp == 0) {
        // ===== TMA producer: the warp walks the loop converged, one elected lane issues (see elect_one_sync) =====
        {
            uint32_t kbg = 0;  // K blocks issued so far by this CTA: stage and phase of the ring
            for (int u = cluster_id; u < units; u += n_clusters) {
                int n_tile, m_tile, z, kbeg, num_kb;
                unit_of(u, n_tile, m_tile, z, kbeg, num_kb);
                for (int kb = 0; kb < num_kb; ++kb, ++kbg) {
                    const uint32_t st = kbg % kStages;
                    const uint32_t ph = (kbg / kStages) & 1;
                    mbar_wait(&empty_bar[st], ph ^ 1);
                    uint8_t* sa = smem + st * STAGE_BYTES;
                    uint8_t* sb = sa + S * A_BYTES;
                    const bool load_a = !(p.debug & 2), load_b = !(p.debug & 4);
                    const int k0 = kbeg + kb * kBK;
                    if (elect_one_sync()) {
                        mbar_expect_tx(&full_bar[st], S * ((load_a ? A_BYTES : 0) + (load_b ? b_bytes : 0)));
#pragma unroll
                        for (int s = 0; s < S; ++s) {
                            // shared operand: plane s is fetched by cluster rank s % CL and multicast to all CL CTAs
                            if (!load_a) {
                            } else if (CL == 1) {
                                if (KMAJOR) tma_load_3d(sa + s * A_BYTES, &mapA, &full_bar[st], k0, m_tile * kBM, s);
                                else tma_load_3d(sa + s * A_BYTES, &mapA, &full_bar[st], m_tile * kBM, k0, s);
                            } else if ((uint32_t)(s % CL) == crank) {
                                if (KMAJOR) tma_load_3d_mc(sa + s * A_BYTES, &mapA, &full_bar[st], k0, m_tile * kBM, s, kMask);
                                else tma_load_3d_mc(sa + s * A_BYTES, &mapA, &full_bar[st], m_tile * kBM, k0, s, kMask);
                            }
                            if (load_b) tma_load_3d(sb + s * b_bytes, &mapB, &full_bar[st], k0, n_tile * bn, s);
                        }
                    }
                    __syncwarp();
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: the warp walks the loop converged, one elected lane issues =====
        {
            // Digit ka of A meets digits 0..S-1-ka of B, landing in groups ka..S-1 = CONSECUTIVE TMEM columns, and
            // the B digit planes are consecutive in shared memory, so those S-ka products are issued as one wide
            // MMA (N = bn (S-ka), at most 256 per instruction): A is re-read from shared memory 8 times per K step
            // instead of 21 -- an N = 64 instruction occupies the tensor pipe for ~55 cycles while doing 32 cycles of work.
            // The issue sequence is fully unrolled per tile width.
            uint32_t kbg = 0, it = 0;  // it = units with a non-empty K range so far (phase of the two TMEM barriers)
            for (int u = cluster_id; u < units; u += n_clusters) {
                int n_tile, m_tile, z, kbeg, num_kb;
                unit_of(u, n_tile, m_tile, z, kbeg, num_kb);
                if (num_kb == 0) continue;  // (the epilogue stores zeros without consulting TMEM)
                if (it > 0) {               // the epilogue warps have drained the accumulators of the previous unit
                    mbar_wait(&tmem_empty_bar, (it - 1) & 1);
                    tc_fence_after();
                }
                ++it;
                for (int kb = 0; kb < num_kb; ++kb, ++kbg) {
                    const uint32_t st = kbg % kStages;
                    const uint32_t ph = (kbg / kStages) & 1;
                    mbar_wait(&full_bar[st], ph);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + st * STAGE_BYTES);
                    const uint32_t sb = sa + S * A_BYTES;
                    if (elect_one_sync()) {
                    bool wide = (p.debug & 1) != 0;   // (debug: no MMAs at all)
                    if constexpr (kBN > 64) {
                        wide = wide || bn > 64;
                        if (p.debug & 1) {
                        } else if (bn == 128) issue_kblock<S, KMAJOR, 128>(sa, sb, tmem_base, kb == 0);
                        else if (bn == 112) issue_kblock<S, KMAJOR, 112>(sa, sb, tmem_base, kb == 0);
                        else if (bn == 96) issue_kblock<S, KMAJOR, 96>(sa, sb, tmem_base, kb == 0);
                        else if (bn == 80) issue_kblock<S, KMAJOR, 80>(sa, sb, tmem_base, kb == 0);
                    }
                    if (wide) {
                    } else if (bn == 64) issue_kblock<S, KMAJOR, 64>(sa, sb, tmem_base, kb == 0);
                    else if (bn == 56) issue_kblock<S, KMAJOR, 56>(sa, sb, tmem_base, kb == 0);
                    else if (bn == 48) issue_kblock<S, KMAJOR, 48>(sa, sb, tmem_base, kb == 0);
                    else if (bn == 40) issue_kblock<S, KMAJOR, 40>(sa, sb, tmem_base, kb == 0);
                    else if (bn == 32) issue_kblock<S, KMAJOR, 32>(sa, sb, tmem_base, kb == 0);
                    else if (bn == 24) issue_kblock<S, KMAJOR, 24>(sa, sb, tmem_base, kb == 0);
                    else issue_kblock<S, KMAJOR, 16>(sa, sb, tmem_base, kb == 0);
                    // frees the stage (in every CTA of the cluster) once these MMAs have read it
                    if (CL == 1) umma_commit(&empty_bar[st]);
                    else umma_commit_mc(&empty_bar[st], kMask);
                    }
                    __syncwarp();
                }
                if (elect_one_sync()) umma_commit(&tmem_full_bar);
                __syncwarp();
            }
        }
    } else {
        // ===== epilogue: TMEM -> registers -> fp64 recombination -> global =====
        const int quarter = warp & 3;              // TMEM lane quarter this warp may read
        const int row_in_tile = quarter * 32 + lane;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(quarter * 32) << 16);
        uint32_t it = 0;  // units with a non-empty K range so far
        for (int u = cluster_id; u < units; u += n_clusters) {
            int n_tile, m_tile, z, kbeg, num_kb;
            unit_of(u, n_tile, m_tile, z, kbeg, num_kb);
            const int row = m_tile * kBM + row_in_tile;
            double cadd[16];
            auto fetch_cadd = [&](int c0) {
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const int col = n_tile * bn + c0 + j;
                    cadd[j] = (row < p.rows && col < p.cols && c0 + j < bn) ? p.c_add[(long long)col * p.ldc + row] : 0.0;
                }
            };
            if (CADD) fetch_cadd(0);
            if (num_kb > 0) {
                mbar_wait(&tmem_full_bar, it & 1);
                tc_fence_after();
                ++it;
            }
            double* C = z >= 0 ? p.C + (long long)z * p.c_split_stride : p.tail_C + (long long)(-1 - z) * p.tail_split_stride;
            const long long ldc = z >= 0 ? p.ldc : p.tail_ldc;
            const double rs = (p.row_scale != nullptr && row < p.rows) ? p.row_scale[row] : 1.0;
#pragma unroll 1
            for (int c0 = 0; c0 < bn; c0 += 16) {
                double acc[16];
                double cur[16];
                if (CADD) {  // this chunk's addends are in registers; request the next chunk's before touching TMEM
#pragma unroll
                    for (int j = 0; j < 16; ++j) cur[j] = cadd[j];
                    if (c0 + 16 < bn) fetch_cadd(c0 + 16);
                }
                if (num_kb > 0) {
                    // all S group loads of this chunk in flight before the one wait (a wait per load serialised S TMEM round trips)
                    uint32_t r[S][16];
#pragma unroll
                    for (int g = 0; g < S; ++g) tmem_ld16(lane_addr + (uint32_t)(g * bn + c0), r[g]);
                    tmem_ld_wait();
                    if (c0 + 16 >= bn) {  // last chunk read: hand TMEM back to the MMA warp before the arithmetic and the stores
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&tmem_empty_bar);
                    }
#pragma unroll
                    for (int j = 0; j < 16; ++j) acc[j] = (double)(int)r[S - 1][j];
#pragma unroll
                    for (int g = S - 2; g >= 0; --g) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) acc[j] = acc[j] * p.inv_radix + (double)(int)r[g][j];  // 1/R per group
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 16; ++j) acc[j] = 0.0;
                }
                if (row < p.rows) {
                    const int col0 = n_tile * bn + c0;
                    // columns of this tile that are real outputs (a width of 8 mod 16 ends in the middle of the last chunk)
                    const int cend = min(p.cols, n_tile * bn + bn);
#pragma unroll
                    for (int j = 0; j < 16; j += 2) {
                        const int col = col0 + j;
                        // group g = 0 carries weight R^-2 (digits k = l = 1)
                        double v0 = acc[j] * (p.inv_radix * p.inv_radix) * rs, v1 = acc[j + 1] * (p.inv_radix * p.inv_radix) * rs;
                        if (p.col_scale != nullptr) {
                            if (col < cend) v0 *= p.col_scale[col];
                            if (col + 1 < cend) v1 *= p.col_scale[col + 1];
                        }
                        if (p.trans_out) {  // a warp's 32 rows are 32 consecutive doubles of one output row: coalesced
                            if (CADD) {
                                v0 += cur[j];
                                v1 += cur[j + 1];
                            }
                            if (col < cend) C[(long long)col * ldc + row] = v0;
                            if (col + 1 < cend) C[(long long)(col + 1) * ldc + row] = v1;
                        } else if (col + 1 < cend) {
                            *reinterpret_cast<double2*>(C + (long long)row * ldc + col) = make_double2(v0, v1);
                        } else if (col < cend) {
                            C[(long long)row * ldc + col] = v0;
                        }
                    }
                }
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    if (CL > 1) cluster_sync_all();  // nobody leaves while a peer can still multicast into it or arrive on its barriers
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

// ---- digit extraction -----------------------------------------------------------------------------
// v = x * 2^-E in (-0.5, 0.5);  repeat: t = R v, d = rint(t), v = t - d.  |t| <= R/2, so |d| <= 64 for R = 128 (every step
// exact in binary64) and |d| <= 127 for R = 254 (t = 254 v rounds at the 2^-53 level -- far below the last digit kept).
template <int S>
__device__ __forceinline__ void split_digits(double x, double inv_scale, double radix, int8_t (&d)[S]) {
    double v = x * inv_scale;
#pragma unroll
    for (int k = 0; k < S; ++k) {
        const double t = __dmul_rn(v, radix);  // no FMA contraction with the subtraction below: digits are then exactly
                                               // what the same three binary64 operations give anywhere (numpy in the tests)
        const double r = rint(t);
        d[k] = (int8_t)(int)r;
        v = __dsub_rn(t, r);
    }
}

// Power-of-two scale 2^E with max * 2^-E < 0.5 (so the first digit stays within [-64, 64]).
__device__ __forceinline__ double pow2_above(double amax) {
    if (!(amax <= 1.7976931348623157e308)) return __longlong_as_double(0x7ff8000000000000LL);  // non-finite data: NaN out
    if (!(amax > 0.0)) return 1.0;
    int e;
    frexp(amax, &e);       // amax = f * 2^e, f in [0.5, 1)
    return ldexp(1.0, e + 1);
}

// Slices of a row-major fp64 matrix [rows][ld_in] into out[s][rows][ld_out] (int8), one scale per row
// (row_scale != nullptr: value 2^E_row) or a single scale.  Columns in [cols, ld_out) are zero-filled.
// ZERO_DIAG: the diagonal entry of each row is taken as 0 (the unit diagonal of ry is added back exactly by the consumer).
template <int S, bool ZERO_DIAG = false>
__global__ void slice_rows_kernel(const double* __restrict__ in, long long ld_in, int rows, int cols,
                                  const double* __restrict__ row_scale, const double* __restrict__ one_scale,
                                  int8_t* __restrict__ out, long long ld_out, long long slice_stride, double radix) {
    const long long r = blockIdx.x;  // rows on grid.x (up to 2^31 - 1), column blocks on grid.y
    const int c4 = (blockIdx.y * blockDim.x + threadIdx.x) * 4;
    if (r >= rows || c4 >= ld_out) return;
    const double inv = 1.0 / (row_scale ? row_scale[r] : one_scale[0]);
    int8_t d[4][S];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int c = c4 + j;
        const double x = (c < cols && !(ZERO_DIAG && c == r)) ? in[r * ld_in + c] : 0.0;
        split_digits<S>(x, inv, radix, d[j]);
    }
#pragma unroll
    for (int k = 0; k < S; ++k) {
        char4 v = make_char4(d[0][k], d[1][k], d[2][k], d[3][k]);
        *reinterpret_cast<char4*>(out + (long long)k * slice_stride + r * ld_out + c4) = v;
    }
}

// Digit planes of Y (N x ldy, row-major fp64) with one scale per column (exponent per factor), written TRANSPOSED:
// out[s][c][r], samples contiguous -- the K-major factor-side operand of the second contraction.  One CTA of 32 x 8
// threads turns a 128-row x 32-column block of Y around through shared memory (coalesced 256 B reads of Y, 128 B
// writes per digit plane and factor).
template <int S>
__global__ void __launch_bounds__(256) slice_cols_t_kernel(const double* __restrict__ in, long long ld_in, long long rows,
                                                           int cols, const double* __restrict__ col_scale,
                                                           int8_t* __restrict__ out, long long ld_out, long long slice_stride,
                                                           double radix) {
    constexpr int PITCH = 132;  // 33 words: the 32 columns of one row land in different banks
    __shared__ __align__(4) int8_t t[S][32][PITCH];
    const int tx = threadIdx.x, ty = threadIdx.y;
    const long long r0 = (long long)blockIdx.x * 128;
    const int c0 = blockIdx.y * 32;
    const int c = c0 + tx;
    const double inv = (c < cols) ? 1.0 / col_scale[c] : 1.0;
#pragma unroll 4
    for (int i = 0; i < 16; ++i) {
        const int rr = ty + 8 * i;
        const long long r = r0 + rr;
        const double x = (c < cols && r < rows) ? in[r * ld_in + c] : 0.0;
        int8_t d[S];
        split_digits<S>(x, inv, radix, d);
#pragma unroll
        for (int k = 0; k < S; ++k) t[k][tx][rr] = d[k];
    }
    __syncthreads();
    const int tid = ty * 32 + tx;
    const int w = tid & 31;        // 4-byte word of the 128-byte row
    if (r0 + 4 * w >= ld_out) return;
    for (int idx = tid >> 5; idx < S * 32; idx += 8) {
        const int k = idx >> 5, cc = idx & 31;
        if (c0 + cc < cols)
            *reinterpret_cast<uint32_t*>(out + (long long)k * slice_stride + (long long)(c0 + cc) * ld_out + r0 + 4 * w) =
                *reinterpret_cast<const uint32_t*>(&t[k][cc][4 * w]);
    }
}

// max |a[r][c]| over a row (one CTA of 256 threads per row) -> scale[r] = 2^E;  used for A (W or grad).
// skip_diag: leave a[r][r] out of the maximum (square matrices sliced with ZERO_DIAG).
// x_scale / out_scale (optional): out_scale[r] = x_scale[0] * scale[r], the output scale of Y = X~ A^T.
// dot_b / dot_out (optional): dot_out[r] = sum_c a[r][c] * dot_b[r][c] in the same pass (Bj of the search direction,
// linearcorex.py:302, rides on the pass that finds the exponent of grad's row).
__global__ void row_scale_kernel(const double* __restrict__ a, long long ld, int cols, double* __restrict__ scale,
                                 int skip_diag = 0, const double* __restrict__ x_scale = nullptr,
                                 double* __restrict__ out_scale = nullptr, const double* __restrict__ dot_b = nullptr,
                                 double* __restrict__ dot_out = nullptr) {
    __shared__ double scratch[8];
    const double* ra = a + (long long)blockIdx.x * ld;
    const double* rb = dot_b ? dot_b + (long long)blockIdx.x * ld : nullptr;
    double mx = 0.0, dot = 0.0;
    if (skip_diag || ((uintptr_t)ra & 15) != 0 || (rb != nullptr && ((uintptr_t)rb & 15) != 0)) {
        for (int i = threadIdx.x; i < cols; i += 256) {
            const double v = ra[i];
            if (!(skip_diag && i == (int)blockIdx.x)) mx = lcx::amax_acc(mx, v);
            if (rb) dot += v * rb[i];
        }
    } else {  // 16-byte loads, eight values in flight per thread (a row of W is 400 KB at n = 50 000)
        const double2* ra2 = reinterpret_cast<const double2*>(ra);
        const double2* rb2 = reinterpret_cast<const double2*>(rb);
        const int pairs = cols >> 1;
        double m1 = 0.0, m2 = 0.0, m3 = 0.0, d1 = 0.0, d2 = 0.0, d3 = 0.0;
        int i = threadIdx.x;
        for (; i + 768 < pairs; i += 1024) {
            const double2 v0 = ra2[i], v1 = ra2[i + 256], v2 = ra2[i + 512], v3 = ra2[i + 768];
            mx = lcx::amax_acc(lcx::amax_acc(mx, v0.x), v0.y);
            m1 = lcx::amax_acc(lcx::amax_acc(m1, v1.x), v1.y);
            m2 = lcx::amax_acc(lcx::amax_acc(m2, v2.x), v2.y);
            m3 = lcx::amax_acc(lcx::amax_acc(m3, v3.x), v3.y);
            if (rb2) {
                const double2 b0 = rb2[i], b1 = rb2[i + 256], b2 = rb2[i + 512], b3 = rb2[i + 768];
                dot += v0.x * b0.x + v0.y * b0.y;
                d1 += v1.x * b1.x + v1.y * b1.y;
                d2 += v2.x * b2.x + v2.y * b2.y;
                d3 += v3.x * b3.x + v3.y * b3.y;
            }
        }
        for (; i < pairs; i += 256) {
            const double2 v = ra2[i];
            mx = lcx::amax_acc(lcx::amax_acc(mx, v.x), v.y);
            if (rb2) {
                const double2 b = rb2[i];
                dot += v.x * b.x + v.y * b.y;
            }
        }
        if ((cols & 1) && threadIdx.x == 0) {
            mx = lcx::amax_acc(mx, ra[cols - 1]);
            if (rb) dot += ra[cols - 1] * rb[cols - 1];
        }
        mx = fmax(fmax(mx, m1), fmax(m2, m3));
        dot = (dot + d1) + (d2 + d3);
    }
    mx = block_max_256(mx, scratch);
    if (rb) dot = block_sum_256(dot, scratch);
    if (threadIdx.x == 0) {
        const double sc = pow2_above(mx);
        scale[blockIdx.x] = sc;
        if (out_scale != nullptr) out_scale[blockIdx.x] = x_scale[0] * sc;
        if (rb) dot_out[blockIdx.x] = dot;
    }
}

// ---- per-COLUMN scales (the m x m x n products on the int8 engine: an operand contracted over its rows needs an
// exponent that is constant along the contraction, i.e. one per column) ----
// part[slab][c] = max |a[r][c]| over the rows of one slab (columns across threads: coalesced; four loads in flight)
__global__ void __launch_bounds__(256) col_absmax_partial_kernel(const double* __restrict__ a, long long ld, int rows, int cols,
                                                                 int rows_per_slab, double* __restrict__ part, long long ldp) {
    // two columns per thread (16-byte loads; ld is a multiple of 16 so the pair never leaves the row), four rows in flight
    const int c = (blockIdx.x * 256 + threadIdx.x) * 2;
    if (c >= cols) return;
    const int r0 = blockIdx.y * rows_per_slab;
    const int r1 = min(rows, r0 + rows_per_slab);
    double x0 = 0.0, x1 = 0.0, x2 = 0.0, x3 = 0.0, y0 = 0.0, y1 = 0.0, y2 = 0.0, y3 = 0.0;
    int r = r0;
    for (; r + 3 < r1; r += 4) {
        const double2 v0 = *reinterpret_cast<const double2*>(a + (long long)r * ld + c);
        const double2 v1 = *reinterpret_cast<const double2*>(a + (long long)(r + 1) * ld + c);
        const double2 v2 = *reinterpret_cast<const double2*>(a + (long long)(r + 2) * ld + c);
        const double2 v3 = *reinterpret_cast<const double2*>(a + (long long)(r + 3) * ld + c);
        x0 = lcx::amax_acc(x0, v0.x); y0 = lcx::amax_acc(y0, v0.y);
        x1 = lcx::amax_acc(x1, v1.x); y1 = lcx::amax_acc(y1, v1.y);
        x2 = lcx::amax_acc(x2, v2.x); y2 = lcx::amax_acc(y2, v2.y);
        x3 = lcx::amax_acc(x3, v3.x); y3 = lcx::amax_acc(y3, v3.y);
    }
    for (; r < r1; ++r) {
        const double2 v = *reinterpret_cast<const double2*>(a + (long long)r * ld + c);
        x0 = lcx::amax_acc(x0, v.x); y0 = lcx::amax_acc(y0, v.y);
    }
    part[(long long)blockIdx.y * ldp + c] = fmax(fmax(x0, x1), fmax(x2, x3));
    if (c + 1 < cols) part[(long long)blockIdx.y * ldp + c + 1] = fmax(fmax(y0, y1), fmax(y2, y3));
}
// scale[c] = 2^E above the column maximum
__global__ void col_scale_finish_kernel(const double* __restrict__ part, int slabs, long long ldp, int cols,
                                        double* __restrict__ scale) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cols) return;
    double mx = 0.0;
    for (int s = 0; s < slabs; ++s) mx = fmax(mx, part[(long long)s * ldp + c]);
    scale[c] = pow2_above(mx);
}
// slice_rows_kernel with one scale per COLUMN: out[s][r][c] = digit s of in[r][c] / col_scale[c]
template <int S>
__global__ void slice_colscaled_kernel(const double* __restrict__ in, long long ld_in, int rows, int cols,
                                       const double* __restrict__ col_scale, int8_t* __restrict__ out, long long ld_out,
                                       long long slice_stride, double radix) {
    const long long r = blockIdx.x;
    const int c4 = (blockIdx.y * blockDim.x + threadIdx.x) * 4;
    if (r >= rows || c4 >= ld_out) return;
    int8_t d[4][S];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int c = c4 + j;
        const double x = (c < cols) ? in[r * ld_in + c] : 0.0;
        const double inv = (c < cols) ? 1.0 / col_scale[c] : 1.0;
        split_digits<S>(x, inv, radix, d[j]);
    }
#pragma unroll
    for (int k = 0; k < S; ++k) {
        char4 v = make_char4(d[0][k], d[1][k], d[2][k], d[3][k]);
        *reinterpret_cast<char4*>(out + (long long)k * slice_stride + r * ld_out + c4) = v;
    }
}

// Column statistics of Y (N x ldy): per-slab partial max|Y| and sum Y^2 -> part[slab][2][ldp]
__global__ void __launch_bounds__(256) y_stats_kernel(const double* __restrict__ y, long long ldy, long long rows, int cols,
                                                      int rows_per_slab, double* __restrict__ part, long long ldp) {
    __shared__ double rm[8][32], rs[8][32];
    const int c = blockIdx.x * 32 + threadIdx.x;
    const long long r0 = (long long)blockIdx.y * rows_per_slab;
    const long long r1 = min(rows, r0 + (long long)rows_per_slab);
    double mx = 0.0, sq = 0.0;
    if (c < cols) {
        for (long long r = r0 + threadIdx.y; r < r1; r += 8) {
            const double v = y[r * ldy + c];
            mx = lcx::amax_acc(mx, v);
            sq += v * v;
        }
    }
    rm[threadIdx.y][threadIdx.x] = mx;
    rs[threadIdx.y][threadIdx.x] = sq;
    __syncthreads();
    if (threadIdx.y == 0 && c < cols) {
        double a = 0.0, b = 0.0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            a = fmax(a, rm[k][threadIdx.x]);
            b += rs[k][threadIdx.x];
        }
        part[((long long)blockIdx.y * 2 + 0) * ldp + c] = a;
        part[((long long)blockIdx.y * 2 + 1) * ldp + c] = b;
    }
}

// Combine the slab partials: colsq[c] = sum, yscale[c] = 2^E from max; dscale[c] = x_scale * yscale[c]
__global__ void y_stats_finish_kernel(const double* __restrict__ part, int slabs, long long ldp, int cols,
                                      const double* __restrict__ x_scale, double* __restrict__ colsq,
                                      double* __restrict__ yscale, double* __restrict__ dscale) {
    // one CTA of 256 threads per column; fixed-order block reduction keeps the sum deterministic
    __shared__ double scratch[8];
    const int c = blockIdx.x;
    if (c >= cols) return;
    double mx = 0.0, sq = 0.0;
    for (int s = threadIdx.x; s < slabs; s += 256) {
        mx = fmax(mx, part[((long long)s * 2 + 0) * ldp + c]);
        sq += part[((long long)s * 2 + 1) * ldp + c];
    }
    mx = block_max_256(mx, scratch);
    sq = block_sum_256(sq, scratch);
    if (threadIdx.x == 0) {
        if (colsq) colsq[c] = sq;
        const double sc = pow2_above(mx);
        yscale[c] = sc;
        dscale[c] = x_scale[0] * sc;
    }
}

// dst[r][c] = sum_t src[t][r][c], t in index order (rows x cols; leading dimensions ld_src / ld_dst; split t at t * stride):
// folds the tail partials of the two-level split (GemmParams::tail_*) into the slot the uniform walk left unwritten.
__global__ void __launch_bounds__(256) tail_fold_kernel(const double* __restrict__ src, int splits, long long stride,
                                                        long long ld_src, double* __restrict__ dst, long long ld_dst, int rows,
                                                        int cols) {
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    if (i >= (long long)rows * cols) return;
    const int r = (int)(i / cols), c = (int)(i - (long long)r * cols);
    const double* p0 = src + (long long)r * ld_src + c;
    double acc = p0[0];
    int t = 1;
    for (; t + 3 < splits; t += 4) {  // four loads in flight, added in index order
        const double v0 = p0[(long long)t * stride], v1 = p0[(long long)(t + 1) * stride];
        const double v2 = p0[(long long)(t + 2) * stride], v3 = p0[(long long)(t + 3) * stride];
        acc += v0; acc += v1; acc += v2; acc += v3;
    }
    for (; t < splits; ++t) acc += p0[(long long)t * stride];
    dst[(long long)r * ld_dst + c] = acc;
}

// cscale[j] = x_scale * a_scale[j]   (output scale of Y = X~ A^T)
__global__ void mul_scale_kernel(const double* __restrict__ x_scale, const double* __restrict__ a_scale, double* __restrict__ out,
                                 int m) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < m) out[j] = x_scale[0] * a_scale[j];
}

// Global max |x| of the N x n block (per-CTA partial max, then one CTA finishes) -> scale[0] = 2^E
__global__ void __launch_bounds__(256) absmax_partial_kernel(const double* __restrict__ x, long long ld, long long rows, int cols,
                                                             double* __restrict__ part) {
    __shared__ double scratch[8];
    double mx = 0.0;
    for (long long r = blockIdx.x; r < rows; r += gridDim.x) {
        const double* xr = x + r * ld;
        for (int c = threadIdx.x; c < cols; c += 256) mx = lcx::amax_acc(mx, xr[c]);
    }
    mx = block_max_256(mx, scratch);
    if (threadIdx.x == 0) part[blockIdx.x] = mx;
}
__global__ void absmax_finish_kernel(const double* __restrict__ part, int nparts, double* __restrict__ scale) {
    __shared__ double scratch[8];
    double mx = 0.0;
    for (int i = threadIdx.x; i < nparts; i += 256) mx = fmax(mx, part[i]);
    mx = block_max_256(mx, scratch);
    if (threadIdx.x == 0) scale[0] = pow2_above(mx);
}

// ---- Gram route (N >= n: the fit depends on X~ only through X~^T X~ / N, linearcorex.py:196-213 builds the same products
// "without explicitly constructing the covariance matrix" because it targets n >> N) -------------------------------------
// Digit planes of a column block of X~, turned around: out[s][c][r] = in[s][r][c0 + c] for c < ncols -- the K-major
// factor-side operand (samples contiguous) of X~^T X~[:, block].  One CTA of 32 x 8 threads per 128 x 128 byte tile and
// plane (coalesced 128 B reads along the variables, 128 B writes along the samples).
__global__ void __launch_bounds__(256) transpose_planes_kernel(const int8_t* __restrict__ in, long long ld_in, long long rows,
                                                               long long in_slice_stride, int c0, int ncols,
                                                               int8_t* __restrict__ out, long long ld_out,
                                                               long long out_slice_stride) {
    constexpr int PITCH = 132;
    __shared__ __align__(4) int8_t t[128][PITCH];
    const int tx = threadIdx.x, ty = threadIdx.y;
    const long long r0 = (long long)blockIdx.x * 128;
    const int cb = blockIdx.y * 128;   // column offset inside the block
    const int8_t* src = in + (long long)blockIdx.z * in_slice_stride;
    int8_t* dst = out + (long long)blockIdx.z * out_slice_stride;
#pragma unroll 4
    for (int i = 0; i < 16; ++i) {
        const int rr = ty + 8 * i;
        const long long r = r0 + rr;
        uint32_t w = 0;
        if (r < rows && c0 + cb + 4 * tx < ld_in) w = *reinterpret_cast<const uint32_t*>(src + r * ld_in + c0 + cb + 4 * tx);
        t[4 * tx + 0][rr] = (int8_t)(w & 0xff);
        t[4 * tx + 1][rr] = (int8_t)((w >> 8) & 0xff);
        t[4 * tx + 2][rr] = (int8_t)((w >> 16) & 0xff);
        t[4 * tx + 3][rr] = (int8_t)((w >> 24) & 0xff);
    }
    __syncthreads();
    if (r0 + 4 * tx >= ld_out) return;
    for (int c = ty; c < 128; c += 8) {
        if (cb + c < ncols)
            *reinterpret_cast<uint32_t*>(dst + (long long)(cb + c) * ld_out + r0 + 4 * tx) =
                *reinterpret_cast<const uint32_t*>(&t[c][4 * tx]);
    }
}

// out[i] = x_scale^2 * factor  (output scale of X~^T X~ / N: both operands carry the exponent of X~)
__global__ void gram_scale_kernel(const double* __restrict__ x_scale, double factor, double* __restrict__ out, int count) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) out[i] = x_scale[0] * x_scale[0] * factor;
}

// g[i][j] = g[j][i] for i > j (the build fills row a from the start of a's column block to n: the upper triangle)
__global__ void __launch_bounds__(256) mirror_upper_kernel(double* __restrict__ g, long long ld, int n) {
    __shared__ double t[32][33];
    const int ti = blockIdx.y, tj = blockIdx.x;   // destination tile (rows ti, cols tj), ti >= tj
    if (ti < tj) return;
    const int tx = threadIdx.x, ty = threadIdx.y;
#pragma unroll
    for (int k = 0; k < 4; ++k) {   // source tile (rows tj, cols ti)
        const int r = tj * 32 + ty + 8 * k, c = ti * 32 + tx;
        t[ty + 8 * k][tx] = (r < n && c < n) ? g[(long long)r * ld + c] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int r = ti * 32 + ty + 8 * k, c = tj * 32 + tx;
        if (r < n && c < n && r > c) g[(long long)r * ld + c] = t[tx][ty + 8 * k];
    }
}

// ---- host side -----------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (fn == nullptr) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// 3-D uint8 tensor map over slices[s][rows][ld]: dims (inner = ld-extent `inner`, rows, s).
inline int make_slice_map(CUtensorMap* map, const void* base, long long inner, long long rows, int slices, long long ld,
                          long long slice_stride, int box_inner, int box_rows, bool swizzle128) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return fail(-2, "cuTensorMapEncodeTiled", "driver entry point unavailable");
    cuuint64_t dims[3] = {(cuuint64_t)inner, (cuuint64_t)rows, (cuuint64_t)slices};
    cuuint64_t strides[2] = {(cuuint64_t)ld, (cuuint64_t)slice_stride};
    cuuint32_t box[3] = {(cuuint32_t)box_inner, (cuuint32_t)box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult rc = fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (rc != CUDA_SUCCESS) return fail(-2, "cuTensorMapEncodeTiled", "encode failed (check alignment / strides)");
    return 0;
}

template <int S, bool KMAJOR, int CL, bool CADD = false>
inline int launch_oz_gemm_cl(const CUtensorMap& mapA, const CUtensorMap& mapB, GemmParams p, dim3 grid, cudaStream_t st) {
    constexpr int SMEM = stages_for(S) * S * (kBM * kBK + bn_max(S) * kBK) + 1024;
    static PerDeviceOnce configured = {};
    static int resident[64] = {};  // clusters of this kernel that fit on the device at once, per device ordinal
    auto kern = oz_gemm_kernel<S, KMAJOR, CL, CADD>;
    if (configured.first_time()) LCX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    // grid = (N tiles of THIS launch starting at p.n_tile0, M tiles, K splits); p.n_tiles = all N tiles of the product.
    // Padded N tiles (to a multiple of the cluster size) load zeros (TMA OOB fill) and store nothing.
    p.n_groups = (int)round_up(grid.x, CL) / CL;
    p.m_tiles = (int)grid.y;
    p.k_splits = (int)grid.z;
    const long long units = (p.main_units > 0 ? (long long)p.main_units : (long long)p.n_groups * p.m_tiles * p.k_splits) + p.tail_units;
    {
        static int dbg = -1;
        if (dbg < 0) {
            const char* env = getenv("LCX_OZ_DEBUG");
            dbg = env ? atoi(env) : 0;
        }
        p.debug = dbg;
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = SMEM;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int dev = 0;
    LCX_CUDA(cudaGetDevice(&dev));
    dev &= 63;
    if (resident[dev] == 0) {
        int n = 0, sms = 0;
        cfg.gridDim = dim3(CL * 1024);
        if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess || n <= 0) {
            cudaGetLastError();
            LCX_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
            n = sms / CL;
        }
        resident[dev] = n > 0 ? n : 1;
    }
    const long long clusters = units < resident[dev] ? units : resident[dev];
    LCX_REQUIRE(clusters * CL < (1LL << 31), "grid too large");
    cfg.gridDim = dim3((unsigned)(clusters * CL));
    LCX_CUDA(cudaLaunchKernelEx(&cfg, kern, mapA, mapB, p));
    return 0;
}

// Pairs of N tiles share the M-side operand through TMA multicast (clusters of 1 and of 4 measured slower: multicast does
// not lower the bytes delivered per SM, and clusters of 4 fit only 132 SMs).  A padded cluster slot would occupy an SM for the whole K loop and take a full copy
// of the X~ tile for nothing, so an odd tile count runs as pairs plus one final cluster of three (m = 192: 3 tiles in
// 5.9 ms instead of 7.0 ms), and a single tile as a cluster of one.
template <int S, bool KMAJOR, bool CADD = false>
inline int launch_oz_gemm(const CUtensorMap& mapA, const CUtensorMap& mapB, GemmParams p, dim3 grid, cudaStream_t st) {
    const int n_tiles = (int)grid.x;
    p.n_tiles = n_tiles;
    p.n_tile0 = 0;
    if (n_tiles >= 2) {
        if (n_tiles % 2 == 0) return launch_oz_gemm_cl<S, KMAJOR, 2, CADD>(mapA, mapB, p, grid, st);
        if (n_tiles > 3) {
            grid.x = (unsigned)(n_tiles - 3);
            const int rc = launch_oz_gemm_cl<S, KMAJOR, 2, CADD>(mapA, mapB, p, grid, st);
            if (rc != 0) return rc;
        }
        p.n_tile0 = n_tiles - 3;
        grid.x = 3;
        return launch_oz_gemm_cl<S, KMAJOR, 3, CADD>(mapA, mapB, p, grid, st);
    }
    return launch_oz_gemm_cl<S, KMAJOR, 1, CADD>(mapA, mapB, p, grid, st);
}

}  // namespace oz
}  // namespace lcx
