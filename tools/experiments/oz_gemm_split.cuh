// Record of a measured dead end (DESIGN.md 7), not compiled into the product: the split path of oz_gemm_kernel at S = 6.
// Group g collects the digit pairs with k + l = g.  The side launch accumulates groups 0-1 (3 of the 21 plane products) and
// stores them as int32; the main launch accumulates groups 2-5, whose four accumulators fit 128-wide tiles in TMEM, so one CTA
// owns a 128-row tile across all m <= 128 factors and the X~ tile reaches one SM instead of both SMs of a pair.  The main
// epilogue continues Horner's rule with the side sums, so every output is bit-identical to the pair path.  Measured at
// config 3 with tools/experiments/oz_split_probe.cu (profiles/r07_oz_split_probe_config3.txt): bit-identical, and slower --
// main + side 1.21 x the pair for the first contraction and 1.01 x for the second.  The kernel is oz_gemm_kernel
// (csrc/ozaki_i8.cuh) with a compile-time group window [G0, G1], as it stood before bn = 56 rows were issued as 8 MMAs per K
// step instead of 9 (issue_kblock_window keeps the 4 + 1 / 2 + 1 split of that time).
// Include after ozaki_i8.cuh.
#pragma once
#include "ozaki_i8.cuh"

namespace lcx {
namespace oz {

__host__ __device__ constexpr int stages_for_planes(int planes, int bn) {
    return (220 * 1024) / (planes * (kBM * kBK + bn * kBK)) >= 4 ? 4 : (220 * 1024) / (planes * (kBM * kBK + bn * kBK));
}
// Group window [G0, G1] of one launch (split path, S = 6 and m <= 128): the launch accumulates only the groups
// g = k + l in [G0, G1], so it needs digit planes 0..G1 of both operands and G1 - G0 + 1 accumulators, which fit 128-wide
// tiles whenever there are at most 4 of them.  The full window [0, S - 1] is the ordinary contraction.
__host__ __device__ constexpr int window_planes(int G1) { return G1 + 1; }
__host__ __device__ constexpr int window_bn(int G0, int G1) { return bn_max(G1 - G0 + 1); }
__host__ __device__ constexpr int window_stages(int G0, int G1) {
    return stages_for_planes(window_planes(G1), window_bn(G0, G1));
}
// Split path of S = 6: groups 0..1 (3 of the 21 plane products) in a side launch that stores them as int32, groups 2..5
// in the main launch, which adds the side sums in the same Horner order as the full window.
constexpr int kSplitS = 6, kSplitG = 2;

// All MMAs of one 64-deep K block for a tile of compile-time width BN (multiple of 16, <= bn_max(S)).
// BN % 16 == 8 (equal-width tiles such as 56): N = BN c is a legal UMMA N only for even c, so an odd plane count issues its
// last plane as one instruction of N = BN + 8.  That plane always lands in the LAST group (g = S - 1): the 8 extra columns
// fall into unused TMEM above the accumulators, and the 8 extra B rows it reads are whatever follows that plane in the stage.
//
// Window [G0, G1] (default: all S groups): digit ka of A meets digits max(0, G0 - ka) .. G1 - ka of B, and group g sits at
// TMEM column (g - G0) BN.  ka = 0 reaches every group of the window, so the first K step of ka = 0 still initialises all.
template <int S, bool KMAJOR, int BN, int G0 = 0, int G1 = S - 1>
__device__ __forceinline__ void issue_kblock_window(uint32_t sa, uint32_t sb, uint32_t tmem_base, bool first_block) {
    static_assert(0 <= G0 && G0 <= G1 && G1 <= S - 1, "group window");
    constexpr int A_BYTES = kBM * kBK;
    constexpr int B_BYTES = BN * kBK;        // digit planes of B are packed at the tile's own width
    constexpr bool ODD8 = (BN % 16) != 0;
    constexpr int CMAX = ODD8 ? ((256 / BN) & ~1) : (256 / BN);  // digit planes of B per instruction (N <= 256)
    static_assert(BN % 8 == 0 && BN >= 16 && CMAX >= 1, "tile width");
#pragma unroll
    for (int kk = 0; kk < kBK / 32; ++kk) {
#pragma unroll
        for (int ka = 0; ka <= G1; ++ka) {
            constexpr int kMaxInstr = S;     // upper bound on instructions per (kk, ka); the loop below exits on q0
            int q0 = G0 > ka ? G0 - ka : 0;
#pragma unroll
            for (int it = 0; it < kMaxInstr; ++it) {
                const int left = G1 + 1 - ka - q0;
                if (left <= 0) break;
                int cnt = left < CMAX ? left : CMAX;
                int n = BN * cnt;
                if (ODD8) {
                    if (cnt >= 2) { cnt &= ~1; n = BN * cnt; }
                    else n = BN + 8;         // the row's last plane: spills 8 columns above group S - 1
                }
                const uint32_t idesc = make_idesc_i8(kBM, n, KMAJOR ? 0 : 1, 0);
                // K-major: rows at 64 B pitch, 8-row swizzle atoms of 512 B (SBO); a K step is +32 B inside the span; the
                // next B plane starts BN/8 atoms further, i.e. N simply continues.
                // MN-major A: K rows of 128 B (SW128, atoms of 8 rows = 1 KB); a K step is 32 rows = 4 KB.
                const uint64_t da = KMAJOR ? make_smem_desc(sa + ka * A_BYTES + kk * 32, 16, 512, 4)
                                           : make_smem_desc(sa + ka * A_BYTES + kk * 4096, 8192, 1024, 2);
                const uint64_t db = make_smem_desc(sb + q0 * B_BYTES + kk * 32, 16, 512, 4);
                const uint32_t acc = (!first_block || kk > 0 || ka > 0) ? 1u : 0u;
                umma_i8(tmem_base + (uint32_t)((ka + q0 - G0) * BN), da, db, idesc, acc);
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
//
// G0, G1: group window (see window_bn).  G0 = 0 < G1 < S - 1 is the side launch of the split path: it stores the int32 group
// sums to side_buf instead of recombining them; G0 > 0 is the main launch: its Horner recombination continues below G0 with
// the side sums of the same unit, so the result is bit-identical to the full window.
template <int S, bool KMAJOR, int CL, bool CADD = false, int G0 = 0, int G1 = S - 1>
__global__ void __launch_bounds__(kThreads, 1)
oz_gemm_window_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const GemmParams p,
                      int32_t* const side_buf) {
    constexpr int NP = window_planes(G1);       // digit planes of each operand in a stage
    constexpr int NG = G1 - G0 + 1;             // accumulator groups in TMEM
    constexpr bool SIDE_OUT = G0 == 0 && G1 < S - 1;
    constexpr bool SIDE_IN = G0 > 0;
    static_assert(!SIDE_IN || G1 == S - 1, "the main launch of the split path ends at the last group");
    constexpr int kBN = window_bn(G0, G1);
    constexpr int kStages = window_stages(G0, G1);
    constexpr int A_BYTES = kBM * kBK;          // 8 KB per slice either way
    constexpr int B_BYTES = kBN * kBK;          // 4 KB (8 KB) per slice (full-width tile)
    constexpr int STAGE_BYTES = NP * (A_BYTES + B_BYTES);
    constexpr uint32_t TMEM_COLS = (NG * kBN + 8 <= 128) ? 128 : (NG * kBN + 8 <= 256 ? 256 : 512);  // (+ 8 spill columns)
    static_assert(NG * kBN <= 512, "accumulators exceed TMEM");
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
                    uint8_t* sb = sa + NP * A_BYTES;
                    const bool load_a = !(p.debug & 2), load_b = !(p.debug & 4);
                    const int k0 = kbeg + kb * kBK;
                    if (elect_one_sync()) {
                        mbar_expect_tx(&full_bar[st], NP * ((load_a ? A_BYTES : 0) + (load_b ? b_bytes : 0)));
#pragma unroll
                        for (int s = 0; s < NP; ++s) {
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
                    const uint32_t sb = sa + NP * A_BYTES;
                    if (elect_one_sync()) {
                    bool wide = (p.debug & 1) != 0;   // (debug: no MMAs at all)
                    if constexpr (kBN > 64) {
                        wide = wide || bn > 64;
                        if (p.debug & 1) {
                        } else if (bn == 128) issue_kblock_window<S, KMAJOR, 128, G0, G1>(sa, sb, tmem_base, kb == 0);
                        else if (bn == 112) issue_kblock_window<S, KMAJOR, 112, G0, G1>(sa, sb, tmem_base, kb == 0);
                        else if (bn == 96) issue_kblock_window<S, KMAJOR, 96, G0, G1>(sa, sb, tmem_base, kb == 0);
                        else if (bn == 80) issue_kblock_window<S, KMAJOR, 80, G0, G1>(sa, sb, tmem_base, kb == 0);
                    }
                    if (wide) {
                    } else if (bn == 64) issue_kblock_window<S, KMAJOR, 64, G0, G1>(sa, sb, tmem_base, kb == 0);
                    else if (bn == 56) issue_kblock_window<S, KMAJOR, 56, G0, G1>(sa, sb, tmem_base, kb == 0);
                    else if (bn == 48) issue_kblock_window<S, KMAJOR, 48, G0, G1>(sa, sb, tmem_base, kb == 0);
                    else if (bn == 40) issue_kblock_window<S, KMAJOR, 40, G0, G1>(sa, sb, tmem_base, kb == 0);
                    else if (bn == 32) issue_kblock_window<S, KMAJOR, 32, G0, G1>(sa, sb, tmem_base, kb == 0);
                    else if (bn == 24) issue_kblock_window<S, KMAJOR, 24, G0, G1>(sa, sb, tmem_base, kb == 0);
                    else issue_kblock_window<S, KMAJOR, 16, G0, G1>(sa, sb, tmem_base, kb == 0);
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
                    // this unit's side sums: [group][column][row], a warp reads 128 consecutive bytes per group and column
                    int32_t* side = SIDE_OUT || SIDE_IN ? side_buf + (long long)u * (SIDE_OUT ? NG : G0) * bn * kBM : nullptr;
                    int32_t sv[SIDE_IN ? G0 : 1][16];
                    if (SIDE_IN) {
#pragma unroll
                        for (int g = 0; g < G0; ++g)
#pragma unroll
                            for (int j = 0; j < 16; ++j)
                                sv[g][j] = c0 + j < bn ? side[((long long)g * bn + c0 + j) * kBM + row_in_tile] : 0;
                    }
                    // all group loads of this chunk in flight before the one wait (a wait per load serialised S TMEM round trips)
                    uint32_t r[NG][16];
#pragma unroll
                    for (int g = 0; g < NG; ++g) tmem_ld16(lane_addr + (uint32_t)(g * bn + c0), r[g]);
                    tmem_ld_wait();
                    if (c0 + 16 >= bn) {  // last chunk read: hand TMEM back to the MMA warp before the arithmetic and the stores
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&tmem_empty_bar);
                    }
                    if (SIDE_OUT) {
#pragma unroll
                        for (int g = 0; g < NG; ++g)
#pragma unroll
                            for (int j = 0; j < 16; ++j)
                                if (c0 + j < bn) side[((long long)g * bn + c0 + j) * kBM + row_in_tile] = (int32_t)r[g][j];
                        continue;
                    }
#pragma unroll
                    for (int j = 0; j < 16; ++j) acc[j] = (double)(int)r[NG - 1][j];
#pragma unroll
                    for (int g = S - 2; g >= G0; --g) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) acc[j] = acc[j] * p.inv_radix + (double)(int)r[g - G0][j];  // 1/R per group
                    }
                    if (SIDE_IN) {
#pragma unroll
                        for (int g = G0 - 1; g >= 0; --g) {
#pragma unroll
                            for (int j = 0; j < 16; ++j) acc[j] = acc[j] * p.inv_radix + (double)sv[g][j];
                        }
                    }
                } else if (SIDE_OUT) {
                    continue;
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

template <int S, bool KMAJOR, int CL, bool CADD = false, int G0 = 0, int G1 = S - 1>
inline int launch_oz_gemm_window(const CUtensorMap& mapA, const CUtensorMap& mapB, GemmParams p, int32_t* side, dim3 grid,
                                 cudaStream_t st) {
    constexpr int SMEM = window_stages(G0, G1) * window_planes(G1) * (kBM * kBK + window_bn(G0, G1) * kBK) + 1024;
    static PerDeviceOnce configured = {};
    static int resident[64] = {};  // clusters of this kernel that fit on the device at once, per device ordinal
    auto kern = oz_gemm_window_kernel<S, KMAJOR, CL, CADD, G0, G1>;
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
    LCX_CUDA(cudaLaunchKernelEx(&cfg, kern, mapA, mapB, p, side));
    return 0;
}

// Split path (S = kSplitS, one tile of bn = round_up(m, 16) <= 128 factors): one CTA per 128-row tile and no multicast.  The
// side launch runs groups 0 .. kSplitG - 1 over the same units first and leaves their int32 sums in `side`; the main launch
// accumulates the other groups (18 of the 21 plane products) and recombines all of them.  An SM then receives the X~ tile
// once per K block instead of once per CTA of a pair (DESIGN.md 4).
template <bool KMAJOR>
inline int launch_oz_gemm_split(const CUtensorMap& mapA, const CUtensorMap& mapB, GemmParams p, int32_t* side, dim3 grid,
                                 cudaStream_t st) {
    LCX_REQUIRE(grid.x == 1 && p.bn <= window_bn(kSplitG, kSplitS - 1) && side != nullptr, "split path: one tile of <= 128 factors");
    p.n_tiles = 1;
    p.n_tile0 = 0;
    LCX_TRY((launch_oz_gemm_window<kSplitS, KMAJOR, 1, false, 0, kSplitG - 1>(mapA, mapB, p, side, grid, st)));
    return launch_oz_gemm_window<kSplitS, KMAJOR, 1, false, kSplitG, kSplitS - 1>(mapA, mapB, p, side, grid, st);
}
// int32 values of the side buffer for `units` work units of tile width bn
inline long long split_side_ints(long long units, int bn) { return units * kSplitG * bn * kBM; }

}  // namespace oz
}  // namespace lcx
