// Host-side state of liblcx_b200.so: workspace layout (every array of a bound problem lives in ONE caller-provided
// workspace), launch plans, the session handle.  Included by lcx_api.cu only.
#pragma once
#include "../../include/lcx_b200.h"

#include <float.h>
#include <math.h>

#include "common.cuh"
#include "corex_kernels.cuh"
#include "dgemm_mma.cuh"
#include "fused_allreduce.cuh"
#include "lowrank_kernels.cuh"
#include "lu_solve.cuh"
#include "ozaki_i8.cuh"
#include "preprocess_kernels.cuh"

namespace lcx {
thread_local char g_err[512] = "";
constexpr int kSMs = 148;  // B200; plans (and therefore workspace sizes) are fixed for this part
constexpr int kMaxSplitsX = 32;
constexpr int kProfEv = 5;
constexpr int kMaxSplitsSmall = 148;

__global__ void axpy_kernel(const double* __restrict__ W, const double* __restrict__ U, double eta, double* __restrict__ W2,
                            int m, int n, long long ld) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int j = blockIdx.y;
    if (i < n && j < m) W2[(long long)j * ld + i] = W[(long long)j * ld + i] + eta * U[(long long)j * ld + i];
}

// out = c1 * D + e2 * u     (_sig, linearcorex.py:212)
__global__ void sig_finish_kernel(const double* __restrict__ D, const double* __restrict__ u, double c1, double e2,
                                  double* __restrict__ out, int m, int n, long long ld) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int j = blockIdx.y;
    if (i < n && j < m) out[(long long)j * ld + i] = c1 * D[(long long)j * ld + i] + e2 * u[(long long)j * ld + i];
}
}  // namespace lcx

using namespace lcx;

// internal (non-exported) workspace slots appended after the public enum
enum {
    I_T = LCX_A_COUNT,  // m x ld   rinv/(1+Qi-Si^2), also z of get_covariance and R of _update_syn
    I_PART,             // split-K partials
    I_COLSQ,            // K1 per-CTA column-sum-of-squares partials
    I_SPART,            // scalar partials
    I_W2,               // m   sum_i W^2
    I_BJ,               // m
    I_F,                // m   row scale factors
    I_UJDIAG,           // m   diag(W rho^T)
    I_ROWMI,            // m
    I_SQRTY,            // m
    I_RYINV,            // m x ldm  scratch (H of the search direction)
    I_AUG,              // scratch of the pivoted LU solve (lu_solve.cuh): work | LU | perm | status
    I_XS,               // split modes: int8 digit slices of X~   [S][N_local][ld8]
    I_AS,               //              int8 digit slices of A    [S][m][ld8]
    I_YS,               //              int8 digit slices of Y, transposed  [S][m][ldk8]
    I_OZV,              //              scales: x(16) | a(ldm) | c(ldm) | y(ldm) | d(ldm)
    I_YSTAT,            //              per-slab column max / sum of squares of Y
    I_AMAX,             //              per-CTA partial max |X~|
    I_MMA,              // m x m x n products on the int8 engine: row-scaled digit slices of the left operand  [S][m][ld8]
    I_MMB,              //              row-scaled digit slices of the right operand (K-major, contraction over variables)
    I_MMC,              //              column-scaled digit slices of the operand contracted over its rows (factors)
    I_MMQ,              //              row-scaled digit slices of the m x m factor (ry or H)  [S][m][ldm8]
    I_MMV,              //              scales: col partial max (32 x ld) | col scale (ld) | row scales a, b, q (3 x ldm)
    I_TAIL1,            // two-level split of the first contraction: partials of the tail units  [splits][tail rows][ldy]
    I_TAIL2,            //              of the second contraction  [splits][m][tail variables]
    I_COUNT
};

struct Slot {
    long long off, rows, cols, ld;
};

struct Layout {
    Slot slot[I_COUNT][2];
    long long total;
    long long ld, ldm, ldy;
    GemmPlan plan_k1, plan_k2, plan_mm, plan_mn;  // K1, K2, (m x m over n), (m x n over m)
    int nstrips;
    // split-integer modes (ozaki_i8.cuh)
    int S;                       // digits per operand, 0 = DMMA mode
    long long ld8, ldk8;         // byte leading dimensions of the X~/A slices and of the transposed Y slices (samples)
    int oz_splits, oz_chunk;     // split-K of the second contraction (over samples)
    int oz1_splits, oz1_chunk;   // split-K of the first contraction (over variables), only when row tiles are scarce
    // two-level split (TwoLevel below): the last tail_tiles M tiles run their last K chunk cut tail_splits ways
    int oz_tail_tiles, oz_tail_splits, oz_tail_chunk;     // second contraction (M tiles = 128 variables)
    int oz_build_splits, oz_build_chunk;                  // the uniform split over samples (what lcx_gram_build walks)
    int oz1_tail_tiles, oz1_tail_splits, oz1_tail_chunk;  // first contraction (M tiles = 128 samples)
    int ystat_slabs;
    int oz_kmax;                 // longest contraction one int32 accumulator group may see: 2^31 / ((R/2)^2 S)
    // the four m x m x n products of an iteration (ry, Qij, H, H W) on the same int8 engine (large m only)
    int mm_i8;                   // 0 = DMMA (dgemm_mma.cuh)
    long long ldm8;              // byte leading dimension of the digit slices of an m x m matrix
    int mm_splits, mm_chunk;     // split-K over the variables of the m x m outputs
    int mm_slabs, mm_slab_rows;  // row slabs of the per-column maximum
};

static int digits_for(int precision) {
    if (precision == LCX_PRECISION_FP64) return 0;
    const char* env = getenv("LCX_SPLIT_DIGITS");
    if (env && atoi(env) >= 3 && atoi(env) <= 7) return atoi(env);
    if (precision == LCX_PRECISION_FAST) return 3;          // 24 bits: fp32-equivalent products
    if (precision == LCX_PRECISION_FP64_SPLIT5) return 5;   // 40 bits
    if (precision == LCX_PRECISION_FP64_SPLIT7) return 7;   // 56 bits: finer than binary64's own 53-bit significand
    return 6;                                               // 48 bits: truncation at the level of binary64 rounding
}
// LCX_MM_I8=1 / 0 forces the int8 engine for the m x m x n products on / off; otherwise it is used from m = 384 factors
// (measured on a B200: m = 500, n = 50 000: direction 3.70 -> 3.19 ms, trial 2.25 -> 1.50 ms; m = 256, n = 8 000: 5 % slower --
// the products grow with m^2 n, the extra digit slicing with m n).
static int mm_i8_for(int S, int n, int m) {
    if (S <= 0 || round_up(m, 64) > (1 << 14)) return 0;
    const char* env = getenv("LCX_MM_I8");
    if (env) return atoi(env) != 0;
    return m >= 384 && n >= 2048;
}
constexpr int kYStatRows = 512;
constexpr int kAmaxCtas = 592;

static long long align16(long long v) { return round_up(v, 16); }

// Cost of one work unit of the persistent split-integer contraction beyond its K blocks, in units of one 64-deep K block
// (drain of the accumulators that the next unit's operand fill does not hide + the ring restart).
constexpr double kOzUnitFixedKb = 4.0;

// Two-level split of a contraction whose uniform units (M tiles x K splits, one cluster per unit and N group) do not fill whole
// rounds of the resident clusters: R full rounds of the uniform units, and the r units left over -- the last K chunk of the
// last few M tiles -- cut t = #clusters / r ways so that they fill ONE more short round instead of a long, mostly idle one.
// 12 500 samples per rank (config 3 on 8 GPUs), second contraction: 79 tiles on 74 cluster pairs = 1 round of 196 K blocks + 5
// tiles x 14 splits of 14 K blocks (cost 218 in K-block units) instead of 7 uniform splits in 8 rounds of 28 + 4 (266).
// Cost model as everywhere: rounds x (K blocks per unit + the per-unit fixed cost) + what the combine of the partials costs.
struct TwoLevel {
    int splits, chunk;                       // uniform level
    int tail_tiles, tail_splits, tail_chunk; // 0 tiles: plain uniform split
    double cost;
};
static TwoLevel plan_two_level(long long K, int m_tiles, int n_groups, int smin, int smax, double combine_per_split) {
    const int clusters = kSMs / 2;
    TwoLevel best = {0, 0, 0, 0, 0, 1e300};  // (only plans WITH a tail are returned; cost 1e300 = none exists)
    for (int s0 = smin; s0 <= max(smin, smax); ++s0) {
        const int chunk = (int)round_up(cdiv(K, s0), oz::kBK);
        const int sp = cdiv(K, chunk);
        if (sp < smin) continue;
        const long long U = (long long)n_groups * m_tiles * sp;
        const long long R = U / clusters, r = U - R * clusters;
        const int rt = cdiv(r, n_groups);
        if (r == 0 || R == 0 || rt > m_tiles) continue;
        const long long klast = K - (long long)(sp - 1) * chunk;
        int t = (int)min((long long)(clusters / (rt * n_groups)), max(1LL, (long long)cdiv(klast, oz::kBK) / 2));
        if (t <= 1) continue;
        const int tchunk = (int)round_up(cdiv(klast, t), oz::kBK);
        t = cdiv(klast, tchunk);
        if (t <= 1) continue;
        const double cost = (double)R * (chunk / oz::kBK + kOzUnitFixedKb) + (tchunk / oz::kBK + kOzUnitFixedKb) +
                            (sp > 1 ? combine_per_split * sp : 0.0) + 4.0;  // + the fold launch
        if (cost < best.cost - 1e-9) best = TwoLevel{sp, chunk, rt, t, tchunk, cost};
    }
    return best;
}
// LCX_OZ_TAIL=0 switches the two-level split off; it needs pairs of N tiles in one launch.
static bool oz_tail_allowed(int m, int S) {
    const char* env = getenv("LCX_OZ_TAIL");
    if (env && atoi(env) == 0) return false;
    return cdiv(m, oz::bn_max(S)) % 2 == 0;
}

// Gram product plan (host_gram.cuh): `full` row tiles run as whole waves with the full contraction, the remaining ones split
// over K `splits` ways so that they fill one more short wave.  full = 0: not applicable (the generic split-K plan is used).
struct GramPlan {
    int full, rest, splits, chunk;
};
static GramPlan gram_plan(int n, int m, int S, int oz_kmax) {
    GramPlan g = {0, 0, 1, 0};
    const int n_tiles = cdiv(m, oz::bn_max(S)), m_tiles = cdiv(n, oz::kBM);
    const int clusters = kSMs / 2;
    if (n_tiles != 2 || n > oz_kmax) return g;
    g.full = (m_tiles / clusters) * clusters;
    g.rest = m_tiles - g.full;
    if (g.full == 0 || g.rest == 0) return g;
    const int kblocks = cdiv(n, oz::kBK);
    const int sp = max(1, min(clusters / g.rest, kblocks / 4));
    g.chunk = (int)round_up(cdiv(n, sp), oz::kBK);
    g.splits = cdiv(n, g.chunk);
    return g;
}

// gram: the bound "data" is the n x n matrix X~^T X~ / N (Nl = n rows); only the first contraction runs, with its output stored
// factor-major (transposed), so its split-K partials are m x ld each.
static Layout make_layout(long long Nl, int n, int m, int precision, bool gram = false) {
    Layout L;
    memset(&L, 0, sizeof(L));
    L.S = digits_for(precision);
    if (L.S > 0) {
        const long long half = oz::kRadix / 2;
        L.oz_kmax = (int)(((1LL << 31) / (half * half * L.S)) / 64 * 64);
        if (L.oz_kmax > 65536) L.oz_kmax = 65536;
    }
    L.ld = round_up(n, 16);
    L.ldm = round_up(m, 16);
    L.ldy = round_up(m, 8);
    // few samples (N << 128 * 148 rows): split the first contraction over the variables as well
    const bool k1_split = (long long)cdiv(Nl, 128) * cdiv(m, 128) < kSMs / 2;
    L.plan_k1 = plan_gemm((int)Nl, m, n, kSMs, k1_split ? 16 : 1, k1_split);
    L.plan_k2 = plan_gemm(n, m, (int)Nl, kSMs, kMaxSplitsX, true);
    L.plan_mm = plan_gemm(m, m, n, kSMs, kMaxSplitsSmall, true);
    L.plan_mn = plan_gemm_kn(m, n, m, kSMs);
    L.nstrips = cdiv(n, kStripCols);
    long long cur = 0;
    auto put = [&](int id, int set, long long rows, long long cols, long long ld) {
        L.slot[id][set] = Slot{cur, rows, cols, ld};
        cur = align16(cur + rows * ld);
    };
    const long long mn = m;
    for (int set = 0; set < 2; ++set) {
        put(LCX_A_W, set, mn, n, L.ld);
        put(LCX_A_RHO, set, mn, n, L.ld);
        put(LCX_A_INVRHO, set, mn, n, L.ld);
        put(LCX_A_RHOINVRHO, set, mn, n, L.ld);
        put(LCX_A_QIJ, set, mn, n, L.ld);
        put(LCX_A_SI, set, 1, n, L.ld);
        put(LCX_A_QISI2, set, 1, n, L.ld);
        put(LCX_A_RY, set, mn, m, L.ldm);
        put(LCX_A_UJ, set, 1, m, L.ldm);
    }
    auto put1 = [&](int id, long long rows, long long cols, long long ld) {
        put(id, 0, rows, cols, ld);
        L.slot[id][1] = L.slot[id][0];
    };
    put1(LCX_A_GRAD, mn, n, L.ld);
    put1(LCX_A_UPDATE, mn, n, L.ld);
    put1(LCX_A_RDIR, mn, n, L.ld);
    put1(LCX_A_D, mn + cdiv(m, L.ld), n, L.ld);  // D (m x ld) immediately followed by s (m values)
    put1(LCX_A_MI, mn, n, L.ld);
    put1(LCX_A_XZ, mn, n, L.ld);
    put1(LCX_A_XY, mn, n, L.ld);
    put1(LCX_A_X2Y, 1, n, L.ld);
    put1(LCX_A_IXY, 1, n, L.ld);
    put1(LCX_A_YJ2, 1, m, L.ldm);
    put1(LCX_A_IYX, 1, m, L.ldm);
    put1(LCX_A_TCS, 1, m, L.ldm);
    put1(LCX_A_TCDIRECT, 1, m, L.ldm);
    put1(LCX_A_CY, mn, m, L.ldm);
    put1(LCX_A_Y, Nl, m, L.ldy);
    put1(LCX_A_SCALARS, 1, 16, 16);
    put1(I_T, mn, n, L.ld);
    long long part = 0;
    if (L.plan_k2.splits > 1) part = max(part, (long long)L.plan_k2.splits * mn * L.ld);
    if (L.plan_mm.splits > 1) part = max(part, (long long)L.plan_mm.splits * mn * L.ldm);
    if (L.plan_k1.splits > 1) part = max(part, (long long)L.plan_k1.splits * Nl * L.ldy);
    put1(I_PART, 1, max(part, 16LL), max(part, 16LL));
    put1(I_COLSQ, L.plan_k1.grid.x, m, L.ldy);
    const long long spart = max(3LL * L.nstrips, (long long)m * cdiv(n, 256));
    put1(I_SPART, 1, spart, spart);
    put1(I_W2, 1, m, L.ldm);
    put1(I_BJ, 1, m, L.ldm);
    put1(I_F, 1, m, L.ldm);
    put1(I_UJDIAG, 1, m, L.ldm);
    put1(I_ROWMI, 1, m, L.ldm);
    put1(I_SQRTY, 1, m, L.ldm);
    put1(I_RYINV, mn, m, L.ldm);
    put1(I_AUG, 1, lu::scratch_doubles(m), lu::scratch_doubles(m));
    L.ystat_slabs = cdiv(Nl, kYStatRows);
    put1(I_OZV, 1, 16 + 4 * L.ldm, 16 + 4 * L.ldm);
    put1(I_YSTAT, (long long)L.ystat_slabs * 2, m, L.ldm);
    if (L.S > 0) {
        L.ld8 = round_up(n, 128);
        L.ldk8 = round_up(Nl, 128);
        // second contraction: 128 x 64 tiles over (variables x factors), split over samples to fill whole waves;
        // at most oz_kmax samples per split keeps every int32 accumulator exact
        const long long tiles = (long long)cdiv(n, oz::kBM) * cdiv(m, oz::bn_max(L.S));
        const int kblocks = cdiv(Nl, oz::kBK);
        // time model in units of one 64-deep K block: waves x (K blocks per CTA + the per-unit fixed cost kOzUnitFixedKb)
        // + the partial-buffer round trip; measured at 12.5k and 100k rows per GPU
        int best = 1;
        double best_cost = 1e300;
        const int smin = cdiv(Nl, L.oz_kmax), smax = (int)min(64LL, (long long)max(1, kblocks / 8));
        for (int sp = smin; sp <= max(smin, smax); ++sp) {
            const long long ctas = tiles * sp;
            const long long waves = (ctas + kSMs - 1) / kSMs;
            const double kb = ceil((double)kblocks / sp);
            const double cost = (double)waves * (kb + kOzUnitFixedKb) + (sp > 1 ? 1.5 * sp : 0.0);
            if (cost < best_cost - 1e-9) { best_cost = cost; best = sp; }
        }
        L.oz_chunk = (int)round_up(cdiv(Nl, best), oz::kBK);
        L.oz_splits = cdiv(Nl, L.oz_chunk);
        L.oz_build_splits = L.oz_splits;
        L.oz_build_chunk = L.oz_chunk;
        const bool tail_ok = !gram && oz_tail_allowed(m, L.S);
        if (tail_ok) {
            const TwoLevel t2 = plan_two_level(Nl, cdiv(n, oz::kBM), cdiv(cdiv(m, oz::bn_max(L.S)), 2), smin, max(smin, smax), 1.5);
            if (t2.tail_tiles > 0 && t2.cost < best_cost) {
                L.oz_chunk = t2.chunk; L.oz_splits = t2.splits;
                L.oz_tail_tiles = t2.tail_tiles; L.oz_tail_splits = t2.tail_splits; L.oz_tail_chunk = t2.tail_chunk;
            }
        }
        {   // first contraction: same cost model over its (row tile x factor tile) grid
            const long long tiles1 = (long long)cdiv(Nl, oz::kBM) * cdiv(m, oz::bn_max(L.S));
            const int kblocks1 = cdiv(n, oz::kBK);
            int b1 = cdiv(n, L.oz_kmax);
            double c1best = 1e300;
            const int s1min = cdiv(n, L.oz_kmax);  // int32 exactness of every accumulator group
            for (int sp = s1min; sp <= max(s1min, min(8, kblocks1 / 16)); ++sp) {
                const long long waves = (tiles1 * sp + kSMs - 1) / kSMs;
                const double cost = (double)waves * (ceil((double)kblocks1 / sp) + kOzUnitFixedKb) + (sp > 1 ? 4.0 * sp : 0.0);
                if (cost < c1best - 1e-9) { c1best = cost; b1 = sp; }
            }
            L.oz1_chunk = (int)round_up(cdiv(n, b1), oz::kBK);
            L.oz1_splits = cdiv(n, L.oz1_chunk);
            if (tail_ok) {
                const TwoLevel t1 = plan_two_level(n, cdiv(Nl, oz::kBM), cdiv(cdiv(m, oz::bn_max(L.S)), 2), s1min,
                                                   max(s1min, min(8, kblocks1 / 16)), 4.0);
                if (t1.tail_tiles > 0 && t1.cost < c1best) {
                    L.oz1_chunk = t1.chunk; L.oz1_splits = t1.splits;
                    L.oz1_tail_tiles = t1.tail_tiles; L.oz1_tail_splits = t1.tail_splits; L.oz1_tail_chunk = t1.tail_chunk;
                }
            }
        }
        long long part = max((long long)L.oz_splits * mn * L.ld, L.oz1_splits > 1 ? (long long)L.oz1_splits * Nl * L.ldy : 0LL);
        if (gram) {
            part = max(part, (long long)L.oz1_splits * mn * L.ld);
            part = max(part, (long long)gram_plan(n, m, L.S, L.oz_kmax).splits * mn * L.ld);
            // sharded over ranks (host_gram.cuh) a rank's few row tiles are split up to kSMs / 2 / tiles ways: with at least
            // two ranks and 128-variable tiles that is at most min(kSMs / 2, K blocks / 4) partials
            part = max(part, (long long)min(kSMs / 2, max(1, cdiv(n, oz::kBK) / 4)) * mn * L.ld);
        }
        if (part > L.slot[I_PART][0].cols) {  // grow the split-K partial buffer (it is the last big slot before these)
            put1(I_PART, 1, part, part);
        }
        const long long xs8 = ((long long)L.S * Nl * L.ld8 + 7) / 8;   // int8 planes counted in doubles (64-bit sizes:
        const long long as8 = ((long long)L.S * mn * L.ld8 + 7) / 8;   // the target shape has 1.5e10 doubles of planes)
        const long long ys8 = ((long long)L.S * mn * L.ldk8 + 7) / 8;
        put1(I_XS, 1, xs8, xs8);
        put1(I_AS, 1, as8, as8);
        put1(I_YS, 1, ys8, ys8);
        put1(I_AMAX, 1, kAmaxCtas, kAmaxCtas);
        {
            const long long t1 = max(16LL, (long long)L.oz1_tail_splits * L.oz1_tail_tiles * oz::kBM * L.ldy);
            const long long t2 = max(16LL, (long long)L.oz_tail_splits * mn * L.oz_tail_tiles * oz::kBM);
            put1(I_TAIL1, 1, t1, t1);
            put1(I_TAIL2, 1, t2, t2);
        }
        L.mm_i8 = mm_i8_for(L.S, n, m);
        if (L.mm_i8) {
            L.ldm8 = round_up(m, 128);
            {   // m x m outputs, contraction over the variables: split to fill the SMs, never beyond the int32-exact length
                const long long tiles_mm = (long long)cdiv(m, oz::kBM) * cdiv(m, oz::bn_max(L.S));
                const int kblocks_mm = cdiv(n, oz::kBK);
                const int smin_mm = cdiv(n, L.oz_kmax);
                int bmm = smin_mm;
                double cbest = 1e300;
                for (int sp = smin_mm; sp <= max(smin_mm, min(64, kblocks_mm / 8)); ++sp) {
                    const long long waves = (tiles_mm * sp + kSMs - 1) / kSMs;
                    const double cost = (double)waves * (ceil((double)kblocks_mm / sp) + kOzUnitFixedKb) + 1.5 * sp;
                    if (cost < cbest - 1e-9) { cbest = cost; bmm = sp; }
                }
                L.mm_chunk = (int)round_up(cdiv(n, bmm), oz::kBK);
                L.mm_splits = cdiv(n, L.mm_chunk);
            }
            L.mm_slabs = (int)min(32LL, (long long)cdiv(m, 8));
            L.mm_slab_rows = cdiv(m, L.mm_slabs);
            const long long need = (long long)L.mm_splits * mn * L.ldm;
            if (need > L.slot[I_PART][0].cols) put1(I_PART, 1, need, need);
            const long long pl8 = ((long long)L.S * mn * L.ld8 + 7) / 8;
            const long long q8 = ((long long)L.S * mn * L.ldm8 + 7) / 8;
            put1(I_MMA, 1, pl8, pl8);
            put1(I_MMB, 1, pl8, pl8);
            put1(I_MMC, 1, pl8, pl8);
            put1(I_MMQ, 1, q8, q8);
            put1(I_MMV, 1, 33 * L.ld + 3 * L.ldm, 33 * L.ld + 3 * L.ldm);
        }
    }
    L.total = cur;
    if (getenv("LCX_PLAN_DEBUG") && L.S > 0)
        fprintf(stderr, "[lcx plan] Nl=%lld n=%d m=%d gram=%d | K1: splits %d chunk %d tail %d tiles x %d splits (chunk %d) | K2: splits %d "
                "chunk %d tail %d tiles x %d splits (chunk %d)\n", Nl, n, m, (int)gram, L.oz1_splits, L.oz1_chunk, L.oz1_tail_tiles,
                L.oz1_tail_splits, L.oz1_tail_chunk, L.oz_splits, L.oz_chunk, L.oz_tail_tiles, L.oz_tail_splits, L.oz_tail_chunk);
    return L;
}

struct lcx_session {
    int device, precision;
    cudaStream_t stream;
    lcx_allreduce_fn hook;
    void* hook_user;
    long long launches;
    double* mailbox;  // pinned host, 16 doubles (a slot of the process-wide block, lcx_api.cu)
    bool mailbox_pooled;
    unsigned long long mailbox_seq;   // sequence number of the last post_mailbox_kernel (slot 16 of the mailbox)
    bool bound;
    const double* xt;
    bool gram;        // the bound matrix is X~^T X~ / N (lcx_bind_gram): a "pass pair" is ONE product G A^T (host_gram.cuh)
    long long Nl, Nt, ldx;
    // CUDA graphs of the loop body (lcx_run_stage_ns): direction + first trial + mailbox copy of one iteration, one graph per
    // physical parity of the moment sets, re-captured when eps changes.  Captured and replayed on gstream (a blocking stream:
    // capture is not allowed on the legacy default stream torch hands over).
    cudaStream_t gstream;
    cudaEvent_t gevent;
    cudaGraphExec_t graph_exec[2];
    double graph_eps;
    long long graph_launches[2];
    int graph_warm[2];  // iterations already run without capture on this parity (kernel attributes are configured there)
    int d_splits;     // > 1: the last Gram product left its split-K partials in I_PART for the consumer to add (host_gram.cuh)
    int n, m;
    double* ws;
    Layout L;
    int cur;  // which physical set is "set 0" (current)
    // optional device-side timing of the two X contractions (bench.py roofline); events are
    // recorded on the session stream around each launch and resolved at lcx_profile_read
    bool prof_on;
    cudaEvent_t* prof_ev;      // kProfEv per pair: [0] before K1, [1] after K1, [3] before K2, [4] before the split-K combine /
                               // rank exchange, [2] after it
    int prof_pending, prof_cap;
    double prof_k1_ms, prof_k2_ms, prof_x_ms;
    long long prof_pairs;
    // sample sharding over NVLink peers (fused_allreduce.cuh); peers.world <= 1 means off
    far::Peers peers;
    unsigned long long ar_calls;
    // split-integer modes: TMA descriptors over the digit slices
    CUtensorMap map_x_k1, map_a_k1, map_x_k2, map_y_k2;
    int oz_bn;        // width of every factor tile (equal split of the m factors; multiple of 8, >= 16)
    // m x m x n products on the int8 engine (L.mm_i8)
    CUtensorMap map_mm_a, map_mm_b, map_mn_c, map_mn_q;
    int8_t* mma() const { return (int8_t*)(ws + L.slot[I_MMA][0].off); }
    int8_t* mmb() const { return (int8_t*)(ws + L.slot[I_MMB][0].off); }
    int8_t* mmc() const { return (int8_t*)(ws + L.slot[I_MMC][0].off); }
    int8_t* mmq() const { return (int8_t*)(ws + L.slot[I_MMQ][0].off); }
    double* mm_colpart() const { return ws + L.slot[I_MMV][0].off; }
    double* mm_colscale() const { return ws + L.slot[I_MMV][0].off + 32 * L.ld; }
    double* mm_scale_a() const { return ws + L.slot[I_MMV][0].off + 33 * L.ld; }
    double* mm_scale_b() const { return ws + L.slot[I_MMV][0].off + 33 * L.ld + L.ldm; }
    double* mm_scale_q() const { return ws + L.slot[I_MMV][0].off + 33 * L.ld + 2 * L.ldm; }
    int8_t* xs() const { return (int8_t*)(ws + L.slot[I_XS][0].off); }
    int8_t* as() const { return (int8_t*)(ws + L.slot[I_AS][0].off); }
    int8_t* ys() const { return (int8_t*)(ws + L.slot[I_YS][0].off); }
    double* oz_xscale() const { return ws + L.slot[I_OZV][0].off; }
    double* oz_ascale() const { return ws + L.slot[I_OZV][0].off + 16; }
    double* oz_cscale() const { return ws + L.slot[I_OZV][0].off + 16 + L.ldm; }
    double* oz_yscale() const { return ws + L.slot[I_OZV][0].off + 16 + 2 * L.ldm; }
    double* oz_dscale() const { return ws + L.slot[I_OZV][0].off + 16 + 3 * L.ldm; }

    double* ptr(int id, int set = 0) const {
        // with NVLink peers the exchanged block (D and the column sums of squares behind it) IS the output region of this
        // rank's symmetric buffer: the exchange kernel's last phase stores the sums there directly, no copy-out
        if (id == LCX_A_D && peers.world > 1) return peers.base[peers.rank] + 2 * peers.count;
        const int phys = (id <= LCX_A_UJ) ? (set ^ cur) : 0;
        return ws + L.slot[id][phys].off;
    }
    long long off(int id, int set = 0) const {
        const int phys = (id <= LCX_A_UJ) ? (set ^ cur) : 0;
        return L.slot[id][phys].off;
    }
};

#define S_REQUIRE_BOUND(s)                                                        \
    do {                                                                          \
        if (!(s)) return fail(LCX_ERR_ARG, "session", "null session");            \
        if (!(s)->bound) return fail(LCX_ERR_STATE, "session", "no bound problem"); \
        LCX_CUDA(cudaSetDevice((s)->device));                                     \
    } while (0)

#define LAUNCHED(s) ((s)->launches++)

static int combine_and_allreduce(lcx_session* s, const double* part, int splits, long long stride, int rows, int cols,
                                 long long ld, double* dst_body, double* tail, int ntail);

static dim3 grid_mn(int m, int n) { return dim3(cdiv(n, 256), m); }
