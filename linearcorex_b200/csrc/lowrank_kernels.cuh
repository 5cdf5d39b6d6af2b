// Scoring held-out data under the fitted covariance (Corex.score_samples / mahalanobis / get_precision).
//
// For discourage_overlap=True the estimate of get_covariance (linearcorex.py:447-451) is exactly low rank plus diagonal:
//   z = rhoinvrho / (1 + Si),  Z = z / sqrt(1 - eps^2)     (m x n)
//   Sigma = S (Z^T Z + Delta) S,   S = diag(theta[1]),   Delta = diag(1 - sum_j Z_ji^2)
// (np.fill_diagonal only replaces the diagonal).  With Woodbury and Sylvester, for Delta > 0:
//   K = I_m + Z Delta^-1 Z^T = G G^T      B = G^-1 Z Delta^-1      (m x n)
//   Sigma^-1 = S^-1 (Delta^-1 - B^T B) S^-1
//   log det Sigma = 2 sum_i log sd_i + sum_i log Delta_i + 2 sum_k log G_kk
//   q(x) = sum_i x~_i^2 / Delta_i - |B x~|^2,   x~ = (x - mean) / sd
// so a sample costs O(n m) and the factor O(n m^2 + m^3) instead of O(n^2) and O(n^3).
//
//   factor_prep_kernel    Z Delta^-1/2 (operand of K), Z Delta^-1 (right-hand sides of B), 1/Delta, per-column log terms
//   chol_factor_kernel    K = G G^T (K arrives without its identity), written in lu_solve.cuh's `lup` layout so that
//                         lu_solve_kernel performs G^-1 = diag(G)^-1 L^-1; one CTA in shared memory for m <= 160, the
//                         cooperative grid with one grid barrier per column beyond that (modelled on lu_factor_kernel)
//   logdet_kernel         fixed-order log det Sigma + the status word for the host mailbox
//   score_standardize_kernel   x~ (standardize_kernel's arithmetic) and s_l = sum_i x~_li^2 / Delta_i in one pass
//   score_finish_kernel   q_l = s_l - sum_j Y_lj^2 and log p_l from Y = X~ B^T (the DMMA projection)
//   precision_finish_kernel    (delta_ik / Delta_i - (B^T B)_ik) / (sd_i sd_k) of one row block
//   eye_kernel            the identity that lu_solve_kernel turns into G^-1 (H = G^-1 G^-T, the m x m matrix conditioning needs)
//   condition_rows_kernel conditional mean of the missing entries, q_O and log p(x_O) of a row, one CTA per row: the
//                         order-p system of Path A or B in shared memory (p <= 160) or in a per-CTA global slab; in its
//                         kCondSample mode also conditional standard deviations and draws from the same factor
//   normal_fill_kernel    counter-based standard normals (Philox4x32-10 + Box-Muller), the U of sampling
//   sample_prep_kernel    Z and sqrt(Delta) for sampling, Delta as factor_prep_kernel forms it
//   sample_finish_kernel  theta0 + theta1 (U Z + sqrt(Delta) eps), eps generated in registers
//   given_prep_kernel     conditioning on a fixed column set O: Z_O Delta_O^-1/2, Z_O Delta_O^-1, the gathered theta and
//                         1/Delta of O, Z_T and Delta_T of the targets T, with factor_prep_kernel's Delta_i
//   given_std_kernel      theta1_t sqrt(Delta_t + |p_t|^2), the conditional standard deviation of target t
//   given_mean_finish_kernel   theta0_T + theta1_T (V P) of a row block (the conditional means)
//   given_cov_finish_kernel    theta1_T (Delta_T + P^T P) theta1_T of a row block (the conditional covariance)
#pragma once
#include "common.cuh"
#include "lu_solve.cuh"
#include "preprocess_kernels.cuh"

namespace lcx {
namespace lowrank {

// Z_ji and Delta_i (the m factors summed in index order) of column i, c = 1 + Si_i: the one definition that scoring,
// conditioning and sampling share, so that all of them see the same Delta bit for bit.
__device__ __forceinline__ double lowrank_z(const double* __restrict__ rinv, long long ldr, int j, int i, double c,
                                            double inv_sqrt_scale) {
    return rinv[(long long)j * ldr + i] / c * inv_sqrt_scale;
}
__device__ __forceinline__ double lowrank_delta(const double* __restrict__ rinv, long long ldr, int m, int i, double c,
                                                double inv_sqrt_scale) {
    double acc = 0.0;
    for (int j = 0; j < m; ++j) {
        const double z = lowrank_z(rinv, ldr, j, i, c, inv_sqrt_scale);
        acc += z * z;
    }
    return 1.0 - acc;
}

// One thread per variable i.  rinv: ld ldr; zh, zd: ld ldz.  status[1] = 1 when some Delta_i <= 0 (Sigma is then not treated
// as positive definite).
__global__ void factor_prep_kernel(const double* __restrict__ rinv, const double* __restrict__ si, long long ldr, long long ldz,
                                   int m, int n, double inv_sqrt_scale, const double* __restrict__ sd, double* __restrict__ zh,
                                   double* __restrict__ zd, double* __restrict__ dinv, double* __restrict__ ldiag,
                                   int* __restrict__ status) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double c = 1.0 + si[i];
    const double delta = lowrank_delta(rinv, ldr, m, i, c, inv_sqrt_scale);
    if (!(delta > 0.0)) status[1] = 1;
    const double di = 1.0 / delta, rs = sqrt(di);
    dinv[i] = di;
    ldiag[i] = 2.0 * log(sd[i]) + log(delta);
    for (int j = 0; j < m; ++j) {
        const double z = lowrank_z(rinv, ldr, j, i, c, inv_sqrt_scale);
        zh[(long long)j * ldz + i] = z * rs;
        zd[(long long)j * ldz + i] = z * di;
    }
}

// ---- counter-based standard normals (Corex.sample, sample_missing) ---------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11; Random123's constants).  Normal j of stream (seed, tag, row, draw) comes from the
// counter (j / 2, draw, row mod 2^32, row / 2^32 + 2^24 tag) under the key (seed mod 2^32, seed / 2^32): two uniforms in
// (0, 1] of 53 bits each, u1 from words 0/1 and u2 from words 2/3, then Box-Muller, z_2t = sqrt(-2 ln u1) cospi(2 u2) and
// z_2t+1 = sqrt(-2 ln u1) sinpi(2 u2).  It depends on nothing else, so results are the same under any grid, row blocking or
// split of the rows between calls.  Tag 0: sample (columns 0..m-1 are u, m..m+n-1 eps); tag 1: conditional draws of the
// missing entries (sample_missing); tag 2: draws given a fixed column set (ConditionalGaussian.sample: columns 0..m-1 are u,
// m..m+|T|-1 eps in the order of the targets).
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return c;
}
__device__ __forceinline__ uint4 philox_words(unsigned long long seed, int tag, long long row, long long draw, long long t) {
    const unsigned long long ur = (unsigned long long)row;
    return philox4x32_10(make_uint4((uint32_t)t, (uint32_t)draw, (uint32_t)ur, (uint32_t)(ur >> 32) + ((uint32_t)tag << 24)),
                         (uint32_t)seed, (uint32_t)(seed >> 32));
}
__device__ __forceinline__ double uniform53(uint32_t hi, uint32_t lo) {  // (0, 1], exact
    return (double)((((unsigned long long)hi << 21) | (lo >> 11)) + 1ULL) * 0x1p-53;
}
__device__ __forceinline__ double2 normal_pair(unsigned long long seed, int tag, long long row, long long draw, long long t) {
    const uint4 w = philox_words(seed, tag, row, draw, t);
    const double r = sqrt(-2.0 * log(uniform53(w.x, w.y)));
    double s, c;
    sincospi(2.0 * uniform53(w.z, w.w), &s, &c);
    return make_double2(r * c, r * s);
}
__device__ __forceinline__ double normal_at(unsigned long long seed, int tag, long long row, long long draw, long long j) {
    const double2 z = normal_pair(seed, tag, row, draw, j >> 1);
    return (j & 1) ? z.y : z.x;
}

// out (rows x ldo): out[r][j] = normal j of stream (seed, tag, row0 + r, draw) for j < cols, plus base[r][j] when base (ld
// ldo) is given; words (optional, rows x ldw) the four Philox words behind normals 2t and 2t + 1 at words[r][4t .. 4t + 3].
// One thread per counter.
__global__ void __launch_bounds__(256) normal_fill_kernel(unsigned long long seed, int tag, long long row0, long long rows,
                                                          long long draw, int cols, const double* __restrict__ base,
                                                          double* __restrict__ out, long long ldo,
                                                          uint32_t* __restrict__ words, long long ldw) {
    const long long pairs = (cols + 1) / 2;
    for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < rows * pairs; e += (long long)gridDim.x * 256) {
        const long long r = e / pairs, t = e % pairs;
        const double2 z = normal_pair(seed, tag, row0 + r, draw, t);
        out[r * ldo + 2 * t] = base ? base[r * ldo + 2 * t] + z.x : z.x;
        if (2 * t + 1 < cols) out[r * ldo + 2 * t + 1] = base ? base[r * ldo + 2 * t + 1] + z.y : z.y;
        if (words) {
            const uint4 w = philox_words(seed, tag, row0 + r, draw, t);
            uint32_t* o = words + r * ldw + 4 * t;
            o[0] = w.x, o[1] = w.y, o[2] = w.z, o[3] = w.w;
        }
    }
}

// One thread per variable i: Z (m x ldz) and sqrt(Delta) of Sigma~ = Z^T Z + Delta, with factor_prep_kernel's Delta_i.
// scalars[0] = 1 when some Delta_i <= 0 (the host reads it through the mailbox).
__global__ void sample_prep_kernel(const double* __restrict__ rinv, const double* __restrict__ si, long long ldr, long long ldz,
                                   int m, int n, double inv_sqrt_scale, double* __restrict__ z, double* __restrict__ sqd,
                                   double* __restrict__ scalars) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double c = 1.0 + si[i];
    const double delta = lowrank_delta(rinv, ldr, m, i, c, inv_sqrt_scale);
    if (!(delta > 0.0)) scalars[0] = 1.0;
    sqd[i] = sqrt(delta);
    for (int j = 0; j < m; ++j) z[(long long)j * ldz + i] = lowrank_z(rinv, ldr, j, i, c, inv_sqrt_scale);
}

// out (rows x ldo) holds Y = U Z on entry and theta0 + theta1 (Y + sqrt(Delta) eps) on exit, eps_i = normal m + i of stream
// (seed, tag, row0 + r, draw), generated here and never stored.  One thread per Philox counter (two normals).  sample: tag 0,
// draw 0; ConditionalGaussian.sample: tag 2, n = |T|, the gathered theta and sqrt(Delta) of the targets.
__global__ void __launch_bounds__(256) sample_finish_kernel(double* __restrict__ out, long long ldo, long long rows, int m, int n,
                                                            const double* __restrict__ sqd, const double* __restrict__ mean,
                                                            const double* __restrict__ sd, unsigned long long seed,
                                                            long long row0, int tag, long long draw) {
    const long long t0 = m >> 1, pairs = ((long long)(m + n - 1) >> 1) - t0 + 1;
    for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < rows * pairs; e += (long long)gridDim.x * 256) {
        const long long r = e / pairs, t = t0 + e % pairs;
        const double2 z = normal_pair(seed, tag, row0 + r, draw, t);
        const long long i0 = 2 * t - m;
        if (i0 >= 0) {
            double* o = out + r * ldo + i0;
            *o = mean[i0] + sd[i0] * (*o + sqd[i0] * z.x);
        }
        if (i0 + 1 < n) {
            double* o = out + r * ldo + i0 + 1;
            *o = mean[i0 + 1] + sd[i0 + 1] * (*o + sqd[i0 + 1] * z.y);
        }
    }
}

constexpr int kCholThreads = 512;
constexpr int kCholSmemMaxM = lu::kSmemMaxM;

// K = I + P (P symmetric positive semi-definite, m x m, ld ldp_in) factored without pivoting: step k scales column k by
// 1 / a_kk and updates the trailing rows, exactly lu_factor_kernel's elimination with the pivot fixed at row k.  The trailing
// matrix stays symmetric, so the pivots a_kk are G_kk^2 and the multipliers a_rk / a_kk are G_rk / G_kk.  Output in the lup
// layout of lu_solve_kernel: L = G diag(G)^-1 below the diagonal, diag(G) on it, zeros above, perm = identity.
// lpiv[k] = log a_kk = 2 log G_kk.  status[0] = 1 when a pivot is <= 0 (K is then not positive definite).
template <bool IN_SMEM>
__global__ void __launch_bounds__(kCholThreads) chol_factor_kernel(const double* __restrict__ P, long long ldp_in, int m,
                                                                   double* work_global, double* __restrict__ lup, long long ldl,
                                                                   int* __restrict__ perm, double* __restrict__ lpiv,
                                                                   int* __restrict__ status) {
    extern __shared__ __align__(16) unsigned char chol_smem_raw[];
    double* work = IN_SMEM ? reinterpret_cast<double*>(chol_smem_raw) : work_global;
    const long long ldw = lu::factor_ld(m, IN_SMEM);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nwarps_cta = kCholThreads / 32;
    const long long gtid = (long long)blockIdx.x * kCholThreads + tid;
    const long long gthreads = (long long)gridDim.x * kCholThreads;
    auto ld_w = [&](long long idx) -> double { return IN_SMEM ? work[idx] : __ldcg(work + idx); };
    auto st_w = [&](long long idx, double v) { if (IN_SMEM) work[idx] = v; else __stcg(work + idx, v); };
    auto sync_all = [&]() {
        if (IN_SMEM) __syncthreads();
        else cooperative_groups::this_grid().sync();
    };
    for (long long e = gtid; e < (long long)m * m; e += gthreads) {
        const int r = (int)(e / m), c = (int)(e % m);
        st_w(r * ldw + c, P[(long long)r * ldp_in + c] + (r == c ? 1.0 : 0.0));
    }
    sync_all();
    for (int k = 0; k < m; ++k) {
        const double piv = ld_w(k * ldw + k);
        if (!(piv > 0.0) && gtid == 0) status[0] = 1;
        const double pinv = 1.0 / piv;
        const long long prow = (long long)k * ldw;
        const int gw = blockIdx.x * nwarps_cta + warp, gws = gridDim.x * nwarps_cta;
        for (int r = k + 1 + gw; r < m; r += gws) {
            const long long row = (long long)r * ldw;
            const double l = ld_w(row + k) * pinv;
            for (int c = k + 1 + lane; c < m; c += 32) st_w(row + c, ld_w(row + c) - l * ld_w(prow + c));
            __syncwarp();
            if (lane == 0) st_w(row + k, l);
        }
        sync_all();
    }
    for (long long e = gtid; e < (long long)m * m; e += gthreads) {
        const int r = (int)(e / m), c = (int)(e % m);
        const double v = ld_w(r * ldw + c);
        lup[(long long)r * ldl + c] = c < r ? v : (c == r ? sqrt(v) : 0.0);
    }
    for (long long r = gtid; r < m; r += gthreads) {
        perm[r] = (int)r;
        lpiv[r] = log(ld_w(r * ldw + r));
    }
}

// logdet[0] = sum_i ldiag_i + sum_k lpiv_k (fixed order); scalars[0] = status (0 = positive definite), scalars[1] = logdet.
__global__ void __launch_bounds__(256) logdet_kernel(const double* __restrict__ ldiag, int n, const double* __restrict__ lpiv,
                                                     int m, const int* __restrict__ status, double* __restrict__ logdet,
                                                     double* __restrict__ scalars) {
    __shared__ double red[8];
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) a += ldiag[i];
    for (int k = threadIdx.x; k < m; k += 256) b += lpiv[k];
    a = block_sum_256(a, red);
    b = block_sum_256(b, red);
    if (threadIdx.x == 0) {
        const double v = a + b;
        logdet[0] = v;
        scalars[0] = (status[0] != 0 || status[1] != 0) ? 1.0 : 0.0;
        scalars[1] = v;
    }
}

// One CTA per row: out = x~ (fp64, ld = ldo, columns >= n zeroed) with standardize_kernel's per-element arithmetic in mode 0
// ('standard'; g() is never applied here), and ssq[r] = sum_i x~_ri^2 dinv_i.  Thread t owns the column groups 4t + 1024k
// whatever the load width (VEC: 16-byte loads), so the reduction order -- and the result -- depends on nothing but n.
// MASK (conditioning): a missing entry (NaN, or the marker when has_marker) is not imputed but set to 0 in out and left
// out of ssq; miss[r * n + 0 .. nmiss[r]) lists the missing columns in ascending order and miss[r * n + n - 1 - j] the j-th
// observed one; raw (optional, ld ldr) receives the observed entries as binary64.  An observed entry goes through exactly
// the arithmetic of MASK = false, so a complete row gives the same out and ssq bit for bit.
// FLAG (conditioning on a fixed column set, where no entry may be missing): a missing entry is zeroed and left out of ssq as
// with MASK, no lists are written, and raw[0] (one double) is set to 1.0.
template <typename T, bool VEC, bool MASK, bool FLAG = false>
__global__ void __launch_bounds__(256) score_standardize_kernel(const T* __restrict__ x, long long N, int n, long long ldx,
                                                                int has_marker, double marker, int marker_is_nan,
                                                                const double* __restrict__ impute, const double* __restrict__ mean,
                                                                const double* __restrict__ sd, const double* __restrict__ dinv,
                                                                double* __restrict__ out, long long ldo, double* __restrict__ ssq,
                                                                int* __restrict__ miss, int* __restrict__ nmiss,
                                                                double* __restrict__ raw, long long ldr) {
    __shared__ double red[8];
    __shared__ int wcount[8];
    const long long r = blockIdx.x;
    if (r >= N) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double acc = 0.0;
    int base = 0;  // missing entries in the chunks before this one (MASK)
    for (int c0 = 0; c0 < ldo; c0 += 256 * 4) {
        const int i0 = c0 + threadIdx.x * 4;
        double v[4] = {0.0, 0.0, 0.0, 0.0}, o[4];
        bool mis[4] = {false, false, false, false};
        if (i0 < ldo) {
            if (VEC && i0 + 3 < n) {
                load_row_vec<T, 4>(x + r * ldx + i0, v);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (i0 + j < n) v[j] = (double)x[r * ldx + i0 + j];
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int i = i0 + j;
                o[j] = 0.0;
                if ((MASK || FLAG) && i < n) mis[j] = (v[j] != v[j]) || (has_marker && !marker_is_nan && v[j] == marker);
                if (FLAG && mis[j]) raw[0] = 1.0;
                if (i < n && !mis[j]) {
                    o[j] = standardize_value(v[j], i, has_marker, marker, marker_is_nan, 0, impute, mean, sd);
                    acc += o[j] * o[j] * dinv[i];
                    if (MASK && raw) raw[r * ldr + i] = v[j];
                }
            }
            // ldo is a multiple of 16 doubles and i0 of 4: 16-byte stores
            *reinterpret_cast<double2*>(out + r * ldo + i0) = make_double2(o[0], o[1]);
            *reinterpret_cast<double2*>(out + r * ldo + i0 + 2) = make_double2(o[2], o[3]);
        }
        if (MASK) {  // block-wide exclusive scan of the missing counts: the lists come out in column order
            const int cnt = (int)mis[0] + (int)mis[1] + (int)mis[2] + (int)mis[3];
            int incl = cnt;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl += t;
            }
            if (lane == 31) wcount[warp] = incl;
            __syncthreads();
            int before = base + incl - cnt, total = 0;
            for (int w = 0; w < 8; ++w) {
                if (w < warp) before += wcount[w];
                total += wcount[w];
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int i = i0 + j;
                if (i >= n) break;
                if (mis[j]) miss[r * n + before++] = i;
                else miss[r * n + n - 1 - (i - before)] = i;
            }
            base += total;
            __syncthreads();
        }
    }
    acc = block_sum_256(acc, red);
    if (threadIdx.x == 0) {
        ssq[r] = acc;
        if (MASK) nmiss[r] = base;
    }
}

// One warp per row: maha = ssq - sum_j Y_rj^2 (fixed shuffle tree), logpdf = -(n log 2 pi + log det Sigma + maha) / 2.
__global__ void __launch_bounds__(256) score_finish_kernel(const double* __restrict__ y, long long ldy, const double* __restrict__ ssq,
                                                           long long N, int m, const double* __restrict__ logdet, double n_log_2pi,
                                                           double* __restrict__ maha, double* __restrict__ logpdf) {
    const long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= N) return;
    double a = 0.0;
    for (int j = lane; j < m; j += 32) {
        const double v = y[r * ldy + j];
        a += v * v;
    }
    a = warp_sum(a);
    if (lane == 0) {
        const double q = ssq[r] - a;
        maha[r] = q;
        logpdf[r] = -0.5 * (n_log_2pi + logdet[0] + q);
    }
}

// out (rows x ldc) holds rows [row0, row0 + rows) of B^T B; turned into the same rows of Sigma^-1.
__global__ void precision_finish_kernel(double* __restrict__ out, long long ldc, int row0, int rows, int n,
                                        const double* __restrict__ dinv, const double* __restrict__ sd) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    const int r = blockIdx.y;
    if (k < n && r < rows) {
        const int i = row0 + r;
        const double v = (i == k ? dinv[i] : 0.0) - out[(long long)r * ldc + k];
        out[(long long)r * ldc + k] = v / (sd[i] * sd[k]);
    }
}

// out (m x ldo) = I_m: the right-hand sides from which lu_solve_kernel forms G^-1 (for H = G^-1 G^-T)
__global__ void eye_kernel(double* __restrict__ out, long long ldo, int m) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
    if (c < m) out[(long long)r * ldo + c] = r == c ? 1.0 : 0.0;
}

// ---- conditioning on the observed entries (Corex.impute, score_samples(missing='marginalize')) --------------------------
// Row with missing set M (k = |M|) and observed set O, standardised space, x~° = x~ with the missing entries zeroed:
//   c = B x~° (m),  g = B_M^T c (k),  s° = sum_O x~_i^2 / Delta_i,   Lambda = Sigma~^-1 = Delta^-1 - B^T B
//   x^_M = Lambda_MM^-1 g,  q_O = s° - |c|^2 - g^T x^_M,
//   log det Sigma_OO = log det Sigma - 2 sum_M log sd_i + log det Lambda_MM.
// Path A (order k):  Lambda_MM = Delta_M^-1 - B_M^T B_M.
// Path B (order m):  E = H + sum_O Delta_i b_i b_i^T  (= I - sum_M Delta_i b_i b_i^T, formed from PSD terms only),
//   Lambda_MM^-1 g = Delta_M g + Delta_M B_M^T E^-1 B_M Delta_M g,  log det Lambda_MM = log det E - sum_M log Delta_i.
// The path with the smaller cost estimate wins; its order decides the size class (cond_class).
// kCondSample mode, with W = L D L^T the factor of the row's system (Lambda_MM for Path A, E for Path B):
//   Path A  var_a = sum_r (L^-1 e_a)_r^2 / d_r                        draw x^ + L^-T D^-1/2 eps
//   Path B  var_a = Delta_a + Delta_a^2 sum_r (L^-1 b_a)_r^2 / d_r     draw x^ + Delta_M^1/2 eps1 + Delta_M B_M^T L^-T D^-1/2 eps2
// (Cov of the Path B draw: Delta_M + Delta_M B_M^T E^-1 B_M Delta_M = Lambda_MM^-1.)  A row with nothing observed solves E = H,
// Path B with O empty: std 1 in standardised units, unconditional draws.  eps: tag-1 normals of stream (row, draw), columns
// 0..k-1 over the missing columns in ascending order, then (Path B) k..k+m-1 for eps2.
constexpr int kCondThreads = 256;
constexpr int kCondChunk = 16;       // gathered vectors staged per pass of the matrix build
constexpr int kCondSmallMax = 64;    // class 1: the order-p matrix in shared memory, several CTAs per SM
constexpr int kCondSmemMax = 160;    // class 2: one CTA per SM, p (p|1) + kCondChunk p doubles <= 227 KB
enum CondCount { kCountTrivial = 0, kCountSmall, kCountSmem, kCountGlobal, kCountPathA, kCountPathB, kCondCounts = 8 };
enum CondMode { kCondMean = 0, kCondSample = 1 };  // mean (+ q_O, log p); mean + optional std and draws

__host__ __device__ inline bool cond_path_a(long long k, long long n, long long m) {
    const double a = (double)k * k * m + (double)k * k * k / 3.0;
    const double b = (double)(n - k) * m * m + (double)m * m * m / 3.0;
    return a <= b;
}
// order of the system a row with k of n entries missing solves (0: nothing to solve); in kCondSample mode a row with nothing
// observed solves E = H, of order m
__host__ __device__ inline int cond_order(int k, int n, int m, bool sample = false) {
    if (k == 0) return 0;
    if (k == n) return sample ? m : 0;
    return cond_path_a(k, n, m) ? k : m;
}
__host__ __device__ inline int cond_class(int p) {
    return p == 0 ? kCountTrivial : p <= kCondSmallMax ? kCountSmall : p <= kCondSmemMax ? kCountSmem : kCountGlobal;
}
__host__ __device__ inline long long cond_matrix_doubles(int p) { return (long long)p * (p | 1) + (long long)kCondChunk * p; }

// In-place solve of W v = rhs for W = L D L^T as left by the elimination (multipliers below the diagonal, pivots on it).
// Every v_r is updated in a fixed order (columns ascending, then descending).  Returns sum_r y_r^2 / d_r (y = L^-1 rhs),
// which is rhs^T W^-1 rhs, on every thread.
__device__ __forceinline__ double cond_ldl_solve(const double* W, int ldw, int p, double* v, double* red) {
    const int tid = threadIdx.x;
    for (int c = 0; c < p; ++c) {
        const double yc = v[c];
        for (int r = c + 1 + tid; r < p; r += kCondThreads) v[r] -= W[(long long)r * ldw + c] * yc;
        __syncthreads();
    }
    double quad = 0.0;
    for (int r = tid; r < p; r += kCondThreads) {
        const double y = v[r], d = W[(long long)r * ldw + r];
        quad += y * y / d;
        v[r] = y / d;
    }
    quad = block_sum_256(quad, red);
    for (int c = p - 1; c > 0; --c) {
        const double xc = v[c];
        for (int r = tid; r < c; r += kCondThreads) v[r] -= W[(long long)c * ldw + r] * xc;
        __syncthreads();
    }
    return quad;
}

// V[t] <- L^-1 V[t] for the kCondChunk right-hand sides V[t] = V + t p, L the unit lower factor in W; V[t]_r = 0 for r < c0.
// The caller synchronises before.
__device__ __forceinline__ void cond_fwd_chunk(const double* W, int ldw, int p, double* V, int c0) {
    for (int c = c0; c < p - 1; ++c) {
        double vc[kCondChunk];
#pragma unroll
        for (int t = 0; t < kCondChunk; ++t) vc[t] = V[(long long)t * p + c];
        for (int r = c + 1 + threadIdx.x; r < p; r += kCondThreads) {
            const double l = W[(long long)r * ldw + c];
#pragma unroll
            for (int t = 0; t < kCondChunk; ++t) V[(long long)t * p + r] -= l * vc[t];
        }
        __syncthreads();
    }
}

// V[t] <- L^-T V[t] for the kCondChunk right-hand sides.  The caller synchronises before.
__device__ __forceinline__ void cond_back_chunk(const double* W, int ldw, int p, double* V) {
    for (int c = p - 1; c > 0; --c) {
        double vc[kCondChunk];
#pragma unroll
        for (int t = 0; t < kCondChunk; ++t) vc[t] = V[(long long)t * p + c];
        for (int r = threadIdx.x; r < c; r += kCondThreads) {
            const double l = W[(long long)c * ldw + r];
#pragma unroll
            for (int t = 0; t < kCondChunk; ++t) V[(long long)t * p + r] -= l * vc[t];
        }
        __syncthreads();
    }
}

// One CTA per row of the rows whose order lies in [pmin, pmax] (persistent grid, rows blockIdx.x + t gridDim.x).
// IN_SMEM: the order-p matrix and the staged vectors in dynamic shared memory; otherwise in this CTA's slab of `slabs`
// (slab_doubles each).  vec (ld ldv): the row of x~° on entry, g and then x^_M on exit; y (ld ldy): c on entry, Path B's
// B_M Delta_M g and E^-1 of it on exit.  Outputs optional: xout (ld ldxo) receives mean + sd x^ at the missing columns,
// maha / logpdf q_O and log p(x_O).  counts (kCondCounts) += rows per class and per path.
// MODE == kCondSample (maha, logpdf and logdet unused; xout required): sdo (optional, ld ldo, zero on entry) receives sd sqrt(var)
// at the missing columns; draws (optional) n_draws completed rows per row, draw d of row r at draws + d draw_stride + r ldo,
// drawn from stream (seed, 1, row0 + r, d).
template <bool IN_SMEM, int MODE = kCondMean>
__global__ void __launch_bounds__(kCondThreads) condition_rows_kernel(
    const int* __restrict__ miss, const int* __restrict__ nmiss, long long N, int n, int m, const double* __restrict__ b,
    long long ldb, const double* __restrict__ h, long long ldh, const double* __restrict__ dinv, const double* __restrict__ mean,
    const double* __restrict__ sd, const double* __restrict__ logdet, double log_2pi, const double* __restrict__ ssq, double* vec,
    long long ldv, double* y, long long ldy, int pmin, int pmax, double* slabs, long long slab_doubles, double* __restrict__ xout,
    long long ldxo, double* __restrict__ maha, double* __restrict__ logpdf, unsigned long long* __restrict__ counts,
    double* __restrict__ sdo, double* __restrict__ draws, long long ldo, long long draw_stride, unsigned long long seed,
    long long row0, int n_draws) {
    constexpr bool SAMPLE = MODE == kCondSample;
    extern __shared__ __align__(16) unsigned char cond_smem_raw[];
    __shared__ double red[8];
    __shared__ double wt[kCondChunk];
    __shared__ double s_c2;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double* work = IN_SMEM ? reinterpret_cast<double*>(cond_smem_raw) : slabs + (long long)blockIdx.x * slab_doubles;
    for (long long r = blockIdx.x; r < N; r += gridDim.x) {
        const int k = nmiss[r];
        const int p = cond_order(k, n, m, SAMPLE);
        if (p < pmin || p > pmax) continue;
        const int* ml = miss + r * n;
        double* g = vec + r * ldv;
        double* c = y + r * ldy;
        if (warp == 0) {  // |c|^2 exactly as score_finish_kernel sums |Y_r|^2
            double a = 0.0;
            for (int j = lane; j < m; j += 32) {
                const double v = c[j];
                a += v * v;
            }
            a = warp_sum(a);
            if (lane == 0) s_c2 = a;
        }
        __syncthreads();
        const double c2 = s_c2;
        double q = 0.0, lp = 0.0;
        if (k == 0) {  // complete row: score_finish_kernel's arithmetic
            if constexpr (!SAMPLE) {
                q = ssq[r] - c2;
                lp = -0.5 * (__dmul_rn((double)n, log_2pi) + logdet[0] + q);  // the host's n log 2 pi: no contraction into an fma
            }
        } else if (k == n && !SAMPLE) {  // nothing observed: x^ = 0, log p = 0
            if (xout)
                for (int i = tid; i < n; i += kCondThreads) xout[r * ldxo + i] = mean[i];
        } else {
            bool path_a = p == k;
            if constexpr (SAMPLE) path_a = path_a && k < n;  // nothing observed: Path B with O empty, even when m = n
            // g = B_M^T c, and the fixed-order sums of log sd_i and -log Delta_i over M
            double lsd = 0.0, ldel = 0.0;
            for (int a = tid; a < k; a += kCondThreads) {
                const int i = ml[a];
                double acc = 0.0;
                for (int j = 0; j < m; ++j) acc += b[(long long)j * ldb + i] * c[j];
                g[a] = acc;
                lsd += log(sd[i]);
                ldel += log(dinv[i]);  // -log Delta_i
            }
            lsd = block_sum_256(lsd, red);
            ldel = block_sum_256(ldel, red);
            // the order-p matrix: lower triangle of D0 + sum_t w_t u_t u_t^T, then mirrored
            const int ldw = p | 1;
            double* W = work;
            double* U = work + (long long)p * ldw;
            for (long long e = tid; e < (long long)p * p; e += kCondThreads) {
                const int rr = (int)(e / p), cc = (int)(e % p);
                W[(long long)rr * ldw + cc] = path_a ? (rr == cc ? dinv[ml[rr]] : 0.0) : h[(long long)rr * ldh + cc];
            }
            const int T = path_a ? m : n - k;  // Path A: the m rows of B_M; Path B: the observed columns of B
            for (int t0 = 0; t0 < T; t0 += kCondChunk) {
                __syncthreads();
                if (tid < kCondChunk) {
                    const int t = t0 + tid;
                    wt[tid] = t >= T ? 0.0 : (path_a ? -1.0 : 1.0 / dinv[ml[n - 1 - t]]);
                }
                for (int e = tid; e < kCondChunk * p; e += kCondThreads) {
                    double u = 0.0;
                    if (path_a) {
                        const int t = e / p, a = e % p;
                        if (t0 + t < T) u = b[(long long)(t0 + t) * ldb + ml[a]];
                        U[(long long)t * p + a] = u;
                    } else {  // consecutive threads read consecutive observed columns of one factor row
                        const int t = e % kCondChunk, j = e / kCondChunk;
                        if (t0 + t < T) u = b[(long long)j * ldb + ml[n - 1 - (t0 + t)]];
                        U[(long long)t * p + j] = u;
                    }
                }
                __syncthreads();
                for (int rr = warp; rr < p; rr += kCondThreads / 32) {
                    double wu[kCondChunk];
#pragma unroll
                    for (int t = 0; t < kCondChunk; ++t) wu[t] = wt[t] * U[(long long)t * p + rr];
                    for (int cc = lane; cc <= rr; cc += 32) {
                        double acc = W[(long long)rr * ldw + cc];
#pragma unroll
                        for (int t = 0; t < kCondChunk; ++t) acc = fma(wu[t], U[(long long)t * p + cc], acc);
                        W[(long long)rr * ldw + cc] = acc;
                    }
                }
            }
            __syncthreads();
            for (long long e = tid; e < (long long)p * p; e += kCondThreads) {
                const int rr = (int)(e / p), cc = (int)(e % p);
                if (cc > rr) W[(long long)rr * ldw + cc] = W[(long long)cc * ldw + rr];
            }
            __syncthreads();
            // unpivoted elimination (chol_factor_kernel's): pivots d_k on the diagonal, multipliers below it
            double ldet = 0.0;
            for (int kk = 0; kk < p; ++kk) {
                const double piv = W[(long long)kk * ldw + kk];
                ldet += log(piv);
                const double pinv = 1.0 / piv;
                const long long prow = (long long)kk * ldw;
                for (int rr = kk + 1 + warp; rr < p; rr += kCondThreads / 32) {
                    const long long row = (long long)rr * ldw;
                    const double l = W[row + kk] * pinv;
                    for (int cc = kk + 1 + lane; cc < p; cc += 32) W[row + cc] -= l * W[prow + cc];
                    __syncwarp();
                    if (lane == 0) W[row + kk] = l;
                }
                __syncthreads();
            }
            double gx;
            if (path_a) {
                gx = cond_ldl_solve(W, ldw, p, g, red);  // g <- Lambda_MM^-1 g; g^T x^ = g^T Lambda_MM^-1 g
            } else {
                // c <- B_M Delta_M g, then E^-1 of it
                for (int j = tid; j < m; j += kCondThreads) {
                    double acc = 0.0;
                    for (int a = 0; a < k; ++a) acc += b[(long long)j * ldb + ml[a]] * (g[a] / dinv[ml[a]]);
                    c[j] = acc;
                }
                __syncthreads();
                cond_ldl_solve(W, ldw, p, c, red);
                double part = 0.0;
                for (int a = tid; a < k; a += kCondThreads) {
                    const int i = ml[a];
                    double acc = g[a];
                    for (int j = 0; j < m; ++j) acc += b[(long long)j * ldb + i] * c[j];
                    const double xh = acc / dinv[i];
                    part += g[a] * xh;
                    g[a] = xh;
                }
                gx = block_sum_256(part, red);
                ldet += ldel;
            }
            q = ssq[r] - c2 - gx;
            if constexpr (!SAMPLE) lp = -0.5 * (__dmul_rn((double)(n - k), log_2pi) + (logdet[0] - 2.0 * lsd + ldet) + q);
            if (xout)
                for (int a = tid; a < k; a += kCondThreads) {
                    const int i = ml[a];
                    xout[r * ldxo + i] = mean[i] + sd[i] * g[a];
                }
            if constexpr (SAMPLE) {
                double* V = work + (long long)p * ldw;  // the staging area of the build: kCondChunk right-hand sides of length p
                if (sdo)
                    for (int a0 = 0; a0 < k; a0 += kCondChunk) {
                        const int nb = min(kCondChunk, k - a0);
                        __syncthreads();
                        for (int e = tid; e < kCondChunk * p; e += kCondThreads) {
                            double u = 0.0;
                            if (path_a) {  // e_a
                                const int t = e / p, rr = e % p;
                                if (t < nb && rr == a0 + t) u = 1.0;
                                V[(long long)t * p + rr] = u;
                            } else {  // b_a: consecutive threads read consecutive missing columns of one factor row
                                const int t = e % kCondChunk, j = e / kCondChunk;
                                if (t < nb) u = b[(long long)j * ldb + ml[a0 + t]];
                                V[(long long)t * p + j] = u;
                            }
                        }
                        __syncthreads();
                        cond_fwd_chunk(W, ldw, p, V, path_a ? a0 : 0);
                        for (int t = warp; t < nb; t += kCondThreads / 32) {
                            double acc = 0.0;
                            for (int rr = lane; rr < p; rr += 32) {
                                const double v = V[(long long)t * p + rr];
                                acc += v * v / W[(long long)rr * ldw + rr];
                            }
                            acc = warp_sum(acc);
                            if (lane == 0) {
                                const int i = ml[a0 + t];
                                double var = acc;
                                if (!path_a) {
                                    const double dl = 1.0 / dinv[i];
                                    var = dl + dl * dl * acc;
                                }
                                sdo[r * ldo + i] = sd[i] * sqrt(var);
                            }
                        }
                    }
                if (draws) {
                    const long long grow = row0 + r;
                    const int j0 = path_a ? 0 : k;  // eps (Path A) or eps2 (Path B)
                    for (int d0 = 0; d0 < n_draws; d0 += kCondChunk) {
                        const int nd = min(kCondChunk, n_draws - d0);
                        __syncthreads();
                        for (int e = tid; e < kCondChunk * p; e += kCondThreads) {  // D^-1/2 eps of draw d0 + t
                            const int t = e / p, rr = e % p;
                            V[e] = t < nd ? normal_at(seed, 1, grow, d0 + t, j0 + rr) / sqrt(W[(long long)rr * ldw + rr]) : 0.0;
                        }
                        __syncthreads();
                        cond_back_chunk(W, ldw, p, V);
                        for (int a = tid; a < k; a += kCondThreads) {
                            const int i = ml[a];
                            double bv[kCondChunk];  // Path B: (B_M^T L^-T D^-1/2 eps2)_a, factors summed in index order
#pragma unroll
                            for (int t = 0; t < kCondChunk; ++t) bv[t] = 0.0;
                            if (!path_a)
                                for (int j = 0; j < m; ++j) {
                                    const double bj = b[(long long)j * ldb + i];
#pragma unroll
                                    for (int t = 0; t < kCondChunk; ++t) bv[t] += bj * V[(long long)t * p + j];
                                }
                            const double dl = 1.0 / dinv[i];
#pragma unroll
                            for (int t = 0; t < kCondChunk; ++t) {
                                if (t >= nd) break;
                                const double v = path_a ? V[(long long)t * p + a]
                                                        : sqrt(dl) * normal_at(seed, 1, grow, d0 + t, a) + dl * bv[t];
                                draws[(d0 + t) * draw_stride + r * ldo + i] = mean[i] + sd[i] * (g[a] + v);
                            }
                        }
                    }
                }
            }
            if (tid == 0 && counts) atomicAdd(counts + (path_a ? kCountPathA : kCountPathB), 1ULL);
        }
        if constexpr (SAMPLE) {  // observed entries of every draw: the input's binary64, as xout holds it
            if (draws && k < n)
                for (long long e = tid; e < (long long)n_draws * (n - k); e += kCondThreads) {
                    const int d = (int)(e / (n - k)), i = ml[n - 1 - (int)(e % (n - k))];
                    draws[d * draw_stride + r * ldo + i] = xout[r * ldxo + i];
                }
        }
        if (tid == 0) {
            if (maha) maha[r] = q;
            if (logpdf) logpdf[r] = lp;
            if (counts) atomicAdd(counts + cond_class(p), 1ULL);
        }
        __syncthreads();
    }
}

// ---- conditioning on a fixed column set (ConditionalGaussian) -----------------------------------------------------------
// Observed columns O, targets T (disjoint), standardised space, Sigma~ = Z^T Z + Delta:
//   E_O = I + Z_O Delta_O^-1 Z_O^T = L L^T,   A = L^-1 Z_O Delta_O^-1 (m x |O|),   P = L^-1 Z_T (m x |T|)
//   v = A x~_O,  E[x~_T | x~_O] = P^T v,  Cov[x~_T | x~_O] = Delta_T + P^T P,  q_O = sum_O x~_i^2 / Delta_i - |v|^2,
//   log det Sigma_OO = sum_O (2 log sd_i + log Delta_i) + 2 sum_k log L_kk,   draw x~_T = P^T (v + u) + Delta_T^1/2 eps.
// E_O - I, its factor, the sweeps for A and P and log det are lcx_lowrank_factor's pieces run on the gathered columns.

// One thread per selected column: t < no is observed column obs[t], t >= no target column tgt[t - no].  Observed: zh, zd (m x
// ldo) = Z_O Delta_O^-1/2, Z_O Delta_O^-1 (factor_prep_kernel's arithmetic), ocols = [theta0_O | theta1_O | 1/Delta_O] (rows of
// no), ldiag = 2 log sd + log Delta.  Targets: zt (m x ldt) = Z_T, tcols rows 0..3 of nt = [theta0_T | theta1_T | Delta_T |
// sqrt(Delta_T)].  status[1] = 1 when a selected Delta_i <= 0; scalars[2] = 1 when an index lies outside [0, n).
__global__ void given_prep_kernel(const double* __restrict__ rinv, const double* __restrict__ si, long long ldr, int m, int n,
                                  double inv_sqrt_scale, const double* __restrict__ mean, const double* __restrict__ sd,
                                  const int* __restrict__ obs, int no, const int* __restrict__ tgt, int nt, double* __restrict__ zh,
                                  double* __restrict__ zd, long long ldo, double* __restrict__ ocols, double* __restrict__ ldiag,
                                  double* __restrict__ zt, long long ldt, double* __restrict__ tcols, int* __restrict__ status,
                                  double* __restrict__ scalars) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= no + nt) return;
    const bool is_obs = t < no;
    const int a = is_obs ? t : t - no;
    const int i = is_obs ? obs[a] : tgt[a];
    if (i < 0 || i >= n) {
        scalars[2] = 1.0;
        return;
    }
    const double c = 1.0 + si[i];
    const double delta = lowrank_delta(rinv, ldr, m, i, c, inv_sqrt_scale);
    if (!(delta > 0.0)) status[1] = 1;
    if (is_obs) {
        const double di = 1.0 / delta, rs = sqrt(di);
        ocols[a] = mean[i];
        ocols[no + a] = sd[i];
        ocols[2 * no + a] = di;
        ldiag[a] = 2.0 * log(sd[i]) + log(delta);
        for (int j = 0; j < m; ++j) {
            const double z = lowrank_z(rinv, ldr, j, i, c, inv_sqrt_scale);
            zh[(long long)j * ldo + a] = z * rs;
            zd[(long long)j * ldo + a] = z * di;
        }
    } else {
        tcols[a] = mean[i];
        tcols[nt + a] = sd[i];
        tcols[2 * nt + a] = delta;
        tcols[3 * nt + a] = sqrt(delta);
        for (int j = 0; j < m; ++j) zt[(long long)j * ldt + a] = lowrank_z(rinv, ldr, j, i, c, inv_sqrt_scale);
    }
}

// tcols row 4 = theta1_t sqrt(Delta_t + sum_k P_kt^2) (k ascending), one thread per target
__global__ void given_std_kernel(const double* __restrict__ p, long long ldp, int m, int nt, double* __restrict__ tcols) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nt) return;
    double acc = 0.0;
    for (int k = 0; k < m; ++k) {
        const double v = p[(long long)k * ldp + t];
        acc += v * v;
    }
    tcols[4 * nt + t] = tcols[nt + t] * sqrt(tcols[2 * nt + t] + acc);
}

// out (rows x ldo) holds V P on entry and theta0_T + theta1_T (V P) on exit
__global__ void __launch_bounds__(256) given_mean_finish_kernel(double* __restrict__ out, long long ldo, long long rows, int nt,
                                                                const double* __restrict__ tcols) {
    for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < rows * nt; e += (long long)gridDim.x * 256) {
        const long long r = e / nt;
        const int t = (int)(e % nt);
        double* o = out + r * ldo + t;
        *o = tcols[t] + tcols[nt + t] * *o;
    }
}

// out (rows x ldc) holds rows [row0, row0 + rows) of P^T P; turned into the same rows of theta1_T (Delta_T + P^T P) theta1_T
__global__ void given_cov_finish_kernel(double* __restrict__ out, long long ldc, int row0, int rows, int nt,
                                        const double* __restrict__ tcols) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    const int r = blockIdx.y;
    if (k < nt && r < rows) {
        const int i = row0 + r;
        const double v = (i == k ? tcols[2 * nt + i] : 0.0) + out[(long long)r * ldc + k];
        out[(long long)r * ldc + k] = v * (tcols[nt + i] * tcols[nt + k]);
    }
}

}  // namespace lowrank
}  // namespace lcx
