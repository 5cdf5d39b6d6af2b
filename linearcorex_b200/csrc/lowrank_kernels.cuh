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
//                         order-p system of Path A or B in shared memory (p <= 160) or in a per-CTA global slab
#pragma once
#include "common.cuh"
#include "lu_solve.cuh"
#include "preprocess_kernels.cuh"

namespace lcx {
namespace lowrank {

// One thread per variable i; the m factors are summed in index order.  rinv: ld ldr; zh, zd: ld ldz.  status[1] = 1 when some
// Delta_i <= 0 (Sigma is then not treated as positive definite).
__global__ void factor_prep_kernel(const double* __restrict__ rinv, const double* __restrict__ si, long long ldr, long long ldz,
                                   int m, int n, double inv_sqrt_scale, const double* __restrict__ sd, double* __restrict__ zh,
                                   double* __restrict__ zd, double* __restrict__ dinv, double* __restrict__ ldiag,
                                   int* __restrict__ status) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double c = 1.0 + si[i];
    double acc = 0.0;
    for (int j = 0; j < m; ++j) {
        const double z = rinv[(long long)j * ldr + i] / c * inv_sqrt_scale;
        acc += z * z;
    }
    const double delta = 1.0 - acc;
    if (!(delta > 0.0)) status[1] = 1;
    const double di = 1.0 / delta, rs = sqrt(di);
    dinv[i] = di;
    ldiag[i] = 2.0 * log(sd[i]) + log(delta);
    for (int j = 0; j < m; ++j) {
        const double z = rinv[(long long)j * ldr + i] / c * inv_sqrt_scale;
        zh[(long long)j * ldz + i] = z * rs;
        zd[(long long)j * ldz + i] = z * di;
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
template <typename T, bool VEC, bool MASK>
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
                if (MASK && i < n) mis[j] = (v[j] != v[j]) || (has_marker && !marker_is_nan && v[j] == marker);
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
constexpr int kCondThreads = 256;
constexpr int kCondChunk = 16;       // gathered vectors staged per pass of the matrix build
constexpr int kCondSmallMax = 64;    // class 1: the order-p matrix in shared memory, several CTAs per SM
constexpr int kCondSmemMax = 160;    // class 2: one CTA per SM, p (p|1) + kCondChunk p doubles <= 227 KB
enum CondCount { kCountTrivial = 0, kCountSmall, kCountSmem, kCountGlobal, kCountPathA, kCountPathB, kCondCounts = 8 };

__host__ __device__ inline bool cond_path_a(long long k, long long n, long long m) {
    const double a = (double)k * k * m + (double)k * k * k / 3.0;
    const double b = (double)(n - k) * m * m + (double)m * m * m / 3.0;
    return a <= b;
}
// order of the system a row with k of n entries missing solves (0: nothing to solve)
__host__ __device__ inline int cond_order(int k, int n, int m) {
    if (k == 0 || k == n) return 0;
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

// One CTA per row of the rows whose order lies in [pmin, pmax] (persistent grid, rows blockIdx.x + t gridDim.x).
// IN_SMEM: the order-p matrix and the staged vectors in dynamic shared memory; otherwise in this CTA's slab of `slabs`
// (slab_doubles each).  vec (ld ldv): the row of x~° on entry, g and then x^_M on exit; y (ld ldy): c on entry, Path B's
// B_M Delta_M g and E^-1 of it on exit.  Outputs optional: xout (ld ldxo) receives mean + sd x^ at the missing columns,
// maha / logpdf q_O and log p(x_O).  counts (kCondCounts) += rows per class and per path.
template <bool IN_SMEM>
__global__ void __launch_bounds__(kCondThreads) condition_rows_kernel(
    const int* __restrict__ miss, const int* __restrict__ nmiss, long long N, int n, int m, const double* __restrict__ b,
    long long ldb, const double* __restrict__ h, long long ldh, const double* __restrict__ dinv, const double* __restrict__ mean,
    const double* __restrict__ sd, const double* __restrict__ logdet, double log_2pi, const double* __restrict__ ssq, double* vec,
    long long ldv, double* y, long long ldy, int pmin, int pmax, double* slabs, long long slab_doubles, double* __restrict__ xout,
    long long ldxo, double* __restrict__ maha, double* __restrict__ logpdf, unsigned long long* __restrict__ counts) {
    extern __shared__ __align__(16) unsigned char cond_smem_raw[];
    __shared__ double red[8];
    __shared__ double wt[kCondChunk];
    __shared__ double s_c2;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double* work = IN_SMEM ? reinterpret_cast<double*>(cond_smem_raw) : slabs + (long long)blockIdx.x * slab_doubles;
    for (long long r = blockIdx.x; r < N; r += gridDim.x) {
        const int k = nmiss[r];
        const int p = cond_order(k, n, m);
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
            q = ssq[r] - c2;
            lp = -0.5 * (__dmul_rn((double)n, log_2pi) + logdet[0] + q);  // the host's n log 2 pi: no contraction into an fma
        } else if (k == n) {  // nothing observed: x^ = 0, log p = 0
            if (xout)
                for (int i = tid; i < n; i += kCondThreads) xout[r * ldxo + i] = mean[i];
        } else {
            const bool path_a = p == k;
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
            lp = -0.5 * (__dmul_rn((double)(n - k), log_2pi) + (logdet[0] - 2.0 * lsd + ldet) + q);
            if (xout)
                for (int a = tid; a < k; a += kCondThreads) {
                    const int i = ml[a];
                    xout[r * ldxo + i] = mean[i] + sd[i] * g[a];
                }
            if (tid == 0 && counts) atomicAdd(counts + (path_a ? kCountPathA : kCountPathB), 1ULL);
        }
        if (tid == 0) {
            if (maha) maha[r] = q;
            if (logpdf) logpdf[r] = lp;
            if (counts) atomicAdd(counts + cond_class(p), 1ULL);
        }
        __syncthreads();
    }
}

}  // namespace lowrank
}  // namespace lcx
