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
template <typename T, bool VEC>
__global__ void __launch_bounds__(256) score_standardize_kernel(const T* __restrict__ x, long long N, int n, long long ldx,
                                                                int has_marker, double marker, int marker_is_nan,
                                                                const double* __restrict__ impute, const double* __restrict__ mean,
                                                                const double* __restrict__ sd, const double* __restrict__ dinv,
                                                                double* __restrict__ out, long long ldo, double* __restrict__ ssq) {
    __shared__ double red[8];
    const long long r = blockIdx.x;
    if (r >= N) return;
    double acc = 0.0;
    for (int i0 = threadIdx.x * 4; i0 < ldo; i0 += 256 * 4) {
        double v[4] = {0.0, 0.0, 0.0, 0.0}, o[4];
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
            if (i < n) {
                o[j] = standardize_value(v[j], i, has_marker, marker, marker_is_nan, 0, impute, mean, sd);
                acc += o[j] * o[j] * dinv[i];
            }
        }
        // ldo is a multiple of 16 doubles and i0 of 4: 16-byte stores
        *reinterpret_cast<double2*>(out + r * ldo + i0) = make_double2(o[0], o[1]);
        *reinterpret_cast<double2*>(out + r * ldo + i0 + 2) = make_double2(o[2], o[3]);
    }
    acc = block_sum_256(acc, red);
    if (threadIdx.x == 0) ssq[r] = acc;
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

}  // namespace lowrank
}  // namespace lcx
