// m x m linear solves of the details path: X = A^-1 B for the n right-hand sides of
//   X_i Z_j = np.linalg.solve(ry, rho).T            (linearcorex.py:280)
//   X_i Z_j = np.linalg.solve(cy, X_i Y_j^T).T      (linearcorex.py:366)
// done the way LAPACK's dgesv does them -- LU with partial pivoting (first largest |a_rk|), then the two triangular
// solves -- instead of forming an inverse.  A zero pivot sets the status word; the caller turns it into the error numpy
// raises there (LinAlgError: Singular matrix).
//
//   lu_factor_kernel<true>   one CTA, the matrix in shared memory (m <= 160: every fit of the synergy variant calls this
//                            once per iteration with m ~ 10, so latency is what matters)
//   lu_factor_kernel<false>  cooperative grid (up to 64 CTAs), the matrix in L2, ONE grid-wide barrier per pivot step:
//                            rows are never swapped physically (an index list is), so during step k the pivot row is
//                            read-only and every other active row is owned by exactly one warp.  m = 500: ~1.5 ms
//                            against ~50 ms for the single-CTA Gauss-Jordan it replaces.
//   lu_solve_kernel          one CTA per 32 right-hand sides: the m x 32 tile lives in shared memory (m <= 832; in place
//                            in the output beyond that) through both sweeps; rows of L / U are fetched with one
//                            coalesced load per 32 multiply-adds and broadcast by shuffle.
#pragma once
#include <cooperative_groups.h>

#include "common.cuh"

namespace lcx {
namespace lu {

namespace cg = cooperative_groups;

constexpr int kFactorThreads = 512;
constexpr int kSmemMaxM = 160;    // m*(m|1) doubles must fit in 227 KB of shared memory
constexpr int kSolveCols = 32;
constexpr int kSolveRows = 8;     // row groups (warps) of the solve kernel
constexpr int kSolveSmemMaxM = 832;

__host__ __device__ inline long long factor_ld(int m, bool in_smem) { return in_smem ? (m | 1) : (long long)((m + 1) & ~1); }

// LU = P A with unit lower L below the diagonal and U on and above it, rows in pivot order; perm[k] = source row of row k.
// status[0] = 1 if a pivot was exactly zero (numpy: LinAlgError), else 0.
template <bool IN_SMEM>
__global__ void __launch_bounds__(kFactorThreads) lu_factor_kernel(const double* __restrict__ A, long long lda, int m,
                                                                 double* work_global, double* __restrict__ lup, long long ldp,
                                                                 int* __restrict__ perm, int* __restrict__ status) {
    extern __shared__ __align__(16) unsigned char lu_smem_raw[];
    __shared__ double red_val[kFactorThreads / 32];
    __shared__ int red_idx[kFactorThreads / 32];
    __shared__ double s_pinv;
    __shared__ int s_prow;
    int* list = reinterpret_cast<int*>(lu_smem_raw);                                      // m ints
    double* work = IN_SMEM ? reinterpret_cast<double*>(lu_smem_raw + (((size_t)m * 4 + 15) & ~(size_t)15)) : work_global;
    const long long ldw = factor_ld(m, IN_SMEM);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nwarps_cta = kFactorThreads / 32;
    const long long gtid = (long long)blockIdx.x * kFactorThreads + tid;
    const long long gthreads = (long long)gridDim.x * kFactorThreads;
    auto ld_w = [&](long long idx) -> double { return IN_SMEM ? work[idx] : __ldcg(work + idx); };
    auto st_w = [&](long long idx, double v) { if (IN_SMEM) work[idx] = v; else __stcg(work + idx, v); };
    auto sync_all = [&]() {
        if (IN_SMEM) __syncthreads();
        else cg::this_grid().sync();
    };
    for (long long e = gtid; e < (long long)m * m; e += gthreads) {
        const int r = (int)(e / m), c = (int)(e % m);
        st_w(r * ldw + c, A[(long long)r * lda + c]);
    }
    for (int r = tid; r < m; r += kFactorThreads) list[r] = r;
    if (gtid == 0) status[0] = 0;
    sync_all();
    for (int k = 0; k < m; ++k) {
        // ---- pivot: first largest |a_rk| over the active rows (every CTA finds it for itself) ----
        double best = -1.0;
        int bi = k;
        for (int r = k + tid; r < m; r += kFactorThreads) {
            const double v = fabs(ld_w(list[r] * ldw + k));
            if (v > best) { best = v; bi = r; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
        }
        if (lane == 0) { red_val[warp] = best; red_idx[warp] = bi; }
        __syncthreads();
        if (tid == 0) {
            double b = red_val[0];
            int ix = red_idx[0];
            for (int w = 1; w < nwarps_cta; ++w)
                if (red_val[w] > b || (red_val[w] == b && red_idx[w] < ix)) { b = red_val[w]; ix = red_idx[w]; }
            const int t = list[k];
            list[k] = list[ix];
            list[ix] = t;
            const double piv = ld_w(list[k] * ldw + k);
            if (!(b > 0.0) && blockIdx.x == 0) status[0] = 1;
            s_pinv = 1.0 / piv;
            s_prow = list[k];
        }
        __syncthreads();
        // ---- eliminate column k from the active rows: one warp per row ----
        const double pinv = s_pinv;
        const long long prow = (long long)s_prow * ldw;
        const int gw = blockIdx.x * nwarps_cta + warp, gws = gridDim.x * nwarps_cta;
        for (int r = k + 1 + gw; r < m; r += gws) {
            const long long row = (long long)list[r] * ldw;
            const double l = ld_w(row + k) * pinv;
            for (int c = k + 1 + lane; c < m; c += 32) st_w(row + c, ld_w(row + c) - l * ld_w(prow + c));
            __syncwarp();
            if (lane == 0) st_w(row + k, l);
        }
        sync_all();
    }
    // rows in pivot order
    for (long long e = gtid; e < (long long)m * m; e += gthreads) {
        const int r = (int)(e / m), c = (int)(e % m);
        lup[(long long)r * ldp + c] = ld_w(list[r] * ldw + c);
    }
    if (blockIdx.x == 0)
        for (int r = tid; r < m; r += kFactorThreads) perm[r] = list[r];
}

// X[:, col0:col0+32] = U^-1 L^-1 B[perm, col0:col0+32].  IN_SMEM: X may alias B (a CTA reads its whole tile before it
// writes); otherwise the tile is worked on in place in X and X must not alias B.
// status_out (optional): the factorisation's status word as a double, for the host mailbox.
template <bool IN_SMEM>
__global__ void __launch_bounds__(kSolveCols* kSolveRows) lu_solve_kernel(const double* __restrict__ lup, long long ldp,
                                                                        const int* __restrict__ perm, int m,
                                                                        const double* B, long long ldb, double* X,
                                                                        long long ldx, int n, const int* __restrict__ status,
                                                                        double* __restrict__ status_out) {
    extern __shared__ __align__(16) unsigned char lu_smem_raw[];
    double* tile = reinterpret_cast<double*>(lu_smem_raw);
    const int c = threadIdx.x & 31, g = threadIdx.x >> 5;
    const int col = blockIdx.x * kSolveCols + c;
    const bool live = col < n;
    auto xs = [&](int r) -> double& { return IN_SMEM ? tile[r * kSolveCols + c] : X[(long long)r * ldx + col]; };
    if (blockIdx.x == 0 && threadIdx.x == 0 && status_out) *status_out = (double)status[0];
    if (IN_SMEM) {
        for (int r = g; r < m; r += kSolveRows) tile[r * kSolveCols + c] = live ? B[(long long)perm[r] * ldb + col] : 0.0;
    } else {
        for (int r = g; r < m; r += kSolveRows)
            if (live) X[(long long)r * ldx + col] = B[(long long)perm[r] * ldb + col];
    }
    __syncthreads();
    // ---- L y = P b (unit lower) ----
    for (int r0 = 0; r0 < m; r0 += kSolveRows) {
        const int r = r0 + g;
        if (r < m && r0 > 0) {
            const double* Lr = lup + (long long)r * ldp;
            double s0 = 0.0, s1 = 0.0;
            for (int k0 = 0; k0 < r0; k0 += 32) {
                const double lv = (k0 + c < r0) ? Lr[k0 + c] : 0.0;
                const int kn = min(32, r0 - k0);
                int kk = 0;
                for (; kk + 1 < kn; kk += 2) {
                    const double a0 = __shfl_sync(0xffffffffu, lv, kk), a1 = __shfl_sync(0xffffffffu, lv, kk + 1);
                    if (live) {
                        s0 += a0 * xs(k0 + kk);
                        s1 += a1 * xs(k0 + kk + 1);
                    }
                }
                if (kk < kn) {
                    const double a0 = __shfl_sync(0xffffffffu, lv, kk);
                    if (live) s0 += a0 * xs(k0 + kk);
                }
            }
            if (live) xs(r) -= s0 + s1;
        }
        __syncthreads();
        if (g == 0 && live) {
            const int rn = min(kSolveRows, m - r0);
            for (int i = 1; i < rn; ++i) {
                const double* Lr = lup + (long long)(r0 + i) * ldp + r0;
                double v = xs(r0 + i);
                for (int j = 0; j < i; ++j) v -= Lr[j] * xs(r0 + j);
                xs(r0 + i) = v;
            }
        }
        __syncthreads();
    }
    // ---- U x = y ----
    for (int r1 = m; r1 > 0; r1 -= kSolveRows) {
        const int r = r1 - 1 - g;
        if (r >= 0 && r1 < m) {
            const double* Ur = lup + (long long)r * ldp;
            double s0 = 0.0, s1 = 0.0;
            for (int k0 = r1; k0 < m; k0 += 32) {
                const double uv = (k0 + c < m) ? Ur[k0 + c] : 0.0;
                const int kn = min(32, m - k0);
                int kk = 0;
                for (; kk + 1 < kn; kk += 2) {
                    const double a0 = __shfl_sync(0xffffffffu, uv, kk), a1 = __shfl_sync(0xffffffffu, uv, kk + 1);
                    if (live) {
                        s0 += a0 * xs(k0 + kk);
                        s1 += a1 * xs(k0 + kk + 1);
                    }
                }
                if (kk < kn) {
                    const double a0 = __shfl_sync(0xffffffffu, uv, kk);
                    if (live) s0 += a0 * xs(k0 + kk);
                }
            }
            if (live) xs(r) -= s0 + s1;
        }
        __syncthreads();
        if (g == 0 && live) {
            const int rn = min(kSolveRows, r1);
            for (int i = 0; i < rn; ++i) {
                const int rr = r1 - 1 - i;
                const double* Ur = lup + (long long)rr * ldp;
                double v = xs(rr);
                for (int j = 0; j < i; ++j) v -= Ur[r1 - 1 - j] * xs(r1 - 1 - j);
                xs(rr) = v / Ur[rr];
            }
        }
        __syncthreads();
    }
    if (IN_SMEM && live)
        for (int r = g; r < m; r += kSolveRows) X[(long long)r * ldx + col] = tile[r * kSolveCols + c];
}

// scratch: work (m x ldw) | lup (m x m) | perm (m ints) | status (2 ints)
inline long long scratch_doubles(int m) {
    const long long ldw = (m + 1) & ~1;
    return (long long)m * ldw + (long long)m * m + (m + 1) / 2 + 8;
}

struct Scratch {
    double* work;
    double* lup;
    int* perm;
    int* status;
};
inline Scratch carve(double* scratch, int m) {
    Scratch s;
    const long long ldw = (m + 1) & ~1;
    s.work = scratch;
    s.lup = scratch + (long long)m * ldw;
    s.perm = reinterpret_cast<int*>(s.lup + (long long)m * m);
    s.status = s.perm + ((m + 1) & ~1);
    return s;
}

// Enqueue the two triangular sweeps X = U^-1 L^-1 B[perm] of a factor in the lup layout (ld ldp) on `st`.
inline int launch_solve(const double* lup, long long ldp, const int* perm, int m, const double* B, long long ldb, double* X,
                        long long ldx, int n, const int* status, double* status_out, cudaStream_t st, long long* launches) {
    static PerDeviceOnce attr_s = {};
    if (m > kSolveSmemMaxM && X == B) return fail(-1, "lu::solve", "in-place solve needs m <= 832");
    const int tiles = (n + kSolveCols - 1) / kSolveCols;
    if (m <= kSolveSmemMaxM) {
        const size_t smem = (size_t)m * kSolveCols * sizeof(double);
        if (attr_s.first_time())
            LCX_CUDA(cudaFuncSetAttribute(lu_solve_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024));
        lu_solve_kernel<true><<<tiles, kSolveCols * kSolveRows, smem, st>>>(lup, ldp, perm, m, B, ldb, X, ldx, n, status,
                                                                          status_out);
    } else {
        lu_solve_kernel<false><<<tiles, kSolveCols * kSolveRows, 0, st>>>(lup, ldp, perm, m, B, ldb, X, ldx, n, status,
                                                                        status_out);
    }
    if (launches) ++*launches;
    LCX_CUDA(cudaGetLastError());
    return 0;
}

// Enqueue X = A^-1 B on `st`.  Returns a negative code on a launch error.
inline int solve(const double* A, long long lda, int m, const double* B, long long ldb, double* X, long long ldx, int n,
                 double* scratch, double* status_out, cudaStream_t st, long long* launches) {
    Scratch sc = carve(scratch, m);
    static PerDeviceOnce attr_f_smem = {}, attr_f_coop = {};
    if (m <= kSmemMaxM) {
        const size_t smem = (((size_t)m * 4 + 15) & ~(size_t)15) + (size_t)m * (m | 1) * sizeof(double);
        if (attr_f_smem.first_time())
            LCX_CUDA(cudaFuncSetAttribute(lu_factor_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024));
        lu_factor_kernel<true><<<1, kFactorThreads, smem, st>>>(A, lda, m, nullptr, sc.lup, m, sc.perm, sc.status);
    } else {
        int grid = (m + 15) / 16;
        if (grid > 64) grid = 64;
        const size_t smem = ((size_t)m * 4 + 15) & ~(size_t)15;
        if (attr_f_coop.first_time())
            LCX_CUDA(cudaFuncSetAttribute(lu_factor_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024));
        const double* a = A;
        double* work = sc.work;
        double* lup = sc.lup;
        long long ldp = m;
        int* perm = sc.perm;
        int* status = sc.status;
        void* args[] = {&a, &lda, &m, &work, &lup, &ldp, &perm, &status};
        LCX_CUDA(cudaLaunchCooperativeKernel((void*)lu_factor_kernel<false>, dim3(grid), dim3(kFactorThreads), args, smem, st));
    }
    if (launches) ++*launches;
    return launch_solve(sc.lup, m, sc.perm, m, B, ldb, X, ldx, n, sc.status, status_out, st, launches);
}

}  // namespace lu
}  // namespace lcx
