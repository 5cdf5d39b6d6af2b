// Column statistics, mean imputation and standardisation (linearcorex.py:397-429, :483-510).
//
// Raw X arrives as float32 or float64, row-major N x n (ld = ldx).  Three passes, each a column
// reduction over a row slab per CTA (blockDim = 32 x 8, grid = strips x slabs) followed by a
// fixed-order combine of the slab partials.  When rows are sharded over ranks the caller
// all-reduces the combined vectors between passes (SURVEY.md section 8(e)).
#pragma once
#include "common.cuh"
#include "ozaki_i8.cuh"

namespace lcx {

// V consecutive elements of a row as doubles: one 16-byte load per 4 floats / 2 doubles when V == 4 (the caller
// guarantees 16-byte alignment: base pointer, leading dimension and first column all multiples of 4 elements).
template <typename T, int V>
__device__ __forceinline__ void load_row_vec(const T* __restrict__ p, double (&o)[V]) {
    if constexpr (V == 1) {
        o[0] = (double)p[0];
    } else if constexpr (sizeof(T) == 4) {
        const float4 v = *reinterpret_cast<const float4*>(p);
        o[0] = (double)v.x; o[1] = (double)v.y; o[2] = (double)v.z; o[3] = (double)v.w;
    } else {
        const double2 a = *reinterpret_cast<const double2*>(p), b = *reinterpret_cast<const double2*>(p + 2);
        o[0] = a.x; o[1] = a.y; o[2] = b.x; o[3] = b.y;
    }
}

__device__ __forceinline__ bool is_missing_d(double d, int has_marker, double marker, int marker_is_nan) {
    if (!has_marker) return false;
    return (d != d) || (!marker_is_nan && d == marker);  // NaN is always missing once a marker is set (:505)
}

// pass 1: part_sum[slab][i] = sum of observed x, part_cnt[slab][i] = number observed (finite, not missing)
// Each thread owns V adjacent columns (V = 4: 16-byte loads) and every eighth row of the slab; a column's rows are
// summed in the same order whatever V is, so the result does not depend on the vector width.
template <typename T, int V>
__global__ void __launch_bounds__(256) colstats_sum_kernel(const T* __restrict__ x, long long N, int n, long long ldx,
                                                           int rows_per_slab, int has_marker, double marker,
                                                           int marker_is_nan, double* __restrict__ part_sum,
                                                           double* __restrict__ part_cnt, long long ldp) {
    __shared__ double rs[8][32 * V], rc[8][32 * V];
    const int i0 = (blockIdx.x * 32 + threadIdx.x) * V;
    const long long r0 = (long long)blockIdx.y * rows_per_slab;
    const long long r1 = min(N, r0 + rows_per_slab);
    double s[V], c[V];
#pragma unroll
    for (int j = 0; j < V; ++j) s[j] = c[j] = 0.0;
    if (i0 < n) {
#pragma unroll 2
        for (long long r = r0 + threadIdx.y; r < r1; r += 8) {
            double v[V];
            load_row_vec<T, V>(x + r * ldx + i0, v);
#pragma unroll
            for (int j = 0; j < V; ++j) {
                const bool obs = has_marker ? (!is_missing_d(v[j], has_marker, marker, marker_is_nan) && isfinite(v[j])) : true;
                if (obs) { s[j] += v[j]; c[j] += 1.0; }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < V; ++j) {
        rs[threadIdx.y][threadIdx.x * V + j] = s[j];
        rc[threadIdx.y][threadIdx.x * V + j] = c[j];
    }
    __syncthreads();
    for (int t = threadIdx.y * 32 + threadIdx.x; t < 32 * V; t += 256) {
        const int i = blockIdx.x * 32 * V + t;
        if (i < n) {
            double a = 0.0, b = 0.0;
#pragma unroll
            for (int k = 0; k < 8; ++k) { a += rs[k][t]; b += rc[k][t]; }
            part_sum[(long long)blockIdx.y * ldp + i] = a;
            part_cnt[(long long)blockIdx.y * ldp + i] = b;
        }
    }
}

// pass 2: part[slab][i] = sum over observed rows of (x - mean_i)^2   (imputed entries contribute 0)
template <typename T, int V>
__global__ void __launch_bounds__(256) colstats_sqdev_kernel(const T* __restrict__ x, long long N, int n, long long ldx,
                                                             int rows_per_slab, int has_marker, double marker,
                                                             int marker_is_nan, const double* __restrict__ mean,
                                                             double* __restrict__ part, double* __restrict__ part_max,
                                                             long long ldp) {
    // part_max (optional): per-slab max |x - mean| -- bounds |X~| before X~ exists (streamed digit slicing)
    __shared__ double rs[8][32 * V], rm[8][32 * V];
    const int i0 = (blockIdx.x * 32 + threadIdx.x) * V;
    const long long r0 = (long long)blockIdx.y * rows_per_slab;
    const long long r1 = min(N, r0 + rows_per_slab);
    double s[V], mx[V], mu[V];
#pragma unroll
    for (int j = 0; j < V; ++j) {
        s[j] = mx[j] = 0.0;
        mu[j] = (i0 + j < n) ? mean[i0 + j] : 0.0;
    }
    if (i0 < n) {
#pragma unroll 2
        for (long long r = r0 + threadIdx.y; r < r1; r += 8) {
            double v[V];
            load_row_vec<T, V>(x + r * ldx + i0, v);
#pragma unroll
            for (int j = 0; j < V; ++j) {
                if (!is_missing_d(v[j], has_marker, marker, marker_is_nan)) {
                    const double d = v[j] - mu[j];
                    s[j] += d * d;
                    mx[j] = amax_acc(mx[j], d);
                }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < V; ++j) {
        rs[threadIdx.y][threadIdx.x * V + j] = s[j];
        rm[threadIdx.y][threadIdx.x * V + j] = mx[j];
    }
    __syncthreads();
    for (int t = threadIdx.y * 32 + threadIdx.x; t < 32 * V; t += 256) {
        const int i = blockIdx.x * 32 * V + t;
        if (i < n) {
            double a = 0.0, b = 0.0;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                a += rs[k][t];
                b = fmax(b, rm[k][t]);
            }
            part[(long long)blockIdx.y * ldp + i] = a;
            if (part_max) part_max[(long long)blockIdx.y * ldp + i] = b;
        }
    }
}

// out[i] = max_slab part[slab][i]
__global__ void combine_slabs_max_kernel(const double* __restrict__ part, int slabs, long long ldp, double* __restrict__ out,
                                         int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        double a = 0.0;
        for (int s = 0; s < slabs; ++s) a = fmax(a, part[(long long)s * ldp + i]);
        out[i] = a;
    }
}

// out[i] = sum_slab part[slab][i]
__global__ void combine_slabs_kernel(const double* __restrict__ part, int slabs, long long ldp, double* __restrict__ out,
                                     int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        double a = 0.0;
        for (int s = 0; s < slabs; ++s) a += part[(long long)s * ldp + i];
        out[i] = a;
    }
}

// mean = sum / cnt
__global__ void finish_mean_kernel(const double* __restrict__ sum, const double* __restrict__ cnt, double* __restrict__ mean,
                                   int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) mean[i] = sum[i] / cnt[i];
}

// std = max(sqrt(sq / denom), 1e-10); denom = n_obs ('standard', :413) or N_total ('outliers', np.std :421)
__global__ void finish_std_kernel(const double* __restrict__ sq, const double* __restrict__ cnt, double n_total,
                                  int use_nobs, double* __restrict__ sd, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) sd[i] = fmax(sqrt(sq[i] / (use_nobs ? cnt[i] : n_total)), 1e-10);
}

__device__ __forceinline__ double squash_tails(double z) {  // g(), :483-487
    const double core = fmin(fmax(z, -4.0), 4.0);
    return core + tanh(z - core);
}

// One element of X~ (column i): a missing entry takes impute[i] first (:404); mode 0 = 'standard' (x - mean) / std (:415),
// 1 = 'outliers' (the same + g(), :423), 2 = 'none' (cast only).
__device__ __forceinline__ double standardize_value(double d, int i, int has_marker, double marker, int marker_is_nan, int mode,
                                                    const double* __restrict__ impute, const double* __restrict__ mean,
                                                    const double* __restrict__ sd) {
    if (is_missing_d(d, has_marker, marker, marker_is_nan)) d = impute[i];
    if (mode == 2) return d;
    const double o = (d - mean[i]) / sd[i];
    return mode == 1 ? squash_tails(o) : o;
}

// X~ = (x - mean)/std  [+ g()];  missing entries take the column mean first (:404, :415, :423).
// mode: 0 = 'standard', 1 = 'outliers', 2 = 'none' (cast only).  Output fp64, ld = ldo, columns >= n zeroed.
template <typename T, int V>
__global__ void standardize_kernel(const T* __restrict__ x, long long N, int n, long long ldx, int has_marker,
                                   double marker, int marker_is_nan, int mode, const double* __restrict__ impute,
                                   const double* __restrict__ mean, const double* __restrict__ sd,
                                   double* __restrict__ out, long long ldo) {
    const int i0 = (blockIdx.y * blockDim.x + threadIdx.x) * V;  // rows on grid.x (up to 2^31-1), column blocks on grid.y
    const long long r = blockIdx.x;
    if (i0 >= ldo || r >= N) return;
    double v[V], o[V];
    if (i0 < n) {
        load_row_vec<T, V>(x + r * ldx + i0, v);
    }
#pragma unroll
    for (int j = 0; j < V; ++j) {
        const int i = i0 + j;
        o[j] = i < n ? standardize_value(v[j], i, has_marker, marker, marker_is_nan, mode, impute, mean, sd) : 0.0;
    }
    if constexpr (V == 1) {
        out[r * ldo + i0] = o[0];
    } else {  // ldo is a multiple of 16 doubles and i0 of 4: 16-byte stores
        *reinterpret_cast<double2*>(out + r * ldo + i0) = make_double2(o[0], o[1]);
        *reinterpret_cast<double2*>(out + r * ldo + i0 + 2) = make_double2(o[2], o[3]);
    }
}

// Split modes: standardise + g() + impute + digit-slice in ONE pass over the raw input -- X~ goes straight from the fp32 / fp64
// source into its S int8 planes (out[s][row0 + r][c]) and never exists in binary64: 4 (or 8) bytes read and S bytes written per
// element instead of 12 + 8 + S + 8 through standardize_kernel, absmax and slice_rows.  The exponent of X~ must be known
// beforehand (lcx_set_x_scale: max |x - mean| / std per column comes out of the squared-deviation pass).  The arithmetic of
// each element is standardize_kernel's followed by split_digits's, operation for operation: the planes are bit-identical.
template <typename T, int S, int V>
__global__ void __launch_bounds__(128) standardize_slice_kernel(const T* __restrict__ x, long long N, int n, long long ldx,
                                                                int has_marker, double marker, int marker_is_nan, int mode,
                                                                const double* __restrict__ impute, const double* __restrict__ mean,
                                                                const double* __restrict__ sd, double* x_scale,
                                                                int8_t* __restrict__ out, long long ld_out,
                                                                long long slice_stride, double radix) {
    const int c4 = (blockIdx.y * blockDim.x + threadIdx.x) * 4;   // four columns per thread: one char4 store per plane
    const long long r = blockIdx.x;
    if (c4 >= ld_out || r >= N) return;
    const double inv = 1.0 / x_scale[0];
    double v[4] = {0.0, 0.0, 0.0, 0.0};
    if (V == 4) {
        if (c4 + 3 < n) {
            load_row_vec<T, 4>(x + r * ldx + c4, v);
        } else {
            for (int j = 0; j < 4; ++j)
                if (c4 + j < n) v[j] = (double)x[r * ldx + c4 + j];
        }
    } else {
        for (int j = 0; j < 4; ++j)
            if (c4 + j < n) v[j] = (double)x[r * ldx + c4 + j];
    }
    int8_t d[4][S];
    bool poison = false;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int i = c4 + j;
        double o = 0.0;
        if (i < n) {
            o = standardize_value(v[j], i, has_marker, marker, marker_is_nan, mode, impute, mean, sd);
            poison = poison || !(fabs(o) <= 1.7976931348623157e308);
        }
        oz::split_digits<S>(o, inv, radix, d[j]);
    }
    // A non-finite X~ entry (an inf in the data, a column with no observed value: mean = 0 / 0) has no digits.  The reference's
    // float64 products turn NaN there; here the exponent of X~ is poisoned, and with it every product of the planes.
    if (poison) x_scale[0] = __longlong_as_double(0x7ff8000000000000LL);
#pragma unroll
    for (int k = 0; k < S; ++k) {
        char4 w = make_char4(d[0][k], d[1][k], d[2][k], d[3][k]);
        *reinterpret_cast<char4*>(out + (long long)k * slice_stride + r * ld_out + c4) = w;
    }
}

}  // namespace lcx
