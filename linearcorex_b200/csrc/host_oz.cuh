// Host plumbing of the split-integer (int8 digit plane) engine: digit slicing, tensor maps, the X pass pair and the
// m x m x n products as launches of oz_gemm_kernel (ozaki_i8.cuh).  Included by lcx_api.cu after host_session.cuh.
#pragma once
#include "host_session.cuh"

// ---- split-integer plumbing (ozaki_i8.cuh) -------------------------------------------------------
template <int S>
static int oz_slice_x_t(lcx_session* s) {
    const Layout& L = s->L;
    oz::absmax_partial_kernel<<<kAmaxCtas, 256, 0, s->stream>>>(s->xt, s->ldx, s->Nl, s->n, s->ws + L.slot[I_AMAX][0].off);
    LAUNCHED(s);
    oz::absmax_finish_kernel<<<1, 256, 0, s->stream>>>(s->ws + L.slot[I_AMAX][0].off, kAmaxCtas, s->oz_xscale());
    LAUNCHED(s);
    dim3 grid((unsigned)s->Nl, cdiv(L.ld8, 4 * 128));
    oz::slice_rows_kernel<S><<<grid, 128, 0, s->stream>>>(s->xt, s->ldx, (int)s->Nl, s->n, nullptr, s->oz_xscale(), s->xs(), L.ld8,
                                                        s->Nl * L.ld8, (double)oz::kRadix);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}

static int oz_prepare(lcx_session* s, bool streamed) {
    const Layout& L = s->L;
    LCX_REQUIRE(L.oz1_chunk <= L.oz_kmax && L.oz_chunk <= L.oz_kmax, "contraction chunk exceeds the int32-exact length");
    if (!streamed) switch (L.S) {
        case 3: LCX_TRY(oz_slice_x_t<3>(s)); break;
        case 4: LCX_TRY(oz_slice_x_t<4>(s)); break;
        case 5: LCX_TRY(oz_slice_x_t<5>(s)); break;
        case 6: LCX_TRY(oz_slice_x_t<6>(s)); break;
        case 7: LCX_TRY(oz_slice_x_t<7>(s)); break;
        default: return fail(LCX_ERR_STATE, "oz_prepare", "bad digit count");
    }
    // X~ slices as the M operand of Y = X~ A^T (K-major: inner = variables, 64 B boxes) and as the M operand of
    // D = X~^T Y (MN-major: inner = variables, 128 B boxes over 64 sample rows); the factor-side operands are K-major:
    // A slices (inner = variables) and the transposed Y slices (inner = samples).
    LCX_TRY(oz::make_slice_map(&s->map_x_k1, s->xs(), s->n, s->Nl, L.S, L.ld8, s->Nl * L.ld8, oz::kBK, oz::kBM, false));
    // the factors are split into equal tiles: m = 100, bn_max = 64 -> 2 tiles of 56 (not 64 + 48), so the CTAs that share an
    // X~ tile by multicast carry the same work; widths of 8 mod 16 use the spill form of the wide MMAs (ozaki_i8.cuh)
    const int bnm = oz::bn_max(L.S);
    const int n_tiles = cdiv(s->m, bnm);
    s->oz_bn = (int)max(16LL, round_up(cdiv(s->m, n_tiles), bnm > 64 ? 16 : 8));
    const int bn = s->oz_bn;
    LCX_TRY(oz::make_slice_map(&s->map_a_k1, s->as(), s->n, s->m, L.S, L.ld8, (long long)s->m * L.ld8, oz::kBK, bn, false));
    LCX_TRY(oz::make_slice_map(&s->map_x_k2, s->xs(), s->n, s->Nl, L.S, L.ld8, s->Nl * L.ld8, oz::kBM, oz::kBK, true));
    LCX_TRY(oz::make_slice_map(&s->map_y_k2, s->ys(), s->Nl, s->m, L.S, L.ldk8, (long long)s->m * L.ldk8, oz::kBK, bn, false));
    if (L.mm_i8) {
        LCX_REQUIRE(L.mm_chunk <= L.oz_kmax && round_up(s->m, oz::kBK) <= L.oz_kmax, "contraction chunk exceeds the int32-exact length");
        const long long st_n = (long long)s->m * L.ld8, st_q = (long long)s->m * L.ldm8;
        // ry = W rho^T, H = T rinv^T: both operands K-major over the variables (M side 128-row boxes, N side bn-row boxes)
        LCX_TRY(oz::make_slice_map(&s->map_mm_a, s->mma(), s->n, s->m, L.S, L.ld8, st_n, oz::kBK, oz::kBM, false));
        LCX_TRY(oz::make_slice_map(&s->map_mm_b, s->mmb(), s->n, s->m, L.S, L.ld8, st_n, oz::kBK, bn, false));
        // Qij = ry rinv, grad += H W: M side = variables of the m x n operand (MN-major, contraction over its m rows),
        // N side = the m x m factor, K-major
        LCX_TRY(oz::make_slice_map(&s->map_mn_c, s->mmc(), s->n, s->m, L.S, L.ld8, st_n, oz::kBM, oz::kBK, true));
        LCX_TRY(oz::make_slice_map(&s->map_mn_q, s->mmq(), s->m, s->m, L.S, L.ldm8, st_q, oz::kBK, bn, false));
    }
    return 0;
}

template <int S>
static int oz_pair_t(lcx_session* s, const double* A, double* svec, cudaEvent_t* ev, bool first_only, bool want_tail,
                     const double* dot_b, double* dot_out) {
    const Layout& L = s->L;
    const int m = s->m, n = s->n;
    double* Y = s->ptr(LCX_A_Y);
    double* D = s->ptr(LCX_A_D);
    // ---- Y = X~ A^T ----
    oz::row_scale_kernel<<<m, 256, 0, s->stream>>>(A, L.ld, n, s->oz_ascale(), 0, s->oz_xscale(), s->oz_cscale(), dot_b, dot_out);
    LAUNCHED(s);
    oz::slice_rows_kernel<S><<<dim3(m, cdiv(L.ld8, 4 * 128)), 128, 0, s->stream>>>(A, L.ld, m, n, s->oz_ascale(), nullptr, s->as(), L.ld8,
                                                                              (long long)m * L.ld8, (double)oz::kRadix);
    LAUNCHED(s);
    {
        oz::GemmParams p;
        memset(&p, 0, sizeof(p));
        const bool split1 = L.oz1_splits > 1;
        p.C = split1 ? s->ptr(I_PART) : Y;
        p.ldc = L.ldy; p.c_split_stride = split1 ? s->Nl * L.ldy : 0;
        p.col_scale = s->oz_cscale();
        p.inv_radix = 1.0 / (double)oz::kRadix;
        p.rows = (int)s->Nl; p.cols = m; p.k_total = n; p.k_chunk = L.oz1_chunk;
        p.bn = s->oz_bn;
        const int row0 = (cdiv(s->Nl, oz::kBM) - L.oz1_tail_tiles) * oz::kBM;
        if (L.oz1_tail_tiles > 0) {  // two-level split (host_session.cuh: plan_two_level): the last row tiles' last K chunk, cut finer
            const int groups = cdiv(cdiv(m, oz::bn_max(S)), 2), m_tiles = cdiv(s->Nl, oz::kBM);
            p.main_units = groups * (m_tiles * L.oz1_splits - L.oz1_tail_tiles);
            p.tail_units = groups * L.oz1_tail_tiles * L.oz1_tail_splits;
            p.tail_m_tile0 = m_tiles - L.oz1_tail_tiles; p.tail_m_tiles = L.oz1_tail_tiles;
            p.tail_kbase = (L.oz1_splits - 1) * L.oz1_chunk; p.tail_kchunk = L.oz1_tail_chunk;
            p.tail_C = s->ptr(I_TAIL1) - (long long)row0 * L.ldy;
            p.tail_ldc = L.ldy; p.tail_split_stride = (long long)L.oz1_tail_tiles * oz::kBM * L.ldy;
        }
        LCX_TRY((oz::launch_oz_gemm<S, true>(s->map_x_k1, s->map_a_k1, p,
                                             dim3(cdiv(m, oz::bn_max(S)), cdiv(s->Nl, oz::kBM), L.oz1_splits), s->stream)));
        LAUNCHED(s);
        if (L.oz1_tail_tiles > 0) {
            double* dst = (split1 ? s->ptr(I_PART) + (long long)(L.oz1_splits - 1) * s->Nl * L.ldy : Y) + (long long)row0 * L.ldy;
            const int rows = (int)(s->Nl - row0);
            oz::tail_fold_kernel<<<cdiv((long long)rows * m, 256), 256, 0, s->stream>>>(
                s->ptr(I_TAIL1), L.oz1_tail_splits, (long long)L.oz1_tail_tiles * oz::kBM * L.ldy, L.ldy, dst, L.ldy, rows, m);
            LAUNCHED(s);
        }
        if (split1) {
            LCX_TRY(launch_reduce_splits(s->ptr(I_PART), L.oz1_splits, s->Nl * L.ldy, Y, (int)s->Nl, m, L.ldy, s->stream));
            LAUNCHED(s);
        }
    }
    if (ev) LCX_CUDA(cudaEventRecord(ev[1], s->stream));
    if (ev) LCX_CUDA(cudaEventRecord(ev[3], s->stream));
    // ---- column max / sum of squares of Y, digit slices of Y ----
    double* ystat = s->ws + L.slot[I_YSTAT][0].off;
    oz::y_stats_kernel<<<dim3(cdiv(m, 32), L.ystat_slabs), dim3(32, 8), 0, s->stream>>>(Y, L.ldy, s->Nl, m, kYStatRows, ystat, L.ldm);
    LAUNCHED(s);
    oz::y_stats_finish_kernel<<<m, 256, 0, s->stream>>>(ystat, L.ystat_slabs, L.ldm, m, s->oz_xscale(), svec, s->oz_yscale(),
                                                                  s->oz_dscale());
    LAUNCHED(s);
    if (first_only) {  // _norm (:215-228): only Y and its column sums of squares are needed
        LCX_CUDA(cudaGetLastError());
        return 0;
    }
    oz::slice_cols_t_kernel<S><<<dim3((unsigned)cdiv(s->Nl, 128), cdiv(m, 32)), dim3(32, 8), 0, s->stream>>>(
        Y, L.ldy, s->Nl, m, s->oz_yscale(), s->ys(), L.ldk8, (long long)m * L.ldk8, (double)oz::kRadix);
    LAUNCHED(s);
    // ---- D = (X~^T Y)^T: tiles of 128 variables x 64 factors, stored factor-major, split over samples ----
    {
        oz::GemmParams p;
        memset(&p, 0, sizeof(p));
        const bool split = L.oz_splits > 1;
        p.C = split ? s->ptr(I_PART) : D;
        p.ldc = L.ld; p.c_split_stride = split ? (long long)m * L.ld : 0;
        p.col_scale = s->oz_dscale();
        p.inv_radix = 1.0 / (double)oz::kRadix;
        p.rows = n; p.cols = m; p.k_total = (int)s->Nl; p.k_chunk = L.oz_chunk;
        p.bn = s->oz_bn;
        p.trans_out = 1;
        const int var0 = (cdiv(n, oz::kBM) - L.oz_tail_tiles) * oz::kBM;
        const long long tld = (long long)L.oz_tail_tiles * oz::kBM;
        if (L.oz_tail_tiles > 0) {  // two-level split: the last variable tiles' last sample chunk, cut finer
            const int groups = cdiv(cdiv(m, oz::bn_max(S)), 2), m_tiles = cdiv(n, oz::kBM);
            p.main_units = groups * (m_tiles * L.oz_splits - L.oz_tail_tiles);
            p.tail_units = groups * L.oz_tail_tiles * L.oz_tail_splits;
            p.tail_m_tile0 = m_tiles - L.oz_tail_tiles; p.tail_m_tiles = L.oz_tail_tiles;
            p.tail_kbase = (L.oz_splits - 1) * L.oz_chunk; p.tail_kchunk = L.oz_tail_chunk;
            p.tail_C = s->ptr(I_TAIL2) - var0;
            p.tail_ldc = tld; p.tail_split_stride = (long long)m * tld;
        }
        LCX_TRY((oz::launch_oz_gemm<S, false>(s->map_x_k2, s->map_y_k2, p,
                                              dim3(cdiv(m, oz::bn_max(S)), cdiv(n, oz::kBM), L.oz_splits), s->stream)));
        LAUNCHED(s);
        if (L.oz_tail_tiles > 0) {
            double* dst = (split ? s->ptr(I_PART) + (long long)(L.oz_splits - 1) * m * L.ld : D) + var0;
            oz::tail_fold_kernel<<<cdiv((long long)m * (n - var0), 256), 256, 0, s->stream>>>(
                s->ptr(I_TAIL2), L.oz_tail_splits, (long long)m * tld, tld, dst, L.ld, m, n - var0);
            LAUNCHED(s);
        }
        if (ev) LCX_CUDA(cudaEventRecord(ev[4], s->stream));
        LCX_TRY(combine_and_allreduce(s, split ? s->ptr(I_PART) : D, split ? L.oz_splits : 1, (long long)m * L.ld, m, n, L.ld, D, svec,
                                      want_tail ? m : 0));
    }
    LCX_CUDA(cudaGetLastError());
    return 0;
}

static int oz_pair(lcx_session* s, const double* A, double* svec, cudaEvent_t* ev, bool first_only, bool want_tail,
                   const double* dot_b = nullptr, double* dot_out = nullptr) {
    switch (s->L.S) {
        case 3: return oz_pair_t<3>(s, A, svec, ev, first_only, want_tail, dot_b, dot_out);
        case 4: return oz_pair_t<4>(s, A, svec, ev, first_only, want_tail, dot_b, dot_out);
        case 5: return oz_pair_t<5>(s, A, svec, ev, first_only, want_tail, dot_b, dot_out);
        case 6: return oz_pair_t<6>(s, A, svec, ev, first_only, want_tail, dot_b, dot_out);
        case 7: return oz_pair_t<7>(s, A, svec, ev, first_only, want_tail, dot_b, dot_out);
    }
    return fail(LCX_ERR_STATE, "oz_pair", "bad digit count");
}

// ---- the m x m x n products of an iteration on the int8 engine (L.mm_i8; same kernel, same digit scheme) ----------
// out (m x m) = left right^T over the variables, both m x n: each operand gets one exponent per factor row; split-K
// partials are combined in fixed order and np.fill_diagonal is applied there (raw diagonal -> diag_out).
template <int S>
static int oz_square_t(lcx_session* s, const double* left, const double* right, double* out, double diag_value,
                       double* diag_out) {
    const Layout& L = s->L;
    const int m = s->m, n = s->n;
    const dim3 gs(m, cdiv(L.ld8, 4 * 128));
    const long long st_n = (long long)m * L.ld8;
    oz::row_scale_kernel<<<m, 256, 0, s->stream>>>(left, L.ld, n, s->mm_scale_a());
    LAUNCHED(s);
    oz::slice_rows_kernel<S><<<gs, 128, 0, s->stream>>>(left, L.ld, m, n, s->mm_scale_a(), nullptr, s->mma(), L.ld8, st_n,
                                                       (double)oz::kRadix);
    LAUNCHED(s);
    oz::row_scale_kernel<<<m, 256, 0, s->stream>>>(right, L.ld, n, s->mm_scale_b());
    LAUNCHED(s);
    oz::slice_rows_kernel<S><<<gs, 128, 0, s->stream>>>(right, L.ld, m, n, s->mm_scale_b(), nullptr, s->mmb(), L.ld8, st_n,
                                                       (double)oz::kRadix);
    LAUNCHED(s);
    oz::GemmParams p;
    memset(&p, 0, sizeof(p));
    const long long out_count = (long long)m * L.ldm;
    p.C = s->ptr(I_PART);
    p.ldc = L.ldm; p.c_split_stride = out_count;
    p.row_scale = s->mm_scale_a();
    p.col_scale = s->mm_scale_b();
    p.inv_radix = 1.0 / (double)oz::kRadix;
    p.rows = m; p.cols = m; p.k_total = n; p.k_chunk = L.mm_chunk;
    p.bn = s->oz_bn;
    LCX_TRY((oz::launch_oz_gemm<S, true>(s->map_mm_a, s->map_mm_b, p,
                                         dim3(cdiv(m, oz::bn_max(S)), cdiv(m, oz::kBM), L.mm_splits), s->stream)));
    LAUNCHED(s);
    LCX_TRY(launch_reduce_splits(s->ptr(I_PART), L.mm_splits, out_count, out, m, m, L.ldm, s->stream,
                                 diag_out ? diag_out : s->ptr(I_F), diag_value));
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}

// out (m x n, factor-major) = c_add + Q V with Q m x m and V m x n: the contraction runs over V's rows, so V gets one
// exponent per COLUMN (variable) and Q one per row; tiles of 128 variables x 64 factors like the second X contraction.
// unit_diag: Q has an exact unit diagonal (ry after np.fill_diagonal, :263).  Its digits would be spent on that 1 while the
// off-diagonal correlations are 1e-2 and below, so the product runs on Q - I and the caller passes c_add = V.
template <int S>
static int oz_mn_t(lcx_session* s, const double* Q, const double* V, double* out, const double* c_add, bool unit_diag) {
    const Layout& L = s->L;
    const int m = s->m, n = s->n;
    oz::col_absmax_partial_kernel<<<dim3(cdiv(n, 512), L.mm_slabs), 256, 0, s->stream>>>(V, L.ld, m, n, L.mm_slab_rows,
                                                                                       s->mm_colpart(), L.ld);
    LAUNCHED(s);
    oz::col_scale_finish_kernel<<<cdiv(n, 256), 256, 0, s->stream>>>(s->mm_colpart(), L.mm_slabs, L.ld, n, s->mm_colscale());
    LAUNCHED(s);
    oz::slice_colscaled_kernel<S><<<dim3(m, cdiv(L.ld8, 4 * 128)), 128, 0, s->stream>>>(V, L.ld, m, n, s->mm_colscale(), s->mmc(),
                                                                                      L.ld8, (long long)m * L.ld8, (double)oz::kRadix);
    LAUNCHED(s);
    oz::row_scale_kernel<<<m, 256, 0, s->stream>>>(Q, L.ldm, m, s->mm_scale_q(), unit_diag ? 1 : 0);
    LAUNCHED(s);
    const dim3 gq(m, cdiv(L.ldm8, 4 * 128));
    if (unit_diag)
        oz::slice_rows_kernel<S, true><<<gq, 128, 0, s->stream>>>(Q, L.ldm, m, m, s->mm_scale_q(), nullptr, s->mmq(), L.ldm8,
                                                                 (long long)m * L.ldm8, (double)oz::kRadix);
    else
        oz::slice_rows_kernel<S><<<gq, 128, 0, s->stream>>>(Q, L.ldm, m, m, s->mm_scale_q(), nullptr, s->mmq(), L.ldm8,
                                                           (long long)m * L.ldm8, (double)oz::kRadix);
    LAUNCHED(s);
    oz::GemmParams p;
    memset(&p, 0, sizeof(p));
    p.C = out;
    p.ldc = L.ld; p.c_split_stride = 0;
    p.row_scale = s->mm_colscale();
    p.col_scale = s->mm_scale_q();
    p.inv_radix = 1.0 / (double)oz::kRadix;
    p.rows = n; p.cols = m; p.k_total = m; p.k_chunk = (int)round_up(m, oz::kBK);
    p.bn = s->oz_bn;
    p.trans_out = 1;
    p.c_add = c_add;
    LCX_TRY((oz::launch_oz_gemm<S, false, true>(s->map_mn_c, s->map_mn_q, p,
                                          dim3(cdiv(m, oz::bn_max(S)), cdiv(n, oz::kBM), 1), s->stream)));
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}

static int oz_square(lcx_session* s, const double* left, const double* right, double* out, double diag_value, double* diag_out) {
    switch (s->L.S) {
        case 3: return oz_square_t<3>(s, left, right, out, diag_value, diag_out);
        case 4: return oz_square_t<4>(s, left, right, out, diag_value, diag_out);
        case 5: return oz_square_t<5>(s, left, right, out, diag_value, diag_out);
        case 6: return oz_square_t<6>(s, left, right, out, diag_value, diag_out);
        case 7: return oz_square_t<7>(s, left, right, out, diag_value, diag_out);
    }
    return fail(LCX_ERR_STATE, "oz_square", "bad digit count");
}

static int oz_mn(lcx_session* s, const double* Q, const double* V, double* out, const double* c_add, bool unit_diag) {
    switch (s->L.S) {
        case 3: return oz_mn_t<3>(s, Q, V, out, c_add, unit_diag);
        case 4: return oz_mn_t<4>(s, Q, V, out, c_add, unit_diag);
        case 5: return oz_mn_t<5>(s, Q, V, out, c_add, unit_diag);
        case 6: return oz_mn_t<6>(s, Q, V, out, c_add, unit_diag);
        case 7: return oz_mn_t<7>(s, Q, V, out, c_add, unit_diag);
    }
    return fail(LCX_ERR_STATE, "oz_mn", "bad digit count");
}

template <int S>
static int oz_slice_block_t(lcx_session* s, const double* xt, long long row0, long long rows, long long ldx) {
    const Layout& L = s->L;
    dim3 grid((unsigned)rows, cdiv(L.ld8, 4 * 128));
    oz::slice_rows_kernel<S><<<grid, 128, 0, s->stream>>>(xt, ldx, (int)rows, s->n, nullptr, s->oz_xscale(), s->xs() + row0 * L.ld8,
                                                        L.ld8, s->Nl * L.ld8, (double)oz::kRadix);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}
