// Gram route of the split-integer engine.  Every quantity of the fit depends on the data only through X~^T X~ / N: _sig
// (linearcorex.py:196-213) is u -> (X~^T X~ / N) u^T, and sum_l Y_lj^2 / N = a_j^T (X~^T X~ / N) a_j.  The reference never
// forms that n x n matrix because it targets n >> N (its docstring at :197-198); for N >= n forming it ONCE turns the two
// N x n x m contractions of every iteration into one n x n x m product.
//   lcx_gram_build : G = X~^T X~ / N from the bound digit planes -- column block by column block through the SAME second-
//                    contraction kernel (variables on M, MN-major X~ planes; the block's planes turned around as the K-major
//                    factor-side operand), upper triangle only, exact int32 group sums, fixed-order split-K combine.
//   lcx_bind_gram  : digit planes of G (one exponent: it is a correlation matrix) as the M operand of the FIRST contraction.
//   gram_pair      : D = (G A^T)^T stored factor-major, s_j = sum_i A_ji D_ji.
// Included by lcx_api.cu after host_oz.cuh.
#pragma once
#include "host_oz.cuh"

static long long gram_tbuf_doubles(const lcx_session* s, int block_cols) {
    return ((long long)s->L.S * block_cols * s->L.ldk8 + 7) / 8;
}

static long long gram_scratch_doubles(const lcx_session* s, int block_cols, long long ldg) {
    return round_up(block_cols, 16) + align16(gram_tbuf_doubles(s, block_cols)) +
           (s->L.oz_build_splits > 1 ? (long long)s->L.oz_build_splits * block_cols * ldg : 0LL) + 64;
}

template <int S>
static int gram_build_t(lcx_session* s, double* g, long long ldg, int B, double* scratch) {
    const Layout& L = s->L;
    const int n = s->n;
    double* scale = scratch;
    int8_t* tbuf = (int8_t*)(scratch + round_up(B, 16));
    double* part = scratch + round_up(B, 16) + align16(gram_tbuf_doubles(s, B));
    const long long t_stride = (long long)B * L.ldk8;
    const int splits = L.oz_build_splits;
    oz::gram_scale_kernel<<<cdiv(B, 256), 256, 0, s->stream>>>(s->oz_xscale(), 1.0 / (double)s->Nt, scale, B);
    LAUNCHED(s);
    for (int c0 = 0; c0 < n; c0 += B) {
        const int nb = min(B, n - c0);
        oz::transpose_planes_kernel<<<dim3((unsigned)cdiv(s->Nl, 128), cdiv(nb, 128), S), dim3(32, 8), 0, s->stream>>>(
            s->xs(), L.ld8, s->Nl, s->Nl * L.ld8, c0, nb, tbuf, L.ldk8, t_stride);
        LAUNCHED(s);
        // equal-width tiles of the block's columns (the last block may be narrower than B)
        const int bnm = oz::bn_max(S);
        const int n_tiles = cdiv(nb, bnm);
        const int bn = (int)max(16LL, round_up(cdiv(nb, n_tiles), bnm > 64 ? 16 : 8));
        CUtensorMap map_a, map_b;
        // rows (variables) from the start of this column block: the upper triangle
        LCX_TRY(oz::make_slice_map(&map_a, s->xs() + c0, n - c0, s->Nl, S, L.ld8, s->Nl * L.ld8, oz::kBM, oz::kBK, true));
        LCX_TRY(oz::make_slice_map(&map_b, tbuf, s->Nl, nb, S, L.ldk8, t_stride, oz::kBK, bn, false));
        oz::GemmParams p;
        memset(&p, 0, sizeof(p));
        double* dst = g + (long long)c0 * ldg + c0;
        p.C = splits > 1 ? part : dst;
        p.ldc = ldg;
        p.c_split_stride = splits > 1 ? (long long)B * ldg : 0;
        p.col_scale = scale;
        p.inv_radix = 1.0 / (double)oz::kRadix;
        p.rows = n - c0; p.cols = nb; p.k_total = (int)s->Nl; p.k_chunk = L.oz_build_chunk;
        p.bn = bn;
        p.trans_out = 1;
        LCX_TRY((oz::launch_oz_gemm<S, false>(map_a, map_b, p, dim3(n_tiles, cdiv(n - c0, oz::kBM), splits), s->stream)));
        LAUNCHED(s);
        if (splits > 1) {
            LCX_TRY(launch_reduce_splits(part, splits, (long long)B * ldg, dst, nb, n - c0, ldg, s->stream));
            LAUNCHED(s);
        }
    }
    oz::mirror_upper_kernel<<<dim3(cdiv(n, 32), cdiv(n, 32)), dim3(32, 8), 0, s->stream>>>(g, ldg, n);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}

static int gram_build(lcx_session* s, double* g, long long ldg, int B, double* scratch) {
    switch (s->L.S) {
        case 3: return gram_build_t<3>(s, g, ldg, B, scratch);
        case 4: return gram_build_t<4>(s, g, ldg, B, scratch);
        case 5: return gram_build_t<5>(s, g, ldg, B, scratch);
        case 6: return gram_build_t<6>(s, g, ldg, B, scratch);
        case 7: return gram_build_t<7>(s, g, ldg, B, scratch);
    }
    return fail(LCX_ERR_STATE, "gram_build", "bad digit count");
}

// dot_b / dot_out: dot_out_j = sum_i A_ji dot_b_ji rides on the row-maximum pass over A.  leave_partials: with a split product
// the m x ld partials stay in I_PART (s->d_splits of them) for a consumer that adds them itself.
// D = (G A^T)^T (m x ld, factor-major) and optionally svec_j = sum_i A_ji D_ji = a_j^T G a_j (the column sums of squares of
// Y = X~ A^T divided by N).  ev (optional): [0] recorded by the caller; [1]/[3]/[4]/[2] after the product.
template <int S>
static int gram_pair_t(lcx_session* s, const double* A, double* svec, cudaEvent_t* ev, const double* dot_b, double* dot_out,
                       bool leave_partials) {
    const Layout& L = s->L;
    const int m = s->m, n = s->n;
    double* D = s->ptr(LCX_A_D);
    oz::row_scale_kernel<<<m, 256, 0, s->stream>>>(A, L.ld, n, s->oz_ascale(), 0, s->oz_xscale(), s->oz_cscale(), dot_b, dot_out);
    LAUNCHED(s);
    oz::slice_rows_kernel<S><<<dim3(m, cdiv(L.ld8, 4 * 128)), 128, 0, s->stream>>>(A, L.ld, m, n, s->oz_ascale(), nullptr, s->as(), L.ld8,
                                                                              (long long)m * L.ld8, (double)oz::kRadix);
    LAUNCHED(s);
    oz::GemmParams p;
    memset(&p, 0, sizeof(p));
    p.ldc = L.ld;
    p.col_scale = s->oz_cscale();
    p.inv_radix = 1.0 / (double)oz::kRadix;
    p.rows = n; p.cols = m; p.k_total = n;
    p.bn = s->oz_bn;
    p.trans_out = 1;
    s->d_splits = 1;
    const int n_tiles = cdiv(m, oz::bn_max(S));
    if (s->peers.world > 1) {
        // Row tiles of G shard over the ranks: this rank computes the columns of D that belong to its tiles (split over K
        // to fill its SMs), then the slabs are exchanged in place (far::gather_cols_kernel).  The m x n phase that follows
        // is replicated on bit-identical D.
        const int P = s->peers.world, m_tiles = cdiv(n, oz::kBM);
        const int per = cdiv(m_tiles, P);
        const int t0 = min(m_tiles, s->peers.rank * per), t1 = min(m_tiles, t0 + per);
        const int mine = t1 - t0;
        const int clusters = kSMs / 2, kblocks = cdiv(n, oz::kBK);
        const long long col0 = (long long)t0 * oz::kBM;
        const int ncols = (int)(min((long long)L.ld, (long long)t1 * oz::kBM) - col0);
        if (mine > 0) {
            // split count by the planner's cost model (rounds x (K blocks per unit + the per-unit fixed cost) + combine), never
            // below the int32-exact minimum: 40 tiles x 157 K blocks on 74 pairs -> 3 splits (2 rounds of 53) instead of 1 x 157
            const int smin = cdiv(n, L.oz_kmax), smax = max(smin, min(clusters, max(1, kblocks / 4)));
            int sp = smin;
            double best = 1e300;
            for (int c = smin; c <= smax; ++c) {
                const int rounds = cdiv((long long)mine * c, clusters);
                const double cost = rounds * (ceil((double)kblocks / c) + kOzUnitFixedKb) + (c > 1 ? 1.5 * c : 0.0);
                if (cost < best - 1e-9) { best = cost; sp = c; }
            }
            const int chunk = (int)round_up(cdiv(n, sp), oz::kBK);
            const int splits = cdiv(n, chunk);
            LCX_REQUIRE((long long)splits * m * L.ld <= L.slot[I_PART][0].cols, "split-K partial buffer too small");
            p.m_tile0 = t0;
            p.k_chunk = chunk;
            p.C = splits > 1 ? s->ptr(I_PART) : D;
            p.c_split_stride = splits > 1 ? (long long)m * L.ld : 0;
            LCX_TRY((oz::launch_oz_gemm<S, true>(s->map_x_k1, s->map_a_k1, p, dim3(n_tiles, mine, splits), s->stream)));
            LAUNCHED(s);
            if (splits > 1) {
                LCX_TRY(launch_reduce_splits(s->ptr(I_PART) + col0, splits, (long long)m * L.ld, D + col0, m,
                                             (int)min((long long)n - col0, (long long)mine * oz::kBM), L.ld, s->stream));
                LAUNCHED(s);
            }
        }
        if (ev) {
            LCX_CUDA(cudaEventRecord(ev[1], s->stream));
            LCX_CUDA(cudaEventRecord(ev[3], s->stream));
            LCX_CUDA(cudaEventRecord(ev[4], s->stream));
        }
        {
            unsigned long long epoch0 = 2ULL * s->ar_calls;
            s->ar_calls++;
            far::Peers pp = s->peers;
            int rows = m, c0 = (int)col0, nc = max(0, ncols);
            long long ldd = L.ld;
            void* args[] = {&pp, &rows, &ldd, &c0, &nc, &epoch0};
            LCX_CUDA(cudaLaunchCooperativeKernel((void*)far::gather_cols_kernel, dim3(kSMs), dim3(512), args, 0, s->stream));
            LAUNCHED(s);
        }
    } else {
    // Whole waves of full-K row tiles straight into D, then the remaining r < #clusters row tiles split over K so that they
    // fill one more (short) wave: 79 tiles on 74 pairs = 157 + 12 K blocks instead of 5 rounds of 40 + the per-unit drains.
    const GramPlan gp = gram_plan(n, m, S, L.oz_kmax);
    if (gp.full > 0) {
        p.C = D;
        p.c_split_stride = 0;
        p.k_chunk = (int)round_up(n, oz::kBK);
        LCX_TRY((oz::launch_oz_gemm<S, true>(s->map_x_k1, s->map_a_k1, p, dim3(n_tiles, gp.full, 1), s->stream)));
        LAUNCHED(s);
        if (gp.rest > 0) {
            const long long col0 = (long long)gp.full * oz::kBM;
            p.m_tile0 = gp.full;
            p.k_chunk = gp.chunk;
            p.C = gp.splits > 1 ? s->ptr(I_PART) : D;
            p.c_split_stride = gp.splits > 1 ? (long long)m * L.ld : 0;
            LCX_TRY((oz::launch_oz_gemm<S, true>(s->map_x_k1, s->map_a_k1, p, dim3(n_tiles, gp.rest, gp.splits), s->stream)));
            LAUNCHED(s);
            if (gp.splits > 1) {
                LCX_TRY(launch_reduce_splits(s->ptr(I_PART) + col0, gp.splits, (long long)m * L.ld, D + col0, m, (int)(n - col0),
                                             L.ld, s->stream));
                LAUNCHED(s);
            }
        }
        if (ev) {
            LCX_CUDA(cudaEventRecord(ev[1], s->stream));
            LCX_CUDA(cudaEventRecord(ev[3], s->stream));
            LCX_CUDA(cudaEventRecord(ev[4], s->stream));
        }
    } else {
    const bool split = L.oz1_splits > 1;
    p.C = split ? s->ptr(I_PART) : D;
    p.c_split_stride = split ? (long long)m * L.ld : 0;
    p.k_chunk = L.oz1_chunk;
    LCX_TRY((oz::launch_oz_gemm<S, true>(s->map_x_k1, s->map_a_k1, p, dim3(cdiv(m, oz::bn_max(S)), cdiv(n, oz::kBM), L.oz1_splits),
                                         s->stream)));
    LAUNCHED(s);
    if (ev) LCX_CUDA(cudaEventRecord(ev[1], s->stream));
    if (ev) LCX_CUDA(cudaEventRecord(ev[3], s->stream));
    if (ev) LCX_CUDA(cudaEventRecord(ev[4], s->stream));
    if (split && leave_partials && svec == nullptr) {
        s->d_splits = L.oz1_splits;  // the consumer (direction_stage2) adds the partials itself, in index order
    } else if (split) {
        LCX_TRY(launch_reduce_splits(s->ptr(I_PART), L.oz1_splits, (long long)m * L.ld, D, m, n, L.ld, s->stream));
        LAUNCHED(s);
    }
    }
    }
    if (svec) {
        row_dot_kernel<<<m, 256, 0, s->stream>>>(A, D, svec, n, L.ld);
        LAUNCHED(s);
    }
    LCX_CUDA(cudaGetLastError());
    return 0;
}

static int gram_pair(lcx_session* s, const double* A, double* svec, cudaEvent_t* ev, const double* dot_b = nullptr,
                     double* dot_out = nullptr, bool leave_partials = false) {
    switch (s->L.S) {
        case 3: return gram_pair_t<3>(s, A, svec, ev, dot_b, dot_out, leave_partials);
        case 4: return gram_pair_t<4>(s, A, svec, ev, dot_b, dot_out, leave_partials);
        case 5: return gram_pair_t<5>(s, A, svec, ev, dot_b, dot_out, leave_partials);
        case 6: return gram_pair_t<6>(s, A, svec, ev, dot_b, dot_out, leave_partials);
        case 7: return gram_pair_t<7>(s, A, svec, ev, dot_b, dot_out, leave_partials);
    }
    return fail(LCX_ERR_STATE, "gram_pair", "bad digit count");
}
