// The steps of one fit iteration as sequences of launches on the session stream (no host synchronisation here):
// the X pass pair + exchange, the moment tail, direction and trial.  Included by lcx_api.cu after host_oz.cuh.
#pragma once
#include <atomic>

#include "host_oz.cuh"
#include "host_gram.cuh"

// ---- GEMM plumbing -----------------------------------------------------------------------------
// Sum over ranks of [body = sum_z part[z] (rows x ld, valid cols) | tail (ntail doubles)] -> dst_body / dst_tail.
// Peer path: ONE kernel (split-K combine + two-shot all-reduce over NVLink peer memory).  Otherwise the fixed-order
// local combine followed by the installed hook (NCCL through torch.distributed), or nothing on a single rank.
static int combine_and_allreduce(lcx_session* s, const double* part, int splits, long long stride, int rows, int cols,
                                 long long ld, double* dst_body, double* tail, int ntail) {
    const long long body = (long long)rows * ld;
    if (s->peers.world > 1) {
        LCX_REQUIRE(body + ntail <= s->peers.count, "peer buffer too small");
        const int slot = (int)(s->ar_calls & 1);
        unsigned long long epoch0 = 2ULL * s->ar_calls;
        s->ar_calls++;
        far::Peers pp = s->peers;
        const double* tl = tail;
        void* args[] = {&pp, &part, &splits, &stride, &rows, &cols, &ld, &tl, &ntail, (void*)&slot, &epoch0};
        LCX_CUDA(cudaLaunchCooperativeKernel((void*)far::reduce_allreduce_kernel, dim3(kSMs), dim3(512), args, 0, s->stream));
        LAUNCHED(s);
        const double* out = s->peers.base[s->peers.rank] + 2 * s->peers.count;
        if ((rows > 0 ? dst_body == out : true) && (ntail > 0 ? tail == out + body : true)) return 0;  // D lives there already
        if (rows > 0 && ntail > 0 && tail == dst_body + body) {  // D and the sums of squares are adjacent: one copy
            LCX_CUDA(cudaMemcpyAsync(dst_body, out, (size_t)(body + ntail) * sizeof(double), cudaMemcpyDeviceToDevice, s->stream));
            return 0;
        }
        if (rows > 0)
            LCX_CUDA(cudaMemcpyAsync(dst_body, out, (size_t)body * sizeof(double), cudaMemcpyDeviceToDevice, s->stream));
        if (ntail > 0)
            LCX_CUDA(cudaMemcpyAsync(tail, out + body, (size_t)ntail * sizeof(double), cudaMemcpyDeviceToDevice, s->stream));
        return 0;
    }
    if (rows > 0 && (splits > 1 || part != dst_body)) {
        LCX_TRY(launch_reduce_splits(part, splits, stride, dst_body, rows, cols, ld, s->stream));
        LAUNCHED(s);
    }
    if (s->hook) {
        // body and tail are contiguous in the workspace (D is followed by the column sums of squares)
        const long long off = (rows > 0 ? dst_body : tail) - s->ws;
        if (s->hook(s->hook_user, off, (rows > 0 ? body : 0) + ntail) != 0)
            return fail(LCX_ERR_STATE, "allreduce hook", "hook reported failure");
    }
    return 0;
}

static int run_gemm(lcx_session* s, GemmLayout lay, const GemmPlan& pl, GemmArgs a, double* part, long long out_count,
                    bool leave_partials = false) {
    // out_count = number of doubles of one full output (rows * ldc) -- the split stride
    if (pl.splits > 1 && leave_partials) {
        LCX_REQUIRE(a.Cadd == nullptr, "split-K with Cadd is not supported");
        a.C = part;
        a.c_split_stride = out_count;
        LCX_TRY(launch_gemm(lay, pl, a, s->stream));
        LAUNCHED(s);
    } else if (pl.splits > 1) {
        double* final_c = a.C;
        const double* cadd = a.Cadd;
        LCX_REQUIRE(cadd == nullptr, "split-K with Cadd is not supported");
        a.C = part;
        a.c_split_stride = out_count;
        LCX_TRY(launch_gemm(lay, pl, a, s->stream));
        LAUNCHED(s);
        const int out_rows = a.trans_out ? a.N : a.M, out_cols = a.trans_out ? a.M : a.N;
        LCX_TRY(launch_reduce_splits(part, pl.splits, out_count, final_c, out_rows, out_cols, a.ldc, s->stream));
        LAUNCHED(s);
    } else {
        a.c_split_stride = 0;
        LCX_TRY(launch_gemm(lay, pl, a, s->stream));
        LAUNCHED(s);
    }
    return 0;
}

// m x m product over the variables (ry, H): split-K GEMM whose fixed-order combine also performs np.fill_diagonal
// (raw diagonal -> diag_out if given, diag_value stored) -- one launch less than combine + diag kernel.
static int run_square_gemm(lcx_session* s, GemmArgs a, double diag_value, double* diag_out) {
    const Layout& L = s->L;
    const int m = s->m;
    const long long out_count = (long long)m * L.ldm;
    if (L.plan_mm.splits > 1) {
        double* final_c = a.C;
        a.C = s->ptr(I_PART);
        a.c_split_stride = out_count;
        LCX_TRY(launch_gemm(kLayoutKK, L.plan_mm, a, s->stream));
        LAUNCHED(s);
        LCX_TRY(launch_reduce_splits(s->ptr(I_PART), L.plan_mm.splits, out_count, final_c, m, m, L.ldm, s->stream,
                                     diag_out ? diag_out : s->ptr(I_F), diag_value));
        LAUNCHED(s);
    } else {
        double* final_c = a.C;
        LCX_TRY(run_gemm(s, kLayoutKK, L.plan_mm, a, s->ptr(I_PART), out_count));
        diag_fix_kernel<<<cdiv(m, 128), 128, 0, s->stream>>>(final_c, L.ldm, m, diag_value, diag_out);
        LAUNCHED(s);
    }
    return 0;
}

// Y = X~ A^T (+ colsq into D's tail), D = X~^T Y summed over splits, then the rank all-reduce.
// dot_b / dot_out (optional): dot_out_j = sum_i A_ji dot_b_ji, taken in the first pass over A where the route has one (split
// modes), by a row_dot launch otherwise.  leave_partials: the Gram route may hand D over as split-K partials (s->d_splits).
static int xpair(lcx_session* s, const double* A, bool want_colsq, const double* dot_b = nullptr, double* dot_out = nullptr,
                 bool leave_partials = false) {
    const Layout& L = s->L;
    const int m = s->m, n = s->n;
    double* Y = s->ptr(LCX_A_Y);
    double* D = s->ptr(LCX_A_D);
    double* svec = D + (long long)m * L.ld;
    cudaEvent_t* ev = nullptr;
    if (s->prof_on && s->prof_pending < s->prof_cap) ev = s->prof_ev + kProfEv * s->prof_pending;
    if (ev) LCX_CUDA(cudaEventRecord(ev[0], s->stream));
    if (s->gram) {  // one product with the n x n Gram matrix instead of the two passes over X~ (host_gram.cuh)
        LCX_TRY(gram_pair(s, A, want_colsq ? svec : nullptr, ev, dot_b, dot_out, leave_partials));
        if (ev) {
            LCX_CUDA(cudaEventRecord(ev[2], s->stream));
            s->prof_pending++;
        }
    } else if (L.S > 0) {
        LCX_TRY(oz_pair(s, A, svec, ev, false, want_colsq, dot_b, dot_out));
        if (ev) {
            LCX_CUDA(cudaEventRecord(ev[2], s->stream));
            s->prof_pending++;
        }
    } else {
    if (dot_out) {
        row_dot_kernel<<<m, 256, 0, s->stream>>>(A, dot_b, dot_out, n, L.ld);
        LAUNCHED(s);
    }
    {   // K1
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = s->xt; a.B = A; a.C = Y;
        a.M = (int)s->Nl; a.N = m; a.K = n;
        a.lda = s->ldx; a.ldb = L.ld; a.ldc = L.ldy;
        const bool k1_split = L.plan_k1.splits > 1;
        a.colsq_part = (want_colsq && !k1_split) ? s->ptr(I_COLSQ) : nullptr;
        a.ld_colsq = (int)L.ldy;
        LCX_TRY(run_gemm(s, kLayoutKK, L.plan_k1, a, k1_split ? s->ptr(I_PART) : nullptr, s->Nl * L.ldy));
        if (ev) LCX_CUDA(cudaEventRecord(ev[1], s->stream));
        if (want_colsq && k1_split) {  // split over variables: the sums of squares come from the reduced Y
            double* ystat = s->ws + L.slot[I_YSTAT][0].off;
            oz::y_stats_kernel<<<dim3(cdiv(m, 32), L.ystat_slabs), dim3(32, 8), 0, s->stream>>>(Y, L.ldy, s->Nl, m, kYStatRows, ystat,
                                                                                          L.ldm);
            LAUNCHED(s);
            oz::y_stats_finish_kernel<<<m, 256, 0, s->stream>>>(ystat, L.ystat_slabs, L.ldm, m, s->oz_xscale(), svec, s->oz_yscale(),
                                                               s->oz_dscale());
            LAUNCHED(s);
        } else if (want_colsq) {
            reduce_colsq_kernel<<<cdiv(m, 128), 128, 0, s->stream>>>(s->ptr(I_COLSQ), L.plan_k1.grid.x, (int)L.ldy, svec, m);
            LAUNCHED(s);
        }
    }
    {   // K2: (X~^T Y)^T written factor-major
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = s->xt; a.B = Y; a.C = D;
        a.M = n; a.N = m; a.K = (int)s->Nl;
        a.lda = s->ldx; a.ldb = L.ldy; a.ldc = L.ld;
        a.trans_out = 1;
        if (ev) LCX_CUDA(cudaEventRecord(ev[3], s->stream));  // K2 starts after the (tiny) colsq reduction
        LCX_TRY(run_gemm(s, kLayoutMN, L.plan_k2, a, s->ptr(I_PART), (long long)m * L.ld, true));
        if (ev) LCX_CUDA(cudaEventRecord(ev[4], s->stream));
        const bool split = L.plan_k2.splits > 1;
        LCX_TRY(combine_and_allreduce(s, split ? s->ptr(I_PART) : D, split ? L.plan_k2.splits : 1, (long long)m * L.ld, m, n, L.ld,
                                      D, svec, want_colsq ? m : 0));
        if (ev) {
            LCX_CUDA(cudaEventRecord(ev[2], s->stream));
            s->prof_pending++;
        }
    }
    }
    LCX_CUDA(cudaGetLastError());
    return 0;
}

// scalars: 16 device doubles to post; default: the bound workspace's LCX_A_SCALARS (free-standing calls pass their own).
static int read_mailbox(lcx_session* s, const double* scalars = nullptr) {
    if (scalars == nullptr) scalars = s->ptr(LCX_A_SCALARS);
    const unsigned long long seq = ++s->mailbox_seq;
    post_mailbox_kernel<<<1, 32, 0, s->stream>>>(scalars, s->mailbox, seq);
    LAUNCHED(s);
    volatile unsigned long long* flag = reinterpret_cast<volatile unsigned long long*>(s->mailbox + 16);
    unsigned polls = 0;
    while (*flag != seq) {
        if ((++polls & 0x3fffu) == 0) {  // every ~16k polls: has the stream failed, or drained without the flag landing?
            const cudaError_t q = cudaStreamQuery(s->stream);
            if (q == cudaSuccess) {
                if (*flag == seq) break;
                LCX_CUDA(cudaStreamSynchronize(s->stream));
                if (*flag != seq) return fail(LCX_ERR_CUDA, "read_mailbox", "the mailbox post never arrived");
                break;
            }
            if (q != cudaErrorNotReady) return fail(LCX_ERR_CUDA, "read_mailbox", cudaGetErrorString(q));
        }
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    return 0;
}

// ry, Qij, Qi-Si^2, TC, uj for `set`, given rho/invrho/rinv/Si (and W) of that set.
static int moments_tail(lcx_session* s, int set, double c1, double e2, int uj_mode) {
    const Layout& L = s->L;
    const int m = s->m, n = s->n;
    double* W = s->ptr(LCX_A_W, set);
    double* rho = s->ptr(LCX_A_RHO, set);
    double* rinv = s->ptr(LCX_A_RHOINVRHO, set);
    double* ry = s->ptr(LCX_A_RY, set);
    double* Qij = s->ptr(LCX_A_QIJ, set);
    if (L.mm_i8) {  // both products as exact int8 digit-plane products on tcgen05
        LCX_TRY(oz_square(s, W, rho, ry, 1.0, s->ptr(I_UJDIAG)));
        LCX_TRY(oz_mn(s, ry, rinv, Qij, rinv, true));  // Qij = rinv + (ry - I) rinv
    } else {
    {   // ry = W rho^T  (:261), diag -> 1 (:263); the diagonal before the fill is uj by linearity
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = W; a.B = rho; a.C = ry;
        a.M = m; a.N = m; a.K = n;
        a.lda = L.ld; a.ldb = L.ld; a.ldc = L.ldm;
        LCX_TRY(run_square_gemm(s, a, 1.0, s->ptr(I_UJDIAG)));
    }
    {   // Qij = ry rinv  (:266)
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = ry; a.B = rinv; a.C = Qij;
        a.M = m; a.N = n; a.K = m;
        a.lda = L.ldm; a.ldb = L.ld; a.ldc = L.ld;
        LCX_TRY(run_gemm(s, kLayoutKN, L.plan_mn, a, nullptr, 0));
    }
    }
    moments_stage2_kernel<<<L.nstrips, dim3(kStripCols, kStripRows), 0, s->stream>>>(
        rho, rinv, Qij, s->ptr(LCX_A_SI, set), s->ptr(LCX_A_QISI2, set), s->ptr(I_SPART), m, n, L.ld);
    LAUNCHED(s);
    moments_finish_kernel<<<1, 256, 0, s->stream>>>(s->ptr(I_SPART), L.nstrips, uj_mode,
                                                   s->ptr(LCX_A_D) + (long long)m * L.ld, s->ptr(I_W2), s->ptr(I_UJDIAG), c1,
                                                   e2, s->ptr(LCX_A_UJ, set), m, s->ptr(LCX_A_SCALARS));
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}

// full from-X moment evaluation of W(set) into `set`
static int moments_from_x(lcx_session* s, int set, double eps) {
    const Layout& L = s->L;
    const int m = s->m, n = s->n;
    const double c1 = (1.0 - eps * eps) / (double)s->Nt, e2 = eps * eps;
    double* W = s->ptr(LCX_A_W, set);
    LCX_TRY(xpair(s, W, true));
    row_dot_kernel<<<m, 256, 0, s->stream>>>(W, W, s->ptr(I_W2), n, L.ld);
    LAUNCHED(s);
    moments_stage1_kernel<true><<<L.nstrips, dim3(kStripCols, kStripRows), 0, s->stream>>>(
        s->ptr(LCX_A_D), W, nullptr, nullptr, nullptr, 0.0, c1, e2, nullptr, s->ptr(LCX_A_RHO, set),
        s->ptr(LCX_A_INVRHO, set), s->ptr(LCX_A_RHOINVRHO, set), s->ptr(LCX_A_SI, set), m, n, L.ld);
    LAUNCHED(s);
    return moments_tail(s, set, c1, e2, 0);
}

static int enqueue_direction(lcx_session* s, double eps) {
    const Layout& L = s->L;
    const int m = s->m, n = s->n;
    const double c1 = (1.0 - eps * eps) / (double)s->Nt, e2 = eps * eps;
    double* W = s->ptr(LCX_A_W);
    double* rho = s->ptr(LCX_A_RHO);
    double* rinv = s->ptr(LCX_A_RHOINVRHO);
    double* G = s->ptr(LCX_A_GRAD);
    double* T = s->ptr(I_T);
    double* H = s->ptr(I_RYINV);  // m x ldm scratch (the inverse buffer is idle outside the details path)
    direction_stage1_kernel<<<grid_mn(m, n), 256, 0, s->stream>>>(W, rho, s->ptr(LCX_A_INVRHO), rinv, s->ptr(LCX_A_QIJ),
                                                                s->ptr(LCX_A_SI), s->ptr(LCX_A_QISI2), s->ptr(LCX_A_UJ), T, G,
                                                                m, n, L.ld);
    LAUNCHED(s);
    if (L.mm_i8) {
        LCX_TRY(oz_square(s, T, rinv, H, 0.0, nullptr));  // H = T rinv^T, diag -> 0 (:294-295)
        LCX_TRY(oz_mn(s, H, W, G, G, false));             // grad = G0 + H W (:300)
    } else {
    {   // H = T rinv^T, diag -> 0 (:294-295)
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = T; a.B = rinv; a.C = H;
        a.M = m; a.N = m; a.K = n;
        a.lda = L.ld; a.ldb = L.ld; a.ldc = L.ldm;
        LCX_TRY(run_square_gemm(s, a, 0.0, nullptr));
    }
    {   // grad = G0 + H W (:300), in place over G0
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = H; a.B = W; a.C = G; a.Cadd = G;
        a.M = m; a.N = n; a.K = m;
        a.lda = L.ldm; a.ldb = L.ld; a.ldc = L.ld;
        LCX_TRY(run_gemm(s, kLayoutKN, L.plan_mn, a, nullptr, 0));
    }
    }
    // X~^T (X~ grad^T): the one pass over X of this iteration (:301); Bj = sum_i rho grad (:302) rides on its first pass over grad
    s->d_splits = 1;
    LCX_TRY(xpair(s, G, false, rho, s->ptr(I_BJ), true));
    const dim3 g2(cdiv(n, 256), m);
    const bool parts = s->d_splits > 1;
    direction_stage2_kernel<<<g2, 256, 0, s->stream>>>(W, rho, G, parts ? s->ptr(I_PART) : s->ptr(LCX_A_D), s->ptr(LCX_A_UJ),
                                                     s->ptr(I_BJ), c1, e2, s->ptr(LCX_A_UPDATE), s->ptr(LCX_A_RDIR),
                                                     s->ptr(I_SPART), m, n, L.ld, s->d_splits, (long long)m * L.ld);
    LAUNCHED(s);
    // (a last-CTA sum inside direction_stage2 was measured slower: 4 000 CTAs queue on one arrival counter)
    sum_partials_kernel<<<1, 256, 0, s->stream>>>(s->ptr(I_SPART), (int)(g2.x * g2.y), s->ptr(LCX_A_SCALARS) + 2);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}

static int enqueue_trial(lcx_session* s, double eps, double eta, int exact) {
    const Layout& L = s->L;
    const int m = s->m, n = s->n;
    const double c1 = (1.0 - eps * eps) / (double)s->Nt, e2 = eps * eps;
    if (exact) {
        axpy_kernel<<<grid_mn(m, n), 256, 0, s->stream>>>(s->ptr(LCX_A_W), s->ptr(LCX_A_UPDATE), eta, s->ptr(LCX_A_W, 1), m, n,
                                                        L.ld);
        LAUNCHED(s);
        LCX_TRY(moments_from_x(s, 1, eps));
    } else {
        moments_stage1_kernel<false><<<L.nstrips, dim3(kStripCols, kStripRows), 0, s->stream>>>(
            nullptr, s->ptr(LCX_A_W), s->ptr(LCX_A_UPDATE), s->ptr(LCX_A_RHO), s->ptr(LCX_A_RDIR), eta, c1, e2,
            s->ptr(LCX_A_W, 1), s->ptr(LCX_A_RHO, 1), s->ptr(LCX_A_INVRHO, 1), s->ptr(LCX_A_RHOINVRHO, 1),
            s->ptr(LCX_A_SI, 1), m, n, L.ld);
        LAUNCHED(s);
        LCX_TRY(moments_tail(s, 1, c1, e2, 1));
    }
    return 0;
}

// X (m x ldx, n columns) = A^-1 B by LU with partial pivoting (np.linalg.solve, linearcorex.py:280 / :366).  The status word
// of the factorisation lands in scalars[8] (read back with the mailbox: non-zero = singular matrix).
static int run_solve(lcx_session* s, const double* a, long long lda, const double* b, long long ldb, double* x, long long ldx) {
    LCX_TRY(lu::solve(a, lda, s->m, b, ldb, x, ldx, s->n, s->ptr(I_AUG), s->ptr(LCX_A_SCALARS) + 8, s->stream, &s->launches));
    return 0;
}

// shared tail of the details computations: MI, X_i^2|Y, I(X_i;Y), TCs, TC_no_overlap, TC_direct, additivity
static int details_tail(lcx_session* s, const double* other, const double* yj2_in) {
    const Layout& L = s->L;
    const int m = s->m, n = s->n;
    details_cols_kernel<<<L.nstrips, dim3(kStripCols, kStripRows), 0, s->stream>>>(
        s->ptr(LCX_A_RHO), s->ptr(LCX_A_XZ), other, s->ptr(LCX_A_MI), s->ptr(LCX_A_X2Y), s->ptr(LCX_A_IXY), s->ptr(I_SPART),
        m, n, L.ld);
    LAUNCHED(s);
    row_dot_kernel<<<m, 256, 0, s->stream>>>(s->ptr(LCX_A_MI), nullptr, s->ptr(I_ROWMI), n, L.ld);
    LAUNCHED(s);
    details_finish_kernel<<<1, 256, 0, s->stream>>>(s->ptr(I_SPART), L.nstrips, s->ptr(LCX_A_UJ), yj2_in, s->ptr(I_ROWMI),
                                                   s->ptr(LCX_A_YJ2), s->ptr(LCX_A_IYX), s->ptr(LCX_A_TCS),
                                                   s->ptr(LCX_A_TCDIRECT), s->ptr(I_SQRTY), m, s->ptr(LCX_A_SCALARS) + 4);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}
