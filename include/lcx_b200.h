/* lcx_b200.h -- C ABI of the B200-native Linear CorEx fit-loop library (liblcx_b200.so).
 *
 * This is the drop-in boundary for the hot path of gregversteeg/LinearCorex
 * (linearcorex/linearcorex.py, class Corex).  The reference has no FFI of its own: its only
 * accelerator seam is the `if self.gpu:` cudamat branch (cm.CUDAMatrix / cm.dot / .asarray at
 * linearcorex.py:199-208, :217-223, :240-256, :340-352, :427-428), which ships Y and X^T Y back to
 * the host after every GEMM.  The entry points below replace that seam one level up -- the array
 * math of _calculate_moments_{ns,syn}, _sig, _norm, _update_{ns,syn}, preprocess, transform and
 * get_covariance -- and are what a ctypes binding inside the reference would call (INTEGRATION.md).
 *
 * Conventions
 *   - Every function returns an int: 0 = ok, LCX_QUICK_FAIL (1) = "max uj >= 1" (the reference's
 *     `return False`, linearcorex.py:250-251), negative = error; lcx_last_error() gives the text.
 *     No exception ever crosses this boundary.
 *   - The library owns no array memory.  X~, the workspace and every output are device pointers
 *     supplied by the caller (torch tensors in the shipped host code) with explicit sizes and
 *     leading dimensions.  The session holds only launch state, a stream, a small pinned mailbox
 *     for the O(1) scalars that gate host control flow, and pointers into the caller's workspace.
 *   - All work is enqueued on the session's stream.  A call synchronises that stream only when it
 *     returns host scalars (TC, max uj, tangent).
 *   - Factor-major arrays (W, rho, ...) are m x n row-major with leading dimension lcx_ld(n)
 *     (n rounded up to 16); the n x m arrays of the reference (X_i Y_j, X_i Z_j) are stored
 *     transposed in that same layout.
 *   - Sessions are not thread-safe; one host thread per GPU (one process per GPU under torchrun).
 *   - Rows of X may be sharded across ranks: lcx_set_allreduce() installs the hook the library
 *     calls wherever the reference's single-process sum over samples must become a sum over ranks.
 */
#ifndef LCX_B200_H
#define LCX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LCX_OK 0
#define LCX_QUICK_FAIL 1
#define LCX_ERR_ARG (-1)
#define LCX_ERR_CUDA (-2)
#define LCX_ERR_STATE (-3)
#define LCX_ERR_SINGULAR (-4) /* a pivot of the details-path solve was exactly zero: numpy raises LinAlgError there */
#define LCX_ERR_NOT_PD (-5)   /* the covariance estimate is not (treated as) positive definite: lcx_lowrank_factor */

/* precision modes */
#define LCX_PRECISION_FP64 0   /* DMMA (mma.sync m8n8k4 f64) contractions, everything in binary64 */
#define LCX_PRECISION_FAST 1   /* opt-in fast mode: split-integer tcgen05 (kind::i8) X contractions, 3 digits = 24 bits
                                  (fp32-equivalent products, like 3xTF32), everything else binary64; parity 1e-4 */
#define LCX_PRECISION_FP64_SPLIT 2 /* FP64-faithful split-integer tcgen05 X contractions: 6 radix-254 digits = 48 bits below
                                      the row/column maximum (truncation at the level of binary64 rounding; measured parity
                                      1e-11 or better against the reference's float64 path), everything else binary64 */
#define LCX_PRECISION_FP64_SPLIT5 3 /* the same with 5 digits = 40 bits: 30 % faster, parity 1e-9 on fits of up to ~700
                                       iterations (2e-9 on the 2400-iteration adni fixture) */
#define LCX_PRECISION_FP64_SPLIT7 4 /* 7 digits = 56 bits, finer than binary64's 53-bit significand: for ill-conditioned fits
                                       (pure-noise data, extreme outliers) where the 48-bit mode's perturbation is amplified
                                       past 1e-9; 28 instead of 21 plane products, two pipeline stages */

/* input dtypes of raw X */
#define LCX_F32 0
#define LCX_F64 1

/* gaussianize modes (linearcorex.py:407-423) */
#define LCX_GAUSS_STANDARD 0
#define LCX_GAUSS_OUTLIERS 1
#define LCX_GAUSS_NONE 2

/* workspace arrays addressable through lcx_array_info(); "set" 0 = current moments, 1 = trial */
enum lcx_array {
    LCX_A_W = 0,        /* m x ld   weights `ws`                                   (set) */
    LCX_A_RHO,          /* m x ld   moments['rho']                                 (set) */
    LCX_A_INVRHO,       /* m x ld   moments['invrho']                              (set) */
    LCX_A_RHOINVRHO,    /* m x ld   moments['rhoinvrho']                           (set) */
    LCX_A_QIJ,          /* m x ld   moments['Qij']                                 (set) */
    LCX_A_SI,           /* ld       moments['Si']                                  (set) */
    LCX_A_QISI2,        /* ld       moments['Qi-Si^2'] (ns) / moments['Qi'] (syn)  (set) */
    LCX_A_RY,           /* m x ldm  moments['ry']                                  (set) */
    LCX_A_UJ,           /* m        moments['uj']                                  (set) */
    LCX_A_GRAD,         /* m x ld   grad of _update_ns (:296-300)                        */
    LCX_A_UPDATE,       /* m x ld   update (:303)                                        */
    LCX_A_RDIR,         /* m x ld   _sig(update)                                         */
    LCX_A_D,            /* m x ld (+ m) all-reduce buffer: X~^T(X~ A^T) then sum Y^2     */
    LCX_A_MI,           /* m x ld   moments['MI']                                        */
    LCX_A_XZ,           /* m x ld   moments['X_i Z_j']^T                                 */
    LCX_A_XY,           /* m x ld   moments['X_i Y_j']^T                                 */
    LCX_A_X2Y,          /* ld       moments['X_i^2 | Y']                                 */
    LCX_A_IXY,          /* ld       moments['I(X_i ; Y)']                                */
    LCX_A_YJ2,          /* m        moments['Y_j^2']                                     */
    LCX_A_IYX,          /* m        moments['I(Y_j ; X)']                                */
    LCX_A_TCS,          /* m        moments['TCs']                                       */
    LCX_A_TCDIRECT,     /* m        moments['TC_direct']                                 */
    LCX_A_CY,           /* m x ldm  moments['cy'] (syn)                                  */
    LCX_A_Y,            /* N_local x ldy   Y = X~ A^T of the last projection             */
    LCX_A_SCALARS,      /* 16       [0] TC [1] max uj [2] tangent [4] TC_no_overlap [5] sum I(X_i;Y)
                                    [6] additivity [7] sum I(Y_j;X) [8] status of the details-path solve */
    LCX_A_COUNT
};

typedef struct lcx_session lcx_session;

/* Sum `count` doubles at workspace offset `offset` (in doubles) over all ranks, in place, ordered
 * on the session stream.  Installed by multi-GPU callers; NULL (default) = single rank. */
typedef int (*lcx_allreduce_fn)(void* user, long long offset, long long count);

/* ---- lifecycle ------------------------------------------------------------------------------ */
int lcx_version(void);
const char* lcx_last_error(void);
int lcx_session_create(lcx_session** out, int device, int precision);
int lcx_session_destroy(lcx_session* s);
int lcx_set_stream(lcx_session* s, void* cuda_stream);
int lcx_set_allreduce(lcx_session* s, lcx_allreduce_fn fn, void* user);
/* Sample sharding over NVLink peer memory (preferred over the hook when every rank can map every other rank's
 * buffer): `bases[r]` = rank r's copy of one symmetric buffer of lcx_peer_buffer_doubles() doubles, zero-filled
 * before the first call on any rank.  With peers set, the split-K combine of X~^T Y and the sum over ranks run as
 * ONE kernel (two-shot reduce-scatter / all-gather with P2P loads and stores, release/acquire flags), and every
 * rank ends with bit-identical moments.  Call after lcx_bind; world <= 1 or bases == NULL switches it off. */
long long lcx_peer_buffer_doubles(int n_vars, int n_factors);
int lcx_set_peer_allreduce(lcx_session* s, int world, int rank, void* const* bases, long long buffer_doubles);
int lcx_launch_count(lcx_session* s, long long* launches);   /* kernels launched so far by this session */
/* Device-side timing of the two X contractions (CUDA events on the session stream around each launch).
 * lcx_profile_read synchronises the stream and returns accumulated milliseconds and the pair count. */
int lcx_profile_enable(lcx_session* s, int on);
int lcx_profile_read(lcx_session* s, double* k1_ms, double* k2_ms, long long* pairs, int reset);
/* The same with the second contraction split into the kernel itself and what follows it: the split-K combine and the
 * exchange over ranks (lcx_profile_read's k2_ms is their sum). */
int lcx_profile_read_phases(lcx_session* s, double* k1_ms, double* k2_ms, double* exchange_ms, long long* pairs, int reset);

/* ---- layout --------------------------------------------------------------------------------- */
long long lcx_ld(int n_vars);                       /* leading dimension of m x n arrays */
long long lcx_ldy(int n_factors);                   /* leading dimension of Y            */
/* Doubles the caller must provide to lcx_bind for a problem of this size. */
long long lcx_workspace_doubles(long long n_rows_local, int n_vars, int n_factors, int precision);
/* Bind a preprocessed data block X~ (n_rows_local x n_vars, fp64, ld = ldx) and a workspace.
 * n_rows_total = sum of n_rows_local over ranks (the reference's n_samples, :110).
 * LCX_PRECISION_FP64: xt must stay valid while the session is bound.  Split modes: xt is converted to int8 digit
 * planes inside the workspace before lcx_bind returns and may be released by the caller afterwards. */
int lcx_bind(lcx_session* s, const double* xt, long long n_rows_local, long long n_rows_total, int n_vars,
             long long ldx, int n_factors, double* workspace, long long workspace_doubles);
/* Streamed binding for data whose fp64 X~ does not fit beside its digit planes (split modes only): call lcx_bind with
 * xt == NULL, then lcx_set_x_scale(max |X~|) once and lcx_slice_block for every row block [row0, row0 + rows) of X~
 * (any order, each row exactly once) before the first fit step.  A NaN or infinite max_abs (non-finite data) sets a NaN
 * scale: every product then comes out NaN, which is what the reference's float64 path does with such data. */
int lcx_set_x_scale(lcx_session* s, double max_abs);
int lcx_slice_block(lcx_session* s, const double* xt, long long row0, long long rows, long long ldx);
/* The same for raw rows: lcx_standardize (:397-429, :483-487, :497-510) and lcx_slice_block fused into one pass -- the fp32 /
 * fp64 source goes straight into the int8 digit planes of rows [row0, row0 + n_rows), X~ never exists in binary64 (4 or 8
 * bytes read + S written per element).  Bit-identical planes to the two-call sequence. */
int lcx_standardize_slice(lcx_session* s, const void* x, int dtype, long long row0, long long n_rows, long long ldx,
                          int has_marker, double marker, int gauss_mode, const double* impute, const double* mean,
                          const double* sd);
/* ---- Gram route (N >= n) ------------------------------------------------------------------------------------------
 * Every quantity of the fit depends on the data only through X~^T X~ / N: _sig (linearcorex.py:196-213) is
 * u -> (X~^T X~ / N) u^T and sum_l Y_lj^2 / N = a_j^T (X~^T X~ / N) a_j (:248, :227).  The reference avoids the n x n matrix
 * because it targets n >> N (:197-198); for N >= n forming it once replaces the two N x n x m contractions of every
 * iteration by one n x n x m product.
 * lcx_gram_build: g (n x ldg fp64 device, ldg = lcx_ld(n)) = this rank's X~^T X~ / n_rows_total, from the digit planes of a
 *   split-mode session bound to X~ (exact int8 digit products on tcgen05, upper triangle computed and mirrored).  The
 *   caller sums g over ranks.  block_cols (multiple of 128) = variables per pass over X~.
 * lcx_bind_gram: bind a (second) split-mode session to the summed matrix; every fit-loop entry point below then works
 *   unchanged on it -- lcx_sig, lcx_moments_*, lcx_direction_*, lcx_trial_ns, lcx_update_syn -- and needs no exchange
 *   between ranks (each rank holds the same matrix).  g may be released after the call. */
long long lcx_gram_scratch_doubles(lcx_session* s, int block_cols);
int lcx_gram_build(lcx_session* s, double* g, long long ldg, int block_cols, double* scratch, long long scratch_doubles);
long long lcx_gram_workspace_doubles(int n_vars, int n_factors, int precision);
int lcx_bind_gram(lcx_session* s, const double* g, long long ldg, int n_vars, int n_factors, double* workspace,
                  long long workspace_doubles);
/* Split modes: location of the int8 digit planes ([digits][rows][ld_bytes], offset in doubles from the workspace base) of
 * which = 0: X~ (rows = local samples, cols = variables), 1: the last small operand A (W or grad; rows = factors,
 * cols = variables), 2: Y, stored transposed (rows = factors, cols = local samples); and of their scales (1 value for
 * X~, one per factor otherwise).  For inspection and the bit-exact digit tests. */
int lcx_digit_planes_info(lcx_session* s, int which, long long* offset, int* digits, long long* rows, long long* cols,
                          long long* ld_bytes, long long* scale_offset, int* radix);
/* Offset (in doubles, from the workspace base), rows, cols and leading dimension of an array. */
int lcx_array_info(lcx_session* s, int array_id, int set, long long* offset, long long* rows, long long* cols,
                   long long* ld);

/* ---- preprocessing: linearcorex.py:397-429 (preprocess), :497-510 (mean_impute), :483-487 (g) --- */
/* pass 1: per-column sum and count of observed entries -> sum[n], cnt[n] (device).  scratch: slab partials */
int lcx_colstats_sum(lcx_session* s, const void* x, int dtype, long long n_rows, int n_vars, long long ldx,
                     int has_marker, double marker, double* sum, double* cnt, double* scratch,
                     long long scratch_doubles);
/* mean = sum / cnt  (after the caller all-reduced sum and cnt) */
int lcx_colstats_mean(lcx_session* s, const double* sum, const double* cnt, double* mean, int n_vars);
/* pass 2: per-column sum of squared deviations of observed entries -> sq[n] */
/* maxdev (optional, device, n): per-column max |x - mean| over observed entries, so that max |X~| is known before
 * X~ exists (streamed digit slicing) */
int lcx_colstats_sqdev(lcx_session* s, const void* x, int dtype, long long n_rows, int n_vars, long long ldx,
                       int has_marker, double marker, const double* mean, double* sq, double* maxdev, double* scratch,
                       long long scratch_doubles);
/* std = clip(sqrt(sq / (use_nobs ? cnt : n_rows_total)), 1e-10)   (:413 vs :421) */
int lcx_colstats_std(lcx_session* s, const double* sq, const double* cnt, double n_rows_total, int use_nobs,
                     double* sd, int n_vars);
/* X~ = g?((impute(x) - mean) / std), fp64, ld = ldo (columns >= n_vars zero-filled).  Missing entries
 * take impute[i] -- the column mean of the data being preprocessed (mean_impute runs on transform()
 * inputs too, :389/:404), which differs from theta's mean outside fit. */
int lcx_standardize(lcx_session* s, const void* x, int dtype, long long n_rows, int n_vars, long long ldx,
                    int has_marker, double marker, int gauss_mode, const double* impute, const double* mean,
                    const double* sd, double* out, long long ldo);
long long lcx_colstats_scratch_doubles(long long n_rows, int n_vars);

/* ---- the two X contractions ----------------------------------------------------------------- */
/* Y = X~ A^T  (:247, :210, :226, :394) and optionally colsq[j] = sum_l Y_lj^2 (:248, :227).
 * Free-standing (no bound problem needed): used by transform().  scratch >= lcx_project_scratch_doubles. */
int lcx_project(lcx_session* s, const double* xt, long long n_rows, int n_vars, long long ldx, const double* a,
                long long lda, int n_factors, double* y, long long ldy, double* colsq, double* scratch,
                long long scratch_doubles);
long long lcx_project_scratch_doubles(long long n_rows, int n_factors);
/* _sig (:196-213) on the bound X~: out = (1-eps^2) (X~^T (X~ u^T))^T / N + eps^2 u, all m x ld device arrays */
int lcx_sig(lcx_session* s, const double* u, double eps, double* out);

/* ---- fit-loop steps on the bound problem ----------------------------------------------------- */
int lcx_set_w(lcx_session* s, const double* host_w, long long host_ld);          /* upload ws (m x n) into set 0 */
int lcx_get_w(lcx_session* s, double* host_w, long long host_ld);                /* download set 0 ws           */
int lcx_init_scale(lcx_session* s, double eps);                                  /* ws /= 10 _norm(x, ws)  (:117) */
int lcx_stage_rescale(lcx_session* s, double eps, double eps_prev);              /* :130-133                      */
int lcx_permute_rows(lcx_session* s, const int* host_order);                     /* ws = ws[order]         (:162) */
/* _calculate_moments_ns(x, ws, quick=True) from X~ for set 0 (:236-276).  Returns LCX_QUICK_FAIL when
 * max uj >= 1 and check_uj != 0.  tc / max_uj are host outputs. */
int lcx_moments_ns(lcx_session* s, double eps, int check_uj, double* tc, double* max_uj);
/* the quick=False extras (:277-287) for set 0; host outputs: TC_no_overlap, additivity */
int lcx_details_ns(lcx_session* s, double* tc_no_overlap, double* additivity);
/* search direction of _update_ns (:292-305); host output: update_tangent */
int lcx_direction_ns(lcx_session* s, double eps, double* tangent);
/* one backtracking trial (:320-321): set 1 <- moments of ws + eta*update.
 * exact = 0: through the linearity of _sig (no pass over X);  exact = 1: from X~ like the reference. */
int lcx_trial_ns(lcx_session* s, double eps, double eta, int exact, double* tc, double* max_uj);
/* direction + first (linear) trial at `eta` enqueued back to back with ONE host synchronisation; the trial is
 * speculative -- discard it when tangent >= 0 (:306-311) */
int lcx_direction_trial_ns(lcx_session* s, double eps, double eta, double* tangent, double* tc, double* max_uj);
/* Up to max_iter iterations of one annealing stage -- the loop body of fit (:137-151) including _update_ns's backtracking
 * (:312-334) -- without returning to the caller between iterations.  Outputs per iteration i < *n_done: tc[i], tangent[i],
 * eta[i] (accepted step; 0 when tangent >= 0, :306-311), trials[i], quick_fails[i].  *stop_reason: 0 = max_iter done,
 * 1 = |delta TC| < tol (:152), 2 = the update yielded invalid moments (:144-149; iteration *n_done - 1, not applied). */
int lcx_run_stage_ns(lcx_session* s, double eps, double tol, int exact_trials, int max_iter, double tc_start, int* n_done,
                     int* stop_reason, double* tc, double* tangent, double* eta, int* trials, int* quick_fails);
int lcx_accept_trial(lcx_session* s);                                            /* set 0 <-> set 1 (:333-334)   */
/* _calculate_moments_syn (:336-373) for set 0; host output TC */
int lcx_moments_syn(lcx_session* s, double* tc, double* additivity);
/* _update_syn (:375-384): ws <- (1-eta) ws + eta (R - H ws), then moments_syn */
int lcx_update_syn(lcx_session* s, double eta, double* tc, double* additivity);

/* ---- get_covariance (:443-455) ---------------------------------------------------------------- */
/* rows [row0, row0+rows) of the n x n covariance into out (rows x ldc, device).  synergy = 0: ns formula
 * with eps; synergy = 1: X_i Z_j X_i Y_j^T.  sd = theta[1] (device, n). */
int lcx_get_covariance(lcx_session* s, int synergy, double eps, const double* sd, int row0, int rows, double* out,
                       long long ldc);
/* The same row block from explicit factors, with no bound problem (a model restored from a pickle holds only host
 * moments, which is all the reference reads at :443-455):  out = diag(sd) fill_diagonal(left^T right / scale, 1) diag(sd),
 * left / right factor-major n_factors x ld device arrays -- ns: left = right = rhoinvrho / (1 + Si), scale = 1 - eps^2;
 * synergy: left = X_i Z_j^T, right = X_i Y_j^T, scale = 1. */
int lcx_covariance_rows(lcx_session* s, const double* left, const double* right, long long ld, int n_factors, int n_vars,
                        double scale, const double* sd, int row0, int rows, double* out, long long ldc);

/* ---- scoring under the covariance estimate (ns variant; no bound problem needed) ------------------------------------
 * The ns estimate is low rank plus diagonal:  Sigma = S (Z^T Z + Delta) S  with  Z = rhoinvrho / (1 + Si) / sqrt(1 - eps^2),
 * Delta = diag(1 - sum_j Z_ji^2),  S = diag(sd).  With K = I + Z Delta^-1 Z^T = G G^T and B = G^-1 Z Delta^-1 (Woodbury):
 *   Sigma^-1 = S^-1 (Delta^-1 - B^T B) S^-1,   log det Sigma = 2 sum log sd + sum log Delta + 2 sum log G_kk.
 * lcx_lowrank_factor: rhoinvrho (m x ld), si (n), sd (n) device -> b (m x ldb), dinv (n) = 1 / Delta, logdet (1 double), all
 *   device, enqueued on the stream; ONE mailbox read returns the status: LCX_ERR_NOT_PD when some Delta_i <= 0 or a pivot of
 *   K is <= 0 (Delta_i <= 0 is a conservative test).  scratch >= lcx_lowrank_scratch_doubles(m, n).
 * lcx_score_rows: raw fp32 / fp64 rows (ld ldx) -> maha[l] = (x~_l)^T C^-1 x~_l (squared Mahalanobis distance, C = S^-1 Sigma
 *   S^-1) and logpdf[l] = log N(x_l; mean, Sigma), device, with x~ = (impute(x) - mean) / sd (lcx_standardize's 'standard'
 *   arithmetic).  All binary64 (DMMA); rows never share a reduction, so results do not depend on how rows are blocked.
 *   scratch >= lcx_score_scratch_doubles(n_rows, n_vars, n_factors).
 * lcx_precision_rows: rows [row0, row0 + rows) of Sigma^-1 into out (rows x ldc, device); row0 even, ldc even. */
long long lcx_lowrank_scratch_doubles(int n_factors, int n_vars);
int lcx_lowrank_factor(lcx_session* s, const double* rhoinvrho, const double* si, long long ld, int n_factors, int n_vars,
                       double eps, const double* sd, double* b, long long ldb, double* dinv, double* logdet, double* scratch,
                       long long scratch_doubles);
long long lcx_score_scratch_doubles(long long n_rows, int n_vars, int n_factors);
int lcx_score_rows(lcx_session* s, const void* x, int dtype, long long n_rows, int n_vars, long long ldx, int has_marker,
                   double marker, const double* impute, const double* mean, const double* sd, const double* b, long long ldb,
                   int n_factors, const double* dinv, const double* logdet, double* maha, double* logpdf, double* scratch,
                   long long scratch_doubles);
int lcx_precision_rows(lcx_session* s, const double* b, long long ldb, int n_factors, int n_vars, const double* dinv,
                       const double* sd, int row0, int rows, double* out, long long ldc);

/* ---- conditioning on the observed entries (ns variant) -----------------------------------------------------------------
 * For a row with missing set M and observed set O, in standardised space (x~ = (x - mean) / sd, Lambda = Delta^-1 - B^T B):
 *   x^_M = E[x~_M | x~_O] = Lambda_MM^-1 B_M^T B x~°  (x~° = x~ with the missing entries zeroed),
 *   q_O = x~_O^T (Sigma~_OO)^-1 x~_O,   log p(x_O) = log N(x_O; mean_O, Sigma_OO).
 * Each row solves one SPD system without pivoting, of order |M| (Lambda_MM) or m (E = H + sum_O Delta_i b_i b_i^T, Woodbury),
 * whichever has the smaller flop estimate (|M|^2 m + |M|^3 / 3 against |O| m^2 + m^3 / 3).
 * lcx_lowrank_factor_h: lcx_lowrank_factor (same b, dinv, logdet bit for bit) plus h (m x ldh, device) = H = G^-1 G^-T, under
 *   the same single mailbox read.  ldh even, >= m.  scratch >= lcx_lowrank_h_scratch_doubles(m, n).
 * lcx_condition_rows: raw fp32 / fp64 rows (ld ldx) as in lcx_score_rows, but a missing entry -- NaN, or the marker when
 *   has_marker -- is conditioned on instead of imputed by a column mean; no imputation means are needed.  Optional device
 *   outputs: imputed (n_rows x ldi): observed entries copied as binary64, missing ones mean + sd x^; maha = q_O; logpdf =
 *   log p(x_O).  A complete row gives lcx_score_rows' maha and logpdf bit for bit; a row with nothing observed gives x^ = 0
 *   and q = log p = 0.  Every per-row sum runs in an order fixed by n and the row's own mask, so results do not depend on how
 *   rows are blocked.  class_counts (optional, host, 8 long longs; the call then synchronises the stream): rows with nothing
 *   to solve, rows whose system has order <= 64, <= 160 (both in shared memory), > 160 (per-CTA global slab), rows on the
 *   order-|M| path, on the order-m path.  scratch >= lcx_condition_scratch_doubles(n_rows, n_vars, n_factors). */
long long lcx_lowrank_h_scratch_doubles(int n_factors, int n_vars);
int lcx_lowrank_factor_h(lcx_session* s, const double* rhoinvrho, const double* si, long long ld, int n_factors, int n_vars,
                         double eps, const double* sd, double* b, long long ldb, double* dinv, double* logdet, double* h, long long ldh,
                         double* scratch, long long scratch_doubles);
long long lcx_condition_scratch_doubles(long long n_rows, int n_vars, int n_factors);
int lcx_condition_rows(lcx_session* s, const void* x, int dtype, long long n_rows, int n_vars, long long ldx, int has_marker,
                       double marker, const double* mean, const double* sd, const double* b, long long ldb, int n_factors,
                       const double* h, long long ldh, const double* dinv, const double* logdet, double* imputed, long long ldi,
                       double* maha, double* logpdf, long long* class_counts, double* scratch, long long scratch_doubles);
/* lcx_condition_sample_rows: lcx_condition_rows' standardisation, projection and per-row systems (imputed required and
 *   bit-identical to lcx_condition_rows'; no maha / logpdf), plus, from the same L D L^T factor of each row's system:
 *   std (optional, n_rows x ldo, device): theta1_i sqrt(var(x_i | x_O)) at the missing entries, exactly 0.0 at observed ones;
 *     Path A var = diag(Lambda_MM^-1) by forward sweeps on e_a, Path B var_a = Delta_a + Delta_a^2 b_a^T E^-1 b_a.
 *   draws (optional, device): n_draws completed rows per row, draw d of row r at draws + d draw_stride + r ldo (draw_stride >=
 *     n_rows ldo): the observed entries as imputed holds them, the missing ones theta0 + theta1 (x^ + v) with v ~ N(0, Lambda_MM^-1):
 *     Path A v = L^-T D^-1/2 eps, Path B v = Delta_M^1/2 eps1 + Delta_M B_M^T L^-T D^-1/2 eps2, eps from lcx_normal_fill's stream
 *     (seed, tag 1, row0 + r, d).
 *   A row with nothing observed solves E = H (order m): std theta1, unconditional draws.  A complete row has std 0 and draws
 *   equal to the row.  Every per-row sum runs in a fixed order, so results do not depend on the row blocking; row0 is the global
 *   index of the first row, so a split of the rows between calls or ranks gives the same draws.  class_counts as for
 *   lcx_condition_rows (rows with nothing observed count as order-m, Path B).
 *   scratch >= lcx_condition_sample_scratch_doubles(n_rows, n_vars, n_factors). */
long long lcx_condition_sample_scratch_doubles(long long n_rows, int n_vars, int n_factors);
int lcx_condition_sample_rows(lcx_session* s, const void* x, int dtype, long long n_rows, int n_vars, long long ldx, int has_marker,
                              double marker, const double* mean, const double* sd, const double* b, long long ldb, int n_factors,
                              const double* h, long long ldh, const double* dinv, double* imputed, long long ldi, double* std_out,
                              double* draws, long long ldo, long long draw_stride, unsigned long long seed, long long row0,
                              int n_draws, long long* class_counts, double* scratch, long long scratch_doubles);

/* ---- sampling from the fitted Gaussian (ns variant) ---------------------------------------------------------------------
 * lcx_normal_fill: out[r][j] (n_rows x ldo, device) = standard normal j of the stream (seed, tag, row0 + r, draw), j < n_cols.
 *   Philox4x32-10 with counter (j / 2, draw, row mod 2^32, row / 2^32 + 2^24 tag) and key (seed mod 2^32, seed / 2^32); two
 *   53-bit uniforms in (0, 1], u1 from words 0/1 and u2 from words 2/3, ((w_hi 2^21 + w_lo / 2^11) + 1) 2^-53; Box-Muller
 *   z_2t = sqrt(-2 ln u1) cospi(2 u2), z_2t+1 = sqrt(-2 ln u1) sinpi(2 u2).  A normal depends on nothing else.  words
 *   (optional, n_rows x ldw uint32, ldw >= 4 ceil(n_cols / 2)) receives the Philox words of counter t at [4t, 4t + 4).
 *   Tags: 0 = lcx_sample_rows (columns 0..m-1 are u, m..m+n-1 eps), 1 = lcx_condition_sample_rows.
 * lcx_sample_rows: rows row0 .. row0 + n_rows - 1 of the stream of draws x = mean + sd (Z^T u + Delta^1/2 eps) from
 *   N(mean, Sigma), Sigma = S (Z^T Z + Delta) S as for lcx_lowrank_factor (same inputs, same Delta bit for bit), into out
 *   (n_rows x ldo, device, ldo even).  O(n m) per row: Z and sqrt(Delta) by one column kernel, U (n_rows x m) by
 *   lcx_normal_fill, Y = U Z on the DMMA engine, and a finish pass that generates eps in registers.  Row r depends only on
 *   (seed, row0 + r), not on n_rows.  ONE mailbox read returns LCX_ERR_NOT_PD when some Delta_i <= 0.
 *   scratch >= lcx_sample_scratch_doubles(n_rows, n_vars, n_factors). */
int lcx_normal_fill(lcx_session* s, unsigned long long seed, int tag, long long row0, long long n_rows, long long draw, int n_cols,
                    double* out, long long ldo, unsigned int* words, long long ldw);
long long lcx_sample_scratch_doubles(long long n_rows, int n_vars, int n_factors);
int lcx_sample_rows(lcx_session* s, const double* rhoinvrho, const double* si, long long ld, int n_factors, int n_vars, double eps,
                    const double* mean, const double* sd, unsigned long long seed, long long row0, long long n_rows, double* out,
                    long long ldo, double* scratch, long long scratch_doubles);

/* ---- raw FP64 tensor-core GEMM (unit tests / building block) ----------------------------------- */
/* layout: 0 = A[M][K], B[N][K];  1 = A[K][M], B[K][N];  2 = A[M][K], B[K][N].  C = A*B (+ cadd), optionally
 * stored transposed.  scratch holds split-K partials (may be NULL with max_splits <= 1). */
int lcx_gemm_f64(lcx_session* s, int layout, int M, int N, int K, const double* a, long long lda, const double* b,
                 long long ldb, double* c, long long ldc, int trans_out, const double* cadd, int max_splits,
                 double* scratch, long long scratch_doubles);
/* x (m x ldx, n_rhs columns) = a^-1 b for an m x m device matrix a and m x n_rhs right-hand sides b, by LU with partial
 * pivoting and two triangular sweeps -- what np.linalg.solve does at linearcorex.py:280 and :366 (x may alias b for
 * m <= 832).  Returns LCX_ERR_SINGULAR on an exactly zero pivot.  scratch >= lcx_solve_scratch_doubles(m). */
long long lcx_solve_scratch_doubles(int m);
int lcx_solve(lcx_session* s, const double* a, long long lda, int m, const double* b, long long ldb, double* x,
              long long ldx, int n_rhs, double* scratch, long long scratch_doubles);

#ifdef __cplusplus
}
#endif
#endif /* LCX_B200_H */
