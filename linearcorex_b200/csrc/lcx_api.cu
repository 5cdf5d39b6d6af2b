// C ABI of liblcx_b200.so -- see include/lcx_b200.h for the contract and the reference lines each
// entry point replaces.  Host orchestration only; the arithmetic lives in dgemm_mma.cuh,
// corex_kernels.cuh and preprocess_kernels.cuh.
#include "host_session.cuh"
#include "host_oz.cuh"
#include "host_steps.cuh"

// ---- lifecycle ---------------------------------------------------------------------------------
// Mailboxes (32 pinned doubles per session) come from one process-wide page-locked block: cudaHostAlloc / cudaFreeHost cost
// 10-80 ms each once the process maps 100+ GB of device memory (measured: the Gram route's re-bind spent 0.08-0.17 s in
// them), and both synchronise the device.  64 slots; a 65th concurrent session falls back to its own allocation.
#include <mutex>
namespace {
std::mutex g_mailbox_mutex;
double* g_mailbox_pool = nullptr;
unsigned long long g_mailbox_used = 0;
constexpr int kMailboxSlots = 64, kMailboxDoubles = 32;  // 16 scalars + the sequence number of post_mailbox_kernel (+ padding)

double* mailbox_acquire(bool* pooled) {
    std::lock_guard<std::mutex> lock(g_mailbox_mutex);
    if (g_mailbox_pool == nullptr &&
        cudaHostAlloc((void**)&g_mailbox_pool, kMailboxSlots * kMailboxDoubles * sizeof(double), cudaHostAllocPortable) != cudaSuccess) {
        g_mailbox_pool = nullptr;
        cudaGetLastError();
    }
    if (g_mailbox_pool != nullptr) {
        for (int i = 0; i < kMailboxSlots; ++i) {
            if (!(g_mailbox_used >> i & 1ULL)) {
                g_mailbox_used |= 1ULL << i;
                *pooled = true;
                return g_mailbox_pool + i * kMailboxDoubles;
            }
        }
    }
    double* own = nullptr;
    *pooled = false;
    if (cudaHostAlloc((void**)&own, kMailboxDoubles * sizeof(double), cudaHostAllocPortable) != cudaSuccess) return nullptr;
    return own;
}

void mailbox_release(double* box, bool pooled) {
    if (box == nullptr) return;
    if (!pooled) {
        cudaFreeHost(box);
        return;
    }
    std::lock_guard<std::mutex> lock(g_mailbox_mutex);
    g_mailbox_used &= ~(1ULL << ((box - g_mailbox_pool) / kMailboxDoubles));
}
}  // namespace

extern "C" int lcx_version(void) { return 100; }
extern "C" const char* lcx_last_error(void) { return g_err; }

extern "C" int lcx_session_create(lcx_session** out, int device, int precision) {
    LCX_REQUIRE(out != nullptr, "out is null");
    LCX_REQUIRE(precision >= LCX_PRECISION_FP64 && precision <= LCX_PRECISION_FP64_SPLIT7, "unknown precision mode");
    LCX_CUDA(cudaSetDevice(device));
    int major = 0;  // (cudaGetDeviceProperties takes ~0.1 s once the process holds large page-locked / device mappings)
    LCX_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    if (major != 10) return fail(LCX_ERR_STATE, "lcx_session_create", "this library is built for sm_100a (B200) only");
    lcx_session* s = new lcx_session();
    memset(s, 0, sizeof(*s));
    s->device = device;
    s->precision = precision;
    s->stream = 0;
    s->mailbox = mailbox_acquire(&s->mailbox_pooled);
    if (s->mailbox == nullptr) {
        delete s;
        return fail(LCX_ERR_CUDA, "lcx_session_create", "no page-locked memory for the mailbox");
    }
    for (int i = 0; i < kMailboxDoubles; ++i) s->mailbox[i] = 0.0;  // (a recycled slot still holds its last owner's sequence number)
    *out = s;
    return 0;
}

extern "C" int lcx_profile_enable(lcx_session* s, int on) {
    LCX_REQUIRE(s != nullptr, "null session");
    LCX_CUDA(cudaSetDevice(s->device));
    if (on && s->prof_ev == nullptr) {
        s->prof_cap = 4096;
        s->prof_ev = new cudaEvent_t[kProfEv * s->prof_cap];
        for (int i = 0; i < kProfEv * s->prof_cap; ++i) LCX_CUDA(cudaEventCreate(&s->prof_ev[i]));
    }
    s->prof_on = on != 0;
    return 0;
}

static int profile_resolve(lcx_session* s) {
    LCX_CUDA(cudaSetDevice(s->device));
    LCX_CUDA(cudaStreamSynchronize(s->stream));
    for (int i = 0; i < s->prof_pending; ++i) {
        cudaEvent_t* ev = s->prof_ev + kProfEv * i;
        float a = 0.f, b = 0.f, c = 0.f;
        LCX_CUDA(cudaEventElapsedTime(&a, ev[0], ev[1]));
        LCX_CUDA(cudaEventElapsedTime(&b, ev[3], ev[4]));
        LCX_CUDA(cudaEventElapsedTime(&c, ev[4], ev[2]));
        s->prof_k1_ms += a;
        s->prof_k2_ms += b;
        s->prof_x_ms += c;
        s->prof_pairs++;
    }
    s->prof_pending = 0;
    return 0;
}

extern "C" int lcx_profile_read(lcx_session* s, double* k1_ms, double* k2_ms, long long* pairs, int reset) {
    LCX_REQUIRE(s != nullptr, "null session");
    LCX_TRY(profile_resolve(s));
    if (k1_ms) *k1_ms = s->prof_k1_ms;
    if (k2_ms) *k2_ms = s->prof_k2_ms + s->prof_x_ms;
    if (pairs) *pairs = s->prof_pairs;
    if (reset) {
        s->prof_k1_ms = s->prof_k2_ms = s->prof_x_ms = 0.0;
        s->prof_pairs = 0;
    }
    return 0;
}

extern "C" int lcx_profile_read_phases(lcx_session* s, double* k1_ms, double* k2_ms, double* exchange_ms, long long* pairs,
                                       int reset) {
    LCX_REQUIRE(s != nullptr, "null session");
    LCX_TRY(profile_resolve(s));
    if (k1_ms) *k1_ms = s->prof_k1_ms;
    if (k2_ms) *k2_ms = s->prof_k2_ms;
    if (exchange_ms) *exchange_ms = s->prof_x_ms;
    if (pairs) *pairs = s->prof_pairs;
    if (reset) {
        s->prof_k1_ms = s->prof_k2_ms = s->prof_x_ms = 0.0;
        s->prof_pairs = 0;
    }
    return 0;
}

static void graphs_invalidate(lcx_session* s) {
    for (int i = 0; i < 2; ++i) {
        if (s->graph_exec[i]) cudaGraphExecDestroy(s->graph_exec[i]);
        s->graph_exec[i] = nullptr;
    }
}

extern "C" int lcx_session_destroy(lcx_session* s) {
    if (!s) return 0;
    graphs_invalidate(s);
    if (s->gstream) cudaStreamDestroy(s->gstream);
    if (s->gevent) cudaEventDestroy(s->gevent);
    if (s->prof_ev) {
        for (int i = 0; i < kProfEv * s->prof_cap; ++i) cudaEventDestroy(s->prof_ev[i]);
        delete[] s->prof_ev;
    }
    mailbox_release(s->mailbox, s->mailbox_pooled);
    delete s;
    return 0;
}

extern "C" int lcx_set_stream(lcx_session* s, void* cuda_stream) {
    LCX_REQUIRE(s != nullptr, "null session");
    s->stream = (cudaStream_t)cuda_stream;
    return 0;
}

extern "C" int lcx_set_allreduce(lcx_session* s, lcx_allreduce_fn fn, void* user) {
    LCX_REQUIRE(s != nullptr, "null session");
    s->hook = fn;
    s->hook_user = user;
    return 0;
}

extern "C" long long lcx_peer_buffer_doubles(int n_vars, int n_factors) {
    if (n_vars <= 0 || n_factors <= 0) return -1;
    const long long count = (long long)n_factors * round_up(n_vars, 16) + round_up(n_factors, 16);
    return 3 * count + 4 * far::kMaxRanks;
}

extern "C" int lcx_set_peer_allreduce(lcx_session* s, int world, int rank, void* const* bases, long long buffer_doubles) {
    S_REQUIRE_BOUND(s);
    if (world <= 1 || bases == nullptr) {
        s->peers.world = 0;
        return 0;
    }
    LCX_REQUIRE(world <= far::kMaxRanks && rank >= 0 && rank < world, "bad world / rank (at most 8 ranks)");
    LCX_REQUIRE(buffer_doubles >= lcx_peer_buffer_doubles(s->n, s->m), "peer buffer too small (see lcx_peer_buffer_doubles)");
    for (int r = 0; r < world; ++r) {
        LCX_REQUIRE(bases[r] != nullptr && ((uintptr_t)bases[r] % 16 == 0), "bad peer pointer");
        s->peers.base[r] = (double*)bases[r];
    }
    s->peers.world = world;
    s->peers.rank = rank;
    s->peers.count = (long long)s->m * s->L.ld + s->L.ldm;
    s->ar_calls = 0;
    return 0;
}

extern "C" int lcx_launch_count(lcx_session* s, long long* launches) {
    LCX_REQUIRE(s != nullptr && launches != nullptr, "null argument");
    *launches = s->launches;
    return 0;
}

// ---- layout ------------------------------------------------------------------------------------
extern "C" long long lcx_ld(int n_vars) { return round_up(n_vars, 16); }
extern "C" long long lcx_ldy(int n_factors) { return round_up(n_factors, 8); }

extern "C" long long lcx_workspace_doubles(long long n_rows_local, int n_vars, int n_factors, int precision) {
    if (n_rows_local < 0 || n_vars <= 0 || n_factors <= 0 || precision < 0 || precision > LCX_PRECISION_FP64_SPLIT7) return -1;
    return make_layout(n_rows_local, n_vars, n_factors, precision).total;
}

static int bind_common(lcx_session* s, const double* xt, long long n_rows_local, long long n_rows_total, int n_vars,
                       long long ldx, int n_factors, double* workspace, long long workspace_doubles, bool gram) {
    LCX_REQUIRE(s != nullptr, "null session");
    LCX_REQUIRE(workspace != nullptr, "null device pointer");
    LCX_REQUIRE(xt != nullptr || s->precision != LCX_PRECISION_FP64,
                "xt may be NULL only in the split modes (digit planes are then filled by lcx_slice_block)");
    LCX_REQUIRE(n_rows_local > 0 && n_rows_local < (1LL << 31) && n_rows_total >= (gram ? 1 : n_rows_local), "bad row counts");
    LCX_REQUIRE(n_vars > 0 && n_factors > 0, "bad shape");
    LCX_REQUIRE(ldx >= n_vars && ldx % 2 == 0, "ldx must be even and >= n_vars");
    LCX_REQUIRE(((uintptr_t)xt % 16 == 0) && ((uintptr_t)workspace % 128 == 0), "misaligned device pointer");
    const bool streamed = (xt == nullptr);
    Layout L = make_layout(n_rows_local, n_vars, n_factors, s->precision, gram);
    LCX_REQUIRE(workspace_doubles >= L.total, "workspace too small (see lcx_workspace_doubles)");
    LCX_CUDA(cudaSetDevice(s->device));
    s->xt = xt;
    s->gram = gram;
    s->Nl = n_rows_local;
    s->Nt = n_rows_total;
    s->ldx = ldx;
    s->n = n_vars;
    s->m = n_factors;
    s->ws = workspace;
    s->L = L;
    s->cur = 0;
    graphs_invalidate(s);
    s->graph_warm[0] = s->graph_warm[1] = 0;
    s->d_splits = 1;
    s->bound = true;
    s->peers.world = 0;  // a new problem starts single-rank until lcx_set_peer_allreduce is called for it
    // everything except Y starts at zero so padding never carries NaNs into an all-reduce
    const long long y_off = L.slot[LCX_A_Y][0].off;
    LCX_CUDA(cudaMemsetAsync(workspace, 0, (size_t)y_off * sizeof(double), s->stream));
    const long long y_end = align16(y_off + n_rows_local * L.ldy);
    LCX_CUDA(cudaMemsetAsync(workspace + y_end, 0, (size_t)(L.total - y_end) * sizeof(double), s->stream));
    if (L.S > 0) {
        LCX_TRY(oz_prepare(s, streamed));  // digit slices of X~; after this X~ itself is never read again in the split modes,
        LCX_CUDA(cudaStreamSynchronize(s->stream));  // so the caller may release it as soon as lcx_bind returns
        s->xt = nullptr;
    }
    return 0;
}

extern "C" int lcx_bind(lcx_session* s, const double* xt, long long n_rows_local, long long n_rows_total, int n_vars,
                        long long ldx, int n_factors, double* workspace, long long workspace_doubles) {
    return bind_common(s, xt, n_rows_local, n_rows_total, n_vars, ldx, n_factors, workspace, workspace_doubles, false);
}

// ---- Gram route (host_gram.cuh) -----------------------------------------------------------------------------------
extern "C" long long lcx_gram_scratch_doubles(lcx_session* s, int block_cols) {
    if (!s || !s->bound || s->L.S <= 0 || s->gram || block_cols < 128 || block_cols % 128 != 0) return -1;
    return gram_scratch_doubles(s, block_cols, round_up(s->n, 16));
}

extern "C" int lcx_gram_build(lcx_session* s, double* g, long long ldg, int block_cols, double* scratch, long long scratch_doubles) {
    S_REQUIRE_BOUND(s);
    LCX_REQUIRE(s->L.S > 0 && !s->gram, "lcx_gram_build needs a split-mode session bound to X~");
    LCX_REQUIRE(g != nullptr && scratch != nullptr, "null device pointer");
    LCX_REQUIRE(block_cols >= 128 && block_cols % 128 == 0, "block_cols must be a positive multiple of 128");
    LCX_REQUIRE(ldg == round_up(s->n, 16), "ldg must be lcx_ld(n_vars)");
    LCX_REQUIRE(((uintptr_t)g % 128 == 0) && ((uintptr_t)scratch % 128 == 0), "misaligned device pointer");
    LCX_REQUIRE(scratch_doubles >= gram_scratch_doubles(s, block_cols, ldg), "scratch too small (see lcx_gram_scratch_doubles)");
    return gram_build(s, g, ldg, block_cols, scratch);
}

extern "C" long long lcx_gram_workspace_doubles(int n_vars, int n_factors, int precision) {
    if (n_vars <= 0 || n_factors <= 0 || precision <= LCX_PRECISION_FP64 || precision > LCX_PRECISION_FP64_SPLIT7) return -1;
    return make_layout(n_vars, n_vars, n_factors, precision, true).total;
}

extern "C" int lcx_bind_gram(lcx_session* s, const double* g, long long ldg, int n_vars, int n_factors, double* workspace,
                             long long workspace_doubles) {
    LCX_REQUIRE(s != nullptr && g != nullptr, "null argument");
    LCX_REQUIRE(s->precision != LCX_PRECISION_FP64, "the Gram route runs on the split-integer engine (choose a split precision)");
    return bind_common(s, g, n_vars, 1, n_vars, ldg, n_factors, workspace, workspace_doubles, true);
}

// ---- streamed digit slicing (X~ never materialised as a whole: the 1M x 20k target on one GPU) -------------------
extern "C" int lcx_set_x_scale(lcx_session* s, double max_abs) {
    S_REQUIRE_BOUND(s);
    LCX_REQUIRE(s->L.S > 0, "only meaningful in the split modes");
    LCX_REQUIRE(!(max_abs < 0.0), "max_abs must be a non-negative bound on |X~|");
    int e = 0;
    double scale = 1.0;
    if (!(max_abs <= DBL_MAX)) {
        scale = NAN;  // non-finite data: every product comes out NaN, as in the reference's float64 path
    } else if (max_abs > 0.0) {
        frexp(max_abs, &e);
        scale = ldexp(1.0, e + 1);
    }
    LCX_CUDA(cudaMemcpyAsync(s->oz_xscale(), &scale, sizeof(double), cudaMemcpyHostToDevice, s->stream));
    LCX_CUDA(cudaStreamSynchronize(s->stream));
    return 0;
}

extern "C" int lcx_slice_block(lcx_session* s, const double* xt, long long row0, long long rows, long long ldx) {
    S_REQUIRE_BOUND(s);
    LCX_REQUIRE(s->L.S > 0, "only meaningful in the split modes");
    LCX_REQUIRE(xt != nullptr && row0 >= 0 && rows > 0 && row0 + rows <= s->Nl && ldx >= s->n, "bad row block");
    switch (s->L.S) {
        case 3: return oz_slice_block_t<3>(s, xt, row0, rows, ldx);
        case 4: return oz_slice_block_t<4>(s, xt, row0, rows, ldx);
        case 5: return oz_slice_block_t<5>(s, xt, row0, rows, ldx);
        case 6: return oz_slice_block_t<6>(s, xt, row0, rows, ldx);
        case 7: return oz_slice_block_t<7>(s, xt, row0, rows, ldx);
    }
    return fail(LCX_ERR_STATE, "lcx_slice_block", "bad digit count");
}

extern "C" int lcx_array_info(lcx_session* s, int array_id, int set, long long* offset, long long* rows, long long* cols,
                              long long* ld) {
    S_REQUIRE_BOUND(s);
    LCX_REQUIRE(array_id >= 0 && array_id < LCX_A_COUNT && (set == 0 || set == 1), "bad array id / set");
    const int phys = (array_id <= LCX_A_UJ) ? (set ^ s->cur) : 0;
    const Slot& sl = s->L.slot[array_id][phys];
    if (offset) *offset = (array_id == LCX_A_D) ? (long long)(s->ptr(LCX_A_D) - s->ws) : sl.off;  // (peer buffer when sharded)
    if (rows) *rows = (array_id == LCX_A_D) ? s->m : sl.rows;
    if (cols) *cols = sl.cols;
    if (ld) *ld = sl.ld;
    return 0;
}

// Where the int8 digit planes and their power-of-two scales live (split modes; for inspection and bit-exact tests).
extern "C" int lcx_digit_planes_info(lcx_session* s, int which, long long* offset, int* digits, long long* rows,
                                     long long* cols, long long* ld_bytes, long long* scale_offset, int* radix) {
    S_REQUIRE_BOUND(s);
    const Layout& L = s->L;
    LCX_REQUIRE(L.S > 0, "no digit planes in the DMMA mode");
    LCX_REQUIRE(which >= 0 && which <= 2, "which: 0 = X~, 1 = A (last small operand), 2 = Y");
    const int slot = which == 0 ? I_XS : (which == 1 ? I_AS : I_YS);
    if (offset) *offset = L.slot[slot][0].off;
    if (digits) *digits = L.S;
    if (rows) *rows = which == 0 ? s->Nl : s->m;          // the Y planes are stored transposed: [factor][sample]
    if (cols) *cols = which == 2 ? s->Nl : s->n;
    if (ld_bytes) *ld_bytes = which == 2 ? L.ldk8 : L.ld8;
    if (scale_offset) *scale_offset = L.slot[I_OZV][0].off + (which == 0 ? 0 : (which == 1 ? 16 : 16 + 2 * L.ldm));
    if (radix) *radix = oz::kRadix;
    return 0;
}

// ---- preprocessing -----------------------------------------------------------------------------
static const int kSlabRows = 4096;

extern "C" long long lcx_colstats_scratch_doubles(long long n_rows, int n_vars) {
    return 2LL * cdiv(n_rows, kSlabRows) * round_up(n_vars, 16) + 32;
}

// 16-byte row loads are possible when the base pointer and the leading dimension are multiples of 4 elements
template <typename T>
static bool vec4_ok(const T* x, long long ldx) { return ((uintptr_t)x % 16 == 0) && (ldx % 4 == 0); }

template <typename T, bool W>
static int colstats_sum_t(lcx_session* s, const T* x, long long N, int n, long long ldx, int has_marker, double marker,
                          double* sum, double* cnt, double* scratch, const double* w) {
    const int slabs = cdiv(N, kSlabRows);
    const long long ldp = round_up(n, 16);
    double* ps = scratch;
    double* pc = scratch + (long long)slabs * ldp;
    const dim3 block(32, 8);
    if (vec4_ok(x, ldx))
        colstats_sum_kernel<T, 4, W><<<dim3(cdiv(n, 128), slabs), block, 0, s->stream>>>(x, N, n, ldx, kSlabRows, has_marker,
                                                                                       marker, marker != marker, ps, pc, ldp, w);
    else
        colstats_sum_kernel<T, 1, W><<<dim3(cdiv(n, 32), slabs), block, 0, s->stream>>>(x, N, n, ldx, kSlabRows, has_marker,
                                                                                      marker, marker != marker, ps, pc, ldp, w);
    LAUNCHED(s);
    combine_slabs_kernel<<<cdiv(n, 256), 256, 0, s->stream>>>(ps, slabs, ldp, sum, n);
    LAUNCHED(s);
    combine_slabs_kernel<<<cdiv(n, 256), 256, 0, s->stream>>>(pc, slabs, ldp, cnt, n);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int lcx_colstats_sum(lcx_session* s, const void* x, int dtype, long long n_rows, int n_vars, long long ldx,
                                int has_marker, double marker, double* sum, double* cnt, double* scratch,
                                long long scratch_doubles) {
    LCX_REQUIRE(s && x && sum && cnt && scratch, "null argument");
    LCX_REQUIRE(n_rows > 0 && n_vars > 0 && ldx >= n_vars, "bad shape");
    LCX_REQUIRE(scratch_doubles >= lcx_colstats_scratch_doubles(n_rows, n_vars), "scratch too small");
    LCX_CUDA(cudaSetDevice(s->device));
    if (dtype == LCX_F32)
        return colstats_sum_t<float, false>(s, (const float*)x, n_rows, n_vars, ldx, has_marker, marker, sum, cnt, scratch, nullptr);
    if (dtype == LCX_F64)
        return colstats_sum_t<double, false>(s, (const double*)x, n_rows, n_vars, ldx, has_marker, marker, sum, cnt, scratch, nullptr);
    return fail(LCX_ERR_ARG, "lcx_colstats_sum", "unknown dtype");
}

extern "C" int lcx_row_scale(lcx_session* s, const double* w, long long n_rows, double n_rows_total, double w_total,
                             double* r) {
    LCX_REQUIRE(s && w && r, "null argument");
    LCX_REQUIRE(n_rows > 0 && n_rows_total > 0.0 && w_total > 0.0 && w_total <= DBL_MAX, "bad row count or weight total");
    LCX_CUDA(cudaSetDevice(s->device));
    row_scale_kernel<<<(unsigned)cdiv(n_rows, 256), 256, 0, s->stream>>>(w, n_rows, n_rows_total, w_total, r);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int lcx_colstats_sum_w(lcx_session* s, const void* x, int dtype, long long n_rows, int n_vars, long long ldx,
                                  int has_marker, double marker, double* sum, double* cnt, double* scratch,
                                  long long scratch_doubles, const double* w) {
    LCX_REQUIRE(s && x && sum && cnt && scratch && w, "null argument");
    LCX_REQUIRE(n_rows > 0 && n_vars > 0 && ldx >= n_vars, "bad shape");
    LCX_REQUIRE(scratch_doubles >= lcx_colstats_scratch_doubles(n_rows, n_vars), "scratch too small");
    LCX_CUDA(cudaSetDevice(s->device));
    if (dtype == LCX_F32)
        return colstats_sum_t<float, true>(s, (const float*)x, n_rows, n_vars, ldx, has_marker, marker, sum, cnt, scratch, w);
    if (dtype == LCX_F64)
        return colstats_sum_t<double, true>(s, (const double*)x, n_rows, n_vars, ldx, has_marker, marker, sum, cnt, scratch, w);
    return fail(LCX_ERR_ARG, "lcx_colstats_sum_w", "unknown dtype");
}

extern "C" int lcx_colstats_mean(lcx_session* s, const double* sum, const double* cnt, double* mean, int n_vars) {
    LCX_REQUIRE(s && sum && cnt && mean && n_vars > 0, "bad argument");
    LCX_CUDA(cudaSetDevice(s->device));
    finish_mean_kernel<<<cdiv(n_vars, 256), 256, 0, s->stream>>>(sum, cnt, mean, n_vars);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}

template <typename T, bool W>
static int colstats_sqdev_t(lcx_session* s, const T* x, long long N, int n, long long ldx, int has_marker, double marker,
                            const double* mean, double* sq, double* maxdev, double* scratch, const double* w, const double* r) {
    const int slabs = cdiv(N, kSlabRows);
    const long long ldp = round_up(n, 16);
    double* pmax = maxdev ? scratch + (long long)slabs * ldp : nullptr;
    const dim3 block(32, 8);
    if (vec4_ok(x, ldx))
        colstats_sqdev_kernel<T, 4, W><<<dim3(cdiv(n, 128), slabs), block, 0, s->stream>>>(
            x, N, n, ldx, kSlabRows, has_marker, marker, marker != marker, mean, scratch, pmax, ldp, w, r);
    else
        colstats_sqdev_kernel<T, 1, W><<<dim3(cdiv(n, 32), slabs), block, 0, s->stream>>>(
            x, N, n, ldx, kSlabRows, has_marker, marker, marker != marker, mean, scratch, pmax, ldp, w, r);
    LAUNCHED(s);
    combine_slabs_kernel<<<cdiv(n, 256), 256, 0, s->stream>>>(scratch, slabs, ldp, sq, n);
    LAUNCHED(s);
    if (maxdev) {
        combine_slabs_max_kernel<<<cdiv(n, 256), 256, 0, s->stream>>>(pmax, slabs, ldp, maxdev, n);
        LAUNCHED(s);
    }
    LCX_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int lcx_colstats_sqdev(lcx_session* s, const void* x, int dtype, long long n_rows, int n_vars, long long ldx,
                                  int has_marker, double marker, const double* mean, double* sq, double* maxdev,
                                  double* scratch, long long scratch_doubles) {
    LCX_REQUIRE(s && x && mean && sq && scratch, "null argument");
    LCX_REQUIRE(n_rows > 0 && n_vars > 0 && ldx >= n_vars, "bad shape");
    LCX_REQUIRE(scratch_doubles >= lcx_colstats_scratch_doubles(n_rows, n_vars), "scratch too small");
    LCX_CUDA(cudaSetDevice(s->device));
    if (dtype == LCX_F32)
        return colstats_sqdev_t<float, false>(s, (const float*)x, n_rows, n_vars, ldx, has_marker, marker, mean, sq, maxdev, scratch,
                                              nullptr, nullptr);
    if (dtype == LCX_F64)
        return colstats_sqdev_t<double, false>(s, (const double*)x, n_rows, n_vars, ldx, has_marker, marker, mean, sq, maxdev,
                                               scratch, nullptr, nullptr);
    return fail(LCX_ERR_ARG, "lcx_colstats_sqdev", "unknown dtype");
}

extern "C" int lcx_colstats_sqdev_w(lcx_session* s, const void* x, int dtype, long long n_rows, int n_vars, long long ldx,
                                    int has_marker, double marker, const double* mean, double* sq, double* maxdev,
                                    double* scratch, long long scratch_doubles, const double* w, const double* r) {
    LCX_REQUIRE(s && x && mean && sq && scratch && w && r, "null argument");
    LCX_REQUIRE(n_rows > 0 && n_vars > 0 && ldx >= n_vars, "bad shape");
    LCX_REQUIRE(scratch_doubles >= lcx_colstats_scratch_doubles(n_rows, n_vars), "scratch too small");
    LCX_CUDA(cudaSetDevice(s->device));
    if (dtype == LCX_F32)
        return colstats_sqdev_t<float, true>(s, (const float*)x, n_rows, n_vars, ldx, has_marker, marker, mean, sq, maxdev, scratch,
                                             w, r);
    if (dtype == LCX_F64)
        return colstats_sqdev_t<double, true>(s, (const double*)x, n_rows, n_vars, ldx, has_marker, marker, mean, sq, maxdev,
                                              scratch, w, r);
    return fail(LCX_ERR_ARG, "lcx_colstats_sqdev_w", "unknown dtype");
}

extern "C" int lcx_colstats_std(lcx_session* s, const double* sq, const double* cnt, double n_rows_total, int use_nobs,
                                double* sd, int n_vars) {
    LCX_REQUIRE(s && sq && cnt && sd && n_vars > 0, "bad argument");
    LCX_CUDA(cudaSetDevice(s->device));
    finish_std_kernel<<<cdiv(n_vars, 256), 256, 0, s->stream>>>(sq, cnt, n_rows_total, use_nobs, sd, n_vars);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}

template <bool W>
static int standardize_d(lcx_session* s, const void* x, int dtype, long long n_rows, int n_vars, long long ldx, int has_marker,
                         double marker, int gauss_mode, const double* impute, const double* mean, const double* sd, double* out,
                         long long ldo, const double* r) {
    LCX_REQUIRE(s && x && out, "null argument");
    LCX_REQUIRE(gauss_mode == LCX_GAUSS_NONE || (mean && sd), "mean/std required");
    LCX_REQUIRE(has_marker == 0 || impute != nullptr, "imputation means required when a missing marker is set");
    LCX_REQUIRE(n_rows > 0 && n_vars > 0 && ldx >= n_vars && ldo >= n_vars, "bad shape");
    LCX_CUDA(cudaSetDevice(s->device));
    const int nan_marker = marker != marker;
    const bool v4 = (ldo % 4 == 0) && ((uintptr_t)out % 16 == 0) &&
                    (dtype == LCX_F32 ? vec4_ok((const float*)x, ldx) : vec4_ok((const double*)x, ldx));
    const dim3 grid((unsigned)n_rows, cdiv(ldo, v4 ? 1024 : 256));
    if (dtype == LCX_F32 && v4)
        standardize_kernel<float, 4, W><<<grid, 256, 0, s->stream>>>((const float*)x, n_rows, n_vars, ldx, has_marker, marker,
                                                                nan_marker, gauss_mode, impute, mean, sd, out, ldo, r);
    else if (dtype == LCX_F32)
        standardize_kernel<float, 1, W><<<grid, 256, 0, s->stream>>>((const float*)x, n_rows, n_vars, ldx, has_marker, marker,
                                                                nan_marker, gauss_mode, impute, mean, sd, out, ldo, r);
    else if (dtype == LCX_F64 && v4)
        standardize_kernel<double, 4, W><<<grid, 256, 0, s->stream>>>((const double*)x, n_rows, n_vars, ldx, has_marker, marker,
                                                                 nan_marker, gauss_mode, impute, mean, sd, out, ldo, r);
    else if (dtype == LCX_F64)
        standardize_kernel<double, 1, W><<<grid, 256, 0, s->stream>>>((const double*)x, n_rows, n_vars, ldx, has_marker, marker,
                                                                 nan_marker, gauss_mode, impute, mean, sd, out, ldo, r);
    else
        return fail(LCX_ERR_ARG, "lcx_standardize", "unknown dtype");
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int lcx_standardize(lcx_session* s, const void* x, int dtype, long long n_rows, int n_vars, long long ldx,
                               int has_marker, double marker, int gauss_mode, const double* impute, const double* mean,
                               const double* sd, double* out, long long ldo) {
    return standardize_d<false>(s, x, dtype, n_rows, n_vars, ldx, has_marker, marker, gauss_mode, impute, mean, sd, out, ldo,
                                nullptr);
}

extern "C" int lcx_standardize_w(lcx_session* s, const void* x, int dtype, long long n_rows, int n_vars, long long ldx,
                                 int has_marker, double marker, int gauss_mode, const double* impute, const double* mean,
                                 const double* sd, double* out, long long ldo, const double* r) {
    LCX_REQUIRE(r != nullptr, "null argument");
    return standardize_d<true>(s, x, dtype, n_rows, n_vars, ldx, has_marker, marker, gauss_mode, impute, mean, sd, out, ldo, r);
}

template <typename T, int S, bool W>
static int standardize_slice_t(lcx_session* s, const T* x, long long row0, long long rows, long long ldx, int has_marker,
                               double marker, int mode, const double* impute, const double* mean, const double* sd,
                               const double* r) {
    const Layout& L = s->L;
    const dim3 grid((unsigned)rows, cdiv(L.ld8, 4 * 128));
    int8_t* out = s->xs() + row0 * L.ld8;
    const int nan_marker = marker != marker;
    if (vec4_ok(x, ldx))
        standardize_slice_kernel<T, S, 4, W><<<grid, 128, 0, s->stream>>>(x, rows, s->n, ldx, has_marker, marker, nan_marker, mode,
                                                                     impute, mean, sd, s->oz_xscale(), out, L.ld8,
                                                                     s->Nl * L.ld8, (double)oz::kRadix, r);
    else
        standardize_slice_kernel<T, S, 1, W><<<grid, 128, 0, s->stream>>>(x, rows, s->n, ldx, has_marker, marker, nan_marker, mode,
                                                                     impute, mean, sd, s->oz_xscale(), out, L.ld8,
                                                                     s->Nl * L.ld8, (double)oz::kRadix, r);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}

template <typename T, bool W>
static int standardize_slice_d(lcx_session* s, const T* x, long long row0, long long rows, long long ldx, int has_marker,
                               double marker, int mode, const double* impute, const double* mean, const double* sd,
                               const double* r) {
    switch (s->L.S) {
        case 3: return standardize_slice_t<T, 3, W>(s, x, row0, rows, ldx, has_marker, marker, mode, impute, mean, sd, r);
        case 4: return standardize_slice_t<T, 4, W>(s, x, row0, rows, ldx, has_marker, marker, mode, impute, mean, sd, r);
        case 5: return standardize_slice_t<T, 5, W>(s, x, row0, rows, ldx, has_marker, marker, mode, impute, mean, sd, r);
        case 6: return standardize_slice_t<T, 6, W>(s, x, row0, rows, ldx, has_marker, marker, mode, impute, mean, sd, r);
        case 7: return standardize_slice_t<T, 7, W>(s, x, row0, rows, ldx, has_marker, marker, mode, impute, mean, sd, r);
    }
    return fail(LCX_ERR_STATE, "lcx_standardize_slice", "bad digit count");
}

// lcx_standardize + lcx_slice_block in one pass over the raw rows (split modes, after lcx_bind(xt = NULL) + lcx_set_x_scale)
template <bool W>
static int standardize_slice_any(lcx_session* s, const void* x, int dtype, long long row0, long long n_rows, long long ldx,
                                 int has_marker, double marker, int gauss_mode, const double* impute, const double* mean,
                                 const double* sd, const double* r) {
    S_REQUIRE_BOUND(s);
    LCX_REQUIRE(s->L.S > 0 && !s->gram, "only meaningful in the split modes, on a session bound to X~");
    LCX_REQUIRE(x != nullptr && row0 >= 0 && n_rows > 0 && row0 + n_rows <= s->Nl && ldx >= s->n, "bad row block");
    LCX_REQUIRE(gauss_mode == LCX_GAUSS_NONE || (mean && sd), "mean/std required");
    LCX_REQUIRE(has_marker == 0 || impute != nullptr, "imputation means required when a missing marker is set");
    if (dtype == LCX_F32)
        return standardize_slice_d<float, W>(s, (const float*)x, row0, n_rows, ldx, has_marker, marker, gauss_mode, impute, mean,
                                             sd, r);
    if (dtype == LCX_F64)
        return standardize_slice_d<double, W>(s, (const double*)x, row0, n_rows, ldx, has_marker, marker, gauss_mode, impute, mean,
                                              sd, r);
    return fail(LCX_ERR_ARG, "lcx_standardize_slice", "unknown dtype");
}

extern "C" int lcx_standardize_slice(lcx_session* s, const void* x, int dtype, long long row0, long long n_rows, long long ldx,
                                     int has_marker, double marker, int gauss_mode, const double* impute, const double* mean,
                                     const double* sd) {
    return standardize_slice_any<false>(s, x, dtype, row0, n_rows, ldx, has_marker, marker, gauss_mode, impute, mean, sd, nullptr);
}

// r: the row scales of rows [row0, row0 + n_rows) (r[0] belongs to row row0)
extern "C" int lcx_standardize_slice_w(lcx_session* s, const void* x, int dtype, long long row0, long long n_rows, long long ldx,
                                       int has_marker, double marker, int gauss_mode, const double* impute, const double* mean,
                                       const double* sd, const double* r) {
    LCX_REQUIRE(r != nullptr, "null argument");
    return standardize_slice_any<true>(s, x, dtype, row0, n_rows, ldx, has_marker, marker, gauss_mode, impute, mean, sd, r);
}

// ---- exported steps ----------------------------------------------------------------------------
extern "C" long long lcx_project_scratch_doubles(long long n_rows, int n_factors) {
    return (long long)cdiv(n_rows, 128) * round_up(n_factors, 8) + 16;
}

extern "C" int lcx_project(lcx_session* s, const double* xt, long long n_rows, int n_vars, long long ldx, const double* a,
                           long long lda, int n_factors, double* y, long long ldy, double* colsq, double* scratch,
                           long long scratch_doubles) {
    LCX_REQUIRE(s && xt && a && y, "null argument");
    LCX_REQUIRE(n_rows > 0 && n_rows < (1LL << 31) && n_vars > 0 && n_factors > 0, "bad shape");
    LCX_REQUIRE(colsq == nullptr || (scratch != nullptr && scratch_doubles >= lcx_project_scratch_doubles(n_rows, n_factors)),
                "scratch too small for the column sums");
    LCX_CUDA(cudaSetDevice(s->device));
    GemmPlan pl = plan_gemm((int)n_rows, n_factors, n_vars, kSMs, 1, false);
    GemmArgs g;
    memset(&g, 0, sizeof(g));
    g.A = xt; g.B = a; g.C = y;
    g.M = (int)n_rows; g.N = n_factors; g.K = n_vars;
    g.lda = ldx; g.ldb = lda; g.ldc = ldy;
    const int ldp = (int)round_up(n_factors, 8);
    g.colsq_part = colsq ? scratch : nullptr;
    g.ld_colsq = ldp;
    LCX_TRY(launch_gemm(kLayoutKK, pl, g, s->stream));
    LAUNCHED(s);
    if (colsq) {
        reduce_colsq_kernel<<<cdiv(n_factors, 128), 128, 0, s->stream>>>(scratch, pl.grid.x, ldp, colsq, n_factors);
        LAUNCHED(s);
    }
    LCX_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int lcx_sig(lcx_session* s, const double* u, double eps, double* out) {
    S_REQUIRE_BOUND(s);
    LCX_REQUIRE(u && out, "null argument");
    LCX_TRY(xpair(s, u, false));
    const double c1 = (1.0 - eps * eps) / (double)s->Nt, e2 = eps * eps;
    sig_finish_kernel<<<grid_mn(s->m, s->n), 256, 0, s->stream>>>(s->ptr(LCX_A_D), u, c1, e2, out, s->m, s->n, s->L.ld);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int lcx_set_w(lcx_session* s, const double* host_w, long long host_ld) {
    S_REQUIRE_BOUND(s);
    LCX_REQUIRE(host_w && host_ld >= s->n, "bad host array");
    LCX_CUDA(cudaMemcpy2DAsync(s->ptr(LCX_A_W), s->L.ld * sizeof(double), host_w, host_ld * sizeof(double),
                               (size_t)s->n * sizeof(double), s->m, cudaMemcpyHostToDevice, s->stream));
    LCX_CUDA(cudaStreamSynchronize(s->stream));
    return 0;
}

extern "C" int lcx_get_w(lcx_session* s, double* host_w, long long host_ld) {
    S_REQUIRE_BOUND(s);
    LCX_REQUIRE(host_w && host_ld >= s->n, "bad host array");
    LCX_CUDA(cudaMemcpy2DAsync(host_w, host_ld * sizeof(double), s->ptr(LCX_A_W), s->L.ld * sizeof(double),
                               (size_t)s->n * sizeof(double), s->m, cudaMemcpyDeviceToHost, s->stream));
    LCX_CUDA(cudaStreamSynchronize(s->stream));
    return 0;
}

extern "C" int lcx_init_scale(lcx_session* s, double eps) {
    S_REQUIRE_BOUND(s);
    const Layout& L = s->L;
    const int m = s->m, n = s->n;
    double* W = s->ptr(LCX_A_W);
    double* svec = s->ptr(LCX_A_D) + (long long)m * L.ld;
    if (s->gram) {
        LCX_TRY(gram_pair(s, W, svec, nullptr));
    } else if (L.S > 0) {
        LCX_TRY(oz_pair(s, W, svec, nullptr, true, true));
    } else {
        LCX_TRY(lcx_project(s, s->xt, s->Nl, n, s->ldx, W, L.ld, m, s->ptr(LCX_A_Y), L.ldy, svec, s->ptr(I_COLSQ),
                            lcx_project_scratch_doubles(s->Nl, m)));
    }
    if (!s->gram)  // (on the Gram route a_j^T G a_j is already the sum over all samples, identical on every rank)
        LCX_TRY(combine_and_allreduce(s, nullptr, 1, 0, 0, 0, L.ld, nullptr, svec, m));  // sum of Y^2 over ranks
    row_dot_kernel<<<m, 256, 0, s->stream>>>(W, W, s->ptr(I_W2), n, L.ld);
    LAUNCHED(s);
    const double c1 = (1.0 - eps * eps) / (double)s->Nt, e2 = eps * eps;
    init_scale_kernel<<<cdiv(m, 128), 128, 0, s->stream>>>(svec, s->ptr(I_W2), c1, e2, s->ptr(I_F), m);
    LAUNCHED(s);
    scale_rows_kernel<<<grid_mn(m, n), 256, 0, s->stream>>>(W, s->ptr(I_F), m, n, L.ld);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int lcx_stage_rescale(lcx_session* s, double eps, double eps_prev) {
    S_REQUIRE_BOUND(s);
    const Layout& L = s->L;
    const int m = s->m, n = s->n;
    double* W = s->ptr(LCX_A_W);
    row_dot_kernel<<<m, 256, 0, s->stream>>>(W, W, s->ptr(I_W2), n, L.ld);
    LAUNCHED(s);
    stage_scale_kernel<<<cdiv(m, 128), 128, 0, s->stream>>>(s->ptr(I_W2), s->ptr(LCX_A_UJ), eps, eps_prev, s->ptr(I_F), m);
    LAUNCHED(s);
    scale_rows_kernel<<<grid_mn(m, n), 256, 0, s->stream>>>(W, s->ptr(I_F), m, n, L.ld);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int lcx_permute_rows(lcx_session* s, const int* host_order) {
    S_REQUIRE_BOUND(s);
    LCX_REQUIRE(host_order != nullptr, "null order");
    const Layout& L = s->L;
    double* W = s->ptr(LCX_A_W);
    double* tmp = s->ptr(LCX_A_GRAD);
    for (int j = 0; j < s->m; ++j) {
        LCX_REQUIRE(host_order[j] >= 0 && host_order[j] < s->m, "order out of range");
        LCX_CUDA(cudaMemcpyAsync(tmp + (long long)j * L.ld, W + (long long)host_order[j] * L.ld, L.ld * sizeof(double),
                                 cudaMemcpyDeviceToDevice, s->stream));
    }
    LCX_CUDA(cudaMemcpyAsync(W, tmp, (size_t)s->m * L.ld * sizeof(double), cudaMemcpyDeviceToDevice, s->stream));
    return 0;
}

extern "C" int lcx_moments_ns(lcx_session* s, double eps, int check_uj, double* tc, double* max_uj) {
    S_REQUIRE_BOUND(s);
    LCX_TRY(moments_from_x(s, 0, eps));
    LCX_TRY(read_mailbox(s));
    if (tc) *tc = s->mailbox[0];
    if (max_uj) *max_uj = s->mailbox[1];
    return (check_uj && s->mailbox[1] >= 1.0) ? LCX_QUICK_FAIL : LCX_OK;
}

extern "C" int lcx_direction_ns(lcx_session* s, double eps, double* tangent) {
    S_REQUIRE_BOUND(s);
    LCX_TRY(enqueue_direction(s, eps));
    LCX_TRY(read_mailbox(s));
    if (tangent) *tangent = s->mailbox[2];
    return 0;
}

extern "C" int lcx_trial_ns(lcx_session* s, double eps, double eta, int exact, double* tc, double* max_uj) {
    S_REQUIRE_BOUND(s);
    LCX_TRY(enqueue_trial(s, eps, eta, exact));
    LCX_TRY(read_mailbox(s));
    if (tc) *tc = s->mailbox[0];
    if (max_uj) *max_uj = s->mailbox[1];
    return (s->mailbox[1] >= 1.0) ? LCX_QUICK_FAIL : LCX_OK;
}

// Direction (:292-305) and the first backtracking trial at `eta` (:320-321) enqueued back to back, ONE host
// synchronisation for update_tangent, TC and max uj.  The trial is speculative: if update_tangent >= 0 the caller
// discards it (the reference returns before trying, :306-311).  Linear trials only (an exact trial costs a pass pair).
extern "C" int lcx_direction_trial_ns(lcx_session* s, double eps, double eta, double* tangent, double* tc, double* max_uj) {
    S_REQUIRE_BOUND(s);
    LCX_TRY(enqueue_direction(s, eps));
    LCX_TRY(enqueue_trial(s, eps, eta, 0));
    LCX_TRY(read_mailbox(s));
    if (tangent) *tangent = s->mailbox[2];
    if (tc) *tc = s->mailbox[0];
    if (max_uj) *max_uj = s->mailbox[1];
    return (s->mailbox[1] >= 1.0) ? LCX_QUICK_FAIL : LCX_OK;
}

// Iteration graphs pay only where an iteration is bound by the host's launch rate: arrays of at most kGraphMaxElems elements
// (README demo, big5: kernels of 2-3 us).  Measured on a B200 (tools/small_configs.py, profiles/r02_cuda_graph_ab.txt): README
// demo 0.124 -> 0.075 ms per iteration; at config 3 a replay is 50 us SLOWER per iteration than stream launches (the host
// waits for every iteration, so a graph's launch latency is exposed while stream launches run ahead of 5-30 us kernels), and a
// capture costs ~1 ms, so a stage must run kGraphAfter iterations on a parity before it is captured.  Single-rank sessions
// only (the rank exchange is a cooperative kernel / a host hook).
constexpr long long kGraphMaxElems = 1 << 17;
constexpr int kGraphAfter = 8;
static bool graphs_enabled(const lcx_session* s) {
    if (s->peers.world > 1 || s->hook != nullptr || s->prof_on) return false;
    return (long long)s->m * s->n <= kGraphMaxElems;
}

// Direction (:292-305) + the eta = 1 trial (:320-321) + the mailbox copy of ONE iteration, replayed from a CUDA graph: ~17
// launches become one cudaGraphLaunch.  Returns 1 when the iteration must be enqueued plainly instead (the first kGraphAfter
// iterations of a stage on this parity: kernel attributes are configured outside a capture, and short stages never pay one).
static int iteration_graph(lcx_session* s, double eps) {
    const int par = s->cur;
    if (s->graph_eps != eps) {
        graphs_invalidate(s);
        s->graph_eps = eps;
        for (int i = 0; i < 2; ++i)
            if (s->graph_warm[i] > 0) s->graph_warm[i] = 0;  // (a negative count = capture failed once: stay on plain launches)
    }
    if (s->graph_exec[par] == nullptr) {
        if (s->graph_warm[par] < kGraphAfter) {
            s->graph_warm[par]++;
            return 1;
        }
        if (s->gstream == nullptr) {
            LCX_CUDA(cudaStreamCreate(&s->gstream));
            LCX_CUDA(cudaEventCreateWithFlags(&s->gevent, cudaEventDisableTiming));
        }
        cudaStream_t user = s->stream;
        const long long l0 = s->launches;
        LCX_CUDA(cudaStreamBeginCapture(s->gstream, cudaStreamCaptureModeRelaxed));
        s->stream = s->gstream;
        int rc = enqueue_direction(s, eps);
        if (rc >= 0) rc = enqueue_trial(s, eps, 1.0, 0);
        cudaError_t ce = cudaSuccess;
        if (rc >= 0)
            ce = cudaMemcpyAsync(s->mailbox, s->ptr(LCX_A_SCALARS), 16 * sizeof(double), cudaMemcpyDeviceToHost, s->gstream);
        s->stream = user;
        cudaGraph_t g = nullptr;
        const cudaError_t ee = cudaStreamEndCapture(s->gstream, &g);
        s->graph_launches[par] = s->launches - l0;
        s->launches = l0;
        if (rc < 0 || ce != cudaSuccess || ee != cudaSuccess || g == nullptr) {
            if (g) cudaGraphDestroy(g);
            cudaGetLastError();
            s->graph_warm[par] = -1000000;  // capture is not possible here: stay on plain launches
            return rc < 0 ? rc : 1;
        }
        const cudaError_t ie = cudaGraphInstantiate(&s->graph_exec[par], g, 0);
        cudaGraphDestroy(g);
        if (ie != cudaSuccess) {
            cudaGetLastError();
            s->graph_exec[par] = nullptr;
            s->graph_warm[par] = -1000000;
            return 1;
        }
    }
    // everything queued on the caller's stream comes first; the host waits for the graph below, so what follows is ordered too
    LCX_CUDA(cudaEventRecord(s->gevent, s->stream));
    LCX_CUDA(cudaStreamWaitEvent(s->gstream, s->gevent, 0));
    LCX_CUDA(cudaGraphLaunch(s->graph_exec[par], s->gstream));
    s->launches += s->graph_launches[par];
    LCX_CUDA(cudaStreamSynchronize(s->gstream));
    return 0;
}

// The loop body of fit (:137-151) with _update_ns's backtracking (:290-334) for up to max_iter iterations of ONE annealing
// stage, entirely on this side of the ABI: between two iterations the GPU waits only for the mailbox read and a few
// branches, not for an interpreter.  Per iteration i < *n_done: tc[i] (the objective after it), tangent[i], eta[i] (accepted
// step, 0 if none), trials[i], quick_fails[i].  *stop_reason: 0 = max_iter iterations done, 1 = |delta TC| < tol (:152),
// 2 = the update produced invalid moments (the reference prints an error and returns, :144-149; iteration *n_done - 1 is
// the failing one and was not applied).  tc_start = TC of the current moments (the caller holds it).
extern "C" int lcx_run_stage_ns(lcx_session* s, double eps, double tol, int exact_trials, int max_iter, double tc_start,
                                int* n_done, int* stop_reason, double* tc, double* tangent, double* eta, int* trials,
                                int* quick_fails) {
    S_REQUIRE_BOUND(s);
    LCX_REQUIRE(n_done && stop_reason && tc && tangent && eta && trials && quick_fails && max_iter >= 0, "bad argument");
    double tc_cur = tc_start;
    *n_done = 0;
    *stop_reason = 0;
    const double eta_min = tol < 1e-10 ? tol : 1e-10;
    for (int it = 0; it < max_iter; ++it) {
        const double last_tc = tc_cur;
        bool have_first = false, mailbox_ready = false;
        if (exact_trials) {
            LCX_TRY(enqueue_direction(s, eps));
        } else {  // direction and the eta = 1 trial share one host synchronisation (discarded if tangent >= 0)
            int plain = 1;
            if (graphs_enabled(s)) {
                plain = iteration_graph(s, eps);
                if (plain < 0) return plain;
            }
            if (plain) {
                LCX_TRY(enqueue_direction(s, eps));
                LCX_TRY(enqueue_trial(s, eps, 1.0, 0));
            }
            have_first = true;
            mailbox_ready = !plain;  // a replayed graph ends with the mailbox copy and the host has already waited for it
        }
        if (!mailbox_ready) LCX_TRY(read_mailbox(s));
        const double tang = s->mailbox[2];
        tangent[it] = tang;
        eta[it] = 0.0;
        trials[it] = 0;
        quick_fails[it] = 0;
        *n_done = it + 1;
        if (!(tang >= 0)) {  // (:306-311 returns the unchanged moments when tangent >= 0)
            double e = 1.0;
            int last_fail = -1;  // -1: no trial ran, 1: the last trial hit max uj >= 1, 0: it produced moments
            double tc_trial = 0.0;
            while (true) {
                if (e < eta_min) break;  // :316-319
                if (have_first) {
                    have_first = false;
                } else {
                    LCX_TRY(enqueue_trial(s, eps, e, exact_trials));
                    LCX_TRY(read_mailbox(s));
                }
                tc_trial = s->mailbox[0];
                trials[it]++;
                if (s->mailbox[1] >= 1.0) {  // TEST 1 (:322-326)
                    last_fail = 1;
                    quick_fails[it]++;
                    e *= 0.5;
                    continue;
                }
                last_fail = 0;
                if (!(-tc_trial <= -tc_cur + 0.1 * e * tang)) {  // TEST 2, first Wolfe condition (:327-332)
                    e *= 0.5;
                    continue;
                }
                break;
            }
            eta[it] = e;
            if (last_fail != 0) {
                tc[it] = tc_cur;
                *stop_reason = 2;
                return 0;
            }
            s->cur ^= 1;  // accept (:333-334)
            tc_cur = tc_trial;
        }
        tc[it] = tc_cur;
        const double delta = fabs(tc_cur - last_tc);
        if (delta < tol) {
            *stop_reason = 1;
            return 0;
        }
    }
    return 0;
}

extern "C" int lcx_accept_trial(lcx_session* s) {
    S_REQUIRE_BOUND(s);
    s->cur ^= 1;
    return 0;
}

extern "C" int lcx_details_ns(lcx_session* s, double* tc_no_overlap, double* additivity) {
    S_REQUIRE_BOUND(s);
    const Layout& L = s->L;
    const int m = s->m, n = s->n;
    double* rho = s->ptr(LCX_A_RHO);
    // X_i Z_j = solve(ry, rho)^T (:280)
    LCX_TRY(run_solve(s, s->ptr(LCX_A_RY), L.ldm, rho, L.ld, s->ptr(LCX_A_XZ), L.ld));
    LCX_TRY(details_tail(s, rho, nullptr));
    // X_i Y_j = rho^T sqrt(Y_j^2) (:279)
    scale_rows_out_kernel<<<grid_mn(m, n), 256, 0, s->stream>>>(rho, s->ptr(I_SQRTY), s->ptr(LCX_A_XY), m, n, L.ld);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    LCX_TRY(read_mailbox(s));
    if (s->mailbox[8] != 0.0) return fail(LCX_ERR_SINGULAR, "lcx_details_ns", "Singular matrix (ry)");
    if (tc_no_overlap) *tc_no_overlap = s->mailbox[4];
    if (additivity) *additivity = s->mailbox[6];
    return 0;
}

extern "C" int lcx_moments_syn(lcx_session* s, double* tc, double* additivity) {
    S_REQUIRE_BOUND(s);
    const Layout& L = s->L;
    const int m = s->m, n = s->n;
    double* W = s->ptr(LCX_A_W);
    double* XY = s->ptr(LCX_A_XY);
    double* cy = s->ptr(LCX_A_CY);
    double* rinv = s->ptr(LCX_A_RHOINVRHO);
    LCX_TRY(xpair(s, W, false));
    // X_i Y_j = X~^T Y / N (:354)
    sig_finish_kernel<<<grid_mn(m, n), 256, 0, s->stream>>>(s->ptr(LCX_A_D), s->ptr(LCX_A_D), 1.0 / (double)s->Nt, 0.0, XY, m, n,
                                                          L.ld);
    LAUNCHED(s);
    {   // cy = W XY + yscale^2 I (:355)
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = W; a.B = XY; a.C = cy;
        a.M = m; a.N = m; a.K = n;
        a.lda = L.ld; a.ldb = L.ld; a.ldc = L.ldm;
        LCX_TRY(run_gemm(s, kLayoutKK, L.plan_mm, a, s->ptr(I_PART), (long long)m * L.ldm));
        diag_add_kernel<<<cdiv(m, 128), 128, 0, s->stream>>>(cy, L.ldm, m, 1.0);
        LAUNCHED(s);
    }
    syn_ry_kernel<<<dim3(cdiv(m, 128), m), 128, 0, s->stream>>>(cy, L.ldm, m, s->ptr(LCX_A_RY), s->ptr(LCX_A_YJ2),
                                                              s->ptr(I_SQRTY));
    LAUNCHED(s);
    syn_stage1_kernel<<<L.nstrips, dim3(kStripCols, kStripRows), 0, s->stream>>>(
        XY, s->ptr(I_SQRTY), s->ptr(LCX_A_RHO), s->ptr(LCX_A_INVRHO), rinv, s->ptr(LCX_A_SI), m, n, L.ld);
    LAUNCHED(s);
    {   // Qij = ry rinv (:361)
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = s->ptr(LCX_A_RY); a.B = rinv; a.C = s->ptr(LCX_A_QIJ);
        a.M = m; a.N = n; a.K = m;
        a.lda = L.ldm; a.ldb = L.ld; a.ldc = L.ld;
        LCX_TRY(run_gemm(s, kLayoutKN, L.plan_mn, a, nullptr, 0));
    }
    syn_qi_kernel<<<L.nstrips, dim3(kStripCols, kStripRows), 0, s->stream>>>(rinv, s->ptr(LCX_A_QIJ), s->ptr(LCX_A_QISI2), m, n,
                                                                           L.ld);
    LAUNCHED(s);
    // X_i Z_j = solve(cy, XY^T)^T (:366)
    LCX_TRY(run_solve(s, cy, L.ldm, XY, L.ld, s->ptr(LCX_A_XZ), L.ld));
    // sqrtY currently holds sqrt(Yj2); details_finish rewrites it with the same values
    LCX_TRY(details_tail(s, XY, s->ptr(LCX_A_YJ2)));
    syn_tc_kernel<<<1, 32, 0, s->stream>>>(s->ptr(LCX_A_SCALARS) + 4, s->ptr(LCX_A_SCALARS));
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    LCX_TRY(read_mailbox(s));
    if (s->mailbox[8] != 0.0) return fail(LCX_ERR_SINGULAR, "lcx_moments_syn", "Singular matrix (cy)");
    if (tc) *tc = s->mailbox[0];
    if (additivity) *additivity = s->mailbox[6];
    return 0;
}

extern "C" int lcx_update_syn(lcx_session* s, double eta, double* tc, double* additivity) {
    S_REQUIRE_BOUND(s);
    const Layout& L = s->L;
    const int m = s->m, n = s->n;
    double* W = s->ptr(LCX_A_W);
    double* Rm = s->ptr(I_T);
    double* H = s->ptr(LCX_A_CY);       // rebuilt by moments_syn below
    double* Sm = s->ptr(LCX_A_GRAD);
    syn_colscale_kernel<<<grid_mn(m, n), 256, 0, s->stream>>>(s->ptr(LCX_A_XZ), s->ptr(LCX_A_X2Y), Rm, m, n, L.ld);
    LAUNCHED(s);
    {   // H = (XZ^T / X2Y) XZ, diag -> 0 (:378-379)
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = Rm; a.B = s->ptr(LCX_A_XZ); a.C = H;
        a.M = m; a.N = m; a.K = n;
        a.lda = L.ld; a.ldb = L.ld; a.ldc = L.ldm;
        LCX_TRY(run_square_gemm(s, a, 0.0, nullptr));
    }
    {   // S = H W (:381)
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = H; a.B = W; a.C = Sm;
        a.M = m; a.N = n; a.K = m;
        a.lda = L.ldm; a.ldb = L.ld; a.ldc = L.ld;
        LCX_TRY(run_gemm(s, kLayoutKN, L.plan_mn, a, nullptr, 0));
    }
    syn_mix_kernel<<<grid_mn(m, n), 256, 0, s->stream>>>(W, Rm, Sm, eta, W, m, n, L.ld);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return lcx_moments_syn(s, tc, additivity);
}

// rows [row0, row0 + rows) of  diag(sd) fill_diagonal(left^T right / scale, 1) diag(sd)   (:447-451, :453-454); left / right are
// factor-major m x ld device arrays.  Free-standing: needs no bound problem.
static int covariance_rows(lcx_session* s, const double* left, const double* right, long long ld, int m, int n, double scale,
                           const double* sd, int row0, int rows, double* out, long long ldc) {
    GemmPlan pl = plan_gemm(rows, n, m, kSMs, 1, false);
    GemmArgs a;
    memset(&a, 0, sizeof(a));
    a.A = left + row0; a.B = right; a.C = out;
    a.M = rows; a.N = n; a.K = m;
    a.lda = ld; a.ldb = ld; a.ldc = ldc;
    LCX_TRY(launch_gemm(kLayoutMN, pl, a, s->stream));
    LAUNCHED(s);
    cov_finish_kernel<<<dim3(cdiv(n, 256), rows), 256, 0, s->stream>>>(out, ldc, row0, rows, n, scale, sd);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int lcx_get_covariance(lcx_session* s, int synergy, double eps, const double* sd, int row0, int rows, double* out,
                                  long long ldc) {
    S_REQUIRE_BOUND(s);
    const Layout& L = s->L;
    const int m = s->m, n = s->n;
    LCX_REQUIRE(sd && out, "null argument");
    LCX_REQUIRE(row0 >= 0 && rows > 0 && row0 + rows <= n && row0 % 2 == 0, "bad row block (row0 must be even)");
    LCX_REQUIRE(ldc >= n && ldc % 2 == 0, "ldc must be even and >= n");
    if (!synergy) {
        double* z = s->ptr(I_T);
        cov_z_kernel<<<grid_mn(m, n), 256, 0, s->stream>>>(s->ptr(LCX_A_RHOINVRHO), s->ptr(LCX_A_SI), z, m, n, L.ld);
        LAUNCHED(s);
        return covariance_rows(s, z, z, L.ld, m, n, 1.0 - eps * eps, sd, row0, rows, out, ldc);
    }
    return covariance_rows(s, s->ptr(LCX_A_XZ), s->ptr(LCX_A_XY), L.ld, m, n, 1.0, sd, row0, rows, out, ldc);
}

extern "C" int lcx_covariance_rows(lcx_session* s, const double* left, const double* right, long long ld, int n_factors,
                                   int n_vars, double scale, const double* sd, int row0, int rows, double* out, long long ldc) {
    LCX_REQUIRE(s && left && right && sd && out, "null argument");
    LCX_REQUIRE(n_factors > 0 && n_vars > 0 && ld >= n_vars && ld % 2 == 0, "bad shape (ld must be even and >= n_vars)");
    LCX_REQUIRE(row0 >= 0 && rows > 0 && row0 + rows <= n_vars && row0 % 2 == 0, "bad row block (row0 must be even)");
    LCX_REQUIRE(ldc >= n_vars && ldc % 2 == 0, "ldc must be even and >= n_vars");
    LCX_REQUIRE(((uintptr_t)left % 16 == 0) && ((uintptr_t)right % 16 == 0) && ((uintptr_t)out % 16 == 0), "misaligned device pointer");
    LCX_CUDA(cudaSetDevice(s->device));
    return covariance_rows(s, left, right, ld, n_factors, n_vars, scale, sd, row0, rows, out, ldc);
}

extern "C" int lcx_gemm_f64(lcx_session* s, int layout, int M, int N, int K, const double* a, long long lda, const double* b,
                            long long ldb, double* c, long long ldc, int trans_out, const double* cadd, int max_splits,
                            double* scratch, long long scratch_doubles) {
    LCX_REQUIRE(s && a && b && c, "null argument");
    LCX_REQUIRE(layout >= 0 && layout <= 2 && M > 0 && N > 0 && K > 0, "bad shape/layout");
    LCX_CUDA(cudaSetDevice(s->device));
    const long long out_rows = trans_out ? N : M;
    const long long out_count = out_rows * ldc;
    int ms = max_splits;
    if (scratch == nullptr || cadd != nullptr) ms = 1;
    if (ms > 1 && out_count > 0) ms = (int)min((long long)ms, scratch_doubles / out_count);
    if (ms < 1) ms = 1;
    GemmPlan pl = plan_gemm(M, N, K, kSMs, ms, ms > 1);
    GemmArgs g;
    memset(&g, 0, sizeof(g));
    g.A = a; g.B = b; g.C = c; g.Cadd = cadd;
    g.M = M; g.N = N; g.K = K;
    g.lda = lda; g.ldb = ldb; g.ldc = ldc;
    g.trans_out = trans_out;
    return run_gemm(s, (GemmLayout)layout, pl, g, scratch, out_count);
}

extern "C" long long lcx_solve_scratch_doubles(int m) { return m > 0 ? lu::scratch_doubles(m) : -1; }

extern "C" int lcx_solve(lcx_session* s, const double* a, long long lda, int m, const double* b, long long ldb, double* x,
                         long long ldx, int n_rhs, double* scratch, long long scratch_doubles) {
    LCX_REQUIRE(s && a && b && x && scratch && m > 0 && n_rhs > 0, "bad argument");
    LCX_REQUIRE(lda >= m && ldb >= n_rhs && ldx >= n_rhs, "bad leading dimension");
    LCX_REQUIRE(scratch_doubles >= lu::scratch_doubles(m), "scratch too small (see lcx_solve_scratch_doubles)");
    LCX_CUDA(cudaSetDevice(s->device));
    lu::Scratch sc = lu::carve(scratch, m);
    LCX_TRY(lu::solve(a, lda, m, b, ldb, x, ldx, n_rhs, scratch, nullptr, s->stream, &s->launches));
    int status = 0;
    LCX_CUDA(cudaMemcpyAsync(&status, sc.status, sizeof(int), cudaMemcpyDeviceToHost, s->stream));
    LCX_CUDA(cudaStreamSynchronize(s->stream));
    if (status != 0) return fail(LCX_ERR_SINGULAR, "lcx_solve", "Singular matrix");
    return 0;
}

// ---- scoring under the covariance estimate (lowrank_kernels.cuh) ---------------------------------------------------------
namespace {
// scratch of lcx_lowrank_factor: zh | zd (m x ldz each) | K - I (m x ldk) | split-K partials | work of the cooperative factor |
// lup (m x m) | perm (m ints) | status (2 ints) | per-column log terms (n) | log pivots (m) | mailbox scalars (16)
// [| G^-1 (m x ldk), lcx_lowrank_factor_h only]
struct LowrankScratch {
    double *zh, *zd, *kmat, *part, *work, *lup, *ldiag, *lpiv, *scalars, *ginv;
    int *perm, *status;
    long long ldz, ldk, total;
    GemmPlan plan;
};
LowrankScratch lowrank_carve(double* base, int m, int n, bool with_h) {
    LowrankScratch c;
    c.ldz = round_up(n, 16);
    c.ldk = round_up(m, 16);
    c.plan = plan_gemm(m, m, n, kSMs, kMaxSplitsSmall, true);
    long long cur = 0;
    auto take = [&](long long count) {
        double* p = base ? base + cur : nullptr;
        cur = align16(cur + count);
        return p;
    };
    c.zh = take((long long)m * c.ldz);
    c.zd = take((long long)m * c.ldz);
    c.kmat = take((long long)m * c.ldk);
    c.part = take(c.plan.splits > 1 ? (long long)c.plan.splits * m * c.ldk : 16);
    c.work = take(m <= lowrank::kCholSmemMaxM ? 16 : (long long)m * lu::factor_ld(m, false));
    c.lup = take((long long)m * m);
    c.perm = reinterpret_cast<int*>(take((m + 1) / 2 + 1));
    c.status = reinterpret_cast<int*>(take(1));
    c.ldiag = take(n);
    c.lpiv = take(m);
    c.scalars = take(16);
    c.ginv = with_h ? take((long long)m * c.ldk) : nullptr;
    c.total = cur;
    return c;
}
}  // namespace

extern "C" long long lcx_lowrank_scratch_doubles(int n_factors, int n_vars) {
    if (n_factors <= 0 || n_vars <= 0) return -1;
    return lowrank_carve(nullptr, n_factors, n_vars, false).total;
}

extern "C" long long lcx_lowrank_h_scratch_doubles(int n_factors, int n_vars) {
    if (n_factors <= 0 || n_vars <= 0) return -1;
    return lowrank_carve(nullptr, n_factors, n_vars, true).total;
}

// K - I = (Z Delta^-1/2)(Z Delta^-1/2)^T from the n columns of c.zh (zero when n = 0), then K = G G^T into c.lup / c.lpiv
// (chol_factor_kernel: one CTA in shared memory for m <= 160, the cooperative grid beyond)
static int gram_chol(lcx_session* s, const LowrankScratch& c, int m, int n) {
    if (n == 0) {
        LCX_CUDA(cudaMemsetAsync(c.kmat, 0, (size_t)m * c.ldk * sizeof(double), s->stream));
    } else {  // both operands K-contiguous, split-K over the variables, fixed-order combine; the identity is added where the
              // factorisation loads K
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = c.zh; a.B = c.zh; a.C = c.kmat;
        a.M = m; a.N = m; a.K = n;
        a.lda = c.ldz; a.ldb = c.ldz; a.ldc = c.ldk;
        LCX_TRY(run_gemm(s, kLayoutKK, c.plan, a, c.part, (long long)m * c.ldk));
    }
    static PerDeviceOnce attr_smem = {}, attr_coop = {};
    if (m <= lowrank::kCholSmemMaxM) {
        const size_t smem = (size_t)m * (m | 1) * sizeof(double);
        if (attr_smem.first_time())
            LCX_CUDA(cudaFuncSetAttribute(lowrank::chol_factor_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024));
        lowrank::chol_factor_kernel<true><<<1, lowrank::kCholThreads, smem, s->stream>>>(c.kmat, c.ldk, m, nullptr, c.lup, m, c.perm,
                                                                                        c.lpiv, c.status);
    } else {
        if (attr_coop.first_time())
            LCX_CUDA(cudaFuncSetAttribute(lowrank::chol_factor_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024));
        const int grid = min(64, (m + 15) / 16);
        const double* kmat = c.kmat;
        long long ldk = c.ldk, ldl = m;
        int mm = m;
        double* work = c.work;
        double* lup = c.lup;
        int* perm = c.perm;
        double* lpiv = c.lpiv;
        int* status = c.status;
        void* args[] = {&kmat, &ldk, &mm, &work, &lup, &ldl, &perm, &lpiv, &status};
        LCX_CUDA(cudaLaunchCooperativeKernel((void*)lowrank::chol_factor_kernel<false>, dim3(grid), dim3(lowrank::kCholThreads), args, 0,
                                             s->stream));
    }
    LAUNCHED(s);
    return 0;
}

// lcx_lowrank_factor, and with h != nullptr also H = G^-1 G^-T (m x ldh) before the one mailbox read
static int lowrank_factor(lcx_session* s, const char* who, const double* rhoinvrho, const double* si, long long ld, int n_factors,
                          int n_vars, double eps, const double* sd, double* b, long long ldb, double* dinv, double* logdet, double* h,
                          long long ldh, double* scratch, long long scratch_doubles) {
    LCX_REQUIRE(s && rhoinvrho && si && sd && b && dinv && logdet && scratch, "null argument");
    const int m = n_factors, n = n_vars;
    LCX_REQUIRE(m > 0 && n > 0 && ld >= n && ldb >= n && ldb % 2 == 0, "bad shape (ldb must be even and >= n_vars)");
    LCX_REQUIRE(eps >= 0.0 && eps < 1.0, "eps must lie in [0, 1)");
    const bool with_h = h != nullptr;
    LCX_REQUIRE(scratch_doubles >= lowrank_carve(nullptr, m, n, with_h).total,
                with_h ? "scratch too small (see lcx_lowrank_h_scratch_doubles)" : "scratch too small (see lcx_lowrank_scratch_doubles)");
    LCX_REQUIRE(((uintptr_t)scratch % 16 == 0) && ((uintptr_t)b % 16 == 0), "misaligned device pointer");
    LCX_REQUIRE(!with_h || (ldh >= m && ldh % 2 == 0 && (uintptr_t)h % 16 == 0), "bad h (ldh must be even and >= n_factors)");
    LCX_CUDA(cudaSetDevice(s->device));
    const LowrankScratch c = lowrank_carve(scratch, m, n, with_h);
    LCX_CUDA(cudaMemsetAsync(c.status, 0, 2 * sizeof(int), s->stream));
    lowrank::factor_prep_kernel<<<cdiv(n, 256), 256, 0, s->stream>>>(rhoinvrho, si, ld, c.ldz, m, n, 1.0 / sqrt(1.0 - eps * eps), sd,
                                                                     c.zh, c.zd, dinv, c.ldiag, c.status);
    LAUNCHED(s);
    LCX_TRY(gram_chol(s, c, m, n));
    // B = G^-1 (Z Delta^-1) = diag(G)^-1 L^-1 (Z Delta^-1): the details path's triangular sweeps, identity permutation
    LCX_TRY(lu::launch_solve(c.lup, m, c.perm, m, c.zd, c.ldz, b, ldb, n, c.status, nullptr, s->stream, &s->launches));
    if (with_h) {  // G^-1 = the same sweeps on the identity (held in h until the product overwrites it), H = G^-1 (G^-1)^T
        lowrank::eye_kernel<<<dim3(cdiv(m, 256), m), 256, 0, s->stream>>>(h, ldh, m);
        LAUNCHED(s);
        LCX_TRY(lu::launch_solve(c.lup, m, c.perm, m, h, ldh, c.ginv, c.ldk, m, c.status, nullptr, s->stream, &s->launches));
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = c.ginv; a.B = c.ginv; a.C = h;
        a.M = m; a.N = m; a.K = m;
        a.lda = c.ldk; a.ldb = c.ldk; a.ldc = ldh;
        LCX_TRY(run_gemm(s, kLayoutKK, plan_gemm(m, m, m, kSMs, 1, false), a, nullptr, (long long)m * ldh));
    }
    lowrank::logdet_kernel<<<1, 256, 0, s->stream>>>(c.ldiag, n, c.lpiv, m, c.status, logdet, c.scalars);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    LCX_TRY(read_mailbox(s, c.scalars));
    if (s->mailbox[0] != 0.0) return fail(LCX_ERR_NOT_PD, who, "Matrix is not positive definite");
    return 0;
}

extern "C" int lcx_lowrank_factor(lcx_session* s, const double* rhoinvrho, const double* si, long long ld, int n_factors, int n_vars,
                                  double eps, const double* sd, double* b, long long ldb, double* dinv, double* logdet, double* scratch,
                                  long long scratch_doubles) {
    return lowrank_factor(s, "lcx_lowrank_factor", rhoinvrho, si, ld, n_factors, n_vars, eps, sd, b, ldb, dinv, logdet, nullptr, 0,
                          scratch, scratch_doubles);
}

extern "C" int lcx_lowrank_factor_h(lcx_session* s, const double* rhoinvrho, const double* si, long long ld, int n_factors,
                                    int n_vars, double eps, const double* sd, double* b, long long ldb, double* dinv, double* logdet,
                                    double* h, long long ldh, double* scratch, long long scratch_doubles) {
    LCX_REQUIRE(h != nullptr, "null argument");
    return lowrank_factor(s, "lcx_lowrank_factor_h", rhoinvrho, si, ld, n_factors, n_vars, eps, sd, b, ldb, dinv, logdet, h, ldh,
                          scratch, scratch_doubles);
}

extern "C" long long lcx_score_scratch_doubles(long long n_rows, int n_vars, int n_factors) {
    if (n_rows <= 0 || n_vars <= 0 || n_factors <= 0) return -1;
    return align16(n_rows * round_up(n_vars, 16)) + align16(n_rows) + align16(n_rows * round_up(n_factors, 8));
}

extern "C" int lcx_score_rows(lcx_session* s, const void* x, int dtype, long long n_rows, int n_vars, long long ldx, int has_marker,
                              double marker, const double* impute, const double* mean, const double* sd, const double* b, long long ldb,
                              int n_factors, const double* dinv, const double* logdet, double* maha, double* logpdf, double* scratch,
                              long long scratch_doubles) {
    LCX_REQUIRE(s && x && mean && sd && b && dinv && logdet && maha && logpdf && scratch, "null argument");
    LCX_REQUIRE(has_marker == 0 || impute != nullptr, "imputation means required when a missing marker is set");
    LCX_REQUIRE(n_rows > 0 && n_rows < (1LL << 31) && n_vars > 0 && n_factors > 0 && ldx >= n_vars && ldb >= n_vars && ldb % 2 == 0,
                "bad shape");
    LCX_REQUIRE(scratch_doubles >= lcx_score_scratch_doubles(n_rows, n_vars, n_factors),
                "scratch too small (see lcx_score_scratch_doubles)");
    LCX_REQUIRE(((uintptr_t)scratch % 16 == 0) && ((uintptr_t)b % 16 == 0), "misaligned device pointer");
    LCX_CUDA(cudaSetDevice(s->device));
    const long long ld = round_up(n_vars, 16), ldy = round_up(n_factors, 8);
    double* xt = scratch;
    double* ssq = xt + align16(n_rows * ld);
    double* y = ssq + align16(n_rows);
    const int nan_marker = marker != marker;
    if (dtype == LCX_F32 && vec4_ok((const float*)x, ldx))
        lowrank::score_standardize_kernel<float, true, false><<<(unsigned)n_rows, 256, 0, s->stream>>>(
            (const float*)x, n_rows, n_vars, ldx, has_marker, marker, nan_marker, impute, mean, sd, dinv, xt, ld, ssq, nullptr, nullptr,
            nullptr, 0);
    else if (dtype == LCX_F32)
        lowrank::score_standardize_kernel<float, false, false><<<(unsigned)n_rows, 256, 0, s->stream>>>(
            (const float*)x, n_rows, n_vars, ldx, has_marker, marker, nan_marker, impute, mean, sd, dinv, xt, ld, ssq, nullptr, nullptr,
            nullptr, 0);
    else if (dtype == LCX_F64 && vec4_ok((const double*)x, ldx))
        lowrank::score_standardize_kernel<double, true, false><<<(unsigned)n_rows, 256, 0, s->stream>>>(
            (const double*)x, n_rows, n_vars, ldx, has_marker, marker, nan_marker, impute, mean, sd, dinv, xt, ld, ssq, nullptr, nullptr,
            nullptr, 0);
    else if (dtype == LCX_F64)
        lowrank::score_standardize_kernel<double, false, false><<<(unsigned)n_rows, 256, 0, s->stream>>>(
            (const double*)x, n_rows, n_vars, ldx, has_marker, marker, nan_marker, impute, mean, sd, dinv, xt, ld, ssq, nullptr, nullptr,
            nullptr, 0);
    else
        return fail(LCX_ERR_ARG, "lcx_score_rows", "unknown dtype");
    LAUNCHED(s);
    // Y = X~ B^T on the DMMA engine (transform's projection, no split-K: every row's sums run in the same order)
    LCX_TRY(lcx_project(s, xt, n_rows, n_vars, ld, b, ldb, n_factors, y, ldy, nullptr, nullptr, 0));
    lowrank::score_finish_kernel<<<cdiv(n_rows, 8), 256, 0, s->stream>>>(y, ldy, ssq, n_rows, n_factors, logdet,
                                                                         (double)n_vars * log(2.0 * M_PI), maha, logpdf);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}

// rows [row0, row0 + rows) of Sigma^-1 = S^-1 (Delta^-1 - B^T B) S^-1: B^T B on the DMMA engine in get_covariance's layout
// (z^T z), then the diagonal and the scales.  The twin of lcx_covariance_rows.
extern "C" int lcx_precision_rows(lcx_session* s, const double* b, long long ldb, int n_factors, int n_vars, const double* dinv,
                                  const double* sd, int row0, int rows, double* out, long long ldc) {
    LCX_REQUIRE(s && b && dinv && sd && out, "null argument");
    LCX_REQUIRE(n_factors > 0 && n_vars > 0 && ldb >= n_vars && ldb % 2 == 0, "bad shape (ldb must be even and >= n_vars)");
    LCX_REQUIRE(row0 >= 0 && rows > 0 && row0 + rows <= n_vars && row0 % 2 == 0, "bad row block (row0 must be even)");
    LCX_REQUIRE(ldc >= n_vars && ldc % 2 == 0, "ldc must be even and >= n_vars");
    LCX_REQUIRE(((uintptr_t)b % 16 == 0) && ((uintptr_t)out % 16 == 0), "misaligned device pointer");
    LCX_CUDA(cudaSetDevice(s->device));
    GemmPlan pl = plan_gemm(rows, n_vars, n_factors, kSMs, 1, false);
    GemmArgs a;
    memset(&a, 0, sizeof(a));
    a.A = b + row0; a.B = b; a.C = out;
    a.M = rows; a.N = n_vars; a.K = n_factors;
    a.lda = ldb; a.ldb = ldb; a.ldc = ldc;
    LCX_TRY(launch_gemm(kLayoutMN, pl, a, s->stream));
    LAUNCHED(s);
    lowrank::precision_finish_kernel<<<dim3(cdiv(n_vars, 256), rows), 256, 0, s->stream>>>(out, ldc, row0, rows, n_vars, dinv, sd);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}

// ---- conditioning on the observed entries (lowrank_kernels.cuh: score_standardize_kernel<MASK>, condition_rows_kernel) ----
namespace {
// scratch of lcx_condition_rows: x~° (rows x ld) | s° (rows) | c (rows x ldy) | missing / observed lists (rows x n ints) |
// missing counts (rows ints) | class counters (kCondCounts) | per-CTA slabs of the global class
struct ConditionScratch {
    double *xt, *ssq, *y, *slabs;
    int *miss, *nmiss;
    unsigned long long* counts;
    long long ld, ldy, slab_doubles, total;
    int pmax, nslabs;
};
ConditionScratch condition_carve(double* base, long long rows, int n, int m, bool sample = false) {
    ConditionScratch c;
    c.ld = round_up(n, 16);
    c.ldy = round_up(m, 8);
    c.pmax = 0;
    for (int k = 1; k <= n; ++k) c.pmax = max(c.pmax, lowrank::cond_order(k, n, m, sample));
    c.slab_doubles = c.nslabs = 0;
    if (c.pmax > lowrank::kCondSmemMax) {  // at most 2 CTAs per SM, and about 1 GB of slabs
        c.slab_doubles = align16(lowrank::cond_matrix_doubles(c.pmax));
        c.nslabs = (int)max(1LL, min(min((long long)2 * kSMs, rows), (1LL << 27) / c.slab_doubles));
    }
    long long cur = 0;
    auto take = [&](long long count) {
        double* p = base ? base + cur : nullptr;
        cur = align16(cur + count);
        return p;
    };
    c.xt = take(rows * c.ld);
    c.ssq = take(rows);
    c.y = take(rows * c.ldy);
    c.miss = reinterpret_cast<int*>(take((rows * n + 1) / 2));
    c.nmiss = reinterpret_cast<int*>(take((rows + 1) / 2));
    c.counts = reinterpret_cast<unsigned long long*>(take(lowrank::kCondCounts));
    c.slabs = take((long long)c.nslabs * c.slab_doubles);
    c.total = cur;
    return c;
}

// the kCondSample outputs of condition_rows_kernel (all zero in kCondMean mode)
struct CondSampleOut {
    double *sdo, *draws;
    long long ldo, draw_stride;
    unsigned long long seed;
    long long row0;
    int n_draws;
};

template <bool IN_SMEM, int MODE>
int launch_condition(lcx_session* s, const ConditionScratch& c, long long n_rows, int n, int m, const double* b, long long ldb,
                     const double* h, long long ldh, const double* dinv, const double* mean, const double* sd, const double* logdet,
                     int pmin, int pmax, double* imputed, long long ldi, double* maha, double* logpdf,
                     unsigned long long* counts, const CondSampleOut& so) {
    static PerDeviceOnce attr = {};
    auto kern = lowrank::condition_rows_kernel<IN_SMEM, MODE>;
    const size_t smem = IN_SMEM ? (size_t)lowrank::cond_matrix_doubles(pmax) * sizeof(double) : 0;
    if (IN_SMEM && attr.first_time())
        LCX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)(lowrank::cond_matrix_doubles(lowrank::kCondSmemMax) * sizeof(double))));
    int grid = c.nslabs;
    if (IN_SMEM) {
        int per_sm = 0;
        LCX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, lowrank::kCondThreads, smem));
        grid = (int)min(n_rows, (long long)max(per_sm, 1) * kSMs);
    }
    kern<<<grid, lowrank::kCondThreads, smem, s->stream>>>(
        c.miss, c.nmiss, n_rows, n, m, b, ldb, h, ldh, dinv, mean, sd, logdet, log(2.0 * M_PI), c.ssq, c.xt, c.ld, c.y, c.ldy, pmin,
        pmax, c.slabs, c.slab_doubles, imputed, ldi, maha, logpdf, counts, so.sdo, so.draws, so.ldo, so.draw_stride, so.seed, so.row0,
        so.n_draws);
    LAUNCHED(s);
    return 0;
}

// the body of lcx_condition_rows / lcx_condition_sample_rows after the argument checks: the masked standardisation, the
// projection c = X~° B^T and the three size classes
template <int MODE>
int condition_rows(lcx_session* s, const char* who, const void* x, int dtype, long long n_rows, int n, long long ldx, int has_marker,
                   double marker, const double* mean, const double* sd, const double* b, long long ldb, int m, const double* h,
                   long long ldh, const double* dinv, const double* logdet, double* imputed, long long ldi, double* maha,
                   double* logpdf, const CondSampleOut& so, long long* class_counts, double* scratch) {
    LCX_CUDA(cudaSetDevice(s->device));
    const ConditionScratch c = condition_carve(scratch, n_rows, n, m, MODE == lowrank::kCondSample);
    const int nan_marker = marker != marker;
    LCX_CUDA(cudaMemsetAsync(c.counts, 0, lowrank::kCondCounts * sizeof(unsigned long long), s->stream));
#define LCX_MASK_LAUNCH(T, V)                                                                                                  \
    lowrank::score_standardize_kernel<T, V, true><<<(unsigned)n_rows, 256, 0, s->stream>>>(                                    \
        (const T*)x, n_rows, n, ldx, has_marker, marker, nan_marker, nullptr, mean, sd, dinv, c.xt, c.ld, c.ssq, c.miss, c.nmiss, \
        imputed, ldi)
    if (dtype == LCX_F32 && vec4_ok((const float*)x, ldx))
        LCX_MASK_LAUNCH(float, true);
    else if (dtype == LCX_F32)
        LCX_MASK_LAUNCH(float, false);
    else if (dtype == LCX_F64 && vec4_ok((const double*)x, ldx))
        LCX_MASK_LAUNCH(double, true);
    else if (dtype == LCX_F64)
        LCX_MASK_LAUNCH(double, false);
    else
        return fail(LCX_ERR_ARG, who, "unknown dtype");
#undef LCX_MASK_LAUNCH
    LAUNCHED(s);
    // c = X~° B^T: lcx_score_rows' projection, so a complete row gets the same c bit for bit
    LCX_TRY(lcx_project(s, c.xt, n_rows, n, c.ld, b, ldb, m, c.y, c.ldy, nullptr, nullptr, 0));
    // size classes by the order p of a row's system: [0, 64] and (64, 160] in shared memory, beyond in the slabs
    LCX_TRY((launch_condition<true, MODE>(s, c, n_rows, n, m, b, ldb, h, ldh, dinv, mean, sd, logdet, 0,
                                          min(c.pmax, lowrank::kCondSmallMax), imputed, ldi, maha, logpdf, c.counts, so)));
    if (c.pmax > lowrank::kCondSmallMax)
        LCX_TRY((launch_condition<true, MODE>(s, c, n_rows, n, m, b, ldb, h, ldh, dinv, mean, sd, logdet, lowrank::kCondSmallMax + 1,
                                              min(c.pmax, lowrank::kCondSmemMax), imputed, ldi, maha, logpdf, c.counts, so)));
    if (c.pmax > lowrank::kCondSmemMax)
        LCX_TRY((launch_condition<false, MODE>(s, c, n_rows, n, m, b, ldb, h, ldh, dinv, mean, sd, logdet, lowrank::kCondSmemMax + 1,
                                               c.pmax, imputed, ldi, maha, logpdf, c.counts, so)));
    LCX_CUDA(cudaGetLastError());
    if (class_counts) {
        unsigned long long hc[lowrank::kCondCounts];
        LCX_CUDA(cudaMemcpyAsync(hc, c.counts, sizeof(hc), cudaMemcpyDeviceToHost, s->stream));
        LCX_CUDA(cudaStreamSynchronize(s->stream));
        for (int i = 0; i < lowrank::kCondCounts; ++i) class_counts[i] = (long long)hc[i];
    }
    return 0;
}
}  // namespace

extern "C" long long lcx_condition_scratch_doubles(long long n_rows, int n_vars, int n_factors) {
    if (n_rows <= 0 || n_vars <= 0 || n_factors <= 0) return -1;
    return condition_carve(nullptr, n_rows, n_vars, n_factors).total;
}

extern "C" long long lcx_condition_sample_scratch_doubles(long long n_rows, int n_vars, int n_factors) {
    if (n_rows <= 0 || n_vars <= 0 || n_factors <= 0) return -1;
    return condition_carve(nullptr, n_rows, n_vars, n_factors, true).total;
}

extern "C" int lcx_condition_rows(lcx_session* s, const void* x, int dtype, long long n_rows, int n_vars, long long ldx, int has_marker,
                                  double marker, const double* mean, const double* sd, const double* b, long long ldb, int n_factors,
                                  const double* h, long long ldh, const double* dinv, const double* logdet, double* imputed,
                                  long long ldi, double* maha, double* logpdf, long long* class_counts, double* scratch,
                                  long long scratch_doubles) {
    LCX_REQUIRE(s && x && mean && sd && b && h && dinv && logdet && scratch, "null argument");
    LCX_REQUIRE(n_rows > 0 && n_rows < (1LL << 31) && n_vars > 0 && n_factors > 0 && ldx >= n_vars && ldb >= n_vars && ldb % 2 == 0 &&
                    ldh >= n_factors,
                "bad shape");
    LCX_REQUIRE(imputed == nullptr || ldi >= n_vars, "bad shape (ldi must be >= n_vars)");
    LCX_REQUIRE(scratch_doubles >= lcx_condition_scratch_doubles(n_rows, n_vars, n_factors),
                "scratch too small (see lcx_condition_scratch_doubles)");
    LCX_REQUIRE(((uintptr_t)scratch % 16 == 0) && ((uintptr_t)b % 16 == 0), "misaligned device pointer");
    const CondSampleOut none = {};
    return condition_rows<lowrank::kCondMean>(s, "lcx_condition_rows", x, dtype, n_rows, n_vars, ldx, has_marker, marker, mean, sd, b,
                                              ldb, n_factors, h, ldh, dinv, logdet, imputed, ldi, maha, logpdf, none, class_counts,
                                              scratch);
}

extern "C" int lcx_condition_sample_rows(lcx_session* s, const void* x, int dtype, long long n_rows, int n_vars, long long ldx,
                                         int has_marker, double marker, const double* mean, const double* sd, const double* b,
                                         long long ldb, int n_factors, const double* h, long long ldh, const double* dinv,
                                         double* imputed, long long ldi, double* std_out, double* draws, long long ldo,
                                         long long draw_stride, unsigned long long seed, long long row0, int n_draws,
                                         long long* class_counts, double* scratch, long long scratch_doubles) {
    LCX_REQUIRE(s && x && mean && sd && b && h && dinv && imputed && scratch, "null argument");
    LCX_REQUIRE(n_rows > 0 && n_rows < (1LL << 31) && n_vars > 0 && n_factors > 0 && ldx >= n_vars && ldb >= n_vars && ldb % 2 == 0 &&
                    ldh >= n_factors && ldi >= n_vars,
                "bad shape");
    LCX_REQUIRE((std_out == nullptr && draws == nullptr) || ldo >= n_vars, "bad shape (ldo must be >= n_vars)");
    LCX_REQUIRE(draws == nullptr || (n_draws > 0 && draw_stride >= n_rows * ldo), "bad draws (n_draws > 0, draw_stride >= n_rows ldo)");
    LCX_REQUIRE(row0 >= 0, "row0 must be >= 0");
    LCX_REQUIRE(scratch_doubles >= lcx_condition_sample_scratch_doubles(n_rows, n_vars, n_factors),
                "scratch too small (see lcx_condition_sample_scratch_doubles)");
    LCX_REQUIRE(((uintptr_t)scratch % 16 == 0) && ((uintptr_t)b % 16 == 0), "misaligned device pointer");
    LCX_CUDA(cudaSetDevice(s->device));
    if (std_out) LCX_CUDA(cudaMemsetAsync(std_out, 0, (size_t)n_rows * ldo * sizeof(double), s->stream));  // observed entries: 0
    const CondSampleOut so = {std_out, draws, ldo, draw_stride, seed, row0, draws ? n_draws : 0};
    return condition_rows<lowrank::kCondSample>(s, "lcx_condition_sample_rows", x, dtype, n_rows, n_vars, ldx, has_marker, marker, mean,
                                                sd, b, ldb, n_factors, h, ldh, dinv, nullptr, imputed, ldi, nullptr, nullptr, so,
                                                class_counts, scratch);
}

// ---- sampling from the fitted Gaussian (lowrank_kernels.cuh: normal_fill_kernel, sample_prep_kernel, sample_finish_kernel) ----
namespace {
// scratch of lcx_sample_rows: Z (m x ldz) | sqrt(Delta) (n) | mailbox scalars (16) | U (rows x ldu)
struct SampleScratch {
    double *z, *sqd, *scalars, *u;
    long long ldz, ldu, total;
};
SampleScratch sample_carve(double* base, long long rows, int n, int m) {
    SampleScratch c;
    c.ldz = round_up(n, 16);
    c.ldu = round_up(m, 8);
    long long cur = 0;
    auto take = [&](long long count) {
        double* p = base ? base + cur : nullptr;
        cur = align16(cur + count);
        return p;
    };
    c.z = take((long long)m * c.ldz);
    c.sqd = take(n);
    c.scalars = take(16);
    c.u = take(rows * c.ldu);
    c.total = cur;
    return c;
}
int normal_fill(lcx_session* s, unsigned long long seed, int tag, long long row0, long long rows, long long draw, int cols,
                double* out, long long ldo, uint32_t* words, long long ldw, const double* base = nullptr) {
    const long long work = rows * ((cols + 1) / 2);
    lowrank::normal_fill_kernel<<<(unsigned)min((long long)cdiv(work, 256), (long long)kSMs * 16), 256, 0, s->stream>>>(
        seed, tag, row0, rows, draw, cols, base, out, ldo, words, ldw);
    LAUNCHED(s);
    return 0;
}
}  // namespace

extern "C" int lcx_normal_fill(lcx_session* s, unsigned long long seed, int tag, long long row0, long long n_rows, long long draw,
                               int n_cols, double* out, long long ldo, unsigned int* words, long long ldw) {
    LCX_REQUIRE(s && out, "null argument");
    LCX_REQUIRE(tag >= 0 && tag < 256 && row0 >= 0 && n_rows > 0 && row0 + n_rows <= (1LL << 56) && draw >= 0 && draw < (1LL << 32) &&
                    n_cols > 0 && ldo >= n_cols && (words == nullptr || ldw >= 4LL * ((n_cols + 1) / 2)),
                "bad argument");
    LCX_CUDA(cudaSetDevice(s->device));
    LCX_TRY(normal_fill(s, seed, tag, row0, n_rows, draw, n_cols, out, ldo, words, ldw));
    LCX_CUDA(cudaGetLastError());
    return 0;
}

extern "C" long long lcx_sample_scratch_doubles(long long n_rows, int n_vars, int n_factors) {
    if (n_rows <= 0 || n_vars <= 0 || n_factors <= 0) return -1;
    return sample_carve(nullptr, n_rows, n_vars, n_factors).total;
}

extern "C" int lcx_sample_rows(lcx_session* s, const double* rhoinvrho, const double* si, long long ld, int n_factors, int n_vars,
                               double eps, const double* mean, const double* sd, unsigned long long seed, long long row0,
                               long long n_rows, double* out, long long ldo, double* scratch, long long scratch_doubles) {
    LCX_REQUIRE(s && rhoinvrho && si && mean && sd && out && scratch, "null argument");
    const int m = n_factors, n = n_vars;
    LCX_REQUIRE(m > 0 && n > 0 && ld >= n && n_rows > 0 && n_rows < (1LL << 31) && ldo >= n && ldo % 2 == 0, "bad shape (ldo must be even)");
    LCX_REQUIRE(row0 >= 0 && row0 + n_rows <= (1LL << 56), "bad row0");
    LCX_REQUIRE(eps >= 0.0 && eps < 1.0, "eps must lie in [0, 1)");
    LCX_REQUIRE(scratch_doubles >= lcx_sample_scratch_doubles(n_rows, n, m), "scratch too small (see lcx_sample_scratch_doubles)");
    LCX_REQUIRE(((uintptr_t)scratch % 16 == 0) && ((uintptr_t)out % 16 == 0), "misaligned device pointer");
    LCX_CUDA(cudaSetDevice(s->device));
    const SampleScratch c = sample_carve(scratch, n_rows, n, m);
    LCX_CUDA(cudaMemsetAsync(c.scalars, 0, 16 * sizeof(double), s->stream));
    lowrank::sample_prep_kernel<<<cdiv(n, 256), 256, 0, s->stream>>>(rhoinvrho, si, ld, c.ldz, m, n, 1.0 / sqrt(1.0 - eps * eps), c.z,
                                                                     c.sqd, c.scalars);
    LAUNCHED(s);
    LCX_TRY(normal_fill(s, seed, 0, row0, n_rows, 0, m, c.u, c.ldu, nullptr, 0));
    {   // Y = U Z into out: predict's layout (A row-major rows x m, B factor-major m x n), no split-K, so every entry sums its
        // m products in the same order whatever the row blocking
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = c.u; a.B = c.z; a.C = out;
        a.M = (int)n_rows; a.N = n; a.K = m;
        a.lda = c.ldu; a.ldb = c.ldz; a.ldc = ldo;
        LCX_TRY(run_gemm(s, kLayoutKN, plan_gemm((int)n_rows, n, m, kSMs, 1, false), a, nullptr, 0));
    }
    const long long work = n_rows * (((long long)(m + n - 1) >> 1) - (m >> 1) + 1);
    lowrank::sample_finish_kernel<<<(unsigned)min((long long)cdiv(work, 256), (long long)kSMs * 16), 256, 0, s->stream>>>(
        out, ldo, n_rows, m, n, c.sqd, mean, sd, seed, row0, 0, 0);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    LCX_TRY(read_mailbox(s, c.scalars));
    if (s->mailbox[0] != 0.0) return fail(LCX_ERR_NOT_PD, "lcx_sample_rows", "Matrix is not positive definite");
    return 0;
}

// ---- conditioning on a fixed column set (lowrank_kernels.cuh: given_*_kernel and the pieces of lcx_lowrank_factor) -------
namespace {
// scratch of lcx_conditional_factor: lcx_lowrank_factor's for the |O| observed columns (zh, zd, K - I, ..., log terms of O) |
// Z_T (m x ldt)
struct GivenFactorScratch {
    LowrankScratch f;
    double* zt;
    long long ldt, total;
};
GivenFactorScratch given_factor_carve(double* base, int m, int no, int nt) {
    GivenFactorScratch c;
    c.f = lowrank_carve(base, m, max(no, 1), false);
    c.ldt = round_up(max(nt, 1), 16);
    c.zt = base ? base + c.f.total : nullptr;
    c.total = c.f.total + align16((long long)m * c.ldt);
    return c;
}

// scratch of lcx_conditional_rows / lcx_conditional_sample_rows: x~_O (rows x ldx) | s (rows) | V (rows x ldv) | q, log p when
// the caller wants neither (rows each) | mailbox scalars (16) | V + U of a draw (rows x ldv)
struct GivenRowsScratch {
    double *xt, *ssq, *v, *maha, *logpdf, *scalars, *u;
    long long ldx, ldv, total;
};
GivenRowsScratch given_rows_carve(double* base, long long rows, int no, int m) {
    GivenRowsScratch c;
    c.ldx = round_up(max(no, 1), 16);
    c.ldv = round_up(m, 8);
    long long cur = 0;
    auto take = [&](long long count) {
        double* p = base ? base + cur : nullptr;
        cur = align16(cur + count);
        return p;
    };
    c.xt = take(rows * c.ldx);
    c.ssq = take(rows);
    c.v = take(rows * c.ldv);
    c.maha = take(rows);
    c.logpdf = take(rows);
    c.scalars = take(16);
    c.u = take(rows * c.ldv);
    c.total = cur;
    return c;
}

// x~_O and s = sum_O x~_i^2 / Delta_i (score_standardize_kernel, FLAG mode: a missing entry raises scalars[0]), then V = X~_O A^T
// by lcx_score_rows' projection (no split-K: every row's sums run in an order fixed by |O|).  |O| = 0: V = 0, s = 0.
int given_project(lcx_session* s, const char* who, const GivenRowsScratch& c, const void* x, int dtype, long long n_rows, int no,
                  long long ldx, int has_marker, double marker, const double* a, long long lda, const double* ocols, int m) {
    LCX_CUDA(cudaMemsetAsync(c.scalars, 0, 16 * sizeof(double), s->stream));
    if (no == 0) {
        LCX_CUDA(cudaMemsetAsync(c.ssq, 0, n_rows * sizeof(double), s->stream));
        LCX_CUDA(cudaMemsetAsync(c.v, 0, n_rows * c.ldv * sizeof(double), s->stream));
        return 0;
    }
    const int nan_marker = marker != marker;
#define LCX_FLAG_LAUNCH(T, V)                                                                                                    \
    lowrank::score_standardize_kernel<T, V, false, true><<<(unsigned)n_rows, 256, 0, s->stream>>>(                               \
        (const T*)x, n_rows, no, ldx, has_marker, marker, nan_marker, nullptr, ocols, ocols + no, ocols + 2 * no, c.xt, c.ldx, c.ssq, \
        nullptr, nullptr, c.scalars, 0)
    if (dtype == LCX_F32 && vec4_ok((const float*)x, ldx))
        LCX_FLAG_LAUNCH(float, true);
    else if (dtype == LCX_F32)
        LCX_FLAG_LAUNCH(float, false);
    else if (dtype == LCX_F64 && vec4_ok((const double*)x, ldx))
        LCX_FLAG_LAUNCH(double, true);
    else if (dtype == LCX_F64)
        LCX_FLAG_LAUNCH(double, false);
    else
        return fail(LCX_ERR_ARG, who, "unknown dtype");
#undef LCX_FLAG_LAUNCH
    LAUNCHED(s);
    return lcx_project(s, c.xt, n_rows, no, c.ldx, a, lda, m, c.v, c.ldv, nullptr, nullptr, 0);
}

// out (rows x ldo) = left (rows x ldv) P on the DMMA engine: sample's layout, no split-K, so every entry sums its m products in
// the same order whatever the row blocking
int given_times_p(lcx_session* s, const double* left, long long ldv, long long rows, const double* p, long long ldp, int m, int nt,
                  double* out, long long ldo) {
    GemmArgs g;
    memset(&g, 0, sizeof(g));
    g.A = left; g.B = p; g.C = out;
    g.M = (int)rows; g.N = nt; g.K = m;
    g.lda = ldv; g.ldb = ldp; g.ldc = ldo;
    return run_gemm(s, kLayoutKN, plan_gemm((int)rows, nt, m, kSMs, 1, false), g, nullptr, 0);
}

int given_status(lcx_session* s, const char* who, const GivenRowsScratch& c) {
    LCX_CUDA(cudaGetLastError());
    LCX_TRY(read_mailbox(s, c.scalars));
    if (s->mailbox[0] != 0.0) return fail(LCX_ERR_MISSING, who, "a row has a missing entry in an observed column");
    return 0;
}
}  // namespace

extern "C" long long lcx_conditional_factor_scratch_doubles(int n_factors, int n_obs, int n_tgt) {
    if (n_factors <= 0 || n_obs < 0 || n_tgt < 0) return -1;
    return given_factor_carve(nullptr, n_factors, n_obs, n_tgt).total;
}

extern "C" int lcx_conditional_factor(lcx_session* s, const double* rhoinvrho, const double* si, long long ld, int n_factors,
                                      int n_vars, double eps, const double* mean, const double* sd, const int* observed, int n_obs,
                                      const int* targets, int n_tgt, double* a, long long lda, double* p, long long ldp,
                                      double* ocols, double* tcols, double* logdet, double* scratch, long long scratch_doubles) {
    LCX_REQUIRE(s && rhoinvrho && si && mean && sd && logdet && scratch, "null argument");
    LCX_REQUIRE(n_obs == 0 || (observed && a && ocols), "null argument (observed, a, ocols)");
    LCX_REQUIRE(n_tgt == 0 || (targets && p && tcols), "null argument (targets, p, tcols)");
    const int m = n_factors, n = n_vars, no = n_obs, nt = n_tgt;
    LCX_REQUIRE(m > 0 && n > 0 && ld >= n && no >= 0 && nt >= 0 && (long long)no + nt <= n, "bad shape");
    LCX_REQUIRE(no == 0 || (lda >= no && lda % 2 == 0 && (uintptr_t)a % 16 == 0), "bad a (lda must be even and >= n_obs)");
    LCX_REQUIRE(nt == 0 || (ldp >= nt && ldp % 2 == 0 && (uintptr_t)p % 16 == 0), "bad p (ldp must be even and >= n_tgt)");
    LCX_REQUIRE(eps >= 0.0 && eps < 1.0, "eps must lie in [0, 1)");
    LCX_REQUIRE(scratch_doubles >= lcx_conditional_factor_scratch_doubles(m, no, nt),
                "scratch too small (see lcx_conditional_factor_scratch_doubles)");
    LCX_REQUIRE((uintptr_t)scratch % 16 == 0, "misaligned device pointer");
    LCX_CUDA(cudaSetDevice(s->device));
    const GivenFactorScratch c = given_factor_carve(scratch, m, no, nt);
    LCX_CUDA(cudaMemsetAsync(c.f.status, 0, 2 * sizeof(int), s->stream));
    LCX_CUDA(cudaMemsetAsync(c.f.scalars, 0, 16 * sizeof(double), s->stream));
    if (no + nt > 0) {
        lowrank::given_prep_kernel<<<cdiv(no + nt, 256), 256, 0, s->stream>>>(
            rhoinvrho, si, ld, m, n, 1.0 / sqrt(1.0 - eps * eps), mean, sd, observed, no, targets, nt, c.f.zh, c.f.zd, c.f.ldz, ocols,
            c.f.ldiag, c.zt, c.ldt, tcols, c.f.status, c.f.scalars);
        LAUNCHED(s);
    }
    // E_O - I and E_O = L L^T exactly as lcx_lowrank_factor forms K on all columns; then A and P by the same sweeps as B
    LCX_TRY(gram_chol(s, c.f, m, no));
    if (no > 0) LCX_TRY(lu::launch_solve(c.f.lup, m, c.f.perm, m, c.f.zd, c.f.ldz, a, lda, no, c.f.status, nullptr, s->stream, &s->launches));
    if (nt > 0) {
        LCX_TRY(lu::launch_solve(c.f.lup, m, c.f.perm, m, c.zt, c.ldt, p, ldp, nt, c.f.status, nullptr, s->stream, &s->launches));
        lowrank::given_std_kernel<<<cdiv(nt, 256), 256, 0, s->stream>>>(p, ldp, m, nt, tcols);
        LAUNCHED(s);
    }
    lowrank::logdet_kernel<<<1, 256, 0, s->stream>>>(c.f.ldiag, no, c.f.lpiv, m, c.f.status, logdet, c.f.scalars);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    LCX_TRY(read_mailbox(s, c.f.scalars));
    if (s->mailbox[2] != 0.0) return fail(LCX_ERR_ARG, "lcx_conditional_factor", "column index out of range");
    if (s->mailbox[0] != 0.0) return fail(LCX_ERR_NOT_PD, "lcx_conditional_factor", "Matrix is not positive definite");
    return 0;
}

extern "C" long long lcx_conditional_scratch_doubles(long long n_rows, int n_obs, int n_factors) {
    if (n_rows <= 0 || n_obs < 0 || n_factors <= 0) return -1;
    return given_rows_carve(nullptr, n_rows, n_obs, n_factors).total;
}

extern "C" int lcx_conditional_rows(lcx_session* s, const void* x, int dtype, long long n_rows, int n_obs, long long ldx, int has_marker,
                                    double marker, const double* a, long long lda, const double* ocols, const double* p, long long ldp,
                                    int n_tgt, const double* tcols, int n_factors, const double* logdet, double* pred, long long ldpred,
                                    double* maha, double* logpdf, double* scratch, long long scratch_doubles) {
    const int m = n_factors, no = n_obs, nt = n_tgt;
    LCX_REQUIRE(s && logdet && scratch && (no == 0 || (x && a && ocols)) && (nt == 0 || (p && tcols)), "null argument");
    LCX_REQUIRE(n_rows > 0 && n_rows < (1LL << 31) && no >= 0 && nt >= 0 && m > 0 && ldx >= no && (no == 0 || lda >= no) &&
                    (nt == 0 || ldp >= nt),
                "bad shape");
    LCX_REQUIRE(pred == nullptr || nt == 0 || (ldpred >= nt && ldpred % 2 == 0 && (uintptr_t)pred % 16 == 0),
                "bad pred (ldpred must be even and >= n_tgt)");
    LCX_REQUIRE(scratch_doubles >= lcx_conditional_scratch_doubles(n_rows, no, m), "scratch too small (see lcx_conditional_scratch_doubles)");
    LCX_REQUIRE((uintptr_t)scratch % 16 == 0 && (no == 0 || (uintptr_t)a % 16 == 0), "misaligned device pointer");
    LCX_CUDA(cudaSetDevice(s->device));
    const GivenRowsScratch c = given_rows_carve(scratch, n_rows, no, m);
    LCX_TRY(given_project(s, "lcx_conditional_rows", c, x, dtype, n_rows, no, ldx, has_marker, marker, a, lda, ocols, m));
    if (pred && nt > 0) {
        LCX_TRY(given_times_p(s, c.v, c.ldv, n_rows, p, ldp, m, nt, pred, ldpred));
        const long long work = n_rows * nt;
        lowrank::given_mean_finish_kernel<<<(unsigned)min((long long)cdiv(work, 256), (long long)kSMs * 16), 256, 0, s->stream>>>(
            pred, ldpred, n_rows, nt, tcols);
        LAUNCHED(s);
    }
    if (maha || logpdf) {  // q = s - |V_r|^2 and log p with |O| and log det Sigma_OO: score_finish_kernel's arithmetic
        lowrank::score_finish_kernel<<<cdiv(n_rows, 8), 256, 0, s->stream>>>(c.v, c.ldv, c.ssq, n_rows, m, logdet,
                                                                             (double)no * log(2.0 * M_PI), maha ? maha : c.maha,
                                                                             logpdf ? logpdf : c.logpdf);
        LAUNCHED(s);
    }
    return given_status(s, "lcx_conditional_rows", c);
}

extern "C" int lcx_conditional_sample_rows(lcx_session* s, const void* x, int dtype, long long n_rows, int n_obs, long long ldx,
                                           int has_marker, double marker, const double* a, long long lda, const double* ocols,
                                           const double* p, long long ldp, int n_tgt, const double* tcols, int n_factors,
                                           double* draws, long long ldo, long long draw_stride, unsigned long long seed,
                                           long long row0, int n_draws, double* scratch, long long scratch_doubles) {
    const int m = n_factors, no = n_obs, nt = n_tgt;
    LCX_REQUIRE(s && scratch && (no == 0 || (x && a && ocols)) && (nt == 0 || (p && tcols && draws)), "null argument");
    LCX_REQUIRE(n_rows > 0 && n_rows < (1LL << 31) && no >= 0 && nt >= 0 && m > 0 && ldx >= no && (no == 0 || lda >= no) &&
                    (nt == 0 || ldp >= nt),
                "bad shape");
    LCX_REQUIRE(nt == 0 || (ldo >= nt && ldo % 2 == 0 && (uintptr_t)draws % 16 == 0), "bad draws (ldo must be even and >= n_tgt)");
    LCX_REQUIRE(n_draws > 0 && (nt == 0 || n_draws == 1 || (draw_stride >= n_rows * ldo && draw_stride % 2 == 0)),
                "bad draws (n_draws > 0, draw_stride even and >= n_rows ldo)");
    LCX_REQUIRE(row0 >= 0 && row0 + n_rows <= (1LL << 56), "bad row0");
    LCX_REQUIRE(scratch_doubles >= lcx_conditional_scratch_doubles(n_rows, no, m), "scratch too small (see lcx_conditional_scratch_doubles)");
    LCX_REQUIRE((uintptr_t)scratch % 16 == 0 && (no == 0 || (uintptr_t)a % 16 == 0), "misaligned device pointer");
    LCX_CUDA(cudaSetDevice(s->device));
    const GivenRowsScratch c = given_rows_carve(scratch, n_rows, no, m);
    LCX_TRY(given_project(s, "lcx_conditional_sample_rows", c, x, dtype, n_rows, no, ldx, has_marker, marker, a, lda, ocols, m));
    if (nt > 0)
        for (int d = 0; d < n_draws; ++d) {  // V + u (tag-2 normals 0..m-1), (V + u) P, then + Delta_T^1/2 eps (normals m..m+|T|-1)
            double* out = draws + (long long)d * draw_stride;
            LCX_TRY(normal_fill(s, seed, 2, row0, n_rows, d, m, c.u, c.ldv, nullptr, 0, c.v));
            LCX_TRY(given_times_p(s, c.u, c.ldv, n_rows, p, ldp, m, nt, out, ldo));
            const long long work = n_rows * (((long long)(m + nt - 1) >> 1) - (m >> 1) + 1);
            lowrank::sample_finish_kernel<<<(unsigned)min((long long)cdiv(work, 256), (long long)kSMs * 16), 256, 0, s->stream>>>(
                out, ldo, n_rows, m, nt, tcols + 3 * (long long)nt, tcols, tcols + nt, seed, row0, 2, d);
            LAUNCHED(s);
        }
    return given_status(s, "lcx_conditional_sample_rows", c);
}

// rows [row0, row0 + rows) of theta1_T (Delta_T + P^T P) theta1_T: P^T P on the DMMA engine in lcx_precision_rows' layout, then the
// diagonal and the scales
extern "C" int lcx_conditional_covariance_rows(lcx_session* s, const double* p, long long ldp, int n_factors, int n_tgt,
                                               const double* tcols, int row0, int rows, double* out, long long ldc) {
    LCX_REQUIRE(s && p && tcols && out, "null argument");
    LCX_REQUIRE(n_factors > 0 && n_tgt > 0 && ldp >= n_tgt && ldp % 2 == 0, "bad shape (ldp must be even and >= n_tgt)");
    LCX_REQUIRE(row0 >= 0 && rows > 0 && row0 + rows <= n_tgt && row0 % 2 == 0 && rows < 65536, "bad row block (row0 must be even)");
    LCX_REQUIRE(ldc >= n_tgt && ldc % 2 == 0, "ldc must be even and >= n_tgt");
    LCX_REQUIRE(((uintptr_t)p % 16 == 0) && ((uintptr_t)out % 16 == 0), "misaligned device pointer");
    LCX_CUDA(cudaSetDevice(s->device));
    GemmArgs g;
    memset(&g, 0, sizeof(g));
    g.A = p + row0; g.B = p; g.C = out;
    g.M = rows; g.N = n_tgt; g.K = n_factors;
    g.lda = ldp; g.ldb = ldp; g.ldc = ldc;
    LCX_TRY(launch_gemm(kLayoutMN, plan_gemm(rows, n_tgt, n_factors, kSMs, 1, false), g, s->stream));
    LAUNCHED(s);
    lowrank::given_cov_finish_kernel<<<dim3(cdiv(n_tgt, 256), rows), 256, 0, s->stream>>>(out, ldc, row0, rows, n_tgt, tcols);
    LAUNCHED(s);
    LCX_CUDA(cudaGetLastError());
    return 0;
}
