// The split path of oz_gemm_kernel at S = 6 (groups 0-1 in a side launch, groups 2-5 in a main launch, one CTA per 128-row
// tile of all m <= 128 factors) against the pair path (two 56-wide tiles on a CTA pair sharing X~ by multicast), on the same
// digit planes, in one process: device time of each launch (CUDA events, launches alternated) and a bitwise comparison of
// every output the two paths write (Y, the split-K and tail partials of D).  The planes are made by the library's own kernels
// from Gaussian data, so the digit statistics are those of a real fit.  K-split plans are passed in as printed by
// LCX_PLAN_DEBUG (the default is config 3: 100 000 x 10 000 x 100).  Not part of the product.  Build + run on a GPU box:
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 --expt-relaxed-constexpr -I linearcorex_b200/csrc -I tools/experiments \
//        -o tools/experiments/bin/oz_split_probe tools/experiments/oz_split_probe.cu -lcuda && tools/experiments/bin/oz_split_probe
//   args: N n m  k1_splits k1_chunk k1_tail_tiles k1_tail_splits k1_tail_chunk  k2_splits k2_chunk k2_tail_tiles k2_tail_splits
//         k2_tail_chunk  repeats
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <cuda_runtime.h>

namespace lcx { thread_local char g_err[512] = ""; }
#include "ozaki_i8.cuh"
#include "oz_gemm_split.cuh"

using namespace lcx;
using namespace lcx::oz;

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(2); } } while (0)
#define TRY(x) do { if ((x) != 0) { printf("error %s at %s:%d\n", g_err, __FILE__, __LINE__); exit(2); } } while (0)

__device__ double gauss(unsigned long long i, unsigned long long seed) {
    auto mix = [](unsigned long long z) {
        z += 0x9e3779b97f4a7c15ULL; z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL; z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL;
        return z ^ (z >> 31);
    };
    const unsigned long long a = mix(i * 2 + seed * 0x1234567ULL), b = mix(i * 2 + 1 + seed * 0x1234567ULL);
    const double u1 = ((a >> 11) + 1) * (1.0 / 9007199254740993.0), u2 = (b >> 11) * (1.0 / 9007199254740992.0);
    return sqrt(-2.0 * log(u1)) * cos(6.283185307179586 * u2);
}
__global__ void fill_kernel(double* x, long long rows, int cols, long long ld, double scale, unsigned long long seed) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * ld) return;
    const long long r = i / ld;
    const int c = (int)(i - r * ld);
    x[i] = c < cols ? scale * gauss((unsigned long long)(r * cols + c), seed) : 0.0;
}
__global__ void count_diff_kernel(const unsigned long long* a, const unsigned long long* b, long long n, unsigned long long* out) {
    long long cnt = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        cnt += a[i] != b[i];
    if (cnt) atomicAdd(out, (unsigned long long)cnt);
}
static unsigned long long count_diff(const double* a, const double* b, long long n) {
    unsigned long long* d;
    CK(cudaMalloc(&d, 8));
    CK(cudaMemset(d, 0, 8));
    count_diff_kernel<<<1184, 256>>>((const unsigned long long*)a, (const unsigned long long*)b, n, d);
    unsigned long long h = 0;
    CK(cudaMemcpy(&h, d, 8, cudaMemcpyDeviceToHost));
    CK(cudaFree(d));
    return h;
}

struct Plan { int splits, chunk, tail_tiles, tail_splits, tail_chunk; };

int main(int argc, char** argv) {
    long long N = 100000; int n = 10000, m = 100;
    Plan k1 = {1, 10048, 0, 0, 0}, k2 = {7, 14336, 35, 2, 7040};
    int reps = 10;
    if (argc >= 4) { N = atoll(argv[1]); n = atoi(argv[2]); m = atoi(argv[3]); }
    if (argc >= 14) {
        k1 = {atoi(argv[4]), atoi(argv[5]), atoi(argv[6]), atoi(argv[7]), atoi(argv[8])};
        k2 = {atoi(argv[9]), atoi(argv[10]), atoi(argv[11]), atoi(argv[12]), atoi(argv[13])};
    }
    if (argc >= 15) reps = atoi(argv[14]);
    constexpr int S = 6;
    const long long ld = round_up(n, 16), ld8 = round_up(n, 128), ldk8 = round_up(N, 128), ldy = round_up(m, 8);
    const int bn_pair = (int)std::max(16LL, round_up(cdiv(m, cdiv(m, bn_max(S))), 8));
    const int bn_split = (int)round_up(m, 16);
    printf("shape N=%lld n=%d m=%d  bn pair %d split %d  K1 %d x %d tail %d x %d (%d)  K2 %d x %d tail %d x %d (%d)\n", N, n, m, bn_pair,
           bn_split, k1.splits, k1.chunk, k1.tail_tiles, k1.tail_splits, k1.tail_chunk, k2.splits, k2.chunk, k2.tail_tiles,
           k2.tail_splits, k2.tail_chunk);

    double *x, *a, *scal;
    int8_t *xs, *as, *ys;
    CK(cudaMalloc(&x, N * ld * 8));
    CK(cudaMalloc(&a, (long long)m * ld * 8));
    CK(cudaMalloc(&scal, 8 * (16 + 8 * 1024 + 4096)));
    double* xscale = scal; double* ascale = scal + 16; double* cscale = ascale + 1024; double* yscale = cscale + 1024;
    double* dscale = yscale + 1024; double* colsq = dscale + 1024; double* part = colsq + 1024;
    CK(cudaMalloc(&xs, (long long)S * N * ld8));
    CK(cudaMalloc(&as, (long long)S * m * ld8));
    CK(cudaMalloc(&ys, (long long)S * m * ldk8));
    fill_kernel<<<cdiv(N * ld, 256), 256>>>(x, N, n, ld, 1.0, 1);
    fill_kernel<<<cdiv((long long)m * ld, 256), 256>>>(a, m, n, ld, 0.1 / sqrt((double)n), 2);
    absmax_partial_kernel<<<592, 256>>>(x, ld, N, n, part);
    absmax_finish_kernel<<<1, 256>>>(part, 592, xscale);
    slice_rows_kernel<S><<<dim3((unsigned)N, cdiv(ld8, 512)), 128>>>(x, ld, (int)N, n, nullptr, xscale, xs, ld8, N * ld8, (double)kRadix);
    row_scale_kernel<<<m, 256>>>(a, ld, n, ascale, 0, xscale, cscale);
    slice_rows_kernel<S><<<dim3(m, cdiv(ld8, 512)), 128>>>(a, ld, m, n, ascale, nullptr, as, ld8, (long long)m * ld8, (double)kRadix);
    CK(cudaDeviceSynchronize());
    CK(cudaFree(x));

    CUtensorMap map_x_k1, map_x_k2, map_a_pair, map_a_split, map_y_pair, map_y_split;
    TRY(make_slice_map(&map_x_k1, xs, n, N, S, ld8, N * ld8, kBK, kBM, false));
    TRY(make_slice_map(&map_x_k2, xs, n, N, S, ld8, N * ld8, kBM, kBK, true));
    TRY(make_slice_map(&map_a_pair, as, n, m, S, ld8, (long long)m * ld8, kBK, bn_pair, false));
    TRY(make_slice_map(&map_a_split, as, n, m, S, ld8, (long long)m * ld8, kBK, bn_split, false));
    TRY(make_slice_map(&map_y_pair, ys, N, m, S, ldk8, (long long)m * ldk8, kBK, bn_pair, false));
    TRY(make_slice_map(&map_y_split, ys, N, m, S, ldk8, (long long)m * ldk8, kBK, bn_split, false));

    // outputs: [split][rows][ld] partials (+ tails), one set per path
    const long long c1 = (long long)k1.splits * N * ldy, t1 = std::max(16LL, (long long)k1.tail_splits * k1.tail_tiles * kBM * ldy);
    const long long c2 = (long long)k2.splits * m * ld, t2 = std::max(16LL, (long long)k2.tail_splits * m * k2.tail_tiles * kBM);
    double *c1p, *c1s, *t1p, *t1s, *c2p, *c2s, *t2p, *t2s;
    CK(cudaMalloc(&c1p, c1 * 8)); CK(cudaMalloc(&c1s, c1 * 8)); CK(cudaMalloc(&t1p, t1 * 8)); CK(cudaMalloc(&t1s, t1 * 8));
    CK(cudaMalloc(&c2p, c2 * 8)); CK(cudaMalloc(&c2s, c2 * 8)); CK(cudaMalloc(&t2p, t2 * 8)); CK(cudaMalloc(&t2s, t2 * 8));
    for (auto pr : {std::make_pair(c1p, c1), std::make_pair(c1s, c1), std::make_pair(t1p, t1), std::make_pair(t1s, t1),
                    std::make_pair(c2p, c2), std::make_pair(c2s, c2), std::make_pair(t2p, t2), std::make_pair(t2s, t2)})
        CK(cudaMemset(pr.first, 0, pr.second * 8));
    const int mt1 = cdiv(N, kBM), mt2 = cdiv(n, kBM);
    const long long units_max = std::max((long long)mt1 * k1.splits + k1.tail_tiles * k1.tail_splits,
                                         (long long)mt2 * k2.splits + k2.tail_tiles * k2.tail_splits);
    int32_t* side;
    CK(cudaMalloc(&side, split_side_ints(units_max, bn_split) * 4));

    auto params = [&](bool second, bool split_path, double* C, double* T) {
        GemmParams p;
        memset(&p, 0, sizeof(p));
        const Plan& pl = second ? k2 : k1;
        p.C = C;
        p.inv_radix = 1.0 / (double)kRadix;
        p.bn = split_path ? bn_split : bn_pair;
        p.cols = m;
        if (!second) {
            p.ldc = ldy; p.c_split_stride = N * ldy; p.col_scale = cscale; p.rows = (int)N; p.k_total = n;
        } else {
            p.ldc = ld; p.c_split_stride = (long long)m * ld; p.col_scale = dscale; p.rows = n; p.k_total = (int)N; p.trans_out = 1;
        }
        p.k_chunk = pl.chunk;
        const int mt = second ? mt2 : mt1;
        if (pl.tail_tiles > 0) {
            const int groups = 1;  // m <= 128
            p.main_units = groups * (mt * pl.splits - pl.tail_tiles);
            p.tail_units = groups * pl.tail_tiles * pl.tail_splits;
            p.tail_m_tile0 = mt - pl.tail_tiles; p.tail_m_tiles = pl.tail_tiles;
            p.tail_kbase = (pl.splits - 1) * pl.chunk; p.tail_kchunk = pl.tail_chunk;
            const long long row0 = (long long)(mt - pl.tail_tiles) * kBM;
            if (!second) {
                p.tail_C = T - row0 * ldy; p.tail_ldc = ldy; p.tail_split_stride = (long long)pl.tail_tiles * kBM * ldy;
            } else {
                const long long tld = (long long)pl.tail_tiles * kBM;
                p.tail_C = T - row0; p.tail_ldc = tld; p.tail_split_stride = (long long)m * tld;
            }
        }
        return p;
    };
    auto run = [&](bool second, bool split_path, int which, cudaStream_t st) {  // which: 0 both launches, 1 side only, 2 main only
        GemmParams p = second ? params(true, split_path, split_path ? c2s : c2p, split_path ? t2s : t2p)
                              : params(false, split_path, split_path ? c1s : c1p, split_path ? t1s : t1p);
        const Plan& pl = second ? k2 : k1;
        const dim3 grid(split_path ? 1 : cdiv(m, bn_max(S)), second ? mt2 : mt1, pl.splits);
        const CUtensorMap& ma = second ? map_x_k2 : map_x_k1;
        const CUtensorMap& mb = second ? (split_path ? map_y_split : map_y_pair) : (split_path ? map_a_split : map_a_pair);
        if (!split_path) {
            if (second) TRY((launch_oz_gemm<S, false>(ma, mb, p, grid, st)));
            else TRY((launch_oz_gemm<S, true>(ma, mb, p, grid, st)));
        } else if (which == 0) {
            if (second) TRY(launch_oz_gemm_split<false>(ma, mb, p, side, grid, st));
            else TRY(launch_oz_gemm_split<true>(ma, mb, p, side, grid, st));
        } else {
            p.n_tiles = 1; p.n_tile0 = 0;  // (what launch_oz_gemm_split sets)
            if (which == 1) {
                if (second) TRY((launch_oz_gemm_window<S, false, 1, false, 0, kSplitG - 1>(ma, mb, p, side, grid, st)));
                else TRY((launch_oz_gemm_window<S, true, 1, false, 0, kSplitG - 1>(ma, mb, p, side, grid, st)));
            } else {
                if (second) TRY((launch_oz_gemm_window<S, false, 1, false, kSplitG, S - 1>(ma, mb, p, side, grid, st)));
                else TRY((launch_oz_gemm_window<S, true, 1, false, kSplitG, S - 1>(ma, mb, p, side, grid, st)));
            }
        }
        CK(cudaGetLastError());
    };

    // K1 by the pair path -> Y (split partials summed in order), then the Y planes for K2 (as the library makes them)
    run(false, false, 0, 0);
    CK(cudaDeviceSynchronize());
    double* Y;
    CK(cudaMalloc(&Y, N * ldy * 8));
    CK(cudaMemcpy(Y, c1p, N * ldy * 8, cudaMemcpyDeviceToDevice));  // split 0 only: Y needs plausible statistics, not exact sums
    const int slabs = cdiv(N, 512);
    double* ystat;
    CK(cudaMalloc(&ystat, (long long)slabs * 2 * round_up(m, 16) * 8));
    y_stats_kernel<<<dim3(cdiv(m, 32), slabs), dim3(32, 8)>>>(Y, ldy, N, m, 512, ystat, round_up(m, 16));
    y_stats_finish_kernel<<<m, 256>>>(ystat, slabs, round_up(m, 16), m, xscale, colsq, yscale, dscale);
    slice_cols_t_kernel<S><<<dim3((unsigned)cdiv(N, 128), cdiv(m, 32)), dim3(32, 8)>>>(Y, ldy, N, m, yscale, ys, ldk8,
                                                                                     (long long)m * ldk8, (double)kRadix);
    CK(cudaDeviceSynchronize());

    // correctness: every output word of the two paths
    run(false, true, 0, 0);
    run(true, false, 0, 0);
    run(true, true, 0, 0);
    CK(cudaDeviceSynchronize());
    printf("bitwise differences: K1 C %llu / %lld, K1 tail %llu, K2 C %llu / %lld, K2 tail %llu\n", count_diff(c1p, c1s, c1), c1,
           count_diff(t1p, t1s, t1), count_diff(c2p, c2s, c2), c2, count_diff(t2p, t2s, t2));

    // timing: launches alternated, median over the repeats
    cudaEvent_t ev[2];
    CK(cudaEventCreate(&ev[0])); CK(cudaEventCreate(&ev[1]));
    const char* names[8] = {"K1 pair", "K1 split", "K1 side", "K1 main", "K2 pair", "K2 split", "K2 side", "K2 main"};
    std::vector<float> t[8];
    for (int r = 0; r < reps + 2; ++r) {
        for (int c = 0; c < 8; ++c) {
            const bool second = c >= 4, split_path = (c & 3) != 0;
            const int which = (c & 3) == 0 ? 0 : (c & 3) - 1;
            CK(cudaEventRecord(ev[0]));
            run(second, split_path, which, 0);
            CK(cudaEventRecord(ev[1]));
            CK(cudaEventSynchronize(ev[1]));
            float ms = 0;
            CK(cudaEventElapsedTime(&ms, ev[0], ev[1]));
            if (r >= 2) t[c].push_back(ms);
        }
    }
    for (int c = 0; c < 8; ++c) {
        std::sort(t[c].begin(), t[c].end());
        printf("%-9s median %.4f ms  min %.4f  max %.4f\n", names[c], t[c][t[c].size() / 2], t[c].front(), t[c].back());
    }
    const double p1 = t[0][t[0].size() / 2], s1 = t[1][t[1].size() / 2], p2 = t[4][t[4].size() / 2], s2 = t[5][t[5].size() / 2];
    printf("split / pair: K1 %.3f  K2 %.3f  both %.3f\n", s1 / p1, s2 / p2, (s1 + s2) / (p1 + p2));
    return 0;
}
