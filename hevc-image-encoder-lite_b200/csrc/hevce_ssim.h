// hevce_ssim.h -- mean SSIM of a picture, with scikit-image's defaults as HEVCeval.py uses them: uniform 7x7 window,
// sample covariance (N / (N - 1)), K1 = 0.01, K2 = 0.03, data_range = 256, mean over the (H-6) x (W-6) window centres
// whose window lies inside the picture.
//
// It compares two H x W planes at the padded size: the coded picture -- the sample the encoder reads at each padded
// position, src[min(y, src_h - 1)][min(x, src_w - 1)] (the load of encode_picture in hevce_core.h) -- and the plane
// being measured (the reconstruction or the decoded picture).  hevce_cuda.cu runs these functions in hevce_ssim_kernel
// and hevce_ssim_mean_kernel; tests/sim/hevce_simssim.cpp runs the same source on the host.
//
// One CTA covers one 32x32 block of window centres, block b of a picture at the place of CTU b: centres
// (y0 + 3 + r, x0 + 3 + c), 0 <= r, c < 32.  Since H and W are multiples of 32, the picture's (H/32) x (W/32) blocks
// hold all its centres.
//   load     38 x 38 samples of both planes from (y0, x0); samples outside the picture are 0 and reach no valid centre;
//   hsum     per tile row and centre column, the horizontal 7-sums of a, b, a^2, b^2 and ab: exact integers
//            (at most 7 * 255^2 before the vertical pass, 49 * 255^2 after);
//   centre   thread t takes centre column t % 32 and rows 4 (t / 32) .. 4 (t / 32) + 3: it slides the vertical 7-sums
//            of the hsums down the column and adds the four centres' SSIM, evaluated in fp64 from the exact sums, in
//            row order;
//   reduce   the threads' sums are added by a fixed tree, and the block writes one fp64 partial.
// hevce_ssim_mean_kernel adds a picture's partials in block order.  No step depends on the grid, the batch or timing,
// so a picture's SSIM is bit-identical however it is batched, chunked or sharded.
#pragma once
#include "hevce_core.h"

namespace HEVCE_NS {

constexpr int SSIM_THREADS = 256;
constexpr int SSIM_WIN = 7;
constexpr int SSIM_TS = CTU + SSIM_WIN - 1;           // tile side: 32 centres + 6 samples of window
constexpr int SSIM_LOAD_ITEMS = SSIM_TS * SSIM_TS;    // one sample of both planes
constexpr int SSIM_HSUM_ITEMS = SSIM_TS * CTU;        // tile row x centre column
constexpr int SSIM_ROWS = CTU * CTU / SSIM_THREADS;  // centre rows per thread

struct SsimTile {
    u8 a[SSIM_TS * SSIM_TS];          // coded picture, a[r * SSIM_TS + c] = sample (y0 + r, x0 + c)
    u8 b[SSIM_TS * SSIM_TS];          // measured plane
    int h[5][SSIM_TS * CTU];          // horizontal 7-sums of a, b, a^2, b^2, ab over columns c .. c+6 of tile row r
    double red[SSIM_THREADS];         // per-thread sums for the block reduction
};

HEVCE_HD inline int ssim_nblk(const Job& job) { return (job.H / CTU) * (job.W / CTU); }

// plane: the picture's H x W plane to measure; job.img / src_h / src_w give the coded picture
HEVCE_HD inline void ssim_load(SsimTile& t, const Job& job, const u8* plane, int blk, int item) {
    const int cw = job.W / CTU, y = (blk / cw) * CTU + item / SSIM_TS, x = (blk % cw) * CTU + item % SSIM_TS;
    const bool in = y < job.H && x < job.W;
    t.a[item] = in ? job.img[(size_t)imin(y, job.src_h - 1) * job.src_w + imin(x, job.src_w - 1)] : (u8)0;
    t.b[item] = in ? plane[(size_t)y * job.W + x] : (u8)0;
}

HEVCE_HD inline void ssim_hsum(SsimTile& t, int item) {
    const int r = item / CTU, c = item % CTU;
    int sa = 0, sb = 0, saa = 0, sbb = 0, sab = 0;
    for (int k = 0; k < SSIM_WIN; k++) {
        const int a = t.a[r * SSIM_TS + c + k], b = t.b[r * SSIM_TS + c + k];
        sa += a; sb += b; saa += a * a; sbb += b * b; sab += a * b;
    }
    t.h[0][item] = sa; t.h[1][item] = sb; t.h[2][item] = saa; t.h[3][item] = sbb; t.h[4][item] = sab;
}

// SSIM of one centre from its window sums s = {Sa, Sb, Saa, Sbb, Sab}.  With N = 49 samples, the means are S/N and the
// sample (co)variances (N Sxy - Sx Sy) / (N (N-1)); multiplying numerator and denominator of SSIM by N^2 (first factor)
// and N (N-1) (second factor) leaves integer terms that are exact in int64, so identical planes give exactly 1.
HEVCE_HD inline double ssim_of_sums(const int (&s)[5]) {
    const long long N = SSIM_WIN * SSIM_WIN, ab = (long long)s[0] * s[1], a2b2 = (long long)s[0] * s[0] + (long long)s[1] * s[1];
    const double C1 = 6.5536 * (double)(N * N), C2 = 58.9824 * (double)(N * (N - 1));   // (0.01 * 256)^2, (0.03 * 256)^2
    const double num = ((double)(2 * ab) + C1) * ((double)(2 * (N * s[4] - ab)) + C2);
    const double den = ((double)a2b2 + C1) * ((double)(N * ((long long)s[2] + s[3]) - a2b2) + C2);
    return num / den;
}

// thread tid's sum over its centres (column tid % 32, rows SSIM_ROWS * (tid / 32) ..), in row order; a centre whose
// window leaves the picture adds nothing
HEVCE_HD inline double ssim_thread_sum(const SsimTile& t, const Job& job, int blk, int tid) {
    const int cw = job.W / CTU, c = tid % CTU, r0 = (tid / CTU) * SSIM_ROWS;
    const int rows_in = job.H - (SSIM_WIN - 1) - (blk / cw) * CTU, cols_in = job.W - (SSIM_WIN - 1) - (blk % cw) * CTU;
    int s[5] = {0, 0, 0, 0, 0};
    for (int k = 0; k < SSIM_WIN - 1; k++)
        for (int v = 0; v < 5; v++) s[v] += t.h[v][(r0 + k) * CTU + c];
    double acc = 0.0;
    for (int r = r0; r < r0 + SSIM_ROWS; r++) {
        for (int v = 0; v < 5; v++) s[v] += t.h[v][(r + SSIM_WIN - 1) * CTU + c];
        if (r < rows_in && c < cols_in) acc += ssim_of_sums(s);
        for (int v = 0; v < 5; v++) s[v] -= t.h[v][r * CTU + c];
    }
    return acc;
}

// one level of the block reduction: threads tid < half add red[tid + half]; half = 128, 64, .., 1 leaves the sum in red[0]
HEVCE_HD inline void ssim_reduce_step(SsimTile& t, int half, int tid) {
    if (tid < half) t.red[tid] += t.red[tid + half];
}

// the picture's mean from its block partials, added in block order
HEVCE_HD inline double ssim_mean(const Job& job, const double* partials) {
    double acc = 0.0;
    for (int b = 0; b < ssim_nblk(job); b++) acc += partials[b];
    return acc / ((double)(job.H - (SSIM_WIN - 1)) * (double)(job.W - (SSIM_WIN - 1)));
}

}   // namespace HEVCE_NS
