// hevce_simssim.cpp -- host build of the SSIM kernels' source (TEST INFRASTRUCTURE ONLY).
//
// Runs the functions of csrc/hevce_ssim.h in one thread, as hevce_ssim_kernel and hevce_ssim_mean_kernel schedule them:
// every CTA of the grid (block, picture), in each CTA every work item of a phase before the next phase (load, hsum),
// then the 256 threads' centre sums, the reduction tree level by level, and the block partial; then every picture's mean
// from its partials.  With order = 1 the blocks of a picture run last to first, and the items of the load and hsum phases
// too: a bit-identical result shows they are independent.
#include <cstring>
#include <vector>

#include "hevce_core.h"
#include "hevce_ssim.h"

using namespace hevce;

// n pictures: srcs[i] (src_h[i] x src_w[i], stride src_w[i]) coded at the padded size H[i] x W[i], planes[i] (H x W).
// ssim[i] receives the mean SSIM.  Returns 0, or -1 for a padded size that is not a positive multiple of 32.
extern "C" int hevce_simssim(int n, const u8* const* srcs, const int* src_h, const int* src_w, const u8* const* planes, const int* H,
                             const int* W, double* ssim, int order) {
    std::vector<Job> jobs((size_t)n);
    std::vector<size_t> first((size_t)n);
    size_t nblk = 0;
    for (int i = 0; i < n; i++) {
        if (H[i] <= 0 || W[i] <= 0 || H[i] % CTU || W[i] % CTU) return -1;
        Job& j = jobs[i];
        memset(&j, 0, sizeof(Job));
        j.img = srcs[i]; j.src_h = src_h[i]; j.src_w = src_w[i];
        j.H = H[i]; j.W = W[i];
        first[i] = nblk;
        nblk += (size_t)ssim_nblk(j);
    }
    std::vector<double> partials(nblk, -1.0);
    auto item = [&](int i, int count) { return order ? count - 1 - i : i; };
    SsimTile t;
    for (int pic = 0; pic < n; pic++) {                      // blockIdx.y
        const Job& job = jobs[pic];
        for (int b = 0; b < ssim_nblk(job); b++) {           // blockIdx.x
            const int blk = item(b, ssim_nblk(job));
            memset(&t, 0x5A, sizeof(t));                     // shared memory starts with whatever was there
            for (int i = 0; i < SSIM_LOAD_ITEMS; i++) ssim_load(t, job, planes[pic], blk, item(i, SSIM_LOAD_ITEMS));
            for (int i = 0; i < SSIM_HSUM_ITEMS; i++) ssim_hsum(t, item(i, SSIM_HSUM_ITEMS));
            for (int tid = 0; tid < SSIM_THREADS; tid++) t.red[tid] = ssim_thread_sum(t, job, blk, tid);
            for (int half = SSIM_THREADS / 2; half > 0; half >>= 1)
                for (int tid = 0; tid < SSIM_THREADS; tid++) ssim_reduce_step(t, half, tid);
            partials[first[pic] + blk] = t.red[0];
        }
    }
    for (int pic = 0; pic < n; pic++) ssim[pic] = ssim_mean(jobs[pic], partials.data() + first[pic]);
    return 0;
}
