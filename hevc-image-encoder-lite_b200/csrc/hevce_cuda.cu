// hevce_cuda.cu -- sm_100a kernels + device-resident sessions of libhevce_b200.so.
//
// The decision kernel (hevce_core.h: encode_picture) is linked in several variants (hevce_variant.cu, hevce_variants.h):
// gangs of 7 / 4 / 2 pictures per CTA, one "wide" picture per CTA, and one picture per CTA or per cluster of two CTAs
// split into parent || child tracks.  This file picks the variant per batch, owns the
// commit / quality / peak kernels and everything between the plain-C API (hevce_api.c) and the device.
//
// Host side here is the thin layer between the plain-C API (hevce_api.c) and the device: buffer management in HBM,
// pinned staging, launches, CUDA-event timing.  No CPU implementation of any encoder stage exists in this library.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <numeric>
#include <thread>
#include <vector>

#include "../../include/hevce.h"
#include "hevce_core.h"
#include "hevce_deblock.h"
#include "hevce_decode.h"
#include "hevce_internal.h"
#include "hevce_ssim.h"
#include "hevce_variants.h"

using namespace hevce;

#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) {                                                                         \
            fprintf(stderr, "libhevce_b200: %s failed: %s (%s:%d)\n", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            return HEVCE_ERR_CUDA;                                                                       \
        }                                                                                                \
    } while (0)

// ------------------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------------------
// Commit pass: one thread per CTU re-encodes the decided CTU with the byte-writing coder.  blockIdx.y = picture.
__global__ void __launch_bounds__(NTC) hevce_commit_kernel(const Job* __restrict__ jobs, const Tables* __restrict__ tables) {
    CommitShared& cs = my_csm();
    for (int i = threadIdx.x; i < (int)(sizeof(Tables) / 4); i += NTC) ((u32*)&cs.tb)[i] = ((const u32*)tables)[i];
    __syncthreads();
    const Job job = jobs[blockIdx.y];
    const int nctu = (job.H / CTU) * (job.W / CTU), ctu = blockIdx.x * NTC + threadIdx.x;
    if (ctu < nctu) commit_ctu(job, ctu, threadIdx.x);
}

// Stream gather: the streams of a batch lie in per-picture slots of worst-case size; this copies each one to its
// 16-byte-aligned place in one contiguous buffer so the host needs a single device-to-host copy.  blockIdx.x = picture.
__global__ void __launch_bounds__(256) hevce_pack_kernel(const Job* __restrict__ jobs, const unsigned long long* __restrict__ dst_off,
                                                         const int* __restrict__ results, u8* __restrict__ dst) {
    const Job job = jobs[blockIdx.x];
    const int len = min(max(results[2 * blockIdx.x], 0), job.out_cap);
    const uint4* src = (const uint4*)job.out;               // stream slots start at multiples of 256 bytes
    uint4* out = (uint4*)(dst + dst_off[blockIdx.x]);
    for (int i = threadIdx.x; i < (len + 15) / 16; i += blockDim.x) out[i] = src[i];
}

// Quality pass (HEVCeMain.c:116-133): sum of squared differences between source and reconstruction over the area both
// cover.  blockIdx.y = picture, a CTA strides over 16-pixel segments of the reconstruction rows.  HBM-bound: 2 B/pixel.
// `plane` is the picture's H x W plane to compare: its reconstruction, or the decoded picture at the same offset.
__device__ __forceinline__ void quality_sse(const Job& job, const u8* __restrict__ plane, unsigned long long* __restrict__ sse) {
    const int hm = min(job.src_h, job.H), wm = min(job.src_w, job.W), segs = (wm + 15) / 16;
    unsigned long long acc = 0;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < (long long)hm * segs; t += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(t / segs), x0 = (int)(t % segs) * 16;
        const uint4 rv = *(const uint4*)(plane + (size_t)y * job.W + x0);   // rows of the plane are 32-byte aligned
        const u32 rw[4] = {rv.x, rv.y, rv.z, rv.w};
        const u8* ip = job.img + (size_t)y * job.src_w + x0;
        unsigned part = 0;
#pragma unroll
        for (int k = 0; k < 16; k++) {
            if (x0 + k < wm) {
                const int d = (int)ip[k] - (int)((rw[k >> 2] >> (8 * (k & 3))) & 0xffu);
                part += (unsigned)(d * d);
            }
        }
        acc += part;
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(sse + blockIdx.y, acc);
}

__global__ void __launch_bounds__(256) hevce_quality_kernel(const Job* __restrict__ jobs, unsigned long long* __restrict__ sse) {
    const Job job = jobs[blockIdx.y];
    quality_sse(job, job.rcon, sse);
}

// the same over the decoded pictures: dec_base holds each picture at its reconstruction's offset from rcon_base
__global__ void __launch_bounds__(256) hevce_decoded_quality_kernel(const Job* __restrict__ jobs, const u8* rcon_base, const u8* dec_base,
                                                                    unsigned long long* __restrict__ sse) {
    const Job job = jobs[blockIdx.y];
    quality_sse(job, dec_base + (job.rcon - rcon_base), sse);
}

// In-loop deblocking filter (hevce_deblock.h): one CTA per (CTU, picture), blockIdx.y = picture.  Reads the
// reconstructions, writes the decoded pictures to dec_base at the reconstructions' offsets from rcon_base.
__global__ void __launch_bounds__(DBK_THREADS) hevce_deblock_kernel(const Job* __restrict__ jobs, const u8* rcon_base, u8* dec_base) {
    __shared__ DbkTile t;
    const Job job = jobs[blockIdx.y];
    const int ctu = blockIdx.x;
    if (ctu >= dbk_nctu(job)) return;
    for (int i = threadIdx.x; i < DBK_LOAD_ITEMS; i += DBK_THREADS) dbk_load(t, job, ctu, i);
    __syncthreads();
    if (dbk_active(job)) {
        for (int i = threadIdx.x; i < DBK_VERT_ITEMS; i += DBK_THREADS) dbk_vertical(t, job, ctu, i);
        __syncthreads();
        for (int i = threadIdx.x; i < DBK_HORZ_ITEMS; i += DBK_THREADS) dbk_horizontal(t, job, ctu, i);
        __syncthreads();
    }
    u8* dec = dec_base + (job.rcon - rcon_base);
    for (int i = threadIdx.x; i < DBK_STORE_ITEMS; i += DBK_THREADS) dbk_store(t, job, ctu, dec, i);
}

// f7: SSIM (hevce_ssim.h).  One CTA per (32x32 block of window centres, picture), blockIdx.y = picture.  The measured
// plane is at the picture's reconstruction offset from rcon_base in plane_base (rcon_base itself, or the decoded
// pictures); block b's partial goes to partials[b] past the picture's first CTU record, so each picture has its own.
__global__ void __launch_bounds__(SSIM_THREADS) hevce_ssim_kernel(const Job* __restrict__ jobs, const u8* rcon_base, const u8* plane_base,
                                                                  const CtuRec* recs_base, double* __restrict__ partials) {
    __shared__ SsimTile t;
    const Job job = jobs[blockIdx.y];
    const int blk = blockIdx.x;
    if (blk >= ssim_nblk(job)) return;
    const u8* plane = plane_base + (job.rcon - rcon_base);
    for (int i = threadIdx.x; i < SSIM_LOAD_ITEMS; i += SSIM_THREADS) ssim_load(t, job, plane, blk, i);
    __syncthreads();
    for (int i = threadIdx.x; i < SSIM_HSUM_ITEMS; i += SSIM_THREADS) ssim_hsum(t, i);
    __syncthreads();
    t.red[threadIdx.x] = ssim_thread_sum(t, job, blk, threadIdx.x);
    __syncthreads();
    for (int half = SSIM_THREADS / 2; half > 0; half >>= 1) {
        ssim_reduce_step(t, half, threadIdx.x);
        __syncthreads();
    }
    if (threadIdx.x == 0) partials[(job.recs - recs_base) + blk] = t.red[0];
}

// a picture's mean SSIM from its block partials, one thread per picture
__global__ void __launch_bounds__(128) hevce_ssim_mean_kernel(const Job* __restrict__ jobs, int n, const CtuRec* recs_base,
                                                              const double* __restrict__ partials, double* __restrict__ ssim) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Job job = jobs[i];
    ssim[i] = ssim_mean(job, partials + (job.recs - recs_base));
}

// f6, the decoder (hevce_decode.h).  A picture's stream: its bytes, header length (first byte of the slice data), length.
struct DecSrc { const u8* data; int start, len; };

// Parse: the CABAC state threads through a picture's whole slice, so one lane of a warp parses one picture (blockIdx.x).
// Fills the picture's CtuRec partition bytes and its (zeroed) level blocks; status[picture] = DEC_OK or DEC_ERR.
__global__ void __launch_bounds__(32) hevce_parse_kernel(const Job* __restrict__ jobs, const DecSrc* __restrict__ src,
                                                         const Tables* __restrict__ tables, int* __restrict__ status) {
    __shared__ Tables tb;
    for (int i = threadIdx.x; i < (int)(sizeof(Tables) / 4); i += 32) ((u32*)&tb)[i] = ((const u32*)tables)[i];
    __syncthreads();
    if (threadIdx.x == 0) {
        const DecSrc s = src[blockIdx.x];
        status[blockIdx.x] = dec_parse_picture(jobs[blockIdx.x], s.data, s.start, s.len, tb);
    }
}

// Reconstruction: one CTA per picture (blockIdx.x), a CTU-row wavefront.  Warp w takes CTU rows w, w + DEC_WARPS, ...; it
// starts CTU (r, c) once row r - 1 has finished CTU c + 1 (the above-right samples), and the lanes of the warp share the
// phases of each TU (reference samples, filtering: one sample each; columns, then rows of the inverse transform and the
// prediction: one line each).  A picture whose parse failed is written as zeros.
constexpr int DEC_WARPS = 8;
struct DecWarp { DecTuWork w; DecTu tus[64]; int nt; };

__global__ void __launch_bounds__(32 * DEC_WARPS) hevce_recon_kernel(const Job* __restrict__ jobs, const int* __restrict__ status) {
    __shared__ DecWarp ws[DEC_WARPS];
    __shared__ int done[DEC_MAX_DIM / CTU];   // CTUs finished per CTU row
    const Job job = jobs[blockIdx.x];
    const int rows = job.H / CTU, cols = job.W / CTU;
    if (status[blockIdx.x] != DEC_OK) {
        for (size_t i = threadIdx.x; i < (size_t)job.H * job.W / 16; i += blockDim.x) ((uint4*)job.rcon)[i] = make_uint4(0, 0, 0, 0);
        return;
    }
    for (int i = threadIdx.x; i < rows; i += blockDim.x) done[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    DecWarp& s = ws[threadIdx.x >> 5];
    volatile int* vdone = done;
    for (int r = threadIdx.x >> 5; r < rows; r += DEC_WARPS) {
        for (int c = 0; c < cols; c++) {
            if (r > 0 && lane == 0) {
                const int need = min(c + 2, cols);
                while (vdone[r - 1] < need) __nanosleep(32);
                __threadfence_block();
            }
            const int ctu = r * cols + c;
            if (lane == 0) s.nt = dec_tu_list(job.recs[ctu], s.tus);
            __syncwarp();
            const s16* lev = job.levs + (size_t)ctu * (CTU * CTU);
            for (int t = 0; t < s.nt; t++) {
                const DecTu u = s.tus[t];
                const int T = u.s, ty = r * CTU + u.y, tx = c * CTU + u.x;
                for (int j = lane; j < dec_ref_items(T); j += 32) dec_ref_item(s.w, job, ty, tx, T, j);
                __syncwarp();
                if (lane == 0) dec_ref_substitute(s.w, T);
                __syncwarp();
                for (int j = lane; j < dec_ref_items(T); j += 32) dec_filter_item(s.w, T, j);
                if (lane < T) dec_column(s.w, lev + u.y * CTU + u.x, T, job.q, lane);
                __syncwarp();
                if (lane < T) dec_row(s.w, job, ty, tx, T, u.m, lane);
                __syncwarp();
            }
            if (lane == 0) {
                __threadfence_block();
                vdone[r] = c + 1;
            }
        }
    }
}

// integer-issue micro-benchmark: 8 independent IMAD chains + 8 independent LOP3/IADD3 chains per thread
__global__ void __launch_bounds__(256) hevce_int_peak_kernel(int iters, int seed, int* sink) {
    int a[8], b[8];
#pragma unroll
    for (int i = 0; i < 8; i++) { a[i] = seed + i * 7 + threadIdx.x; b[i] = seed * 3 + i + blockIdx.x; }
    const int m = seed | 1, c = seed + 11;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 8; i++) {
            a[i] = a[i] * m + c;            // IMAD  (fma pipe)
            b[i] = (b[i] ^ c) + a[i];       // LOP3 + IADD3 (alu pipe)
        }
    }
    int r = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) r ^= a[i] ^ b[i];
    if (r == 0x7fffffff) sink[0] = r;
}

// ------------------------------------------------------------------------------------------------------------
// per-device state
// ------------------------------------------------------------------------------------------------------------
namespace {

struct Variant {
    const char* name;
    int (*prepare)(void);
    int (*launch)(const void*, const int*, int, const void*, int*, const void*, int, void*);
    void (*info)(hevce_variant_info*);
    void (*profile)(unsigned long long*, unsigned long long*);
    hevce_variant_info vi;
    double cost;   // relative time per CTU of one gang when the whole GPU runs this variant (HEVCE_VARIANT_LIST)
};
#if defined(HEVCE_PROFILE_DUMP)
#define HEVCE_VARIANT_ROW(tag, cost) {#tag, hevce_variant_prepare_##tag, hevce_variant_launch_##tag, hevce_variant_info_##tag, hevce_variant_profile_##tag, {}, cost},
#else
#define HEVCE_VARIANT_ROW(tag, cost) {#tag, hevce_variant_prepare_##tag, hevce_variant_launch_##tag, hevce_variant_info_##tag, nullptr, {}, cost},
#endif
Variant g_variants[] = {HEVCE_VARIANT_LIST(HEVCE_VARIANT_ROW)};
constexpr int NVARIANT = (int)(sizeof(g_variants) / sizeof(g_variants[0]));
// set and read by any caller thread; relaxed, as no other data is published through them
std::atomic<int> g_forced_variant{-1};   // hevce_set_variant / HEVCE_VARIANT: -1 = choose per batch
std::atomic<int> g_last_variant{0};

Tables g_host_tables;
std::once_flag g_variants_once;
void variants_init() {
    std::call_once(g_variants_once, [] {
        fill_tables(g_host_tables);
        for (int v = 0; v < NVARIANT; v++) g_variants[v].info(&g_variants[v].vi);
        if (const char* env = getenv("HEVCE_VARIANT"))
            for (int v = 0; v < NVARIANT; v++) if (!strcmp(env, g_variants[v].name)) g_forced_variant.store(v, std::memory_order_relaxed);
    });
}

struct DeviceInfo {
    bool ready = false;
    int sms = 0;
    Tables* d_tables = nullptr;
};
std::mutex g_dev_mutex;
DeviceInfo g_dev[64];

int device_prepare(int device) {
    std::lock_guard<std::mutex> lk(g_dev_mutex);
    if (device < 0 || device >= 64) return HEVCE_ERR_ARG;
    CK(cudaSetDevice(device));
    if (g_dev[device].ready) return 0;
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10 || prop.minor != 0) {   // the cubins are sm_100a: they load on compute capability 10.0 only
        fprintf(stderr, "libhevce_b200: device %d is sm_%d%d; this library is built for sm_100a only\n", device, prop.major, prop.minor);
        return HEVCE_ERR_CUDA;
    }
    variants_init();
    for (int v = 0; v < NVARIANT; v++) CK((cudaError_t)g_variants[v].prepare());
    CK(cudaMalloc((void**)&g_dev[device].d_tables, sizeof(Tables)));
    CK(cudaMemcpy(g_dev[device].d_tables, &g_host_tables, sizeof(Tables), cudaMemcpyHostToDevice));
    g_dev[device].sms = prop.multiProcessorCount;
    g_dev[device].ready = true;
    return 0;
}

// Work units of a batch for a variant with `gang` pictures per CTA: same-size pictures in order of decreasing size,
// -1 in the empty slots of a short gang.  Returns the longest-processing-time-first makespan over `bins` CTAs in CTUs.
long long build_gangs(const std::vector<Job>& jobs, const std::vector<int>& order, int gang, int bins, std::vector<int>* out) {
    const int n = (int)order.size();
    std::vector<long long> load((size_t)std::max(1, bins), 0);   // min-heap by load
    auto cmp = [](long long a, long long b) { return a > b; };
    long long makespan = 0;
    if (out) out->clear();
    for (int i = 0; i < n;) {
        const Job& f = jobs[order[i]];
        int m = 1;
        while (m < gang && i + m < n && jobs[order[i + m]].H == f.H && jobs[order[i + m]].W == f.W) m++;
        if (out)
            for (int k = 0; k < gang; k++) out->push_back(k < m ? order[i + k] : -1);
        std::pop_heap(load.begin(), load.end(), cmp);
        load.back() += (long long)(f.H / CTU) * (f.W / CTU);
        makespan = std::max(makespan, load.back());
        std::push_heap(load.begin(), load.end(), cmp);
        i += m;
    }
    return makespan;
}

// Grow-only buffer of T in device memory, or in pinned host memory: a larger request frees the old allocation first, then
// allocates need + need/8 + slack elements.  The buffer frees itself; its owner selects the device before it goes.
template <class T, bool Pinned = false>
struct GrowBuffer {
    T* p = nullptr;
    size_t cap = 0;
    GrowBuffer() = default;
    GrowBuffer(const GrowBuffer&) = delete;
    GrowBuffer& operator=(const GrowBuffer&) = delete;
    ~GrowBuffer() { release(); }
    void release() {
        if (p) Pinned ? cudaFreeHost(p) : cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    int reserve(size_t need) {
        if (need <= cap) return 0;
        release();
        const size_t want = need + need / 8 + (Pinned ? 4096 : 256);
        CK(Pinned ? cudaHostAlloc((void**)&p, want * sizeof(T), cudaHostAllocDefault) : cudaMalloc((void**)&p, want * sizeof(T)));
        cap = want;
        return 0;
    }
};

// the reference's clamp and padding of a picture (HEVCe.c:1581-1582)
void set_padded_size(Job& j, int ysz, int xsz, int max_dim) {
    j.H = (std::min(ysz, max_dim) + CTU - 1) / CTU * CTU;
    j.W = (std::min(xsz, max_dim) + CTU - 1) / CTU * CTU;
}

}   // namespace

struct hevce_session {
    int device = 0, n = 0, grid = 0, launches = 0, ngangs = 0, variant = 0;
    float kernel_ms = 0.f, commit_ms = 0.f;
    int max_nctu = 0;
    long long h2d = 0, d2h = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;
    std::vector<Job> jobs;
    std::vector<size_t> img_off, rcon_off, out_off;
    std::vector<int> order, results;
    size_t img_total = 0, rcon_total = 0, out_total = 0;
    GrowBuffer<u8> d_img, d_rcon, d_out, d_grec, d_line, d_pack;
    GrowBuffer<Job> d_jobs;
    GrowBuffer<int> d_order, d_results, d_counter;
    GrowBuffer<Scratch> d_slots;
    GrowBuffer<s16> d_glev, d_lev;
    GrowBuffer<CtuRec> d_recs;
    GrowBuffer<unsigned long long> d_sse, d_packoff;
    float quality_ms = 0.f, deblock_ms = 0.f;
    bool encoded = false;   // hevce_session_encode has run since the last configure/upload
    bool deblocked = false; // hevce_session_deblock has run since the last configure/upload/encode
    GrowBuffer<u8> d_dec;   // decoded pictures at the offsets of d_rcon; reserved by the first hevce_session_deblock
    GrowBuffer<double> d_ssim_part, d_ssim;   // SSIM block partials at the CTU offsets, per-picture means
    float ssim_ms = 0.f;
    std::vector<size_t> ctu_off;
    int line_pitch = 0;
    GrowBuffer<u8, true> h_stage;   // pinned staging
};

extern "C" int hevce_internal_get_device(void) { int d = -1; return cudaGetDevice(&d) == cudaSuccess ? d : -1; }
extern "C" void hevce_internal_set_device(int device) { if (device >= 0) cudaSetDevice(device); }

// host-side staging copies (user buffers <-> pinned memory) spread over a few threads: at 100 Mpixel/s a single
// thread's memcpy of a 0.8 GB step is a visible part of the end-to-end time
template <class F>
static void parallel_pictures(int n, size_t total_bytes, F&& fn) {
    // the host cores shared by up to four chunk workers per device and by every visible device (one process per GPU
    // or one process for all of them: either way about that many workers copy at the same time)
    static const unsigned auto_threads = [] {
        int nd = 1;
        if (cudaGetDeviceCount(&nd) != cudaSuccess || nd < 1) nd = 1;
        return std::min(4u, std::max(1u, std::thread::hardware_concurrency() / (4u * (unsigned)nd)));
    }();
    unsigned nt = auto_threads;
    if (total_bytes < ((size_t)16 << 20) || n < 2 * (int)nt) nt = 1;
    if (nt == 1) { for (int i = 0; i < n; i++) fn(i); return; }
    std::vector<std::thread> th;
    for (unsigned t = 0; t < nt; t++)
        th.emplace_back([&, t] { for (int i = (int)t; i < n; i += (int)nt) fn(i); });
    for (auto& x : th) x.join();
}

// The variant (index into the variant table) that finishes these pictures soonest on one device by the
// longest-processing-time estimate: makespan over the SMs in CTUs x the variant's measured time per CTU.
static int choose_variant(int sms, const std::vector<Job>& jobs, const std::vector<int>& order) {
    int best = g_forced_variant.load(std::memory_order_relaxed);
    if (best >= 0) return best;
    double best_t = 0;
    for (int v = 0; v < NVARIANT; v++) {
        const double t = (double)build_gangs(jobs, order, g_variants[v].vi.gang, sms / g_variants[v].vi.cluster, nullptr) * g_variants[v].cost;
        if (best < 0 || t < best_t) { best = v; best_t = t; }
    }
    return best;
}

static void size_order(const std::vector<Job>& jobs, std::vector<int>& order) {   // largest pictures first, same sizes adjacent
    order.resize(jobs.size());
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
        const Job &x = jobs[a], &y = jobs[b];
        const long long ax = (long long)x.H * x.W, ay = (long long)y.H * y.W;
        if (ax != ay) return ax > ay;
        if (x.H != y.H) return x.H > y.H;
        return false;
    });
}

// For a caller that cuts one device's pictures into several chunks that run at the same time (hevce_api.c): the
// variant is chosen for ALL of them together, then forced on every chunk's session.  returns a variant index or < 0.
extern "C" int hevce_internal_choose_variant(int device, int n, const int* ysz, const int* xsz, int max_dim) {
    if (device_prepare(device) || n <= 0) return -1;
    std::vector<Job> jobs((size_t)n);
    for (int i = 0; i < n; i++) set_padded_size(jobs[i], ysz[i], xsz[i], max_dim);
    std::vector<int> order;
    size_order(jobs, order);
    return choose_variant(g_dev[device].sms, jobs, order);
}

extern "C" int hevce_internal_device_sms(int device) { return device_prepare(device) ? 0 : g_dev[device].sms; }

// variant < 0: choose for this batch; max_ctas > 0: the launch uses at most that many CTAs (a chunk that shares the device
// with other chunks' kernels)
extern "C" int hevce_session_configure(hevce_session* s, int n, const int* ysz, const int* xsz, const int* qpd6, int max_dim, int variant, int max_ctas) {
    if (!s || n < 0 || n > 65535 || (n > 0 && (!ysz || !xsz || !qpd6))) return HEVCE_ERR_ARG;   // grid.y of the commit kernel = picture index
    int rc = device_prepare(s->device);
    if (rc) return rc;
    s->encoded = s->deblocked = false;
    s->n = n;
    s->jobs.assign(n, Job());
    s->img_off.assign(n, 0); s->rcon_off.assign(n, 0); s->out_off.assign(n, 0); s->ctu_off.assign(n, 0);
    size_t co = 0;
    s->max_nctu = 0;
    size_t io = 0, ro = 0, oo = 0;
    int maxW = CTU;
    for (int i = 0; i < n; i++) {
        if (ysz[i] <= 0 || xsz[i] <= 0 || qpd6[i] < 0 || qpd6[i] > 4) return HEVCE_ERR_ARG;
        Job& j = s->jobs[i];
        j.src_h = ysz[i]; j.src_w = xsz[i];
        set_padded_size(j, ysz[i], xsz[i], max_dim);
        j.q = qpd6[i];
        j.out_cap = 256 + 2 * j.H * j.W;
        s->img_off[i] = io; s->rcon_off[i] = ro; s->out_off[i] = oo; s->ctu_off[i] = co;
        co += (size_t)(j.H / CTU) * (j.W / CTU);
        s->max_nctu = std::max(s->max_nctu, (j.H / CTU) * (j.W / CTU));
        // only the rows/columns the encoder can touch are transferred (a picture larger than the clamp is cropped)
        io += ((size_t)std::min(j.src_h, j.H) * j.src_w + 255) & ~(size_t)255;
        ro += (size_t)j.H * j.W;
        oo += ((size_t)j.out_cap + 255) & ~(size_t)255;
        maxW = std::max(maxW, j.W);
    }
    s->img_total = io; s->rcon_total = ro; s->out_total = oo;
    if (n == 0) return 0;
    // work units: gangs of same-size pictures, largest pictures first; the variant (pictures per CTA) that finishes the
    // batch soonest by the longest-processing-time estimate: makespan in CTUs x the variant's time per CTU
    size_order(s->jobs, s->order);
    const DeviceInfo& di = g_dev[s->device];
    const int best = (variant >= 0 && variant < NVARIANT) ? variant : choose_variant(di.sms, s->jobs, s->order);
    s->variant = best;
    const int GANGV = g_variants[best].vi.gang;
    std::vector<int> gangs;
    const int CLV = g_variants[best].vi.cluster;          // CTAs per gang
    build_gangs(s->jobs, s->order, GANGV, di.sms / CLV, &gangs);
    s->ngangs = (int)gangs.size() / GANGV;
    s->grid = std::min(s->ngangs, std::max(1, (max_ctas > 0 ? std::min(max_ctas, di.sms) : di.sms) / CLV)) * CLV;
    if ((rc = s->d_img.reserve(io))) return rc;
    if ((rc = s->d_rcon.reserve(ro))) return rc;
    if ((rc = s->d_out.reserve(oo))) return rc;
    if ((rc = s->d_jobs.reserve((size_t)n))) return rc;
    if ((rc = s->d_order.reserve(gangs.size()))) return rc;
    if ((rc = s->d_results.reserve((size_t)2 * n))) return rc;
    if ((rc = s->d_counter.reserve(1))) return rc;
    const size_t g = (size_t)(s->grid / CLV) * GANGV * g_variants[best].vi.tracks, nlev = (size_t)NCAND * LEV_STRIDE + 64, nrec = (size_t)NREC * CTU * CTU;
    s->line_pitch = maxW / 4 + 32;
    if ((rc = s->d_glev.reserve(g * nlev))) return rc;
    if ((rc = s->d_grec.reserve(g * nrec))) return rc;
    if ((rc = s->d_lev.reserve(co * CTU * CTU))) return rc;
    if ((rc = s->d_recs.reserve(co))) return rc;
    if ((rc = s->d_line.reserve(g * (size_t)s->line_pitch))) return rc;
    if ((rc = s->d_slots.reserve(g))) return rc;
    std::vector<Scratch> slots(g);
    for (size_t k = 0; k < g; k++) {
        slots[k].glev = s->d_glev.p + k * nlev;
        slots[k].grec = s->d_grec.p + k * nrec;
        slots[k].msz_line = s->d_line.p + k * (size_t)s->line_pitch;
    }
    for (int i = 0; i < n; i++) {
        Job& j = s->jobs[i];
        j.img = s->d_img.p + s->img_off[i];
        j.rcon = s->d_rcon.p + s->rcon_off[i];
        j.out = s->d_out.p + s->out_off[i];
        j.result = s->d_results.p + 2 * i;
        j.recs = s->d_recs.p + s->ctu_off[i];
        j.levs = s->d_lev.p + s->ctu_off[i] * CTU * CTU;
    }
    CK(cudaMemcpyAsync(s->d_slots.p, slots.data(), g * sizeof(Scratch), cudaMemcpyHostToDevice, s->stream));
    CK(cudaMemcpyAsync(s->d_jobs.p, s->jobs.data(), (size_t)n * sizeof(Job), cudaMemcpyHostToDevice, s->stream));
    CK(cudaMemcpyAsync(s->d_order.p, gangs.data(), gangs.size() * sizeof(int), cudaMemcpyHostToDevice, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    return 0;
}

extern "C" hevce_session* hevce_session_create_empty(int device) {
    if (device_prepare(device)) return nullptr;
    hevce_session* s = new hevce_session;
    s->device = device;
    if (cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreate(&s->ev0) != cudaSuccess ||
        cudaEventCreate(&s->ev1) != cudaSuccess || cudaEventCreate(&s->ev2) != cudaSuccess) {
        fprintf(stderr, "libhevce_b200: cannot create stream/events on device %d\n", device);
        hevce_session_destroy(s);
        return nullptr;
    }
    return s;
}

extern "C" hevce_session* hevce_session_create(int device, int n, const int* ysz, const int* xsz, const int* qpd6) {
    hevce_session* s = hevce_session_create_empty(device);
    if (s && hevce_session_configure(s, n, ysz, xsz, qpd6, hevce_get_max_dim(), -1, 0)) { hevce_session_destroy(s); return nullptr; }
    return s;
}

extern "C" int hevce_session_upload(hevce_session* s, const unsigned char* const* imgs) {
    if (!s || (s->n > 0 && !imgs)) return HEVCE_ERR_ARG;
    CK(cudaSetDevice(s->device));
    if (s->n == 0) return 0;
    int rc = s->h_stage.reserve(s->img_total);
    if (rc) return rc;
    for (int i = 0; i < s->n; i++)
        if (!imgs[i]) return HEVCE_ERR_ARG;
    parallel_pictures(s->n, s->img_total, [&](int i) {
        const Job& j = s->jobs[i];
        memcpy(s->h_stage.p + s->img_off[i], imgs[i], (size_t)std::min(j.src_h, j.H) * j.src_w);
    });
    CK(cudaMemcpyAsync(s->d_img.p, s->h_stage.p, s->img_total, cudaMemcpyHostToDevice, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    s->h2d = (long long)s->img_total;
    s->encoded = s->deblocked = false;
    return 0;
}

extern "C" int hevce_session_encode(hevce_session* s) {
    if (!s) return HEVCE_ERR_ARG;
    s->deblocked = false;
    CK(cudaSetDevice(s->device));
    if (s->n == 0) return 0;
    CK(cudaMemsetAsync(s->d_counter.p, 0, sizeof(int), s->stream));
    CK(cudaMemsetAsync(s->d_results.p, 0, 2 * (size_t)s->n * sizeof(int), s->stream));
    CK(cudaEventRecord(s->ev0, s->stream));
    CK((cudaError_t)g_variants[s->variant].launch(s->d_jobs.p, s->d_order.p, s->ngangs, s->d_slots.p, s->d_counter.p, g_dev[s->device].d_tables, s->grid, s->stream));
    g_last_variant.store(s->variant, std::memory_order_relaxed);
    CK(cudaEventRecord(s->ev1, s->stream));
    {
        const dim3 grid((unsigned)((s->max_nctu + NTC - 1) / NTC), (unsigned)s->n);
        hevce_commit_kernel<<<grid, NTC, sizeof(CommitShared), s->stream>>>(s->d_jobs.p, g_dev[s->device].d_tables);
        CK(cudaGetLastError());
    }
    CK(cudaEventRecord(s->ev2, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    CK(cudaEventElapsedTime(&s->kernel_ms, s->ev0, s->ev1));
    CK(cudaEventElapsedTime(&s->commit_ms, s->ev1, s->ev2));
    s->launches += 2;
    s->encoded = true;
    return 0;
}

extern "C" int hevce_session_download(hevce_session* s, unsigned char* const* pbuffers, unsigned char* const* img_rcons, int* stream_len) {
    if (!s || (s->n > 0 && (!pbuffers || !img_rcons))) return HEVCE_ERR_ARG;
    CK(cudaSetDevice(s->device));
    if (s->n == 0) return 0;
    s->results.resize(2 * (size_t)s->n);
    CK(cudaMemcpyAsync(s->results.data(), s->d_results.p, 2 * (size_t)s->n * sizeof(int), cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    size_t bytes = 0;
    int status = 0;
    for (int i = 0; i < s->n; i++) {
        if (s->results[2 * i + 1] != 0 || s->results[2 * i] < 0 || s->results[2 * i] > s->jobs[i].out_cap) {
            fprintf(stderr, "libhevce_b200: picture %d failed its consistency check (flags %d, len %d)\n", i, s->results[2 * i + 1], s->results[2 * i]);
            status = HEVCE_ERR_STATE;
            s->results[2 * i] = 0;
        }
        bytes += ((size_t)s->results[2 * i] + 15) & ~(size_t)15;
    }
    int rc = s->h_stage.reserve(s->rcon_total + bytes);
    if (rc) return rc;
    // gather the streams on the device (hevce_pack_kernel), then one copy per direction: reconstructions, streams
    std::vector<unsigned long long> poff((size_t)s->n);
    std::vector<size_t> soff((size_t)s->n);
    size_t off = 0;
    for (int i = 0; i < s->n; i++) {
        if (!pbuffers[i] || !img_rcons[i]) return HEVCE_ERR_ARG;
        poff[i] = off;
        soff[i] = s->rcon_total + off;
        off += ((size_t)s->results[2 * i] + 15) & ~(size_t)15;
        if (stream_len) stream_len[i] = s->results[2 * i];
    }
    if ((rc = s->d_pack.reserve(bytes + 16))) return rc;
    if ((rc = s->d_packoff.reserve((size_t)s->n))) return rc;
    CK(cudaMemcpyAsync(s->d_packoff.p, poff.data(), (size_t)s->n * sizeof(unsigned long long), cudaMemcpyHostToDevice, s->stream));
    hevce_pack_kernel<<<s->n, 256, 0, s->stream>>>(s->d_jobs.p, s->d_packoff.p, s->d_results.p, s->d_pack.p);
    CK(cudaGetLastError());
    s->launches += 1;
    CK(cudaMemcpyAsync(s->h_stage.p, s->d_rcon.p, s->rcon_total, cudaMemcpyDeviceToHost, s->stream));
    if (bytes) CK(cudaMemcpyAsync(s->h_stage.p + s->rcon_total, s->d_pack.p, bytes, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    off += s->rcon_total;
    parallel_pictures(s->n, off, [&](int i) {
        const Job& j = s->jobs[i];
        memcpy(img_rcons[i], s->h_stage.p + s->rcon_off[i], (size_t)j.H * j.W);
        memcpy(pbuffers[i], s->h_stage.p + soff[i], (size_t)s->results[2 * i]);
    });
    s->d2h = (long long)(s->rcon_total + bytes + 2 * (size_t)s->n * sizeof(int));
    return status;
}

// f3: per-picture MSE / PSNR against the source, reduced on the device (calcImagePSNR, HEVCeMain.c:116-133), of the
// reconstructions or (decoded) of the decoded pictures
static int session_quality(hevce_session* s, bool decoded, double* mse, double* psnr) {
    CK(cudaSetDevice(s->device));
    if (s->n == 0) return 0;
    int rc = s->d_sse.reserve((size_t)s->n);
    if (rc) return rc;
    CK(cudaMemsetAsync(s->d_sse.p, 0, (size_t)s->n * sizeof(unsigned long long), s->stream));
    long long maxpix = 0;
    for (const Job& j : s->jobs) maxpix = std::max(maxpix, (long long)j.H * j.W);
    const dim3 grid((unsigned)std::max(1LL, std::min(1024LL, (maxpix / 16 + 255) / 256)), (unsigned)s->n);
    CK(cudaEventRecord(s->ev0, s->stream));
    if (decoded) hevce_decoded_quality_kernel<<<grid, 256, 0, s->stream>>>(s->d_jobs.p, s->d_rcon.p, s->d_dec.p, s->d_sse.p);
    else hevce_quality_kernel<<<grid, 256, 0, s->stream>>>(s->d_jobs.p, s->d_sse.p);
    CK(cudaGetLastError());
    CK(cudaEventRecord(s->ev1, s->stream));
    std::vector<unsigned long long> sse((size_t)s->n);
    CK(cudaMemcpyAsync(sse.data(), s->d_sse.p, sse.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    CK(cudaEventElapsedTime(&s->quality_ms, s->ev0, s->ev1));
    s->launches += 1;
    for (int i = 0; i < s->n; i++) {
        const Job& j = s->jobs[i];
        double m = (double)sse[i] / std::min(j.src_h, j.H) / std::min(j.src_w, j.W);
        if (m < 1e-9) m = 1e-9;
        if (mse) mse[i] = m;
        if (psnr) psnr[i] = 10.0 * log10(255 * 255 / m);
    }
    return 0;
}

extern "C" int hevce_session_quality(hevce_session* s, double* mse, double* psnr) {
    if (!s || (s->n > 0 && !mse && !psnr)) return HEVCE_ERR_ARG;
    if (s->n > 0 && !s->encoded) return HEVCE_ERR_STATE;   // nothing has been encoded yet
    return session_quality(s, false, mse, psnr);
}
extern "C" float hevce_session_quality_ms(const hevce_session* s) { return s ? s->quality_ms : 0.f; }

// f5: the decoded pictures of the last encode -- the reconstructions after the in-loop deblocking filter
extern "C" int hevce_session_deblock(hevce_session* s) {
    if (!s) return HEVCE_ERR_ARG;
    if (s->n > 0 && !s->encoded) return HEVCE_ERR_STATE;   // nothing has been encoded yet
    CK(cudaSetDevice(s->device));
    if (s->n > 0) {
        int rc = s->d_dec.reserve(s->rcon_total);
        if (rc) return rc;
        CK(cudaEventRecord(s->ev0, s->stream));
        hevce_deblock_kernel<<<dim3((unsigned)s->max_nctu, (unsigned)s->n), DBK_THREADS, 0, s->stream>>>(s->d_jobs.p, s->d_rcon.p, s->d_dec.p);
        CK(cudaGetLastError());
        CK(cudaEventRecord(s->ev1, s->stream));
        CK(cudaStreamSynchronize(s->stream));
        CK(cudaEventElapsedTime(&s->deblock_ms, s->ev0, s->ev1));
        s->launches += 1;
    }
    s->deblocked = true;
    return 0;
}
extern "C" float hevce_session_deblock_ms(const hevce_session* s) { return s ? s->deblock_ms : 0.f; }

extern "C" int hevce_session_download_decoded(hevce_session* s, unsigned char* const* img_decs) {
    if (!s || (s->n > 0 && !img_decs)) return HEVCE_ERR_ARG;
    if (s->n > 0 && !s->deblocked) return HEVCE_ERR_STATE;
    CK(cudaSetDevice(s->device));
    if (s->n == 0) return 0;
    for (int i = 0; i < s->n; i++)
        if (!img_decs[i]) return HEVCE_ERR_ARG;
    int rc = s->h_stage.reserve(s->rcon_total);
    if (rc) return rc;
    CK(cudaMemcpyAsync(s->h_stage.p, s->d_dec.p, s->rcon_total, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    parallel_pictures(s->n, s->rcon_total, [&](int i) {
        const Job& j = s->jobs[i];
        memcpy(img_decs[i], s->h_stage.p + s->rcon_off[i], (size_t)j.H * j.W);
    });
    return 0;
}

extern "C" int hevce_session_decoded_quality(hevce_session* s, double* mse, double* psnr) {
    if (!s || (s->n > 0 && !mse && !psnr)) return HEVCE_ERR_ARG;
    if (s->n > 0 && !s->deblocked) return HEVCE_ERR_STATE;
    return session_quality(s, true, mse, psnr);
}

// f7: per-picture mean SSIM (hevce_ssim.h) between the coded picture and the reconstruction or (decoded) the decoded
// picture, at the padded size
extern "C" int hevce_session_ssim(hevce_session* s, int decoded, double* ssim) {
    if (!s || (decoded != 0 && decoded != 1) || (s->n > 0 && !ssim)) return HEVCE_ERR_ARG;
    if (s->n > 0 && !(decoded ? s->deblocked : s->encoded)) return HEVCE_ERR_STATE;
    CK(cudaSetDevice(s->device));
    if (s->n == 0) return 0;
    const Job& last = s->jobs[s->n - 1];
    int rc = s->d_ssim_part.reserve(s->ctu_off[s->n - 1] + (size_t)ssim_nblk(last));
    if (!rc) rc = s->d_ssim.reserve((size_t)s->n);
    if (rc) return rc;
    CK(cudaEventRecord(s->ev0, s->stream));
    hevce_ssim_kernel<<<dim3((unsigned)s->max_nctu, (unsigned)s->n), SSIM_THREADS, 0, s->stream>>>(
        s->d_jobs.p, s->d_rcon.p, decoded ? s->d_dec.p : s->d_rcon.p, s->d_recs.p, s->d_ssim_part.p);
    CK(cudaGetLastError());
    hevce_ssim_mean_kernel<<<(s->n + 127) / 128, 128, 0, s->stream>>>(s->d_jobs.p, s->n, s->d_recs.p, s->d_ssim_part.p, s->d_ssim.p);
    CK(cudaGetLastError());
    CK(cudaEventRecord(s->ev1, s->stream));
    CK(cudaMemcpyAsync(ssim, s->d_ssim.p, (size_t)s->n * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    CK(cudaEventElapsedTime(&s->ssim_ms, s->ev0, s->ev1));
    s->launches += 2;
    return 0;
}
extern "C" float hevce_session_ssim_ms(const hevce_session* s) { return s ? s->ssim_ms : 0.f; }

// Decisions of picture i after hevce_session_encode: CU size and luma intra mode per 4x4 unit ((H/4)*(W/4) bytes each),
// CU kind per 8x8 unit ((H/8)*(W/8) bytes: 0 one TU, 1 four TUs, 2 NxN).  Any pointer may be NULL.
extern "C" int hevce_session_partition(hevce_session* s, int i, unsigned char* cu_size, unsigned char* mode, unsigned char* kind) {
    if (!s || i < 0 || i >= s->n) return HEVCE_ERR_ARG;
    if (!s->encoded) return HEVCE_ERR_STATE;               // nothing has been encoded yet
    CK(cudaSetDevice(s->device));
    const Job& j = s->jobs[i];
    std::vector<CtuRec> recs((size_t)(j.H / CTU) * (j.W / CTU));
    CK(cudaMemcpyAsync(recs.data(), s->d_recs.p + s->ctu_off[i], recs.size() * sizeof(CtuRec), cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    unpack_partition(recs.data(), j.H, j.W, cu_size, mode, kind);
    return 0;
}

extern "C" float hevce_session_kernel_ms(const hevce_session* s) { return s ? s->kernel_ms : 0.f; }
extern "C" float hevce_session_commit_ms(const hevce_session* s) { return s ? s->commit_ms : 0.f; }
extern "C" int hevce_session_launches(const hevce_session* s) { return s ? s->launches : 0; }
extern "C" int hevce_session_grid(const hevce_session* s) { return s ? s->grid : 0; }
extern "C" const char* hevce_session_variant(const hevce_session* s) { return s ? g_variants[s->variant].name : ""; }

// Kernel variant used for the batches configured from now on: a tag of HEVCE_VARIANT_LIST, or NULL / "" / "auto" to
// choose per batch.  returns 0, or HEVCE_ERR_ARG for an unknown name.
extern "C" int hevce_set_variant(const char* name) {
    variants_init();
    if (!name || !*name || !strcmp(name, "auto")) { g_forced_variant.store(-1, std::memory_order_relaxed); return 0; }
    for (int v = 0; v < NVARIANT; v++)
        if (!strcmp(name, g_variants[v].name)) { g_forced_variant.store(v, std::memory_order_relaxed); return 0; }
    return HEVCE_ERR_ARG;
}
extern "C" long long hevce_session_h2d_bytes(const hevce_session* s) { return s ? s->h2d : 0; }
extern "C" long long hevce_session_d2h_bytes(const hevce_session* s) { return s ? s->d2h : 0; }

extern "C" void hevce_session_destroy(hevce_session* s) {
    if (!s) return;
    cudaSetDevice(s->device);
    if (s->ev0) cudaEventDestroy(s->ev0);
    if (s->ev1) cudaEventDestroy(s->ev1);
    if (s->ev2) cudaEventDestroy(s->ev2);
    if (s->stream) cudaStreamDestroy(s->stream);
    delete s;
}

// ------------------------------------------------------------------------------------------------------------
// f6: the decoder -- streams of this library back to decoded pictures, separate from the encoder's sessions
// ------------------------------------------------------------------------------------------------------------
extern "C" int hevce_stream_info(const unsigned char* stream, int len, int* ysz, int* xsz, int* qpd6) {
    int H, W, q;
    if (!stream || len <= 0 || dec_header(stream, len, H, W, q) < 0) return HEVCE_ERR_ARG;
    if (ysz) *ysz = H;
    if (xsz) *xsz = W;
    if (qpd6) *qpd6 = q;
    return 0;
}

struct hevce_decoder {
    int device = 0, n = 0, max_nctu = 0;
    bool ran = false;                 // hevce_decoder_run has run since the last upload
    float parse_ms = 0.f, recon_ms = 0.f, deblock_ms = 0.f;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    std::vector<Job> jobs;
    std::vector<DecSrc> src;
    std::vector<size_t> pix_off;
    std::vector<int> status;
    size_t pix_total = 0;
    GrowBuffer<u8> d_bits, d_rcon, d_dec;
    GrowBuffer<Job> d_jobs;
    GrowBuffer<DecSrc> d_src;
    GrowBuffer<int> d_status;
    GrowBuffer<CtuRec> d_recs;
    GrowBuffer<s16> d_levs;
    GrowBuffer<u8, true> h_stage;     // pinned staging
};

extern "C" void hevce_decoder_destroy(hevce_decoder* d) {
    if (!d) return;
    cudaSetDevice(d->device);
    for (cudaEvent_t e : d->ev) if (e) cudaEventDestroy(e);
    if (d->stream) cudaStreamDestroy(d->stream);
    delete d;
}

extern "C" hevce_decoder* hevce_decoder_create(int device) {
    if (device_prepare(device)) return nullptr;
    hevce_decoder* d = new hevce_decoder;
    d->device = device;
    bool ok = cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking) == cudaSuccess;
    for (cudaEvent_t& e : d->ev) ok = ok && cudaEventCreate(&e) == cudaSuccess;
    if (!ok) {
        fprintf(stderr, "libhevce_b200: cannot create stream/events on device %d\n", device);
        hevce_decoder_destroy(d);
        return nullptr;
    }
    return d;
}

// n streams -> device: every header is checked first (HEVCE_ERR_ARG, nothing changed), then the streams go up as one copy
extern "C" int hevce_decoder_upload(hevce_decoder* d, int n, const unsigned char* const* streams, const int* stream_len) {
    if (!d || n < 0 || n > 65535 || (n > 0 && (!streams || !stream_len))) return HEVCE_ERR_ARG;   // grid.y of the deblocking kernel
    std::vector<Job> jobs((size_t)n);
    std::vector<DecSrc> src((size_t)n);
    std::vector<size_t> pix_off((size_t)n), bit_off((size_t)n), ctu_off((size_t)n);
    size_t pix = 0, bits = 0, ctus = 0;
    int max_nctu = 0;
    for (int i = 0; i < n; i++) {
        Job& j = jobs[i];
        memset(&j, 0, sizeof(Job));
        if (!streams[i] || stream_len[i] <= 0 || (src[i].start = dec_header(streams[i], stream_len[i], j.H, j.W, j.q)) < 0) return HEVCE_ERR_ARG;
        src[i].len = stream_len[i];
        j.src_h = j.H; j.src_w = j.W;
        pix_off[i] = pix; bit_off[i] = bits; ctu_off[i] = ctus;
        pix += (size_t)j.H * j.W;
        bits += ((size_t)stream_len[i] + 15) & ~(size_t)15;
        ctus += (size_t)(j.H / CTU) * (j.W / CTU);
        max_nctu = std::max(max_nctu, (j.H / CTU) * (j.W / CTU));
    }
    CK(cudaSetDevice(d->device));
    d->ran = false;
    d->n = n;
    if (n == 0) return 0;
    int rc;
    if ((rc = d->h_stage.reserve(bits))) return rc;
    if ((rc = d->d_bits.reserve(bits))) return rc;
    if ((rc = d->d_rcon.reserve(pix))) return rc;
    if ((rc = d->d_dec.reserve(pix))) return rc;
    if ((rc = d->d_jobs.reserve((size_t)n))) return rc;
    if ((rc = d->d_src.reserve((size_t)n))) return rc;
    if ((rc = d->d_status.reserve((size_t)n))) return rc;
    if ((rc = d->d_recs.reserve(ctus))) return rc;
    if ((rc = d->d_levs.reserve(ctus * CTU * CTU))) return rc;
    parallel_pictures(n, bits, [&](int i) { memcpy(d->h_stage.p + bit_off[i], streams[i], (size_t)stream_len[i]); });
    for (int i = 0; i < n; i++) {
        jobs[i].rcon = d->d_rcon.p + pix_off[i];
        jobs[i].recs = d->d_recs.p + ctu_off[i];
        jobs[i].levs = d->d_levs.p + ctu_off[i] * CTU * CTU;
        src[i].data = d->d_bits.p + bit_off[i];
    }
    CK(cudaMemcpyAsync(d->d_bits.p, d->h_stage.p, bits, cudaMemcpyHostToDevice, d->stream));
    CK(cudaMemcpyAsync(d->d_jobs.p, jobs.data(), (size_t)n * sizeof(Job), cudaMemcpyHostToDevice, d->stream));
    CK(cudaMemcpyAsync(d->d_src.p, src.data(), (size_t)n * sizeof(DecSrc), cudaMemcpyHostToDevice, d->stream));
    CK(cudaStreamSynchronize(d->stream));
    d->jobs.swap(jobs);
    d->src.swap(src);
    d->pix_off.swap(pix_off);
    d->pix_total = pix;
    d->max_nctu = max_nctu;
    return 0;
}

// parse + reconstruction + deblocking of the uploaded streams, synchronous
extern "C" int hevce_decoder_run(hevce_decoder* d) {
    if (!d) return HEVCE_ERR_ARG;
    CK(cudaSetDevice(d->device));
    if (d->n > 0) {
        size_t ctus = 0;
        for (const Job& j : d->jobs) ctus += (size_t)(j.H / CTU) * (j.W / CTU);
        CK(cudaMemsetAsync(d->d_levs.p, 0, ctus * CTU * CTU * sizeof(s16), d->stream));   // the parser writes non-zero levels only
        CK(cudaEventRecord(d->ev[0], d->stream));
        hevce_parse_kernel<<<d->n, 32, 0, d->stream>>>(d->d_jobs.p, d->d_src.p, g_dev[d->device].d_tables, d->d_status.p);
        CK(cudaGetLastError());
        CK(cudaEventRecord(d->ev[1], d->stream));
        hevce_recon_kernel<<<d->n, 32 * DEC_WARPS, 0, d->stream>>>(d->d_jobs.p, d->d_status.p);
        CK(cudaGetLastError());
        CK(cudaEventRecord(d->ev[2], d->stream));
        hevce_deblock_kernel<<<dim3((unsigned)d->max_nctu, (unsigned)d->n), DBK_THREADS, 0, d->stream>>>(d->d_jobs.p, d->d_rcon.p, d->d_dec.p);
        CK(cudaGetLastError());
        CK(cudaEventRecord(d->ev[3], d->stream));
        CK(cudaStreamSynchronize(d->stream));
        CK(cudaEventElapsedTime(&d->parse_ms, d->ev[0], d->ev[1]));
        CK(cudaEventElapsedTime(&d->recon_ms, d->ev[1], d->ev[2]));
        CK(cudaEventElapsedTime(&d->deblock_ms, d->ev[2], d->ev[3]));
    }
    d->ran = true;
    return 0;
}

// decoded pictures -> host (one copy); status[i] (may be NULL) = 0 or HEVCE_ERR_STATE.  Returns HEVCE_ERR_STATE when a
// picture's slice data did not parse (its buffer then holds zeros); the other pictures are decoded all the same.
extern "C" int hevce_decoder_download(hevce_decoder* d, unsigned char* const* img_decs, int* status) {
    if (!d || (d->n > 0 && !img_decs)) return HEVCE_ERR_ARG;
    if (d->n > 0 && !d->ran) return HEVCE_ERR_STATE;
    CK(cudaSetDevice(d->device));
    if (d->n == 0) return 0;
    for (int i = 0; i < d->n; i++)
        if (!img_decs[i]) return HEVCE_ERR_ARG;
    int rc = d->h_stage.reserve(d->pix_total);
    if (rc) return rc;
    d->status.resize((size_t)d->n);
    CK(cudaMemcpyAsync(d->status.data(), d->d_status.p, (size_t)d->n * sizeof(int), cudaMemcpyDeviceToHost, d->stream));
    CK(cudaMemcpyAsync(d->h_stage.p, d->d_dec.p, d->pix_total, cudaMemcpyDeviceToHost, d->stream));
    CK(cudaStreamSynchronize(d->stream));
    parallel_pictures(d->n, d->pix_total, [&](int i) {
        const Job& j = d->jobs[i];
        memcpy(img_decs[i], d->h_stage.p + d->pix_off[i], (size_t)j.H * j.W);
    });
    int ret = 0;
    for (int i = 0; i < d->n; i++) {
        if (status) status[i] = d->status[i] == DEC_OK ? 0 : HEVCE_ERR_STATE;
        if (d->status[i] != DEC_OK) ret = HEVCE_ERR_STATE;
    }
    return ret;
}

extern "C" float hevce_decoder_parse_ms(const hevce_decoder* d) { return d ? d->parse_ms : 0.f; }
extern "C" float hevce_decoder_recon_ms(const hevce_decoder* d) { return d ? d->recon_ms : 0.f; }
extern "C" float hevce_decoder_deblock_ms(const hevce_decoder* d) { return d ? d->deblock_ms : 0.f; }

#if defined(HEVCE_PROFILE_DUMP)
extern "C" __attribute__((visibility("default"))) void hevce_profile_dump(void) {
    unsigned long long c[128], n[128];
    const Variant& last = g_variants[g_last_variant.load(std::memory_order_relaxed)];
    last.profile(c, n);
    printf("variant %s\n", last.name);
    static const char* names[] = {"border", "A", "B", "C", "D+pu/trial", "pu_argmin", "trial(S>8)", "decide", "adopt", "enter", "load", "commit", "misc", "teamA/round", "teamB pixel", "teamB d+cabac", "teamB argmin"};
    unsigned long long tot = 0;
    for (int i = 0; i < P_TA; i++) tot += c[i];   // team tags overlap "D+pu/trial" of the 8x8 nodes
    for (int i = 0; i < P_NTAGS; i++)
        printf("phase %-12s count %10llu cycles %14llu  %5.1f%%  avg %8.0f\n", names[i], n[i], c[i], 100.0 * c[i] / (double)tot, n[i] ? (double)c[i] / n[i] : 0.0);
    for (int sz = 0; sz < 3; sz++)
        for (int w = 0; w < 32; w++)
            if (n[24 + 32 * sz + w] && c[24 + 32 * sz + w] / n[24 + 32 * sz + w] > 1000) printf("%dx%d trial pass, warp %2d: avg %8.0f cycles\n", 8 << sz, 8 << sz, w, (double)c[24 + 32 * sz + w] / n[24 + 32 * sz + w]);
}
#endif

extern "C" int hevce_internal_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

extern "C" double hevce_measure_int_peak(int device) {
    if (device_prepare(device)) return (double)HEVCE_ERR_CUDA;
    int* sink = nullptr;
    if (cudaMalloc((void**)&sink, sizeof(int)) != cudaSuccess) return (double)HEVCE_ERR_CUDA;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    const int iters = 1 << 14, blocks = g_dev[device].sms * 8, threads = 256;
    double best = 0;
    for (int rep = 0; rep < 5; rep++) {
        cudaEventRecord(e0);
        hevce_int_peak_kernel<<<blocks, threads>>>(iters, 12345 + rep, sink);
        cudaEventRecord(e1);
        if (cudaEventSynchronize(e1) != cudaSuccess) { best = (double)HEVCE_ERR_CUDA; break; }
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        // per iteration and thread: 8 IMAD (2 ops each) + 8 LOP3 + 8 IADD3
        const double ops = (double)blocks * threads * iters * (8 * 2 + 8 + 8);
        if (rep > 0) best = std::max(best, ops / (ms * 1e-3));
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    return best;
}
