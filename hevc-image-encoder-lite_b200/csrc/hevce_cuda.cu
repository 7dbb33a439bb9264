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
#include "hevce_internal.h"
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
__global__ void __launch_bounds__(256) hevce_quality_kernel(const Job* __restrict__ jobs, unsigned long long* __restrict__ sse) {
    const Job job = jobs[blockIdx.y];
    const int hm = min(job.src_h, job.H), wm = min(job.src_w, job.W), segs = (wm + 15) / 16;
    unsigned long long acc = 0;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < (long long)hm * segs; t += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(t / segs), x0 = (int)(t % segs) * 16;
        const uint4 rv = *(const uint4*)(job.rcon + (size_t)y * job.W + x0);   // rows of the reconstruction are 32-byte aligned
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
int g_forced_variant = -1;     // hevce_set_variant / HEVCE_VARIANT: -1 = choose per batch
int g_last_variant = 0;

Tables g_host_tables;
std::once_flag g_variants_once;
void variants_init() {
    std::call_once(g_variants_once, [] {
        fill_tables(g_host_tables);
        for (int v = 0; v < NVARIANT; v++) g_variants[v].info(&g_variants[v].vi);
        if (const char* env = getenv("HEVCE_VARIANT"))
            for (int v = 0; v < NVARIANT; v++) if (!strcmp(env, g_variants[v].name)) g_forced_variant = v;
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

template <class T>
int grow(T** p, size_t* cap, size_t need) {   // grow-only device buffer
    if (need <= *cap) return 0;
    if (*p) cudaFree(*p);
    *p = nullptr;
    *cap = 0;
    size_t want = need + need / 8 + 256;
    CK(cudaMalloc((void**)p, want * sizeof(T)));
    *cap = want;
    return 0;
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
    // device buffers (grow-only)
    u8 *d_img = nullptr, *d_rcon = nullptr, *d_out = nullptr;
    size_t c_img = 0, c_rcon = 0, c_out = 0;
    Job* d_jobs = nullptr; size_t c_jobs = 0;
    int* d_order = nullptr; size_t c_order = 0;
    int* d_results = nullptr; size_t c_results = 0;
    int* d_counter = nullptr;
    Scratch* d_slots = nullptr; size_t c_slots = 0;
    s16 *d_glev = nullptr, *d_lev = nullptr; u8 *d_grec = nullptr, *d_line = nullptr;
    size_t c_glev = 0, c_lev = 0, c_grec = 0, c_line = 0;
    CtuRec* d_recs = nullptr; size_t c_recs = 0;
    unsigned long long* d_sse = nullptr; size_t c_sse = 0;
    u8* d_pack = nullptr; size_t c_pack = 0;
    unsigned long long* d_packoff = nullptr; size_t c_packoff = 0;
    float quality_ms = 0.f;
    bool encoded = false;   // hevce_session_encode has run since the last configure/upload
    std::vector<size_t> ctu_off;
    int line_pitch = 0;
    // pinned staging
    u8* h_stage = nullptr; size_t c_stage = 0;
};

// host-side staging copies (user buffers <-> pinned memory) spread over a few threads: at 100 Mpixel/s a single
// thread's memcpy of a 0.8 GB step is a visible part of the end-to-end time
static int g_copy_threads = 0;   // 0 = derive from the host's core count
extern "C" void hevce_internal_set_copy_threads(int n) { g_copy_threads = n; }
extern "C" int hevce_internal_get_device(void) { int d = -1; return cudaGetDevice(&d) == cudaSuccess ? d : -1; }
extern "C" void hevce_internal_set_device(int device) { if (device >= 0) cudaSetDevice(device); }

template <class F>
static void parallel_pictures(int n, size_t total_bytes, F&& fn) {
    // default: the host cores shared by up to four chunk workers per device and by every visible device (one process per GPU
    // or one process for all of them: either way about that many workers copy at the same time)
    static const unsigned auto_threads = [] {
        int nd = 1;
        if (cudaGetDeviceCount(&nd) != cudaSuccess || nd < 1) nd = 1;
        return std::min(4u, std::max(1u, std::thread::hardware_concurrency() / (4u * (unsigned)nd)));
    }();
    unsigned nt = g_copy_threads > 0 ? (unsigned)g_copy_threads : auto_threads;
    if (total_bytes < ((size_t)16 << 20) || n < 2 * (int)nt) nt = 1;
    if (nt == 1) { for (int i = 0; i < n; i++) fn(i); return; }
    std::vector<std::thread> th;
    for (unsigned t = 0; t < nt; t++)
        th.emplace_back([&, t] { for (int i = (int)t; i < n; i += (int)nt) fn(i); });
    for (auto& x : th) x.join();
}

static int stage_reserve(hevce_session* s, size_t need) {
    if (need <= s->c_stage) return 0;
    if (s->h_stage) cudaFreeHost(s->h_stage);
    s->h_stage = nullptr;
    s->c_stage = 0;
    CK(cudaHostAlloc((void**)&s->h_stage, need + need / 8 + 4096, cudaHostAllocDefault));
    s->c_stage = need + need / 8 + 4096;
    return 0;
}

// The variant (index into the variant table) that finishes these pictures soonest on one device by the
// longest-processing-time estimate: makespan over the SMs in CTUs x the variant's measured time per CTU.
static int choose_variant(int sms, const std::vector<Job>& jobs, const std::vector<int>& order) {
    int best = g_forced_variant;
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
    for (int i = 0; i < n; i++) {
        jobs[i].H = (std::min(ysz[i], max_dim) + CTU - 1) / CTU * CTU;
        jobs[i].W = (std::min(xsz[i], max_dim) + CTU - 1) / CTU * CTU;
    }
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
    s->encoded = false;
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
        j.H = (std::min(ysz[i], max_dim) + CTU - 1) / CTU * CTU;     // HEVCe.c:1581-1582
        j.W = (std::min(xsz[i], max_dim) + CTU - 1) / CTU * CTU;
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
    if ((rc = grow(&s->d_img, &s->c_img, io))) return rc;
    if ((rc = grow(&s->d_rcon, &s->c_rcon, ro))) return rc;
    if ((rc = grow(&s->d_out, &s->c_out, oo))) return rc;
    if ((rc = grow(&s->d_jobs, &s->c_jobs, (size_t)n))) return rc;
    if ((rc = grow(&s->d_order, &s->c_order, gangs.size()))) return rc;
    if ((rc = grow(&s->d_results, &s->c_results, (size_t)2 * n))) return rc;
    if (!s->d_counter) CK(cudaMalloc((void**)&s->d_counter, sizeof(int)));
    const size_t g = (size_t)(s->grid / CLV) * GANGV * g_variants[best].vi.tracks, nlev = (size_t)NCAND * LEV_STRIDE + 64, nrec = (size_t)NREC * CTU * CTU;
    s->line_pitch = maxW / 4 + 32;
    if ((rc = grow(&s->d_glev, &s->c_glev, g * nlev))) return rc;
    if ((rc = grow(&s->d_grec, &s->c_grec, g * nrec))) return rc;
    if ((rc = grow(&s->d_lev, &s->c_lev, co * CTU * CTU))) return rc;
    if ((rc = grow(&s->d_recs, &s->c_recs, co))) return rc;
    if ((rc = grow(&s->d_line, &s->c_line, g * (size_t)s->line_pitch))) return rc;
    if ((rc = grow(&s->d_slots, &s->c_slots, g))) return rc;
    std::vector<Scratch> slots(g);
    for (size_t k = 0; k < g; k++) {
        slots[k].glev = s->d_glev + k * nlev;
        slots[k].grec = s->d_grec + k * nrec;
        slots[k].msz_line = s->d_line + k * (size_t)s->line_pitch;
    }
    for (int i = 0; i < n; i++) {
        Job& j = s->jobs[i];
        j.img = s->d_img + s->img_off[i];
        j.rcon = s->d_rcon + s->rcon_off[i];
        j.out = s->d_out + s->out_off[i];
        j.result = s->d_results + 2 * i;
        j.recs = s->d_recs + s->ctu_off[i];
        j.levs = s->d_lev + s->ctu_off[i] * CTU * CTU;
    }
    CK(cudaMemcpyAsync(s->d_slots, slots.data(), g * sizeof(Scratch), cudaMemcpyHostToDevice, s->stream));
    CK(cudaMemcpyAsync(s->d_jobs, s->jobs.data(), (size_t)n * sizeof(Job), cudaMemcpyHostToDevice, s->stream));
    CK(cudaMemcpyAsync(s->d_order, gangs.data(), gangs.size() * sizeof(int), cudaMemcpyHostToDevice, s->stream));
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
    if (s && hevce_session_configure(s, n, ysz, xsz, qpd6, hevce_internal_max_dim(), -1, 0)) { hevce_session_destroy(s); return nullptr; }
    return s;
}

extern "C" int hevce_session_upload(hevce_session* s, const unsigned char* const* imgs) {
    if (!s || (s->n > 0 && !imgs)) return HEVCE_ERR_ARG;
    CK(cudaSetDevice(s->device));
    if (s->n == 0) return 0;
    int rc = stage_reserve(s, s->img_total);
    if (rc) return rc;
    for (int i = 0; i < s->n; i++)
        if (!imgs[i]) return HEVCE_ERR_ARG;
    parallel_pictures(s->n, s->img_total, [&](int i) {
        const Job& j = s->jobs[i];
        memcpy(s->h_stage + s->img_off[i], imgs[i], (size_t)std::min(j.src_h, j.H) * j.src_w);
    });
    CK(cudaMemcpyAsync(s->d_img, s->h_stage, s->img_total, cudaMemcpyHostToDevice, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    s->h2d = (long long)s->img_total;
    s->encoded = false;
    return 0;
}

extern "C" int hevce_session_encode(hevce_session* s) {
    if (!s) return HEVCE_ERR_ARG;
    CK(cudaSetDevice(s->device));
    if (s->n == 0) return 0;
    CK(cudaMemsetAsync(s->d_counter, 0, sizeof(int), s->stream));
    CK(cudaMemsetAsync(s->d_results, 0, 2 * (size_t)s->n * sizeof(int), s->stream));
    CK(cudaEventRecord(s->ev0, s->stream));
    CK((cudaError_t)g_variants[s->variant].launch(s->d_jobs, s->d_order, s->ngangs, s->d_slots, s->d_counter, g_dev[s->device].d_tables, s->grid, s->stream));
    g_last_variant = s->variant;
    CK(cudaEventRecord(s->ev1, s->stream));
    {
        const dim3 grid((unsigned)((s->max_nctu + NTC - 1) / NTC), (unsigned)s->n);
        hevce_commit_kernel<<<grid, NTC, sizeof(CommitShared), s->stream>>>(s->d_jobs, g_dev[s->device].d_tables);
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
    CK(cudaMemcpyAsync(s->results.data(), s->d_results, 2 * (size_t)s->n * sizeof(int), cudaMemcpyDeviceToHost, s->stream));
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
    int rc = stage_reserve(s, s->rcon_total + bytes);
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
    if ((rc = grow(&s->d_pack, &s->c_pack, bytes + 16))) return rc;
    if ((rc = grow(&s->d_packoff, &s->c_packoff, (size_t)s->n))) return rc;
    CK(cudaMemcpyAsync(s->d_packoff, poff.data(), (size_t)s->n * sizeof(unsigned long long), cudaMemcpyHostToDevice, s->stream));
    hevce_pack_kernel<<<s->n, 256, 0, s->stream>>>(s->d_jobs, s->d_packoff, s->d_results, s->d_pack);
    CK(cudaGetLastError());
    s->launches += 1;
    CK(cudaMemcpyAsync(s->h_stage, s->d_rcon, s->rcon_total, cudaMemcpyDeviceToHost, s->stream));
    if (bytes) CK(cudaMemcpyAsync(s->h_stage + s->rcon_total, s->d_pack, bytes, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    off += s->rcon_total;
    parallel_pictures(s->n, off, [&](int i) {
        const Job& j = s->jobs[i];
        memcpy(img_rcons[i], s->h_stage + s->rcon_off[i], (size_t)j.H * j.W);
        memcpy(pbuffers[i], s->h_stage + soff[i], (size_t)s->results[2 * i]);
    });
    s->d2h = (long long)(s->rcon_total + bytes + 2 * (size_t)s->n * sizeof(int));
    return status;
}

// f3: per-picture MSE / PSNR of the last encode, reduced on the device (calcImagePSNR, HEVCeMain.c:116-133)
extern "C" int hevce_session_quality(hevce_session* s, double* mse, double* psnr) {
    if (!s || (s->n > 0 && !mse && !psnr)) return HEVCE_ERR_ARG;
    if (s->n > 0 && !s->encoded) return HEVCE_ERR_STATE;   // nothing has been encoded yet
    CK(cudaSetDevice(s->device));
    if (s->n == 0) return 0;
    int rc = grow(&s->d_sse, &s->c_sse, (size_t)s->n);
    if (rc) return rc;
    CK(cudaMemsetAsync(s->d_sse, 0, (size_t)s->n * sizeof(unsigned long long), s->stream));
    long long maxpix = 0;
    for (const Job& j : s->jobs) maxpix = std::max(maxpix, (long long)j.H * j.W);
    const dim3 grid((unsigned)std::max(1LL, std::min(1024LL, (maxpix / 16 + 255) / 256)), (unsigned)s->n);
    CK(cudaEventRecord(s->ev0, s->stream));
    hevce_quality_kernel<<<grid, 256, 0, s->stream>>>(s->d_jobs, s->d_sse);
    CK(cudaGetLastError());
    CK(cudaEventRecord(s->ev1, s->stream));
    std::vector<unsigned long long> sse((size_t)s->n);
    CK(cudaMemcpyAsync(sse.data(), s->d_sse, sse.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream));
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
extern "C" float hevce_session_quality_ms(const hevce_session* s) { return s ? s->quality_ms : 0.f; }

// Decisions of picture i after hevce_session_encode: CU size and luma intra mode per 4x4 unit ((H/4)*(W/4) bytes each),
// CU kind per 8x8 unit ((H/8)*(W/8) bytes: 0 one TU, 1 four TUs, 2 NxN).  Any pointer may be NULL.
extern "C" int hevce_session_partition(hevce_session* s, int i, unsigned char* cu_size, unsigned char* mode, unsigned char* kind) {
    if (!s || i < 0 || i >= s->n) return HEVCE_ERR_ARG;
    if (!s->encoded) return HEVCE_ERR_STATE;               // nothing has been encoded yet
    CK(cudaSetDevice(s->device));
    const Job& j = s->jobs[i];
    std::vector<CtuRec> recs((size_t)(j.H / CTU) * (j.W / CTU));
    CK(cudaMemcpyAsync(recs.data(), s->d_recs + s->ctu_off[i], recs.size() * sizeof(CtuRec), cudaMemcpyDeviceToHost, s->stream));
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
    if (!name || !*name || !strcmp(name, "auto")) { g_forced_variant = -1; return 0; }
    for (int v = 0; v < NVARIANT; v++)
        if (!strcmp(name, g_variants[v].name)) { g_forced_variant = v; return 0; }
    return HEVCE_ERR_ARG;
}
extern "C" long long hevce_session_h2d_bytes(const hevce_session* s) { return s ? s->h2d : 0; }
extern "C" long long hevce_session_d2h_bytes(const hevce_session* s) { return s ? s->d2h : 0; }

extern "C" void hevce_session_padded_size(const hevce_session* s, int i, int* H, int* W) {
    *H = s->jobs[i].H;
    *W = s->jobs[i].W;
}

extern "C" void hevce_session_destroy(hevce_session* s) {
    if (!s) return;
    cudaSetDevice(s->device);
    cudaFree(s->d_img); cudaFree(s->d_rcon); cudaFree(s->d_out); cudaFree(s->d_jobs); cudaFree(s->d_order);
    cudaFree(s->d_results); cudaFree(s->d_counter); cudaFree(s->d_slots); cudaFree(s->d_glev); cudaFree(s->d_grec);
    cudaFree(s->d_lev); cudaFree(s->d_line); cudaFree(s->d_recs); cudaFree(s->d_sse); cudaFree(s->d_pack); cudaFree(s->d_packoff);
    if (s->h_stage) cudaFreeHost(s->h_stage);
    if (s->ev0) cudaEventDestroy(s->ev0);
    if (s->ev1) cudaEventDestroy(s->ev1);
    if (s->ev2) cudaEventDestroy(s->ev2);
    if (s->stream) cudaStreamDestroy(s->stream);
    delete s;
}

#if defined(HEVCE_PROFILE_DUMP)
extern "C" __attribute__((visibility("default"))) void hevce_profile_dump(void) {
    unsigned long long c[128], n[128];
    g_variants[g_last_variant].profile(c, n);
    printf("variant %s\n", g_variants[g_last_variant].name);
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
