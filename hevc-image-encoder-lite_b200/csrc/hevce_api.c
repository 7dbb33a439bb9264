/*
 * hevce_api.c -- the C API of libhevce_b200.so: plain C host code over the CUDA layer (hevce_cuda.cu).
 *
 *   HEVCImageEncoder       drop-in for the reference entry point (HEVCe.h:5-12, HEVCe.c:1570-1647)
 *   HEVCImageEncoderBatch  n independent pictures, sharded over the selected GPUs by cumulative CTU count,
 *                          no collective (SURVEY.md section 8e)
 *   HEVCImageEncoderBatchDecoded  the same, plus every picture after the in-loop deblocking filter
 *   HEVCImageEncoderBatchTarget   each picture at the coarsest qpd6 whose decoded picture meets a quality target
 *   HEVCImageDecoderBatch  streams of this library back to decoded pictures, sharded the same way
 *
 * A shard (the pictures of one device) is cut into chunks; same-size pictures run as rounds of four chunks on four host
 * threads, each with its own session (stream + pinned staging) and its kernel on a quarter of the SMs, so the
 * host<->device copies of one chunk overlap the kernels of the others.
 *
 * There is no CPU encoder in this library: every picture is encoded by the sm_100a kernels; if no CUDA device can be
 * used the calls fail with HEVCE_ERR_CUDA.
 */
#include <errno.h>
#include <math.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "hevce_internal.h"

#define API __attribute__((visibility("default")))

/* Only HEVCImageEncoderBatchDecoded reaches these two.  Weak references let this file link with a CUDA layer that does not
   define them, such as the CPU stand-in of the chunk-planner test; in libhevce_b200.so hevce_cuda.cu defines both. */
#pragma weak hevce_session_deblock
#pragma weak hevce_session_download_decoded
/* ... and only HEVCImageEncoderBatchTarget these two (it returns HEVCE_ERR_STATE without the ones its metric needs). */
#pragma weak hevce_session_ssim
#pragma weak hevce_session_decoded_quality
/* The same for the decoder (HEVCImageDecoderBatch returns HEVCE_ERR_STATE without them). */
#pragma weak hevce_stream_info
#pragma weak hevce_decoder_create
#pragma weak hevce_decoder_upload
#pragma weak hevce_decoder_run
#pragma weak hevce_decoder_download
#pragma weak hevce_decoder_destroy
#define MAX_DEV 64
#define POOL_PER_DEV 4                        /* cached sessions (grow-only buffers) per device ordinal */
#define CHUNK_PIXELS (768LL * 1024 * 1024)    /* per-chunk bound (padded pixels) so the pinned staging stays modest */
#define CHUNK_PICTURES 32768                  /* ... and pictures (the commit kernel's grid.y is the picture index) */
#define G7_GANG 7                             /* pictures per CTA of the g7 variant */
#define WAVE_PICTURES (148 * G7_GANG)         /* pictures of one full wave of g7 on a B200 */
#define MAX_WORKERS 4                         /* chunk workers per device (= cached sessions per device) */

static pthread_mutex_t g_lock = PTHREAD_MUTEX_INITIALIZER;   /* device list + session pool */
static int g_ndev = -1, g_devs[MAX_DEV];
static int g_max_dim = 8192;
static hevce_session *g_pool[MAX_DEV][POOL_PER_DEV];
static int g_pool_busy[MAX_DEV][POOL_PER_DEV];
static hevce_decoder *g_dec[MAX_DEV];   /* one cached decoder per device ordinal */
static int g_dec_busy[MAX_DEV];

API const char *hevce_version(void) { return "hevce-b200 0.2 (sm_100a)"; }

API int hevce_get_max_dim(void) { return __atomic_load_n(&g_max_dim, __ATOMIC_RELAXED); }

API int hevce_set_max_dim(int max_dim) {
    int old = hevce_get_max_dim();
    if (max_dim >= 32 && max_dim <= 16384) __atomic_store_n(&g_max_dim, max_dim, __ATOMIC_RELAXED);
    return old;
}

/* HEVCE_DEVICES="0,3": every entry must be a visible ordinal; anything else is an error (nothing is cached) */
static int resolve_devices(void) {   /* call with g_lock held; returns the device count or a negative HEVCE_ERR_* */
    int visible, i;
    if (g_ndev >= 0) return g_ndev;
    visible = hevce_internal_device_count();
    {
        const char *env = getenv("HEVCE_DEVICES");
        if (env && *env) {
            int devs[MAX_DEV], nd = 0;
            const char *p = env;
            while (*p) {
                char *end;
                long d;
                errno = 0;
                d = strtol(p, &end, 10);
                if (end == p || errno || d < 0 || d >= visible || nd >= MAX_DEV || (*end && *end != ',')) {
                    fprintf(stderr, "libhevce_b200: HEVCE_DEVICES=\"%s\" is not a list of visible device ordinals (%d visible)\n", env, visible);
                    return visible ? HEVCE_ERR_ARG : HEVCE_ERR_CUDA;
                }
                devs[nd++] = (int)d;
                p = *end ? end + 1 : end;
            }
            if (nd == 0) return HEVCE_ERR_ARG;
            memcpy(g_devs, devs, sizeof(int) * (size_t)nd);
            g_ndev = nd;
            return g_ndev;
        }
    }
    g_ndev = 0;
    for (i = 0; i < visible && i < MAX_DEV; i++) g_devs[g_ndev++] = i;
    return g_ndev;
}

API int hevce_set_devices(int count, const int *ordinals) {
    int i, visible = hevce_internal_device_count();
    if (count < 1 || count > MAX_DEV || !ordinals) return HEVCE_ERR_ARG;
    for (i = 0; i < count; i++)
        if (ordinals[i] < 0 || ordinals[i] >= visible) return visible ? HEVCE_ERR_ARG : HEVCE_ERR_CUDA;
    pthread_mutex_lock(&g_lock);
    g_ndev = count;
    for (i = 0; i < count; i++) g_devs[i] = ordinals[i];
    pthread_mutex_unlock(&g_lock);
    return 0;
}

/* ---- session pool: concurrent callers (and the chunk workers of a shard) get a session each -------------------- */
static hevce_session *pool_acquire(int device, int *slot) {
    int k;
    hevce_session *s = NULL;
    *slot = -1;
    pthread_mutex_lock(&g_lock);
    for (k = 0; k < POOL_PER_DEV && *slot < 0; k++)
        if (!g_pool_busy[device][k] && g_pool[device][k]) *slot = k;
    for (k = 0; k < POOL_PER_DEV && *slot < 0; k++)
        if (!g_pool_busy[device][k]) *slot = k;
    if (*slot >= 0) { g_pool_busy[device][*slot] = 1; s = g_pool[device][*slot]; }
    pthread_mutex_unlock(&g_lock);
    if (!s) {   /* an empty pool slot, or every pooled session is busy (then the session is temporary) */
        s = hevce_session_create_empty(device);
        if (*slot >= 0) {
            pthread_mutex_lock(&g_lock);
            if (s) g_pool[device][*slot] = s;
            else g_pool_busy[device][*slot] = 0;   /* creation failed: the slot is free again */
            pthread_mutex_unlock(&g_lock);
            if (!s) *slot = -1;
        }
    }
    return s;
}

static void pool_release(int device, int slot, hevce_session *s) {
    if (slot < 0) { hevce_session_destroy(s); return; }
    pthread_mutex_lock(&g_lock);
    g_pool_busy[device][slot] = 0;
    pthread_mutex_unlock(&g_lock);
}

/* Free the cached sessions (HBM buffers, pinned staging) of every device.  Sessions in use by a running call stay. */
API void hevce_release(void) {
    int d, k;
    for (d = 0; d < MAX_DEV; d++)
        for (k = 0; k < POOL_PER_DEV; k++) {
            hevce_session *s = NULL;
            pthread_mutex_lock(&g_lock);
            if (!g_pool_busy[d][k]) { s = g_pool[d][k]; g_pool[d][k] = NULL; }
            pthread_mutex_unlock(&g_lock);
            if (s) hevce_session_destroy(s);
        }
    for (d = 0; d < MAX_DEV; d++) {
        hevce_decoder *dec = NULL;
        pthread_mutex_lock(&g_lock);
        if (!g_dec_busy[d]) { dec = g_dec[d]; g_dec[d] = NULL; }
        pthread_mutex_unlock(&g_lock);
        if (dec) hevce_decoder_destroy(dec);
    }
}

typedef struct {
    int device, first, count, status, max_dim, variant, max_ctas;
    unsigned char *const *pbuffers;
    const unsigned char *const *imgs;
    unsigned char *const *rcons;
    unsigned char *const *decs;   /* decoded pictures, or NULL: HEVCImageEncoderBatch */
    const int *ysz, *xsz, *qpd6;
    int *stream_len;
    int metric;                   /* HEVCE_METRIC_* of quality */
    double *quality;              /* decoded pictures' quality, or NULL: only HEVCImageEncoderBatchTarget asks for it */
    /* chunk queue shared by the shard's workers */
    int nchunk, next_chunk;
    int *chunk_first;   /* nchunk + 1 entries; a chunk holds at least one picture, so count + 1 are allocated */
    pthread_mutex_t qlock;
} Shard;

/* the reference's clamp and padding of one picture dimension (HEVCe.c:1581-1582) */
static int padded_dim(int v, int max_dim) { return ((v < max_dim ? v : max_dim) + 31) / 32 * 32; }

static long long padded_pixels(int h, int w, int max_dim) { return (long long)padded_dim(h, max_dim) * padded_dim(w, max_dim); }

/* worker: encode chunks of the shard until the queue is empty */
static void *chunk_worker(void *arg) {
    Shard *sh = (Shard *)arg;
    int slot;
    hevce_session *s = pool_acquire(sh->device, &slot);
    if (!s) {
        pthread_mutex_lock(&sh->qlock);
        if (!sh->status) sh->status = HEVCE_ERR_CUDA;
        pthread_mutex_unlock(&sh->qlock);
        return NULL;
    }
    for (;;) {
        int c, a, m, rc;
        pthread_mutex_lock(&sh->qlock);
        c = sh->status ? sh->nchunk : sh->next_chunk++;
        pthread_mutex_unlock(&sh->qlock);
        if (c >= sh->nchunk) break;
        a = sh->chunk_first[c];
        m = sh->chunk_first[c + 1] - a;
        rc = hevce_session_configure(s, m, sh->ysz + a, sh->xsz + a, sh->qpd6 + a, sh->max_dim, sh->variant, sh->max_ctas);
        if (!rc) rc = hevce_session_upload(s, sh->imgs + a);
        if (!rc) rc = hevce_session_encode(s);
        if (!rc) rc = hevce_session_download(s, sh->pbuffers + a, sh->rcons + a, sh->stream_len + a);
        if (!rc && (sh->decs || sh->quality)) rc = hevce_session_deblock(s);
        if (!rc && sh->quality)
            rc = sh->metric == HEVCE_METRIC_SSIM ? hevce_session_ssim(s, 1, sh->quality + a) : hevce_session_decoded_quality(s, NULL, sh->quality + a);
        if (!rc && sh->decs) rc = hevce_session_download_decoded(s, sh->decs + a);
        if (rc) {
            pthread_mutex_lock(&sh->qlock);
            if (!sh->status) sh->status = rc;
            pthread_mutex_unlock(&sh->qlock);
        }
    }
    pool_release(sh->device, slot, s);
    return NULL;
}

/* Cut the shard into chunks: fills chunk_first, nchunk and max_ctas, returns the number of chunk workers. */
static int plan_chunks(Shard *sh) {
    const int *ys = sh->ysz + sh->first, *xs = sh->xsz + sh->first;
    int done = 0, i, same = 1;
    for (i = 1; i < sh->count && same; i++)
        if (ys[i] != ys[0] || xs[i] != xs[0]) same = 0;
    sh->nchunk = 0;
    sh->max_ctas = 0;
    if (same && sh->count >= 8 * G7_GANG) {
        /* Same-size pictures: rounds of four chunks (multiples of 7 pictures) on four workers, every chunk's kernel on a
           quarter of the SMs.  The four kernels run side by side, so the copies of a chunk overlap the kernels of the
           others, and the small commit kernel that follows a chunk's decision kernel finds that chunk's SMs free (behind
           whole-device kernels it would wait for the next chunk's persistent CTAs to finish). */
        const long long px = padded_pixels(ys[0], xs[0], sh->max_dim) * sh->count;
        int rounds = (int)((px + MAX_WORKERS * CHUNK_PIXELS - 1) / (MAX_WORKERS * CHUNK_PIXELS)), per, sms = hevce_internal_device_sms(sh->device);
        if (rounds < 1) rounds = 1;
        while ((long long)rounds * MAX_WORKERS * (CHUNK_PICTURES - G7_GANG) < sh->count) rounds++;   /* many tiny pictures: the per-chunk picture bound */
        per = (sh->count + rounds * MAX_WORKERS - 1) / (rounds * MAX_WORKERS);
        per = (per + G7_GANG - 1) / G7_GANG * G7_GANG;
        /* more than one wave: cap every chunk's grid at a quarter of the SMs (smaller shards fit side by side anyway) */
        sh->max_ctas = (sms > 0 && sh->count > WAVE_PICTURES) ? (sms + MAX_WORKERS - 1) / MAX_WORKERS : 0;
        for (; done < sh->count; done += per) sh->chunk_first[sh->nchunk++] = sh->first + done;
        sh->chunk_first[sh->nchunk] = sh->first + sh->count;
        return MAX_WORKERS;
    }
    while (done < sh->count) {
        int m = 0, same_c = 1;
        long long px = 0;
        while (done + m < sh->count && m < CHUNK_PICTURES &&
               (m == 0 || px + padded_pixels(ys[done + m], xs[done + m], sh->max_dim) <= CHUNK_PIXELS)) {
            px += padded_pixels(ys[done + m], xs[done + m], sh->max_dim);
            if (ys[done + m] != ys[done] || xs[done + m] != xs[done]) same_c = 0;
            m++;
        }
        /* same-size pictures: whole waves of g7 per chunk, so no chunk ends with a nearly empty wave */
        if (same_c && m > WAVE_PICTURES && done + m < sh->count) m -= m % WAVE_PICTURES;
        sh->chunk_first[sh->nchunk++] = sh->first + done;
        done += m;
    }
    sh->chunk_first[sh->nchunk] = sh->first + sh->count;
    return 2;   /* whole-device kernels: two workers, so one chunk's copies overlap the other's kernels */
}

/* encode pictures [first, first+count) on one device */
static void *shard_main(void *arg) {
    Shard *sh = (Shard *)arg;
    int nworkers, nh = 0, i;
    pthread_t helpers[MAX_WORKERS];
    sh->status = 0;
    sh->next_chunk = 0;
    sh->chunk_first = (int *)malloc(sizeof(int) * (size_t)(sh->count + 1));
    if (!sh->chunk_first) { sh->status = HEVCE_ERR_ARG; return NULL; }
    pthread_mutex_init(&sh->qlock, NULL);
    /* the kernel variant is chosen for the whole shard: its chunks share the device */
    sh->variant = hevce_internal_choose_variant(sh->device, sh->count, sh->ysz + sh->first, sh->xsz + sh->first, sh->max_dim);
    nworkers = plan_chunks(sh);
    if (nworkers > sh->nchunk) nworkers = sh->nchunk;
    for (i = 1; i < nworkers; i++)
        if (pthread_create(&helpers[nh], NULL, chunk_worker, sh) == 0) nh++;
    chunk_worker(sh);
    for (i = 0; i < nh; i++) pthread_join(helpers[i], NULL);
    pthread_mutex_destroy(&sh->qlock);
    free(sh->chunk_first);
    return NULL;
}

/* Contiguous shards with (nearly) equal padded-pixel = CTU counts over ndev devices: shard k holds pictures
   [first[k], first[k] + count[k]) on device dev[k].  Returns the number of shards (devices without pictures get none). */
static int cut_shards(int n, const int *ysz, const int *xsz, int max_dim, int ndev, const int *devs, int *dev, int *first, int *count) {
    long long total = 0, acc = 0;
    int i, k, nshard = 0;
    for (i = 0; i < n; i++) total += padded_pixels(ysz[i], xsz[i], max_dim);
    if (ndev > n) ndev = n;
    for (k = 0, i = 0; k < ndev; k++) {
        int f = i;
        long long want = total * (k + 1) / ndev;
        while (i < n && (k == ndev - 1 || acc + padded_pixels(ysz[i], xsz[i], max_dim) / 2 <= want)) acc += padded_pixels(ysz[i], xsz[i], max_dim), i++;
        if (i == f) continue;
        dev[nshard] = devs[k]; first[nshard] = f; count[nshard] = i - f;
        nshard++;
    }
    return nshard;
}

/* size write-back (HEVCe.c:1643-1644) */
static void write_sizes(int n, int *ysz, int *xsz, int max_dim) {
    int i;
    for (i = 0; i < n; i++) {
        ysz[i] = padded_dim(ysz[i], max_dim);
        xsz[i] = padded_dim(xsz[i], max_dim);
    }
}

/* the batch path of every encoding entry point; img_decs NULL: no decoded pictures; quality NULL: no quality reduction.
   max_dim is the caller's one value for the whole call (sharding, clamp and size write-back); the sizes are not written. */
static int encode_batch(int n, unsigned char *const *pbuffers, const unsigned char *const *imgs, unsigned char *const *img_rcons,
                        unsigned char *const *img_decs, const int *ysz, const int *xsz, const int *qpd6, int *stream_len, int max_dim,
                        int metric, double *quality) {
    Shard shards[MAX_DEV];
    pthread_t threads[MAX_DEV];
    int ndev, devs[MAX_DEV], started[MAX_DEV], i, k, nshard = 0, status = 0, *lens = stream_len, saved_device;
    int cut_dev[MAX_DEV], cut_first[MAX_DEV], cut_count[MAX_DEV];
    if (n < 0) return HEVCE_ERR_ARG;
    if (n == 0) return 0;
    if (!pbuffers || !imgs || !img_rcons || !ysz || !xsz || !qpd6) return HEVCE_ERR_ARG;
    for (i = 0; i < n; i++)
        if (!pbuffers[i] || !imgs[i] || !img_rcons[i] || ysz[i] <= 0 || xsz[i] <= 0 || qpd6[i] < 0 || qpd6[i] > 4) return HEVCE_ERR_ARG;
    pthread_mutex_lock(&g_lock);
    ndev = resolve_devices();
    if (ndev > 0) memcpy(devs, g_devs, sizeof(int) * (size_t)ndev);
    pthread_mutex_unlock(&g_lock);
    if (ndev < 0) return ndev;
    if (ndev == 0) {
        fprintf(stderr, "libhevce_b200: no usable CUDA device (this library has no CPU path)\n");
        return HEVCE_ERR_CUDA;
    }
    if (!lens) lens = (int *)malloc(sizeof(int) * (size_t)n);
    if (!lens) return HEVCE_ERR_ARG;
    saved_device = hevce_internal_get_device();   /* shard 0 runs on this thread and selects its device */
    nshard = cut_shards(n, ysz, xsz, max_dim, ndev, devs, cut_dev, cut_first, cut_count);
    for (k = 0; k < nshard; k++) {
        shards[k].device = cut_dev[k]; shards[k].first = cut_first[k]; shards[k].count = cut_count[k]; shards[k].max_dim = max_dim;
        shards[k].pbuffers = pbuffers; shards[k].imgs = imgs; shards[k].rcons = img_rcons; shards[k].decs = img_decs;
        shards[k].ysz = ysz; shards[k].xsz = xsz; shards[k].qpd6 = qpd6; shards[k].stream_len = lens;
        shards[k].metric = metric; shards[k].quality = quality;
    }
    for (k = 1; k < nshard; k++) {
        started[k] = pthread_create(&threads[k], NULL, shard_main, &shards[k]) == 0;
        if (!started[k]) shard_main(&shards[k]);   /* no thread: run the shard here */
    }
    shard_main(&shards[0]);
    for (k = 1; k < nshard; k++)
        if (started[k]) pthread_join(threads[k], NULL);
    for (k = 0; k < nshard; k++)
        if (shards[k].status && !status) status = shards[k].status;
    if (lens != stream_len) free(lens);
    hevce_internal_set_device(saved_device);      /* leave the caller's current device as it was */
    return status;
}

API int HEVCImageEncoderBatch(int n, unsigned char *const *pbuffers, const unsigned char *const *imgs,
                              unsigned char *const *img_rcons, int *ysz, int *xsz, const int *qpd6, int *stream_len) {
    const int max_dim = hevce_get_max_dim();
    const int rc = encode_batch(n, pbuffers, imgs, img_rcons, NULL, ysz, xsz, qpd6, stream_len, max_dim, 0, NULL);
    if (!rc) write_sizes(n, ysz, xsz, max_dim);
    return rc;
}

API int HEVCImageEncoderBatchDecoded(int n, unsigned char *const *pbuffers, const unsigned char *const *imgs, unsigned char *const *img_rcons,
                                     unsigned char *const *img_decs, int *ysz, int *xsz, const int *qpd6, int *stream_len) {
    const int max_dim = hevce_get_max_dim();
    int i, rc;
    if (!hevce_session_deblock || !hevce_session_download_decoded) return HEVCE_ERR_STATE;   /* linked without them */
    if (n > 0 && !img_decs) return HEVCE_ERR_ARG;
    for (i = 0; i < n; i++)
        if (!img_decs[i]) return HEVCE_ERR_ARG;
    rc = encode_batch(n, pbuffers, imgs, img_rcons, img_decs, ysz, xsz, qpd6, stream_len, max_dim, 0, NULL);
    if (!rc) write_sizes(n, ysz, xsz, max_dim);
    return rc;
}

/* Quality-target search (the rule is in hevce.h).  Each round encodes the pictures still searching, at their probe qpd6,
   through encode_batch.  A picture without a passing probe yet encodes straight into the caller's buffers; one whose
   buffers hold a passing probe encodes into host scratch, copied over only if the new probe passes too.  So the caller's
   buffers always hold the last passing probe, or, while none has passed, the last probe: at the end, the chosen one. */
API int HEVCImageEncoderBatchTarget(int n, unsigned char *const *pbuffers, const unsigned char *const *imgs, unsigned char *const *img_rcons,
                                    unsigned char *const *img_decs, int *ysz, int *xsz, int metric, const double *target, int *qpd6,
                                    double *quality, int *stream_len) {
    const int max_dim = hevce_get_max_dim();
    int i, k, m, rc = 0, *ints;
    int *lo, *hi, *len, *idx, *sub_ys, *sub_xs, *sub_q, *sub_len;
    double *dbls, *qual, *sub_qual;
    unsigned char **ptrs, **sub_pb, **sub_rc, **sub_dec;
    const unsigned char **sub_img;
    if (metric != HEVCE_METRIC_PSNR && metric != HEVCE_METRIC_SSIM) return HEVCE_ERR_ARG;
    if (!hevce_session_deblock || (img_decs && !hevce_session_download_decoded) ||
        (metric == HEVCE_METRIC_SSIM ? !hevce_session_ssim : !hevce_session_decoded_quality))
        return HEVCE_ERR_STATE;   /* linked without a call the metric needs */
    if (n < 0) return HEVCE_ERR_ARG;
    if (n == 0) return 0;
    if (!pbuffers || !imgs || !img_rcons || !ysz || !xsz || !target || !qpd6) return HEVCE_ERR_ARG;
    for (i = 0; i < n; i++)
        if (!pbuffers[i] || !imgs[i] || !img_rcons[i] || (img_decs && !img_decs[i]) || ysz[i] <= 0 || xsz[i] <= 0 || isnan(target[i]))
            return HEVCE_ERR_ARG;
    ints = (int *)malloc(sizeof(int) * 8 * (size_t)n);
    dbls = (double *)malloc(sizeof(double) * 2 * (size_t)n);
    ptrs = (unsigned char **)malloc(sizeof(unsigned char *) * 4 * (size_t)n);
    if (!ints || !dbls || !ptrs) {
        free(ints); free(dbls); free(ptrs);
        return HEVCE_ERR_ARG;
    }
    lo = ints; hi = lo + n; len = hi + n; idx = len + n; sub_ys = idx + n; sub_xs = sub_ys + n; sub_q = sub_xs + n; sub_len = sub_q + n;
    qual = dbls; sub_qual = qual + n;
    sub_pb = ptrs; sub_rc = sub_pb + n; sub_dec = sub_rc + n; sub_img = (const unsigned char **)(sub_dec + n);
    for (i = 0; i < n; i++) lo[i] = -1, hi[i] = 5;
    for (;;) {
        size_t scratch_bytes = 0, off = 0;
        unsigned char *scratch = NULL;
        for (i = 0, m = 0; i < n; i++) {
            if (hi[i] - lo[i] <= 1) continue;
            idx[m] = i; sub_q[m] = (lo[i] + hi[i]) / 2; sub_ys[m] = ysz[i]; sub_xs[m] = xsz[i]; sub_img[m] = imgs[i];
            if (lo[i] >= 0) scratch_bytes += (size_t)padded_pixels(ysz[i], xsz[i], max_dim) * (img_decs ? 4 : 3) + 256;
            m++;
        }
        if (m == 0) break;
        if (scratch_bytes && !(scratch = (unsigned char *)malloc(scratch_bytes))) { rc = HEVCE_ERR_ARG; break; }
        for (k = 0; k < m; k++) {
            i = idx[k];
            if (lo[i] < 0) {
                sub_pb[k] = pbuffers[i]; sub_rc[k] = img_rcons[i]; sub_dec[k] = img_decs ? img_decs[i] : NULL;
            } else {   /* stream (256 + 2 B/pixel), reconstruction, decoded picture */
                const size_t px = (size_t)padded_pixels(ysz[i], xsz[i], max_dim);
                sub_pb[k] = scratch + off; off += 256 + 2 * px;
                sub_rc[k] = scratch + off; off += px;
                sub_dec[k] = NULL;
                if (img_decs) { sub_dec[k] = scratch + off; off += px; }
            }
        }
        rc = encode_batch(m, sub_pb, sub_img, sub_rc, img_decs ? sub_dec : NULL, sub_ys, sub_xs, sub_q, sub_len, max_dim, metric, sub_qual);
        for (k = 0; !rc && k < m; k++) {
            const int pass = sub_qual[k] >= target[idx[k]], direct = lo[idx[k]] < 0;
            i = idx[k];
            if (pass && !direct) {   /* a better passing probe replaces the one in the caller's buffers */
                const size_t px = (size_t)padded_pixels(ysz[i], xsz[i], max_dim);
                memcpy(pbuffers[i], sub_pb[k], (size_t)sub_len[k]);
                memcpy(img_rcons[i], sub_rc[k], px);
                if (img_decs) memcpy(img_decs[i], sub_dec[k], px);
            }
            if (pass || direct) { len[i] = sub_len[k]; qual[i] = sub_qual[k]; }
            if (pass) lo[i] = sub_q[k];
            else hi[i] = sub_q[k];
        }
        free(scratch);
        if (rc) break;
    }
    if (!rc) {
        for (i = 0; i < n; i++) {
            qpd6[i] = lo[i] >= 0 ? lo[i] : 0;
            if (quality) quality[i] = qual[i];
            if (stream_len) stream_len[i] = len[i];
        }
        write_sizes(n, ysz, xsz, max_dim);
    }
    free(ints); free(dbls); free(ptrs);
    return rc;
}

API int HEVCImageEncoder(unsigned char *pbuffer, const unsigned char *img, unsigned char *img_rcon, int *ysz, int *xsz, const int qpd6) {
    int len = 0, rc;
    unsigned char *pb[1];
    const unsigned char *im[1];
    unsigned char *rc_[1];
    if (!ysz || !xsz) return HEVCE_ERR_ARG;
    pb[0] = pbuffer; im[0] = img; rc_[0] = img_rcon;
    rc = HEVCImageEncoderBatch(1, pb, im, rc_, ysz, xsz, &qpd6, &len);
    return rc ? rc : len;
}

/* ---- f6: the decoder ----------------------------------------------------------------------------------------- */
typedef struct {
    int device, first, count, status;
    const unsigned char *const *streams;
    const int *stream_len, *ysz, *xsz;
    unsigned char *const *decs;
    int *pic_status;
} DecShard;

/* decode pictures [first, first+count) on one device, in chunks of at most CHUNK_PIXELS / CHUNK_PICTURES; a chunk whose
   pictures did not all parse does not stop the others */
static void *dec_shard_main(void *arg) {
    DecShard *sh = (DecShard *)arg;
    hevce_decoder *d = NULL;
    int cached = 0, done = 0;
    sh->status = 0;
    pthread_mutex_lock(&g_lock);
    if (!g_dec_busy[sh->device]) { g_dec_busy[sh->device] = 1; cached = 1; d = g_dec[sh->device]; }
    pthread_mutex_unlock(&g_lock);
    if (!d) d = hevce_decoder_create(sh->device);   /* first use, or another call is using the cached one */
    if (d && cached) {
        pthread_mutex_lock(&g_lock);
        g_dec[sh->device] = d;
        pthread_mutex_unlock(&g_lock);
    }
    if (!d) sh->status = HEVCE_ERR_CUDA;
    while (d && done < sh->count) {
        const int a = sh->first + done;
        int m = 0, rc;
        long long px = 0;
        while (done + m < sh->count && m < CHUNK_PICTURES && (m == 0 || px + (long long)sh->ysz[a + m] * sh->xsz[a + m] <= CHUNK_PIXELS))
            px += (long long)sh->ysz[a + m] * sh->xsz[a + m], m++;
        rc = hevce_decoder_upload(d, m, sh->streams + a, sh->stream_len + a);
        if (!rc) rc = hevce_decoder_run(d);
        if (rc) { sh->status = rc; break; }
        rc = hevce_decoder_download(d, sh->decs + a, sh->pic_status ? sh->pic_status + a : NULL);
        done += m;
        if (rc == HEVCE_ERR_STATE) sh->status = rc;   /* pictures that did not parse: the next chunks still run */
        else if (rc) { sh->status = rc; break; }
    }
    if (cached) {
        pthread_mutex_lock(&g_lock);
        g_dec_busy[sh->device] = 0;
        pthread_mutex_unlock(&g_lock);
    } else if (d) {
        hevce_decoder_destroy(d);
    }
    return NULL;
}

API int HEVCImageDecoderBatch(int n, const unsigned char *const *streams, const int *stream_len, unsigned char *const *img_decs, int *status) {
    DecShard shards[MAX_DEV];
    pthread_t threads[MAX_DEV];
    int ndev, devs[MAX_DEV], cut_dev[MAX_DEV], cut_first[MAX_DEV], cut_count[MAX_DEV], started[MAX_DEV], *ys, *xs, i, k, q, nshard, rc = 0,
        saved_device;
    if (!hevce_stream_info || !hevce_decoder_create || !hevce_decoder_upload || !hevce_decoder_run || !hevce_decoder_download ||
        !hevce_decoder_destroy)
        return HEVCE_ERR_STATE;   /* linked without the decoder */
    if (n < 0) return HEVCE_ERR_ARG;
    if (n == 0) return 0;
    if (!streams || !stream_len || !img_decs) return HEVCE_ERR_ARG;
    ys = (int *)malloc(sizeof(int) * (size_t)n);
    xs = (int *)malloc(sizeof(int) * (size_t)n);
    for (i = 0; ys && xs && i < n && !rc; i++)
        if (!streams[i] || !img_decs[i] || hevce_stream_info(streams[i], stream_len[i], &ys[i], &xs[i], &q)) rc = HEVCE_ERR_ARG;
    if (!ys || !xs) rc = HEVCE_ERR_ARG;
    if (!rc) {
        pthread_mutex_lock(&g_lock);
        ndev = resolve_devices();
        if (ndev > 0) memcpy(devs, g_devs, sizeof(int) * (size_t)ndev);
        pthread_mutex_unlock(&g_lock);
        if (ndev < 0) rc = ndev;
        else if (ndev == 0) {
            fprintf(stderr, "libhevce_b200: no usable CUDA device (this library has no CPU path)\n");
            rc = HEVCE_ERR_CUDA;
        }
    }
    if (rc) { free(ys); free(xs); return rc; }
    saved_device = hevce_internal_get_device();   /* shard 0 runs on this thread and selects its device */
    nshard = cut_shards(n, ys, xs, 16384, ndev, devs, cut_dev, cut_first, cut_count);   /* stream sizes are padded already */
    for (k = 0; k < nshard; k++) {
        shards[k].device = cut_dev[k]; shards[k].first = cut_first[k]; shards[k].count = cut_count[k];
        shards[k].streams = streams; shards[k].stream_len = stream_len; shards[k].ysz = ys; shards[k].xsz = xs;
        shards[k].decs = img_decs; shards[k].pic_status = status;
    }
    for (k = 1; k < nshard; k++) {
        started[k] = pthread_create(&threads[k], NULL, dec_shard_main, &shards[k]) == 0;
        if (!started[k]) dec_shard_main(&shards[k]);
    }
    dec_shard_main(&shards[0]);
    for (k = 1; k < nshard; k++)
        if (started[k]) pthread_join(threads[k], NULL);
    for (k = 0; k < nshard; k++)   /* a failed call outranks pictures that did not parse */
        if (shards[k].status && (!rc || rc == HEVCE_ERR_STATE)) rc = shards[k].status;
    free(ys);
    free(xs);
    hevce_internal_set_device(saved_device);   /* leave the caller's current device as it was */
    return rc;
}
