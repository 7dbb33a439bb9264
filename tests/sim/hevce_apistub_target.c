/*
 * hevce_apistub_target.c -- plain-C stand-in for the whole CUDA layer below csrc/hevce_api.c, for
 * HEVCImageEncoderBatchTarget (TEST INFRASTRUCTURE ONLY).  tests/test_host_api_target.py links it alone with the
 * unmodified csrc/hevce_api.c.  Unlike hevce_apistub.c it reads and writes the picture buffers:
 *
 *   - every image buffer starts with a picture id (int32); hevce_session_upload reads it;
 *   - apistub_target_reset(ndev, fail_configure, fail_code) reports ndev devices with 148 SMs each, clears the log, and
 *     lets the k-th configure (counted from 1 over all threads) fail with a chosen code;
 *   - hevce_session_upload logs (configure number, device, id, qpd6, ysz, xsz) for every picture of the session;
 *   - the downloads write the markers (id, qpd6, 'S' / 'R' / 'D') at the start of the stream, reconstruction and decoded
 *     buffers; stream_len = 16 + (5 * id + qpd6) % 200, within the stream capacity of a 32x32 picture;
 *   - the two quality calls return apistub_target_table[id * 5 + qpd6], set by the test, and count their calls; they need
 *     a hevce_session_deblock of the same encode first;
 *   - -DAPISTUB_NO_QUALITY leaves out hevce_session_ssim and hevce_session_decoded_quality.
 */
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

#include "hevce_internal.h"

#define LOG_CAP 65536
#define MAX_ID 4096

struct hevce_session {
    int device, n, configure_no, deblocked;
    const int *ysz, *xsz, *qpd6;
    int id[LOG_CAP];
};

static pthread_mutex_t g_mutex = PTHREAD_MUTEX_INITIALIZER;
static _Thread_local int g_current = 0;
static int g_ndev = 1, g_nconfigure, g_fail_configure, g_fail_code, g_nlog, g_nssim, g_npsnr;
static long long g_log[LOG_CAP][6];
double apistub_target_table[MAX_ID * 5];

void apistub_target_reset(int ndev, int fail_configure, int fail_code) {
    pthread_mutex_lock(&g_mutex);
    g_ndev = ndev;
    g_nconfigure = g_nlog = g_nssim = g_npsnr = 0;
    g_fail_configure = fail_configure;
    g_fail_code = fail_code;
    pthread_mutex_unlock(&g_mutex);
}

/* copies up to cap logged pictures, 6 values each, and returns how many were logged */
int apistub_target_log(long long *rows, int cap) {
    int i, k, n;
    pthread_mutex_lock(&g_mutex);
    n = g_nlog;
    for (i = 0; i < n && i < cap; i++)
        for (k = 0; k < 6; k++) rows[6 * i + k] = g_log[i][k];
    pthread_mutex_unlock(&g_mutex);
    return n;
}

/* quality calls so far: metric 0 = hevce_session_decoded_quality, 1 = hevce_session_ssim */
int apistub_target_quality_calls(int metric) { return metric ? g_nssim : g_npsnr; }

int hevce_internal_device_count(void) { return g_ndev; }
int hevce_internal_get_device(void) { return g_current; }
void hevce_internal_set_device(int device) {
    if (device >= 0) g_current = device;
}
int hevce_internal_device_sms(int device) {
    g_current = device;
    return 148;
}
int hevce_internal_choose_variant(int device, int n, const int *ysz, const int *xsz, int max_dim) {
    (void)n, (void)ysz, (void)xsz, (void)max_dim;
    g_current = device;
    return 0;
}

hevce_session *hevce_session_create_empty(int device) {
    hevce_session *s = (hevce_session *)calloc(1, sizeof(hevce_session));
    if (s) s->device = device;
    g_current = device;
    return s;
}

void hevce_session_destroy(hevce_session *s) { free(s); }

int hevce_session_configure(hevce_session *s, int n, const int *ysz, const int *xsz, const int *qpd6, int max_dim, int variant, int max_ctas) {
    int rc = 0;
    (void)max_dim, (void)variant, (void)max_ctas;
    g_current = s->device;
    if (n > LOG_CAP) return HEVCE_ERR_STATE;
    s->n = n; s->ysz = ysz; s->xsz = xsz; s->qpd6 = qpd6; s->deblocked = 0;
    pthread_mutex_lock(&g_mutex);
    s->configure_no = ++g_nconfigure;
    if (s->configure_no == g_fail_configure) rc = g_fail_code;
    pthread_mutex_unlock(&g_mutex);
    return rc;
}

int hevce_session_upload(hevce_session *s, const unsigned char *const *imgs) {
    int i, rc = 0;
    g_current = s->device;
    pthread_mutex_lock(&g_mutex);
    for (i = 0; i < s->n; i++) {
        memcpy(&s->id[i], imgs[i], sizeof(int));
        if (s->id[i] < 0 || s->id[i] >= MAX_ID || g_nlog >= LOG_CAP) { rc = HEVCE_ERR_STATE; break; }
        {
            long long *e = g_log[g_nlog++];
            e[0] = s->configure_no; e[1] = s->device; e[2] = s->id[i]; e[3] = s->qpd6[i]; e[4] = s->ysz[i]; e[5] = s->xsz[i];
        }
    }
    pthread_mutex_unlock(&g_mutex);
    return rc;
}

int hevce_session_encode(hevce_session *s) {
    g_current = s->device;
    s->deblocked = 0;
    return 0;
}

static void marker(unsigned char *buf, int id, int q, char what) {
    memcpy(buf, &id, sizeof(int));
    memcpy(buf + 4, &q, sizeof(int));
    buf[8] = (unsigned char)what;
}

int hevce_session_download(hevce_session *s, unsigned char *const *pbuffers, unsigned char *const *img_rcons, int *stream_len) {
    int i;
    g_current = s->device;
    for (i = 0; i < s->n; i++) {
        marker(pbuffers[i], s->id[i], s->qpd6[i], 'S');
        marker(img_rcons[i], s->id[i], s->qpd6[i], 'R');
        if (stream_len) stream_len[i] = 16 + (5 * s->id[i] + s->qpd6[i]) % 200;
    }
    return 0;
}

int hevce_session_deblock(hevce_session *s) {
    g_current = s->device;
    s->deblocked = 1;
    return 0;
}

int hevce_session_download_decoded(hevce_session *s, unsigned char *const *img_decs) {
    int i;
    g_current = s->device;
    if (!s->deblocked) return HEVCE_ERR_STATE;
    for (i = 0; i < s->n; i++) marker(img_decs[i], s->id[i], s->qpd6[i], 'D');
    return 0;
}

#ifndef APISTUB_NO_QUALITY
static int quality(hevce_session *s, double *out, int *count) {
    int i;
    g_current = s->device;
    if (!s->deblocked) return HEVCE_ERR_STATE;
    for (i = 0; i < s->n; i++) out[i] = apistub_target_table[s->id[i] * 5 + s->qpd6[i]];
    pthread_mutex_lock(&g_mutex);
    ++*count;
    pthread_mutex_unlock(&g_mutex);
    return 0;
}

int hevce_session_decoded_quality(hevce_session *s, double *mse, double *psnr) {
    if (mse || !psnr) return HEVCE_ERR_ARG;   /* the target search asks for the PSNR only */
    return quality(s, psnr, &g_npsnr);
}

int hevce_session_ssim(hevce_session *s, int decoded, double *ssim) {
    if (decoded != 1) return HEVCE_ERR_ARG;   /* the target search measures the decoded pictures */
    return quality(s, ssim, &g_nssim);
}
#endif
