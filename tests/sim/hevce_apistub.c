/*
 * hevce_apistub.c -- plain-C stand-in for the CUDA layer below csrc/hevce_api.c (TEST INFRASTRUCTURE ONLY).
 *
 * tests/test_host_api.py links it with the unmodified csrc/hevce_api.c, so the sharding, chunking, worker and session
 * pool logic of HEVCImageEncoderBatch runs on the CPU without a kernel, the CUDA runtime or a GPU.  The stub defines
 * every function hevce_api.c calls through hevce_internal.h and hevce.h.  It never dereferences a picture buffer.
 *
 *   - apistub_reset(n, ...) reports n devices with 148 SMs each and clears the call log;
 *   - every call that selects a device in the real layer selects it here, in a per-thread current device;
 *   - hevce_session_configure logs (device, first picture, count, variant, max_ctas, max_dim) under a mutex, with the
 *     first picture counted from the array given to apistub_set_base;
 *   - hevce_internal_choose_variant returns (device + n) % 6, so a test sees one shard's choice reach all its chunks;
 *   - the k-th configure or download (counted from 1 over all threads) can fail with a chosen code;
 *   - hevce_session_download writes each picture's index into stream_len.
 */
#include <pthread.h>
#include <stdlib.h>

#include "hevce_internal.h"

#define LOG_CAP 4096

struct hevce_session {
    int device, n;
    const int *ysz;
};

static pthread_mutex_t g_mutex = PTHREAD_MUTEX_INITIALIZER;
static _Thread_local int g_current = 0;
static int g_ndev = 1;
static const int *g_base;
static long long g_log[LOG_CAP][6];
static int g_nlog, g_nconfigure, g_ndownload, g_fail_configure, g_fail_download, g_fail_code;

void apistub_reset(int ndev, int fail_configure, int fail_download, int fail_code) {
    pthread_mutex_lock(&g_mutex);
    g_ndev = ndev;
    g_nlog = g_nconfigure = g_ndownload = 0;
    g_fail_configure = fail_configure;
    g_fail_download = fail_download;
    g_fail_code = fail_code;
    pthread_mutex_unlock(&g_mutex);
}

void apistub_set_base(const int *ysz) { g_base = ysz; }

/* copies up to cap logged configure calls, 6 values each, and returns how many were logged */
int apistub_calls(long long *rows, int cap) {
    int i, k, n;
    pthread_mutex_lock(&g_mutex);
    n = g_nlog;
    for (i = 0; i < n && i < cap; i++)
        for (k = 0; k < 6; k++) rows[6 * i + k] = g_log[i][k];
    pthread_mutex_unlock(&g_mutex);
    return n;
}

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
    (void)ysz, (void)xsz, (void)max_dim;
    g_current = device;
    return (device + n) % 6;
}

hevce_session *hevce_session_create_empty(int device) {
    hevce_session *s = (hevce_session *)calloc(1, sizeof(hevce_session));
    if (s) s->device = device;
    g_current = device;
    return s;
}

int hevce_session_configure(hevce_session *s, int n, const int *ysz, const int *xsz, const int *qpd6, int max_dim, int variant, int max_ctas) {
    int rc = 0;
    (void)xsz, (void)qpd6;
    g_current = s->device;
    s->n = n;
    s->ysz = ysz;
    pthread_mutex_lock(&g_mutex);
    if (++g_nconfigure == g_fail_configure) rc = g_fail_code;
    if (g_nlog < LOG_CAP) {
        long long *e = g_log[g_nlog++];
        e[0] = s->device; e[1] = ysz - g_base; e[2] = n; e[3] = variant; e[4] = max_ctas; e[5] = max_dim;
    } else {
        rc = HEVCE_ERR_STATE;
    }
    pthread_mutex_unlock(&g_mutex);
    return rc;
}

int hevce_session_upload(hevce_session *s, const unsigned char *const *imgs) {
    (void)imgs;
    g_current = s->device;
    return 0;
}

int hevce_session_encode(hevce_session *s) {
    g_current = s->device;
    return 0;
}

int hevce_session_download(hevce_session *s, unsigned char *const *pbuffers, unsigned char *const *img_rcons, int *stream_len) {
    int i, rc = 0;
    (void)pbuffers, (void)img_rcons;
    g_current = s->device;
    pthread_mutex_lock(&g_mutex);
    if (++g_ndownload == g_fail_download) rc = g_fail_code;
    pthread_mutex_unlock(&g_mutex);
    if (!rc && stream_len)
        for (i = 0; i < s->n; i++) stream_len[i] = (int)(s->ysz - g_base) + i;
    return rc;
}

void hevce_session_destroy(hevce_session *s) { free(s); }
