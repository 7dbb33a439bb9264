/*
 * hevce_apistub_decoder.c -- plain-C stand-in for the decoder calls of the CUDA layer (TEST INFRASTRUCTURE ONLY).
 * tests/test_host_api_decoder.py links it with the unmodified csrc/hevce_api.c and tests/sim/hevce_apistub.c, which
 * stands in for the rest of the CUDA layer.
 *
 *   - a stub stream is 8 bytes: "HVC6", H / 32, W / 32 (one byte each), qpd6, and a last byte that is 1 when the
 *     picture's slice data "does not parse"; hevce_stream_info rejects anything else;
 *   - hevce_decoder_upload logs (device, first picture, count), the first picture counted from the array given to
 *     apistub_decoder_set_base, and checks every header again; the k-th create, upload, run or download (counted from 1
 *     over all threads) can fail with a chosen code;
 *   - hevce_decoder_download writes picture index + 1 into the first byte of each picture and the status of each.
 */
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

#include "hevce_internal.h"

#define DLOG_CAP 4096

struct hevce_decoder {
    int device, n;
    const unsigned char *const *streams;
};

static pthread_mutex_t g_m = PTHREAD_MUTEX_INITIALIZER;
static const unsigned char *const *g_sbase;
static long long g_log[DLOG_CAP][3];
static int g_nlog, g_count[4], g_fail[4], g_code, g_live;

void apistub_decoder_reset(int fail_create, int fail_upload, int fail_run, int fail_download, int code) {
    pthread_mutex_lock(&g_m);
    g_nlog = 0;
    memset(g_count, 0, sizeof(g_count));
    g_fail[0] = fail_create; g_fail[1] = fail_upload; g_fail[2] = fail_run; g_fail[3] = fail_download;
    g_code = code;
    pthread_mutex_unlock(&g_m);
}

void apistub_decoder_set_base(const unsigned char *const *streams) { g_sbase = streams; }

int apistub_decoder_log(long long *rows, int cap) {
    int i, k, n;
    pthread_mutex_lock(&g_m);
    n = g_nlog;
    for (i = 0; i < n && i < cap; i++)
        for (k = 0; k < 3; k++) rows[3 * i + k] = g_log[i][k];
    pthread_mutex_unlock(&g_m);
    return n;
}

int apistub_decoder_calls(int which) { int n; pthread_mutex_lock(&g_m); n = g_count[which]; pthread_mutex_unlock(&g_m); return n; }
int apistub_decoders_live(void) { int n; pthread_mutex_lock(&g_m); n = g_live; pthread_mutex_unlock(&g_m); return n; }

static int counted(int which) {   /* 0 or the injected failure code of this call */
    int rc = 0;
    pthread_mutex_lock(&g_m);
    if (++g_count[which] == g_fail[which]) rc = g_code;
    pthread_mutex_unlock(&g_m);
    return rc;
}

int hevce_stream_info(const unsigned char *s, int len, int *ysz, int *xsz, int *qpd6) {
    if (!s || len != 8 || memcmp(s, "HVC6", 4) || !s[4] || !s[5] || s[6] > 4 || s[7] > 1) return HEVCE_ERR_ARG;
    if (ysz) *ysz = 32 * s[4];
    if (xsz) *xsz = 32 * s[5];
    if (qpd6) *qpd6 = s[6];
    return 0;
}

hevce_decoder *hevce_decoder_create(int device) {
    hevce_decoder *d;
    if (counted(0)) return NULL;
    d = (hevce_decoder *)calloc(1, sizeof(hevce_decoder));
    d->device = device;
    pthread_mutex_lock(&g_m);
    g_live++;
    pthread_mutex_unlock(&g_m);
    return d;
}

void hevce_decoder_destroy(hevce_decoder *d) {
    if (!d) return;
    pthread_mutex_lock(&g_m);
    g_live--;
    pthread_mutex_unlock(&g_m);
    free(d);
}

int hevce_decoder_upload(hevce_decoder *d, int n, const unsigned char *const *streams, const int *stream_len) {
    int i, rc = counted(1);
    hevce_internal_set_device(d->device);
    if (rc) return rc;
    for (i = 0; i < n; i++)
        if (hevce_stream_info(streams[i], stream_len[i], NULL, NULL, NULL)) return HEVCE_ERR_ARG;
    d->n = n;
    d->streams = streams;
    pthread_mutex_lock(&g_m);
    if (g_nlog < DLOG_CAP) {
        g_log[g_nlog][0] = d->device; g_log[g_nlog][1] = streams - g_sbase; g_log[g_nlog][2] = n;
        g_nlog++;
    }
    pthread_mutex_unlock(&g_m);
    return 0;
}

int hevce_decoder_run(hevce_decoder *d) {
    hevce_internal_set_device(d->device);
    return counted(2);
}

int hevce_decoder_download(hevce_decoder *d, unsigned char *const *img_decs, int *status) {
    int i, ret = 0, rc = counted(3);
    hevce_internal_set_device(d->device);
    if (rc) return rc;
    for (i = 0; i < d->n; i++) {
        const int bad = d->streams[i][7];
        img_decs[i][0] = (unsigned char)((d->streams - g_sbase) + i + 1);
        if (status) status[i] = bad ? HEVCE_ERR_STATE : 0;
        if (bad) ret = HEVCE_ERR_STATE;
    }
    return ret;
}
