/*
 * hevce_apistub_decoded.c -- plain-C stand-in for the two session calls of HEVCImageEncoderBatchDecoded (TEST
 * INFRASTRUCTURE ONLY).  tests/test_host_api_decoded.py links it with the unmodified csrc/hevce_api.c and
 * tests/sim/hevce_apistub.c, which stands in for the rest of the CUDA layer.
 *
 *   - apistub_decoded_reset(...) clears the counters and the log; the k-th hevce_session_deblock or
 *     hevce_session_download_decoded (counted from 1 over all threads) can fail with a chosen code;
 *   - hevce_session_download_decoded logs (device, picture, img_decs[i]) for every picture of its chunk, with the
 *     picture counted from the array given to apistub_decoded_set_base;
 *   - both select the session's device, as the real calls do.
 */
#include <pthread.h>
#include <stddef.h>

#include "hevce_internal.h"

#define DEC_LOG_CAP 65536

struct hevce_session {   /* the layout hevce_apistub.c allocates */
    int device, n;
    const int *ysz;
};

static pthread_mutex_t g_dmutex = PTHREAD_MUTEX_INITIALIZER;
static const int *g_dbase;
static long long g_dlog[DEC_LOG_CAP][3];
static int g_ndlog, g_ndeblock, g_ndownload, g_fail_deblock, g_fail_download, g_fail_code;

void apistub_decoded_reset(int fail_deblock, int fail_download_decoded, int fail_code) {
    pthread_mutex_lock(&g_dmutex);
    g_ndlog = g_ndeblock = g_ndownload = 0;
    g_fail_deblock = fail_deblock;
    g_fail_download = fail_download_decoded;
    g_fail_code = fail_code;
    pthread_mutex_unlock(&g_dmutex);
}

void apistub_decoded_set_base(const int *ysz) { g_dbase = ysz; }

/* copies up to cap logged pictures, 3 values each, and returns how many were logged */
int apistub_decoded_log(long long *rows, int cap) {
    int i, k, n;
    pthread_mutex_lock(&g_dmutex);
    n = g_ndlog;
    for (i = 0; i < n && i < cap; i++)
        for (k = 0; k < 3; k++) rows[3 * i + k] = g_dlog[i][k];
    pthread_mutex_unlock(&g_dmutex);
    return n;
}

int apistub_deblocks(void) {
    int n;
    pthread_mutex_lock(&g_dmutex);
    n = g_ndeblock;
    pthread_mutex_unlock(&g_dmutex);
    return n;
}

int hevce_session_deblock(hevce_session *s) {
    int rc = 0;
    hevce_internal_set_device(s->device);
    pthread_mutex_lock(&g_dmutex);
    if (++g_ndeblock == g_fail_deblock) rc = g_fail_code;
    pthread_mutex_unlock(&g_dmutex);
    return rc;
}

int hevce_session_download_decoded(hevce_session *s, unsigned char *const *img_decs) {
    int i, rc = 0;
    hevce_internal_set_device(s->device);
    pthread_mutex_lock(&g_dmutex);
    if (++g_ndownload == g_fail_download) rc = g_fail_code;
    for (i = 0; !rc && i < s->n; i++) {
        if (g_ndlog < DEC_LOG_CAP) {
            long long *e = g_dlog[g_ndlog++];
            e[0] = s->device; e[1] = (s->ysz - g_dbase) + i; e[2] = (long long)(size_t)img_decs[i];
        } else {
            rc = HEVCE_ERR_STATE;
        }
    }
    pthread_mutex_unlock(&g_dmutex);
    return rc;
}
