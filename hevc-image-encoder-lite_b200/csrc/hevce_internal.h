/* hevce_internal.h -- private C interface between hevce_api.c (plain C host code) and hevce_cuda.cu. */
#ifndef HEVCE_INTERNAL_H
#define HEVCE_INTERNAL_H
#include "../../include/hevce.h"
#ifdef __cplusplus
extern "C" {
#endif
int hevce_internal_device_count(void);
int hevce_internal_get_device(void);          /* the calling thread's current CUDA device, -1 if none */
void hevce_internal_set_device(int device);   /* no-op for device < 0 */
hevce_session *hevce_session_create_empty(int device);
int hevce_internal_choose_variant(int device, int n, const int *ysz, const int *xsz, int max_dim);   /* variant index or < 0 */
int hevce_internal_device_sms(int device);   /* 0 on error */
int hevce_session_configure(hevce_session *s, int n, const int *ysz, const int *xsz, const int *qpd6, int max_dim, int variant, int max_ctas);   /* variant < 0: choose; max_ctas 0: no cap */
#ifdef __cplusplus
}
#endif
#endif
