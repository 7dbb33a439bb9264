/*
 * hevce.h -- C ABI of libhevce_b200.so, the B200-native HEVC intra still-image encoder.
 *
 * Drop-in boundary: `HEVCImageEncoder` keeps the exact prototype and semantics of the reference entry point
 * (/root/reference/src/HEVCe.h:5-12, defined at src/HEVCe.c:1570-1647; only in-repo caller src/HEVCeMain.c:197).
 * Everything else in this header is new surface of this repository (batch + device-resident sessions).
 *
 * The library exports ONLY the symbols declared here (the reference exports 50 helper symbols such as `predict`,
 * `transform`, `quantize`; both libraries can therefore be loaded into one process).  All work runs in hand-written
 * sm_100a CUDA kernels; there is no CPU fallback: without a usable CUDA device every entry point returns
 * HEVCE_ERR_CUDA.
 */
#ifndef HEVCE_B200_H
#define HEVCE_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define HEVCE_API __attribute__((visibility("default")))
#else
#define HEVCE_API
#endif

#define HEVCE_ERR_ARG   (-1)   /* null pointer, non-positive size, qpd6 outside 0..4, n < 0                     */
#define HEVCE_ERR_CUDA  (-2)   /* no CUDA device / CUDA runtime failure (message on stderr)                      */
#define HEVCE_ERR_STATE (-3)   /* internal consistency check failed (stream buffer overflow, commit mismatch)    */

/*
 * Replaces: int HEVCImageEncoder(pbuffer, img, img_rcon, ysz, xsz, qpd6)   -- HEVCe.h:5-12, HEVCe.c:1570-1577.
 *   pbuffer  : receives the .h265 byte stream (caller-owned; the reference has no capacity argument either --
 *              header (<= 90 B) + 2 bytes per padded pixel is always enough, see DESIGN.md)
 *   img      : (*ysz) x (*xsz) 8-bit grayscale, row-major, stride *xsz
 *   img_rcon : receives the reconstruction, PADDED size, stride = padded width (HEVCe.c:1628); mandatory
 *   ysz,xsz  : in: picture size; out: size clamped to 8192 and rounded up to a multiple of 32 (HEVCe.c:1581-1582,
 *              1643-1644)
 *   qpd6     : 0..4 (QP = 6*qpd6 + 4)
 * returns the stream length in bytes (HEVCe.c:1646), or a negative HEVCE_ERR_* (the reference cannot fail; a
 * negative return is a compatible extension).  Re-entrant and thread-safe like the reference: concurrent callers each
 * get their own device session (up to four are cached per device), and the caller's current CUDA device is restored.
 */
HEVCE_API int HEVCImageEncoder(unsigned char *pbuffer, const unsigned char *img, unsigned char *img_rcon,
                     int *ysz, int *xsz, const int qpd6);

/*
 * New: n independent pictures in one call; per-picture semantics identical to n calls of HEVCImageEncoder
 * (including the clamp / pad / size write-back).  Pictures may differ in size and qpd6.  The batch is sharded
 * over the selected GPUs by cumulative CTU count, one host thread per device, no collective (pictures are
 * independent; SURVEY.md section 8e).  stream_len[i] receives the length of stream i.
 * returns 0, or a negative HEVCE_ERR_*.
 */
HEVCE_API int HEVCImageEncoderBatch(int n, unsigned char *const *pbuffers, const unsigned char *const *imgs,
                          unsigned char *const *img_rcons, int *ysz, int *xsz, const int *qpd6, int *stream_len);

/* ---- extensions used by the benchmark harness and the multi-process launcher ------------------------------ */

/* Restrict the library to `count` CUDA device ordinals (default: every visible device; the environment
 * variable HEVCE_DEVICES="0,3" does the same).  returns 0 or HEVCE_ERR_*. */
HEVCE_API int hevce_set_devices(int count, const int *ordinals);

/* Size limit applied by the clamp (default 8192 = the reference's MAX_YSZ / MAX_XSZ, HEVCe.c:62-63).  Values up to
 * 16384 reproduce a reference build whose two limits were raised; returns the previous value. */
HEVCE_API int hevce_set_max_dim(int max_dim);
HEVCE_API int hevce_get_max_dim(void);   /* the limit in force; a call captures it once on entry (size output buffers from it) */

/* Free the sessions the library caches between calls (HBM buffers, pinned staging).  Sessions a running call is
 * using stay.  The reference allocates nothing, so it has no counterpart. */
HEVCE_API void hevce_release(void);

/* Kernel variant for the batches configured from now on.  The decision kernel is linked in six variants of the same
 * source: "g7" / "g4" / "g2" = 7 / 4 / 2 same-size pictures per CTA in lock-step (throughput), "w1" = one picture per
 * CTA with all its threads and nearly all shared memory of the SM, "t1" = one picture per CTA whose threads form three
 * tracks so that a 16x16 / 32x32 node's own candidates are evaluated while its children are decided, "c2" = the same
 * tracks on a cluster of two CTAs (two SMs per picture, state exchanged through distributed shared memory; latency: few
 * or large pictures).  NULL, "" or
 * "auto" (default; also the environment variable HEVCE_VARIANT) chooses per batch.  Every variant produces the same
 * bytes.  returns 0, or HEVCE_ERR_ARG for an unknown name. */
HEVCE_API int hevce_set_variant(const char *name);

/* Device-resident session: buffers for a fixed list of pictures on ONE device.  Lets a caller keep inputs in HBM
 * and time the encode kernel alone (bench.py `value`), or overlap its own copies. */
typedef struct hevce_session hevce_session;
HEVCE_API hevce_session *hevce_session_create(int device, int n, const int *ysz, const int *xsz, const int *qpd6);
HEVCE_API int  hevce_session_upload(hevce_session *s, const unsigned char *const *imgs);      /* host -> HBM (pinned staging) */
HEVCE_API int  hevce_session_encode(hevce_session *s);                                        /* decision + commit kernels, synchronous */
HEVCE_API int  hevce_session_download(hevce_session *s, unsigned char *const *pbuffers, unsigned char *const *img_rcons,
                            int *stream_len);                                       /* HBM -> host */
HEVCE_API float hevce_session_kernel_ms(const hevce_session *s);   /* CUDA-event duration of the last hevce_encode_kernel launch */
HEVCE_API float hevce_session_commit_ms(const hevce_session *s);   /* ... of the hevce_commit_kernel launch that follows it */
HEVCE_API int  hevce_session_launches(const hevce_session *s);     /* kernel launches issued so far by this session */
HEVCE_API int  hevce_session_grid(const hevce_session *s);         /* CTAs of the persistent encode grid */
HEVCE_API const char *hevce_session_variant(const hevce_session *s); /* kernel variant chosen for the configured batch */
/* Per-picture quality of the last encode, reduced on the device: mean squared error and PSNR between source and
 * reconstruction over the area both cover, MSE floored at 1e-9 (calcImagePSNR, HEVCeMain.c:116-133, printed by the
 * reference CLI at HEVCeMain.c:201-212).  mse / psnr: n doubles each, either may be NULL.  HEVCE_ERR_STATE before the
 * first hevce_session_encode of the uploaded pictures (the same holds for hevce_session_partition). */
HEVCE_API int  hevce_session_quality(hevce_session *s, double *mse, double *psnr);
HEVCE_API float hevce_session_quality_ms(const hevce_session *s);  /* CUDA-event duration of the last hevce_quality_kernel launch */
/* Decisions of picture i of the last encode as raster maps: CU size (8/16/32) and luma intra mode (0..34) per 4x4 unit,
 * (H/4)*(W/4) bytes each; CU kind per 8x8 unit, (H/8)*(W/8) bytes: 0 = one TU, 1 = four TUs, 2 = NxN (what the
 * reference keeps in map_cu_sz_0 / map_pmode_0, HEVCe.c:1591-1592, plus the transform split).  Any pointer may be NULL. */
HEVCE_API int  hevce_session_partition(hevce_session *s, int i, unsigned char *cu_size, unsigned char *mode, unsigned char *kind);
HEVCE_API long long hevce_session_h2d_bytes(const hevce_session *s);
HEVCE_API long long hevce_session_d2h_bytes(const hevce_session *s);
HEVCE_API void hevce_session_destroy(hevce_session *s);

/* Integer-issue peak of the device: a dependency-free IMAD/LOP3 micro-benchmark; returns int-ops/s (IMAD = 2 ops),
 * or a negative HEVCE_ERR_*.  Used as the roofline denominator companion (SURVEY.md section 8d). */
HEVCE_API double hevce_measure_int_peak(int device);

HEVCE_API const char *hevce_version(void);

#ifdef __cplusplus
}
#endif
#endif
