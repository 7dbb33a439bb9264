/* hevce_variants.h -- private: the kernel variants linked into libhevce_b200.so (see hevce_variant.cu, Makefile). */
#ifndef HEVCE_VARIANTS_H
#define HEVCE_VARIANTS_H

typedef struct hevce_variant_info {
    int gang;                  /* pictures per CTA                                   */
    int threads_per_picture;   /* CTA size = gang * threads_per_picture              */
    int lanes_per_warp;        /* trial-coder lanes hosted by one warp               */
    int wide;                  /* 1: one picture per CTA with the large pool         */
    int tracks;                /* thread tracks per picture (3 = parent || child)    */
    int cluster;               /* CTAs (SMs) per picture: 1, or 2 = tracks on a cluster */
    long long smem_bytes;      /* dynamic shared memory per CTA                      */
} hevce_variant_info;

/* tag, relative time per CTU of one gang when the whole GPU runs this variant: measured on B200 (qpd6=2, 148 gangs of
 * 64x64 pictures, 74 for c2; profiles/r2_variant_latency.log, r2_variant_latency_c2.log), ms per CTU of one gang beside it.
 * A variant's shape is set only by its VDEF_<tag> line in csrc/Makefile; hevce_variant_info_<tag>() reports it. */
#define HEVCE_VARIANT_LIST(X) \
    X(g7, 1.00) /* 8.63 */    \
    X(g4, 0.74) /* 6.38 */    \
    X(g2, 0.63) /* 5.42 */    \
    X(w1, 0.54) /* 4.65 */    \
    X(t1, 0.52) /* 4.46 */    \
    X(c2, 0.30) /* 2.61 */

#ifdef __cplusplus
extern "C" {
#endif
#define HEVCE_DECLARE_VARIANT(tag, cost)                                                                                 \
    int hevce_variant_prepare_##tag(void);                                                                               \
    int hevce_variant_launch_##tag(const void *jobs, const int *gangs, int ngangs, const void *slots, int *counter,      \
                                   const void *tables, int grid, void *stream);                                          \
    void hevce_variant_info_##tag(hevce_variant_info *out);                                                              \
    void hevce_variant_profile_##tag(unsigned long long *cycles, unsigned long long *count);
HEVCE_VARIANT_LIST(HEVCE_DECLARE_VARIANT)
#undef HEVCE_DECLARE_VARIANT
#ifdef __cplusplus
}
#endif
#endif
