// hevce_core.h -- the HEVC intra still-image encoder of this repository: every stage of the hot path
// (reference samples, 35 predictors, integer transforms, simplified RDOQ, reconstruction, CABAC trial coding,
// CU quadtree decision, bitstream commit) as code for ONE CTA that encodes ONE picture.
//
// The file is compiled by nvcc into the sm_100a kernel (hevce_variant.cu).  It contains no CPU fallback: the
// product library only ever runs it on the GPU.  For development the same source is also compiled by g++ into a
// single-threaded *simulator* of the CTA (tests/sim/, test infrastructure only), where every PAR_FOR phase runs
// its work items in a permuted order; bit-exactness under permutation shows the phases are race-free.
//
// Execution model ("bulk-synchronous phases", one CTA = one picture):
//   * CTUs in raster order, CUs in z-order: the CABAC state threads through the whole picture, so this order is
//     forced (SURVEY.md section 7.3-1); the parallel axes are the candidates of a CU node and the batch;
//   * pixel pipeline: the candidates of a node (35 modes x {one TU, four TUs, NxN PU}) are processed together in
//     four phases whose work items are (candidate, line): A = predict + residual + forward column transform,
//     B = forward row transform + RDOQ, C = coefficient-group zero-out + dequantisation + inverse column transform,
//     D = inverse row transform + reconstruction + SSE.  All blocks live in shared memory (padded, conflict-free
//     for both row and column items); only the final levels and reconstructions go to a per-slot L2-resident store;
//   * entropy trials: one lane per candidate runs a private arithmetic coder (full integer state incl. the
//     emulation-prevention bookkeeping, no byte store) from the node snapshot, reading levels one 4x4 group at a time;
//   * thread 0 takes the arg-min with the reference's "last minimum wins" order, the CTA copies the winner's
//     reconstruction / levels / coder state into the live state;
//   * after each CTU the decided tree is re-encoded once by a byte-writing coder (commit pass).
//
// Behavioural parity target: /root/reference/src/HEVCe.c (cited as HEVCe.c:NNN).  Written from scratch.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define HEVCE_HD __host__ __device__
#define HEVCE_NOINLINE __noinline__
#else
#define HEVCE_HD
#define HEVCE_NOINLINE __attribute__((noinline))
#endif

// tuning switches: tools/ab_variants.py builds A/B variants of the library with other values of them
// Consecutive bypass strings of one syntax element coded by ONE put_bypass call (the reference issues one call per bit of
// the last-position suffixes and two per escape level, HEVCe.c:1076-1086, 1154-1169).  Exact for everything observable:
// bypass coding is linear (low = low * 2^n + range * bits) and a byte leaves the window whenever fewer than 12 bits of
// headroom remain, whatever the grouping, so the bytes, their count (the rate, emulation prevention included) and
// {range, nbits} are the same; only WHEN a carry reaches the pending byte can differ (it may still sit in `low` where the
// call-for-call coder has already added it).  Trial and commit coders use the same grouping, so their states still have
// to agree exactly.  tests/test_stages.py: random sequences in both groupings give identical byte streams; the
// call-for-call build equals the reference's putCoef state field by field; measured -5 % kernel time (g7).
#ifndef HEVCE_OPT_BYPMERGE
#define HEVCE_OPT_BYPMERGE 1
#endif
// bit-fields of a coefficient group built two levels at a time (signs gathered by shift + mask, the non-zero mask squeezed
// out of the class field) instead of level by level: 100 instead of 159 instructions per group.  Measured (profiles/
// r2_ab_fastbuild_*.log): -0.7 % on the one-picture-per-CTA cluster variant, +0.6 % on the 7-picture gang, where the longer
// live ranges cost spills at the 72-register cap -- so it is on for the variants with one picture per CTA only.
#ifndef HEVCE_OPT_FASTBUILD
#define HEVCE_OPT_FASTBUILD (HEVCE_OPT_GANG == 1)
#endif
// ---- kernel variant (one translation unit per variant, see hevce_variant.cu): pictures per CTA, threads per picture,
// trial lanes per warp and the pool plan.  GANG x NT threads run in lock-step phases; WIDE = one picture owns the CTA
// and most of the SM's shared memory (all 35 candidates of a 16x16 / 32x32 step in one round).  Measured on B200
// (888 x 64x64, qpd6=2): GANG 6 (80 regs) = GANG 5 (96 regs) > GANG 4 by 12 %; GANG 7 (72 regs, possible since the
// context sets shrank to 26 words) 5.7 % more pictures per second per SM than GANG 6.
#ifndef HEVCE_OPT_GANG
#define HEVCE_OPT_GANG 7
#endif
#ifndef HEVCE_OPT_NT
#define HEVCE_OPT_NT 128
#endif
#ifndef HEVCE_OPT_LPW      // trial-coder lanes per warp: 32 = packed (issue-bound gangs), small = spread (latency-bound)
#define HEVCE_OPT_LPW 32
#endif
#ifndef HEVCE_OPT_WIDE
#define HEVCE_OPT_WIDE 0
#endif
#ifndef HEVCE_OPT_TRACKS   // 1: parent || child -- a picture's threads split into three tracks: the 8x8 chain, the 16x16
#define HEVCE_OPT_TRACKS 0 //    nodes' own candidates, the 32x32 node's own candidates (HEVCE_OPT_TRK_C threads + 2 equal halves of the rest)
#endif
#ifndef HEVCE_OPT_TRK_C
#define HEVCE_OPT_TRK_C HEVCE_OPT_NT
#endif
#ifndef HEVCE_OPT_CLUSTER  // 2: the tracks of a picture on a thread-block cluster of two CTAs (two SMs): rank 0 = track 0 with all
#define HEVCE_OPT_CLUSTER 0 //   its threads, rank 1 = tracks 1 and 2 with half each; state crosses through distributed shared memory
#endif
#ifndef HEVCE_OPT_LPW_P    // trial lanes per warp on the two parent tracks
#define HEVCE_OPT_LPW_P HEVCE_OPT_LPW
#endif
#ifndef HEVCE_NS
#define HEVCE_NS hevce
#endif

namespace HEVCE_NS {

typedef uint8_t u8;
typedef int16_t s16;
typedef uint32_t u32;

// ------------------------------------------------------------------------------------------------------------
// sizes
// ------------------------------------------------------------------------------------------------------------
constexpr int CTU = 32;
constexpr int NT = HEVCE_OPT_NT;   // threads per picture (a multiple of 64)
constexpr int GANG = HEVCE_OPT_GANG;            // pictures per CTA (lock-step groups of NT threads)
constexpr int LPW = HEVCE_OPT_LPW;
constexpr bool WIDE = HEVCE_OPT_WIDE != 0;
// Tracks (parent || child, SURVEY.md section 7.3-1: a node's own candidates depend only on its entry snapshot and on
// samples outside the CU, so they can be evaluated while its children run; only the final ">=" waits): track 0 = the
// 8x8 nodes plus every decision / adoption, track 1 = the candidates of the 16x16 nodes, track 2 = those of the 32x32 node.
constexpr bool TRACKS = HEVCE_OPT_TRACKS != 0;
constexpr int NTRACK = TRACKS ? 3 : 1;
constexpr bool CLUSTER = HEVCE_OPT_CLUSTER != 0;          // tracks on the two CTAs of a cluster (NT threads each)
constexpr int TRK_C = CLUSTER ? NT : TRACKS ? HEVCE_OPT_TRK_C : NT;      // threads of track 0
constexpr int TRK_P = CLUSTER ? NT / 2 : TRACKS ? (NT - TRK_C) / 2 : 0;  // threads of track 1 and of track 2
constexpr int LPW_P = HEVCE_OPT_LPW_P;
constexpr int NTA = (TRK_C / 2) / 32 * 32, NTB = TRK_C - NTA;   // the two thread teams of track 0 on 8x8 nodes: [0, NTA) and [NTA, TRK_C)
static_assert(NT % 32 == 0 && NTA >= 32 && LPW >= 1 && LPW <= 32 && LPW_P >= 1 && LPW_P <= 32, "bad kernel variant");
static_assert(!TRACKS || (GANG == 1 && TRK_C % 64 == 0 && TRK_P % 32 == 0 && TRK_P >= 96 && TRK_C + 2 * TRK_P == (CLUSTER ? 2 * NT : NT)), "bad track split");
static_assert(!CLUSTER || TRACKS, "the cluster variant is a track variant");
HEVCE_HD inline int trk_of_tid(int tid) { return (!TRACKS || tid < TRK_C) ? 0 : tid < TRK_C + TRK_P ? 1 : 2; }
HEVCE_HD inline int trk_t0(int t) { return CLUSTER ? (t == 2 ? TRK_P : 0) : t == 0 ? 0 : t == 1 ? TRK_C : TRK_C + TRK_P; }   // first thread of the track in its CTA
HEVCE_HD inline int trk_size(int t) { return t == 0 ? TRK_C : TRK_P; }
HEVCE_HD inline int trk_lpw(int t) { return t == 0 ? LPW : LPW_P; }
template <int S> struct TrackOf { static constexpr int value = !TRACKS ? 0 : S == 8 ? 0 : S == 16 ? 1 : 2; };
constexpr int NTC = 128;           // threads per block of the commit kernel (one CTU each)
constexpr int NLANE = 70;          // trial-coder lanes with a private context set (the 35 NxN-PU lanes reuse 0..34)
constexpr int NCAND = 105;         // trial-coder lanes of a CU node: 35 one-TU + 35 four-TU + 35 NxN-PU candidates
constexpr int NMODE = 35;
constexpr int NCTX = 91;           // context bytes: the contexts of HEVCe.c:745-759 that a luma-only intra stream can touch
constexpr int CTXW = 23;           // context words per lane (odd: lane-major context sets of consecutive lanes start in different banks)
constexpr int CTXW4 = 9;           // leading words that hold every context a 4x4 luma TU's residual can touch
constexpr int WP = 65;             // pitch of the CTU reconstruction window (row 0 / col 0 = neighbours)
constexpr int IMAX = 0x7fffffff;

// Compact layout (the reference struct also carries the chroma contexts, 142 bytes).  What the residual of a 4x4 luma TU
// touches comes first, so an NxN PU lane initialises words 0..CTXW4-1 only: last_x of 4x4 TUs 0-2, last_y of 4x4 TUs 3-5,
// greater1 6-21 (4 sets x 4), greater2 22-25, sig_coeff 26-52 (27 luma; 4x4 TUs use the first 9); then split_cu 53-55,
// part 56, luma mode 57, chroma mode 58, split_tu 59-61, cbf_luma 62-63, cbf_chroma 64, coded_sub_block 65-66, last_x of
// 8x8 / 16x16 / 32x32 TUs 67-69 / 70-73 / 74-78 (only the 3 / 4 / 5 contexts a TU size can reach, HEVCe.c:1046-1075),
// last_y 79-81 / 82-85 / 86-90.
enum { CX_LASTX4 = 0, CX_LASTY4 = 3, CX_ONE = 6, CX_ABS = 22, CX_SIG = 26, CX_SPLIT_CU = 53, CX_PART = 56, CX_YPM = 57, CX_UVPM = 58,
       CX_SPLIT_TU = 59, CX_YCBF = 62, CX_UVCBF = 64, CX_SIGCG = 65, CX_LASTX = 67, CX_LASTY = 79 };
// first last_x / last_y context of a TU of size 4 << row
HEVCE_HD inline int cx_lastx(int row) { return row == 0 ? CX_LASTX4 : row == 1 ? CX_LASTX : row == 2 ? CX_LASTX + 3 : CX_LASTX + 7; }
HEVCE_HD inline int cx_lasty(int row) { return row == 0 ? CX_LASTY4 : row == 1 ? CX_LASTY : row == 2 ? CX_LASTY + 3 : CX_LASTY + 7; }

HEVCE_HD inline int imin(int a, int b) { return a < b ? a : b; }
HEVCE_HD inline int imax(int a, int b) { return a > b ? a : b; }
HEVCE_HD inline int iclip(int v, int lo, int hi) { return imin(imax(v, lo), hi); }
HEVCE_HD inline int iabs(int v) { return v < 0 ? -v : v; }
HEVCE_HD inline int ilog2(int v) {   // v = 4, 8, 16, 32 -> 2..5
    return v == 4 ? 2 : v == 8 ? 3 : v == 16 ? 4 : 5;
}
HEVCE_HD inline int bitlen(unsigned v) {
#if defined(__CUDA_ARCH__)
    return 32 - __clz((int)v);
#else
    return v ? 32 - __builtin_clz(v) : 0;
#endif
}

// ------------------------------------------------------------------------------------------------------------
// constant tables (filled on the host by fill_tables(), copied to __constant__ and from there to shared memory)
// ------------------------------------------------------------------------------------------------------------
// bin4, sigp4 and rate32 have no reader, and lps4 / next_lps only feed st8.  They stay: dropping them moves the other
// fields, and that layout measured 0.2-0.6 % slower on the gang variants (profiles/r2_notes.md).
struct Tables {
    u32 lps4[64];          // rangeTabLps, one word per state: byte q = LPS range for (range>>6)&3 == q  (HEVCe.c:704-713)
    u8 next_lps[128];      // (state<<1|mps) after an LPS                   (HEVCe.c:702)
    unsigned long long st8[128];   // per ctx = state<<1|mps: bytes 0..3 LPS range by range quarter, byte 4 ctx after an LPS, byte 5 after an MPS
    u32 bin4[4 + 512];     // [4 + ctx*4 + q], ctx = state<<1|mps, q = (range>>6)&3 (range>>6 is 4..7, hence the 4 unused words in front):
                           // byte 0 LPS range, byte 1 ctx after an LPS, byte 2 ctx after an MPS, bits 29..31 LPS renorm shift (HEVCe.c:701-715)
    u8 ctx_iv[4 * CTXW];   // context init values by (compact) context index    (HEVCe.c:763-777)
    u8 scan4[3][16];       // in-CG scan, (y<<2)|x : diag / horizontal / vertical
    u8 inv4[3][16];        // inverse: raster index (y<<2)|x -> scan index
    unsigned long long sigoff[3][4];   // sig_coeff ctx offset (4 bits per scan index) by neighbour pattern (HEVCe.c:1116-1121)
    unsigned long long sig4[3];   // sig_coeff ctx of 4x4 TUs (4 bits per scan index)
    u8 cgdiag[3][64];      // diagonal CG order for 2x2 / 4x4 / 8x8 CG grids, (cy<<3)|cx
    u8 sigp4[16];          // sig_coeff ctx for 4x4 TUs                     (HEVCe.c:1093)
    u8 grp[32];            // last-position group index                     (HEVCe.c:1047)
    u8 gmin[12];           // first position of a group                     (HEVCe.c:1048)
    int rate32[32];        // RDOQ rate estimate of levels 0..31                (HEVCe.c:526-535)
    int drate[8];          // rate(l) - rate(l-1) for l = 1..6; [7] = 0: from 7 on the step is 65536 when l-5 is a power of two, else 0
};

inline void fill_tables(Tables& t) {
    static const u8 LPS[64][4] = {
        {128, 176, 208, 240}, {128, 167, 197, 227}, {128, 158, 187, 216}, {123, 150, 178, 205}, {116, 142, 169, 195},
        {111, 135, 160, 185}, {105, 128, 152, 175}, {100, 122, 144, 166}, {95, 116, 137, 158},  {90, 110, 130, 150},
        {85, 104, 123, 142},  {81, 99, 117, 135},   {77, 94, 111, 128},   {73, 89, 105, 122},   {69, 85, 100, 116},
        {66, 80, 95, 110},    {62, 76, 90, 104},    {59, 72, 86, 99},     {56, 69, 81, 94},     {53, 65, 77, 89},
        {51, 62, 73, 85},     {48, 59, 69, 80},     {46, 56, 66, 76},     {43, 53, 63, 72},     {41, 50, 59, 69},
        {39, 48, 56, 65},     {37, 45, 54, 62},     {35, 43, 51, 59},     {33, 41, 48, 56},     {32, 39, 46, 53},
        {30, 37, 43, 50},     {29, 35, 41, 48},     {27, 33, 39, 45},     {26, 31, 37, 43},     {24, 30, 35, 41},
        {23, 28, 33, 39},     {22, 27, 32, 37},     {21, 26, 30, 35},     {20, 24, 29, 33},     {19, 23, 27, 31},
        {18, 22, 26, 30},     {17, 21, 25, 28},     {16, 20, 23, 27},     {15, 19, 22, 25},     {14, 18, 21, 24},
        {14, 17, 20, 23},     {13, 16, 19, 22},     {12, 15, 18, 21},     {12, 14, 17, 20},     {11, 14, 16, 19},
        {11, 13, 15, 18},     {10, 12, 15, 17},     {10, 12, 14, 16},     {9, 11, 13, 15},      {9, 11, 12, 14},
        {8, 10, 12, 14},      {8, 9, 11, 13},       {7, 9, 11, 12},       {7, 9, 10, 12},       {7, 8, 10, 11},
        {6, 8, 9, 11},        {6, 7, 9, 10},        {6, 7, 8, 9},         {2, 2, 2, 2}};
    static const u8 TRANS_LPS[64] = {0,  0,  1,  2,  2,  4,  4,  5,  6,  7,  8,  9,  9,  11, 11, 12, 13, 13, 15, 15, 16, 16,
                                     18, 18, 19, 19, 21, 21, 22, 22, 23, 24, 24, 25, 26, 26, 27, 27, 28, 29, 29, 30, 30, 30,
                                     31, 32, 32, 33, 33, 33, 34, 34, 35, 35, 35, 36, 36, 36, 37, 37, 37, 38, 38, 63};
    static const u8 HEAD[16] = {139, 141, 157, 184, 184, 63, 153, 138, 138, 111, 141, 94, 138, 182, 154, 154};
    static const u8 LAST[25] = {110, 110, 124, 0, 0, 125, 140, 153, 0, 0, 125, 127, 140, 109, 0, 111, 143, 127, 111, 79, 108, 123, 63, 154, 0};
    static const u8 SIG[44] = {111, 111, 125, 110, 110, 94, 124, 108, 124, 107, 125, 141, 179, 153, 125, 107, 125, 141, 179, 153, 125, 107,
                               125, 141, 179, 153, 125, 141, 140, 139, 182, 182, 152, 136, 152, 136, 153, 136, 139, 111, 136, 139, 111, 111};
    static const u8 ONE[24] = {140, 92, 137, 138, 140, 152, 138, 139, 153, 74, 149, 92, 139, 107, 122, 152, 140, 179, 166, 182, 140, 227, 122, 197};
    static const u8 ABSV[6] = {138, 153, 136, 167, 152, 152};
    static const u8 P4[16] = {0, 1, 4, 5, 2, 3, 4, 5, 6, 6, 8, 8, 7, 7, 8, 8};
    static const u8 GMIN[12] = {0, 1, 2, 3, 4, 6, 8, 12, 16, 24, 0, 0};
    for (int s = 0; s < 64; s++) t.lps4[s] = (u32)LPS[s][0] | ((u32)LPS[s][1] << 8) | ((u32)LPS[s][2] << 16) | ((u32)LPS[s][3] << 24);
    for (int s = 0; s < 64; s++)
        for (int m = 0; m < 2; m++) t.next_lps[(s << 1) | m] = (u8)((TRANS_LPS[s] << 1) | (s == 0 ? !m : m));
    for (int v = 0; v < 128; v++) {
        const unsigned long long nmps = v < 124 ? v + 2 : v;
        t.st8[v] = (unsigned long long)t.lps4[v >> 1] | ((unsigned long long)t.next_lps[v] << 32) | (nmps << 40);
    }
    for (int i = 0; i < 4; i++) t.bin4[i] = 0;
    for (int v = 0; v < 128; v++)
        for (int q = 0; q < 4; q++) {
            const u32 lps = LPS[v >> 1][q], nb = lps < 8 ? 6 : 9 - bitlen(lps), nmps = v < 124 ? v + 2 : v;
            t.bin4[4 + v * 4 + q] = lps | ((u32)t.next_lps[v] << 8) | (nmps << 16) | (nb << 29);
        }
    // the init tables are in the reference's order (luma entries first in every group); only the luma part is kept
    for (int i = 0; i < 4 * CTXW; i++) t.ctx_iv[i] = 154;
    for (int i = 0; i < 12; i++) t.ctx_iv[CX_SPLIT_CU + i] = HEAD[i];   // split_cu .. cbf_chroma keep the reference's order
    for (int row = 0; row < 4; row++)
        for (int i = 0; i < (row < 2 ? 3 : row + 2); i++) t.ctx_iv[cx_lastx(row) + i] = t.ctx_iv[cx_lasty(row) + i] = LAST[5 * row + i];
    t.ctx_iv[CX_SIGCG] = 91;
    t.ctx_iv[CX_SIGCG + 1] = 171;
    for (int i = 0; i < 27; i++) t.ctx_iv[CX_SIG + i] = SIG[i];
    for (int i = 0; i < 16; i++) t.ctx_iv[CX_ONE + i] = ONE[i];
    for (int i = 0; i < 4; i++) t.ctx_iv[CX_ABS + i] = ABSV[i];
    // scans: up-right diagonal / raster / column-major, same pattern inside a CG and over the CG grid (HEVCe.c:1128-1132)
    for (int type = 0; type < 3; type++) {
        int n = 0;
        if (type == 1) { for (int y = 0; y < 4; y++) for (int x = 0; x < 4; x++) t.scan4[type][n++] = (u8)((y << 2) | x); }
        else if (type == 2) { for (int x = 0; x < 4; x++) for (int y = 0; y < 4; y++) t.scan4[type][n++] = (u8)((y << 2) | x); }
        else for (int d = 0; d < 7; d++) for (int y = d < 3 ? d : 3; y >= 0; y--) { int x = d - y; if (x < 4) t.scan4[type][n++] = (u8)((y << 2) | x); }
    }
    for (int type = 0; type < 3; type++) {
        t.sig4[type] = 0;
        for (int k = 0; k < 16; k++) {
            const int p4 = t.scan4[type][k], py = p4 >> 2, px = p4 & 3;
            t.inv4[type][p4] = (u8)k;
            t.sig4[type] |= (unsigned long long)P4[p4] << (4 * k);
        }
        for (int pat = 0; pat < 4; pat++) {
            unsigned long long w = 0;
            for (int k = 0; k < 16; k++) {
                const int p4 = t.scan4[type][k], py = p4 >> 2, px = p4 & 3;
                const int tt = pat == 0 ? py + px : pat == 1 ? 2 * py : 2 * px;
                const unsigned long long off = pat == 3 ? 2u : (tt == 0 ? 2u : tt < 3 ? 1u : 0u);
                w |= off << (4 * k);
            }
            t.sigoff[type][pat] = w;
        }
    }
    for (int g = 0; g < 3; g++) {
        int ncg = 2 << g, n = 0;
        for (int i = 0; i < 64; i++) t.cgdiag[g][i] = 0;
        for (int d = 0; d < 2 * ncg - 1; d++)
            for (int y = d < ncg - 1 ? d : ncg - 1; y >= 0; y--) { int x = d - y; if (x < ncg) t.cgdiag[g][n++] = (u8)((y << 3) | x); }
    }
    for (int i = 0; i < 16; i++) t.sigp4[i] = P4[i];
    for (int i = 0; i < 32; i++) t.grp[i] = (u8)(i < 4 ? i : i < 6 ? 4 : i < 8 ? 5 : i < 12 ? 6 : i < 16 ? 7 : i < 24 ? 8 : 9);
    for (int i = 0; i < 12; i++) t.gmin[i] = GMIN[i];
    for (int l = 0; l < 8; l++) t.drate[l] = l == 1 ? 70000 : l == 2 ? 20000 : l == 3 ? 2000 : l == 4 ? 65536 : (l == 5 || l == 6) ? 32768 : 0;
    for (int l = 0; l < 32; l++)
        t.rate32[l] = l == 0 ? 0 : l == 1 ? 70000 : l == 2 ? 90000 : l == 3 ? 92000 : l == 4 ? 157536 : l == 5 ? 190304 : 92000 + ((4 + 2 * (bitlen((unsigned)(l - 5)) - 1)) << 15);
}

// context initialisation for QP = 6*qpd6+4 (HEVCe.c:727-735)
HEVCE_HD inline u8 ctx_init_value(int iv, int q) {
    int qp = 6 * q + 4;
    int st = iclip(((((iv >> 4) * 5 - 45) * qp) >> 4) + ((iv & 15) << 3) - 16, 1, 126);
    return (u8)(st >= 64 ? ((st - 64) << 1) | 1 : (63 - st) << 1);
}

// ------------------------------------------------------------------------------------------------------------
// RD cost (HEVCe.c:177-185) -- saturating
// ------------------------------------------------------------------------------------------------------------
struct RdK { int wd, wb, ld, lb; };   // weights and the saturation limits IMAX/weight, fixed per picture
HEVCE_HD inline RdK rd_consts(int q) {
    RdK k;
    k.wd = q < 3 ? 11 : q == 3 ? 5 : 1;
    k.wb = q == 0 ? 1 : q == 1 ? 4 : q == 2 ? 16 : q == 3 ? 29 : 23;
    k.ld = q < 3 ? IMAX / 11 : q == 3 ? IMAX / 5 : IMAX;
    k.lb = q == 0 ? IMAX : q == 1 ? IMAX / 4 : q == 2 ? IMAX / 16 : q == 3 ? IMAX / 29 : IMAX / 23;
    return k;
}
HEVCE_HD inline int rd_cost(const RdK& k, int dist, int bits) {
    const int c1 = (k.ld <= dist) ? IMAX : k.wd * dist;
    const int c2 = (k.lb <= bits) ? IMAX : k.wb * bits;
    return (IMAX - c1 <= c2) ? IMAX : c1 + c2;
}

// ------------------------------------------------------------------------------------------------------------
// arithmetic coder (HEVCe.c:797-933).  One coder type serves trials (out == nullptr: full integer state including
// the emulation-prevention bookkeeping that can change the byte count, but no byte store) and the commit pass.
// ------------------------------------------------------------------------------------------------------------
struct Coder { int range, low, nbits, nbytes, held, z, n; };

HEVCE_HD inline void coder_reset(Coder& c) { c.range = 510; c.low = 0; c.nbits = 23; c.nbytes = 0; c.held = 0xff; c.z = 0; c.n = 0; }
HEVCE_HD inline int coder_len(const Coder& c) { return 8 * (c.n + c.nbytes) + 23 - c.nbits; }   // HEVCe.c:835
HEVCE_HD inline bool coder_equal(const Coder& a, const Coder& b) {
    return a.range == b.range && a.low == b.low && a.nbits == b.nbits && a.nbytes == b.nbytes && a.held == b.held && a.z == b.z && a.n == b.n;
}

template <bool EMIT>
struct BacT {
    Coder c;
    u8* out;            // EMIT only: destination of this CTU's bytes
    int cap;            // EMIT only: bytes available at out
    u32 tabs;           // device: shared-space address of Tables::st8, kept in a register (use_tables)

    // The bin table is read with an explicit ld.shared from an address the compiler cannot re-derive: left to itself it
    // rebuilds the shared-window base (S2UR + UMOV + ULEA) in front of every bin.
    HEVCE_HD void use_tables(const Tables& tb) {
#if defined(__CUDA_ARCH__)
        tabs = (u32)__cvta_generic_to_shared(&tb.st8[0]);
        asm volatile("mov.u32 %0, %0;" : "+r"(tabs));
#else
        (void)tb; tabs = 0;
#endif
    }

    HEVCE_HD void emit(int byte) {   // HEVCe.c:821-832
        const int b = byte & 0xff;
        if (EMIT) {
            if (c.z >= 2 && b <= 3) {
                if (c.n < cap) out[c.n] = 3;
                c.n++;
                c.z = 0;
            }
            if (c.n < cap) out[c.n] = (u8)b;
            c.n++;
            c.z = b ? 0 : c.z + 1;
        } else {   // trial: count only, branch-free
            const int epb = (c.z >= 2) & (b <= 3);
            c.n += 1 + epb;
            c.z = b ? 0 : (epb ? 1 : c.z + 1);
        }
    }
    HEVCE_HD void carry_out() {   // HEVCe.c:859-879
        if (c.nbits >= 12) return;
        const int lead = c.low >> (24 - c.nbits);
        c.nbits += 8;
        c.low &= (int)(0xFFFFFFFFu >> c.nbits);
        if (lead == 0xff) c.nbytes++;
        else if (c.nbytes > 0) {
            const int carry = lead >> 8;
            emit(c.held + carry);
            c.held = lead & 0xff;
            for (; c.nbytes > 1; c.nbytes--) emit((0xff + carry) & 0xff);
        } else { c.nbytes = 1; c.held = lead; }
    }
    HEVCE_HD void put_bin(const Tables& tb, int bin, u8& cx) { cx = (u8)bin_step(tb, bin, cx); }
    // one context-coded bin with context byte v; returns the new context byte (HEVCe.c:914-933, both branches computed, then selected)
    HEVCE_HD int bin_step(const Tables& tb, int bin, const int v) {
#if defined(__CUDA_ARCH__)
        u32 lo, hi;
        asm("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(lo), "=r"(hi) : "r"(tabs + (u32)v * 8u));
        // range >> 6 is 4..7: byte 0..3 of lo; the other selector nibbles are 0 and pick byte 0 of the zero operand.  Raw prmt:
        // __byte_perm first masks the selector (one more instruction on the range -> range recurrence).
        u32 lps_u;
        asm("prmt.b32 %0, %1, %2, %3;" : "=r"(lps_u) : "r"(0u), "r"(lo), "r"((u32)c.range >> 6));
        const int lps = (int)lps_u;
#else
        const u32 lo = (u32)tb.st8[v], hi = (u32)(tb.st8[v] >> 32);
        const int lps = (int)((lo >> (8 * ((c.range >> 6) & 3))) & 0xffu);
#endif
        const int rmps = c.range - lps;
        const bool is_lps = ((v ^ bin) & 1) != 0;                   // bin is 0 or 1 at every call site
        // renorm table, HEVCe.c:715: 9 - bitlen(lps) for lps >= 6; the only smaller entry (2, probability state 63) cannot
        // be reached: contexts are initialised to states 1..126 (ctx_init_value) and the MPS transition stops at 62
        const int sh = is_lps ? 9 - bitlen((unsigned)lps) : (rmps < 256 ? 1 : 0);
        if (is_lps) c.low += rmps;
        c.low = (int)((unsigned)c.low << sh);
        c.range = (is_lps ? lps : rmps) << sh;
        c.nbits -= sh;
        const int cxn = (int)((is_lps ? hi : hi >> 8) & 0xffu);
#if !defined(__CUDA_ARCH__)
        if (v >= 126 || (unsigned)bin > 1u || c.range < 256 || c.range > 510) __builtin_trap();
#endif
        carry_out();
        return cxn;
    }
    HEVCE_HD void put_bypass(int bins, int len) {   // HEVCe.c:899-911
        bins &= (1 << len) - 1;
        while (len > 0) {
            const int n = imin(len, 8);
            len -= n;
            const int chunk = (bins >> len) & ((1 << n) - 1);
            c.low = (int)(((unsigned)c.low << n) + (unsigned)(c.range * chunk));
            c.nbits -= n;
            carry_out();
        }
    }
    HEVCE_HD void put_terminate(int bin) {   // HEVCe.c:882-896
        c.range -= 2;
        if (bin) { c.low = (int)((unsigned)(c.low + c.range) << 7); c.range = 256; c.nbits -= 7; }
        else if (c.range < 256) { c.low = (int)((unsigned)c.low << 1); c.range <<= 1; c.nbits--; }
        carry_out();
    }
    HEVCE_HD void finish() {   // HEVCe.c:840-856
        int fill = 0;
        if ((c.low >> (32 - c.nbits)) > 0) { emit(c.held + 1); c.low -= 1 << (32 - c.nbits); }
        else { if (c.nbytes > 0) emit(c.held); fill = 0xff; }
        for (; c.nbytes > 1; c.nbytes--) emit(fill);
        const int t = (c.low >> 8) << c.nbits;
        emit(t >> 16); emit(t >> 8); emit(t);
    }
};
typedef BacT<false> Bac;        // trial coder: full integer state, no byte store
typedef BacT<true> BacCommit;   // commit coder: writes the CTU's bytes

// context set: 4 * CTXW contiguous bytes (lane-major in the shared-memory array of lane-private sets: CTXW is odd, so
// the sets of 32 consecutive lanes start in 32 different banks).  The base pointer is always derived from the picture's
// shared-memory block inside the function that uses it, so the accesses stay LDS/STS.
struct Cx {
    u8* p;
    HEVCE_HD u8& operator[](int k) const { return p[k]; }
};

// ------------------------------------------------------------------------------------------------------------
// syntax elements (HEVCe.c:943-1340)
// ------------------------------------------------------------------------------------------------------------
HEVCE_HD inline void mpm_list(int l, int a, int (&m)[3]) {   // HEVCe.c:958-977
    if (l != a) { m[0] = l; m[1] = a; m[2] = (l != 0 && a != 0) ? 0 : (l + a < 2) ? 26 : 1; }
    else if (l > 1) { m[0] = l; m[1] = ((l + 29) % 32) + 2; m[2] = ((l - 1) % 32) + 2; }
    else { m[0] = 0; m[1] = 1; m[2] = 26; }
}

HEVCE_HD inline int scan_type(int s, int m) {   // HEVCe.c:1134-1150
    if (s <= 8) { if (iabs(m - 26) <= 4) return 1; if (iabs(m - 10) <= 4) return 2; }
    return 0;
}

// ------------------------------------------------------------------------------------------------------------
// transforms
// ------------------------------------------------------------------------------------------------------------
#include "hevce_xform_gen.h"

template <int T> struct Xf;
template <> struct Xf<4>  { static HEVCE_HD void f(const int (&x)[4], int (&y)[4]) { fdst4(x, y); }   static HEVCE_HD void i(const int (&x)[4], int (&y)[4]) { idst4(x, y); } };
template <> struct Xf<8>  { static HEVCE_HD void f(const int (&x)[8], int (&y)[8]) { fdct8(x, y); }   static HEVCE_HD void i(const int (&x)[8], int (&y)[8]) { idct8(x, y); } };
template <> struct Xf<16> { static HEVCE_HD void f(const int (&x)[16], int (&y)[16]) { fdct16(x, y); } static HEVCE_HD void i(const int (&x)[16], int (&y)[16]) { idct16(x, y); } };
template <> struct Xf<32> { static HEVCE_HD void f(const int (&x)[32], int (&y)[32]) { fdct32(x, y); } static HEVCE_HD void i(const int (&x)[32], int (&y)[32]) { idct32(x, y); } };

HEVCE_HD inline int use_filtered(int s, int m) {   // HEVCe.c:274-280 (HEVC intraHorVerDistThres rule)
    if (s == 4 || m == 1) return 0;
    if (m == 0) return 1;
    const int d = imin(iabs(m - 10), iabs(m - 26));
    return d > (s == 8 ? 7 : s == 16 ? 1 : 0);
}

HEVCE_HD inline int intra_angle(int m) {   // HEVCe.c:282
    const int k = m < 18 ? m - 10 : m - 26;   // signed distance to pure HOR / VER
    const int a = iabs(k);
    const int v = a == 0 ? 0 : a == 1 ? 2 : a == 2 ? 5 : a == 3 ? 9 : a == 4 ? 13 : a == 5 ? 17 : a == 6 ? 21 : a == 7 ? 26 : 32;
    return (m < 18) ? (k < 0 ? v : -v) : (k < 0 ? -v : v);
}

// ------------------------------------------------------------------------------------------------------------
// picture-level state
// ------------------------------------------------------------------------------------------------------------
struct CtuRec {          // what the commit pass needs for one CTU (written by the decision kernel)
    Coder start, end;    // coder state before the CTU / after its terminate bin (and the final flush for the last CTU)
    int out_pos;         // byte offset of this CTU's bytes in the stream
    int last;            // 1: last CTU of the picture
    u8 ctx[4 * CTXW];    // contexts at CTU start
    u8 msz[84], mpm[84]; // neighbour maps after the CTU was decided ([1+uy][1+ux], 81 used)
    u8 kind[16];
};

// Decisions of one picture as raster maps (host side; hevce_session_partition and the simulator): CU size and luma
// intra mode per 4x4 unit, CU kind per 8x8 unit (0: one TU, 1: four TUs, 2: NxN)
inline void unpack_partition(const CtuRec* recs, int H, int W, u8* cu_size, u8* mode, u8* kind) {
    const int cw = W / CTU, w4 = W / 4, w8 = W / 8;
    for (int c = 0; c < (H / CTU) * cw; c++) {
        const CtuRec& r = recs[c];
        const int y4 = (c / cw) * 8, x4 = (c % cw) * 8;
        for (int i = 0; i < 64; i++) {
            if (cu_size) cu_size[(size_t)(y4 + i / 8) * w4 + x4 + i % 8] = r.msz[(1 + i / 8) * 9 + 1 + i % 8];
            if (mode) mode[(size_t)(y4 + i / 8) * w4 + x4 + i % 8] = r.mpm[(1 + i / 8) * 9 + 1 + i % 8];
        }
        if (kind)
            for (int i = 0; i < 16; i++) kind[(size_t)(y4 / 2 + i / 4) * w8 + x4 / 2 + i % 4] = r.kind[i];
    }
}

struct Job {
    CtuRec* recs;      // one record per CTU, raster order
    s16* levs;         // CTU*CTU final levels per CTU: CUs at their z-order offset, group-blocked
    const u8* img;     // source picture (device), stride src_w
    u8* rcon;          // reconstruction (device), H x W
    u8* out;           // bitstream (device)
    int* result;       // [0] = stream length, [1] = error flags
    int src_h, src_w;  // original size (clamp + stride, HEVCe.c:1622)
    int H, W;          // clamped + padded size (HEVCe.c:1581-1582)
    int q;             // qpd6
    int out_cap;
};

enum { ERR_OVERFLOW = 1, ERR_COMMIT_MISMATCH = 2 };
enum { P_BORDER, P_A, P_B, P_C, P_D_TRIAL, P_PU_ARGMIN, P_TRIAL, P_DECIDE, P_ADOPT, P_ENTER, P_LOAD, P_COMMIT, P_MISC, P_TA, P_TB_PIX, P_TB_CABAC, P_TB_ARGMIN, P_NTAGS };

constexpr int LEV_STRIDE = CTU * CTU;   // per-candidate level store (all TUs of the candidate)
constexpr int NREC = 70;                // candidates whose reconstruction is kept (one-TU + four-TU)

struct Scratch {       // per picture slot, global memory (L2-resident working set)
    s16* glev;         // [NCAND][LEV_STRIDE] final levels of every candidate of the current node (group-blocked)
    u8* grec;          // [NREC][CTU*CTU] reconstruction of every non-NxN candidate, CU-local raster
    u8* msz_line;      // CU-size map row of the CTU row above, W/4 entries
};

constexpr int POOL_BYTES = TRACKS ? 53248 : WIDE ? 189440 : 18624;
constexpr int AUX_CODER = POOL_BYTES - 1984;       // pool tail: trial-coder results (free whenever they are used)

struct Shared {
    // (field order as measured: moving the candidate arrays in front of the picture state cost the 7-picture variant 3 %)
    alignas(16) u8 pool[POOL_BYTES];    // per-node carve-up: work blocks, predictions, borders (see Plan<S>)        [track]
    u32 lane_ctx[NLANE * CTXW];         // lane-private context sets, lane-major (set L at word L * CTXW)            [track]
    // ---- the picture's state: owned by track 0; the cluster variant pushes [ctx0, ctu_lev) and q into the parent tracks' blocks
    alignas(16) u8 ctx0[4 * CTXW];      // freshly initialised contexts for this picture's qpd6
    alignas(16) u8 live_ctx[4 * CTXW];
    alignas(16) u8 snap_ctx[3][4 * CTXW];
    alignas(16) u8 nxn_ctx[4 * CTXW];
    alignas(16) s16 nxn_lev[4][16];
    u8 orig[CTU * CTU];
    u8 win[(CTU + 1) * WP];
    u8 msz[81], mpm[81];                // [1+uy][1+ux], 4x4 units; row 0 / col 0 = neighbours
    u8 kind[16];                        // per 8x8 unit: 0 one TU, 1 four TUs, 2 NxN
    Coder live, snap[3], nxn_coder;
    s16* ctu_lev;                       // level store of the current CTU (Job::levs + ctu*1024)                     [track 0]
    Scratch sc;                         // this track's global scratch (trial lanes may run on another picture's threads) [track]
    int q;                              // qpd6
    int cand_sse[NCAND], cand_bits[NCAND];   // cand_bits: trial bits; RD cost once a one-TU / four-TU lane has finished  [track]
    unsigned cgnz[NCAND][4];            // non-zero-group bitmaps: one-TU: [0],[1] = low/high word; else [tu]            [track]
    int nxn_pm[4], nxn_cost;            //                                                                           [track 0 from here]
    unsigned nxn_nz[4];
    int part_sse[CTU];
    int win_item;                       // decision of the current node: -1 keep split, 0..NREC-1 candidate, NCAND = NxN
    int stream_pos;
    int error;
    long long prof_last;
    Scratch sc_of[NTRACK];              // the scratch of every track (adoption reads the winner from the evaluating track's)
    unsigned rdv_seq[TRACKS ? 3 : 1];   // cluster variant: rendezvous sequence numbers written by the partner track
};

HEVCE_HD inline Coder* cand_coder(Shared& sm) { return (Coder*)(sm.pool + AUX_CODER); }

// Per-CTA control block behind the picture blocks and the tables: how many picture slots of the gang are live (a short
// gang leaves slots empty; their threads skip the picture and wait at the CTA barrier of the work queue).
struct GangCtl { int nlive; int next; };

// Shared-memory blocks.  Every track of every picture slot owns one `Shared` block (index slot * NTRACK + track): its
// pool, lane contexts, candidate results and scratch pointers are the track's; the picture-level fields (window,
// original, maps, live / snapshot coder state ...) are those of the picture's track-0 block (pic_sm()).  Non-inlined
// functions fetch the blocks through these accessors instead of taking reference parameters: the compiler then knows
// the address space and emits LDS/STS instead of generic loads.  The constant tables exist once per CTA, behind the blocks.
// Cluster variant: a CTA holds the blocks of ITS tracks only (rank 0: track 0; rank 1: tracks 1 and 2); every track works on
// its own block, whose picture-level fields are a mirror that track 0 pushes through distributed shared memory before it
// releases the track (push_picture_state); track 0 fetches a parent track's results the same way (decide_adopt).
#if defined(__CUDACC__)
constexpr int NBLOCK = CLUSTER ? 2 : GANG * NTRACK;           // blocks in one CTA's shared memory
HEVCE_HD inline int local_block(int slot, int trk) { return CLUSTER ? (trk == 2 ? 1 : 0) : slot * NTRACK + trk; }
#else   // the simulators keep all tracks' blocks of a picture side by side, also for the cluster variant
constexpr int NBLOCK = GANG * NTRACK;
HEVCE_HD inline int local_block(int slot, int trk) { return slot * NTRACK + trk; }
#endif
// the block that holds the picture-level state a thread of (slot, trk) works with
HEVCE_HD inline int picture_block(int slot, int trk) { return CLUSTER ? local_block(slot, trk) : local_block(slot, 0); }
#if defined(__CUDA_ARCH__)
extern __shared__ __align__(16) unsigned char hevce_smem[];
__device__ __forceinline__ int cluster_rank() { unsigned r = 0; if (CLUSTER) asm("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return (int)r; }
#define HEVCE_SLOT (CLUSTER ? 0 : (int)(threadIdx.x / NT))
#define HEVCE_PTID ((int)(threadIdx.x % NT))                       /* thread of the picture (cluster: of the CTA) */
#define HEVCE_TRK (CLUSTER ? (cluster_rank() == 0 ? 0 : ((int)threadIdx.x < TRK_P ? 1 : 2)) : trk_of_tid(HEVCE_PTID))
#define HEVCE_TID (HEVCE_PTID - trk_t0(HEVCE_TRK))                 /* thread of the track   */
__device__ __forceinline__ Shared& blk_sm(int b) { return reinterpret_cast<Shared*>(hevce_smem)[b]; }
// track t's block as seen from another CTA of the cluster (generic pointer into that CTA's shared memory)
__device__ __forceinline__ Shared* remote_blk(int t) {
    Shared* p = &blk_sm(local_block(0, t));
#if HEVCE_OPT_CLUSTER
    unsigned long long in = (unsigned long long)p, out;
    asm volatile("mapa.u64 %0, %1, %2;" : "=l"(out) : "l"(in), "r"(t == 0 ? 0 : 1));
    p = (Shared*)out;
#endif
    return p;
}
__device__ __forceinline__ void rdv_signal(unsigned* flag, unsigned v) {   // release everything this track wrote, then raise the partner's flag
    asm volatile("fence.acq_rel.cluster;\n\tst.release.cluster.u32 [%0], %1;" ::"l"(flag), "r"(v) : "memory");
}
__device__ __forceinline__ void rdv_wait(const unsigned* flag, unsigned v) {
    unsigned x;
    do { asm volatile("ld.acquire.cluster.u32 %0, [%1];" : "=r"(x) : "l"(flag) : "memory"); } while (x != v);
    asm volatile("fence.acq_rel.cluster;" ::: "memory");   // also drops this SM's L1 lines of the partner's global scratch
}
__device__ __forceinline__ Tables& my_tb() { return *reinterpret_cast<Tables*>(hevce_smem + NBLOCK * sizeof(Shared)); }
__device__ __forceinline__ GangCtl& gang_ctl() { return *reinterpret_cast<GangCtl*>(hevce_smem + NBLOCK * sizeof(Shared) + sizeof(Tables)); }
__device__ __forceinline__ int gang_live() { return GANG == 1 ? 1 : gang_ctl().nlive; }
#elif defined(__CUDACC__)
#define HEVCE_SLOT 0
#define HEVCE_PTID 0
#define HEVCE_TRK 0
#define HEVCE_TID 0
inline Shared& blk_sm(int) { return *static_cast<Shared*>(nullptr); }   // host pass of nvcc: declared, never executed
inline Shared* remote_blk(int) { return nullptr; }
inline int cluster_rank() { return 0; }
inline Tables& my_tb() { return *static_cast<Tables*>(nullptr); }
inline GangCtl& gang_ctl() { return *static_cast<GangCtl*>(nullptr); }
inline int gang_live() { return GANG; }
extern thread_local int g_sim_trk;   // the host pass parses the simulator macros below, it never runs them
#else
// simulators (tests/sim): HEVCE_SIM_GANG = one host thread per picture of a gang, HEVCE_SIM_TRACKS = one host thread
// per track of one picture, neither = one thread; real barriers between the host threads
extern Shared* g_sim_sms;                                            // NBLOCK blocks
extern Tables* g_sim_tb;
extern int g_sim_nlive;                                              // live pictures of the gang
extern thread_local int g_sim_member;                                // this thread's picture slot
extern thread_local int g_sim_trk;                                   // the track this thread is executing
void sim_barrier(int id, int parties);
#define HEVCE_SLOT g_sim_member
#define HEVCE_TRK g_sim_trk
inline Shared& blk_sm(int b) { return g_sim_sms[b]; }
inline Shared* remote_blk(int t) { return &g_sim_sms[local_block(0, t)]; }   // a "remote" block is just another one here
inline Tables& my_tb() { return *g_sim_tb; }
inline int gang_live() { return g_sim_nlive; }
#endif
#define my_sm() blk_sm(local_block(HEVCE_SLOT, HEVCE_TRK))             /* the executing track's block       */
#define pic_sm() blk_sm(picture_block(HEVCE_SLOT, HEVCE_TRK))          /* the picture-level state (cluster: this track's mirror) */
#define gang_sm(p) blk_sm(local_block((p), 0))                         /* picture p of the gang (track 0)   */
static_assert(AUX_CODER + NREC * (int)sizeof(Coder) <= POOL_BYTES, "pool tail too small");

// ---- thread <-> work mappings (shared by the kernel and the simulators) --------------------------------------------
// Teams: id 0 = all threads of the track, 1 = team A [0, NTA), 2 = team B [NTA, TRK_C) (track 0 only).
HEVCE_HD inline int team_t0(int id) { return id == 2 ? NTA : 0; }
HEVCE_HD inline int team_size(int id, int trk) { return id == 0 ? trk_size(trk) : id == 1 ? NTA : NTB; }
// first work item of track thread `tid` in a phase of team `id` whose item 0 sits on team thread `off` (mod team size);
// n when the thread is not in the team
HEVCE_HD inline int team_first(int tid, int trk, int id, int off, int n) {
    const int r = tid - team_t0(id);
    if (id == 0) return trk == 0 ? (r + TRK_C - off % TRK_C) % TRK_C : (r + TRK_P - off % (TRK_P ? TRK_P : 1)) % (TRK_P ? TRK_P : 1);
    if (id == 1) return (unsigned)r < (unsigned)NTA ? (r + NTA - off % NTA) % NTA : n;
    return (unsigned)r < (unsigned)NTB ? (r + NTB - off % NTB) % NTB : n;
}
// Trial-coder lanes: thread x of a linear thread space hosts lane (x/32)*lpw + x%32 when x%32 < lpw (lpw = 32: every
// thread hosts a lane, lanes packed into full warps; small lpw: few lanes per warp, less divergence per warp).
HEVCE_HD inline int host_lane(int x, int lpw) { return (x & 31) < lpw ? (x >> 5) * lpw + (x & 31) : -1; }
HEVCE_HD inline int lane_capacity(int nthreads, int lpw) { return (nthreads >> 5) * lpw; }
HEVCE_HD inline int round_lanes(int n, int lpw) { return (n + lpw - 1) / lpw * lpw; }   // next warp boundary in lane space
// team-B threads of the live pictures as one linear space: slot * NTB + (tid - NTA); -1 for team-A threads
HEVCE_HD inline int upper_index(int slot, int tid) { return tid >= NTA ? slot * NTB + tid - NTA : -1; }
// Items shared by the team-B threads that host none of the first `nlanes` lanes (whole warps); when every warp hosts a
// lane all team-B threads share them after their lane.  Returns the first item of linear team-B thread `ub`, sets stride.
HEVCE_HD inline int upper_free_first(int ub, int nlanes, int nlive, int n, int& stride) {
    const int nw = nlive * NTB / 32, hostw = imin((nlanes + LPW - 1) / LPW, nw);
    if (ub < 0) { stride = 1; return n; }
    if (hostw == nw) { stride = nw * 32; return ub; }
    stride = (nw - hostw) * 32;
    return ub >= hostw * 32 ? ub - hostw * 32 : n;
}
// barrier ids: 0 work queue (all threads of the CTA), 1 / 2 the teams of track 0, 3 all live threads, 4..6 one track,
// 7 / 8 rendezvous of track 0 with track 1 / 2
enum { BAR_TEAM_A = 1, BAR_TEAM_B = 2, BAR_PICTURES = 3, BAR_TRACK0 = 4, BAR_RDV1 = 7, BAR_RDV2 = 8 };

// work-item phases.  On the GPU a phase is a strided loop over the threads of a track (or team) followed by a barrier;
// in the simulators it is a loop over the items in a permuted order.
#if defined(__CUDA_ARCH__)
// A CTA holds up to GANG pictures of identical size, one per group of NT threads; the groups run the same phases in
// lock-step (barriers over the live pictures), so every warp of the SM executes the same code at the same time.
#define PAR_FOR(item, n) for (int item = HEVCE_TID, st_##item = trk_size(HEVCE_TRK); item < (n); item += st_##item)
#define PAR_FOR_ALL(item, n) for (int item = HEVCE_PTID; item < (n); item += NT)   /* all threads of the picture */
// threads of team `id` of the track only; item 0 starts at team thread `off`
#define PAR_FOR_TEAM(item, n, id, off) for (int item = team_first(HEVCE_TID, HEVCE_TRK, (id), (off), (n)), st_##item = team_size((id), HEVCE_TRK); item < (n); item += st_##item)
// 8x8 nodes split track 0 into two teams that run independent phase chains; a team's barrier spans the same team of
// all live pictures of the gang (their trial lanes are packed across pictures)
#define TEAM_A if (HEVCE_TID < NTA)
#define TEAM_B else
#define TEAM_JOIN() ((void)0)   // the track-wide barrier that follows is the join
#define HEVCE_BAR(id, cnt) asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(cnt) : "memory")
#define TEAM_SYNC(id) HEVCE_BAR(id, gang_live() * ((id) == 1 ? NTA : NTB))
// Trial-coder lanes of all live pictures, hosted by the track's threads (GANG_FOR) or by the team-B threads (GANG_FOR_UPPER)
#define GANG_RT (gang_live())
#define GANG_FOR(L, n) for (int L = host_lane(HEVCE_SLOT * trk_size(HEVCE_TRK) + HEVCE_TID, trk_lpw(HEVCE_TRK)), cap_ = lane_capacity(gang_live() * trk_size(HEVCE_TRK), trk_lpw(HEVCE_TRK)); (unsigned)L < (unsigned)(n); L += cap_)
#define GANG_FOR_UPPER(u, n) for (int u = HEVCE_TID >= NTA ? host_lane(upper_index(HEVCE_SLOT, HEVCE_TID), LPW) : -1, cap_ = lane_capacity(gang_live() * NTB, LPW); (unsigned)u < (unsigned)(n); u += cap_)
// the team-B threads that host none of the `first` lanes share n items of any picture of the gang
#define GANG_FOR_UPPER_FREE(it, first, n) for (int st_ = 1, it = upper_free_first(upper_index(HEVCE_SLOT, HEVCE_TID), (first), gang_live(), (n), st_); it < (n); it += st_)
// end of a phase: the threads of this track (of all live pictures); without tracks that is every live thread
#define PHASE_END() do { if (TRACKS) HEVCE_BAR(BAR_TRACK0 + HEVCE_TRK, gang_live() * trk_size(HEVCE_TRK)); else HEVCE_BAR(BAR_PICTURES, gang_live() * NT); } while (0)
// picture-wide phases (CTU load / store): every thread of the picture; in the cluster variant the threads of rank 0 (= track 0)
#define BAR_ALL() do { if (!CLUSTER) HEVCE_BAR(BAR_PICTURES, gang_live() * NT); else if (HEVCE_TRK == 0) PHASE_END(); } while (0)
#define PAR_FOR_ALL_OWNER (!CLUSTER || HEVCE_TRK == 0)
// Rendezvous of track 0 with parent track t (no-ops for the third track).  START: the node's entry snapshot exists, track t may
// evaluate the node's candidates; END: track t has finished, track 0 may decide.  One CTA: a named barrier over both tracks.
// Cluster: track 0 pushes the picture state into track t's block, then raises a flag in it (release / acquire at cluster
// scope, sequence numbers instead of resets); at the END track t raises a flag in track 0's block.
#define TRACK_START(t, seq) do { \
    if (!CLUSTER) { if (HEVCE_TRK == 0 || HEVCE_TRK == (t)) HEVCE_BAR(BAR_RDV1 - 1 + (t), gang_live() * (TRK_C + TRK_P)); } \
    else if (HEVCE_TRK == 0) { PHASE_END(); push_picture_state(t); PHASE_END(); if (HEVCE_TID == 0) rdv_signal(&remote_blk(t)->rdv_seq[0], (seq)); } \
    else if (HEVCE_TRK == (t)) { if (HEVCE_TID == 0) rdv_wait(&my_sm().rdv_seq[0], (seq)); PHASE_END(); } } while (0)
#define TRACK_END(t, seq) do { \
    if (!CLUSTER) { if (HEVCE_TRK == 0 || HEVCE_TRK == (t)) HEVCE_BAR(BAR_RDV1 - 1 + (t), gang_live() * (TRK_C + TRK_P)); } \
    else if (HEVCE_TRK == (t)) { PHASE_END(); if (HEVCE_TID == 0) rdv_signal(&remote_blk(0)->rdv_seq[t], (seq)); } \
    else if (HEVCE_TRK == 0) { if (HEVCE_TID == 0) rdv_wait(&my_sm().rdv_seq[t], (seq)); PHASE_END(); } } while (0)
#define ON_TRACK(t) if (HEVCE_TRK == (t))
// between the pixel phases A..D of one round: all lines of a candidate's TU are work items of the same warp (T <= 32
// consecutive items, groups start at multiples of T), so the hand-over needs no CTA- or team-wide barrier
#define WARP_SYNC() __syncwarp()
#if defined(HEVCE_PROFILE)   // per-phase latency histogram (development builds only)
extern __device__ unsigned long long g_phase_cycles[128];
extern __device__ unsigned long long g_phase_count[128];
#define PHASE_END_T(tag) do { PHASE_END(); if (threadIdx.x == 0) { Shared& pm_ = pic_sm(); const long long t_ = clock64(); \
    atomicAdd(&g_phase_cycles[tag], (unsigned long long)(t_ - pm_.prof_last)); atomicAdd(&g_phase_count[tag], 1ull); pm_.prof_last = t_; } } while (0)
#define TEAM_PROF_BEGIN() long long tp_ = clock64()
#define TEAM_PROF(tag, lead) do { if (threadIdx.x == (lead)) { const long long t_ = clock64(); \
    atomicAdd(&g_phase_cycles[tag], (unsigned long long)(t_ - tp_)); atomicAdd(&g_phase_count[tag], 1ull); tp_ = t_; } } while (0)
#else
#define PHASE_END_T(tag) PHASE_END()
#define TEAM_PROF_BEGIN() ((void)0)
#define TEAM_PROF(tag, lead) ((void)0)
#endif
#define HEVCE_ATOMIC_OR(p, v) atomicOr((p), (v))
#define HEVCE_ATOMIC_ADD(p, v) atomicAdd((p), (v))
#else
extern int g_sim_order;   // 0 forward, 1 reverse, >=2 multiplicative permutation
inline int sim_item(int i, int n) {
    if (g_sim_order == 0 || n <= 1) return i;
    if (g_sim_order == 1) return n - 1 - i;
    int a = 2 * g_sim_order + 1;
    auto gcd = [](int x, int y) { while (y) { int t = x % y; x = y; y = t; } return x; };
    while (gcd(a, n) != 1) a += 2;
    return (int)(((long long)i * a + 7) % n);
}
#define PAR_FOR(item, n) for (int item##_i = 0, item = 0; item##_i < (n) && ((item = sim_item(item##_i, (n))), true); item##_i++)
#define PAR_FOR_ALL(item, n) PAR_FOR(item, n)
#define PAR_FOR_TEAM(item, n, id, off) PAR_FOR(item, n)
#define WARP_SYNC() ((void)0)
#define TEAM_PROF_BEGIN() ((void)0)
#define TEAM_PROF(tag, lead) ((void)0)
#define PHASE_END_T(tag) PHASE_END()
#if defined(HEVCE_SIM_TRACKS)
// One host thread per track of ONE picture: a thread executes only its own track's sections, the rendezvous and the
// picture-wide barriers are real.  Inside a track the phases run sequentially (teams one after the other).
extern thread_local int g_sim_my_track;                              // the track this host thread stands for
#define ON_TRACK(t) if (g_sim_my_track == (t) && ((g_sim_trk = (t)), true))
#define TRACK_START(t, seq) do { if (g_sim_my_track == 0) { g_sim_trk = 0; if (CLUSTER) push_picture_state(t); } \
    if (g_sim_my_track == 0 || g_sim_my_track == (t)) sim_barrier(BAR_RDV1 - 1 + (t), 2); } while (0)
#define TRACK_END(t, seq) do { if (g_sim_my_track == 0 || g_sim_my_track == (t)) sim_barrier(BAR_RDV1 - 1 + (t), 2); } while (0)
#define BAR_ALL() do { if (!CLUSTER) sim_barrier(BAR_PICTURES, NTRACK); } while (0)   /* cluster: the parent tracks only meet track 0 at the rendezvous */
#define PAR_FOR_ALL_OWNER (g_sim_my_track == 0)                       /* picture-wide loops: run once, by track 0's thread */
#else
// tracks one after the other on the calling thread: a parent's candidates right after its snapshot, then the children
#define ON_TRACK(t) if ((g_sim_trk = (t)), true)
#define TRACK_START(t, seq) do { g_sim_trk = 0; if (CLUSTER) push_picture_state(t); } while (0)
#define TRACK_END(t, seq) ((void)(g_sim_trk = 0))
#define PAR_FOR_ALL_OWNER true
#endif
#if defined(HEVCE_SIM_GANG)
// the two teams of a picture really run side by side: team A on a helper thread, team B on the picture's thread
#define TEAM_A auto team_a_ = [&](int member_) { g_sim_member = member_; g_sim_trk = 0;
#define TEAM_B }; std::thread team_a_thread_(team_a_, g_sim_member);
#define TEAM_JOIN() team_a_thread_.join()
// Host thread m stands for the NT threads of picture slot m: it runs the gang-wide loops for exactly the lane / thread
// indices those threads own on the GPU (same mapping functions), so the cross-picture packing and the barrier structure
// are exercised for real (each thread runs its team A section, then its team B section; the team barriers span the threads).
#define GANG_RT (gang_live())
#define GANG_FOR(L, n) for (int x_ = g_sim_member * trk_size(HEVCE_TRK); x_ < (g_sim_member + 1) * trk_size(HEVCE_TRK); x_++) \
    for (int L = host_lane(x_, trk_lpw(HEVCE_TRK)), cap_ = lane_capacity(gang_live() * trk_size(HEVCE_TRK), trk_lpw(HEVCE_TRK)); (unsigned)L < (unsigned)(n); L += cap_)
#define GANG_FOR_UPPER(u, n) for (int x_ = NTA; x_ < TRK_C; x_++) \
    for (int u = host_lane(upper_index(g_sim_member, x_), LPW), cap_ = lane_capacity(gang_live() * NTB, LPW); (unsigned)u < (unsigned)(n); u += cap_)
#define GANG_FOR_UPPER_FREE(it, first, n) for (int x_ = NTA; x_ < TRK_C; x_++) \
    for (int st_ = 1, it = upper_free_first(upper_index(g_sim_member, x_), (first), gang_live(), (n), st_); it < (n); it += st_)
#define TEAM_SYNC(id) sim_barrier(id, gang_live())
#define PHASE_END() sim_barrier(BAR_PICTURES, gang_live())
#define BAR_ALL() sim_barrier(BAR_PICTURES, gang_live())
#define HEVCE_ATOMIC_OR(p, v) __atomic_fetch_or((p), (v), __ATOMIC_RELAXED)
#define HEVCE_ATOMIC_ADD(p, v) __atomic_fetch_add((p), (v), __ATOMIC_RELAXED)
#else
#define TEAM_A
#define TEAM_B
#define TEAM_JOIN() ((void)0)
#define TEAM_SYNC(id) ((void)0)
#define GANG_RT 1
#define GANG_FOR(L, n) PAR_FOR(L, n)
#define GANG_FOR_UPPER(u, n) PAR_FOR(u, n)
#define GANG_FOR_UPPER_FREE(it, first, n) PAR_FOR(it, n)
#define PHASE_END() ((void)0)
#if !defined(HEVCE_SIM_TRACKS)
#define BAR_ALL() ((void)0)
#define HEVCE_ATOMIC_OR(p, v) (*(p) |= (v))
#define HEVCE_ATOMIC_ADD(p, v) (*(p) += (v))
#else
#define HEVCE_ATOMIC_OR(p, v) __atomic_fetch_or((p), (v), __ATOMIC_RELAXED)
#define HEVCE_ATOMIC_ADD(p, v) __atomic_fetch_add((p), (v), __ATOMIC_RELAXED)
#endif
#endif
#endif

// Cluster variant, on track 0's threads: the picture-level state [ctx0, mirror_end) into track t's block (another CTA's
// shared memory, written through distributed shared memory) before track t is released to evaluate a node.
HEVCE_HD inline void push_picture_state(int t) {
    const Shared& sm = my_sm();
    Shared* dst = remote_blk(t);
    const int w0 = (int)((const u8*)sm.ctx0 - (const u8*)&sm) / 4, w1 = (int)((const u8*)&sm.ctu_lev - (const u8*)&sm) / 4;
    PAR_FOR(i, w1 - w0) ((u32*)dst)[w0 + i] = ((const u32*)&sm)[w0 + i];
    PAR_FOR(one, 1) dst->q = sm.q;
}

struct Avail { int L, LB, A, AR; };
HEVCE_HD inline Avail sub_avail(const Avail& a, int k) {   // HEVCe.c:1376-1379
    Avail r;
    r.L = (k & 1) ? 1 : a.L;
    r.LB = k == 0 ? a.L : k == 2 ? a.LB : 0;
    r.A = (k & 2) ? 1 : a.A;
    r.AR = k == 0 ? a.A : k == 1 ? a.AR : k == 2 ? 1 : 0;
    return r;
}

// window sample relative to CTU pixel (y,x); y or x may be -1
#define HEVCE_WIN(sm, y, x) ((sm).win[(1 + (y)) * WP + 1 + (x)])

// z-order offset of the 8x8 unit at CTU position (y,x) in the CTU level store
HEVCE_HD inline int zoff(int y, int x) {
    const int a = y >> 3, c = x >> 3;
    return (((a & 2) << 2) | ((c & 2) << 1) | ((a & 1) << 1) | (c & 1)) * 64;
}

// Levels of a TU are stored group by group (groups in raster order, gy*ncg+gx), the 16 levels of a group in the
// scan order of the candidate's mode: a trial coder fetches one group with two 16-byte loads.
HEVCE_HD inline void load_group(const s16* p, u32 (&w)[8]) {
#if defined(__CUDA_ARCH__)
    const uint4 a = ((const uint4*)p)[0], b = ((const uint4*)p)[1];
    w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
#else
    for (int i = 0; i < 8; i++) w[i] = (u32)(unsigned short)p[2 * i] | ((u32)(unsigned short)p[2 * i + 1] << 16);
#endif
}

// one coefficient group: bit-fields in scan order, last position (first coded group only), sig flags, greater1/2,
// signs, remaining levels.  w: the 16 levels (8 words), gp: the same group in the store (escape magnitudes).
template <class BAC>
HEVCE_HD inline void code_group(BAC& b, const Tables& tbl, const Cx cx, int s, int st, int lg, int sigbase, const s16* gp, const u32 (&w)[8],
                                int on, int pat, int first_cg, bool is_last, int cy, int cxg, int& c1) {
    const Tables* tb = &tbl;
    // ---- bit-fields of the group, scan order
    unsigned nzm = 0, sgn = 0, cls = 0;
#if !HEVCE_OPT_FASTBUILD
    if (on) {
#pragma unroll
        for (int k = 0; k < 16; k++) {
            const int v = (int)(s16)(w[k >> 1] >> (16 * (k & 1)));
            const unsigned a = (unsigned)imin(iabs(v), 3);
            nzm |= (unsigned)(v != 0) << k;
            sgn |= (unsigned)(v < 0) << k;
            cls |= a << (2 * k);
        }
    }
#else
    if (on) {   // word j holds the levels of scan positions 2j (low half) and 2j+1
        unsigned sg = 0;   // sign of position 2j at bit 2j, of position 2j+1 at bit 16+2j
#pragma unroll
        for (int j = 0; j < 8; j++) {
            sg |= (w[j] >> (15 - 2 * j)) & (0x00010001u << (2 * j));
            const unsigned a0 = (unsigned)imin(iabs((int)(s16)w[j]), 3), a1 = (unsigned)imin(iabs((int)w[j] >> 16), 3);
            cls |= (a0 | (a1 << 2)) << (4 * j);
        }
        sgn = (sg | (sg >> 15)) & 0xffffu;
        unsigned t = (cls | (cls >> 1)) & 0x55555555u;   // non-zero flags on the even bits, then squeezed together
        t = (t | (t >> 1)) & 0x33333333u;
        t = (t | (t >> 2)) & 0x0f0f0f0fu;
        t = (t | (t >> 4)) & 0x00ff00ffu;
        nzm = (t | (t >> 8)) & 0xffffu;
    }
#endif
    int kstart = 15;
    if (is_last) {
        kstart = nzm ? bitlen(nzm) - 1 : 0;
        const int p4 = tb->scan4[st][kstart];
        // last_sig_coeff_xy (HEVCe.c:1046-1087)
        const int y = cy * 4 + (p4 >> 2), x = cxg * 4 + (p4 & 3);
        const int row = lg - 2, sh = s > 4;
        int ty = st == 2 ? x : y, tx = st == 2 ? y : x;
        const int gy = tb->grp[ty], gx = tb->grp[tx], gmax = tb->grp[s - 1];
        const int bx = cx_lastx(row), by = cx_lasty(row);
        for (int i = 0; i < gx; i++) b.put_bin(tbl, 1, cx[bx + (i >> sh)]);
        if (gx < gmax) b.put_bin(tbl, 0, cx[bx + (gx >> sh)]);
        for (int i = 0; i < gy; i++) b.put_bin(tbl, 1, cx[by + (i >> sh)]);
        if (gy < gmax) b.put_bin(tbl, 0, cx[by + (gy >> sh)]);
#if HEVCE_OPT_BYPMERGE
        {   // both suffixes (<= 3 bits each) as one string
            const int nx = gx > 3 ? (gx - 2) >> 1 : 0, ny = gy > 3 ? (gy - 2) >> 1 : 0;
            if (nx + ny) b.put_bypass(((gx > 3 ? tx - tb->gmin[gx] : 0) << ny) | (gy > 3 ? ty - tb->gmin[gy] : 0), nx + ny);
        }
#else
        if (gx > 3) { tx -= tb->gmin[gx]; for (int i = ((gx - 2) >> 1) - 1; i >= 0; i--) b.put_bypass((tx >> i) & 1, 1); }   // one bin per call,
        if (gy > 3) { ty -= tb->gmin[gy]; for (int i = ((gy - 2) >> 1) - 1; i >= 0; i--) b.put_bypass((ty >> i) & 1, 1); }   // as HEVCe.c:1076-1086
#endif
    }
    // ---- sig_coeff_flags (HEVCe.c:1219-1222, context HEVCe.c:1092-1122)
    {
        // one 4-bit field per scan index: the context of a 4x4 TU's position, or the neighbour-pattern offset of a larger TU
        const unsigned long long tab = s == 4 ? tb->sig4[st] : tb->sigoff[st][pat];
        const int base = s == 4 ? CX_SIG : sigbase + (first_cg ? 0 : 3);
        const bool dc = first_cg && s != 4;                         // position 0 of a larger TU has its own context
        int k = is_last ? kstart - 1 : 15;
        const int kend = (!first_cg && (nzm & ~1u) == 0) ? 1 : 0;   // position 0 of a later group is inferred when it is the only one
        for (; k >= kend; k--) {
            int ci = base + (int)((tab >> (4 * k)) & 15u);
            if (dc && k == 0) ci = CX_SIG;
            b.put_bin(tbl, (int)((nzm >> k) & 1u), cx[ci]);
        }
    }
    if (nzm) {
        // ---- greater1 / greater2 flags, signs (HEVCe.c:1229-1252)
        const int set = (first_cg ? 0 : 2) + (c1 == 0);
        int nz = 0, signs = 0, g2 = -1;
        c1 = 1;
        unsigned mm = nzm;
        while (mm) {
            const int k = bitlen(mm) - 1;
            mm &= ~(1u << k);
            signs = (signs << 1) | (int)((sgn >> k) & 1u);
            if (nz < 8) {
                const int a = (int)((cls >> (2 * k)) & 3u), big = a > 1;
                b.put_bin(tbl, big, cx[CX_ONE + 4 * set + c1]);
                if (big) { c1 = 0; if (g2 < 0) g2 = a > 2; else g2 |= 4; }
                else if (c1 > 0 && c1 < 3) c1++;
            }
            nz++;
        }
        int esc = nz > 8;
        if (g2 >= 0) {
            if (g2 & 4) esc = 1;
            g2 &= 1;
            if (c1 == 0) { b.put_bin(tbl, g2, cx[CX_ABS + set]); esc |= g2; }
        }
        b.put_bypass(signs, nz);
        // ---- coeff_abs_level_remaining (HEVCe.c:1254-1266, 1154-1169)
        if (esc) {
            int base = 3, rp = 0, j = 0;
            mm = nzm;
            while (mm) {
                const int k = bitlen(mm) - 1;
                mm &= ~(1u << k);
                int a = (int)((cls >> (2 * k)) & 3u);
                if (a == 3) a = iabs((int)gp[k]);
                int v = a - (j < 8 ? base : 1);
                if (v >= 0) {
                    if (v < (3 << rp)) {
                        const int n = v >> rp;
#if HEVCE_OPT_BYPMERGE
                        b.put_bypass((((1 << (n + 1)) - 2) << rp) | (v & ((1 << rp) - 1)), n + 1 + rp);   // <= 8 bits: one chunk
#else
                        b.put_bypass((1 << (n + 1)) - 2, n + 1);
                        b.put_bypass(v & ((1 << rp) - 1), rp);
#endif
                    } else {
                        int n = rp;
                        v -= 3 << rp;
                        for (; v >= (1 << n); n++) v -= 1 << n;
                        const int pre = 4 + n - rp;
#if HEVCE_OPT_BYPMERGE
                        if (pre + n <= 30) b.put_bypass((((1 << pre) - 2) << n) | v, pre + n);
                        else
#endif
                        {
                            b.put_bypass((1 << pre) - 2, pre);
                            b.put_bypass(v, n);
                        }
                    }
                    if (a > (3 << rp)) rp = imin(rp + 1, 4);
                }
                if (a >= 2) base = 2;
                j++;
            }
        }
    }

}

// residual_coding() of one TU (HEVCe.c:1173-1269), restructured around coefficient groups: the caller supplies the
// bitmap of non-zero 4x4 groups (bit gy*8+gx), so all-zero groups cost one bin and no memory traffic; a coded group
// is reduced to three bit-fields in scan order (non-zero mask, signs, min(|level|,3) classes) that drive every
// context-coded bin; only escape magnitudes are read back from the store.
template <class BAC>
HEVCE_HD inline void put_residual(BAC& b, const Tables& tbl, const Cx cx, int s, int m, const s16* lev, unsigned mlo, unsigned mhi) {
    const Tables* tb = &tbl;
    const int st = scan_type(s, m), lg = ilog2(s), ncg = s >> 2;
    const int sigbase = CX_SIG + 9 + (s >= 16 ? 12 : 0) + ((s == 8 && st) ? 6 : 0);
    auto cgpos = [&](int g, int& cy, int& cxg) {
        if (lg == 2) { cy = 0; cxg = 0; }
        else if (st == 1) { cy = g >> 1; cxg = g & 1; }
        else if (st == 2) { cy = g & 1; cxg = g >> 1; }
        else { const int v = tb->cgdiag[lg - 3][g]; cy = v >> 3; cxg = v & 7; }
    };
    auto bit = [&](int cy, int cxg) -> int { const int k = cy * 8 + cxg; return (int)(((k < 32) ? (mlo >> k) : (mhi >> (k - 32))) & 1u); };
    int gl = 0;
    for (int g = ncg * ncg - 1; g > 0; g--) {
        int cy, cxg;
        cgpos(g, cy, cxg);
        if (bit(cy, cxg)) { gl = g; break; }
    }
    int c1 = 1;
    // groups are visited in reverse scan order; the levels of the next coded group are fetched while the current
    // one is being coded (the store is L2-resident, a fetch costs several hundred cycles)
    u32 w[8];
    int cy, cxg, ncy = 0, ncx = 0;
    cgpos(gl, cy, cxg);
    int on = bit(cy, cxg);
    if (on) load_group(lev + (cy * ncg + cxg) * 16, w);
    for (int g = gl;;) {
        // next group that needs its levels: the next non-zero one, or the first group
        int g2 = g - 1, on2 = 0;
        for (; g2 > 0; g2--) {
            cgpos(g2, ncy, ncx);
            if (bit(ncy, ncx)) { on2 = 1; break; }
        }
        if (g2 == 0) { ncy = 0; ncx = 0; on2 = g > 0 ? bit(0, 0) : 0; }
#if defined(__CUDA_ARCH__)
        if (on2) asm volatile("prefetch.global.L1 [%0];" ::"l"(lev + (ncy * ncg + ncx) * 16));
#endif
        const int first_cg = g == 0;
        {
            const int rgt = cxg < ncg - 1 && bit(cy, cxg + 1), dwn = cy < ncg - 1 && bit(cy + 1, cxg);
            const int pat = (dwn << 1) | rgt;
            if (g != gl && !first_cg) b.put_bin(tbl, on, cx[CX_SIGCG + (pat != 0)]);
            code_group(b, tbl, cx, s, st, lg, sigbase, lev + (cy * ncg + cxg) * 16, w, on, pat, first_cg, g == gl, cy, cxg, c1);
        }
        if (g == 0) break;
        for (int gg = g - 1; gg > g2; gg--) {   // all-zero groups in between: coded_sub_block_flag = 0
            int zy, zx;
            cgpos(gg, zy, zx);
            const int rgt = zx < ncg - 1 && bit(zy, zx + 1), dwn = zy < ncg - 1 && bit(zy + 1, zx);
            b.put_bin(tbl, 0, cx[CX_SIGCG + ((rgt | dwn) != 0)]);
        }
        g = g2; cy = ncy; cxg = ncx; on = on2;
        if (on) load_group(lev + (cy * ncg + cxg) * 16, w);
    }
}

// Where tables and context sets live: the decision kernel keeps them in the picture's Shared block, the commit kernel
// in its own small shared block.  Both are reached through the extern shared array so the accesses stay LDS/STS.
struct CommitShared {
    Tables tb;
    u32 ctx[NTC * CTXW];  // lane-private context sets of the NTC commit threads of a block, lane-major
};
#if defined(__CUDA_ARCH__)
__device__ __forceinline__ CommitShared& my_csm() { return *reinterpret_cast<CommitShared*>(hevce_smem); }
#elif defined(__CUDACC__)
inline CommitShared& my_csm() { return *static_cast<CommitShared*>(nullptr); }
#else
extern CommitShared* g_sim_csm;
inline CommitShared& my_csm() { return *g_sim_csm; }
#endif
struct MainEnv {
    HEVCE_HD static const Tables& tables() { return my_tb(); }
    HEVCE_HD static u8* base(int b) { return (u8*)&blk_sm(b); }   // b: shared-memory block (picture of the gang, track) the lane works for
};
struct CommitEnv {
    HEVCE_HD static const Tables& tables() { return my_csm().tb; }
    HEVCE_HD static u8* base(int) { return (u8*)&my_csm(); }
};

// One coding unit (HEVCe.c:1272-1340, 943-947).
struct CuDesc {
    int s;              // CU size
    int kind;           // 0: 2Nx2N one TU, 1: 2Nx2N four TUs, 2: NxN, 3: residual of one TU only (NxN PU trial, HEVCe.c:1516)
    int split_ctx;      // >= 0: code split_cu_flag = 0 with this context first (only s >= 16 codes it)
    int pm[4], pl[4], pa[4];
    const s16* lev[4];  // levels of TU k
    unsigned mlo[4];    // non-zero-group bitmaps of TU k (low word); mhi: high word of TU 0 (32x32 only)
    unsigned mhi;
};

template <class BAC, class ENV>
HEVCE_HD HEVCE_NOINLINE void code_cu(BAC& bio, int pic, int cx_off, const CuDesc& d) {
    const Tables& tbl = ENV::tables();
    const Cx cx = {ENV::base(pic) + cx_off};
    BAC b = bio;   // coder state in registers for the whole CU
    b.use_tables(tbl);
    const int s = d.s, kind = d.kind;
    if (kind != 3) {
        if (d.split_ctx >= 0 && s >= 16) b.put_bin(tbl, 0, cx[CX_SPLIT_CU + d.split_ctx]);
        if (s == 8) b.put_bin(tbl, kind != 2, cx[CX_PART]);
        // luma modes (HEVCe.c:985-1018)
        const int n = kind == 2 ? 4 : 1;
        int hit[4], mp[4][3];
        for (int i = 0; i < n; i++) {
            mpm_list(d.pl[i], d.pa[i], mp[i]);
            hit[i] = -1;
            for (int j = 0; j < 3; j++) if (mp[i][j] == d.pm[i]) hit[i] = j;
            b.put_bin(tbl, hit[i] >= 0, cx[CX_YPM]);
        }
        for (int i = 0; i < n; i++) {
            if (hit[i] >= 0) {
#if HEVCE_OPT_BYPMERGE
                b.put_bypass(hit[i] > 0 ? 2 + (hit[i] - 1) : 0, hit[i] > 0 ? 2 : 1);   // mpm_idx: 0 / 10 / 11
#else
                b.put_bypass(hit[i] > 0, 1);
                if (hit[i] > 0) b.put_bypass(hit[i] - 1, 1);
#endif
            } else {
                int r = d.pm[i];
                const int hi = imax(mp[i][0], imax(mp[i][1], mp[i][2])), lo = imin(mp[i][0], imin(mp[i][1], mp[i][2]));
                const int mid = mp[i][0] + mp[i][1] + mp[i][2] - hi - lo;
                if (r > hi) r--;
                if (r > mid) r--;
                if (r > lo) r--;
                b.put_bypass(r, 5);
            }
        }
        b.put_bin(tbl, 0, cx[CX_UVPM]);
        if (kind != 2) b.put_bin(tbl, kind == 1, cx[CX_SPLIT_TU + (s == 32 ? 0 : s == 16 ? 1 : 2)]);
        b.put_bin(tbl, 0, cx[CX_UVCBF]);
        b.put_bin(tbl, 0, cx[CX_UVCBF]);
    }
    const int ntu = (kind == 0 || kind == 3) ? 1 : 4, ts = kind == 0 ? s : kind == 3 ? 4 : s >> 1;
    for (int k = 0; k < ntu; k++) {
        const unsigned mlo = d.mlo[k], mhi = k == 0 ? d.mhi : 0u;
        const int on = (mlo | mhi) != 0;
        if (kind != 3) b.put_bin(tbl, on, cx[CX_YCBF + (kind == 0)]);
        if (on || kind == 3) put_residual(b, tbl, cx, ts, d.pm[kind == 2 ? k : 0], d.lev[k], mlo, mhi);
    }
    bio = b;
}

// bitmap of non-zero 4x4 groups of a stored TU (commit pass; the trial path gets it from phase C)
HEVCE_HD inline void scan_groups(const s16* lev, int s, unsigned& mlo, unsigned& mhi) {
    const int ncg = s >> 2;
    mlo = mhi = 0;
    for (int gy = 0; gy < ncg; gy++)
        for (int gx = 0; gx < ncg; gx++) {
            u32 w[8];
            load_group(lev + (gy * ncg + gx) * 16, w);
            if (w[0] | w[1] | w[2] | w[3] | w[4] | w[5] | w[6] | w[7]) { const int k = gy * 8 + gx; if (k < 32) mlo |= 1u << k; else mhi |= 1u << (k - 32); }
        }
}

// ------------------------------------------------------------------------------------------------------------
// pixel pipeline: one group = the same TU (position, size T) of n candidates with consecutive modes
// ------------------------------------------------------------------------------------------------------------
struct Grp {
    int n;              // candidates in this group (0 = group unused this round)
    int cand0;          // index of local candidate 0 in the per-node arrays (glev, cand_sse, cgnz, ...)
    int mode0;          // its intra mode; local candidate c has mode0 + c
    int ty, tx;         // TU origin in CTU coordinates
    Avail av;           // neighbour availability of this TU
    int priv;           // 1: samples inside the CU come from the candidate's own reconstruction (four-TU candidates)
    int cuy, cux, cus;  // CU origin / size
    int tu;             // TU index inside the candidate (levels at tu*T*T, bitmap word)
    int one_tu;         // 1: one-TU candidate (bitmap uses words 0/1)
    int grec;           // 1: reconstruction rows also go to the global store (cand0 < NREC)
    // byte offsets into Shared::pool (offsets, not pointers, so the accesses stay in the shared address space)
    int blk;            // s16 [n][T*T+T]   residual -> coefficients -> tentative levels -> inverse intermediate
    int pred;           // u8  [n][T*T]
    int psum;           // int [n][T*T/4]   per (row, group column) sums for the group zero-out
    int bord;           // u8  shared: [2][4T+4] (unfiltered, filtered); private: [n][4T+4]
    int rec;            // u8  priv: [n][4*T] edges of the candidate's own sub-TUs (bottom rows of TU 0,1; right columns of TU 0,2);
                        //     NxN PU group: [n][16] the PU's reconstruction; -1: none
    int rec_stride, rec_pitch;
};

template <int T> struct Dim {
    static constexpr int LG = T == 4 ? 2 : T == 8 ? 3 : T == 16 ? 4 : 5;
    static constexpr int BLK = T * T + T;      // padded so that column items of neighbouring candidates hit distinct banks
    static constexpr int BS = 4 * T + 4;       // border array: [pad][2T left, bottom first][corner][2T top][pad]
    static constexpr int UNR = T <= 8 ? T : 1; // loops that do not need register arrays stay rolled for the large sizes
};

// phase 0: reference samples (HEVCe.c:196-257) into the unified border array b[0..4T]: b[2T] = corner,
// b[2T-1-i] = left[i], b[2T+1+i] = top[i]; the [1 2 1] filter is then uniform over the array.
// One work item = one border index j for ALL candidates of the group: where sample j comes from (window, the
// candidate's own sub-TU edges, or the constant 128) does not depend on the candidate, so it is resolved once and the
// candidate loop is a uniform fetch / filter / store.
struct BSrc { int kind, off; };   // kind 0: constant 128, 1: window byte offset, 2: offset inside the candidate's edge block

template <int T>
HEVCE_HD inline void border_column(Shared& sm, const Shared& pm, const Grp& g, int j, int c0, int c1) {   // candidates [c0, c1) of a private group
    constexpr int BS = Dim<T>::BS;
    const Avail& a = g.av;
    auto pos = [&](int y, int x) -> BSrc {
        const int yy = g.ty + y, xx = g.tx + x;
        if (g.priv) {   // inside the CU only the sub-TU edges can be asked for: row T-1 (bottom of TU 0/1) or column T-1 (right of TU 0/2)
            const int cy = yy - g.cuy, cx = xx - g.cux;
            if (cy >= 0 && cx >= 0 && cy < g.cus && cx < g.cus) {
                if (cy == T - 1) return BSrc{2, (cx >= T ? T : 0) + (cx & (T - 1))};
                return BSrc{2, 2 * T + (cy >= T ? T : 0) + (cy & (T - 1))};
            }
        }
        return BSrc{1, (1 + yy) * WP + 1 + xx};
    };
    auto corner = [&]() -> BSrc {   // HEVCe.c:212-219
        if (a.L && a.A) return pos(-1, -1);
        if (a.L) return pos(0, -1);
        if (a.A) return pos(-1, 0);
        return BSrc{0, 0};
    };
    auto resolve = [&](int jj) -> BSrc {   // HEVCe.c:221-243
        if (jj == 2 * T) return corner();
        if (jj < 2 * T) {
            const int i = 2 * T - 1 - jj;
            if (i < T ? a.L : a.LB) return pos(i, -1);
            return a.L ? pos(T - 1, -1) : corner();
        }
        const int i = jj - 2 * T - 1;
        if (i < T ? a.A : a.AR) return pos(-1, i);
        return a.A ? pos(-1, T - 1) : corner();
    };
    const bool inner = T > 4 && j > 0 && j < 4 * T;   // the two ends stay unfiltered (HEVCe.c:255-256); 4x4 is never filtered
    const BSrc s0 = resolve(j);
    BSrc sa = s0, sb = s0;
    if (inner) { sa = resolve(j - 1); sb = resolve(j + 1); }
    const u8* win = pm.win;
    if (!g.priv) {
        auto fetch = [&](const BSrc& q) -> int { return q.kind == 1 ? win[q.off] : 128; };
        const int v = fetch(s0);
        sm.pool[g.bord + 1 + j] = (u8)v;
        if (T > 4) sm.pool[g.bord + BS + 1 + j] = (u8)(inner ? (2 + 2 * v + fetch(sa) + fetch(sb)) >> 2 : v);
    } else {
        const u8* edges = sm.pool + g.rec;
        auto fetch = [&](const BSrc& q, int c) -> int { return q.kind == 1 ? win[q.off] : q.kind == 2 ? edges[c * (4 * T) + q.off] : 128; };
        u8* dst = sm.pool + g.bord + 1 + j;
        for (int c = c0; c < c1; c++) {
            int v = fetch(s0, c);
            if (inner && use_filtered(T, g.mode0 + c)) v = (2 + 2 * v + fetch(sa, c) + fetch(sb, c)) >> 2;
            dst[c * BS] = (u8)v;
        }
    }
}

// phase A: prediction of column x (HEVCe.c:262-381), residual, forward column transform (HEVCe.c:514)
template <int T>
HEVCE_HD inline void phase_a_item(Shared& sm, const Shared& pm, const Grp& g, int item) {
    constexpr int LG = Dim<T>::LG, BLK = Dim<T>::BLK, BS = Dim<T>::BS, UNR = Dim<T>::UNR;
    const int c = item >> LG, x = item & (T - 1), m = g.mode0 + c;
    const int bsel = g.priv ? c : (T > 4 && use_filtered(T, m));
    const u8* B = sm.pool + g.bord + bsel * BS + 1 + 2 * T;   // B[k]: k > 0 top[k-1], k < 0 left[-k-1], 0 corner
    const u8* org = pm.orig + g.ty * CTU + g.tx + x;
    u8* pp = sm.pool + g.pred + c * (T * T) + x;
    if (x == 0) {   // per-candidate accumulators of this TU
        const int ci = g.cand0 + c;
        if (g.one_tu) { sm.cgnz[ci][0] = 0; sm.cgnz[ci][1] = 0; sm.cand_sse[ci] = 0; }
        else { sm.cgnz[ci][g.tu] = 0; if (g.tu == 0 || !g.priv) sm.cand_sse[ci] = 0; }
    }
    const bool edge = T <= 16;
    if (m == 0) {
        const int tr = B[T + 1], bl = B[-T - 1], tx = B[1 + x];
#pragma unroll UNR
        for (int y = 0; y < T; y++) pp[y * T] = (u8)(((T - 1 - x) * B[-1 - y] + (x + 1) * tr + (T - 1 - y) * tx + (y + 1) * bl + T) >> (LG + 1));
    } else if (m == 1) {
        int dc = T;
#pragma unroll UNR
        for (int i = 0; i < T; i++) dc += B[-1 - i] + B[1 + i];
        dc >>= LG + 1;
#pragma unroll UNR
        for (int y = 0; y < T; y++) pp[y * T] = (u8)((edge && x == 0 && y > 0) ? (2 + 3 * dc + B[-1 - y]) >> 2 : dc);
        if (edge) pp[0] = (u8)(x == 0 ? (2 + 2 * dc + B[-1] + B[1]) >> 2 : (2 + 3 * dc + B[1 + x]) >> 2);
    } else if (m == 10) {
#pragma unroll UNR
        for (int y = 0; y < T; y++) pp[y * T] = B[-1 - y];
        if (edge) pp[0] = (u8)iclip(((B[1 + x] - B[0]) >> 1) + B[-1], 0, 255);
    } else if (m == 26) {
        const int t = B[1 + x];
#pragma unroll UNR
        for (int y = 0; y < T; y++) pp[y * T] = (u8)((edge && x == 0) ? iclip(((B[-1 - y] - B[0]) >> 1) + t, 0, 255) : t);
    } else {
        const int ang = intra_angle(m), aa = iabs(ang), inv = (8192 + aa / 2) / aa;   // HEVCe.c:283
        if (m < 18) {   // horizontal family: main arm = left, projected side = top
            const int off = ang * (x + 1), oi = off >> 5, of = off & 31;
            auto R = [&](int k) -> int { return k >= 0 ? B[-k] : B[(128 - inv * k) >> 8]; };
            int prev = R(oi + 1);
#pragma unroll UNR
            for (int y = 0; y < T; y++) {
                const int nxt = R(oi + y + 2);
                pp[y * T] = (u8)(((32 - of) * prev + of * nxt + 16) >> 5);
                prev = nxt;
            }
        } else {        // vertical family: main arm = top, projected side = left
            auto R = [&](int k) -> int { return k >= 0 ? B[k] : B[-((128 - inv * k) >> 8)]; };
#pragma unroll UNR
            for (int y = 0; y < T; y++) {
                const int off = ang * (y + 1), oi = off >> 5, of = off & 31, k = oi + x + 1;
                pp[y * T] = (u8)(((32 - of) * R(k) + of * R(k + 1) + 16) >> 5);
            }
        }
    }
    int v[T], o[T];
#pragma unroll
    for (int y = 0; y < T; y++) v[y] = (int)org[y * CTU] - (int)pp[y * T];
    Xf<T>::f(v, o);
    s16* bp = (s16*)(sm.pool + g.blk) + c * BLK + x;
    constexpr int A1 = LG - 1;
#pragma unroll
    for (int k = 0; k < T; k++) bp[k * T] = (s16)((o[k] + (1 << A1 >> 1)) >> A1);
}

// Per-coefficient RDOQ (HEVCe.c:563-586): the level of coefficient cf, unsigned; dl receives |cf| << 14 for the group sums.
// RD cost without the saturation tests of HEVCe.c:182-184: here dist <= 2^24 and rate <= 1.2e6, so neither product nor
// the sum can reach 2^31 and the plain weighted sum is the same number.
struct RdoqK { int dsh, sh, add, wd, wb; };
HEVCE_HD inline RdoqK rdoq_consts(int lg, int q) {
    const RdK rk = rd_consts(q);
    RdoqK k;
    k.dsh = 10 - lg; k.sh = 21 - lg + q; k.add = 1 << k.sh >> 1; k.wd = rk.wd; k.wb = rk.wb;
    return k;
}
HEVCE_HD inline int rdoq_level(int cf, const RdoqK& k, const Tables& tb, int& dl) {
    dl = iabs(cf) << 14;                                         // |cf| <= 32767: the clamps of HEVCe.c:566 cannot trigger
    const int lvl = (dl + k.add) >> k.sh;
    if (lvl <= 0) return 0;
    // Candidates lvl and lvl-1 only: the third one of HEVCe.c:571, lvl-2, can never be picked.  One level is
    // U = 2^(11+q) in units of the distance e; e(lvl) <= U/2, e(lvl-1) = a in [U/2, 3U/2), e(lvl-2) = a + U exactly
    // (2^sh is a multiple of 2^dsh).  qpd6 <= 3: nothing saturates (5U/2 < 46340) and dist(lvl-2) - dist(lvl-1) >=
    // U^2/64 - 1 = 2^(16+2q) - 1; times wd = 11/11/11/5 that is >= 720,885 / 2.9 M / 11.5 M / 21 M against at most
    // wb * 70,000 = 70,000 / 280,000 / 1.12 M / 2.03 M of rate (70,000 is the largest step between neighbouring
    // levels): lvl-1 is strictly cheaper than lvl-2.  qpd6 = 4: dist(lvl-2) saturates to 2^24 - 1 while dist(lvl) <=
    // 2^21, and two levels are worth at most 23 * 131,072 = 3.0 M of rate: lvl is strictly cheaper than lvl-2.
    // The scan keeps the higher level on a tie, so lvl-1 wins iff cost(lvl-1) < cost(lvl), i.e. iff
    // wd * (dist(lvl-1) - dist(lvl)) < wb * (rate(lvl) - rate(lvl-1)); the rate step comes from an 8-entry table
    // (HEVCe.c:526-535: from level 7 on it is 65536 when lvl-5 is a power of two, else 0).  No product reaches 2^31.
    // tests/test_stages.py: every |cf| x TU size x qpd6 against the reference's quantize().
    const int r = dl - (lvl << k.sh);                           // in [-add, add)
    const int e0 = iabs(r) >> k.dsh;
    const int e1 = (r + 2 * k.add) >> k.dsh;                    // distance to lvl-1: positive
    const int d0 = (e0 * e0) >> 7;
    const int d1 = (e1 < 46340 ? e1 * e1 : IMAX) >> 7;          // saturates at qpd6 = 4 only
    const int dr = tb.drate[imin(lvl, 7)] + ((lvl >= 7 && ((lvl - 5) & (lvl - 6)) == 0) ? 65536 : 0);
    return k.wd * (d1 - d0) < k.wb * dr ? lvl - 1 : lvl;
}

// phase B: forward row transform (HEVCe.c:515) + per-coefficient RDOQ (HEVCe.c:563-586); tentative levels replace
// the coefficients in place, the clamped magnitudes are summed per (row, group column) for the zero-out test.
template <int T>
HEVCE_HD inline void phase_b_item(Shared& sm, const Shared& pm, const Grp& g, int item, int q, const RdK& rk) {
    constexpr int LG = Dim<T>::LG, BLK = Dim<T>::BLK, A2 = LG + 6;
    const int c = item >> LG, y = item & (T - 1);
    s16* bp = (s16*)(sm.pool + g.blk) + c * BLK + y * T;
    {
        int v[T], o[T];
#pragma unroll
        for (int x = 0; x < T; x++) v[x] = bp[x];
        Xf<T>::f(v, o);
#pragma unroll
        for (int x = 0; x < T; x++) bp[x] = (s16)((o[x] + (1 << A2 >> 1)) >> A2);
    }
    const RdoqK k = rdoq_consts(LG, q);
    const int thr = 9 << k.sh >> 2;
    const Tables& tb = my_tb();
    int* ps = (int*)(sm.pool + g.psum) + c * (T * T / 4) + y * (T / 4);
#pragma unroll 1
    for (int gx = 0; gx < T / 4; gx++) {
        int sum = 0;
#pragma unroll
        for (int e = 0; e < 4; e++) {
            const int x = gx * 4 + e;
            const int cf = bp[x];
            int dl;
            const int pick = rdoq_level(cf, k, tb, dl);
            bp[x] = (s16)(cf < 0 ? -pick : pick);
            sum += imin(dl, thr);
        }
        ps[gx] = sum;
    }
}

// phase C: group zero-out (HEVCe.c:589-592), final levels -> global store (group-blocked, scan order) + non-zero-group
// bitmap, dequantisation (HEVCe.c:600-615), inverse column transform (HEVCe.c:514 with inverse=1)
template <int T>
HEVCE_HD inline void phase_c_item(Shared& sm, const Scratch& sc, const Grp& g, int item, int q) {
    constexpr int LG = Dim<T>::LG, BLK = Dim<T>::BLK;
    const int c = item >> LG, x = item & (T - 1), gx = x >> 2, ci = g.cand0 + c;
    s16* bp = (s16*)(sm.pool + g.blk) + c * BLK + x;
    const int* ps = (const int*)(sm.pool + g.psum) + c * (T * T / 4) + gx;
    const u8* inv = my_tb().inv4[scan_type(T, g.mode0 + c)] + (x & 3);
    s16* lp = sc.glev + (size_t)ci * LEV_STRIDE + g.tu * (T * T) + gx * 16;
    const int sh = 21 - LG + q, thr = 9 << sh >> 2, qs = 7 - LG + q;
    int v[T], o[T];
    unsigned mlo = 0, mhi = 0;
    int anyc = 0;
#pragma unroll
    for (int gy = 0; gy < T / 4; gy++) {
        const int sum = ps[(gy * 4) * (T / 4)] + ps[(gy * 4 + 1) * (T / 4)] + ps[(gy * 4 + 2) * (T / 4)] + ps[(gy * 4 + 3) * (T / 4)];
        const bool keep = sum >= thr;
        int nzc = 0;
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const int y = gy * 4 + r;
            const int l = keep ? (int)bp[y * T] : 0;
            lp[gy * (T / 4) * 16 + inv[r * 4]] = (s16)l;
            nzc |= l;
            v[y] = iclip(l * (1 << qs), -32768, 32767);
        }
        if (nzc) {
            const int k = gy * 8 + gx;
            if (k < 32) mlo |= 1u << k; else mhi |= 1u << (k - 32);
            anyc = 1;
        }
    }
    if (g.one_tu) {
        if (mlo) HEVCE_ATOMIC_OR(&sm.cgnz[ci][0], mlo);
        if (mhi) HEVCE_ATOMIC_OR(&sm.cgnz[ci][1], mhi);
    } else if (mlo) HEVCE_ATOMIC_OR(&sm.cgnz[ci][g.tu], mlo);
    if (anyc) {
        Xf<T>::i(v, o);
#pragma unroll
        for (int k = 0; k < T; k++) bp[k * T] = (s16)iclip((o[k] + 64) >> 7, -32768, 32767);
    } else {
#pragma unroll
        for (int k = 0; k < T; k++) bp[k * T] = 0;
    }
}

// phase D: inverse row transform (HEVCe.c:515 with inverse=1), reconstruction, SSE (HEVCe.c:165-174)
template <int T>
HEVCE_HD inline void phase_d_item(Shared& sm, const Shared& pm, const Scratch& sc, const Grp& g, int item) {
    constexpr int LG = Dim<T>::LG, BLK = Dim<T>::BLK;
    const int c = item >> LG, y = item & (T - 1), ci = g.cand0 + c;
    const unsigned nzw = g.one_tu ? (sm.cgnz[ci][0] | sm.cgnz[ci][1]) : sm.cgnz[ci][g.tu];
    const s16* bp = (const s16*)(sm.pool + g.blk) + c * BLK + y * T;
    const u8* pp = sm.pool + g.pred + c * (T * T) + y * T;
    const u8* org = pm.orig + (g.ty + y) * CTU + g.tx;
    int v[T], o[T];
    if (nzw) {
#pragma unroll
        for (int x = 0; x < T; x++) v[x] = bp[x];
        Xf<T>::i(v, o);
    } else {
#pragma unroll
        for (int x = 0; x < T; x++) o[x] = 0;
    }
    const int ry = g.ty - g.cuy + y, rx = g.tx - g.cux;
    u8* rs = (g.rec >= 0 && !g.priv) ? sm.pool + g.rec + c * g.rec_stride + ry * g.rec_pitch + rx : nullptr;
    u8* er = nullptr;   // four-TU candidates keep the edges later sub-TUs predict from: bottom row of TU 0/1
    if (g.priv && g.tu < 2 && y == T - 1) er = sm.pool + g.rec + c * (4 * T) + g.tu * T;
    u8* rg = g.grec ? sc.grec + (size_t)ci * (CTU * CTU) + ry * g.cus + rx : nullptr;
    int sse = 0;
#pragma unroll
    for (int x = 0; x < T; x++) {
        const int res = iclip((o[x] + 2048) >> 12, -32768, 32767);
        const int rec = iclip(res + pp[x], 0, 255);
        const int d = (int)org[x] - rec;
        sse += d * d;
        if (rs) rs[x] = (u8)rec;
        if (er) er[x] = (u8)rec;
        if (rg) rg[x] = (u8)rec;
        if (x == T - 1 && g.priv && !(g.tu & 1)) sm.pool[g.rec + c * (4 * T) + 2 * T + (g.tu >> 1) * T + y] = (u8)rec;   // right column of TU 0/2
    }
    HEVCE_ATOMIC_ADD(&sm.cand_sse[ci], sse);
}

// phase runners: one (non-inlined) copy per TU size, shared by all node sizes
typedef int Team;   // team id of a phase: 0 = all threads of the picture, 1 = team A, 2 = team B (team_first / team_size)
template <int T>
HEVCE_HD HEVCE_NOINLINE void run_borders(const Grp& gref, int off, Team tm) {
    Shared& sm = my_sm();
    const Grp g = gref;   // by value: keeps the descriptor in registers instead of re-reading the caller's stack
    if (g.n == 0) return;
    const Shared& pm = pic_sm();
    if (!g.priv) { PAR_FOR_TEAM(j, 4 * T + 1, tm, off) border_column<T>(sm, pm, g, j, 0, 0); }
    else {   // private neighbours: the candidate loop of one border index is shared by four work items
        const int per = (g.n + 3) >> 2;
        PAR_FOR_TEAM(it, 4 * (4 * T + 1), tm, off) {
            const int j = it >> 2, c0 = (it & 3) * per;
            border_column<T>(sm, pm, g, j, c0, imin(g.n, c0 + per));
        }
    }
}
template <int T>
HEVCE_HD HEVCE_NOINLINE void run_phase_a(const Grp& gref, int off, Team tm) {
    Shared& sm = my_sm();
    const Grp g = gref;
    const Shared& pm = pic_sm();
    PAR_FOR_TEAM(item, g.n * T, tm, off) phase_a_item<T>(sm, pm, g, item);
}
template <int T>
HEVCE_HD HEVCE_NOINLINE void run_phase_b(const Grp& gref, int off, int q, Team tm) {
    Shared& sm = my_sm();
    const Grp g = gref;
    const RdK rk = rd_consts(q);
    const Shared& pm = pic_sm();
    PAR_FOR_TEAM(item, g.n * T, tm, off) phase_b_item<T>(sm, pm, g, item, q, rk);
}
template <int T>
HEVCE_HD HEVCE_NOINLINE void run_phase_c(const Scratch& scref, const Grp& gref, int off, int q, Team tm) {
    Shared& sm = my_sm();
    const Grp g = gref;
    const Scratch sc = scref;
    PAR_FOR_TEAM(item, g.n * T, tm, off) phase_c_item<T>(sm, sc, g, item, q);
}
template <int T>
HEVCE_HD HEVCE_NOINLINE void run_phase_d(const Scratch& scref, const Grp& gref, int off, Team tm) {
    Shared& sm = my_sm();
    const Grp g = gref;
    const Scratch sc = scref;
    const Shared& pm = pic_sm();
    PAR_FOR_TEAM(item, g.n * T, tm, off) phase_d_item<T>(sm, pm, sc, g, item);
}
// phase D of a group for every picture of the gang, on the upper-half threads that host no trial lane
template <int T>
HEVCE_HD HEVCE_NOINLINE void run_phase_d_free(const Grp& gref, int first) {
    const Grp g = gref;
    const int per = g.n * T;
    GANG_FOR_UPPER_FREE(it, first, GANG_RT * per) {
        const int pic = it / per;
        Shared& ps = gang_sm(pic);
        const Scratch sc = ps.sc;
        phase_d_item<T>(ps, ps, sc, g, it - pic * per);
    }
}

// shared-memory carve-up of the pool for a node of size S: group 0 = one-TU candidates (T = S), group 1 = four-TU
// candidates (T = S/2), group 2 (S = 8 only) = NxN PU candidates (T = 4)
template <int S> struct Plan {
    static constexpr int H = S / 2;
    // Gang variants (18 KB pool per picture): 16x16 nodes take the one-TU candidates 6 per round beside the four sub-TU
    // rounds; 32x32 nodes run in two stages that reuse the pool: R0 one-TU rounds of 4 candidates (128 line items of
    // T = 32: one full pass), then 3 chunks of 12 four-TU candidates x 4 sub-TUs.
    // Wide variant (one picture per CTA, 185 KB pool): all 35 one-TU candidates in round 0 beside sub-TU 0 of all 35
    // four-TU candidates, then sub-TUs 1..3: four rounds for every node size.
    static constexpr int N0 = (S == 8 || WIDE) ? 35 : S == 16 ? 6 : 4;     // one-TU candidates per round
    static constexpr int N1 = (S == 32 && !WIDE) ? 12 : 35;                // four-TU candidates per chunk
    static constexpr int R0 = (S == 32 && !WIDE) ? 9 : 0;                  // gang 32x32: one-TU-only rounds that come first
    static constexpr int ROUNDS = WIDE ? 4 : S == 32 ? R0 + 12 : S == 16 ? 6 : 4; // gang 16x16: 4 sub-TU rounds + 2 one-TU-only
    static constexpr bool OVERLAY = S == 32 && !WIDE;                      // group 1 reuses group 0's pool space
    // round r: one-TU candidates [g0_m0, g0_m0 + g0_n), four-TU candidates [g1_m0, g1_m0 + g1_n) at sub-TU g1_tu
    static HEVCE_HD int g0_m0(int r) { return r * N0; }
    static HEVCE_HD int g0_n(int r) { return (r < 0 || (OVERLAY && r >= R0)) ? 0 : imax(0, imin(N0, NMODE - r * N0)); }
    static HEVCE_HD int g1_tu(int r) { return (r - R0) & 3; }
    static HEVCE_HD int g1_m0(int r) { return ((r - R0) >> 2) * N1; }
    static HEVCE_HD int g1_n(int r) { return r < R0 ? 0 : imax(0, imin(N1, NMODE - g1_m0(r))); }
    static constexpr int al(int v) { return (v + 15) & ~15; }
    // group 0
    static constexpr int BLK0 = 0;
    static constexpr int PRED0 = BLK0 + al(N0 * Dim<S>::BLK * 2);
    static constexpr int PSUM0 = PRED0 + al(N0 * S * S);
    static constexpr int BORD0 = PSUM0 + al(N0 * S * S);         // S*S/4 ints
    static constexpr int END0 = BORD0 + al(2 * Dim<S>::BS);
    // group 1
    static constexpr int BLK1 = OVERLAY ? 0 : END0;
    static constexpr int PRED1 = BLK1 + al(N1 * Dim<H>::BLK * 2);
    static constexpr int PSUM1 = PRED1 + al(N1 * H * H);
    static constexpr int BORD1 = PSUM1 + al(N1 * H * H);
    static constexpr int REC1 = BORD1 + al(N1 * Dim<H>::BS);
    static constexpr int END1 = REC1 + al(N1 * 4 * H);           // sub-TU edges only
    // group 2 (S == 8)
    static constexpr int BLK2 = END1;
    static constexpr int PRED2 = BLK2 + al(35 * Dim<4>::BLK * 2);
    static constexpr int PSUM2 = PRED2 + al(35 * 16);
    static constexpr int BORD2 = PSUM2 + al(35 * 16);
    static constexpr int REC2 = BORD2 + al(2 * Dim<4>::BS);
    static constexpr int END2 = REC2 + al(35 * 16);
    static constexpr int TOTAL = S == 8 ? END2 : OVERLAY ? (END0 > END1 ? END0 : END1) : END1;
    static_assert(TOTAL <= POOL_BYTES, "shared-memory pool too small");
    static_assert(S != 8 || TOTAL <= AUX_CODER, "8x8 pipeline buffers overlap the trial-coder results");
};

HEVCE_HD inline Bac make_bac(const Coder& c) {
    Bac b;
    b.c = c; b.out = nullptr; b.cap = 0;
    b.use_tables(my_tb());
    return b;
}
HEVCE_HD inline int sm_off(const Shared& sm, const void* p) { return (int)((const u8*)p - (const u8*)&sm); }

// One trial-coder lane: candidates 0..69 code the whole CU from the node snapshot (HEVCe.c:1434-1438, 1470-1474);
// candidates 70..104 are NxN PU modes: residual alone from a fresh coder and fresh contexts (HEVCe.c:1505-1519).
template <int S>
HEVCE_HD inline void trial_lane(int pic, int trk, int cand, int depth, int y0, int x0) {
    Shared& sm = blk_sm(local_block(pic, trk));      // the track's block: lane contexts, candidate results, scratch
    const Shared& pm = blk_sm(picture_block(pic, trk));   // the picture: maps, snapshots
    const int my = 1 + y0 / 4, mx = 1 + x0 / 4;
    const int split_ctx = (S > pm.msz[my * 9 + mx - 1]) + (S > pm.msz[(my - 1) * 9 + mx]);
    const int pmL = pm.mpm[my * 9 + mx - 1], pmA = pm.mpm[(my - 1) * 9 + mx];
    const Scratch& sc = sm.sc;
    constexpr int H = S / 2;
    const bool pu = cand >= 2 * NMODE;
    const int slot = pu ? cand - 2 * NMODE : cand;   // context-set lane
    const int step = cand / NMODE, mode = cand - step * NMODE;
    Bac b = make_bac(pm.snap[depth]);
    if (pu) coder_reset(b.c);
    const int base_len = pu ? coder_len(b.c) : coder_len(pm.snap[depth]);
    u32* lane_cx = sm.lane_ctx + slot * CTXW;
    if (pu) {   // everything the residual of a 4x4 luma TU touches sits in the first CTXW4 words (see the layout at CX_LASTX4)
        const u32* src = (const u32*)pm.ctx0;
#pragma unroll
        for (int k = 0; k < CTXW4; k++) lane_cx[k] = src[k];
    } else {
        const u32* src = (const u32*)pm.snap_ctx[depth];
#pragma unroll
        for (int k = 0; k < CTXW; k++) lane_cx[k] = src[k];
    }
    CuDesc d;
    d.s = S; d.kind = pu ? 3 : step; d.split_ctx = split_ctx;
    d.pm[0] = mode; d.pl[0] = pmL; d.pa[0] = pmA;
    const s16* lev = sc.glev + (size_t)cand * LEV_STRIDE;
    if (step == 1) {
        for (int k = 0; k < 4; k++) { d.lev[k] = lev + k * H * H; d.mlo[k] = sm.cgnz[cand][k]; }
        d.mhi = 0;
    } else {
        d.lev[0] = lev; d.mlo[0] = sm.cgnz[cand][0]; d.mhi = pu ? 0u : sm.cgnz[cand][1];
    }
    code_cu<Bac, MainEnv>(b, local_block(pic, trk), sm_off(sm, lane_cx), d);
    const int bits = coder_len(b.c) - base_len;
    if (pu) sm.cand_bits[cand] = bits;
    else {   // the lane leaves its RD cost (the distortion is complete since phase D) and its end state
        sm.cand_bits[cand] = rd_cost(rd_consts(pm.q), sm.cand_sse[cand], bits);
        cand_coder(sm)[cand] = b.c;
    }
}

// The NxN CU as a whole, trial-coded from the node snapshot (HEVCe.c:1531-1544)
HEVCE_HD inline void nxn_trial(Shared& sm, int pic, int depth, int y0, int x0) {
    const int my = 1 + y0 / 4, mx = 1 + x0 / 4;
    const int pmL = sm.mpm[my * 9 + mx - 1], pmA = sm.mpm[(my - 1) * 9 + mx];
    Bac b = make_bac(sm.snap[depth]);
    for (int i = 0; i < CTXW; i++) ((u32*)sm.nxn_ctx)[i] = ((const u32*)sm.snap_ctx[depth])[i];
    CuDesc d;
    d.s = 8; d.kind = 2; d.split_ctx = (8 > sm.msz[my * 9 + mx - 1]) + (8 > sm.msz[(my - 1) * 9 + mx]); d.mhi = 0;
    for (int k = 0; k < 4; k++) { d.pm[k] = sm.nxn_pm[k]; d.lev[k] = sm.nxn_lev[k]; d.mlo[k] = sm.nxn_nz[k]; }
    d.pl[0] = pmL;     d.pa[0] = pmA;
    d.pl[1] = d.pm[0]; d.pa[1] = sm.mpm[(my - 1) * 9 + mx + 1];
    d.pl[2] = sm.mpm[(my + 1) * 9 + mx - 1]; d.pa[2] = d.pm[0];
    d.pl[3] = d.pm[2]; d.pa[3] = d.pm[1];
    code_cu<Bac, MainEnv>(b, local_block(pic, 0), sm_off(sm, sm.nxn_ctx), d);
    int sse = 0;
    for (int y = 0; y < 8; y++)
        for (int x = 0; x < 8; x++) { const int dd = (int)sm.orig[(y0 + y) * CTU + x0 + x] - HEVCE_WIN(sm, y0 + y, x0 + x); sse += dd * dd; }
    sm.nxn_cost = rd_cost(rd_consts(sm.q), sse, coder_len(b.c) - coder_len(sm.snap[depth]));
    sm.nxn_coder = b.c;
}

// The non-split candidates of one CU node (HEVCe.c:1420-1544): pixel rounds and trial coders.  Runs on the threads of
// the node size's track with that track's pool / scratch; it reads the picture only outside the CU (reference samples,
// neighbour maps) and the node's entry snapshot, so with tracks it runs while the children are being decided.
template <int S>
HEVCE_HD HEVCE_NOINLINE void eval_candidates(int q, int y0, int x0, const Avail& av, int depth) {
    Shared& sm = my_sm();
    const Scratch sc = sm.sc;
    typedef Plan<S> P;
    constexpr int H = S / 2;
    const RdK rk = rd_consts(q);

    // ---- group descriptors (uniform over the threads of a picture)
    auto group0 = [&](int r) -> Grp {   // one-TU candidates: a slice of the 35 modes per round
        Grp g;
        const int m0 = P::g0_m0(r), n = P::g0_n(r);
        g.n = n; g.cand0 = m0; g.mode0 = m0; g.ty = y0; g.tx = x0; g.av = av; g.priv = 0;
        g.cuy = y0; g.cux = x0; g.cus = S; g.tu = 0; g.one_tu = 1; g.grec = 1;
        g.blk = P::BLK0; g.pred = P::PRED0; g.psum = P::PSUM0; g.bord = P::BORD0;
        g.rec = -1; g.rec_stride = 0; g.rec_pitch = 0;
        return g;
    };
    auto group1 = [&](int r) -> Grp {   // four-TU candidates: sub-TU k of a chunk of modes, each with its own reconstruction as neighbour
        Grp g;
        const int k = P::g1_tu(r), m0 = P::g1_m0(r), n = P::g1_n(r);
        g.n = n; g.cand0 = NMODE + m0; g.mode0 = m0; g.ty = y0 + (k >> 1) * H; g.tx = x0 + (k & 1) * H; g.av = sub_avail(av, k); g.priv = 1;
        g.cuy = y0; g.cux = x0; g.cus = S; g.tu = k; g.one_tu = 0; g.grec = 1;
        g.blk = P::BLK1; g.pred = P::PRED1; g.psum = P::PSUM1; g.bord = P::BORD1;
        g.rec = P::REC1; g.rec_stride = 4 * H; g.rec_pitch = 0;
        return g;
    };
    auto group2 = [&](int k) -> Grp {   // 8x8 nodes: NxN PU k, all 35 modes, neighbours from the window (earlier PUs' winners are already there)
        Grp g;
        g.n = 35; g.cand0 = 2 * NMODE; g.mode0 = 0; g.ty = y0 + (k >> 1) * 4; g.tx = x0 + (k & 1) * 4; g.av = sub_avail(av, k); g.priv = 0;
        g.cuy = g.ty; g.cux = g.tx; g.cus = 4; g.tu = 0; g.one_tu = 0; g.grec = 0;
        g.blk = P::BLK2; g.pred = P::PRED2; g.psum = P::PSUM2; g.bord = P::BORD2;
        g.rec = P::REC2; g.rec_stride = 16; g.rec_pitch = 4;
        return g;
    };

    if constexpr (S > 8) {
        const Team all = 0;
        for (int r = 0; r < P::ROUNDS; r++) {
            const Grp g0 = group0(r), g1 = group1(r);
            const int i0 = g0.n * S;
            // ---- phase 0: reference samples (the one-TU border is the same in every round)
            if (r == 0) run_borders<S>(g0, 0, all);
            run_borders<H>(g1, r == 0 ? 4 * S + 1 : 0, all);
            PHASE_END_T(P_BORDER);
            // ---- phases A..D: warp-local hand-over (see WARP_SYNC)
            if (g0.n) run_phase_a<S>(g0, 0, all);
            if (g1.n) run_phase_a<H>(g1, i0, all);
            WARP_SYNC();
            if (g0.n) run_phase_b<S>(g0, 0, q, all);
            if (g1.n) run_phase_b<H>(g1, i0, q, all);
            WARP_SYNC();
            if (g0.n) run_phase_c<S>(sc, g0, 0, q, all);
            if (g1.n) run_phase_c<H>(sc, g1, i0, q, all);
            WARP_SYNC();
            if (g0.n) run_phase_d<S>(sc, g0, 0, all);
            if (g1.n) run_phase_d<H>(sc, g1, i0, all);
            PHASE_END_T(P_D_TRIAL);
        }
    } else {
        // 8x8 nodes: two independent chains.  Team A (lower half of every picture's threads) evaluates the one-TU and
        // four-TU candidates; team B (upper half) walks the four NxN PUs, whose CABAC lanes are the long pole.  Team A
        // reads the window outside the CU only and team B writes it inside the CU only, so the chains meet at the end.
        TEAM_A {
            const Team ta = 1;
            TEAM_PROF_BEGIN();
            for (int r = 0; r < 4; r++) {
                const Grp g0 = group0(r), g1 = group1(r);
                const int i0 = g0.n * S;
                run_borders<S>(g0, 0, ta);
                run_borders<H>(g1, 4 * S + 1, ta);
                TEAM_SYNC(1);
                if (g0.n) run_phase_a<S>(g0, 0, ta);
                run_phase_a<H>(g1, i0, ta);
                WARP_SYNC();
                if (g0.n) run_phase_b<S>(g0, 0, q, ta);
                run_phase_b<H>(g1, i0, q, ta);
                WARP_SYNC();
                if (g0.n) run_phase_c<S>(sc, g0, 0, q, ta);
                run_phase_c<H>(sc, g1, i0, q, ta);
                WARP_SYNC();
                if (g0.n) run_phase_d<S>(sc, g0, 0, ta);
                run_phase_d<H>(sc, g1, i0, ta);
                TEAM_SYNC(1);
                TEAM_PROF(P_TA, 0);
            }
        }
        TEAM_B {
            const Team tb = 2;
            TEAM_PROF_BEGIN();
            for (int k = 0; k < 4; k++) {
                const Grp g2 = group2(k);
                run_borders<4>(g2, 0, tb);
                TEAM_SYNC(2);
                run_phase_a<4>(g2, 0, tb);
                WARP_SYNC();
                run_phase_b<4>(g2, 0, q, tb);
                WARP_SYNC();
                run_phase_c<4>(sc, g2, 0, q, tb);
                TEAM_SYNC(2);
                TEAM_PROF(P_TB_PIX, NTA);
                // NxN PU coders of this PU, all pictures of the gang, packed into full warps; the threads left over
                // reconstruct the candidates meanwhile (phase D of any picture of the gang)
                GANG_FOR_UPPER(u, GANG_RT * NMODE) {
                    const int pic = u / NMODE, m = u - pic * NMODE;
                    trial_lane<S>(pic, 0, 2 * NMODE + m, depth, y0, x0);
                }
                run_phase_d_free<4>(g2, GANG_RT * NMODE);
                TEAM_SYNC(2);
                TEAM_PROF(P_TB_CABAC, NTA);
                PAR_FOR_TEAM(m, NMODE, 2, 0) sm.cand_bits[2 * NMODE + m] = rd_cost(rk, sm.cand_sse[2 * NMODE + m], sm.cand_bits[2 * NMODE + m]);
                TEAM_SYNC(2);
                PAR_FOR_TEAM(i, 16, 2, 0) {   // best PU mode, last minimum wins (HEVCe.c:1521); one sample per thread
                    int best = IMAX, bm = 0;
                    for (int m = 0; m < NMODE; m++) {
                        const int c = sm.cand_bits[2 * NMODE + m];
                        if (best >= c) { best = c; bm = m; }
                    }
                    const int ci = 2 * NMODE + bm;
                    if (i == 0) { sm.nxn_pm[k] = bm; sm.nxn_nz[k] = sm.cgnz[ci][0]; }
                    sm.nxn_lev[k][i] = sc.glev[(size_t)ci * LEV_STRIDE + i];
                    HEVCE_WIN(sm, g2.ty + (i >> 2), g2.tx + (i & 3)) = sm.pool[g2.rec + bm * 16 + i];
                }
                TEAM_SYNC(2);
                TEAM_PROF(P_TB_ARGMIN, NTA);
            }
        }
        TEAM_JOIN();
        PHASE_END_T(P_D_TRIAL);
    }

    // ---- all one-TU / four-TU trial coders of the gang (70 per picture), packed step-major into full warps; for 8x8
    // nodes one more lane per picture codes the NxN CU as a whole
    {
        const int NC = GANG_RT * NMODE;
#if defined(HEVCE_PROFILE) && defined(__CUDA_ARCH__)
        const long long tw0_ = clock64();
#endif
        const int trk = HEVCE_TRK;
        const int NCP = round_lanes(NC, trk_lpw(trk));   // every step starts on a warp boundary: one-TU, four-TU and NxN lanes run
                                               // different code and would serialise inside a shared warp
        GANG_FOR(L, 2 * NCP + (S == 8 ? GANG_RT : 0)) {
            if (L < 2 * NCP) {
                const int step = L >= NCP, r = L - step * NCP, pic = r / NMODE, m = r - pic * NMODE;
                if (r < NC) trial_lane<S>(pic, trk, step * NMODE + m, depth, y0, x0);
            } else nxn_trial(gang_sm(L - 2 * NCP), L - 2 * NCP, depth, y0, x0);
        }
#if defined(HEVCE_PROFILE) && defined(__CUDA_ARCH__)
        __syncwarp();
        if ((threadIdx.x & 31) == 0) {   // per-warp duration of the trial pass, by node size
            constexpr int base = S == 8 ? 24 : S == 16 ? 56 : 88;   // 32 warp slots per node size
            atomicAdd(&g_phase_cycles[base + threadIdx.x / 32], (unsigned long long)(clock64() - tw0_));
            atomicAdd(&g_phase_count[base + threadIdx.x / 32], 1ull);
        }
#endif
    }
    PHASE_END_T(P_TRIAL);
}

// Decision of one CU node and adoption of the winner (HEVCe.c:1440, 1476, 1546-1559), on track 0; `cm` is the block of
// the track that evaluated the node's candidates.
template <int S>
HEVCE_HD HEVCE_NOINLINE void decide_adopt(int q, int y0, int x0, int depth) {
    Shared& sm = my_sm();
    constexpr int CT = TrackOf<S>::value;
    Shared& cm = CT == 0 ? sm : *remote_blk(CT);   // the evaluating track's block (cluster variant: in the other CTA)
    const Scratch sc = sm.sc_of[CT];
    constexpr int N4 = S / 4;
    const RdK rk = rd_consts(q);
    const int my = 1 + y0 / 4, mx = 1 + x0 / 4;
    // split alternative: distortion of what the children left in the window (HEVCe.c:1409-1410)
    if (S > 8) {
        PAR_FOR(row, S) {
            int acc = 0;
            for (int x = 0; x < S; x++) { const int d = (int)sm.orig[(y0 + row) * CTU + x0 + x] - HEVCE_WIN(sm, y0 + row, x0 + x); acc += d * d; }
            sm.part_sse[row] = acc;
        }
        if (CT != 0) PAR_FOR(c, 2 * NMODE) sm.cand_bits[c] = cm.cand_bits[c];   // the parent track's RD costs, fetched in parallel
        PHASE_END_T(P_DECIDE);
    }

    // ---- decision, reference order; every comparison is ">=" so the last minimum wins
    PAR_FOR(one, 1) {
        int best = IMAX, win = -1;
        if (S > 8) {
            int sse = 0;
            for (int r = 0; r < S; r++) sse += sm.part_sse[r];
            best = rd_cost(rk, sse, coder_len(sm.live) - coder_len(sm.snap[depth]));
        }
        for (int c = 0; c < 2 * NMODE; c++) {   // one-TU modes 0..34, then four-TU modes 0..34 (HEVCe.c:1440, 1476)
            const int cost = sm.cand_bits[c];   // RD cost, left by the candidate's trial lane
            if (best >= cost) { best = cost; win = c; }
        }
        if (S == 8 && best >= sm.nxn_cost) win = NCAND;   // HEVCe.c:1546
        sm.win_item = win;
    }
    PHASE_END_T(P_DECIDE);
    const int win = sm.win_item;   // < 0: the split stays: live state, window, levels and maps are already the children's
    // ---- adoption
    s16* clev = sm.ctu_lev + zoff(y0, x0);
    if (win < 0) {
        // nothing to adopt; still take the barrier below (all pictures of a CTA keep the same barrier sequence)
    } else if (win == NCAND) {
        PAR_FOR(i, 64) clev[i] = sm.nxn_lev[i >> 4][i & 15];
        PAR_FOR(i, CTXW) ((u32*)sm.live_ctx)[i] = ((const u32*)sm.nxn_ctx)[i];
        PAR_FOR(one, 1) {
            sm.live = sm.nxn_coder;
            sm.kind[(y0 >> 3) * 4 + (x0 >> 3)] = 2;
            for (int k = 0; k < 4; k++) {
                sm.msz[(my + (k >> 1)) * 9 + mx + (k & 1)] = 8;
                sm.mpm[(my + (k >> 1)) * 9 + mx + (k & 1)] = (u8)sm.nxn_pm[k];
            }
        }
    } else {
        const int step = win >= NMODE, mode = win - step * NMODE;
        const u8* rp = sc.grec + (size_t)win * (CTU * CTU);
        const s16* lp = sc.glev + (size_t)win * LEV_STRIDE;
        PAR_FOR(i, S * S) {
            HEVCE_WIN(sm, y0 + i / S, x0 + i % S) = rp[i];
            clev[i] = lp[i];
        }
        PAR_FOR(i, CTXW) ((u32*)sm.live_ctx)[i] = cm.lane_ctx[win * CTXW + i];
        PAR_FOR(i, N4 * N4) {
            const int idx = (my + i / N4) * 9 + mx + i % N4;
            sm.msz[idx] = (u8)S;
            sm.mpm[idx] = (u8)mode;
        }
        PAR_FOR(i, (S / 8) * (S / 8)) {
            const int n8 = S / 8;
            sm.kind[((y0 >> 3) + i / n8) * 4 + (x0 >> 3) + i % n8] = (u8)step;
        }
        PAR_FOR(one, 1) sm.live = cand_coder(cm)[win];
    }
    PHASE_END_T(P_ADOPT);
}

// without tracks: a node's candidates and its decision by the same threads, after its children
template <int S>
HEVCE_HD inline void eval_node(int q, int y0, int x0, const Avail& av, int depth) {
    eval_candidates<S>(q, y0, x0, av, depth);
    decide_adopt<S>(q, y0, x0, depth);
}

// enter a node: snapshot the live state (HEVCe.c:1364-1365) and, for splittable nodes, code split_cu_flag = 1
template <int S>
HEVCE_HD inline void enter_node(Shared& sm, int y0, int x0, int depth) {
    PAR_FOR(i, CTXW) ((u32*)sm.snap_ctx[depth])[i] = ((const u32*)sm.live_ctx)[i];
    PAR_FOR(one, 1) sm.snap[depth] = sm.live;
    PHASE_END_T(P_ENTER);
    if (S > 8) {
        PAR_FOR(one, 1) {
            const int my = 1 + y0 / 4, mx = 1 + x0 / 4;
            Bac b = make_bac(sm.live);
            const Cx cx = {sm.live_ctx};
            b.put_bin(my_tb(), 1, cx[CX_SPLIT_CU + (S > sm.msz[my * 9 + mx - 1]) + (S > sm.msz[(my - 1) * 9 + mx])]);   // HEVCe.c:943-947
            sm.live = b.c;
        }
        PHASE_END_T(P_ENTER);
    }
}

// Commit pass: re-encode one decided CTU with the byte-writing coder from its recorded start state (replaces the
// reference's per-trial byte buffers).  One thread per CTU in hevce_commit_kernel; CTUs are independent here because
// the decision kernel recorded every CTU's start state and byte offset.
HEVCE_HD inline void commit_cu(BacCommit& b, int cx_off, const CtuRec& r, const s16* ctu_lev, int s, int y0, int x0) {
    const int my = 1 + y0 / 4, mx = 1 + x0 / 4, h = s / 2;
    CuDesc d;
    d.s = s; d.kind = r.kind[(y0 >> 3) * 4 + (x0 >> 3)]; d.split_ctx = -1; d.mhi = 0;
    d.pm[0] = r.mpm[my * 9 + mx];
    d.pl[0] = r.mpm[my * 9 + mx - 1];
    d.pa[0] = r.mpm[(my - 1) * 9 + mx];
    if (d.kind == 2) {
        d.pm[1] = r.mpm[my * 9 + mx + 1]; d.pm[2] = r.mpm[(my + 1) * 9 + mx]; d.pm[3] = r.mpm[(my + 1) * 9 + mx + 1];
        d.pl[1] = d.pm[0]; d.pa[1] = r.mpm[(my - 1) * 9 + mx + 1];
        d.pl[2] = r.mpm[(my + 1) * 9 + mx - 1]; d.pa[2] = d.pm[0];
        d.pl[3] = d.pm[2]; d.pa[3] = d.pm[1];
    }
    const s16* lev = ctu_lev + zoff(y0, x0);
    if (d.kind == 0) { d.lev[0] = lev; scan_groups(lev, s, d.mlo[0], d.mhi); }
    else
        for (int k = 0; k < 4; k++) { unsigned hi; d.lev[k] = lev + k * h * h; scan_groups(d.lev[k], h, d.mlo[k], hi); }
    code_cu<BacCommit, CommitEnv>(b, 0, cx_off, d);
}

HEVCE_HD inline void commit_ctu(const Job& job, int ctu, int lane) {
    CommitShared& cs = my_csm();
    const CtuRec& r = job.recs[ctu];
    const s16* lev = job.levs + (size_t)ctu * (CTU * CTU);
    u32* cw = cs.ctx + lane * CTXW;
    for (int k = 0; k < CTXW; k++) cw[k] = ((const u32*)r.ctx)[k];
    const int cx_off = (int)((u8*)cw - (u8*)&cs);
    const Cx cx = {(u8*)cw};
    BacCommit b;
    b.use_tables(cs.tb);
    b.c = r.start;
    b.out = job.out + r.out_pos;
    b.cap = imax(0, job.out_cap - r.out_pos);
    auto gt = [&](int s, int y, int x) { return (s > r.msz[(1 + y / 4) * 9 + 1 + x / 4 - 1]) + (s > r.msz[(1 + y / 4 - 1) * 9 + 1 + x / 4]); };
    const int whole = r.msz[10] == 32;
    b.put_bin(cs.tb, !whole, cx[CX_SPLIT_CU + gt(32, 0, 0)]);
    if (whole) commit_cu(b, cx_off, r, lev, 32, 0, 0);
    else
        for (int a = 0; a < 4; a++) {
            const int y16 = (a >> 1) * 16, x16 = (a & 1) * 16;
            const int sz = r.msz[(1 + y16 / 4) * 9 + 1 + x16 / 4];
            b.put_bin(cs.tb, sz != 16, cx[CX_SPLIT_CU + gt(16, y16, x16)]);
            const int ncu = sz == 16 ? 1 : 4;
            for (int c = 0; c < ncu; c++) {
                if (sz == 16) commit_cu(b, cx_off, r, lev, 16, y16, x16);
                else commit_cu(b, cx_off, r, lev, 8, y16 + (c >> 1) * 8, x16 + (c & 1) * 8);
            }
        }
    b.put_terminate(r.last);   // HEVCe.c:1630
    if (r.last) b.finish();    // HEVCe.c:1640
    int err = 0;
    if (!coder_equal(b.c, r.end)) err |= ERR_COMMIT_MISMATCH;   // the adopted trial state must be what the bytes produce
    if (!r.last) {
        const u32* nx = (const u32*)job.recs[ctu + 1].ctx;
        for (int k = 0; k < CTXW; k++) if (cw[k] != nx[k]) err |= ERR_COMMIT_MISMATCH;
    }
    if (b.c.n > b.cap) err |= ERR_OVERFLOW;
    if (err) HEVCE_ATOMIC_OR(job.result + 1, err);
}

// stream header (HEVCe.c:665-691): constant NAL units with ue(width), ue(height) spliced into the SPS
HEVCE_HD inline int write_header(u8* out, int q, int H, int W) {
    const u8 VPS[27] = {0, 0, 1, 0x40, 1, 0x0c, 1, 0xff, 0xff, 3, 0x10, 0, 0, 3, 0, 0, 3, 0, 0, 3, 0, 0, 3, 0, 0xb4, 0xf0, 0x24};
    const u8 SPS[22] = {0, 0, 1, 0x42, 1, 1, 3, 0x10, 0, 0, 3, 0, 0, 3, 0, 0, 3, 0, 0, 3, 0, 0xb4};
    const u8 PPS[11] = {0, 0, 1, 0x44, 1, 0xc0, 0x90, 0x91, 0x81, 0xd9, 0x20};
    const u8 SLICE[6] = {0, 0, 1, 0x26, 1, 0xac};
    const u8 SQP[5][2] = {{0x16, 0xde}, {0x10, 0xde}, {0x2b, 0x78}, {0x4d, 0xe0}, {0x97, 0x80}};
    int n = 0;
    for (int i = 0; i < 27; i++) out[n++] = VPS[i];
    for (int i = 0; i < 22; i++) out[n++] = SPS[i];
    unsigned long long acc = 0;   // bit writer, MSB first
    int nb = 0;
    auto put = [&](unsigned v, int len) {
        for (int i = len - 1; i >= 0; i--) {
            acc = (acc << 1) | ((v >> i) & 1);
            if (++nb == 8) { out[n++] = (u8)acc; acc = 0; nb = 0; }
        }
    };
    auto ue = [&](int v) {   // the reference's ue(v): length derived from v+2 (HEVCe.c:642-648)
        int len = 1;
        v++;
        for (int t = v + 1; t != 1; t >>= 1) len += 2;
        put((unsigned)(v & ((1 << ((len + 1) >> 1)) - 1)), (len >> 1) + ((len + 1) >> 1));
    };
    put(0x0a, 4);
    ue(W);
    ue(H);
    put(0x197ee4, 22);
    put(0x681ed1, 24);
    if (nb) { out[n++] = (u8)(acc << (8 - nb)); }
    for (int i = 0; i < 11; i++) out[n++] = PPS[i];
    for (int i = 0; i < 6; i++) out[n++] = SLICE[i];
    out[n++] = SQP[q][0];
    out[n++] = SQP[q][1];
    return n;
}

// ------------------------------------------------------------------------------------------------------------
// one picture (HEVCe.c:1570-1647)
// ------------------------------------------------------------------------------------------------------------
// `scs`: the global scratch of this picture slot, one set per track
HEVCE_HD inline void encode_picture(const Job& job, const Scratch* scs) {
    Shared& sm = pic_sm();
    const Scratch sc = scs[0];
    const int q = job.q, H = job.H, W = job.W;
#define PIC_FOR(item, n) if (PAR_FOR_ALL_OWNER) PAR_FOR_ALL(item, n)   /* picture-wide phase: all threads of the picture */
    PIC_FOR(i, 4 * CTXW) {
        const u8 v = ctx_init_value(my_tb().ctx_iv[i], q);
        sm.ctx0[i] = v;
        sm.live_ctx[i] = v;
    }
    PIC_FOR(i, 81) { sm.msz[i] = CTU; sm.mpm[i] = 1; }
    PIC_FOR(i, W / 4) sc.msz_line[i] = CTU;
    for (int t = 0; t < NTRACK; t++)
        ON_TRACK(t) PAR_FOR(one, 1) my_sm().sc = scs[t];    // every track: its own scratch
    ON_TRACK(0) PAR_FOR(t, NTRACK) sm.sc_of[t] = scs[t];
    unsigned rdv1 = 0, rdv2 = 0;                            // rendezvous counters (uniform over the threads of a track)
    PIC_FOR(one, 1) {
        coder_reset(sm.live);
        sm.error = 0;
        sm.q = q;
        sm.stream_pos = write_header(job.out, q, H, W);
    }
    BAR_ALL();

    int ctu_idx = 0;
    for (int cy = 0; cy < H; cy += CTU) {
        for (int cx = 0; cx < W; cx += CTU, ctu_idx++) {
            const Avail av = {cx > 0, 0, cy > 0, cy > 0 && cx + CTU < W};   // HEVCe.c:1606-1609
            // ---- load: original (edge-replicated), neighbour samples, neighbour maps
            PIC_FOR(i, CTU * CTU) {
                const int y = imin(cy + i / CTU, job.src_h - 1), x = imin(cx + i % CTU, job.src_w - 1);
                sm.orig[i] = job.img[(size_t)y * job.src_w + x];
            }
            PIC_FOR(i, CTU) sm.win[(1 + i) * WP] = cx > 0 ? job.rcon[(size_t)(cy + i) * W + cx - 1] : (u8)0;
            PIC_FOR(j, 2 * CTU + 1) sm.win[j] = cy > 0 ? job.rcon[(size_t)(cy - 1) * W + iclip(cx - 1 + j, 0, W - 1)] : (u8)0;
            PIC_FOR(i, 8) {
                sm.msz[i + 1] = sc.msz_line[cx / 4 + i];                               // above row: CU sizes scroll,
                sm.mpm[i + 1] = 1;                                                     // modes stay DC (HEVCe.c:1634-1637)
                sm.msz[(i + 1) * 9] = cx > 0 ? sm.msz[(i + 1) * 9 + 8] : (u8)CTU;      // left column = previous CTU's last column
                sm.mpm[(i + 1) * 9] = cx > 0 ? sm.mpm[(i + 1) * 9 + 8] : (u8)1;
            }
            CtuRec& rec = job.recs[ctu_idx];
            PIC_FOR(i, CTXW) ((u32*)rec.ctx)[i] = ((const u32*)sm.live_ctx)[i];
            PIC_FOR(one, 1) { sm.live.n = 0; rec.start = sm.live; sm.ctu_lev = job.levs + (size_t)ctu_idx * (CTU * CTU); }
            BAR_ALL();

            // ---- CU quadtree, z-order (HEVCe.c:1403-1413)
            if (!TRACKS) {   // children before the parent's own candidates, everything on the same threads
                enter_node<32>(sm, 0, 0, 0);
                for (int a = 0; a < 4; a++) {
                    const int y16 = (a >> 1) * 16, x16 = (a & 1) * 16;
                    const Avail av16 = sub_avail(av, a);
                    enter_node<16>(sm, y16, x16, 1);
                    for (int c = 0; c < 4; c++) {
                        const int y8 = y16 + (c >> 1) * 8, x8 = x16 + (c & 1) * 8;
                        enter_node<8>(sm, y8, x8, 2);
                        eval_node<8>(q, y8, x8, sub_avail(av16, c), 2);
                    }
                    eval_node<16>(q, y16, x16, av16, 1);
                }
                eval_node<32>(q, 0, 0, av, 0);
            } else {
                // Parent || child: as soon as a node's entry snapshot exists (rendezvous), its own candidates are evaluated
                // on the node size's track while track 0 walks the children; the decision waits for both (second rendezvous).
                ON_TRACK(0) enter_node<32>(sm, 0, 0, 0);
                TRACK_START(2, ++rdv2);
                ON_TRACK(2) eval_candidates<32>(q, 0, 0, av, 0);
                for (int a = 0; a < 4; a++) {
                    const int y16 = (a >> 1) * 16, x16 = (a & 1) * 16;
                    const Avail av16 = sub_avail(av, a);
                    ON_TRACK(0) enter_node<16>(sm, y16, x16, 1);
                    TRACK_START(1, ++rdv1);
                    ON_TRACK(1) eval_candidates<16>(q, y16, x16, av16, 1);
                    ON_TRACK(0) {
                        for (int c = 0; c < 4; c++) {
                            const int y8 = y16 + (c >> 1) * 8, x8 = x16 + (c & 1) * 8;
                            enter_node<8>(sm, y8, x8, 2);
                            eval_node<8>(q, y8, x8, sub_avail(av16, c), 2);
                        }
                    }
                    TRACK_END(1, rdv1);
                    ON_TRACK(0) decide_adopt<16>(q, y16, x16, 1);
                }
                TRACK_END(2, rdv2);
                ON_TRACK(0) decide_adopt<32>(q, 0, 0, 0);
                BAR_ALL();
            }

            // ---- store reconstruction + map row, terminate bin, commit the CTU's bytes
            PIC_FOR(i, CTU * CTU) job.rcon[(size_t)(cy + i / CTU) * W + cx + i % CTU] = HEVCE_WIN(sm, i / CTU, i % CTU);
            PIC_FOR(i, 8) sc.msz_line[cx / 4 + i] = sm.msz[8 * 9 + 1 + i];
            PIC_FOR(i, 81) { rec.msz[i] = sm.msz[i]; rec.mpm[i] = sm.mpm[i]; }
            PIC_FOR(i, 16) rec.kind[i] = sm.kind[i];
            PIC_FOR(one, 1) {
                const int last = cy + CTU >= H && cx + CTU >= W;
                Bac t = make_bac(sm.live);
                t.put_terminate(last);                                                  // HEVCe.c:1630
                if (last) t.finish();                                                   // HEVCe.c:1640
                rec.end = t.c;
                rec.out_pos = sm.stream_pos;
                rec.last = last;
                sm.stream_pos += t.c.n;                                                 // bytes the commit pass will write
                sm.live = t.c;
            }
            BAR_ALL();
        }
    }
    PIC_FOR(one, 1) {
        job.result[0] = sm.stream_pos;
        if (sm.error) HEVCE_ATOMIC_OR(job.result + 1, sm.error);
    }
    BAR_ALL();
#undef PIC_FOR
}

}   // namespace HEVCE_NS
