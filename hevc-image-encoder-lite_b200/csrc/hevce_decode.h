// hevce_decode.h -- a decoder for the HEVC subset this library writes: the header check, the slice-data parser and the
// reconstruction, as HEVCE_HD functions.  hevce_cuda.cu runs them in hevce_parse_kernel and hevce_recon_kernel, then
// hevce_deblock_kernel (hevce_deblock.h) runs unchanged on the result; tests/sim/hevce_simdecode.cpp runs the same source
// on the host in the kernels' phase order.
//
// Accepted streams: exactly the parameter sets and slice header write_header() produces for some picture size H x W
// (multiples of 32, at most DEC_MAX_DIM) and qpd6 0..4, followed by the slice data.  That is one I slice, CTB 32, minimum
// CB 8, TB 4..32, max_transform_hierarchy_depth_intra 1, 4:2:0 with every chroma cbf 0, no sign hiding, transform skip,
// scaling lists, SAO, PCM, tiles or WPP, deblocking on, one QP = 6 * qpd6 + 4.  write_header is the only statement of it.
//
// Parse (one thread per picture; the CABAC state threads through the whole slice): H.265 9.3.4.3 decoding engine with the
// encoder's Tables words, the syntax of 7.3.8 in spec order with the context selection of 9.3.4.2 in the compact CX_*
// layout.  Each CTU fills its CtuRec's msz / mpm / kind bytes as the encoder does (unpack_partition reads them, and so
// does the deblocking filter) and its levels into a 32 x 32 block: coefficient (y, x) of the TU at CTU position
// (ty, tx) is at [(ty + y) * 32 + tx + x].  Every loop is bounded by the syntax; reads past the end of the data return
// zero bits and set an error, so corrupt input ends with status DEC_ERR, never out of bounds.
//
// Reconstruction (8.4.4.2, 8.6): per TU in z-order, reference samples with z-scan availability (6.4.1), substitution and
// [1 2 1] filtering, planar / DC / angular prediction with the edge filters below 32 x 32, flat scaling, the inverse
// DST / DCT with the 16-bit clip between the stages, and the residual added with a clip.  The work of one TU is split
// into phases whose items are independent (reference samples, substitution, filtering, columns, rows).
#pragma once
#include "hevce_core.h"

namespace HEVCE_NS {

constexpr int DEC_MAX_DIM = 16384;
constexpr int DEC_HDR_CAP = 128;   // write_header writes at most 27 + 22 + 8 + 11 + 8 bytes
enum { DEC_OK = 0, DEC_ERR = 1 };

// ---- header check ------------------------------------------------------------------------------------------------
// Size and qpd6 of a stream whose parameter sets and slice header are the bytes write_header(q, H, W) produces.
// Returns the header length (the first byte of the slice data), or -1.
HEVCE_HD inline int dec_header(const u8* s, int len, int& H, int& W, int& q) {
    // pic_width / pic_height_in_luma_samples: ue(v) at bit 4 of the SPS payload that follows the 27-byte VPS and the
    // 22 constant SPS bytes (write_header)
    const int b0 = 8 * (27 + 22) + 4;
    int pos = b0;
    auto bit = [&](int p) -> int { return (p >> 3) < len ? (s[p >> 3] >> (7 - (p & 7))) & 1 : 0; };
    auto ue = [&]() -> int {
        int lz = 0;
        while (lz < 20 && !bit(pos)) { lz++; pos++; }
        if (lz >= 20) return -1;
        pos++;
        int v = 0;
        for (int i = 0; i < lz; i++) v = (v << 1) | bit(pos++);
        return (1 << lz) - 1 + v;
    };
    if (len < 27 + 22 + 4) return -1;
    W = ue();
    H = ue();
    if (H < CTU || W < CTU || H > DEC_MAX_DIM || W > DEC_MAX_DIM || H % CTU || W % CTU) return -1;
    u8 ref[DEC_HDR_CAP];
    for (q = 0; q <= 4; q++) {
        const int n = write_header(ref, q, H, W);
        if (n > len) continue;
        int same = 1;
        for (int i = 0; i < n; i++) same &= s[i] == ref[i];
        if (same) return n;
    }
    return -1;
}

// ---- slice data reader: emulation prevention removed, every read bounded by the length ---------------------------
struct DecBits {
    const u8* p;
    int pos, end;        // next byte, end of the data
    int zeros;           // consecutive zero bytes just read (emulation prevention)
    unsigned long long cache;
    int nc;              // valid bits in cache
    int err;
};

HEVCE_HD inline int dec_byte(DecBits& b) {
    if (b.pos < b.end && b.zeros >= 2 && b.p[b.pos] == 3) { b.pos++; b.zeros = 0; }
    if (b.pos >= b.end) { b.err = 1; return 0; }
    const int v = b.p[b.pos++];
    b.zeros = v ? 0 : b.zeros + 1;
    return v;
}
HEVCE_HD inline unsigned dec_bits(DecBits& b, int n) {   // n <= 24
    while (b.nc < n) { b.cache = (b.cache << 8) | (unsigned)dec_byte(b); b.nc += 8; }
    b.nc -= n;
    return (unsigned)(b.cache >> b.nc) & ((1u << n) - 1);
}

// ---- CABAC decoding engine (9.3.4.3) -------------------------------------------------------------------------------
struct DecCabac {
    DecBits bs;
    unsigned range, value;   // value: the 9-bit ivlOffset
};

HEVCE_HD inline void dec_cabac_init(DecCabac& d, const u8* data, int start, int end) {
    d.bs.p = data; d.bs.pos = start; d.bs.end = end; d.bs.zeros = 0; d.bs.cache = 0; d.bs.nc = 0; d.bs.err = 0;
    d.range = 510;
    d.value = dec_bits(d.bs, 9);
}

// one context-coded bin; cx = state << 1 | mps (Tables::st8: bytes 0..3 LPS range by range quarter, byte 4 the context
// after an LPS, byte 5 after an MPS)
HEVCE_HD inline int dec_bin(DecCabac& d, const Tables& tb, u8& cx) {
    const unsigned long long e = tb.st8[cx & 127];
    const unsigned lps = (unsigned)(e >> (8 * ((d.range >> 6) & 3))) & 0xffu;
    d.range -= lps;
    if (d.value < d.range) {
        cx = (u8)(e >> 40);
        const int bin = cx & 1 ? 1 : 0;   // the MPS does not change on an MPS transition
        if (d.range < 256) { d.range <<= 1; d.value = (d.value << 1) | dec_bits(d.bs, 1); }
        return bin;
    }
    const int bin = !(cx & 1);
    d.value -= d.range;
    const int sh = 9 - bitlen(lps);
    d.range = lps << sh;
    d.value = (d.value << sh) | dec_bits(d.bs, sh);
    cx = (u8)(e >> 32);
    return bin;
}
HEVCE_HD inline int dec_bypass(DecCabac& d) {
    d.value = (d.value << 1) | dec_bits(d.bs, 1);
    if (d.value >= d.range) { d.value -= d.range; return 1; }
    return 0;
}
HEVCE_HD inline unsigned dec_bypass_n(DecCabac& d, int n) {   // n <= 32, first bin most significant
    unsigned v = 0;
    for (int i = 0; i < n; i++) v = (v << 1) | (unsigned)dec_bypass(d);
    return v;
}
HEVCE_HD inline int dec_terminate(DecCabac& d) {
    d.range -= 2;
    if (d.value >= d.range) return 1;   // no renormalization: the last bit read is rbsp_stop_one_bit
    if (d.range < 256) { d.range <<= 1; d.value = (d.value << 1) | dec_bits(d.bs, 1); }
    return 0;
}

// ---- residual_coding (7.3.8.11) of one luma TU of size ts with intra mode m; lev: the TU's first level, stride CTU --
HEVCE_HD HEVCE_NOINLINE void dec_residual(DecCabac& d, const Tables& tb, u8* cx, int ts, int m, s16* lev, int& err) {
    const int st = scan_type(ts, m), lg = ilog2(ts), ncg = ts >> 2;
    const int sigbase = CX_SIG + 9 + (ts >= 16 ? 12 : 0) + ((ts == 8 && st) ? 6 : 0);
    auto cgpos = [&](int g, int& cy, int& cxg) {
        if (lg == 2) { cy = 0; cxg = 0; }
        else if (st == 1) { cy = g >> 1; cxg = g & 1; }
        else if (st == 2) { cy = g & 1; cxg = g >> 1; }
        else { const int v = tb.cgdiag[lg - 3][g]; cy = v >> 3; cxg = v & 7; }
    };
    // last_sig_coeff_x / y prefix (TR, cMax 2 * lg - 1) and suffix
    const int gmax = tb.grp[ts - 1], sh = ts > 4;
    const int bx = cx_lastx(lg - 2), by = cx_lasty(lg - 2);
    int gx = 0, gy = 0;
    while (gx < gmax && dec_bin(d, tb, cx[bx + (gx >> sh)])) gx++;
    while (gy < gmax && dec_bin(d, tb, cx[by + (gy >> sh)])) gy++;
    int lx = gx > 3 ? tb.gmin[gx] + (int)dec_bypass_n(d, (gx - 2) >> 1) : gx;
    int ly = gy > 3 ? tb.gmin[gy] + (int)dec_bypass_n(d, (gy - 2) >> 1) : gy;
    if (st == 2) { const int t = lx; lx = ly; ly = t; }
    // sub-block and scan position of the last coefficient
    const int lcy = ly >> 2, lcx = lx >> 2, kstart = tb.inv4[st][((ly & 3) << 2) | (lx & 3)];
    int gl = 0;
    for (int g = ncg * ncg - 1; g > 0; g--) {
        int cy, cxg;
        cgpos(g, cy, cxg);
        if (cy == lcy && cxg == lcx) { gl = g; break; }
    }
    unsigned long long csbf = 0;   // coded_sub_block_flag, bit cy * 8 + cxg
    auto coded = [&](int cy, int cxg) -> int { return cy < ncg && cxg < ncg ? (int)((csbf >> (cy * 8 + cxg)) & 1u) : 0; };
    int c1 = 1;
    for (int g = gl; g >= 0; g--) {
        int cy, cxg;
        cgpos(g, cy, cxg);
        const int rgt = coded(cy, cxg + 1), dwn = coded(cy + 1, cxg), pat = (dwn << 1) | rgt;
        int on = 1;
        if (g != gl && g != 0) on = dec_bin(d, tb, cx[CX_SIGCG + (pat != 0)]);
        if (!on) continue;
        csbf |= 1ull << (cy * 8 + cxg);
        const int first_cg = g == 0;
        const unsigned long long tab = ts == 4 ? tb.sig4[st] : tb.sigoff[st][pat];
        const int base = ts == 4 ? CX_SIG : sigbase + (first_cg ? 0 : 3);
        unsigned nzm = 0;
        int k = 15;
        if (g == gl) { nzm = 1u << kstart; k = kstart - 1; }
        const int infer_dc = g != gl && g != 0;   // position 0 is inferred significant when nothing else is
        for (; k >= 0; k--) {
            if (k == 0 && infer_dc && nzm == 0) { nzm |= 1u; break; }
            int ci = base + (int)((tab >> (4 * k)) & 15u);
            if (first_cg && ts != 4 && k == 0) ci = CX_SIG;
            nzm |= (unsigned)dec_bin(d, tb, cx[ci]) << k;
        }
        if (!nzm) continue;
        // greater1 / greater2 flags, signs, remaining levels, in reverse scan order
        const int set = (first_cg ? 0 : 2) + (c1 == 0);
        c1 = 1;
        int pos[16], lvl[16], nz = 0, first_g1 = -1, esc = 0;
        for (int kk = 15; kk >= 0; kk--)
            if ((nzm >> kk) & 1u) pos[nz++] = kk;
        esc = nz > 8;
        for (int i = 0; i < nz; i++) {
            lvl[i] = 1;
            if (i < 8) {
                const int big = dec_bin(d, tb, cx[CX_ONE + 4 * set + c1]);
                lvl[i] += big;
                if (big) { c1 = 0; if (first_g1 < 0) first_g1 = i; else esc = 1; }
                else if (c1 > 0 && c1 < 3) c1++;
            }
        }
        if (first_g1 >= 0) {
            const int g2 = dec_bin(d, tb, cx[CX_ABS + set]);
            lvl[first_g1] += g2;
            esc |= g2;
        }
        const unsigned signs = dec_bypass_n(d, nz);
        if (esc) {
            int rp = 0;
            for (int i = 0; i < nz; i++) {
                const int bl = i < 8 ? (i == first_g1 ? 3 : 2) : 1;
                if (lvl[i] != bl) continue;
                // coeff_abs_level_remaining (9.3.3.11): prefix of at most 32 ones, then a TR or k-th order EG suffix
                int p = 0;
                while (p < 32 && dec_bypass(d)) p++;
                if (p == 32) { err = 1; return; }
                long long v;
                if (p < 3) v = ((long long)p << rp) + dec_bypass_n(d, rp);
                else {
                    const int n = p - 3 + rp;
                    v = (((1ll << (p - 3)) + 2) << rp) + (long long)dec_bypass_n(d, n);
                }
                const long long a = lvl[i] + v;
                lvl[i] = a > 32768 ? 32768 : (int)a;   // levels are 16-bit
                if (lvl[i] > (3 << rp)) rp = imin(rp + 1, 4);
            }
        }
        for (int i = 0; i < nz; i++) {
            const int p4 = tb.scan4[st][pos[i]], y = cy * 4 + (p4 >> 2), x = cxg * 4 + (p4 & 3);
            const int neg = (signs >> (nz - 1 - i)) & 1u;
            lev[y * CTU + x] = (s16)(neg ? -lvl[i] : imin(lvl[i], 32767));
        }
    }
}

// ---- one CTU -------------------------------------------------------------------------------------------------------
// Partition maps as the encoder keeps them: msz / mpm [1 + uy][1 + ux] over the 4x4 units of the CTU plus the unit row
// above (CU sizes of the CTU above, modes DC: the above neighbour is unavailable across a CTU row) and the unit column to
// the left (the previous CTU's last column, or size 32 / DC at the picture's left edge); kind per 8x8 unit.
struct DecMaps { u8 msz[81], mpm[81], kind[16]; };

HEVCE_HD HEVCE_NOINLINE void dec_cu(DecCabac& d, const Tables& tb, u8* cx, DecMaps& mp, int s, int y0, int x0, s16* lev, int& err) {
    const int my = 1 + y0 / 4, mx = 1 + x0 / 4, n4 = s / 4;
    const int nxn = s == 8 ? !dec_bin(d, tb, cx[CX_PART]) : 0;   // part_mode: 1 = 2Nx2N
    const int npu = nxn ? 4 : 1;
    int flag[4], mode[4];
    for (int i = 0; i < npu; i++) flag[i] = dec_bin(d, tb, cx[CX_YPM]);
    for (int i = 0; i < npu; i++) {
        const int uy = my + (nxn ? i >> 1 : 0), ux = mx + (nxn ? i & 1 : 0);
        int c[3];
        mpm_list(mp.mpm[uy * 9 + ux - 1], mp.mpm[(uy - 1) * 9 + ux], c);
        if (flag[i]) {
            const int idx = dec_bypass(d) ? 1 + dec_bypass(d) : 0;
            mode[i] = c[idx];
        } else {
            int r = (int)dec_bypass_n(d, 5);
            if (c[0] > c[1]) { const int t = c[0]; c[0] = c[1]; c[1] = t; }
            if (c[0] > c[2]) { const int t = c[0]; c[0] = c[2]; c[2] = t; }
            if (c[1] > c[2]) { const int t = c[1]; c[1] = c[2]; c[2] = t; }
            for (int j = 0; j < 3; j++) if (r >= c[j]) r++;
            mode[i] = r;
        }
        if (nxn) { mp.msz[uy * 9 + ux] = 8; mp.mpm[uy * 9 + ux] = (u8)mode[i]; }
        else
            for (int u = 0; u < n4 * n4; u++) { mp.msz[(my + u / n4) * 9 + mx + u % n4] = (u8)s; mp.mpm[(my + u / n4) * 9 + mx + u % n4] = (u8)mode[i]; }
    }
    if (dec_bin(d, tb, cx[CX_UVPM])) dec_bypass_n(d, 2);   // intra_chroma_pred_mode
    const int split = nxn ? 1 : dec_bin(d, tb, cx[CX_SPLIT_TU + (s == 32 ? 0 : s == 16 ? 1 : 2)]);
    if (dec_bin(d, tb, cx[CX_UVCBF]) | dec_bin(d, tb, cx[CX_UVCBF])) err = 1;   // chroma residual: outside the subset
    const int kind = nxn ? 2 : split;
    for (int u = 0; u < (s / 8) * (s / 8); u++) mp.kind[((y0 >> 3) + u / (s / 8)) * 4 + (x0 >> 3) + u % (s / 8)] = (u8)kind;
    const int ntu = split ? 4 : 1, ts = split ? s / 2 : s;
    for (int k = 0; k < ntu; k++) {
        const int ty = y0 + (k >> 1) * ts, tx = x0 + (k & 1) * ts;
        if (dec_bin(d, tb, cx[CX_YCBF + !split])) dec_residual(d, tb, cx, ts, mode[nxn ? k : 0], lev + ty * CTU + tx, err);
        if (err) return;
    }
}

// coding_quadtree of one CTU and its end_of_slice_segment_flag; returns 0, or DEC_ERR
HEVCE_HD HEVCE_NOINLINE int dec_ctu(DecCabac& d, const Tables& tb, u8* cx, DecMaps& mp, s16* lev, int last) {
    int err = 0;
    auto ctx = [&](int s, int y, int x) { return (s > mp.msz[(1 + y / 4) * 9 + x / 4]) + (s > mp.msz[(y / 4) * 9 + 1 + x / 4]); };
    if (!dec_bin(d, tb, cx[CX_SPLIT_CU + ctx(32, 0, 0)])) dec_cu(d, tb, cx, mp, 32, 0, 0, lev, err);
    else
        for (int a = 0; a < 4 && !err; a++) {
            const int y16 = (a >> 1) * 16, x16 = (a & 1) * 16;
            if (!dec_bin(d, tb, cx[CX_SPLIT_CU + ctx(16, y16, x16)])) dec_cu(d, tb, cx, mp, 16, y16, x16, lev, err);
            else
                for (int c = 0; c < 4 && !err; c++) dec_cu(d, tb, cx, mp, 8, y16 + (c >> 1) * 8, x16 + (c & 1) * 8, lev, err);
        }
    if (err || d.bs.err) return DEC_ERR;
    // end_of_slice_segment_flag: 0 after every CTU but the last.  The reference's flush (BacT::finish, HEVCe.c:840-856)
    // writes the coder's low register without its bit 7, where 9.3.2.5 puts the stop bit, so after the last CTU the
    // offset is either in the terminating interval or one below it; both end the slice.  What follows is not checked.
    if (!last) return dec_terminate(d) || d.bs.err ? DEC_ERR : DEC_OK;
    return d.value + 3 >= d.range && !d.bs.err ? DEC_OK : DEC_ERR;
}

// ---- one picture (hevce_parse_kernel: one thread) --------------------------------------------------------------------
// data / len: the stream, start: its header length (dec_header).  job.recs / job.levs receive the CTUs; levs must be
// zero on entry (only the non-zero levels are written).  After a failure every remaining CTU gets a one-TU 32x32 CU, so
// the records stay valid input for the deblocking filter.  Returns DEC_OK or DEC_ERR.
HEVCE_HD inline int dec_parse_picture(const Job& job, const u8* data, int start, int len, const Tables& tb) {
    DecCabac d;
    dec_cabac_init(d, data, start, len);
    u8 cx[4 * CTXW];
    for (int i = 0; i < 4 * CTXW; i++) cx[i] = ctx_init_value(tb.ctx_iv[i], job.q);
    DecMaps mp;
    const int cw = job.W / CTU, nctu = (job.H / CTU) * cw;
    int status = DEC_OK, c = 0;
    for (; c < nctu && status == DEC_OK; c++) {
        const int cy = c / cw, cxc = c % cw;
        for (int i = 0; i < 8; i++) {
            mp.msz[i + 1] = cy > 0 ? job.recs[c - cw].msz[8 * 9 + 1 + i] : (u8)CTU;
            mp.mpm[i + 1] = 1;
            mp.msz[(i + 1) * 9] = cxc > 0 ? mp.msz[(i + 1) * 9 + 8] : (u8)CTU;
            mp.mpm[(i + 1) * 9] = cxc > 0 ? mp.mpm[(i + 1) * 9 + 8] : (u8)1;
        }
        mp.msz[0] = CTU; mp.mpm[0] = 1;
        status = dec_ctu(d, tb, cx, mp, job.levs + (size_t)c * (CTU * CTU), c == nctu - 1);
        CtuRec& r = job.recs[c];
        for (int i = 0; i < 81; i++) { r.msz[i] = mp.msz[i]; r.mpm[i] = mp.mpm[i]; }
        for (int i = 0; i < 16; i++) r.kind[i] = mp.kind[i];
    }
    if (status != DEC_OK)
        for (int k = c - 1; k < nctu; k++) {
            CtuRec& r = job.recs[k];
            for (int i = 0; i < 81; i++) { r.msz[i] = CTU; r.mpm[i] = 1; }
            for (int i = 0; i < 16; i++) r.kind[i] = 0;
        }
    return status;
}

// ---- reconstruction --------------------------------------------------------------------------------------------------
struct DecTu { u8 y, x, s, m; };   // TU origin in CTU coordinates, size, luma intra mode

// the TUs of a parsed CTU in decoding (z-) order; returns their number (at most 64)
HEVCE_HD inline int dec_tu_list(const CtuRec& r, DecTu* tu) {
    int n = 0;
    auto cu = [&](int s, int y0, int x0) {
        const int kind = r.kind[(y0 >> 3) * 4 + (x0 >> 3)];
        if (kind == 0) { tu[n++] = DecTu{(u8)y0, (u8)x0, (u8)s, r.mpm[(1 + y0 / 4) * 9 + 1 + x0 / 4]}; return; }
        const int h = s / 2;
        for (int k = 0; k < 4; k++) {
            const int y = y0 + (k >> 1) * h, x = x0 + (k & 1) * h;
            tu[n++] = DecTu{(u8)y, (u8)x, (u8)h, r.mpm[(1 + (kind == 2 ? y : y0) / 4) * 9 + 1 + (kind == 2 ? x : x0) / 4]};
        }
    };
    auto sz = [&](int y, int x) { return r.msz[(1 + y / 4) * 9 + 1 + x / 4]; };
    if (sz(0, 0) == 32) cu(32, 0, 0);
    else
        for (int a = 0; a < 4; a++) {
            const int y16 = (a >> 1) * 16, x16 = (a & 1) * 16;
            if (sz(y16, x16) == 16) cu(16, y16, x16);
            else
                for (int c = 0; c < 4; c++) cu(8, y16 + (c >> 1) * 8, x16 + (c & 1) * 8);
        }
    return n;
}

// z-scan order of the 4x4 unit (uy, ux) inside a CTU
HEVCE_HD inline int dec_zs(int uy, int ux) {
    int z = 0;
    for (int b = 0; b < 3; b++) z |= (((ux >> b) & 1) << (2 * b)) | (((uy >> b) & 1) << (2 * b + 1));
    return z;
}

// 6.4.1: is sample (yn, xn) decoded before the TU whose first sample is (yc, xc)?  One slice, no tiles.
HEVCE_HD inline bool dec_available(const Job& job, int yn, int xn, int yc, int xc) {
    if (yn < 0 || xn < 0 || yn >= job.H || xn >= job.W) return false;
    const int cw = job.W / CTU, an = (yn / CTU) * cw + xn / CTU, ac = (yc / CTU) * cw + xc / CTU;
    if (an != ac) return an < ac;
    return dec_zs((yn % CTU) / 4, (xn % CTU) / 4) < dec_zs((yc % CTU) / 4, (xc % CTU) / 4);
}

// Working memory of one TU (one warp's shared memory on the device).  ref / flt: the unified reference array, index j
// = 0 .. 4T: j < 2T is the left column from the bottom (p[-1][2T-1-j]), 2T the corner, j > 2T the top row
// (p[j-2T-1][-1]).  tmp: the residual after the vertical stage, row-major with pitch CTU + 1.
struct DecTuWork {
    u8 ref[4 * CTU + 4], flt[4 * CTU + 4], avail[4 * CTU + 4];
    s16 tmp[CTU * (CTU + 1)];
};
HEVCE_HD inline int dec_ref_items(int T) { return 4 * T + 1; }

// phase 1, item j: reference sample j and whether it is available (8.4.4.2.2)
HEVCE_HD inline void dec_ref_item(DecTuWork& w, const Job& job, int y0, int x0, int T, int j) {
    int yn, xn;
    if (j < 2 * T) { yn = y0 + 2 * T - 1 - j; xn = x0 - 1; }
    else { yn = y0 - 1; xn = x0 + j - 2 * T - 1; }
    const bool a = dec_available(job, yn, xn, y0, x0);
#if defined(__CUDA_ARCH__)
    w.ref[j] = a ? *(volatile const u8*)(job.rcon + (size_t)yn * job.W + xn) : (u8)0;   // written by other warps of the CTA
#else
    w.ref[j] = a ? job.rcon[(size_t)yn * job.W + xn] : (u8)0;
#endif
    w.avail[j] = a;
}

// phase 2 (one item): substitution of the unavailable samples (8.4.4.2.2)
HEVCE_HD inline void dec_ref_substitute(DecTuWork& w, int T) {
    const int n = 4 * T + 1;
    int first = -1;
    for (int j = 0; j < n && first < 0; j++) if (w.avail[j]) first = j;
    if (first < 0) { for (int j = 0; j < n; j++) w.ref[j] = 128; return; }
    if (!w.avail[0]) w.ref[0] = w.ref[first];
    for (int j = 1; j < n; j++) if (!w.avail[j]) w.ref[j] = w.ref[j - 1];
}

// phase 3, item j: the [1 2 1] filter (8.4.4.2.3; strong intra smoothing is off); the two ends stay
HEVCE_HD inline void dec_filter_item(DecTuWork& w, int T, int j) {
    w.flt[j] = (j == 0 || j == 4 * T) ? w.ref[j] : (u8)((w.ref[j - 1] + 2 * w.ref[j] + w.ref[j + 1] + 2) >> 2);
}

// predicted sample (y, x) of a T x T TU with mode m (8.4.4.2.4-6); B[k]: k > 0 top[k-1], k < 0 left[-k-1], 0 corner
HEVCE_HD HEVCE_NOINLINE int dec_pred(const u8* B, int T, int lg, int m, int y, int x) {
    if (m == 0) return ((T - 1 - x) * B[-1 - y] + (x + 1) * B[T + 1] + (T - 1 - y) * B[1 + x] + (y + 1) * B[-T - 1] + T) >> (lg + 1);
    const bool edge = T < 32;
    if (m == 1) {
        int dc = T;
        for (int i = 0; i < T; i++) dc += B[-1 - i] + B[1 + i];
        dc >>= lg + 1;
        if (edge && x == 0 && y == 0) return (B[-1] + 2 * dc + B[1] + 2) >> 2;
        if (edge && y == 0) return (B[1 + x] + 3 * dc + 2) >> 2;
        if (edge && x == 0) return (B[-1 - y] + 3 * dc + 2) >> 2;
        return dc;
    }
    const int ang = intra_angle(m), aa = iabs(ang), inv = aa ? (8192 + aa / 2) / aa : 0;   // |invAngle| (Table 8-5)
    if (m >= 18) {   // vertical family: ref[k] = top, extended to k < 0 by projecting the left column
        if (m == 26 && edge && x == 0) return iclip(B[1 + x] + ((B[-1 - y] - B[0]) >> 1), 0, 255);
        auto R = [&](int k) -> int { return k >= 0 ? B[k] : B[-((128 - inv * k) >> 8)]; };
        const int off = ang * (y + 1), ii = off >> 5, f = off & 31, k = x + ii + 1;
        return f ? ((32 - f) * R(k) + f * R(k + 1) + 16) >> 5 : R(k);   // f = 0: ref[k + 1] may lie past the 2T samples
    }
    if (m == 10 && edge && y == 0) return iclip(B[-1 - y] + ((B[1 + x] - B[0]) >> 1), 0, 255);
    auto R = [&](int k) -> int { return k >= 0 ? B[-k] : B[(128 - inv * k) >> 8]; };
    const int off = ang * (x + 1), ii = off >> 5, f = off & 31, k = y + ii + 1;
    return f ? ((32 - f) * R(k) + f * R(k + 1) + 16) >> 5 : R(k);
}

// phase 4, item x: scaling (8.6.3, flat, QP = 6 q + 4) and the vertical inverse transform of column x (8.6.4.2)
template <int T>
HEVCE_HD HEVCE_NOINLINE void dec_column_t(DecTuWork& w, const s16* lev, int q, int x) {
    constexpr int LG = T == 4 ? 2 : T == 8 ? 3 : T == 16 ? 4 : 5;
    const int qs = 7 - LG + q;
    int v[T], o[T], any = 0;
    for (int k = 0; k < T; k++) { v[k] = iclip(lev[k * CTU + x] * (1 << qs), -32768, 32767); any |= v[k]; }
    if (any) {
        Xf<T>::i(v, o);
        for (int k = 0; k < T; k++) w.tmp[k * (CTU + 1) + x] = (s16)iclip((o[k] + 64) >> 7, -32768, 32767);
    } else {
        for (int k = 0; k < T; k++) w.tmp[k * (CTU + 1) + x] = 0;
    }
}
// phase 5, item y: the horizontal inverse transform of row y, prediction, reconstruction of the TU's row y
template <int T>
HEVCE_HD HEVCE_NOINLINE void dec_row_t(const DecTuWork& w, const Job& job, int y0, int x0, int m, int y) {
    constexpr int LG = T == 4 ? 2 : T == 8 ? 3 : T == 16 ? 4 : 5;
    const u8* B = (T > 4 && use_filtered(T, m) ? w.flt : w.ref) + 2 * T;
    int v[T], o[T], any = 0;
    for (int x = 0; x < T; x++) { v[x] = w.tmp[y * (CTU + 1) + x]; any |= v[x]; }
    if (any) Xf<T>::i(v, o);
    u8* out = job.rcon + (size_t)(y0 + y) * job.W + x0;
#pragma unroll 1
    for (int x = 0; x < T; x++) {
        const int res = any ? (o[x] + 2048) >> 12 : 0;
        out[x] = (u8)iclip(dec_pred(B, T, LG, m, y, x) + res, 0, 255);
    }
}
HEVCE_HD inline void dec_column(DecTuWork& w, const s16* lev, int T, int q, int x) {
    if (T == 4) dec_column_t<4>(w, lev, q, x);
    else if (T == 8) dec_column_t<8>(w, lev, q, x);
    else if (T == 16) dec_column_t<16>(w, lev, q, x);
    else dec_column_t<32>(w, lev, q, x);
}
HEVCE_HD inline void dec_row(const DecTuWork& w, const Job& job, int y0, int x0, int T, int m, int y) {
    if (T == 4) dec_row_t<4>(w, job, y0, x0, m, y);
    else if (T == 8) dec_row_t<8>(w, job, y0, x0, m, y);
    else if (T == 16) dec_row_t<16>(w, job, y0, x0, m, y);
    else dec_row_t<32>(w, job, y0, x0, m, y);
}

}   // namespace HEVCE_NS
