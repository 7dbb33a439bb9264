// hevce_deblock.h -- the HEVC in-loop luma deblocking filter (H.265 section 8.7.2) for the streams this library writes:
// every CU intra, so boundary strength 2 on every transform edge of the 8x8 grid; one QP per picture; no SAO.
//
// The stream header leaves the filter on, so a conforming decoder outputs deblock(reconstruction): that is the decoded
// picture.  hevce_cuda.cu runs these functions in hevce_deblock_kernel; tests/sim/hevce_simdeblock.cpp runs the same
// source on the host, every CTA and every work item in the kernel's phase order.
//
// One CTA filters one CTU of one picture, from the reconstruction into a separate output plane:
//   load        the CTU with a 4-sample halo on every side (rows y0-4 .. y0+35, columns x0-4 .. x0+35) and the
//               transform-block size of every 4x4 unit of the CTU and of the unit rows next to it in the CTUs above
//               and below (their CtuRec msz / kind bytes; nothing else of a CtuRec is read);
//   vertical    edges x0, x0+8, .., x0+32 over all 40 tile rows, in place.  An edge reads 4 and writes 3 samples on
//               each side, so edges 8 apart touch disjoint samples;
//   horizontal  edges y0, y0+8, .., y0+32 over the CTU's 32 columns, in place, on the vertically filtered tile;
//   store       the CTU's 32x32 samples.
// Every vertical edge a horizontal edge of this CTU reads through is in the tile, so each CTA sees the picture with all
// its vertical edges filtered, as 8.7.2 requires.  Neighbouring CTAs filter the edges they share from the same samples
// and each keeps its own side: one read (plus halo) and one write per sample.
#pragma once
#include "hevce_core.h"

namespace HEVCE_NS {

constexpr int DBK_THREADS = 64;
constexpr int DBK_TS = CTU + 8;                    // tile side: the CTU and 4 samples of halo each way
constexpr int DBK_UR = CTU / 4 + 2;                // unit rows of the TU-size map: the row above, the CTU's 8, the row below
constexpr int DBK_LOAD_ITEMS = DBK_TS * 4 + DBK_UR * (CTU / 4);   // per tile row: halo word, 2 x 16 samples, halo word; map units
constexpr int DBK_VERT_ITEMS = 5 * (DBK_TS / 4);   // 5 edges x 10 four-row segments
constexpr int DBK_HORZ_ITEMS = 5 * (CTU / 4);      // 5 edges x 8 four-column segments
constexpr int DBK_STORE_ITEMS = CTU * 2;           // 32 rows x 2 x 16 samples

struct alignas(16) DbkTile {
    u8 px[DBK_TS * DBK_TS];           // px[r * DBK_TS + c] = sample (y0 - 4 + r, x0 - 4 + c); 0 outside the picture
    u8 tu[DBK_UR * (CTU / 4)];        // transform-block size of 4x4 unit (uy, ux) at [(uy + 1) * 8 + ux], uy = -1 .. 8
};

struct alignas(16) Dbk16 { u32 w[4]; };

// beta = BETA[QP] (Table 8-12), tc = TC[QP + 2] for bS = 2, QP = 6 * qpd6 + 4: QP 4 .. 28, so QP + 2 <= 30
HEVCE_HD inline int dbk_beta(int q) { const int qp = 6 * q + 4; return qp < 16 ? 0 : qp - 10; }
HEVCE_HD inline int dbk_tc(int q) { const int t = 6 * q + 6; return t < 18 ? 0 : t < 27 ? 1 : 2; }
// qpd6 0-1: beta = tc = 0, no edge passes d < beta and the decoded picture is the reconstruction
HEVCE_HD inline bool dbk_active(const Job& job) { return dbk_beta(job.q) > 0; }
HEVCE_HD inline int dbk_nctu(const Job& job) { return (job.H / CTU) * (job.W / CTU); }

HEVCE_HD inline void dbk_load(DbkTile& t, const Job& job, int ctu, int item) {
    const int cw = job.W / CTU, y0 = (ctu / cw) * CTU, x0 = (ctu % cw) * CTU;
    if (item < DBK_TS * 4) {
        const int r = item >> 2, k = item & 3, y = y0 - 4 + r;
        u32* d = (u32*)(t.px + r * DBK_TS) + (k == 0 ? 0 : k == 3 ? 9 : 1 + 4 * (k - 1));
        const bool row_in = y >= 0 && y < job.H;
        const u8* s = job.rcon + (size_t)(row_in ? y : 0) * job.W + x0;
        if (k == 1 || k == 2) {                    // 16 samples of the CTU row: rows are 32-byte aligned
            Dbk16 v = {{0, 0, 0, 0}};
            if (row_in) v = *(const Dbk16*)(s + 16 * (k - 1));
            for (int i = 0; i < 4; i++) d[i] = v.w[i];
        } else {                                   // 4 halo samples left or right, absent at the picture border
            const bool in = row_in && (k == 0 ? x0 > 0 : x0 + CTU < job.W);
            d[0] = in ? *(const u32*)(s + (k == 0 ? -4 : CTU)) : 0u;
        }
        return;
    }
    const int m = item - DBK_TS * 4, ur = m / (CTU / 4) - 1, ux = m % (CTU / 4);
    int c = ctu, uy = ur;                          // unit row -1 is row 7 of the CTU above, row 8 is row 0 of the CTU below
    if (ur < 0) { c -= cw; uy = 7; }
    if (ur > 7) { c += cw; uy = 0; }
    int tu = CTU;
    if (c >= 0 && c < dbk_nctu(job)) {             // no CTU there: no segment of that row is filtered
        const CtuRec& rec = job.recs[c];
        const int cu = rec.msz[(1 + uy) * 9 + 1 + ux], kind = rec.kind[(uy >> 1) * 4 + (ux >> 1)];
        tu = kind == 0 ? cu : kind == 1 ? cu >> 1 : 4;
    }
    t.tu[(ur + 1) * (CTU / 4) + ux] = (u8)tu;
}

// One 4-line segment of an edge (8.7.2.5.3, .6, .7).  p points at q0 of line 0; `across` steps from q0 to q1 (p0 is at
// -across), `along` from line to line.
HEVCE_HD inline void dbk_segment(u8* p, int across, int along, int beta, int tc) {
    auto S = [&](int line, int i) -> int { return p[line * along + i * across]; };   // i >= 0: q_i, i < 0: p_(-i-1)
    const int dp0 = iabs(S(0, -3) - 2 * S(0, -2) + S(0, -1)), dp3 = iabs(S(3, -3) - 2 * S(3, -2) + S(3, -1));
    const int dq0 = iabs(S(0, 2) - 2 * S(0, 1) + S(0, 0)), dq3 = iabs(S(3, 2) - 2 * S(3, 1) + S(3, 0));
    const int dpq0 = dp0 + dq0, dpq3 = dp3 + dq3;
    if (dpq0 + dpq3 >= beta) return;
    auto dsam = [&](int line, int dpq) {
        return 2 * dpq < (beta >> 2) && iabs(S(line, -4) - S(line, -1)) + iabs(S(line, 0) - S(line, 3)) < (beta >> 3) &&
               iabs(S(line, -1) - S(line, 0)) < ((5 * tc + 1) >> 1);
    };
    const bool strong = dsam(0, dpq0) && dsam(3, dpq3);
    const int side = (beta + (beta >> 1)) >> 3;
    const bool dep = dp0 + dp3 < side, deq = dq0 + dq3 < side;
    for (int l = 0; l < 4; l++) {
        u8* q = p + l * along;
        const int p0 = q[-across], p1 = q[-2 * across], p2 = q[-3 * across], p3 = q[-4 * across];
        const int q0 = q[0], q1 = q[across], q2 = q[2 * across], q3 = q[3 * across];
        if (strong) {
            const int t2 = 2 * tc;
            q[-across] = (u8)iclip((p2 + 2 * p1 + 2 * p0 + 2 * q0 + q1 + 4) >> 3, p0 - t2, p0 + t2);
            q[-2 * across] = (u8)iclip((p2 + p1 + p0 + q0 + 2) >> 2, p1 - t2, p1 + t2);
            q[-3 * across] = (u8)iclip((2 * p3 + 3 * p2 + p1 + p0 + q0 + 4) >> 3, p2 - t2, p2 + t2);
            q[0] = (u8)iclip((p1 + 2 * p0 + 2 * q0 + 2 * q1 + q2 + 4) >> 3, q0 - t2, q0 + t2);
            q[across] = (u8)iclip((p0 + q0 + q1 + q2 + 2) >> 2, q1 - t2, q1 + t2);
            q[2 * across] = (u8)iclip((p0 + q0 + q1 + 3 * q2 + 2 * q3 + 4) >> 3, q2 - t2, q2 + t2);
        } else {
            int delta = (9 * (q0 - p0) - 3 * (q1 - p1) + 8) >> 4;
            if (iabs(delta) >= tc * 10) continue;
            delta = iclip(delta, -tc, tc);
            q[-across] = (u8)iclip(p0 + delta, 0, 255);
            q[0] = (u8)iclip(q0 - delta, 0, 255);
            const int tc2 = tc >> 1;
            if (dep) q[-2 * across] = (u8)iclip(p1 + iclip((((p2 + p0 + 1) >> 1) - p1 + delta) >> 1, -tc2, tc2), 0, 255);
            if (deq) q[across] = (u8)iclip(q1 + iclip((((q2 + q0 + 1) >> 1) - q1 - delta) >> 1, -tc2, tc2), 0, 255);
        }
    }
}

// Vertical edge x0 + 8e on the tile rows 4s .. 4s+3.  The CTU's outline is always a transform edge (TUs do not cross
// CTUs); an inner edge is one where the Q-side unit's transform block starts.  Picture borders are never filtered.
HEVCE_HD inline void dbk_vertical(DbkTile& t, const Job& job, int ctu, int item) {
    const int cw = job.W / CTU, y0 = (ctu / cw) * CTU, x0 = (ctu % cw) * CTU;
    const int e = item % 5, s = item / 5, x = x0 + 8 * e, y = y0 - 4 + 4 * s;
    if (x == 0 || x >= job.W || y < 0 || y >= job.H) return;
    if (e > 0 && e < 4 && (8 * e) % t.tu[s * (CTU / 4) + 2 * e] != 0) return;
    dbk_segment(t.px + (4 * s) * DBK_TS + 4 + 8 * e, 1, DBK_TS, dbk_beta(job.q), dbk_tc(job.q));
}

// Horizontal edge y0 + 8e on the CTU's columns 4s .. 4s+3.
HEVCE_HD inline void dbk_horizontal(DbkTile& t, const Job& job, int ctu, int item) {
    const int cw = job.W / CTU, y0 = (ctu / cw) * CTU;
    const int e = item % 5, s = item / 5, y = y0 + 8 * e;
    if (y == 0 || y >= job.H) return;
    if (e > 0 && e < 4 && (8 * e) % t.tu[(1 + 2 * e) * (CTU / 4) + s] != 0) return;
    dbk_segment(t.px + (4 + 8 * e) * DBK_TS + 4 + 4 * s, DBK_TS, 1, dbk_beta(job.q), dbk_tc(job.q));
}

// dec: the picture's output plane, H x W like job.rcon
HEVCE_HD inline void dbk_store(const DbkTile& t, const Job& job, int ctu, u8* dec, int item) {
    const int cw = job.W / CTU, y0 = (ctu / cw) * CTU, x0 = (ctu % cw) * CTU;
    const int r = item >> 1, h = item & 1;
    const u32* s = (const u32*)(t.px + (4 + r) * DBK_TS) + 1 + 4 * h;
    Dbk16 v;
    for (int i = 0; i < 4; i++) v.w[i] = s[i];
    *(Dbk16*)(dec + (size_t)(y0 + r) * job.W + x0 + 16 * h) = v;
}

}   // namespace HEVCE_NS
