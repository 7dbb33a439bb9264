// hevce_simdecode.cpp -- host build of the decoder's source (TEST INFRASTRUCTURE ONLY).
//
// Runs the functions of csrc/hevce_decode.h and csrc/hevce_deblock.h over whole pictures in one thread, in the order of
// the kernels: hevce_parse_kernel (every picture), hevce_recon_kernel (every CTU of a picture, every TU of a CTU in z-order,
// the phases of a TU one after the other), hevce_deblock_kernel (as tests/sim/hevce_simdeblock.cpp).  With order = 1 the
// pictures are parsed last to first, the CTUs are reconstructed in the wavefront order of the kernel (CTU (r, c) at step
// c + 2 r, the CTUs of a step last to first) instead of raster order, and the items of every phase run last to first:
// the same output shows the items of a phase are independent and a two-CTU lag between CTU rows is enough.
//
// Built with -DHEVCE_SIMDECODE_MAIN it is a program for the sanitizer build: it decodes every truncation of a stream and
// a number of single-bit corruptions of its slice data, each from a buffer of exactly the stream's length.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "hevce_core.h"
#include "hevce_deblock.h"
#include "hevce_decode.h"

using namespace hevce;

// padded size, qpd6 and header length of a stream, or -1 when its header is rejected
extern "C" int hevce_simdecode_info(const u8* s, int len, int* H, int* W, int* q) {
    int h = 0, w = 0, qq = 0;
    const int n = dec_header(s, len, h, w, qq);
    if (n < 0) return -1;
    *H = h; *W = w; *q = qq;
    return n;
}

// n streams; rcons[i] / decs[i] (H x W of stream i) receive the picture before and after deblocking, cu_sizes / modes
// ((H/4) x (W/4)) and kinds ((H/8) x (W/8)) the parsed partition (any of these four may be NULL), status[i] 0 or 1.
// Returns 0, or -1 when a header is rejected (nothing is decoded then).
extern "C" int hevce_simdecode(int n, const u8* const* streams, const int* lens, u8* const* rcons, u8* const* decs, u8* const* cu_sizes,
                               u8* const* modes, u8* const* kinds, int* status, int order) {
    std::vector<Job> jobs((size_t)n);
    std::vector<int> start((size_t)n);
    std::vector<std::vector<CtuRec>> recs((size_t)n);
    std::vector<std::vector<s16>> levs((size_t)n);
    Tables tb;
    fill_tables(tb);
    for (int i = 0; i < n; i++) {
        Job& j = jobs[i];
        memset(&j, 0, sizeof(Job));
        if ((start[i] = dec_header(streams[i], lens[i], j.H, j.W, j.q)) < 0) return -1;
        const int nctu = (j.H / CTU) * (j.W / CTU);
        recs[i].resize((size_t)nctu);
        memset(recs[i].data(), 0xA5, sizeof(CtuRec) * nctu);
        levs[i].assign((size_t)nctu * CTU * CTU, 0);
        j.recs = recs[i].data();
        j.levs = levs[i].data();
        j.rcon = rcons[i];
    }
    auto item = [&](int i, int count) { return order ? count - 1 - i : i; };
    // hevce_parse_kernel
    for (int k = 0; k < n; k++) {
        const int i = item(k, n);
        status[i] = dec_parse_picture(jobs[i], streams[i], start[i], lens[i], tb);
    }
    // hevce_recon_kernel
    DecTuWork w;
    DecTu tus[64];
    for (int i = 0; i < n; i++) {
        const Job& job = jobs[i];
        const int rows = job.H / CTU, cols = job.W / CTU;
        if (status[i]) { memset(job.rcon, 0, (size_t)job.H * job.W); continue; }
        std::vector<int> seq;
        if (!order) for (int c = 0; c < rows * cols; c++) seq.push_back(c);
        else
            for (int t = 0; t <= cols - 1 + 2 * (rows - 1); t++)
                for (int r = rows - 1; r >= 0; r--)
                    if (t - 2 * r >= 0 && t - 2 * r < cols) seq.push_back(r * cols + t - 2 * r);
        for (int ctu : seq) {
            const int y0 = (ctu / cols) * CTU, x0 = (ctu % cols) * CTU, nt = dec_tu_list(job.recs[ctu], tus);
            const s16* lev = job.levs + (size_t)ctu * (CTU * CTU);
            for (int t = 0; t < nt; t++) {
                const DecTu u = tus[t];
                const int T = u.s, ty = y0 + u.y, tx = x0 + u.x;
                memset(&w, 0x5A, sizeof(w));                   // shared memory starts with whatever was there
                for (int j = 0; j < dec_ref_items(T); j++) dec_ref_item(w, job, ty, tx, T, item(j, dec_ref_items(T)));
                dec_ref_substitute(w, T);
                for (int j = 0; j < dec_ref_items(T); j++) dec_filter_item(w, T, item(j, dec_ref_items(T)));
                for (int x = 0; x < T; x++) dec_column(w, lev + u.y * CTU + u.x, T, job.q, item(x, T));
                for (int y = 0; y < T; y++) dec_row(w, job, ty, tx, T, u.m, item(y, T));
            }
        }
    }
    // hevce_deblock_kernel
    DbkTile t;
    for (int i = 0; i < n; i++) {
        const Job& job = jobs[i];
        if (decs)
            for (int ctu = 0; ctu < dbk_nctu(job); ctu++) {
                memset(&t, 0x5A, sizeof(t));
                for (int k = 0; k < DBK_LOAD_ITEMS; k++) dbk_load(t, job, ctu, item(k, DBK_LOAD_ITEMS));
                if (dbk_active(job)) {
                    for (int k = 0; k < DBK_VERT_ITEMS; k++) dbk_vertical(t, job, ctu, item(k, DBK_VERT_ITEMS));
                    for (int k = 0; k < DBK_HORZ_ITEMS; k++) dbk_horizontal(t, job, ctu, item(k, DBK_HORZ_ITEMS));
                }
                for (int k = 0; k < DBK_STORE_ITEMS; k++) dbk_store(t, job, ctu, decs[i], item(k, DBK_STORE_ITEMS));
            }
        unpack_partition(job.recs, job.H, job.W, cu_sizes ? cu_sizes[i] : nullptr, modes ? modes[i] : nullptr, kinds ? kinds[i] : nullptr);
    }
    return 0;
}

#if defined(HEVCE_SIMDECODE_MAIN)
// usage: hevce_simdecode STREAM FLIPS SEED
// Decodes every truncation of STREAM and FLIPS copies with one bit of the slice data flipped, each from an exactly sized
// heap buffer.  Prints "truncations T flips F ok K rejected R failed E"; exits 1 on a status other than 0 / 1.
static int decode_once(const std::vector<u8>& s, int& rejected) {
    u8* buf = (u8*)malloc(s.size() ? s.size() : 1);
    if (!s.empty()) memcpy(buf, s.data(), s.size());
    int H, W, q, st = -1;
    if (hevce_simdecode_info(buf, (int)s.size(), &H, &W, &q) < 0) { rejected++; free(buf); return 0; }
    std::vector<u8> rcon((size_t)H * W), dec((size_t)H * W);
    u8* r = rcon.data();
    u8* d = dec.data();
    const u8* p = buf;
    const int len = (int)s.size();
    if (hevce_simdecode(1, &p, &len, &r, &d, nullptr, nullptr, nullptr, &st, 0)) rejected++;
    free(buf);
    return st;
}

int main(int argc, char** argv) {
    if (argc != 4) { fprintf(stderr, "usage: %s STREAM FLIPS SEED\n", argv[0]); return 2; }
    FILE* f = fopen(argv[1], "rb");
    if (!f) return 2;
    std::vector<u8> s;
    for (int c; (c = fgetc(f)) != EOF;) s.push_back((u8)c);
    fclose(f);
    const int flips = atoi(argv[2]);
    unsigned long long rng = 0x9E3779B97F4A7C15ull ^ (unsigned long long)atoll(argv[3]);
    int H, W, q;
    const int hdr = hevce_simdecode_info(s.data(), (int)s.size(), &H, &W, &q);
    if (hdr < 0) return 2;
    int ok = 0, rejected = 0, failed = 0, bad = 0;
    auto tally = [&](int st) { if (st == 0) ok++; else if (st == 1) failed++; else bad++; };
    for (size_t L = 0; L <= s.size(); L++) {
        std::vector<u8> t(s.begin(), s.begin() + L);
        const int before = rejected;
        const int st = decode_once(t, rejected);
        if (rejected == before) tally(st);
    }
    const int data_bits = 8 * ((int)s.size() - hdr);
    for (int k = 0; k < flips && data_bits > 0; k++) {
        rng = rng * 6364136223846793005ull + 1442695040888963407ull;
        const int b = (int)((rng >> 33) % (unsigned long long)data_bits);
        std::vector<u8> t = s;
        t[hdr + b / 8] ^= (u8)(0x80 >> (b % 8));
        const int before = rejected;
        const int st = decode_once(t, rejected);
        if (rejected == before) tally(st);
    }
    printf("truncations %zu flips %d ok %d rejected %d failed %d bad %d\n", s.size() + 1, flips, ok, rejected, failed, bad);
    return bad ? 1 : 0;
}
#endif
