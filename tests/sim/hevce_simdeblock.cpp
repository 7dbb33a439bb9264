// hevce_simdeblock.cpp -- host build of the deblocking kernel's source (TEST INFRASTRUCTURE ONLY).
//
// Runs the functions of csrc/hevce_deblock.h over whole pictures in one thread, exactly as hevce_deblock_kernel
// schedules them: every CTA of the grid (CTU, picture), and in each CTA every work item of a phase before the next
// phase (load, vertical edges, horizontal edges, store).  The partition reaches the filter the way it does on the
// device: the raster maps of hevce_session_partition are packed back into CtuRec arrays (the inverse of
// unpack_partition), and every other byte of a record is filled with 0xA5, so reading anything but msz / kind shows up.
// With order = 1 the work items of every phase run last to first: the same output shows a phase's items are independent.
#include <cstring>
#include <vector>

#include "hevce_core.h"
#include "hevce_deblock.h"

using namespace hevce;

static void pack_partition(CtuRec* recs, int H, int W, const u8* cu_size, const u8* kind) {
    const int cw = W / CTU, w4 = W / 4, w8 = W / 8;
    for (int c = 0; c < (H / CTU) * cw; c++) {
        CtuRec& r = recs[c];
        memset(&r, 0xA5, sizeof(CtuRec));
        const int y4 = (c / cw) * 8, x4 = (c % cw) * 8;
        for (int i = 0; i < 64; i++) r.msz[(1 + i / 8) * 9 + 1 + i % 8] = cu_size[(size_t)(y4 + i / 8) * w4 + x4 + i % 8];
        for (int i = 0; i < 16; i++) r.kind[i] = kind[(size_t)(y4 / 2 + i / 4) * w8 + x4 / 2 + i % 4];
    }
}

// n pictures of padded size H[i] x W[i]: rcons[i] (H x W), cu_sizes[i] ((H/4) x (W/4)), kinds[i] ((H/8) x (W/8)),
// qpd6[i]; decs[i] receives the decoded picture (H x W).  Returns 0, or -1 for a size that is not a multiple of 32.
extern "C" int hevce_simdeblock(int n, const u8* const* rcons, const u8* const* cu_sizes, const u8* const* kinds, const int* H, const int* W,
                                const int* qpd6, u8* const* decs, int order) {
    std::vector<std::vector<CtuRec>> recs((size_t)n);
    std::vector<Job> jobs((size_t)n);
    int max_nctu = 0;
    for (int i = 0; i < n; i++) {
        if (H[i] <= 0 || W[i] <= 0 || H[i] % CTU || W[i] % CTU) return -1;
        Job& j = jobs[i];
        memset(&j, 0, sizeof(Job));
        j.H = H[i]; j.W = W[i]; j.q = qpd6[i];
        j.rcon = (u8*)rcons[i];            // read only
        recs[i].resize((size_t)dbk_nctu(j));
        pack_partition(recs[i].data(), H[i], W[i], cu_sizes[i], kinds[i]);
        j.recs = recs[i].data();
        max_nctu = imax(max_nctu, dbk_nctu(j));
    }
    auto item = [&](int i, int count) { return order ? count - 1 - i : i; };
    DbkTile t;
    for (int pic = 0; pic < n; pic++)                        // blockIdx.y
        for (int ctu = 0; ctu < max_nctu; ctu++) {           // blockIdx.x
            const Job& job = jobs[pic];
            if (ctu >= dbk_nctu(job)) continue;
            memset(&t, 0x5A, sizeof(t));                     // shared memory starts with whatever was there
            for (int i = 0; i < DBK_LOAD_ITEMS; i++) dbk_load(t, job, ctu, item(i, DBK_LOAD_ITEMS));
            if (dbk_active(job)) {
                for (int i = 0; i < DBK_VERT_ITEMS; i++) dbk_vertical(t, job, ctu, item(i, DBK_VERT_ITEMS));
                for (int i = 0; i < DBK_HORZ_ITEMS; i++) dbk_horizontal(t, job, ctu, item(i, DBK_HORZ_ITEMS));
            }
            for (int i = 0; i < DBK_STORE_ITEMS; i++) dbk_store(t, job, ctu, decs[pic], item(i, DBK_STORE_ITEMS));
        }
    return 0;
}
