// hevce_simtrack.cpp -- TEST INFRASTRUCTURE ONLY: the kernel source (csrc/hevce_core.h) of a parent || child variant
// compiled for the host with ONE HOST THREAD PER TRACK of one picture: track 0 walks the 8x8 nodes and takes every
// decision, tracks 1 / 2 evaluate the 16x16 / 32x32 nodes' own candidates at the same time; the rendezvous between the
// tracks and the picture-wide barriers are real.  Bit-exactness against the oracle shows that what a parent track reads
// while its children are being decided (reference samples outside the CU, neighbour maps, the entry snapshot) is stable;
// under ThreadSanitizer the run shows that the tracks share no unsynchronised data.
#define HEVCE_SIM_TRACKS 1
#include <pthread.h>

#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>

#include "hevce_core.h"

namespace HEVCE_NS {
int g_sim_order = 0, g_sim_nlive = 1;
Shared* g_sim_sms = nullptr;
Tables* g_sim_tb = nullptr;
CommitShared* g_sim_csm = nullptr;
thread_local int g_sim_member = 0, g_sim_trk = 0, g_sim_my_track = 0;
static pthread_barrier_t g_bar[16];
void sim_barrier(int id, int) { pthread_barrier_wait(&g_bar[id]); }
}   // namespace HEVCE_NS

extern "C" int hevce_simtrack_encode(unsigned char* out, int out_cap, const unsigned char* img, unsigned char* rcon,
                                     int* ysz, int* xsz, int q, int order, int* err) {
    using namespace HEVCE_NS;
    static_assert(TRACKS, "compile with a parent || child variant (VDEF_t1 / VDEF_c2 in csrc/Makefile)");
    g_sim_order = order;
    static Tables tables;
    fill_tables(tables);
    Job job;
    int result[2] = {0, 0};
    job.img = img; job.rcon = rcon; job.out = out; job.result = result;
    job.src_h = *ysz; job.src_w = *xsz;
    job.H = (imin(*ysz, 8192) + CTU - 1) / CTU * CTU;
    job.W = (imin(*xsz, 8192) + CTU - 1) / CTU * CTU;
    job.q = q; job.out_cap = out_cap;
    const int nctu = (job.H / CTU) * (job.W / CTU);
    std::vector<s16> lev((size_t)nctu * CTU * CTU);
    std::vector<CtuRec> recs(nctu);
    job.recs = recs.data(); job.levs = lev.data();
    std::vector<std::vector<s16>> glev(NTRACK);
    std::vector<std::vector<u8>> grec(NTRACK), line(NTRACK);
    Scratch sc[NTRACK];
    for (int t = 0; t < NTRACK; t++) {
        glev[t].resize((size_t)NCAND * LEV_STRIDE + 16); grec[t].resize((size_t)NREC * CTU * CTU); line[t].resize(job.W / 4 + 8);
        sc[t].glev = glev[t].data(); sc[t].grec = grec[t].data(); sc[t].msz_line = line[t].data();
    }
    Shared* sm = new Shared[NTRACK];
    memset(sm, 0xA5, sizeof(Shared) * NTRACK);
    g_sim_sms = sm;
    g_sim_tb = &tables;
    pthread_barrier_init(&g_bar[BAR_PICTURES], nullptr, NTRACK);
    pthread_barrier_init(&g_bar[BAR_RDV1], nullptr, 2);
    pthread_barrier_init(&g_bar[BAR_RDV2], nullptr, 2);
    std::vector<std::thread> th;
    for (int t = 0; t < NTRACK; t++)
        th.emplace_back([&, t] {
            g_sim_my_track = t;
            g_sim_trk = 0;
            g_sim_member = 0;
            encode_picture(job, sc);
        });
    for (auto& x : th) x.join();
    pthread_barrier_destroy(&g_bar[BAR_PICTURES]);
    pthread_barrier_destroy(&g_bar[BAR_RDV1]);
    pthread_barrier_destroy(&g_bar[BAR_RDV2]);
    delete[] sm;
    CommitShared* cs = new CommitShared;
    memset(cs, 0x5A, sizeof(CommitShared));
    cs->tb = tables;
    g_sim_csm = cs;
    for (int c = 0; c < nctu; c++) commit_ctu(job, c, (c * 3) % NTC);
    delete cs;
    *ysz = job.H; *xsz = job.W;
    if (err) *err = result[1];
    return result[0];
}
