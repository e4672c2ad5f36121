// ydrop_emu.cpp -- TEST INFRASTRUCTURE: runs the y-drop extension kernel source (ydrop_warp.cuh) on the CPU through the
// warp emulator, one extension per call. Built by tests/test_ydrop_emu.py with g++ -DYW_EMU.
#include <stdio.h>
#include <stdlib.h>
#include <vector>

#define YW_EMU 1
#include "ydrop_emu.h"
namespace yw { EmuWarp* g_warp = nullptr; }
#include "../../mimeo_b200/csrc/ydrop_warp.cuh"

namespace {
struct Job {
    const uint8_t *tc, *qc; long ta, qa; int dir; yw::Params p; yw::Pool pool; yw::ExtResult* res; int max_s; int phase; uint32_t lay_mask; uint32_t priv_used = 0;
    yw::WalkCache wc;
    long tn = 0, qn = 0; yw::FullCell* rows = nullptr; long cap = 0;
};
Job* g_job;
void lane_main() {
    Job& j = *g_job;
    if (j.phase == 2) {
        yw::ydrop_full_warp(j.tc, j.qc, j.ta, j.qa, j.dir, j.tn, j.qn, j.p, j.rows, j.cap, j.res);
    } else if (j.phase == 0) {
        if (j.max_s >= 64) yw::ydrop_forward_warp<64>(j.tc, j.qc, j.ta, j.qa, j.dir, j.p, j.pool, 0u, 0u, j.priv_used, j.res, j.lay_mask);
        else yw::ydrop_forward_warp<32>(j.tc, j.qc, j.ta, j.qa, j.dir, j.p, j.pool, 0u, 0u, j.priv_used, j.res, j.lay_mask);
    } else {
        yw::ydrop_walk_warp(j.tc, j.qc, j.ta, j.qa, j.dir, j.p, j.pool, j.res, j.wc);
    }
    yw::EmuWarp* w = yw::g_warp;
    w->finished[w->cur] = true;
    // hand over to another live lane, or back to main when all are done
    for (int t = 1; t < 32; t++) {
        const int nx = (w->cur + t) & 31;
        if (!w->finished[nx]) { w->cur = nx; setcontext(&w->ctx[nx]); }
    }
    setcontext(&w->main_ctx);
}
void run_warp() {
    static yw::EmuWarp w;
    static std::vector<char> stacks;
    const size_t SS = 1 << 18;
    if (stacks.empty()) stacks.resize(32 * SS);
    w.arrived = 0; w.gen = 0; w.cur = 0;
    yw::g_warp = &w;
    for (int l = 0; l < 32; l++) {
        w.finished[l] = false;
        getcontext(&w.ctx[l]);
        w.ctx[l].uc_stack.ss_sp = stacks.data() + l * SS;
        w.ctx[l].uc_stack.ss_size = SS;
        w.ctx[l].uc_link = nullptr;
        makecontext(&w.ctx[l], lane_main, 0);
    }
    swapcontext(&w.main_ctx, &w.ctx[0]);
}
}  // namespace

extern "C" {
// out: score, di, dj, nmatch, ncols, status, cells, kbest, chunks_used, widest layout, layouts
int emu_extend(const uint8_t* tc, const uint8_t* qc, long ta, long qa, int dir, int O, int E, int Y, int max_s, int nchunks, unsigned lay_mask, int priv, int* out) {
    std::vector<uint8_t> base((size_t)nchunks * yw::CHUNK_BYTES);
    std::vector<yw::ChunkMeta> meta(nchunks);
    std::vector<uint32_t> next(yw::NSUB, 0);
    std::vector<int16_t> scratch(3 * yw::WIN);
    yw::ExtResult res;
    memset(&res, 0, sizeof(res));
    Job j;
    j.tc = tc; j.qc = qc; j.ta = ta; j.qa = qa; j.dir = dir; j.p = yw::Params{O, E, Y}; j.res = &res; j.max_s = max_s; j.lay_mask = lay_mask;
    j.pool.base = base.data(); j.pool.meta = meta.data(); j.pool.next = next.data();
    j.pool.priv = (uint32_t)priv; j.pool.shared0 = (uint32_t)priv; j.pool.per_sub = (uint32_t)((nchunks - priv) / yw::NSUB);
    j.pool.scratch = scratch.data();
    g_job = &j;
    j.phase = 0; run_warp();
    j.phase = 1; run_warp();
    uint32_t used = 0;
    for (uint32_t s = 0; s < (uint32_t)yw::NSUB; s++) used += next[s] < j.pool.per_sub ? next[s] : j.pool.per_sub;
    out[0] = res.score; out[1] = res.di; out[2] = res.dj; out[3] = res.nmatch; out[4] = res.ncols; out[5] = res.status;
    out[6] = (int)res.cells; out[7] = res.kbest; out[8] = (int)used + (int)j.pool.priv; out[9] = res.max_s; out[10] = res.nlayouts;
    return 0;
}

// The full-row fallback (ydrop_full_warp) of one extension: tn / qn = bases available from the anchor in direction dir.
// out: score, di, dj, nmatch, ncols, status, cells
int emu_full(const uint8_t* tc, const uint8_t* qc, long ta, long qa, int dir, long tn, long qn, int O, int E, int Y, long cap, int* out) {
    std::vector<yw::FullCell> rows((size_t)3 * cap);
    yw::ExtResult res;
    memset(&res, 0, sizeof(res));
    Job j;
    j.tc = tc; j.qc = qc; j.ta = ta; j.qa = qa; j.dir = dir; j.p = yw::Params{O, E, Y}; j.res = &res;
    j.tn = tn; j.qn = qn; j.rows = rows.data(); j.cap = cap;
    g_job = &j;
    j.phase = 2; run_warp();
    out[0] = res.score; out[1] = res.di; out[2] = res.dj; out[3] = res.nmatch; out[4] = res.ncols; out[5] = res.status; out[6] = (int)res.cells;
    return 0;
}
}
