// tandem_report_emu.cpp -- TEST INFRASTRUCTURE: runs the tandem-report kernel source (mimeo_b200/csrc/tandem_report_warp.cuh)
// on the CPU through the warp emulator of ydrop_emu.h, one run per call. Built by tests/test_tandem_report.py with g++ -DYW_EMU.
#include <stdio.h>
#include <stdlib.h>
#include <vector>

#define YW_EMU 1
#include "ydrop_emu.h"
namespace yw {
EmuWarp* g_warp = nullptr;
// the two warp intrinsics of the report kernel that ydrop_emu.h does not restate
inline uint32_t popc(uint32_t v) { return (uint32_t)__builtin_popcount(v); }
inline uint32_t redadd(uint32_t v) { const uint32_t* a = emu_exchange(v); uint32_t s = 0; for (int l = 0; l < 32; l++) s += a[l]; return s; }
}  // namespace yw
#include "../../mimeo_b200/csrc/tandem_report_warp.cuh"

namespace {
struct Job {
    const uint8_t* sc; int L; tr::Params p; int NT; tr::Scratch* sh; tr::Out o;
};
Job* g_job;
void lane_main() {
    Job& j = *g_job;
    if (j.NT == 1) tr::report_warp<1>(j.sc, j.L, j.p, *j.sh, j.o, 0);
    else if (j.NT == 2) tr::report_warp<2>(j.sc, j.L, j.p, *j.sh, j.o, 0);
    else if (j.NT == 4) tr::report_warp<4>(j.sc, j.L, j.p, *j.sh, j.o, 0);
    else tr::report_warp<8>(j.sc, j.L, j.p, *j.sh, j.o, 0);
    yw::EmuWarp* w = yw::g_warp;
    w->finished[w->cur] = true;
    for (int t = 1; t < 32; t++) {
        const int nx = (w->cur + t) & 31;
        if (!w->finished[nx]) { w->cur = nx; setcontext(&w->ctx[nx]); }
    }
    setcontext(&w->main_ctx);
}
void run_warp() {
    static yw::EmuWarp w;
    static std::vector<char> stacks;
    const size_t SS = 1 << 17;
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
// sc: the run in the device `codes` alphabet (L >= 2 bytes); NT: shifts per lane (1, 2, 4, 8; 32 * NT >= P).
// out[0..6] = period, score, matches, count A, C, G, T; cons receives period bytes (room for min(P, L - 1)).
void emu_tandem_report(const uint8_t* sc, int L, int M, int X, int P, int NT, int64_t* out, char* cons) {
    // the scratch is left dirty on purpose: the kernel must clear what it reads
    static tr::Scratch sh;
    memset(&sh, 0xa5, sizeof(sh));
    int32_t period = 0;
    int64_t score = 0;
    uint64_t matches = 0, count[4] = {0, 0, 0, 0}, cons_off = 0;
    Job j;
    j.sc = sc; j.L = L; j.p = tr::Params{M, X, P}; j.NT = NT; j.sh = &sh;
    j.o = tr::Out{&period, &score, &matches, count, &cons_off, cons};
    g_job = &j;
    run_warp();
    out[0] = period; out[1] = score; out[2] = (int64_t)matches;
    for (int b = 0; b < 4; b++) out[3 + b] = (int64_t)count[b];
}
}
