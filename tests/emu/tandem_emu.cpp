// tandem_emu.cpp -- TEST INFRASTRUCTURE: runs the tandem-mask kernel source (mimeo_b200/csrc/tandem_warp.cuh) on the CPU
// through the warp emulator of ydrop_emu.h, one span per call. Built by tests/test_tandem_emu.py with g++ -DYW_EMU.
#include <stdio.h>
#include <stdlib.h>
#include <vector>

#define YW_EMU 1
#include "ydrop_emu.h"
namespace yw { EmuWarp* g_warp = nullptr; }
#include "../../mimeo_b200/csrc/tandem_warp.cuh"

namespace {
struct Job {
    const uint8_t* sc; int n; tw::Params p; int K; int wide; void* store; int* ring; tw::Out o;
};
Job* g_job;
template <int K>
void run_k(Job& j) {
    if (j.wide) tw::tandem_warp<K, uint16_t>(j.sc, j.n, j.p, (uint16_t*)j.store, j.ring, j.o);
    else tw::tandem_warp<K, uint8_t>(j.sc, j.n, j.p, (uint8_t*)j.store, j.ring, j.o);
}
void lane_main() {
    Job& j = *g_job;
    if (j.K == 2) run_k<2>(j);
    else if (j.K == 4) run_k<4>(j);
    else run_k<8>(j);
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
// sc: the span in the device `codes` alphabet (n bytes); K: diagonals per lane (2, 4, 8); wide: 16-bit storage.
// Returns m; the merged runs go to iv_start / iv_end (at most cap), *niv receives their number.
long emu_tandem(const uint8_t* sc, int n, int M, int X, int G, int T, int P, int K, int wide, int64_t* iv_start, int64_t* iv_end,
                unsigned cap, unsigned* niv) {
    const size_t rows = n >= 2 ? (size_t)(2 * n - 3) : 0;
    const size_t elems = rows * 16 * K;
    std::vector<uint8_t> store(elems * (wide ? 2 : 1));
    std::vector<int> ring(tw::RING, -1);
    uint64_t m = 0;
    Job j;
    j.sc = sc; j.n = n; j.p = tw::Params{M, X, G, T, P}; j.K = K; j.wide = wide; j.store = store.data(); j.ring = ring.data();
    j.o = tw::Out{&m, iv_start, iv_end, cap, niv};
    g_job = &j;
    run_warp();
    return (long)m;
}
}
