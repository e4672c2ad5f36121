// tandem_report_warp.cuh -- the tandem-repeat report of `--reportTRF` (DESIGN §2, R1-R6) for ONE masked run by ONE WARP.
//
// Statement (tests/tandem_report_oracle.c computes it literally), for a run u[0..L), L >= 2, D = min(P, L - 1):
//   R1 c[d] = #{x < L - d : u[x] in ACGT, u[x] == u[x+d]} for d = 1..D
//   R2 period p = the smallest d with 10 c[d] >= 9 max c (p = 1 when every c[d] is 0)
//   R3 n_k[b] = #{x = k mod p : u[x] == b}; consensus[k] = argmax_b n_k[b] (ties to the earliest of A, C, G, T; N if none)
//   R4 matches = sum_k max_b n_k[b]   R5 count[b] = sum_k n_k[b]   R6 score = M c[p] - X (L - p - c[p])
//
// R1: lane l owns the shifts d = l + 1 + 32 t, t < NT. The run is staged tile by tile in shared memory as three bit planes
// per 32 bases (base bit 0, base bit 1, A/C/G/T), built with three ballots per word; positions >= L are "other". Word w of
// the run shifted by d is the funnel shift of words w + t and w + t + 1 by l + 1 (clamped: lane 31 takes word w + t + 1
// whole), so every lane reads the same words and a word step is one popc per shift.
// R3: x is cut into S streams x = s mod S, S = p for p >= 32 and the largest multiple of p <= 32 below that. Lane l walks
// the streams l, l + 32, ... with four register counters and adds them to the shared n_k[b] of phase s mod p, so no lane
// walks more than about L / 16 positions. R4, R5: one lane per phase, then warp sums.
//
// The same source is compiled by g++ with YW_EMU defined (tests/emu/tandem_report_emu.cpp, which also supplies yw::popc and
// yw::redadd) against the warp emulator of tests/emu/ydrop_emu.h, so the kernel logic is checked against the oracle on the
// CPU as well.
#pragma once
#include <stdint.h>

#ifdef YW_EMU
#include "ydrop_emu.h"
#define TR_DEV inline
namespace tr {
using yw::atomic_add; using yw::ballot; using yw::funnel_rc; using yw::lane_id; using yw::ld8; using yw::popc; using yw::redadd;
using yw::redmax; using yw::redmin; using yw::shfl; using yw::syncwarp;
}
#else
#include <cuda_runtime.h>
#define TR_DEV __device__ __forceinline__
namespace tr {
TR_DEV int lane_id() { return (int)(threadIdx.x & 31); }
TR_DEV uint32_t shfl(uint32_t v, int src) { return __shfl_sync(0xffffffffu, v, src); }
TR_DEV uint32_t ballot(bool p) { return __ballot_sync(0xffffffffu, p); }
TR_DEV int redmax(int v) { return __reduce_max_sync(0xffffffffu, v); }
TR_DEV int redmin(int v) { return __reduce_min_sync(0xffffffffu, v); }
TR_DEV uint32_t redadd(uint32_t v) { return __reduce_add_sync(0xffffffffu, v); }
TR_DEV void syncwarp() { __syncwarp(); }
TR_DEV uint32_t ld8(const uint8_t* p) { return (uint32_t)__ldg(p); }
TR_DEV uint32_t popc(uint32_t v) { return (uint32_t)__popc(v); }
TR_DEV uint32_t funnel_rc(uint32_t lo, uint32_t hi, uint32_t sh) { return __funnelshift_rc(lo, hi, sh); }
TR_DEV uint32_t atomic_add(uint32_t* p, uint32_t v) { return atomicAdd(p, v); }
}  // namespace tr
#endif

namespace tr {

constexpr int MAX_P = 256;
constexpr int TILE = 64;                // words of 32 bases per staged tile
constexpr uint32_t CODE_OTHER = 8;      // `codes` mirror: base | parity << 2 (A,C,G,T = 0,5,6,3); >= 8 is N / IUPAC / pad

struct Params {
    int M, X, P;
};

struct alignas(16) Word {
    uint32_t lo, hi, v, pad;            // base bit 0, base bit 1, A/C/G/T of 32 consecutive positions
};

// Shared memory of one warp.
struct Scratch {
    Word w[TILE + MAX_P / 32];          // a tile and the words shifts of up to MAX_P read beyond it
    uint32_t n[MAX_P][4];               // n_k[b], b = A, C, G, T
};

// Outputs of all runs; run k writes element k (count: 4k .. 4k + 3, A, C, G, T) and its consensus at cons + cons_off[k]
// (period bytes; room for D).
struct Out {
    int32_t* period;
    int64_t* score;
    uint64_t* matches;
    uint64_t* count;
    const uint64_t* cons_off;
    char* cons;
};

// The report of run k, u[0..L) = sc[0..L), L >= 2. NT: shifts per lane, 32 * NT >= P.
template <int NT>
TR_DEV void report_warp(const uint8_t* sc, int L, const Params& p, Scratch& sh, const Out& o, uint32_t k) {
    const int lane = lane_id();
    const int D = p.P < L - 1 ? p.P : L - 1;
    // ---- R1
    uint32_t c[NT];
#pragma unroll
    for (int t = 0; t < NT; t++) c[t] = 0;
    const int nw = (L + 31) >> 5;
    for (int w0 = 0; w0 < nw; w0 += TILE) {
        const int tw = nw - w0 < TILE ? nw - w0 : TILE;
        syncwarp();                                     // the previous tile is consumed
        for (int j = 0; j < tw + NT; j++) {
            const int64_t x = ((int64_t)(w0 + j) << 5) + lane;
            const uint32_t cd = x < L ? ld8(sc + x) : CODE_OTHER;
            const uint32_t lo = ballot(cd & 1u), hi = ballot(cd & 2u), v = ballot(cd < CODE_OTHER);
            if (lane == (j & 31)) sh.w[j] = Word{lo, hi, v, 0u};
        }
        syncwarp();
        const uint32_t s = (uint32_t)lane + 1u;
        for (int j = 0; j < tw; j++) {
            const Word a = sh.w[j];
            Word prev = a;
#pragma unroll
            for (int t = 0; t < NT; t++) {
                const Word nx = sh.w[j + t + 1];
                const uint32_t lo = funnel_rc(prev.lo, nx.lo, s), hi = funnel_rc(prev.hi, nx.hi, s), v = funnel_rc(prev.v, nx.v, s);
                c[t] += popc(~((a.lo ^ lo) | (a.hi ^ hi)) & a.v & v);
                prev = nx;
            }
        }
    }
    // ---- R2
    int cmax = 0;
#pragma unroll
    for (int t = 0; t < NT; t++)
        if (lane + 1 + 32 * t <= D && (int)c[t] > cmax) cmax = (int)c[t];
    cmax = redmax(cmax);
    int dmin = MAX_P + 1;
#pragma unroll
    for (int t = NT - 1; t >= 0; t--) {
        const int d = lane + 1 + 32 * t;
        if (d <= D && 10 * (int64_t)c[t] >= 9 * (int64_t)cmax) dmin = d;
    }
    const int per = redmin(dmin);
    uint32_t cp = 0;
#pragma unroll
    for (int t = 0; t < NT; t++)
        if (t == (per - 1) >> 5) cp = c[t];
    cp = shfl(cp, (per - 1) & 31);
    // ---- R3
    syncwarp();                                         // the previous run's n_k[b] are read
    for (int i = lane; i < 4 * per; i += 32) sh.n[i >> 2][i & 3] = 0;
    syncwarp();
    const int S = per >= 32 ? per : per * (32 / per);
    for (int st = lane; st < S; st += 32) {
        uint32_t na = 0, nc = 0, ng = 0, ntt = 0;
        for (int64_t x = st; x < L; x += S) {
            const uint32_t cd = ld8(sc + x);
            na += cd == 0u; nc += cd == 5u; ng += cd == 6u; ntt += cd == 3u;
        }
        uint32_t* n = sh.n[st % per];
        if (na) atomic_add(n + 0, na);
        if (nc) atomic_add(n + 1, nc);
        if (ng) atomic_add(n + 2, ng);
        if (ntt) atomic_add(n + 3, ntt);
    }
    syncwarp();
    // ---- consensus, R4, R5
    uint32_t mt = 0, cnt[4] = {0u, 0u, 0u, 0u};
    char* cons = o.cons + o.cons_off[k];
    for (int ph = lane; ph < per; ph += 32) {
        uint32_t best = 0;
        int bb = 4;
#pragma unroll
        for (int b = 0; b < 4; b++) {
            const uint32_t v = sh.n[ph][b];
            cnt[b] += v;
            if (v > best) { best = v; bb = b; }
        }
        mt += best;
        cons[ph] = (char)(0x4E54474341ull >> (8 * bb));                 // bytes A, C, G, T, N
    }
    mt = redadd(mt);
#pragma unroll
    for (int b = 0; b < 4; b++) cnt[b] = redadd(cnt[b]);
    if (lane == 0) {
        o.period[k] = per;
        o.score[k] = (int64_t)p.M * cp - (int64_t)p.X * ((int64_t)L - per - cp);
        o.matches[k] = mt;
#pragma unroll
        for (int b = 0; b < 4; b++) o.count[4 * (size_t)k + b] = cnt[b];
    }
}

}  // namespace tr
