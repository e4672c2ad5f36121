// tandem_warp.cuh -- the tandem-repeat mask of `mimeo map --maxtandem` (DESIGN §2, T1-T4) for ONE span by ONE WARP.
//
// Statement (oracle/tandem_oracle.c computes it literally): local self-alignment of the span s[0..n) inside the strip of
// diagonals d = j - i in [1, P] of the prefix matrix, match +M (A/C/G/T only, case ignored), mismatch / N -X, indel -G,
// no affine part. H = forward (prefix) matrix, H' = backward (suffix) matrix. A pair (p, q), 1 <= q - p <= P, qualifies
// iff H[p][q] + sub(s[p], s[q]) + H'[p+1][q+1] >= T, and masks positions p..q.
//
// Layout: lane l owns the K consecutive diagonals d = K*l + 1 .. K*l + K (K even, so slot s holds odd d iff s is even).
// Both passes walk anti-diagonals a = i + j: cell (i, d) lives on a = 2i + d, its diagonal neighbour (same d) is on a -+ 2
// and its two gap neighbours (d - 1, d + 1) are on a -+ 1. A step updates the slots of one parity in place from the
// other parity, with one SHFL at the lane edge; no scan inside a row, no shared memory in the recurrence.
//   * backward pass first, a = 2n-1 .. 3: stores min(H', T + X) of every cell of rows a = 3 .. 2n-1 (0 where H' is the
//     boundary), one ST per cell, row-major by anti-diagonal so that every step is one coalesced store. The clamp is exact:
//     the other side of the sum is H + sub >= -X, so any H' >= T + X qualifies either way.
//   * forward pass, a = 3 .. 2n-1: the diagonal term dg = H[i-1][j-1] + sub(s[i-1], s[j-1]) of cell (i, j) is exactly
//     the first two terms of best(i-1, j-1), so the pair (i-1, j-1) is tested against the stored H'[i][j] in the same step.
// Scores are int32 (exact: the host refuses M*(n+1) + T + X >= 2^31).
//
// Counting: a qualifying pair (p, q) is recorded as ring[p % RING] = max(., q) in a per-warp ring (distinct cells of one
// step have distinct p, so no two lanes collide). Pair p is complete once a >= 2p + 2 + P; lane 0 then merges the
// complete entries in order of p into maximal runs of masked positions, counts them and optionally writes them out.
//
// The same source is compiled by g++ with YW_EMU defined (tests/emu/tandem_emu.cpp) against the warp emulator of
// tests/emu/ydrop_emu.h, so the kernel logic is checked against the oracle on the CPU as well.
#pragma once
#include <stdint.h>

#ifdef YW_EMU
#include "ydrop_emu.h"
#define TW_DEV inline
namespace tw {
using yw::ballot; using yw::lane_id; using yw::ld8; using yw::redmax; using yw::shfl_down; using yw::shfl_up; using yw::syncwarp;
}
#else
#include <cuda_runtime.h>
#define TW_DEV __device__ __forceinline__
namespace tw {
TW_DEV int lane_id() { return (int)(threadIdx.x & 31); }
TW_DEV uint32_t shfl_up(uint32_t v, int d) { return __shfl_up_sync(0xffffffffu, v, d); }
TW_DEV uint32_t shfl_down(uint32_t v, int d) { return __shfl_down_sync(0xffffffffu, v, d); }
TW_DEV uint32_t ballot(bool p) { return __ballot_sync(0xffffffffu, p); }
TW_DEV int redmax(int v) { return __reduce_max_sync(0xffffffffu, v); }
TW_DEV void syncwarp() { __syncwarp(); }
TW_DEV uint32_t ld8(const uint8_t* p) { return (uint32_t)__ldg(p); }
}  // namespace tw
#endif

namespace tw {

constexpr int RING = 256;           // open pairs of a warp: at most P/2 + 4 values of p, P <= MAX_P
constexpr int MAX_P = 256;
constexpr uint32_t CODE_OTHER = 8;  // `codes` mirror: A,C,G,T = 0,5,6,3; >= 8 is N / IUPAC / pad

struct Params {
    int M, X, G, T, P;
};

struct Out {
    uint64_t* masked;               // m of the span
    int64_t* iv_start;              // merged masked runs (closed, span-local), may be null
    int64_t* iv_end;
    uint32_t iv_cap;
    uint32_t* iv_n;                 // number of runs (may exceed iv_cap; only iv_cap are written)
};

// Lane 0's merge state.
struct Merge {
    int64_t cs = 0, ce = -2, m = 0;
    uint32_t niv = 0;
    bool open = false;
    TW_DEV void add(int64_t p, int64_t q, const Out& o) {
        if (open && p <= ce + 1) { ce = q > ce ? q : ce; return; }
        close(o);
        cs = p; ce = q; open = true;
    }
    TW_DEV void close(const Out& o) {
        if (!open) return;
        m += ce - cs + 1;
        if (o.iv_start && niv < o.iv_cap) { o.iv_start[niv] = cs; o.iv_end[niv] = ce; }
        niv++;
        open = false;
    }
};

// One anti-diagonal a of either pass. SP = parity of the slots updated (0: odd d, a odd; 1: even d, a even).
// FWD: cell (i, j) consumes s[i-1], s[j-1], reads the stored H'[i][j] and tests the pair (i-1, j-1).
// !FWD: cell (i, j) consumes s[i], s[j] and stores min(H'[i][j], T + X).
template <int K, int SP, bool FWD, typename ST>
TW_DEV void step(int (&h)[K], int a, int n, const uint8_t* sc, const Params& p, ST* row, int* ring, int& hi_p) {
    const int lane = lane_id();
    int edge;
    if (SP == 0) { edge = (int)shfl_up((uint32_t)h[K - 1], 1); if (lane == 0) edge = 0; }       // d - 1 of slot 0
    else { edge = (int)shfl_down((uint32_t)h[0], 1); if (lane == 31) edge = 0; }                // d + 1 of slot K-1
    int qp = -1;
#pragma unroll
    for (int t = 0; t < K / 2; t++) {
        const int s = 2 * t + SP;
        const int d = K * lane + 1 + s;
        const int lo = s == 0 ? edge : h[s > 0 ? s - 1 : 0];
        const int hi = s == K - 1 ? edge : h[s + 1 < K ? s + 1 : s];
        const int i = (a - d) >> 1, j = (a + d) >> 1;
        const bool valid = d <= p.P && (FWD ? (a - d >= 2 && a + d <= 2 * n) : (a - d >= 0 && a + d <= 2 * n - 2));
        uint32_t ci = CODE_OTHER, cj = CODE_OTHER;
        if (valid) { ci = ld8(sc + (FWD ? i - 1 : i)); cj = ld8(sc + (FWD ? j - 1 : j)); }
        const int dg = h[s] + ((ci == cj && ci < CODE_OTHER) ? p.M : -p.X);
        const int gp = (lo > hi ? lo : hi) - p.G;
        int v = dg > gp ? dg : gp;
        v = v > 0 ? v : 0;
        ST* cell = row + (K / 2) * lane + t;
        if (FWD) {
            if (valid && dg + (int)*cell >= p.T) {
                const int pp = i - 1, qq = j - 1;
                int* r = ring + (pp & (RING - 1));
                *r = *r > qq ? *r : qq;
                qp = pp > qp ? pp : qp;
            }
        } else {
            const int cap = p.T + p.X;
            *cell = (ST)(valid ? (v < cap ? v : cap) : 0);
        }
        if (valid) h[s] = v;
    }
    if (FWD && ballot(qp >= 0)) {   // rare outside repeats: the ring writes of this step are ordered before the next step's
        const int m = redmax(qp);
        hi_p = m > hi_p ? m : hi_p;
        syncwarp();
    }
}

// Lane 0 merges the ring entries of the complete pairs p <= limit (warp-uniform arguments).
TW_DEV void finalize(int* ring, int& p_done, int hi_p, int limit, Merge& mg, const Out& o) {
    if (limit <= p_done) return;
    if (hi_p > p_done) {
        syncwarp();
        if (lane_id() == 0) {
            const int top = limit < hi_p ? limit : hi_p;
            for (int pp = p_done + 1; pp <= top; pp++) {
                int* r = ring + (pp & (RING - 1));
                if (*r >= 0) { mg.add(pp, *r, o); *r = -1; }
            }
        }
        syncwarp();
    }
    p_done = limit;
}

// The mask of one span s[0..n) = sc[0..n). store: this span's (2n - 3) rows of 16 * K elements (n >= 2).
// ring: RING ints of this warp (shared memory on the device).
template <int K, typename ST>
TW_DEV void tandem_warp(const uint8_t* sc, int n, const Params& p, ST* store, int* ring, const Out& o) {
    static_assert(K % 2 == 0, "K must be even: slot parity must not depend on the lane");
    constexpr int RW = 16 * K;      // elements per stored anti-diagonal
    const int lane = lane_id();
    Merge mg;
    if (n >= 2) {
        const int L = 2 * n - 3;    // anti-diagonals 3 .. 2n-1
        int h[K];
        int hi_p = -1, p_done = -1;
        // ---- backward pass
#pragma unroll
        for (int s = 0; s < K; s++) h[s] = 0;
        for (int k = 0; k + 1 < L; k += 2) {
            const int a = 2 * n - 1 - k;
            step<K, 0, false, ST>(h, a, n, sc, p, store + (size_t)(a - 3) * RW, ring, hi_p);
            step<K, 1, false, ST>(h, a - 1, n, sc, p, store + (size_t)(a - 4) * RW, ring, hi_p);
        }
        step<K, 0, false, ST>(h, 3, n, sc, p, store, ring, hi_p);       // L is odd
        // ---- forward pass
        for (int x = lane; x < RING; x += 32) ring[x] = -1;
#pragma unroll
        for (int s = 0; s < K; s++) h[s] = 0;
        syncwarp();
        for (int k = 0; k + 1 < L; k += 2) {
            const int a = 3 + k;
            step<K, 0, true, ST>(h, a, n, sc, p, store + (size_t)(a - 3) * RW, ring, hi_p);
            step<K, 1, true, ST>(h, a + 1, n, sc, p, store + (size_t)(a - 2) * RW, ring, hi_p);
            const int done = a + 1 - 2 - p.P;                                // pairs with 2p + 2 + P <= a + 1 are complete
            finalize(ring, p_done, hi_p, done >= 0 ? done >> 1 : -1, mg, o);
        }
        step<K, 0, true, ST>(h, 2 * n - 1, n, sc, p, store + (size_t)(2 * n - 4) * RW, ring, hi_p);
        finalize(ring, p_done, hi_p, n, mg, o);
    }
    if (lane == 0) {
        mg.close(o);
        *o.masked = (uint64_t)mg.m;
        if (o.iv_n) *o.iv_n = mg.niv;
    }
}

}  // namespace tw
