// ydrop_warp.cuh -- kernel family (c), second generation: affine-gap y-drop extension by ONE WARP per (anchor, direction),
// two DP cells per 32-bit register (16-bit scores, DPX VIADDMNMX / VIMNMX3 .S16x2), no payload in the recurrence.
//
// Replaces LASTZ's --gapped extension (reference call sites wrappers.py:1025-1037 et al.) under spec D4 of
// oracle/lastz_oracle.c (ydrop_extend): anti-diagonal k is evaluated as a whole; a cell survives iff
// H >= best - ydrop, best = maximum over all EARLIER anti-diagonals; the end of the extension is the first cell in
// (anti-diagonal, row) order that attains the final best. Identity (matches / aligned columns) is recovered by a
// walk-back over the stored H values, with the oracle's tie-breaks (H: M > D > I; D and I: open beats extend).
//
// Forward pass (ydrop_forward_warp):
//   * diagonal-major, like the first generation: lane l owns S consecutive diagonals rbase + S*l .. + S-1 for a whole
//     "layout"; a step evaluates the cells of one parity, so every cell and all but one neighbour live in registers;
//     one SHFL per step moves the edge cell between neighbouring lanes, one warp REDUX.MAX gives the step maximum for
//     the y-drop threshold. No shared memory, no block barrier.
//   * scores are kept in a drifting frame  Ht(i,j) = H(i,j) + E*(i+j) - F : the gap-extension cost vanishes
//     (D = max(Hup - O, Dup): one VIADDMNMX), a substitution adds s + 2E, and the frame offset F is moved every few
//     hundred steps so that everything fits signed 16 bit. Dead cells hold exactly SENT in all three states.
//   * two cells per register: pair c of a parity = (slot 2c+p, slot 2c+p+S/2), so the up / left neighbours of a pair
//     are whole registers of the other parity (no permutes except at the lane edge).
//   * substitution scores come from a byte-permute: with codes  base | parity(base) << 2  the HOXD70 entry is a
//     function of (t ^ q, parity(t)), i.e. an 8-entry byte table = one PRMT for four cells.
//   * the stored H of every step (2 bytes per cell) is written to a chunked trace pool in HBM, coalesced.
// Walk-back (ydrop_walk_warp): one warp per extension; 31 diagonal steps are tested at once (each lane one cell);
// a gap is found by testing up to 320 gap lengths in parallel.
//
// The same source is compiled by g++ with YW_EMU defined (tests/emu/): a fibre-based 32-lane emulator stands in for
// the warp intrinsics, so the kernel logic is checked against the oracle on the CPU as well.
#pragma once
#include <stdint.h>

#ifdef YW_EMU
#include "ydrop_emu.h"
#define YW_DEV inline
#define YW_DEV_NOINLINE inline
#else
#include <cuda_runtime.h>
#define YW_DEV __device__ __forceinline__
#define YW_DEV_NOINLINE __device__ __noinline__
#endif

namespace yw {

// ------------------------------------------------------------------------------------------ constants
// 16-bit budget (signed): a dead state is exactly SENT; an alive H is never below threshold - |bias| and the threshold is
// kept in [SENT + 1600, SENT + 32268 - 1500], so that (a) anything computed from dead neighbours (<= SENT + 225) is below
// every threshold, (b) H - threshold never wraps, (c) alive values (<= threshold + Y + 900) stay below 32767 for Y <= 20000.
constexpr int SENT = -30000;                 // a dead state (all of H, D, I)
constexpr int ALIVE_MIN = SENT + 1000;       // stored values above this are alive
constexpr int INIT_THR = SENT + 1600;        // threshold image right after a frame move (best image = this + Y)
constexpr int REBASE_THR = SENT + 30100;     // move the frame when the threshold image exceeds this
constexpr int WIN = 4096;                    // diagonals of the re-layout scratch (circular), per state
constexpr int CHUNK_BYTES = 65536;           // trace pool chunk
constexpr int BLOCK_STEPS = 8;               // steps per unrolled block (one window load)
constexpr int NSUB = 32;                     // sub-pools of the chunk allocator

// code bytes of the `codes` genome mirror: base | parity(base) << 2 for A,C,G,T = 0,5,6,3; 8 = other (N); 12 = beyond the
// scaffold (pad): a cell that would consume a pad base does not exist
constexpr uint32_t CODE_N = 8, CODE_END = 12;

// ST_BAND: the alive band outgrew the widest layout (64 x 32 diagonals); the caller reruns the item with ydrop_full_warp
enum : int { ST_OK = 0, ST_NOMEM = 1, ST_WIDE = 2, ST_FAIL = 3, ST_BAND = 4 };

struct Params {
    int O, E, Y;          // gap open, gap extend, y-drop
};
// HOXD70 + 125 as bytes, index = (t ^ q) | parity(t) << 2 (see header); N against anything = -100 + 125
constexpr uint32_t TAB_LO = 0x025E0BD8u, TAB_HI = 0x005E0BE1u, U_N = 25u;

struct ChunkMeta {        // 32 bytes
    uint32_t prev;        // previous chunk of the same extension, 0xffffffff = none
    int32_t k0;           // step of row 0
    int32_t nrows;
    int32_t rbase;        // diagonal of lane 0, slot 0
    int32_t S;            // diagonals per lane
    int32_t F;            // frame: H + E*k = stored + bias + F
    int32_t pad0, pad1;
};

// Chunk ids [0, nslots * priv) are private: warp slot s owns [s * priv, (s + 1) * priv) and hands them out with a plain
// counter that runs over all the extensions the slot processes in one launch (no atomics). When the slice is used up the
// trace continues in the shared part: NSUB bump counters over per_sub chunks each. The host resets both between launches,
// after the walk-back kernel has consumed the traces.
struct Pool {
    uint8_t* base;        // nchunks * CHUNK_BYTES
    ChunkMeta* meta;      // nchunks
    uint32_t* next;       // NSUB counters of the shared part
    uint32_t per_sub;     // chunks per shared sub-pool
    uint32_t priv;        // private chunks per warp slot
    uint32_t shared0;     // first chunk id of the shared part
    int16_t* scratch;     // per warp slot: 3 * WIN int16 (re-layout scratch)
};

struct ExtResult {        // one per (anchor, direction)
    int32_t score;        // best H
    int32_t kbest;        // step of the first best
    int32_t bestv;        // stored value of the best in its row
    uint32_t chunk;       // last chunk written
    int32_t status;
    int32_t di, dj, nmatch, ncols;   // filled by the walk-back
    uint32_t cells;       // band cells evaluated (lanes between the first and last alive lane)
    int32_t max_s, nlayouts;         // widest layout used, number of layouts (diagnostics)
};

// ------------------------------------------------------------------------------------------ warp / SIMD primitives
#ifndef YW_EMU
YW_DEV int lane_id() { return (int)(threadIdx.x & 31); }
YW_DEV uint32_t shfl_up(uint32_t v, int d) { return __shfl_up_sync(0xffffffffu, v, d); }
YW_DEV uint32_t shfl_down(uint32_t v, int d) { return __shfl_down_sync(0xffffffffu, v, d); }
YW_DEV uint32_t shfl(uint32_t v, int src) { return __shfl_sync(0xffffffffu, v, src); }
YW_DEV uint32_t ballot(bool p) { return __ballot_sync(0xffffffffu, p); }
YW_DEV int redmax(int v) { return __reduce_max_sync(0xffffffffu, v); }
YW_DEV int redmin(int v) { return __reduce_min_sync(0xffffffffu, v); }
YW_DEV void syncwarp() { __syncwarp(); }
YW_DEV uint32_t atomic_add(uint32_t* p, uint32_t v) { return atomicAdd(p, v); }
YW_DEV uint32_t vadd2(uint32_t a, uint32_t b) { return __vadd2(a, b); }
YW_DEV uint32_t vmax2(uint32_t a, uint32_t b) { return __vmaxs2(a, b); }
YW_DEV uint32_t viaddmax2(uint32_t a, uint32_t b, uint32_t c) { return __viaddmax_s16x2(a, b, c); }
YW_DEV uint32_t vmax3_2(uint32_t a, uint32_t b, uint32_t c) { return __vimax3_s16x2(a, b, c); }
YW_DEV uint32_t prmt(uint32_t a, uint32_t b, uint32_t s) {
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(s));
    return r;
}
YW_DEV uint32_t funnel_r(uint32_t lo, uint32_t hi, uint32_t sh) { return __funnelshift_r(lo, hi, sh); }
YW_DEV uint32_t funnel_rc(uint32_t lo, uint32_t hi, uint32_t sh) { return __funnelshift_rc(lo, hi, sh); }   // shift clamped to 32
YW_DEV uint32_t ld32(const uint8_t* p) { return __ldg(reinterpret_cast<const uint32_t*>(p)); }
YW_DEV uint32_t ld8(const uint8_t* p) { return (uint32_t)__ldg(p); }
YW_DEV void fence() { __threadfence(); }
#endif

YW_DEV uint32_t pack2(int lo, int hi) { return ((uint32_t)lo & 0xffffu) | ((uint32_t)hi << 16); }
YW_DEV int lo16(uint32_t v) { return (int)(int16_t)(v & 0xffffu); }
YW_DEV int hi16(uint32_t v) { return (int)(int16_t)(v >> 16); }
// bytes at byte offset `off` (0..3 + 4*w) of a little-endian word array: word w', funnel by the remainder
template <int N>
YW_DEV uint32_t bytes_at(const uint32_t (&w)[N], int off) {
    const int i = off >> 2, s = (off & 3) * 8;
    return s == 0 ? w[i] : funnel_r(w[i], w[i + 1 < N ? i + 1 : i], (uint32_t)s);
}
template <int N>
YW_DEV uint32_t byte_of(const uint32_t (&w)[N], int n) { return (w[n >> 2] >> ((n & 3) * 8)) & 0xffu; }
// the same with a run-time part r (0..4 bytes) of the offset: word index and byte position stay compile-time constants
template <int N>
YW_DEV uint32_t bytes_at_rt(const uint32_t (&w)[N], int word, int r) { return funnel_rc(w[word], w[word + 1 < N ? word + 1 : word], (uint32_t)r * 8u); }
template <int N>
YW_DEV uint32_t byte_of_rt(const uint32_t (&w)[N], int n, int r) { return (bytes_at_rt(w, n >> 2, r) >> ((n & 3) * 8)) & 0xffu; }

// ------------------------------------------------------------------------------------------ layout
template <int S_> struct Lay {
    static constexpr int S = S_;
    static constexpr int CH = S / 4;                       // pairs per parity
    static constexpr int NG = (CH + 3) / 4;                // selector words per step
    static constexpr int NWC = NG + 1;                     // words of a combined stream (bytes 0 .. CH+3, one spare for funnels)
    static constexpr int NWR = (2 * CH + 4 + 3) / 4 + 1;   // words of a raw stream (bytes 0 .. 2CH+3, one spare)
    static constexpr int ROW_BYTES = 32 * CH * 4;
    static constexpr int ROWS_PER_CHUNK = CHUNK_BYTES / ROW_BYTES;
};

template <int S> struct State {
    uint32_t He[Lay<S>::CH], Ho[Lay<S>::CH], De[Lay<S>::CH], Do[Lay<S>::CH], Ie[Lay<S>::CH], Io[Lay<S>::CH];
};

// What one extension carries between layouts (warp-uniform unless noted).
struct Ctx {
    const uint8_t* tc; const uint8_t* qc;   // code arrays
    int64_t ta, qa;                         // anchor (padded coordinates)
    int dir;
    Params p;
    int bias;             // stored H = T-domain H - bias, bias = 125 - 2E
    int init_best, rebase_at;
    int k;                // last completed step
    int rbase, S;
    int bestT;            // T-domain image of the best at step k+1 (i.e. already advanced by E)
    int F;
    int best_real, kbest, bestv;
    int dead_steps;
    int lo_lane, hi_lane; // alive lanes after the last block
    int alo, ahi;         // exact alive diagonal range when a layout ends
    uint32_t lay_mask;    // allowed layouts: bit S/4
    uint32_t cells;
    int status;
    // trace
    Pool pool;
    uint32_t item, slot;
    uint32_t priv_used;   // private chunks handed out to this extension
    uint32_t chunk;       // current chunk id
    int k0, nrows, cap;
    int16_t* scr;         // this warp's scratch: H, D, I each WIN
};

// ------------------------------------------------------------------------------------------ trace pool
YW_DEV_NOINLINE uint32_t pool_alloc_shared(uint32_t* next, uint32_t per_sub, uint32_t shared0, uint32_t item) {
    uint32_t id = 0xffffffffu;
    if (lane_id() == 0) {
        for (uint32_t t = 0; t < NSUB; t++) {
            const uint32_t sub = (item + t) % NSUB;
            if (*(volatile uint32_t*)&next[sub] >= per_sub) continue;
            const uint32_t idx = atomic_add(&next[sub], 1u);
            if (idx < per_sub) { id = shared0 + sub * per_sub + idx; break; }
        }
    }
    return shfl(id, 0);
}
// close the current chunk (if any) and open a new one whose first row is step k_first
YW_DEV bool chunk_open(Ctx& c, int k_first, int rows_per_chunk) {
    const uint32_t prev = c.chunk;
    if (prev != 0xffffffffu && lane_id() == 0) c.pool.meta[prev].nrows = c.nrows;
    uint32_t id;
    if (c.priv_used < c.pool.priv) id = c.slot * c.pool.priv + c.priv_used++;
    else id = pool_alloc_shared(c.pool.next, c.pool.per_sub, c.pool.shared0, c.item);
    if (id == 0xffffffffu) { c.status = ST_NOMEM; return false; }
    if (lane_id() == 0) {
        ChunkMeta m;
        m.prev = prev; m.k0 = k_first; m.nrows = 0; m.rbase = c.rbase; m.S = c.S; m.F = c.F; m.pad0 = m.pad1 = 0;
        c.pool.meta[id] = m;
    }
    c.chunk = id; c.k0 = k_first; c.nrows = 0; c.cap = rows_per_chunk;
    return true;
}

// ------------------------------------------------------------------------------------------ window streams
// NW words of the byte stream R[n] = codes[a0 + n] (asc) or codes[a0 - n] (desc), n = 0 .. 4*NW-1
template <int NW>
YW_DEV void load_stream(const uint8_t* codes, int64_t a0, bool asc, uint32_t (&out)[NW]) {
    if (asc) {
        const int64_t ab = a0 & ~(int64_t)3;
        const uint32_t sh = (uint32_t)(a0 & 3) * 8;
        uint32_t w[NW + 1];
#pragma unroll
        for (int i = 0; i <= NW; i++) w[i] = ld32(codes + ab + 4 * i);
#pragma unroll
        for (int i = 0; i < NW; i++) out[i] = sh ? funnel_r(w[i], w[i + 1], sh) : w[i];
    } else {
        const int64_t b0 = a0 - (4 * NW - 1);           // lowest address; R[n] = A[4NW-1-n], A ascending from b0
        const int64_t ab = b0 & ~(int64_t)3;
        const uint32_t sh = (uint32_t)(b0 & 3) * 8;
        uint32_t w[NW + 1];
#pragma unroll
        for (int i = 0; i <= NW; i++) w[i] = ld32(codes + ab + 4 * i);
#pragma unroll
        for (int i = 0; i < NW; i++) {
            const uint32_t a = sh ? funnel_r(w[NW - 1 - i], w[NW - i], sh) : w[NW - 1 - i];
            out[i] = prmt(a, 0, 0x0123);                 // byte reverse
        }
    }
}

// ------------------------------------------------------------------------------------------ one step
// PAR = 1: odd step (odd slots), PAR = 0: even step. v = 0..3 = position inside the block: a RUN-TIME value (the block is
// a rolled loop: the kernel is instruction-cache bound when every step of every layout is unrolled), so it only ever
// enters as a funnel-shift amount.
// XC / YC: combined streams (normal blocks), XR / YR: raw streams (special blocks: N or pad bases in sight).
template <int S, bool SPECIAL, int PAR>
YW_DEV void step(State<S>& st, const uint32_t (&XC)[Lay<S>::NWC], const uint32_t (&YC)[Lay<S>::NWC],
                 const uint32_t (&XR)[Lay<S>::NWR], const uint32_t (&YR)[Lay<S>::NWR], int v,
                 uint32_t kopen2, uint32_t negbias2, uint32_t negthr2, uint32_t& hmax2) {
    constexpr int CH = Lay<S>::CH, NG = Lay<S>::NG;
    const uint32_t SENT2 = pack2(SENT, SENT);
    const int lane = lane_id();
    const int xo = v;                                   // T stream offset (both parities)
    const int yo = PAR ? 4 - v : 3 - v;                 // Q stream offset
    uint32_t sc[CH], kill[CH];
    if (!SPECIAL) {
#pragma unroll
        for (int g = 0; g < NG; g++) {
            const uint32_t sel = bytes_at_rt(XC, g, xo) ^ bytes_at_rt(YC, g, yo);
            const uint32_t r0 = prmt(TAB_LO, TAB_HI, sel & 0xffffu);
            if (4 * g + 0 < CH) sc[4 * g + 0] = prmt(r0, 0, 0x4140);
            if (4 * g + 1 < CH) sc[4 * g + 1] = prmt(r0, 0, 0x4342);
            if (4 * g + 2 < CH) {
                const uint32_t r1 = prmt(TAB_LO, TAB_HI, sel >> 16);
                sc[4 * g + 2] = prmt(r1, 0, 0x4140);
                if (4 * g + 3 < CH) sc[4 * g + 3] = prmt(r1, 0, 0x4342);
            }
        }
    } else {
#pragma unroll
        for (int c = 0; c < CH; c++) {
            uint32_t u[2], kl[2];
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const uint32_t t = byte_of_rt(XR, c + h * CH, xo), q = byte_of_rt(YR, c + h * CH, yo);
                const bool end = ((t & 12u) == 12u) || ((q & 12u) == 12u);
                const bool n = ((t | q) & 8u) != 0;
                const uint32_t idx = (t ^ (q & 3u)) & 7u;
                const uint32_t tv = (idx & 4u) ? TAB_HI : TAB_LO;
                u[h] = n ? U_N : ((tv >> ((idx & 3u) * 8)) & 0xffu);
                kl[h] = end ? 0xffffu : 0u;
            }
            sc[c] = u[0] | (u[1] << 16);
            kill[c] = kl[0] | (kl[1] << 16);
        }
    }
    // the one cell of a neighbouring lane
    uint32_t eH, eX;
    if (PAR == 0) {        // up of pair 0 = (previous lane's last odd slot, own odd slot S/2-1)
        uint32_t ph = shfl_up(st.Ho[CH - 1], 1), pd = shfl_up(st.Do[CH - 1], 1);
        if (lane == 0) { ph = SENT2; pd = SENT2; }
        eH = prmt(ph, st.Ho[CH - 1], 0x5432); eX = prmt(pd, st.Do[CH - 1], 0x5432);
    } else {               // left of pair CH-1 = (own even slot S/2, next lane's slot 0)
        uint32_t nh = shfl_down(st.He[0], 1), ni = shfl_down(st.Ie[0], 1);
        if (lane == 31) { nh = SENT2; ni = SENT2; }
        eH = prmt(st.He[0], nh, 0x5432); eX = prmt(st.Ie[0], ni, 0x5432);
    }
#pragma unroll
    for (int c = 0; c < CH; c++) {
        uint32_t uH, uD, lH, lI, self;
        if (PAR == 0) {
            uH = c == 0 ? eH : st.Ho[c > 0 ? c - 1 : 0]; uD = c == 0 ? eX : st.Do[c > 0 ? c - 1 : 0];
            lH = st.Ho[c]; lI = st.Io[c]; self = st.He[c];
        } else {
            uH = st.He[c]; uD = st.De[c];
            lH = c == CH - 1 ? eH : st.He[c + 1 < CH ? c + 1 : c]; lI = c == CH - 1 ? eX : st.Ie[c + 1 < CH ? c + 1 : c];
            self = st.Ho[c];
        }
        const uint32_t nd = viaddmax2(uH, kopen2, uD);          // D = max(Hup - O, Dup)            (T domain)
        const uint32_t ni = viaddmax2(lH, kopen2, lI);          // I = max(Hleft - O, Ileft)
        const uint32_t mv = vadd2(self, sc[c]);                 // M = Hdiag + s + 2E
        const uint32_t nh = vmax3_2(mv, nd, ni);
        uint32_t dead = prmt(vadd2(nh, negthr2), 0, 0xBB99);    // 0xffff where H < threshold
        if (SPECIAL) dead |= kill[c];
        const uint32_t hs = vadd2(nh, negbias2);
        const uint32_t oh = (hs & ~dead) | (SENT2 & dead);
        const uint32_t od = (nd & ~dead) | (SENT2 & dead);
        const uint32_t oi = (ni & ~dead) | (SENT2 & dead);
        if (PAR == 0) { st.He[c] = oh; st.De[c] = od; st.Ie[c] = oi; } else { st.Ho[c] = oh; st.Do[c] = od; st.Io[c] = oi; }
    }
    // maximum of the step's cells of this lane: a tree, not a chain (it sits on the critical path to the next threshold)
    {
        uint32_t m[CH];
#pragma unroll
        for (int c = 0; c < CH; c++) m[c] = PAR == 0 ? st.He[c] : st.Ho[c];
#pragma unroll
        for (int n = CH; n > 1; n = (n + 2) / 3) {
#pragma unroll
            for (int x = 0; x < (n + 2) / 3; x++) {
                const uint32_t a = m[3 * x], b = 3 * x + 1 < n ? m[3 * x + 1] : a, d = 3 * x + 2 < n ? m[3 * x + 2] : a;
                m[x] = vmax3_2(a, b, d);
            }
        }
        hmax2 = m[0];
    }
}

template <int S>
YW_DEV void store_row(uint8_t* row, const uint32_t (&h)[Lay<S>::CH]) {
    constexpr int CH = Lay<S>::CH;
    uint32_t* p = reinterpret_cast<uint32_t*>(row) + lane_id() * CH;
#ifdef YW_EMU
#pragma unroll
    for (int c = 0; c < CH; c++) p[c] = h[c];
#else
    if (CH % 4 == 0) {
#pragma unroll
        for (int c = 0; c + 3 < CH; c += 4) *reinterpret_cast<uint4*>(p + c) = make_uint4(h[c], h[c + 1], h[c + 2], h[c + 3]);
    } else if (CH % 2 == 0) {
#pragma unroll
        for (int c = 0; c + 1 < CH; c += 2) *reinterpret_cast<uint2*>(p + c) = make_uint2(h[c], h[c + 1]);
    } else {
#pragma unroll
        for (int c = 0; c < CH; c++) p[c] = h[c];
    }
#endif
}

// after a step: the step maximum (stored domain) -> running best, threshold of the next step, dead-step count.
// Branch-free: the hot loop should not carry reconvergence points.
YW_DEV void after_step(Ctx& c, uint32_t hmax2) {
    const uint32_t both = vmax2(hmax2, prmt(hmax2, hmax2, 0x1032));
    const int bmax = lo16((uint32_t)redmax((int)both));
    c.k++;
    const int stepmax = bmax + c.bias;                 // T domain
    const bool alive = bmax > ALIVE_MIN;
    c.dead_steps = alive ? 0 : c.dead_steps + 1;
    const bool better = alive && stepmax > c.bestT;
    c.kbest = better ? c.k : c.kbest;
    c.bestv = better ? bmax : c.bestv;
    c.best_real = better ? stepmax + c.F - c.p.E * c.k : c.best_real;
    c.bestT = (better ? stepmax : c.bestT) + c.p.E;    // image of the best on the next anti-diagonal
}

// ------------------------------------------------------------------------------------------ one layout
template <int S>
YW_DEV void load_state(const Ctx& c, State<S>& st) {
    constexpr int CH = Lay<S>::CH;
    const int16_t* H = c.scr; const int16_t* D = c.scr + WIN; const int16_t* I = c.scr + 2 * WIN;
    const int d0 = c.rbase + S * lane_id();
#pragma unroll
    for (int x = 0; x < CH; x++) {
        const int a = (d0 + 2 * x) & (WIN - 1), b = (d0 + 2 * x + S / 2) & (WIN - 1);
        const int a1 = (d0 + 2 * x + 1) & (WIN - 1), b1 = (d0 + 2 * x + 1 + S / 2) & (WIN - 1);
        st.He[x] = pack2(H[a], H[b]); st.De[x] = pack2(D[a], D[b]); st.Ie[x] = pack2(I[a], I[b]);
        st.Ho[x] = pack2(H[a1], H[b1]); st.Do[x] = pack2(D[a1], D[b1]); st.Io[x] = pack2(I[a1], I[b1]);
    }
}
template <int S>
YW_DEV void dump_state(const Ctx& c, const State<S>& st) {
    constexpr int CH = Lay<S>::CH;
    int16_t* H = c.scr; int16_t* D = c.scr + WIN; int16_t* I = c.scr + 2 * WIN;
    const int d0 = c.rbase + S * lane_id();
#pragma unroll
    for (int x = 0; x < CH; x++) {
        const int a = (d0 + 2 * x) & (WIN - 1), b = (d0 + 2 * x + S / 2) & (WIN - 1);
        const int a1 = (d0 + 2 * x + 1) & (WIN - 1), b1 = (d0 + 2 * x + 1 + S / 2) & (WIN - 1);
        H[a] = (int16_t)lo16(st.He[x]); H[b] = (int16_t)hi16(st.He[x]); D[a] = (int16_t)lo16(st.De[x]); D[b] = (int16_t)hi16(st.De[x]);
        I[a] = (int16_t)lo16(st.Ie[x]); I[b] = (int16_t)hi16(st.Ie[x]);
        H[a1] = (int16_t)lo16(st.Ho[x]); H[b1] = (int16_t)hi16(st.Ho[x]); D[a1] = (int16_t)lo16(st.Do[x]); D[b1] = (int16_t)hi16(st.Do[x]);
        I[a1] = (int16_t)lo16(st.Io[x]); I[b1] = (int16_t)hi16(st.Io[x]);
    }
}

// move the frame by delta: every alive value drops by delta, dead stays SENT
template <int S>
YW_DEV void rebase_state(State<S>& st, int delta) {
    constexpr int CH = Lay<S>::CH;
    const uint32_t floor2 = pack2(SENT + delta, SENT + delta), neg2 = pack2(-delta, -delta);
#pragma unroll
    for (int x = 0; x < CH; x++) {
        st.He[x] = vadd2(vmax2(st.He[x], floor2), neg2); st.Ho[x] = vadd2(vmax2(st.Ho[x], floor2), neg2);
        st.De[x] = vadd2(vmax2(st.De[x], floor2), neg2); st.Do[x] = vadd2(vmax2(st.Do[x], floor2), neg2);
        st.Ie[x] = vadd2(vmax2(st.Ie[x], floor2), neg2); st.Io[x] = vadd2(vmax2(st.Io[x], floor2), neg2);
    }
}

template <int S, bool SPECIAL>
YW_DEV void run_block(Ctx& c, State<S>& st, const uint32_t (&XC)[Lay<S>::NWC], const uint32_t (&YC)[Lay<S>::NWC],
                      const uint32_t (&XR)[Lay<S>::NWR], const uint32_t (&YR)[Lay<S>::NWR], uint8_t* rowp, uint32_t& alive2) {
    const uint32_t kopen2 = pack2(c.bias - c.p.O, c.bias - c.p.O), negbias2 = pack2(-c.bias, -c.bias);
    const uint32_t SENT2 = pack2(SENT, SENT);
    alive2 = SENT2;
#pragma unroll 1
    for (int v = 0; v < BLOCK_STEPS / 2; v++) {
        if (c.dead_steps >= 2) break;
        uint32_t hm1 = SENT2, hm0 = SENT2;
        {
            const int thr = c.bestT - c.p.Y;
            step<S, SPECIAL, 1>(st, XC, YC, XR, YR, v, kopen2, negbias2, pack2(-thr, -thr), hm1);
            store_row<S>(rowp, st.Ho); rowp += Lay<S>::ROW_BYTES; c.nrows++;
            after_step(c, hm1);
        }
        if (c.dead_steps < 2) {
            const int thr = c.bestT - c.p.Y;
            step<S, SPECIAL, 0>(st, XC, YC, XR, YR, v, kopen2, negbias2, pack2(-thr, -thr), hm0);
            store_row<S>(rowp, st.He); rowp += Lay<S>::ROW_BYTES; c.nrows++;
            after_step(c, hm0);
        }
        alive2 = vmax2(hm1, hm0);
    }
}

// diagonals a layout of S per lane can hold with one free lane and 16 diagonals of slack on both sides
YW_DEV int usable(int S) { return 32 * S - 2 * (S + 16); }
// smallest allowed layout that holds `need` diagonals (+ hysteresis), 0 if none
YW_DEV int pick_layout(uint32_t mask, int need, int hyst, int max_S) {
    for (int S = 8; S <= max_S; S += 4)
        if (((mask >> (S >> 2)) & 1u) && need + hyst <= usable(S)) return S;     // mask bits exist only for instantiated layouts
    return 0;
}

// raw code streams of the block that starts after step kb, for this lane
template <int S>
YW_DEV void load_windows(const Ctx& c, int kb, uint32_t (&XR)[Lay<S>::NWR], uint32_t (&YR)[Lay<S>::NWR]) {
    constexpr int NWR = Lay<S>::NWR;
    const int lane = lane_id();
    const int64_t ib = ((int64_t)kb + c.rbase + (int64_t)S * lane) >> 1, jb = ((int64_t)kb - c.rbase - (int64_t)S * lane) >> 1;
    if (c.dir > 0) { load_stream<NWR>(c.tc, c.ta + ib, true, XR); load_stream<NWR>(c.qc, c.qa + jb + 3, false, YR); }
    else { load_stream<NWR>(c.tc, c.ta - ib - 1, false, XR); load_stream<NWR>(c.qc, c.qa - jb - 4, true, YR); }
}

// Runs blocks in layout (c.rbase, S) until the extension ends or the layout has to change. State comes from and goes
// back to the scratch.
template <int S>
YW_DEV void run_layout(Ctx& c, bool first) {
    constexpr int CH = Lay<S>::CH, NWC = Lay<S>::NWC, NWR = Lay<S>::NWR;
    const int lane = lane_id();
    State<S> st;
    load_state<S>(c, st);
    if (!chunk_open(c, first ? 0 : c.k + 1, Lay<S>::ROWS_PER_CHUNK)) return;
    if (first) {          // row 0: the anchor cell
        store_row<S>(c.pool.base + (size_t)c.chunk * CHUNK_BYTES, st.He);
        c.nrows = 1;
    }
    uint32_t XN[NWR], YN[NWR];                 // raw streams of the coming block
    load_windows<S>(c, c.k, XN, YN);
    for (;;) {
        // frame
        if (c.bestT > c.rebase_at) {
            const int delta = c.bestT - c.init_best;
            rebase_state<S>(st, delta);
            c.bestT -= delta; c.F += delta;
            if (!chunk_open(c, c.k + 1, Lay<S>::ROWS_PER_CHUNK)) break;
        } else if (c.nrows + BLOCK_STEPS > c.cap) {
            if (!chunk_open(c, c.k + 1, Lay<S>::ROWS_PER_CHUNK)) break;
        }
        // windows of this block: kb = c.k (even), cells of lane: i0 = ib + v + 1, j0 = jb + v (+1 on even steps).
        // X[n] = t(ib + 1 + n), Y[n] = q(jb + 4 - n);  dir +1: t(i) = T[ta + i - 1], dir -1: t(i) = T[ta - i].
        // The loads were issued one block ago (software pipeline); the ones for the next block (ib + 4, jb + 4) go out now.
        uint32_t XR[NWR], YR[NWR];
#pragma unroll
        for (int w = 0; w < NWR; w++) { XR[w] = XN[w]; YR[w] = YN[w]; }
        load_windows<S>(c, c.k + BLOCK_STEPS, XN, YN);
        uint32_t flags = 0;
#pragma unroll
        for (int w = 0; w < NWR; w++) flags |= (XR[w] | YR[w]) & 0x08080808u;
        const bool special = ballot(flags != 0) != 0;
        uint32_t XC[NWC], YC[NWC];
#pragma unroll
        for (int w = 0; w < NWC; w++) {
            XC[w] = XR[w] | (bytes_at(XR, 4 * w + CH) << 4);
            YC[w] = (YR[w] & 0x03030303u) | ((bytes_at(YR, 4 * w + CH) & 0x03030303u) << 4);
        }
        uint8_t* rowp = c.pool.base + (size_t)c.chunk * CHUNK_BYTES + (size_t)c.nrows * Lay<S>::ROW_BYTES;
        uint32_t alive2;
        if (special) run_block<S, true>(c, st, XC, YC, XR, YR, rowp, alive2);
        else run_block<S, false>(c, st, XC, YC, XR, YR, rowp, alive2);
        if (c.dead_steps >= 2) break;
        // alive lanes (from the last odd and even step of the block)
        const int lm = lo16(vmax2(alive2, prmt(alive2, alive2, 0x1032)));
        const uint32_t am = ballot(lm > ALIVE_MIN);
        if (am == 0) { c.lo_lane = c.hi_lane = 16; }
        else {
#ifdef YW_EMU
            c.lo_lane = __builtin_ctz(am); c.hi_lane = 31 - __builtin_clz(am);
#else
            c.lo_lane = __ffs(am) - 1; c.hi_lane = 31 - __clz(am);
#endif
        }
        c.cells += (uint32_t)(c.hi_lane - c.lo_lane + 1) * (S / 2) * BLOCK_STEPS;
#ifdef YW_EMU_TRACE
        if (lane == 0) fprintf(stderr, "[fw] k %d S %d rbase %d lanes %d..%d bestT %d best %d dead %d special %d\n", c.k, S, c.rbase, c.lo_lane, c.hi_lane, c.bestT, c.best_real, c.dead_steps, (int)special);
#endif
        // the band may move one diagonal per step: a free lane on both sides covers the next block (S >= BLOCK_STEPS)
        if (c.lo_lane < 1 || c.hi_lane > 30) break;
        // shrink when a smaller layout would do (with hysteresis; lane granularity overestimates the need, which is safe)
        { const int ps = pick_layout(c.lay_mask, (c.hi_lane - c.lo_lane + 1) * S, 64, S - 4); if (ps != 0) break; }
    }
    {   // exact range of alive diagonals (every slot holds its diagonal's latest cell)
        int dlo = INT32_MAX, dhi = INT32_MIN;
        const int d0 = c.rbase + S * lane;
#pragma unroll
        for (int x = 0; x < CH; x++) {
            if (lo16(st.He[x]) > ALIVE_MIN) { dlo = dlo < d0 + 2 * x ? dlo : d0 + 2 * x; dhi = dhi > d0 + 2 * x ? dhi : d0 + 2 * x; }
            if (hi16(st.He[x]) > ALIVE_MIN) { dlo = dlo < d0 + 2 * x + S / 2 ? dlo : d0 + 2 * x + S / 2; dhi = dhi > d0 + 2 * x + S / 2 ? dhi : d0 + 2 * x + S / 2; }
            if (lo16(st.Ho[x]) > ALIVE_MIN) { dlo = dlo < d0 + 2 * x + 1 ? dlo : d0 + 2 * x + 1; dhi = dhi > d0 + 2 * x + 1 ? dhi : d0 + 2 * x + 1; }
            if (hi16(st.Ho[x]) > ALIVE_MIN) { dlo = dlo < d0 + 2 * x + 1 + S / 2 ? dlo : d0 + 2 * x + 1 + S / 2; dhi = dhi > d0 + 2 * x + 1 + S / 2 ? dhi : d0 + 2 * x + 1 + S / 2; }
        }
        c.alo = redmin(dlo); c.ahi = redmax(dhi);
    }
    if (lane == 0 && c.chunk != 0xffffffffu) c.pool.meta[c.chunk].nrows = c.nrows;
    dump_state<S>(c, st);
    syncwarp();
}

// One extension by one warp. Returns through res; the trace stays in the pool for the walk-back. MAXS = widest layout
// this instantiation may use (32: the common kernel; 64: the wide-band kernel, more registers).
template <int MAXS>
YW_DEV void ydrop_forward_warp(const uint8_t* tcodes, const uint8_t* qcodes, int64_t ta, int64_t qa, int dir, Params p,
                               Pool pool, uint32_t item, uint32_t warp_slot, uint32_t& priv_used, ExtResult* res, uint32_t lay_mask) {
    constexpr int max_S = MAXS;
    Ctx c;
    c.tc = tcodes; c.qc = qcodes; c.ta = ta; c.qa = qa; c.dir = dir; c.p = p;
    c.bias = 125 - 2 * p.E;
    c.lay_mask = lay_mask; c.alo = c.ahi = 0;
    c.k = 0; c.S = pick_layout(lay_mask, 1, 0, max_S); c.rbase = -16 * c.S;
    c.init_best = INIT_THR + p.Y; c.rebase_at = REBASE_THR + p.Y;
    c.F = -c.bias - c.init_best;               // stored H(0,0) = 0 + 0 - bias - F = init_best
    c.bestT = c.init_best + c.bias + p.E;      // image of best = 0 on anti-diagonal 1
    c.best_real = 0; c.kbest = 0; c.bestv = c.init_best;
    c.dead_steps = 0; c.lo_lane = c.hi_lane = 16; c.cells = 0; c.status = ST_OK;
    c.pool = pool; c.item = item; c.slot = warp_slot; c.priv_used = priv_used; c.chunk = 0xffffffffu; c.k0 = 0; c.nrows = 0; c.cap = 0;
    c.scr = pool.scratch + (size_t)warp_slot * 3 * WIN;
    const int lane = lane_id();
    {
        uint32_t* w = reinterpret_cast<uint32_t*>(c.scr);
        const uint32_t s2 = pack2(SENT, SENT);
        for (int x = lane * 4; x < 3 * WIN / 2; x += 128) { w[x] = s2; w[x + 1] = s2; w[x + 2] = s2; w[x + 3] = s2; }
    }
    syncwarp();
    if (lane == 0) c.scr[0] = (int16_t)c.init_best;
    syncwarp();
    bool first = true;
    int maxs = 0, nlay = 0;
    while (c.status == ST_OK) {
        maxs = c.S > maxs ? c.S : maxs; nlay++;
        if (c.S == 8) run_layout<8>(c, first);
        else if (c.S == 12) run_layout<12>(c, first);
        else if (c.S == 16) run_layout<16>(c, first);
        else if (c.S == 20) run_layout<20>(c, first);
        else if (c.S == 24) run_layout<24>(c, first);
        else if (c.S == 32) run_layout<32>(c, first);
        else {
            if constexpr (MAXS >= 64) {
                if (c.S == 48) run_layout<48>(c, first);
                else if (c.S == 64) run_layout<64>(c, first);
                else c.status = ST_FAIL;
            } else {
                c.status = ST_FAIL;
            }
        }
        first = false;
        if (c.status != ST_OK || c.dead_steps >= 2) break;
        // next layout: the smallest allowed one that holds the alive diagonals [alo, ahi], centred on them
        if (c.ahi < c.alo) break;                      // nothing alive (the dead-step test normally catches this first)
        const int need = c.ahi - c.alo + 1;
        int ns = pick_layout(c.lay_mask, need, 0, max_S);
        if (ns == 0) { c.status = max_S >= 64 ? ST_BAND : ST_WIDE; break; }    // the caller reruns the item: wide kernel, then full rows
        const int slack = (32 * ns - need) / 2;
        c.S = ns;
        c.rbase = (c.alo - slack) & ~1;
    }
    priv_used = c.priv_used;
    if (lane == 0) {
        ExtResult r;
        r.score = c.best_real; r.kbest = c.kbest; r.bestv = c.bestv; r.chunk = c.chunk; r.status = c.status;
        r.di = r.dj = r.nmatch = r.ncols = 0; r.cells = c.cells; r.max_s = maxs; r.nlayouts = nlay;
        *res = r;
    }
}

// ------------------------------------------------------------------------------------------ walk-back
constexpr int DEADV = INT32_MIN;
constexpr int WCACHE = 16;          // chunk metas kept per walker (current + predecessors)

struct WalkCache {                  // per warp, in shared memory (or plain memory in the emulator)
    ChunkMeta m[WCACHE];
    uint32_t id[WCACHE];
    int n;
};

// H + E*k of cell (k, d), DEADV if dead / never stored. Searches the cached chunks (newest first).
YW_DEV int trace_val(const Pool& pool, const WalkCache& wc, int bias, int k, int d) {
    if (k < 0) return DEADV;
    for (int x = 0; x < wc.n; x++) {
        const ChunkMeta& m = wc.m[x];
        if (k >= m.k0) {
            if (k - m.k0 >= m.nrows) return DEADV;
            const int off = d - m.rbase - (k & 1);
            if (off < 0 || off >= 32 * m.S) return DEADV;
            const int ln = off / m.S, cell = (off - ln * m.S) >> 1, CHm = m.S >> 2;
            const int pair = cell % CHm, half = cell / CHm;
            const int16_t* row = reinterpret_cast<const int16_t*>(pool.base + (size_t)wc.id[x] * CHUNK_BYTES + (size_t)(k - m.k0) * (32 * CHm * 4));
            const int v = row[(ln * CHm + pair) * 2 + half];
            return v > ALIVE_MIN ? v + bias + m.F : DEADV;
        }
    }
    // older than the cache (many short chunks in a row): follow the chain in memory
    uint32_t id = wc.n ? wc.m[wc.n - 1].prev : 0xffffffffu;
    while (id != 0xffffffffu) {
        const ChunkMeta m = pool.meta[id];
        if (k >= m.k0) {
            if (k - m.k0 >= m.nrows) return DEADV;
            const int off = d - m.rbase - (k & 1);
            if (off < 0 || off >= 32 * m.S) return DEADV;
            const int ln = off / m.S, cell = (off - ln * m.S) >> 1, CHm = m.S >> 2;
            const int pair = cell % CHm, half = cell / CHm;
            const int16_t* row = reinterpret_cast<const int16_t*>(pool.base + (size_t)id * CHUNK_BYTES + (size_t)(k - m.k0) * (32 * CHm * 4));
            const int v = row[(ln * CHm + pair) * 2 + half];
            return v > ALIVE_MIN ? v + bias + m.F : DEADV;
        }
        id = m.prev;
    }
    return DEADV;
}

// make wc.m[0] the chunk that holds step k; keep as many predecessors as fit
YW_DEV void cache_seek(const Pool& pool, WalkCache& wc, int k) {
    const int lane = lane_id();
    // drop chunks newer than k
    int drop = 0;
    while (drop < wc.n && wc.m[drop].k0 > k) drop++;
    if (drop) {
        syncwarp();
        ChunkMeta mm; uint32_t ii = 0;
        const bool mv = lane + drop < wc.n;
        if (mv) { mm = wc.m[lane + drop]; ii = wc.id[lane + drop]; }
        syncwarp();
        if (mv) { wc.m[lane] = mm; wc.id[lane] = ii; }
        syncwarp();
        if (lane == 0) wc.n -= drop;
        syncwarp();
    }
    // refill the tail
    for (;;) {
        const int n = wc.n;
        const uint32_t id = n > 0 ? wc.m[n - 1].prev : 0xffffffffu;
        syncwarp();                                   // every lane has read the state before lane 0 changes it
        if (n >= WCACHE || id == 0xffffffffu) break;
        if (lane == 0) { wc.m[n] = pool.meta[id]; wc.id[n] = id; wc.n = n + 1; }
        syncwarp();
    }
}

YW_DEV uint32_t score_u(uint32_t t, uint32_t q) {      // s + 125 for code bytes
    if ((t | q) & 8u) return U_N;
    const uint32_t idx = (t ^ (q & 3u)) & 7u;
    const uint32_t tv = (idx & 4u) ? TAB_HI : TAB_LO;
    return (tv >> ((idx & 3u) * 8)) & 0xffu;
}

YW_DEV void ydrop_walk_warp(const uint8_t* tcodes, const uint8_t* qcodes, int64_t ta, int64_t qa, int dir, Params p,
                            Pool pool, ExtResult* res, WalkCache& wc) {
    const int lane = lane_id();
    const int bias = 125 - 2 * p.E;
    ExtResult r = *res;
    if (r.status != ST_OK) return;
    if (r.kbest == 0) { if (lane == 0) { res->di = res->dj = res->nmatch = res->ncols = 0; } return; }
    // cache: start from the last chunk
    if (lane == 0) { wc.m[0] = pool.meta[r.chunk]; wc.id[0] = r.chunk; wc.n = 1; }
    syncwarp();
    // walk to the chunk holding kbest
    while (wc.m[0].k0 > r.kbest) {
        const uint32_t id = wc.m[0].prev;
        syncwarp();
        if (lane == 0) { wc.m[0] = pool.meta[id]; wc.id[0] = id; }
        syncwarp();
    }
    cache_seek(pool, wc, r.kbest);
    int k = r.kbest, d;
    {   // end cell: the smallest row (= smallest diagonal) on anti-diagonal kbest whose stored value is the best
        const ChunkMeta m = wc.m[0];
        const int CHm = m.S >> 2;
        const int16_t* row = reinterpret_cast<const int16_t*>(pool.base + (size_t)wc.id[0] * CHUNK_BYTES + (size_t)(k - m.k0) * (32 * CHm * 4));
        int dmin = INT32_MAX;
        for (int x = 0; x < 2 * CHm; x++) {
            const int pair = x >> 1, half = x & 1;
            if (row[(lane * CHm + pair) * 2 + half] == r.bestv) {
                const int cell = half * CHm + pair;
                const int dd = m.rbase + m.S * lane + 2 * cell + (k & 1);
                dmin = dd < dmin ? dd : dmin;
            }
        }
        d = redmin(dmin);
        if (d == INT32_MAX) { if (lane == 0) res->status = ST_FAIL; return; }
    }
    int i = (k + d) >> 1, j = (k - d) >> 1;
    const int di = i, dj = j;
#ifdef YW_EMU_TRACE
    if (lane == 0) fprintf(stderr, "[wb] end cell k %d d %d (i %d j %d) score %d\n", k, d, i, j, r.score);
#endif
    int nm = 0, nc = 0;
    bool fail = false;
    const int gmax = (p.Y - p.O) / p.E + 2;           // no gap is longer: it would fall below the y-drop threshold
    while (k > 0 && !fail) {
        cache_seek(pool, wc, k);
        // ---- diagonal run: lane l tests cell (k - 2l, d) = (i - l, j - l)
        const int kl = k - 2 * lane;
        const int v = trace_val(pool, wc, bias, kl, d);
        const int vn = (int)shfl_down((uint32_t)v, 1);
        const int il = i - lane, jl = j - lane;
        bool isM = false, match = false;
        if (lane < 31 && il >= 1 && jl >= 1 && v != DEADV && vn != DEADV) {
            const uint32_t t = dir > 0 ? ld8(tcodes + ta + il - 1) : ld8(tcodes + ta - il);
            const uint32_t q = dir > 0 ? ld8(qcodes + qa + jl - 1) : ld8(qcodes + qa - jl);
            const int s2e = (int)score_u(t, q) - 125 + 2 * p.E;
            isM = vn + s2e == v;
            match = ((t | q) & 8u) == 0 && ((t ^ q) & 3u) == 0;
        }
        const uint32_t bm = ballot(isM), bmatch = ballot(match);
#ifdef YW_EMU
        const int run = __builtin_ctz(~bm);
#else
        const int run = __ffs(~bm) - 1;
#endif
        const uint32_t rmask = run >= 32 ? 0xffffffffu : ((1u << run) - 1u);
#ifdef YW_EMU
        nm += __builtin_popcount(bmatch & rmask);
#else
        nm += __popc(bmatch & rmask);
#endif
        nc += run; k -= 2 * run; i -= run; j -= run;
#ifdef YW_EMU_TRACE
        if (lane == 0) fprintf(stderr, "[wb] run %d -> k %d d %d i %d j %d nm %d nc %d\n", run, k, d, i, j, nm, nc);
#endif
        if (run == 31 || k == 0) continue;
        // ---- a gap ends at (k, d): D first (vertical: (i-g, j)), then I
        const int h = (int)shfl((uint32_t)v, run);
        int glen = 0, gdir = 0;
        for (int pass = 0; pass < 2 && glen == 0; pass++) {
            const int sd = pass == 0 ? -1 : +1;
            bool stop = false;
            for (int r0 = 0; r0 < gmax && !stop; r0 += 32) {
                const int g = r0 + lane + 1;
                const int vg = trace_val(pool, wc, bias, k - g, d + sd * g);
                const uint32_t bf = ballot(vg != DEADV && vg - p.O == h), bd = ballot(vg == DEADV);
#ifdef YW_EMU
                const int f = bf ? __builtin_ctz(bf) : 32, z = bd ? __builtin_ctz(bd) : 32;
#else
                const int f = bf ? __ffs(bf) - 1 : 32, z = bd ? __ffs(bd) - 1 : 32;
#endif
                if (f < z) { glen = r0 + f + 1; gdir = sd; stop = true; }
                else if (z < 32) stop = true;
            }
        }
#ifdef YW_EMU_TRACE
        if (lane == 0) fprintf(stderr, "[wb] gap len %d dir %d at k %d d %d h %d\n", glen, gdir, k, d, h);
#endif
        if (glen == 0) { fail = true; break; }
        k -= glen; d += gdir * glen;
        if (gdir < 0) i -= glen; else j -= glen;
    }
    if (i != 0 || j != 0 || d != 0) fail = true;
    if (lane == 0) {
        res->di = di; res->dj = dj; res->nmatch = nm; res->ncols = nc;
        if (fail) res->status = ST_FAIL;
    }
}


// ------------------------------------------------------------------------------------------ full-row fallback
// The extensions whose band outgrows the widest layout (ST_BAND; e.g. y-drop 20000 with cheap gaps from an anchor inside a
// repeat pair: the alive cells of one anti-diagonal then span more than 2048 diagonals). The spec's recurrence (the oracle's
// ydrop_extend, D4) evaluated literally in 32-bit scores: every cell between the alive ranges of the two previous
// anti-diagonals, three rows of FullCell in `rows` (3 * cap cells), (nmatch, ncols) carried along each state instead of a
// trace. One warp, lane l takes cells clo + l, clo + l + 32, ...; slow, but only the rare ST_BAND items take it.
// tn / qn = bases available from the anchor in the extension direction. Fills score, di, dj, nmatch, ncols, cells; status =
// ST_OK, or ST_FAIL if an anti-diagonal needs more than cap cells.
struct FullCell { int32_t h, d, i, hm, hc, dm, dc, im, ic; };
constexpr int FULL_NEG = INT32_MIN / 4;

YW_DEV int full_sub(uint32_t a, uint32_t b) {
    if (a >= CODE_N || b >= CODE_N) return -100;
    const int tab[16] = {91, -114, -31, -123, -114, 100, -125, -31, -31, -125, 100, -114, -123, -31, -114, 91};
    return tab[((a & 3u) << 2) | (b & 3u)];
}

YW_DEV void ydrop_full_warp(const uint8_t* __restrict__ tcodes, const uint8_t* __restrict__ qcodes, int64_t ta, int64_t qa, int dir,
                            int64_t tn, int64_t qn, const Params& p, FullCell* rows, int64_t cap, ExtResult* res) {
    const int lane = lane_id();
    FullCell *p2 = rows, *p1 = rows + cap, *cur = rows + 2 * cap;
    int64_t b2 = 0, lo2 = 0, hi2 = -1, b1 = 0, lo1 = 0, hi1 = 0;   // row base (index of slot 0), alive range; k-1 = anti-diagonal 0
    if (lane == 0) { FullCell z = {0, FULL_NEG, FULL_NEG, 0, 0, 0, 0, 0, 0}; p1[0] = z; }
    syncwarp();
    int best = 0, r_score = 0, r_di = 0, r_dj = 0, r_nm = 0, r_nc = 0, status = ST_OK;
    uint64_t cells = 0;
    for (int64_t k = 1; k <= tn + qn; k++) {
        int64_t clo = INT64_MAX, chi = INT64_MIN;
        if (hi1 >= lo1) { clo = lo1; chi = hi1 + 1; }
        if (hi2 >= lo2) { if (lo2 + 1 < clo) clo = lo2 + 1; if (hi2 + 1 > chi) chi = hi2 + 1; }
        if (clo == INT64_MAX) break;
        if (clo < 0) clo = 0;
        if (clo < k - qn) clo = k - qn;
        if (chi > k) chi = k;
        if (chi > tn) chi = tn;
        int64_t nlo = INT64_MAX, nhi = INT64_MIN;
        int amax = FULL_NEG;
        if (chi >= clo) {
            if (chi - clo + 1 > cap) { status = ST_FAIL; break; }
            const int thr = best - p.Y;
            for (int64_t i = clo + lane; i <= chi; i += 32) {
                const int64_t j = k - i;
                FullCell c = {FULL_NEG, FULL_NEG, FULL_NEG, 0, 0, 0, 0, 0, 0};
                if (i - 1 >= lo1 && i - 1 <= hi1) {                       // up: (i-1, j) on k-1
                    const FullCell u = p1[i - 1 - b1];
                    if (u.h > FULL_NEG) {
                        const int op = u.h - p.O - p.E, ex = u.d > FULL_NEG ? u.d - p.E : FULL_NEG;
                        if (op >= ex) { c.d = op; c.dm = u.hm; c.dc = u.hc; } else { c.d = ex; c.dm = u.dm; c.dc = u.dc; }
                    }
                }
                if (i >= lo1 && i <= hi1) {                               // left: (i, j-1) on k-1
                    const FullCell l = p1[i - b1];
                    if (l.h > FULL_NEG) {
                        const int op = l.h - p.O - p.E, ex = l.i > FULL_NEG ? l.i - p.E : FULL_NEG;
                        if (op >= ex) { c.i = op; c.im = l.hm; c.ic = l.hc; } else { c.i = ex; c.im = l.im; c.ic = l.ic; }
                    }
                }
                int mval = FULL_NEG, mm = 0, mc = 0;                      // diagonal: (i-1, j-1) on k-2
                if (i >= 1 && j >= 1 && i - 1 >= lo2 && i - 1 <= hi2) {
                    const FullCell g = p2[i - 1 - b2];
                    if (g.h > FULL_NEG) {
                        const uint32_t a = ld8(tcodes + (dir > 0 ? ta + i - 1 : ta - i)), b = ld8(qcodes + (dir > 0 ? qa + j - 1 : qa - j));
                        mval = g.h + full_sub(a, b); mm = g.hm + (a == b && a < CODE_N ? 1 : 0); mc = g.hc + 1;
                    }
                }
                if (mval >= c.d && mval >= c.i) { c.h = mval; c.hm = mm; c.hc = mc; }
                else if (c.d >= c.i) { c.h = c.d; c.hm = c.dm; c.hc = c.dc; }
                else { c.h = c.i; c.hm = c.im; c.hc = c.ic; }
                if (c.h <= FULL_NEG || c.h < thr) { c.h = c.d = c.i = FULL_NEG; }
                else {
                    if (i < nlo) nlo = i;
                    nhi = i;
                    if (c.h > amax) amax = c.h;
                }
                cur[i - clo] = c;
            }
            cells += (uint64_t)(chi - clo + 1);
        }
        syncwarp();
        // the first cell (smallest i) that beats the best of all earlier anti-diagonals, as the sequential scan finds it
        const int m = redmax(amax);
        const int lo_i = redmin(nlo == INT64_MAX ? INT32_MAX : (int)nlo), hi_i = redmax(nhi == INT64_MIN ? INT32_MIN : (int)nhi);
        if (m > best) {
            int first = INT32_MAX;
            for (int64_t i = clo + lane; i <= chi; i += 32) if (cur[i - clo].h == m) { first = (int)i; break; }
            first = redmin(first);
            const FullCell c = cur[first - clo];
            best = m; r_score = m; r_di = first; r_dj = (int)(k - first); r_nm = c.hm; r_nc = c.hc;
        }
        FullCell* t = p2; p2 = p1; b2 = b1; lo2 = lo1; hi2 = hi1; p1 = cur; cur = t;
        b1 = clo;
        if (hi_i >= lo_i && lo_i != INT32_MAX) { lo1 = lo_i; hi1 = hi_i; } else { lo1 = 0; hi1 = -1; }
        syncwarp();
    }
    if (lane == 0) {
        res->score = r_score; res->di = r_di; res->dj = r_dj; res->nmatch = r_nm; res->ncols = r_nc;
        res->cells = (uint32_t)(cells > 0xffffffffull ? 0xffffffffull : cells); res->status = status;
    }
}

}  // namespace yw
