// seed.cu -- kernel family (a): 12-of-19 spaced-seed position table and lookup, fused with the
// leader test and a bounded first-stage gap-free extension that discards the (overwhelmingly
// random) seed hits which provably cannot reach --hspthresh.
//
// Replaces LASTZ's seed position table + seed_hit_search + the start of its gap-free extension
// (reached from mimeo through wrappers.py:1025-1037 / 786-798 / 645-653; SURVEY.md 9.1).
//
//   seed_keys_kernel     every target position -> 24-bit key of its 19-mer window (or "invalid")
//   radix_sort_bits      positions sorted by key (stable, deterministic)
//   bucket_offsets_kernel  key -> [begin,end) in the sorted position list (2^24+1 offsets)
//   seed_scan_kernel     per query position: 13 probes (exact + 12 single-transition variants);
//                        per candidate target position: run-leader test (spec D1), then an exact
//                        x-drop extension bounded to 60 columns right / 90 left. Hits whose
//                        extension terminated inside the bounds with score < K are dead (they can
//                        never become an HSP and, by spec D2, leave no trace); everything else is
//                        a survivor and is appended as (diagonal, query position) for stage 2.
#include "primitives.cuh"
#include "seq.cuh"
#include "internal.cuh"
#include "xdrop_table.cuh"

namespace mb2 {

constexpr uint32_t KEY_INVALID = 1u << 24;
constexpr int S1_WINDOW = 30;        // columns per first-stage window = 10 table chunks of 3 columns
constexpr int S1_RIGHT_WINDOWS = 2;  // 60 columns
constexpr int S1_LEFT_WINDOWS = 3;   // 90 columns (19 of them are the seed itself)
constexpr int S1_TAB = XT_SIZE;      // 3 columns of merged 4-bit codes -> packed {sum, max prefix, min prefix}

__global__ void __launch_bounds__(256)
seed_keys_kernel(GenomeView T, uint32_t p_lo, uint32_t n, uint32_t* __restrict__ keys, uint32_t* __restrict__ pos) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const uint32_t p = p_lo + k;
    const uint32_t nw = nwindow32(T.sm, p) & SEED_WINDOW_MASK19;    // non-ACGT or soft-masked: no seed word
    keys[k] = nw ? KEY_INVALID : seed_key(window32(T.pk, p));
    pos[k] = p;
}

// off[k] = first index in sorted keys with key >= k, for k in [0, 2^24]; sorted keys end with KEY_INVALID entries
__global__ void __launch_bounds__(256)
bucket_offsets_kernel(const uint32_t* __restrict__ keys, uint32_t n, uint32_t* __restrict__ off) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx > n) return;
    const int64_t prev = idx == 0 ? -1 : (int64_t)keys[idx - 1];
    const int64_t cur = idx == n ? (int64_t)KEY_INVALID : (int64_t)min(keys[idx], KEY_INVALID);
    for (int64_t k = prev + 1; k <= cur; k++) off[k] = idx;
}

void build_seed_table(const Genome& T, uint32_t p_lo, uint32_t p_hi, SeedTable& tab) {
    const uint32_t n = p_hi - p_lo;
    ProfScope ps("seed_table_build");
    DevBuf<uint32_t> k0(n), k1(n), v0(n), v1(n);
    launch(seed_keys_kernel, cdiv(n, 256), 256, 0, view(T), p_lo, n, k0.get(), v0.get());
    const int w = radix_sort_bits<uint32_t, uint32_t>(k0.get(), k1.get(), v0.get(), v1.get(), n, 0, 25);
    tab.off.alloc((size_t)KEY_INVALID + 1);
    launch(bucket_offsets_kernel, cdiv((size_t)n + 1, 256), 256, 0, w ? k1.get() : k0.get(), n, tab.off.get());
    tab.pos = std::move(w ? v1 : v0);
    tab.p_lo = p_lo; tab.p_hi = p_hi;
}

// First-stage table over merged codes: three columns of 4 bits, m = t ^ q on the base bits and t | q on the parity and
// non-ACGT bits (nib_merge). That is enough to score a column: a set bit 3 scores SCORE_N; otherwise x = t ^ q decides HOXD70
// except for x = 0 (A/A 91, C/C 100) and x = 3 (A/T -123, C/G -125), whose two bases have equal parity, so the OR is the target's.
// N columns inside the table keep the chunk rule exact (-100 lies within HOXD70's range: prefix sums inside a chunk still differ
// by at most 250 < X). Entry: bits 22..31 = s0+s1+s2 (signed), bits 13..21 = 125 + max prefix sum, bits 0..12 = 125 + X + min
// prefix sum. State of a lane: (best, D) with D = (best - run) + 125 >= 125; a chunk is
//   terminate iff min_field < D;   DM = max(D, max_field);   best += DM - D;   D = DM - sum
// (the rule of xdrop_table.cuh with D shifted by X - 250). A finished lane parks at D = S1_DONE, where every later chunk is
// a no-op on best.
// The index of a chunk is its 12 bits of merged code with bits 2..3 (parity and N of the first column) xor bits 8..9 (x of the
// third column; s1_prepare). The bank of a lookup is index bits 0..4, and the 32 hits of a batch mostly share one query
// window: of the plain code only x of the first column and one bit of x of the second vary with the target there (8 banks,
// about 5.2 wavefronts per lookup for random bases against 2.0 for 32 banks); with the xor all five bits do.
constexpr int S1_DONE = 1 << 24;
constexpr int S1_D0 = 125;                     // run = best = 0
constexpr int S1_MAX_XDROP = 8191 - 125 - 300; // min field fits 13 bits
__device__ __forceinline__ uint32_t s1_entry(uint32_t idx, int X) {
    const uint32_t code = idx ^ (((idx >> 8) & 3u) << 2);
    int sum = 0, mx = INT_MIN, mn = INT_MAX;
    for (int c = 0; c < 3; c++) {
        const uint32_t nib = (code >> (4 * c)) & 15u, t = (nib >> 2) & 1u;   // t: A or C, with the column's parity
        sum += (nib & 8u) ? SCORE_N : sub_lut((t << 2) | (t ^ (nib & 3u)));
        mx = max(mx, sum); mn = min(mn, sum);
    }
    return ((uint32_t)sum << 22) | ((uint32_t)(mx + 125) << 13) | (uint32_t)(mn + X + 125);
}
// bits [s, s + 32) of the 128-bit window w for a compile-time s in (-32, 128); negative s shifts left
__device__ __forceinline__ uint32_t s1_bits(const uint32_t (&w)[4], int s) {
    if (s < 0) return w[0] << (-s);
    const int j = s >> 5, r = s & 31;
    return r == 0 ? w[j] : (j < 3 ? __funnelshift_r(w[j], w[j + 1], r) : w[3] >> r);
}
// A window of merged codes (first column in the low bits of w[0]) made ready for xdrop_window30: returns whether one of its
// 30 columns is non-ACGT, then applies the index xor of every chunk.
__device__ __forceinline__ bool s1_prepare(uint32_t (&w)[4]) {
    const bool an = (((w[0] | w[1] | w[2]) & 0x88888888u) | (w[3] & 0x00888888u)) != 0;
    constexpr uint32_t SW0 = 0x0C00C00Cu, SW1 = 0xC00C00C0u, SW2 = 0x00C00C00u, SW3 = 0x0000C00Cu;   // bits 12k + 2, 12k + 3
    w[0] ^= __funnelshift_r(w[0], w[1], 6) & SW0;
    w[1] ^= __funnelshift_r(w[1], w[2], 6) & SW1;
    w[2] ^= __funnelshift_r(w[2], w[3], 6) & SW2;
    w[3] ^= (w[3] >> 6) & SW3;
    return an;
}
// 30 columns of a prepared window; updates (best, D) of the lane exactly as the column-by-column rule would.
// tab_sa = shared-space address of the table. nchunks counts the chunks a lane entered while still open, except that a window
// with a non-ACGT column (an) that is entered while open counts all 10 (the count the scan has always reported).
template <uint32_t VOTES>
__device__ __forceinline__ void xdrop_window30(uint32_t tab_sa, uint32_t m10, uint32_t m9, const uint32_t (&w)[4], bool an,
                                               int& best, int& D, uint32_t& nchunks) {
    const bool all10 = an && D < S1_DONE / 2;
    uint32_t parked = 0;                       // sum of D at chunk entry: S1_DONE per parked chunk + (< 2^24 in total) for the open ones
    int entered = S1_WINDOW / 3;
#pragma unroll
    for (int k = 0; k < S1_WINDOW / 3; k++) {
        if ((VOTES >> k) & 1u) { if (__all_sync(0xffffffffu, D >= S1_DONE / 2)) { entered = k; break; } }
        // byte address = table + 4 * (12 bits of chunk k)
        const uint32_t addr = (s1_bits(w, 12 * k - 2) & 0x3FFCu) + tab_sa;
        uint32_t e;
        asm("ld.shared.u32 %0, [%1];" : "=r"(e) : "r"(addr));
        parked += (uint32_t)D;
        // The max-prefix and sum fields are cut out with multiplies (fma pipe) instead of shifts and masks (alu pipe, the busier
        // one): (e * 2^10) hi-multiplied by 2^9 = bits 13..21, e hi-multiplied by 2^10 = e >> 22 (signed). The multipliers arrive
        // in registers so that they stay multiplies.
        const bool term = (int)(e & 0x1FFFu) < D;
        const int dm = max(D, (int)__umulhi(e * m10, m9));
        best += dm - D;
        D = term ? S1_DONE : dm - __mulhi((int)e, (int)m10);
    }
    nchunks += all10 ? (uint32_t)(S1_WINDOW / 3) : (uint32_t)entered - (parked >> 24);
}
// (best, D) of one side in a deferred record: best < 2^16 (at most 90 columns of at most +100), an open D < 2^13 (the min
// field); a terminated side stores 0xFFFF in the D half.
__device__ __forceinline__ uint32_t s1_pack(int best, int D) {
    return (uint32_t)best | ((D < S1_DONE / 2 ? (uint32_t)D : 0xFFFFu) << 16);
}
__device__ __forceinline__ void s1_unpack(uint32_t w, int& best, int& D) {
    best = (int)(w & 0xFFFFu);
    D = (w >> 16) == 0xFFFFu ? S1_DONE : (int)(w >> 16);
}

// Merged code of target and query nb words (see s1_entry): M ? t ^ q : t | q with M = 0x33333333, one LOP3 (LUT 0x7A for
// the operands t, M, q; written out because ptxas splits the plain expression into three)
__device__ __forceinline__ uint32_t nib_merge(uint32_t t, uint32_t q) {
    uint32_t m;
    asm("lop3.b32 %0, %1, %2, %3, 0x7A;" : "=r"(m) : "r"(t), "r"(0x33333333u), "r"(q));
    return m;
}
// the eight 4-bit groups of a word in reverse order: a byte reversal, then M ? x >> 4 : x << 4 with M = 0x0F0F0F0F (LUT 0xE2
// for the operands x >> 4, M, x << 4)
__device__ __forceinline__ uint32_t nib_rev(uint32_t x) {
    x = __byte_perm(x, 0u, 0x0123u);
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0xE2;" : "=r"(r) : "r"(x >> 4), "r"(0x0F0F0F0Fu), "r"(x << 4));
    return r;
}
// NW words of nb codes = the 8 NW columns from column p (p in the low bits of w[0]), read as NW / 2 + 1 aligned 8-byte loads
template <int NW>
__device__ __forceinline__ void nib_span(const uint32_t* __restrict__ nb, uint32_t p, uint32_t (&w)[NW]) {
    const uint32_t w0 = (p >> 3) & ~1u, sh = (p & 7u) * 4u;
    const bool odd = p & 8u;
    uint32_t x[NW + 2];
#pragma unroll
    for (int i = 0; i < NW / 2 + 1; i++) {
        const uint2 v = *reinterpret_cast<const uint2*>(nb + w0 + 2 * i);
        x[2 * i] = v.x; x[2 * i + 1] = v.y;
    }
#pragma unroll
    for (int m = 0; m < NW; m++) w[m] = __funnelshift_r(odd ? x[m + 1] : x[m], odd ? x[m + 2] : x[m + 1], sh);
}
// Leader test on 19 merged columns (l0: columns 0..7, l1: 8..15, l2: 16..18) that hold no non-ACGT base: do they form a seed
// hit, i.e. x = 0 in every care column, or (transition) x = 2 in exactly one and 0 in the others?
__device__ __forceinline__ bool seed_match_merged(uint32_t l0, uint32_t l1, uint32_t l2, bool transition) {
    const uint32_t x0 = l0 & 0x30030333u, x1 = l1 & 0x30303003u, x2 = l2 & 0x333u;   // x bits of the care columns
    if ((x0 | x1 | x2) == 0) return true;
    return transition && ((x0 | x1 | x2) & 0x11111111u) == 0 && __popc(x0) + __popc(x1) + __popc(x2) == 1;
}

// Appends the survivors of a warp (diagonal, query position) at one atomically reserved range of surv.
__device__ __forceinline__ void append_survivors(bool survivor, uint32_t hi, uint32_t hj, uint32_t diag_bias, int lane,
                                                 uint64_t* __restrict__ surv, uint32_t surv_cap, unsigned long long* __restrict__ counters) {
    const uint32_t smask = __ballot_sync(0xffffffffu, survivor);
    if (smask) {
        unsigned long long basev = 0;
        if (lane == __ffs(smask) - 1) basev = atomicAdd(&counters[0], (unsigned long long)__popc(smask));
        basev = __shfl_sync(0xffffffffu, basev, __ffs(smask) - 1);
        if (survivor) {
            const unsigned long long slot = basev + __popc(smask & ((1u << lane) - 1u));
            if (slot < surv_cap) surv[slot] = ((uint64_t)(hi - hj + diag_bias) << 32) | hj;
        }
    }
}

// ---- load-balanced scan --------------------------------------------------------------------------------------
// Every WARP works on its own: no CTA barrier after the table build. A warp takes 32 consecutive query positions per
// round (lane = position); rounds are handed out by an atomic counter. Phase A: the 13 bucket ranges of each position are looked up, the non-empty ones are
// compacted (warp scans, three probes at a time) into the warp's ring of descriptors {first hit number, first index in pos[], query position};
// hit numbers are cumulative over the warp's whole life. Phase B: whenever 32 hits are pending, lane l takes hit
// `consumed + l`, finds its descriptor (one OR-reduction over the next 32 descriptors + a popcount), and runs the leader test and the bounded x-drop
// (30-column windows, 3 columns per table lookup). Leftover hits (< 32) wait for the next round, so batches are always
// full except for the very last one of a warp. All loads of a batch that do not depend on the x-drop outcome (leader
// windows, first right and left windows) are issued together.
// A batch runs right window 0 and left windows 0 and 1. Right window 1 (needed by about 12 % of random hits, but by some lane
// of almost every batch) and left window 2 (about 2.5 %) would cost the whole warp for a few lanes, so a hit that is still
// open on the right after window 0 or on the left after window 1 is deferred instead: its state
// (target and query position, (best, D) of both sides) goes to the warp's queue of deferred hits, and whenever 32 are queued
// (and once more at the end of the warp's work) a drain batch resumes them, one per lane, where their batch left them.
// Which hits survive and how many chunks each enters do not depend on which lanes share a warp.
constexpr int SC_NT = 256;                 // threads per CTA
constexpr int SC_WARPS = SC_NT / 32;
constexpr int SC_NPROBE = 13;
constexpr int SC_HALF = 3;                 // probes appended per step: at most 3 * 32 = 96 descriptors
constexpr int SC_STEPS = (SC_NPROBE + SC_HALF - 1) / SC_HALF;   // steps per round
constexpr int SC_RING = 128;               // descriptors per warp: < 32 pending (every descriptor holds >= 1 hit) + 96 new
                                           // (a small ring keeps shared memory low, which leaves the SM more L1 for the gathers)
constexpr int SC_DQ = 64;                  // deferred hits per warp: < 32 queued (drained at 32) + at most 32 from one batch

// Window b >= 1 of the right or the left side of hit (hi, hj) in extension order (the left side reversed), prepared, for a lane
// whose side is still open (D); zero columns (a no-op) otherwise. an: the window holds a non-ACGT column.
__device__ __forceinline__ void s1_later_window(const GenomeView& T, const GenomeView& Q, uint32_t hi, uint32_t hj, bool right, int b, int D,
                                                uint32_t (&w)[4], bool& an) {
    w[0] = w[1] = w[2] = w[3] = 0; an = false;
    if (D >= S1_DONE / 2) return;
    const uint32_t d = right ? SEED_SPAN + S1_WINDOW * b : SEED_SPAN - S1_WINDOW * b - 32;
    uint32_t t[4], q[4];
    nib_span<4>(T.nb, hi + d, t); nib_span<4>(Q.nb, hj + d, q);
    if (right) {
#pragma unroll
        for (int i = 0; i < 4; i++) w[i] = nib_merge(t[i], q[i]);
    } else {
#pragma unroll
        for (int i = 0; i < 4; i++) w[i] = nib_rev(nib_merge(t[3 - i], q[3 - i]));
    }
    an = s1_prepare(w);
}

template <int MINB, uint32_t TAILVOTES>
__global__ void __launch_bounds__(SC_NT, MINB)
seed_scan_kernel(GenomeView T, GenomeView Q, const uint32_t* __restrict__ off, const uint32_t* __restrict__ pos,
                 uint32_t q_lo, uint32_t q_n, int X, int K, int transition, uint32_t diag_bias,
                 uint64_t* __restrict__ surv, uint32_t surv_cap, unsigned long long* __restrict__ counters) {
    __shared__ uint32_t s1tab[S1_TAB];
    __shared__ uint32_t r_cum[SC_WARPS][SC_RING], r_b0[SC_WARPS][SC_RING], r_j[SC_WARPS][SC_RING];
    __shared__ uint4 r_defer[SC_WARPS][SC_DQ];     // deferred hits {hi, hj, s1_pack(right), s1_pack(left)}
    __shared__ unsigned long long sh_stat[3];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int e = tid; e < S1_TAB; e += SC_NT) s1tab[e] = s1_entry((uint32_t)e, X);
    const uint32_t s1tab_sa = (uint32_t)__cvta_generic_to_shared(s1tab);
    const uint32_t s1_m10 = q_n ? 1024u : 0u, s1_m9 = q_n ? 512u : 0u;     // 2^10, 2^9 (q_n > 0 always; see xdrop_window30)
    if (tid < 3) sh_stat[tid] = 0;
    __syncthreads();
    uint32_t* __restrict__ rc = r_cum[warp];
    uint32_t* __restrict__ rb = r_b0[warp];
    uint32_t* __restrict__ rj = r_j[warp];
    uint4* __restrict__ dq = r_defer[warp];
    const int nprobe = transition ? SC_NPROBE : 1;
    const uint32_t nrounds = (q_n + 31) / 32;
    // Rounds are handed out dynamically (counters[CNT_WORK], zeroed by the caller): hits per round vary by orders of magnitude
    // between unique sequence and repeat families, and with a static stride the resident warps ran dry one after another
    // (ncu: 40 % warps active of a theoretical 50 %; C4 scan 480 -> 407 ms). A warp's step = (round, part): SC_HALF probes of
    // the round's 32 positions at a time.
    uint32_t round = 0;
    int part = SC_STEPS;                    // SC_STEPS: the current round is used up
    bool exhausted = false;
    uint32_t head = 0, tail = 0;            // ring positions (monotone, used modulo SC_RING)
    uint32_t cum_tail = 0, consumed = 0;    // hits appended / processed so far (wrapping arithmetic)
    uint32_t dq_head = 0, dq_tail = 0;      // deferred hits drained / queued so far (monotone, used modulo SC_DQ)
    unsigned long long n_lead = 0, n_cells = 0, n_hits = 0;
    for (;;) {
        // ---------------- phase A: append half rounds until a full batch is pending
        while (cum_tail - consumed < 32u && !exhausted) {
            if (part == SC_STEPS) {
                unsigned long long r = 0;
                if (lane == 0) r = atomicAdd(&counters[CNT_WORK], 1ull);
                r = __shfl_sync(0xffffffffu, r, 0);
                if (r >= nrounds) { exhausted = true; break; }
                round = (uint32_t)r; part = 0;
            }
            const int p0 = part * SC_HALF, p1 = min(SC_NPROBE, p0 + SC_HALF);
            part++;
            const uint32_t jrel = round * 32 + lane;
            const uint32_t j = q_lo + jrel;
            const bool jvalid = jrel < q_n && (nwindow32(Q.sm, j) & SEED_WINDOW_MASK19) == 0;
            uint32_t key = 0;
            if (jvalid) key = seed_key(window32(Q.pk, j));
            uint32_t b0[SC_HALF], cnt[SC_HALF];
            uint32_t mine = 0, nne = 0;
#pragma unroll
            for (int q = 0; q < SC_HALF; q++) {
                const int pr = p0 + q;
                uint32_t c = 0, b = 0;
                if (jvalid && pr < p1 && pr < nprobe) {
                    const uint32_t kk = pr == 0 ? key : key ^ (2u << (2 * (pr - 1)));
                    b = off[kk];
                    c = off[kk + 1] - b;
                }
                b0[q] = b; cnt[q] = c;
                mine += c; nne += c ? 1u : 0u;
            }
            // exclusive scans over the lanes of (hits, non-empty descriptors); descriptor order = (lane, probe)
            uint32_t sh = mine, sn = nne;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t th = __shfl_up_sync(0xffffffffu, sh, d), tn = __shfl_up_sync(0xffffffffu, sn, d);
                if (lane >= d) { sh += th; sn += tn; }
            }
            const uint32_t tot_h = __shfl_sync(0xffffffffu, sh, 31), tot_n = __shfl_sync(0xffffffffu, sn, 31);
            uint32_t run = cum_tail + sh - mine, slot = tail + sn - nne;
#pragma unroll
            for (int q = 0; q < SC_HALF; q++) {
                if (cnt[q]) {
                    const uint32_t w = slot & (SC_RING - 1);
                    rc[w] = run; rb[w] = b0[q]; rj[w] = j;
                    run += cnt[q]; slot++;
                }
            }
            tail += tot_n; cum_tail += tot_h; n_hits += (lane == 0) ? tot_h : 0;
            __syncwarp();
        }
        const uint32_t pending = cum_tail - consumed, queued = dq_tail - dq_head;
        if (pending == 0 && queued == 0) break;
        uint32_t hi = 0, hj = 0, nchunks = 0;
        int best_r = 0, dr = S1_DONE, best_l = 0, dl = S1_DONE;
        bool live;
        if (queued >= 32u || pending == 0) {
            // ---------------- drain: up to 32 deferred hits, one per lane, resume from their stored (best, D)
            static_assert(S1_RIGHT_WINDOWS == 2 && S1_LEFT_WINDOWS == 3, "a batch runs right window 0 and left windows 0, 1; a drain the rest");
            const uint32_t nd = min(queued, 32u);
            live = (uint32_t)lane < nd;
            if (live) {
                const uint4 r = dq[(dq_head + (uint32_t)lane) & (SC_DQ - 1)];
                hi = r.x; hj = r.y;
                s1_unpack(r.z, best_r, dr);
                s1_unpack(r.w, best_l, dl);
            }
            dq_head += nd;
            uint32_t w[4]; bool an;
            if (!__all_sync(0xffffffffu, dr >= S1_DONE / 2)) {
                s1_later_window(T, Q, hi, hj, true, 1, dr, w, an);
                xdrop_window30<TAILVOTES>(s1tab_sa, s1_m10, s1_m9, w, an, best_r, dr, nchunks);
            }
            if (!__all_sync(0xffffffffu, dl >= S1_DONE / 2)) {
                s1_later_window(T, Q, hi, hj, false, 2, dl, w, an);
                xdrop_window30<TAILVOTES>(s1tab_sa, s1_m10, s1_m9, w, an, best_l, dl, nchunks);
            }
        } else {
            // ---------------- phase B: one batch of up to 32 hits, one per lane
            const uint32_t nb = min(pending, 32u);
            live = (uint32_t)lane < nb;
            const uint32_t h = consumed + (uint32_t)lane;
            uint32_t e_last = head;
            {
                // Descriptor of every hit of the batch without a search: rc[head] <= consumed < rc[head + 1] (invariant of `head`) and
                // every descriptor holds at least one hit, so the batch lies inside descriptors head .. head + 31. Lane i looks at
                // descriptor head + i; the ones that START inside the batch (at offset 1..31) set a bit at their offset; the
                // descriptor of the hit at offset l is head + (bits at or below l).
                const uint32_t di = head + (uint32_t)lane;
                const bool dv = (int32_t)(tail - di) > 0;
                const uint32_t ci = dv ? rc[di & (SC_RING - 1)] : 0u;
                const uint32_t first = ci - consumed;                   // wrapping; >= 1 for lane > 0
                const uint32_t starts = __reduce_or_sync(0xffffffffu, (dv && lane > 0 && first < 32u) ? (1u << first) : 0u);
                if (live) {
                    const uint32_t lo = head + (uint32_t)__popc(starts & ((2u << lane) - 1u));
                    e_last = lo;
                    hi = pos[rb[lo & (SC_RING - 1)] + (h - rc[lo & (SC_RING - 1)])];
                    hj = rj[lo & (SC_RING - 1)];
                }
            }
            // Everything the batch needs that does not depend on the x-drop outcome: leader window (p - 1), first right window
            // (p + 19) and first left window (p - 13). All three lie inside the 64 columns from p - 13: the nb codes of both
            // sequences there are read with five aligned 8-byte loads each, merged once, and the windows are cut out of the merged
            // words. After the bank fix of the extension table the scan is bound by the integer ALU pipe (ncu on C4: alu pipe
            // 74 % busy, L1 data pipe 65 %, DRAM 11 %; profiles/r2_seed_scan_c4_v2_ncu_summary.txt); taking the pos[] and target
            // gathers of the next batch off the critical path (a pipelined variant, measured) changed nothing and was dropped.
            uint32_t rw[4] = {0, 0, 0, 0}, fw[4] = {0, 0, 0, 0};
            bool ra = false, fa = false;
            if (live) {
                uint32_t bt[8], bq[8], m[8];
                nib_span<8>(T.nb, hi - 13, bt); nib_span<8>(Q.nb, hj - 13, bq);
#pragma unroll
                for (int i = 0; i < 8; i++) m[i] = nib_merge(bt[i], bq[i]);
                const uint32_t l0 = __funnelshift_r(m[1], m[2], 16), l1 = __funnelshift_r(m[2], m[3], 16), l2 = m[3] >> 16;
                // not seedable: a non-ACGT column (bit 3 of the merged code), or a soft-masked one when either genome has lower
                // case (uniform; such a genome hands out an sm plane of its own)
                const uint32_t ln = (T.sm != T.nm || Q.sm != Q.nm) ? (nwindow32(T.sm, hi - 1) | nwindow32(Q.sm, hj - 1)) & SEED_WINDOW_MASK19
                                                                   : ((l0 | l1) & 0x88888888u) | (l2 & 0x888u);
                // spec D1: only run leaders are candidates
                if (ln == 0 && seed_match_merged(l0, l1, l2, transition != 0)) live = false; else n_lead++;
#pragma unroll
                for (int i = 0; i < 4; i++) { rw[i] = m[4 + i]; fw[i] = nib_rev(m[3 - i]); }
                ra = s1_prepare(rw); fa = s1_prepare(fw);
            }
            // Right of the seed: window 0 of 30 columns. Left, from the last seed column downwards: windows 0 and 1, reversed so
            // that the same forward-order table applies. The first window of either side comes out of the block above and runs
            // without polling (some lane of 32 is practically always still open at its end; on the left its first 19 columns are
            // the seed itself); left window 1 (needed by ~90 % of hits) is skipped when all lanes are done and polled inside.
            if (live) { dr = S1_D0; dl = S1_D0; }
            xdrop_window30<0u>(s1tab_sa, s1_m10, s1_m9, rw, ra, best_r, dr, nchunks);
            xdrop_window30<0u>(s1tab_sa, s1_m10, s1_m9, fw, fa, best_l, dl, nchunks);
            if (!__all_sync(0xffffffffu, dl >= S1_DONE / 2)) {
                uint32_t w[4]; bool an;
                s1_later_window(T, Q, hi, hj, false, 1, dl, w, an);
                xdrop_window30<TAILVOTES>(s1tab_sa, s1_m10, s1_m9, w, an, best_l, dl, nchunks);
            }
            // a hit still open on either side goes to the queue and is decided by a drain, also one whose best_r + best_l already
            // reaches K: stage1_cells counts every chunk a hit is open in
            const bool defer = live && (dr < S1_DONE / 2 || dl < S1_DONE / 2);
            const uint32_t dmask = __ballot_sync(0xffffffffu, defer);
            if (defer) {
                dq[(dq_tail + (uint32_t)__popc(dmask & ((1u << lane) - 1u))) & (SC_DQ - 1)] =
                    make_uint4(hi, hj, s1_pack(best_r, dr), s1_pack(best_l, dl));
                live = false;
            }
            dq_tail += (uint32_t)__popc(dmask);
            // retire the batch: descriptors that are fully consumed leave the ring
            consumed += nb;
            uint32_t e = __shfl_sync(0xffffffffu, e_last, (int)nb - 1);
            const uint32_t next_cum = (e + 1 < tail) ? rc[(e + 1) & (SC_RING - 1)] : cum_tail;
            head = ((int32_t)(next_cum - consumed) > 0) ? e : e + 1;
        }
        n_cells += 3ull * nchunks;
        // dead iff both sides terminated inside their bounds with a total below K (spec D2: failed extensions leave no trace)
        append_survivors(live && (dr < S1_DONE / 2 || dl < S1_DONE / 2 || best_r + best_l >= K), hi, hj, diag_bias, lane, surv, surv_cap, counters);
        __syncwarp();
    }
    // statistics
    if (n_lead) atomicAdd(&sh_stat[1], n_lead);
    if (n_cells) atomicAdd(&sh_stat[2], n_cells);
    if (n_hits) atomicAdd(&sh_stat[0], n_hits);
    __syncthreads();
    if (tid < 3 && sh_stat[tid]) atomicAdd(&counters[1 + tid], sh_stat[tid]);
}

// Enqueue the scan of query positions [q_lo, q_hi) against a built table. Survivors are appended to surv.
void seed_scan(const Genome& T, const Genome& Q, const SeedTable& tab, uint32_t q_lo, uint32_t q_hi, const AlignParams& p,
               uint64_t* surv, uint32_t surv_cap, unsigned long long* counters) {
    const uint32_t n = q_hi - q_lo;
    if (n == 0) return;
    MB2_REQUIRE(p.xdrop >= XT_MIN_XDROP, -2, "x-drop below 251 is not supported by the three-column extension table");
    MB2_REQUIRE(p.xdrop <= S1_MAX_XDROP, -2, "x-drop above 7766 is not supported by the first-stage extension table");
    ProfScope ps("seed_scan");
    const unsigned nrounds = cdiv(n, 32);
    // resident CTAs per SM: 4 (56 registers, no spill; default) or 3; the scan hides its gather latencies with resident warps
    // (C4: 5 % slower with 3; 5 CTAs at 48 registers: no faster). MB2_SCAN_MINB overrides.
    static const int minb = getenv("MB2_SCAN_MINB") ? atoi(getenv("MB2_SCAN_MINB")) : 4;
    auto go = [&](auto kern) {
        int per_sm = 0;
        MB2_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, SC_NT, 0));
        // persistent: exactly one resident wave of CTAs; every warp strides over the 32-position rounds
        const unsigned grid = std::min<unsigned>(cdiv(nrounds, SC_WARPS), (unsigned)ctx().sm_count * (unsigned)std::max(1, per_sm));
        launch(kern, grid, SC_NT, 0, view(T), view(Q), tab.off.get(), tab.pos.get(), q_lo, n, p.xdrop,
               p.hspthresh, p.transition, (uint32_t)Q.G, surv, surv_cap, counters);
    };
    // later windows are polled before chunks 3, 6 and 8 (measured on C4: 4/7, 2/4/6/8 and 1/3/5/7/9 are all within 0.6 %)
    if (minb <= 3) go(seed_scan_kernel<3, 0x148u>); else go(seed_scan_kernel<4, 0x148u>);
}

}  // namespace mb2
