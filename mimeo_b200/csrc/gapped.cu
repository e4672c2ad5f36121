// gapped.cu -- kernel family (c): anchors + affine-gap y-drop extension, anti-diagonal dynamic
// programming, integer only (no tensor cores: this is not a dense contraction).
//
// Replaces LASTZ's --gapped stage (SURVEY.md 9.1) under spec D4/D5 of oracle/lastz_oracle.c:
//   * every chained HSP is reduced to an anchor = centre of its best 31-column window;
//   * per tile, anchors are taken best-first; an anchor inside the bounding box of an alignment
//     already reported for the tile is skipped;
//   * from the anchor the alignment is extended forwards and backwards by an affine-gap DP
//     (open 400, extend 30) evaluated one anti-diagonal at a time; a cell survives iff
//     H >= best - ydrop, where best is the maximum over all earlier anti-diagonals. The three DP
//     states each carry (matches, aligned columns) of their arg-max path, so identity needs no
//     traceback;
//   * keep the alignment if forward + backward score >= gappedthresh.
//
// Schedule. Under spec D5 an extension depends only on its anchor, never on the alignments reported
// before it; only the SKIP decision is sequential. So the stage runs in rounds:
//   gp_select_kernel   one warp per tile walks the tile's anchors best-first as far as results exist
//                      (accept / skip exactly as the sequential rule says), then schedules extensions
//                      for anchors that are still undecided: the first undecided one, plus -- as
//                      speculation -- the best anchor of every other "cluster" of the chain (run of
//                      chain members with small gaps, which one alignment usually swallows whole);
//   gp_extend_kernel   one CTA per (anchor, direction), all tiles in one launch.
// Speculation changes which extensions are computed early, never the result: a speculative result is
// only used when the sequential walk reaches its anchor and finds it uncovered.
#include <algorithm>

#include "primitives.cuh"
#include "seq.cuh"
#include "internal.cuh"
#include "ydrop_warp.cuh"

namespace mb2 {

constexpr int GP_CLUSTER_GAP = 1000;     // chain members further apart than this (either axis) start a new speculation cluster

__device__ __forceinline__ int sub_lut3(uint32_t idx) {
    const uint64_t lo = 0xE183648E85E18E5Bull, hi = 0x5B8EE1858E6483E1ull;
    const uint64_t v = (idx & 8) ? hi : lo;
    return (int)(int8_t)(v >> ((idx & 7) * 8));
}

// ---- ordering of the chain members: per tile, score descending, then canonical (s1, s2)
__global__ void __launch_bounds__(256)
anchor_keys_kernel(const uint32_t* __restrict__ tile, const int32_t* __restrict__ score, const uint8_t* __restrict__ in_chain,
                   uint32_t n, uint64_t* __restrict__ key, uint32_t* __restrict__ idx, uint32_t* __restrict__ mflag) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    // non-members sort behind every real tile
    key[k] = in_chain[k] ? (((uint64_t)tile[k] << 31) | (uint64_t)(0x7fffffff - score[k])) : ~0ull;
    idx[k] = k;
    mflag[k] = in_chain[k] ? 1u : 0u;
}
__global__ void __launch_bounds__(256)
anchor_heads_kernel(const uint64_t* __restrict__ key, uint32_t n, uint32_t* __restrict__ flag) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const bool member = key[k] != ~0ull;
    flag[k] = (member && (k == 0 || (key[k] >> 31) != (key[k - 1] >> 31))) ? 1u : 0u;
}
__global__ void __launch_bounds__(256)
anchor_starts_kernel(const uint32_t* __restrict__ flag, const uint32_t* __restrict__ flag_off, uint32_t n, uint32_t* __restrict__ seg_start) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    if (flag[k]) seg_start[flag_off[k]] = k;
}
// speculation clusters over the members in canonical (= chain) order: mlist[r] = HSP index of the r-th member
__global__ void __launch_bounds__(256)
member_list_kernel(const uint32_t* __restrict__ mflag, const uint32_t* __restrict__ mrank, uint32_t n, uint32_t* __restrict__ mlist) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n || !mflag[k]) return;
    mlist[mrank[k]] = k;
}
__global__ void __launch_bounds__(256)
cluster_heads_kernel(const uint32_t* __restrict__ mlist, uint32_t nmember, const uint32_t* __restrict__ tile, const int32_t* __restrict__ hs1,
                     const int32_t* __restrict__ hs2, const int32_t* __restrict__ hlen, uint32_t* __restrict__ head) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nmember) return;
    uint32_t h = 1;
    if (r > 0) {
        const uint32_t g = mlist[r], pg = mlist[r - 1];
        const int g1 = hs1[g] - (hs1[pg] + hlen[pg]), g2 = hs2[g] - (hs2[pg] + hlen[pg]);
        h = (tile[g] != tile[pg] || g1 > GP_CLUSTER_GAP || g2 > GP_CLUSTER_GAP || g1 < -GP_CLUSTER_GAP || g2 < -GP_CLUSTER_GAP) ? 1u : 0u;
    }
    head[r] = h;
}
__global__ void __launch_bounds__(256)
cluster_ids_kernel(const uint32_t* __restrict__ mlist, uint32_t nmember, const uint32_t* __restrict__ head, const uint32_t* __restrict__ head_off,
                   uint32_t* __restrict__ cluster_of) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nmember) return;
    cluster_of[mlist[r]] = head_off[r] + head[r] - 1u;
}

struct Ext { int score, di, dj, nmatch, ncols; };

// Exact shortcut for the trivial alignment of a scaffold with itself. When target and query are the SAME N-free
// sequence and the anchor lies on the main diagonal, the y-drop DP has a closed form: every column (x,x) is a match
// scoring s(b,b) > 0, and any other path to an anti-diagonal k uses at most min(i,j) <= k/2 aligned columns, each
// worth at most s(b,b) of its row base, minus gap costs -- so the main-diagonal cell is the strict maximum of every
// even anti-diagonal, is never pruned, and the extension ends at the scaffold end with score = sum of s(b,b),
// matches = columns = length. (Proof in DESIGN.md; sequences with any non-ACGT base take the general DP.)
__device__ Ext selfdiag_extend_warp(const GenomeView& T, uint32_t p0, uint32_t p1) {
    // count C/G bases in padded-coordinate range [p0, p1): 2-bit code has exactly one bit set for C (01) and G (10)
    int cg = 0;
    if (p1 > p0) {
        const uint32_t w0 = p0 >> 5, w1 = (p1 - 1) >> 5;
        for (uint32_t w = w0 + (threadIdx.x & 31); w <= w1; w += 32) {
            uint64_t x = T.pk[w];
            uint64_t m = (x ^ (x >> 1)) & 0x5555555555555555ull;
            if (w == w0 && (p0 & 31)) m &= ~0ull << (2 * (p0 & 31));
            if (w == w1 && (p1 & 31)) m &= ~0ull >> (64 - 2 * (p1 & 31));
            cg += __popcll(m);
        }
    }
    const int tot = __reduce_add_sync(0xffffffffu, cg);
    const int n = (int)(p1 - p0);
    Ext r;
    r.score = 91 * (n - tot) + 100 * tot; r.di = n; r.dj = n; r.nmatch = n; r.ncols = n;
    return r;
}

// Anchors of all chain members at once (slot x = position in the (tile, score desc) order): centre of the best
// 31-column window of the HSP (first maximum), the whole HSP if it is shorter. One CTA per member; every thread slides a
// window over its own contiguous share of the window positions, then the CTA keeps the first maximum.
constexpr int AP_NT = 128;
constexpr int AP_LONG = 16384;       // HSPs with more windows than this are split over AP_PARTS CTAs (second kernel)
constexpr int AP_PARTS = 32;
constexpr int AP_LONG_SLOTS = 64;

// windows [w0, w1) of one HSP by one thread: best window sum and its first position (strict > keeps the first)
__device__ __forceinline__ void ap_scan(const GenomeView& T, const GenomeView& Q, uint32_t ts, uint32_t qs, int w0, int w1, int& best, int& bw) {
    // 32 column scores at a time from registers: words of 32 bases / 32 N flags starting at column c
    auto score_at = [](uint64_t wt, uint64_t wq, uint32_t an, int t) -> int {
        return ((an >> t) & 1u) ? SCORE_N : sub_lut3((uint32_t)(((wt >> (2 * t)) & 3) << 2) | (uint32_t)((wq >> (2 * t)) & 3));
    };
    best = INT_MIN; bw = INT_MAX;
    if (w0 >= w1) return;
    int sum = 0;
    {
        const uint64_t wt = window32(T.pk, ts + w0), wq = window32(Q.pk, qs + w0);
        const uint32_t an = nwindow32(T.nm, ts + w0) | nwindow32(Q.nm, qs + w0);
#pragma unroll
        for (int t = 0; t < 31; t++) sum += score_at(wt, wq, an, t);
    }
    best = sum; bw = w0;
    // window w = w0 + 1 + 32 b + t: column w + 30 enters, column w - 1 leaves
    for (int wb = w0 + 1; wb < w1; wb += 32) {
        const uint64_t et = window32(T.pk, ts + wb + 30), eq = window32(Q.pk, qs + wb + 30);
        const uint32_t en = nwindow32(T.nm, ts + wb + 30) | nwindow32(Q.nm, qs + wb + 30);
        const uint64_t lt = window32(T.pk, ts + wb - 1), lq = window32(Q.pk, qs + wb - 1);
        const uint32_t ln = nwindow32(T.nm, ts + wb - 1) | nwindow32(Q.nm, qs + wb - 1);
#pragma unroll
        for (int t = 0; t < 32; t++) {
            sum += score_at(et, eq, en, t) - score_at(lt, lq, ln, t);
            if (wb + t < w1 && sum > best) { best = sum; bw = wb + t; }
        }
    }
}
// first maximum over the CTA (highest sum, then lowest window); valid in thread 0
__device__ __forceinline__ void ap_reduce(int& best, int& bw, int* sh_best, int* sh_w) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int wbest = __reduce_max_sync(0xffffffffu, best);
    const int wbw = __reduce_min_sync(0xffffffffu, best == wbest ? bw : INT_MAX);
    if (lane == 0) { sh_best[warp] = wbest; sh_w[warp] = wbw; }
    __syncthreads();
    if (threadIdx.x == 0) {
        int b = sh_best[0], w = sh_w[0];
        for (int k = 1; k < AP_NT / 32; k++)
            if (sh_best[k] > b || (sh_best[k] == b && sh_w[k] < w)) { b = sh_best[k]; w = sh_w[k]; }
        best = b; bw = w;
    }
}
// (sum, window) packed so that "higher sum, then lower window" is plain unsigned max
__device__ __forceinline__ unsigned long long ap_pack(int sum, int w) {
    return ((unsigned long long)((uint32_t)sum ^ 0x80000000u) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)w);
}

__global__ void __launch_bounds__(AP_NT)
anchor_points_kernel(GenomeView T, GenomeView Q, const uint32_t* __restrict__ tile, const int32_t* __restrict__ hs1, const int32_t* __restrict__ hs2,
                     const int32_t* __restrict__ hlen, const uint32_t* __restrict__ order, uint32_t nmember,
                     int32_t* __restrict__ a1, int32_t* __restrict__ a2, uint32_t* __restrict__ long_list, uint32_t* __restrict__ nlong,
                     unsigned long long* __restrict__ long_key) {
    __shared__ int sh_best[AP_NT / 32], sh_w[AP_NT / 32];
    const int tid = threadIdx.x;
    const uint32_t x = blockIdx.x;
    const uint32_t g = order[x], tl = tile[g];
    const uint32_t ts = T.off[tl / (uint32_t)Q.nscaf] + (uint32_t)hs1[g], qs = Q.off[tl % (uint32_t)Q.nscaf] + (uint32_t)hs2[g];
    const int len = hlen[g];
    if (len <= 31) {
        if (tid == 0) { a1[x] = hs1[g] + len / 2; a2[x] = hs2[g] + len / 2; }
        return;
    }
    const int nwin = len - 30;                       // window w covers columns [w, w + 30]
    if (nwin > AP_LONG) {                            // split over several CTAs by anchor_points_long_kernel
        if (tid == 0) { const uint32_t k = atomicAdd(nlong, 1u); long_list[k] = x; long_key[k] = 0ull; }
        return;
    }
    const int chunk = (nwin + AP_NT - 1) / AP_NT;
    int best, bw;
    ap_scan(T, Q, ts, qs, tid * chunk, min(nwin, tid * chunk + chunk), best, bw);
    ap_reduce(best, bw, sh_best, sh_w);
    if (tid == 0) { a1[x] = hs1[g] + bw + 15; a2[x] = hs2[g] + bw + 15; }
}
// grid (AP_PARTS, AP_LONG_SLOTS): CTA (p, s) scans part p of the long HSPs s, s + AP_LONG_SLOTS, ...
__global__ void __launch_bounds__(AP_NT)
anchor_points_long_kernel(GenomeView T, GenomeView Q, const uint32_t* __restrict__ tile, const int32_t* __restrict__ hs1, const int32_t* __restrict__ hs2,
                          const int32_t* __restrict__ hlen, const uint32_t* __restrict__ order, const uint32_t* __restrict__ long_list,
                          const uint32_t* __restrict__ nlong, unsigned long long* __restrict__ long_key) {
    __shared__ int sh_best[AP_NT / 32], sh_w[AP_NT / 32];
    const int tid = threadIdx.x;
    const uint32_t n = *nlong;
    for (uint32_t k = blockIdx.y; k < n; k += gridDim.y) {
        const uint32_t x = long_list[k];
        const uint32_t g = order[x], tl = tile[g];
        const uint32_t ts = T.off[tl / (uint32_t)Q.nscaf] + (uint32_t)hs1[g], qs = Q.off[tl % (uint32_t)Q.nscaf] + (uint32_t)hs2[g];
        const int nwin = hlen[g] - 30;
        const int part = (nwin + AP_PARTS - 1) / AP_PARTS;
        const int p0 = (int)blockIdx.x * part, p1 = min(nwin, p0 + part);
        const int chunk = (max(p1 - p0, 0) + AP_NT - 1) / AP_NT;
        int best, bw;
        ap_scan(T, Q, ts, qs, p0 + tid * chunk, min(p1, p0 + tid * chunk + chunk), best, bw);
        ap_reduce(best, bw, sh_best, sh_w);
        if (tid == 0 && best != INT_MIN) atomicMax(&long_key[k], ap_pack(best, bw));
        __syncthreads();
    }
}
__global__ void __launch_bounds__(64)
anchor_points_finish_kernel(const int32_t* __restrict__ hs1, const int32_t* __restrict__ hs2, const uint32_t* __restrict__ order,
                            const uint32_t* __restrict__ long_list, const uint32_t* __restrict__ nlong,
                            const unsigned long long* __restrict__ long_key, int32_t* __restrict__ a1, int32_t* __restrict__ a2) {
    const uint32_t n = *nlong;
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        const uint32_t x = long_list[k], g = order[x];
        const int w = (int)(0xFFFFFFFFu - (uint32_t)(long_key[k] & 0xFFFFFFFFull));
        a1[x] = hs1[g] + w + 15; a2[x] = hs2[g] + w + 15;
    }
}

// Per (slot, direction) status of an extension.
enum : uint8_t { GX_NONE = 0, GX_NARROW = 1, GX_NEED_WIDE = 2, GX_WIDE = 3 };

struct GpWork {
    // per slot x (position in the (tile, score desc) order of the chain members)
    const uint32_t* order; const int32_t *a1, *a2; const uint32_t* cluster_of;
    uint8_t* status;                 // [2 * nmember]: slot * 2 + direction (0 forward, 1 backward)
    int32_t *e_score, *e_di, *e_dj, *e_nm, *e_nc;   // [2 * nmember] one-sided extension results
    uint32_t* stamp;                 // per cluster: last round that scheduled one of its members
    uint32_t *items_narrow, *items_wide, *items_full;   // work lists of this round: slot * 2 + direction
    uint32_t* counts;                // {narrow, wide, full rows (band wider than the wide kernel)}
};

constexpr int SEL_PEND = 64;         // pending (computed, not yet accepted) boxes a warp remembers while scheduling

// One warp per tile. Phase 1 replays the sequential rule as far as results exist; phase 2 schedules.
__global__ void __launch_bounds__(128)
gp_select_kernel(GpWork W, const uint32_t* __restrict__ tile, uint32_t nmember, const uint32_t* __restrict__ seg_start, uint32_t nseg,
                 uint32_t* __restrict__ resume, uint32_t* __restrict__ nkept_arr, uint32_t round, int gthr,
                 int32_t* __restrict__ o_s1, int32_t* __restrict__ o_e1, int32_t* __restrict__ o_s2, int32_t* __restrict__ o_e2,
                 int32_t* __restrict__ o_score, int32_t* __restrict__ o_nm, int32_t* __restrict__ o_nc, uint32_t* __restrict__ o_tile,
                 uint32_t* __restrict__ o_keep, unsigned long long* __restrict__ counters) {
    __shared__ int pend[128 / 32][SEL_PEND][4];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t seg = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (seg >= nseg) return;
    const uint32_t a = seg_start[seg];
    const uint32_t b = (seg + 1 < nseg) ? seg_start[seg + 1] : nmember;
    uint32_t x = a + resume[seg];
    uint32_t nk = nkept_arr[seg];
    if (x >= b) return;
    unsigned long long accepted = 0;
    auto covered = [&](int p1, int p2) -> bool {                 // spec D5: bounding-box test against reported alignments
        int cov = 0;
        for (uint32_t kk = lane; kk < nk; kk += 32)
            cov |= (p1 >= o_s1[a + kk] && p1 < o_e1[a + kk] && p2 >= o_s2[a + kk] && p2 < o_e2[a + kk]) ? 1 : 0;
        return __any_sync(0xffffffffu, cov);
    };
    auto ready = [&](uint32_t y) -> bool {
        const uint8_t f = W.status[2 * y], r = W.status[2 * y + 1];
        return (f == GX_NARROW || f == GX_WIDE) && (r == GX_NARROW || r == GX_WIDE);
    };
    // ---------------- phase 1: resolve in best-first order while results exist
    for (; x < b; x++) {
        const int p1 = W.a1[x], p2 = W.a2[x];
        if (covered(p1, p2)) continue;
        if (!ready(x)) break;
        accepted++;
        const int score = W.e_score[2 * x] + W.e_score[2 * x + 1];
        if (score >= gthr) {
            if (lane == 0) {
                const uint32_t o = a + nk;
                o_s1[o] = p1 - W.e_di[2 * x + 1]; o_e1[o] = p1 + W.e_di[2 * x]; o_s2[o] = p2 - W.e_dj[2 * x + 1]; o_e2[o] = p2 + W.e_dj[2 * x];
                o_score[o] = score; o_nm[o] = W.e_nm[2 * x] + W.e_nm[2 * x + 1]; o_nc[o] = W.e_nc[2 * x] + W.e_nc[2 * x + 1];
                o_tile[o] = tile[W.order[x]]; o_keep[o] = 1;
            }
            nk++;
            __syncwarp();
        }
    }
    if (lane == 0) {
        resume[seg] = x - a; nkept_arr[seg] = nk;
        if (accepted) atomicAdd(&counters[CNT_ANCHORS], accepted);
    }
    __syncwarp();
    if (x >= b) return;
    // ---------------- phase 2: schedule. Boxes of results that wait for their turn count as covered FOR SCHEDULING only.
    int npend = 0;
    for (uint32_t y0 = x; y0 < b; y0 += 32) {
        const uint32_t y = y0 + lane;
        const bool have = y < b && ready(y);
        const uint32_t m = __ballot_sync(0xffffffffu, have);
        if (have) {
            const int slot = npend + __popc(m & ((1u << lane) - 1u));
            if (slot < SEL_PEND) {
                const int p1 = W.a1[y], p2 = W.a2[y];
                pend[wib][slot][0] = p1 - W.e_di[2 * y + 1]; pend[wib][slot][1] = p1 + W.e_di[2 * y];
                pend[wib][slot][2] = p2 - W.e_dj[2 * y + 1]; pend[wib][slot][3] = p2 + W.e_dj[2 * y];
            }
        }
        npend = min(SEL_PEND, npend + __popc(m));
    }
    __syncwarp();
    for (uint32_t y = x; y < b; y++) {
        const uint8_t sf = W.status[2 * y], sr = W.status[2 * y + 1];
        const bool is_ready = (sf == GX_NARROW || sf == GX_WIDE) && (sr == GX_NARROW || sr == GX_WIDE);
        if (is_ready) continue;
        const uint32_t cl = W.cluster_of[W.order[y]];
        if (y != x && W.stamp[cl] == round) continue;             // one speculative extension per cluster and round
        const int p1 = W.a1[y], p2 = W.a2[y];
        if (y != x) {
            if (covered(p1, p2)) continue;                        // will be skipped when its turn comes
            int cov = 0;
            for (int kk = lane; kk < npend; kk += 32)
                cov |= (p1 >= pend[wib][kk][0] && p1 < pend[wib][kk][1] && p2 >= pend[wib][kk][2] && p2 < pend[wib][kk][3]) ? 1 : 0;
            if (__any_sync(0xffffffffu, cov)) continue;           // probably inside an alignment that is waiting for its turn
        }
        if (lane < 2) {
            const uint8_t s = lane == 0 ? sf : sr;
            if (s == GX_NONE) {
                W.items_narrow[atomicAdd(&W.counts[0], 1u)] = 2 * y + lane;
                W.status[2 * y + lane] = GX_NARROW;
            } else if (s == GX_NEED_WIDE) {
                W.items_wide[atomicAdd(&W.counts[1], 1u)] = 2 * y + lane;
                W.status[2 * y + lane] = GX_WIDE;
            }
        }
        if (lane == 0) W.stamp[cl] = round;
        __syncwarp();
    }
}

// ---- y-drop extension (ydrop_warp.cuh): one warp per work item = (anchor, direction)
constexpr int GP_WARPS_PER_SM = 24;  // most resident one-warp CTAs per SM of any variant of the extension kernel (sizes the scratch slots)
constexpr int ST_CLOSED = 100;       // ExtResult.status of an item answered by the closed form (no trace to walk back)

// Persistent grid of one-warp CTAs; items are handed out by an atomic counter. MAXS = 32: common kernel (bands up to 928
// diagonals); 64: wide bands (rerun of the few items the common kernel hands back).
template <int MAXS, int MINB>
__global__ void __launch_bounds__(32, MINB)
gp_forward_kernel(GenomeView T, GenomeView Q, GpWork W, const uint32_t* __restrict__ items, uint32_t nitems, uint32_t* __restrict__ next_item,
                  const uint32_t* __restrict__ tile, yw::Params prm, const int32_t* __restrict__ same_q, yw::Pool pool,
                  yw::ExtResult* __restrict__ res, unsigned long long* __restrict__ counters, uint32_t lay_mask) {
    const int lane = threadIdx.x;
    uint32_t priv_used = 0;                 // private trace chunks this warp slot has handed out in this launch
    for (;;) {
        uint32_t w = 0;
        if (lane == 0) w = atomicAdd(next_item, 1u);
        w = __shfl_sync(0xffffffffu, w, 0);
        if (w >= nitems) break;
        const uint32_t item = items[w];
        const uint32_t x = item >> 1, dir = item & 1u;
        const uint32_t tl = tile[W.order[x]];
        const uint32_t tsc = tl / (uint32_t)Q.nscaf, qsc = tl % (uint32_t)Q.nscaf;
        const uint32_t toff = T.off[tsc], qoff = Q.off[qsc];
        const int tlen = (int)T.len[tsc];
        const int a1 = W.a1[x], a2 = W.a2[x];
        if (same_q[tsc] == (int)qsc && a1 == a2 && T.nfree[tsc]) {
            const Ext r = dir == 0 ? selfdiag_extend_warp(T, toff + a1, toff + tlen) : selfdiag_extend_warp(T, toff, toff + a1);
            if (lane == 0) {
                W.e_score[item] = r.score; W.e_di[item] = r.di; W.e_dj[item] = r.dj; W.e_nm[item] = r.nmatch; W.e_nc[item] = r.ncols;
                res[item].status = ST_CLOSED;
            }
            continue;
        }
        yw::ydrop_forward_warp<MAXS>(T.codes, Q.codes, (int64_t)toff + a1, (int64_t)qoff + a2, dir == 0 ? +1 : -1, prm, pool, item, blockIdx.x,
                                     priv_used, &res[item], lay_mask);
        __syncwarp();
        if (lane == 0) {
            const yw::ExtResult r = res[item];
            atomicAdd(&counters[CNT_GAPPED_CELLS], (unsigned long long)r.cells);
            if (r.status == yw::ST_NOMEM) { W.status[item] = GX_NONE; atomicAdd(&counters[CNT_WORK], 1ull); }       // scheduled again next round
            else if (r.status == yw::ST_WIDE) W.status[item] = GX_NEED_WIDE;
            else if (r.status == yw::ST_BAND) W.items_full[atomicAdd(&W.counts[2], 1u)] = item;     // gp_full_kernel, same round
            else if (r.status != yw::ST_OK) atomicAdd(&counters[CNT_ERR], 1ull);
        }
    }
}

// walk-back of every traced item of the round: one warp per item (the traces of a round stay in the pool until the host
// resets it for the next round)
__global__ void __launch_bounds__(128)
gp_walk_kernel(GenomeView T, GenomeView Q, GpWork W, const uint32_t* __restrict__ items, uint32_t nitems, const uint32_t* __restrict__ tile,
               yw::Params prm, yw::Pool pool, yw::ExtResult* __restrict__ res, unsigned long long* __restrict__ counters) {
    __shared__ yw::WalkCache wc[4];
    const uint32_t w = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (w >= nitems) return;
    const uint32_t item = items[w];
    if (res[item].status != yw::ST_OK) return;
    const uint32_t x = item >> 1, dir = item & 1u;
    const uint32_t tl = tile[W.order[x]];
    const uint32_t tsc = tl / (uint32_t)Q.nscaf, qsc = tl % (uint32_t)Q.nscaf;
    const int64_t ta = (int64_t)T.off[tsc] + W.a1[x], qa = (int64_t)Q.off[qsc] + W.a2[x];
    yw::ydrop_walk_warp(T.codes, Q.codes, ta, qa, dir == 0 ? +1 : -1, prm, pool, &res[item], wc[threadIdx.x >> 5]);
    __syncwarp();
    if ((threadIdx.x & 31) == 0) {
        const yw::ExtResult r = res[item];
        W.e_score[item] = r.score; W.e_di[item] = r.di; W.e_dj[item] = r.dj; W.e_nm[item] = r.nmatch; W.e_nc[item] = r.ncols;
        if (r.status != yw::ST_OK) atomicAdd(&counters[CNT_ERR], 1ull);
    }
}

// the round's ST_BAND items (alive band wider than the wide kernel's 2048 diagonals): the spec's recurrence on full rows,
// one warp per item (yw::ydrop_full_warp); `rows` holds 3 * cap cells per warp
constexpr int GP_FULL_WARPS = 32;
constexpr int64_t GP_FULL_CAP = 1 << 16;
__global__ void __launch_bounds__(32)
gp_full_kernel(GenomeView T, GenomeView Q, GpWork W, uint32_t* __restrict__ next_item, const uint32_t* __restrict__ tile, yw::Params prm,
               yw::FullCell* __restrict__ rows, yw::ExtResult* __restrict__ res, unsigned long long* __restrict__ counters) {
    const int lane = threadIdx.x;
    const uint32_t nitems = W.counts[2];
    yw::FullCell* my = rows + (size_t)blockIdx.x * 3 * GP_FULL_CAP;
    for (;;) {
        uint32_t w = 0;
        if (lane == 0) w = atomicAdd(next_item, 1u);
        w = __shfl_sync(0xffffffffu, w, 0);
        if (w >= nitems) break;
        const uint32_t item = W.items_full[w];
        const uint32_t x = item >> 1, dir = item & 1u;
        const uint32_t tl = tile[W.order[x]];
        const uint32_t tsc = tl / (uint32_t)Q.nscaf, qsc = tl % (uint32_t)Q.nscaf;
        const int a1 = W.a1[x], a2 = W.a2[x];
        const int64_t tn = dir == 0 ? (int64_t)T.len[tsc] - a1 : a1, qn = dir == 0 ? (int64_t)Q.len[qsc] - a2 : a2;
        yw::ydrop_full_warp(T.codes, Q.codes, (int64_t)T.off[tsc] + a1, (int64_t)Q.off[qsc] + a2, dir == 0 ? +1 : -1, tn, qn, prm, my,
                            GP_FULL_CAP, &res[item]);
        __syncwarp();
        if (lane == 0) {
            const yw::ExtResult r = res[item];
            atomicAdd(&counters[CNT_GAPPED_CELLS], (unsigned long long)r.cells);
            W.e_score[item] = r.score; W.e_di[item] = r.di; W.e_dj[item] = r.dj; W.e_nm[item] = r.nmatch; W.e_nc[item] = r.ncols;
            if (r.status != yw::ST_OK) atomicAdd(&counters[CNT_ERR], 1ull);
        }
    }
}

// launch order of the round's items: the higher-scoring anchor first (long extensions start early, short ones fill the tail)
__global__ void __launch_bounds__(256)
gp_item_keys_kernel(GpWork W, const uint32_t* __restrict__ items, uint32_t nitems, const int32_t* __restrict__ hscore, uint32_t* __restrict__ key) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nitems) return;
    const int sc = hscore[W.order[items[k] >> 1]];
    key[k] = 0xffffffu - (uint32_t)min(sc, 0xffffff);
}

// Trace pool + re-layout scratch of the extension kernels: one device arena, grown on demand, kept between calls.
struct TraceArena {
    uint8_t* base = nullptr; yw::ChunkMeta* meta = nullptr; uint32_t* next = nullptr; int16_t* scratch = nullptr;
    size_t nchunks = 0; int nslots = 0;
};
static TraceArena g_trace;
// allowed layouts (diagonals per lane) as a bit mask, bit S/4
static uint32_t layout_mask(const char* env, const char* dflt) {
    const char* e = getenv(env);
    std::string v = (e && *e) ? e : dflt;
    uint32_t m = 0;
    size_t pos = 0;
    while (pos < v.size()) {
        const size_t c = v.find(',', pos);
        const int S = atoi(v.substr(pos, c == std::string::npos ? std::string::npos : c - pos).c_str());
        if (S == 8 || S == 12 || S == 16 || S == 20 || S == 24 || S == 32) m |= 1u << (S >> 2);
        if (c == std::string::npos) break;
        pos = c + 1;
    }
    return m ? m : (1u << 4) | (1u << 6) | (1u << 8);
}
void gapped_release_scratch() {
    if (g_trace.base) cudaFree(g_trace.base);
    if (g_trace.meta) cudaFree(g_trace.meta);
    if (g_trace.next) cudaFree(g_trace.next);
    if (g_trace.scratch) cudaFree(g_trace.scratch);
    g_trace = TraceArena();
}
static yw::Pool trace_pool(int nslots) {
    Ctx& cx = ctx();
    if (!g_trace.base) {
        size_t free_b = 0, total_b = 0;
        MB2_CUDA(cudaMemGetInfo(&free_b, &total_b));
        size_t want = (size_t)96 << 30;                                   // 2 bytes per evaluated DP cell of one round (capped at 45 % of the free memory)
        if (const char* e = getenv("MB2_TRACE_POOL_MB")) { const double v = atof(e); if (v > 0) want = (size_t)(v * 1048576.0); }
        want = std::min(want, free_b / 20 * 9);
        size_t nchunks = want / yw::CHUNK_BYTES / yw::NSUB * yw::NSUB;
        MB2_REQUIRE(nchunks >= (size_t)yw::NSUB, -3, "gapped stage: not enough device memory for the trace pool");
        MB2_CUDA(cudaStreamSynchronize(cx.stream));
        MB2_CUDA(cudaMalloc((void**)&g_trace.base, nchunks * yw::CHUNK_BYTES));
        MB2_CUDA(cudaMalloc((void**)&g_trace.meta, nchunks * sizeof(yw::ChunkMeta)));
        MB2_CUDA(cudaMalloc((void**)&g_trace.next, yw::NSUB * sizeof(uint32_t)));
        g_trace.nchunks = nchunks;
    }
    if (g_trace.nslots < nslots) {
        MB2_CUDA(cudaStreamSynchronize(cx.stream));
        if (g_trace.scratch) MB2_CUDA(cudaFree(g_trace.scratch));
        MB2_CUDA(cudaMalloc((void**)&g_trace.scratch, (size_t)nslots * 3 * yw::WIN * sizeof(int16_t)));
        g_trace.nslots = nslots;
    }
    yw::Pool p;
    p.base = g_trace.base; p.meta = g_trace.meta; p.next = g_trace.next; p.scratch = g_trace.scratch;
    // a third of the pool is private (one slice per resident warp: no atomics, reused by every extension of that warp), the
    // rest is shared by the extensions whose trace outgrows their slice (50 kbp alignments: ~80 MB each)
    p.priv = (uint32_t)(g_trace.nchunks / 3 / (size_t)nslots);
    p.shared0 = p.priv * (uint32_t)nslots;
    p.per_sub = (uint32_t)((g_trace.nchunks - p.shared0) / yw::NSUB);
    return p;
}

__global__ void __launch_bounds__(256)
aln_gather_kernel(const uint32_t* __restrict__ keep, const uint32_t* __restrict__ keep_off, uint32_t n,
                  const uint32_t* __restrict__ i_tile, const int32_t* __restrict__ i_s1, const int32_t* __restrict__ i_e1,
                  const int32_t* __restrict__ i_s2, const int32_t* __restrict__ i_e2, const int32_t* __restrict__ i_score,
                  const int32_t* __restrict__ i_nm, const int32_t* __restrict__ i_nc,
                  uint32_t* __restrict__ o_tile, int32_t* __restrict__ o_s1, int32_t* __restrict__ o_e1, int32_t* __restrict__ o_s2,
                  int32_t* __restrict__ o_e2, int32_t* __restrict__ o_score, int32_t* __restrict__ o_nm, int32_t* __restrict__ o_nc) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n || !keep[k]) return;
    const uint32_t o = keep_off[k];
    o_tile[o] = i_tile[k]; o_s1[o] = i_s1[k]; o_e1[o] = i_e1[k]; o_s2[o] = i_s2[k]; o_e2[o] = i_e2[k];
    o_score[o] = i_score[k]; o_nm[o] = i_nm[k]; o_nc[o] = i_nc[k];
}

// ungapped mode (--gapped off): every chain member becomes an alignment row; matches counted here
__global__ void __launch_bounds__(128)
ungapped_rows_kernel(GenomeView T, GenomeView Q, const uint32_t* __restrict__ tile, const int32_t* __restrict__ hs1,
                     const int32_t* __restrict__ hs2, const int32_t* __restrict__ hlen, const int32_t* __restrict__ hscore,
                     const uint8_t* __restrict__ in_chain, uint32_t n,
                     int32_t* __restrict__ o_s1, int32_t* __restrict__ o_e1, int32_t* __restrict__ o_s2, int32_t* __restrict__ o_e2,
                     int32_t* __restrict__ o_score, int32_t* __restrict__ o_nm, int32_t* __restrict__ o_nc, uint32_t* __restrict__ o_tile,
                     uint32_t* __restrict__ o_keep) {
    const int lane = threadIdx.x & 31;
    const uint32_t g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (g >= n || !in_chain[g]) return;
    const uint32_t tl = tile[g];
    const uint32_t ts = T.off[tl / (uint32_t)Q.nscaf] + hs1[g], qs = Q.off[tl % (uint32_t)Q.nscaf] + hs2[g];
    int nm = 0;
    for (int c = lane; c < hlen[g]; c += 32)
        nm += (!(isn_at(T.nm, ts + c) | isn_at(Q.nm, qs + c)) && base_at(T.pk, ts + c) == base_at(Q.pk, qs + c)) ? 1 : 0;
    nm = __reduce_add_sync(0xffffffffu, nm);
    if (lane == 0) {
        o_s1[g] = hs1[g]; o_e1[g] = hs1[g] + hlen[g]; o_s2[g] = hs2[g]; o_e2[g] = hs2[g] + hlen[g];
        o_score[g] = hscore[g]; o_nm[g] = nm; o_nc[g] = hlen[g]; o_tile[g] = tl; o_keep[g] = 1;
    }
}

void gapped_extend(const Genome& T, const Genome& Q, const HspSet& h, const DevBuf<uint8_t>& in_chain, const AlignParams& p,
                   const int32_t* h_same_q, AlnSet& out, unsigned long long* counters) {
    out.n = 0;
    const uint32_t n = h.n;
    if (n == 0) return;
    Ctx& cx = ctx();
    DevBuf<uint32_t> r_tile(n), keep(n), keep_off(n), d_nout(1);
    DevBuf<int32_t> r_s1(n), r_e1(n), r_s2(n), r_e2(n), r_score(n), r_nm(n), r_nc(n);
    MB2_CUDA(cudaMemsetAsync(keep.get(), 0, (size_t)n * sizeof(uint32_t), cx.stream));
    if (!p.gapped) {
        launch(ungapped_rows_kernel, cdiv((size_t)n * 32, 128), 128, 0, view(T), view(Q), h.tile.get(), h.s1.get(), h.s2.get(),
               h.len.get(), h.score.get(), in_chain.get(), n, r_s1.get(), r_e1.get(), r_s2.get(), r_e2.get(), r_score.get(),
               r_nm.get(), r_nc.get(), r_tile.get(), keep.get());
    } else {
        ProfScope ps("gapped");
        // order the chain members: (tile, score desc), stable over the canonical order
        int tb = 1; while (tb < 33 && (((uint64_t)T.nscaf * (uint64_t)Q.nscaf) >> tb)) tb++;
        DevBuf<uint64_t> k0(n), k1(n);
        DevBuf<uint32_t> i0(n), i1(n), mflag(n), mrank(n), d_nmember(1);
        launch(anchor_keys_kernel, cdiv(n, 256), 256, 0, h.tile.get(), h.score.get(), in_chain.get(), n, k0.get(), i0.get(), mflag.get());
        const int w = radix_sort_bits<uint64_t, uint32_t>(k0.get(), k1.get(), i0.get(), i1.get(), n, 0, std::min(64, tb + 31));
        const uint64_t* skey = w ? k1.get() : k0.get();
        const uint32_t* order = w ? i1.get() : i0.get();
        DevBuf<uint32_t> flag(n), flag_off(n), seg_start(n), d_nseg(1);
        launch(anchor_heads_kernel, cdiv(n, 256), 256, 0, skey, n, flag.get());
        exclusive_scan_u32(flag.get(), flag_off.get(), n, d_nseg.get());
        launch(anchor_starts_kernel, cdiv(n, 256), 256, 0, flag.get(), flag_off.get(), n, seg_start.get());
        exclusive_scan_u32(mflag.get(), mrank.get(), n, d_nmember.get());
        uint32_t h_nseg = 0, h_nmember = 0;
        MB2_CUDA(cudaMemcpyAsync(&h_nseg, d_nseg.get(), sizeof(uint32_t), cudaMemcpyDeviceToHost, cx.stream));
        MB2_CUDA(cudaMemcpyAsync(&h_nmember, d_nmember.get(), sizeof(uint32_t), cudaMemcpyDeviceToHost, cx.stream));
        // same_q[t] = query scaffold that is the identical sequence as target scaffold t (or -1): enables the closed form
        std::vector<int32_t> same(T.nscaf, -1);
        for (int t = 0; t < T.nscaf; t++) {
            if (h_same_q) same[t] = h_same_q[t];
            else if (Q.fwd_src_id != 0 && Q.fwd_src_id == T.id && t < Q.nfwd) same[t] = t;
        }
        DevBuf<int32_t> d_same(T.nscaf);
        MB2_CUDA(cudaMemcpyAsync(d_same.get(), same.data(), T.nscaf * sizeof(int32_t), cudaMemcpyHostToDevice, cx.stream));
        MB2_CUDA(cudaStreamSynchronize(cx.stream));
        if (h_nmember) {
            const uint32_t nm = h_nmember;
            // speculation clusters along the chains
            DevBuf<uint32_t> mlist(nm), chead(nm), chead_off(nm), cluster_of(n), stamp(nm);
            launch(member_list_kernel, cdiv(n, 256), 256, 0, mflag.get(), mrank.get(), n, mlist.get());
            launch(cluster_heads_kernel, cdiv(nm, 256), 256, 0, mlist.get(), nm, h.tile.get(), h.s1.get(), h.s2.get(), h.len.get(), chead.get());
            exclusive_scan_u32(chead.get(), chead_off.get(), nm);
            launch(cluster_ids_kernel, cdiv(nm, 256), 256, 0, mlist.get(), nm, chead.get(), chead_off.get(), cluster_of.get());
            MB2_CUDA(cudaMemsetAsync(stamp.get(), 0, (size_t)nm * sizeof(uint32_t), cx.stream));
            // anchors, per-slot state
            DevBuf<int32_t> a1(nm), a2(nm), e_score(2 * (size_t)nm), e_di(2 * (size_t)nm), e_dj(2 * (size_t)nm), e_nm(2 * (size_t)nm), e_nc(2 * (size_t)nm);
            DevBuf<uint8_t> status(2 * (size_t)nm);
            DevBuf<uint32_t> items_n(2 * (size_t)nm), items_w(2 * (size_t)nm), items_f(2 * (size_t)nm), counts(3), resume(h_nseg), nkept(h_nseg);
            MB2_CUDA(cudaMemsetAsync(status.get(), 0, 2 * (size_t)nm, cx.stream));
            MB2_CUDA(cudaMemsetAsync(resume.get(), 0, (size_t)h_nseg * sizeof(uint32_t), cx.stream));
            MB2_CUDA(cudaMemsetAsync(nkept.get(), 0, (size_t)h_nseg * sizeof(uint32_t), cx.stream));
            const GenomeView tv = view(T), qv = view(Q);
            DevBuf<uint32_t> long_list(nm), d_nlong(1);
            DevBuf<unsigned long long> long_key(nm);
            MB2_CUDA(cudaMemsetAsync(d_nlong.get(), 0, sizeof(uint32_t), cx.stream));
            launch(anchor_points_kernel, nm, AP_NT, 0, tv, qv, h.tile.get(), h.s1.get(), h.s2.get(), h.len.get(), order, nm,
                   a1.get(), a2.get(), long_list.get(), d_nlong.get(), long_key.get());
            launch(anchor_points_long_kernel, dim3(AP_PARTS, AP_LONG_SLOTS), AP_NT, 0, tv, qv, h.tile.get(), h.s1.get(), h.s2.get(), h.len.get(),
                   order, (const uint32_t*)long_list.get(), (const uint32_t*)d_nlong.get(), long_key.get());
            launch(anchor_points_finish_kernel, 4, 64, 0, h.s1.get(), h.s2.get(), order, (const uint32_t*)long_list.get(),
                   (const uint32_t*)d_nlong.get(), (const unsigned long long*)long_key.get(), a1.get(), a2.get());
            GpWork W;
            W.order = order; W.a1 = a1.get(); W.a2 = a2.get(); W.cluster_of = cluster_of.get(); W.status = status.get();
            W.e_score = e_score.get(); W.e_di = e_di.get(); W.e_dj = e_dj.get(); W.e_nm = e_nm.get(); W.e_nc = e_nc.get();
            W.stamp = stamp.get(); W.items_narrow = items_n.get(); W.items_wide = items_w.get(); W.items_full = items_f.get(); W.counts = counts.get();
            static const bool dbg = getenv("MB2_GP_DEBUG") != nullptr;
            cudaEvent_t ev0 = nullptr, ev1 = nullptr;
            if (dbg) { cudaEventCreate(&ev0); cudaEventCreate(&ev1); }
            MB2_REQUIRE(p.ydrop >= YDROP_MIN && p.ydrop <= YDROP_MAX && p.gap_open >= 0 && p.gap_open <= GAP_OPEN_MAX &&
                        p.gap_extend >= GAP_EXTEND_MIN && p.gap_extend <= GAP_EXTEND_MAX,
                        -2, "gapped stage: y-drop / gap penalties outside the range the 16-bit extension kernel supports");
            const yw::Params prm{p.gap_open, p.gap_extend, p.ydrop};
            const int nslots = cx.sm_count * GP_WARPS_PER_SM;
            const yw::Pool pool = trace_pool(nslots);
            yw::Pool pool_wide = pool;
            pool_wide.priv = 0;              // the wide-band kernel runs in the same round: its traces go to the shared part only
            DevBuf<yw::ExtResult> res(2 * (size_t)nm);
            DevBuf<uint32_t> next_item(3);
            DevBuf<yw::FullCell> full_rows;  // allocated by the first round that has an item for gp_full_kernel
            unsigned long long h_nomem_before = 0;
            uint32_t prev_sched = 0, conc = (uint32_t)nslots;      // items launched last round; CTAs (= concurrent extensions) allowed
            for (uint32_t round = 1;; round++) {
                MB2_CUDA(cudaMemsetAsync(counts.get(), 0, 3 * sizeof(uint32_t), cx.stream));
                launch(gp_select_kernel, cdiv((size_t)h_nseg * 32, 128), 128, 0, W, h.tile.get(), nm, seg_start.get(), h_nseg, resume.get(), nkept.get(),
                       round, p.gappedthresh, r_s1.get(), r_e1.get(), r_s2.get(), r_e2.get(), r_score.get(), r_nm.get(), r_nc.get(), r_tile.get(),
                       keep.get(), counters);
                uint32_t h_counts[2] = {0, 0};
                unsigned long long h_nomem = 0;
                MB2_CUDA(cudaMemcpyAsync(h_counts, counts.get(), sizeof(h_counts), cudaMemcpyDeviceToHost, cx.stream));
                MB2_CUDA(cudaMemcpyAsync(&h_nomem, counters + CNT_WORK, sizeof(h_nomem), cudaMemcpyDeviceToHost, cx.stream));
                MB2_CUDA(cudaStreamSynchronize(cx.stream));
                if (dbg) {
                    float ms = 0;
                    if (round > 1) { cudaEventSynchronize(ev1); cudaEventElapsedTime(&ms, ev0, ev1); }
                    fprintf(stderr, "[gapped] members %u tiles %u | extend of round %u took %.3f ms (%llu items deferred: trace pool full) | round %u schedules %u + wide %u\n",
                            nm, h_nseg, round - 1, ms, h_nomem - h_nomem_before, round, h_counts[0], h_counts[1]);
                    cudaEventRecord(ev0, cx.stream);
                }
                if (h_counts[0] == 0 && h_counts[1] == 0) break;
                // items that ran out of trace pool were put back; if NONE of the previous round finished, one extension alone
                // does not fit the pool. Otherwise run fewer extensions at a time: as many as finished last round.
                const unsigned long long deferred = h_nomem - h_nomem_before;
                MB2_REQUIRE(deferred == 0 || deferred < prev_sched || conc > 1, -3,
                            "gapped stage: the trace pool is too small for a single extension (raise MB2_TRACE_POOL_MB)");
                // Deferred items are normal (a round's traces fill the pool, the rest fail fast and come back). Only when NOT ONE
                // extension of a round finished were the extensions in flight too long to fit side by side: run fewer at a time.
                if (prev_sched && deferred >= prev_sched) conc = std::max<uint32_t>(1, conc / 2);
                prev_sched = h_counts[0] + h_counts[1];
                h_nomem_before = h_nomem;
                MB2_CUDA(cudaMemsetAsync(pool.next, 0, yw::NSUB * sizeof(uint32_t), cx.stream));      // previous round's traces are consumed
                MB2_CUDA(cudaMemsetAsync(next_item.get(), 0, 3 * sizeof(uint32_t), cx.stream));
                static const uint32_t lay_narrow = layout_mask("MB2_GP_LAYOUTS", "16,24,32"), lay_wide = lay_narrow | (1u << 12) | (1u << 16);
                static const bool sort_items = !getenv("MB2_GP_NOSORT");
                static const int occ = getenv("MB2_GP_OCC") ? atoi(getenv("MB2_GP_OCC")) : 16;
                const uint32_t* it_n = items_n.get();
                DevBuf<uint32_t> sk0, sk1, si1;
                if (sort_items && h_counts[0] > (uint32_t)nslots) {
                    sk0.alloc(h_counts[0]); sk1.alloc(h_counts[0]); si1.alloc(h_counts[0]);
                    launch(gp_item_keys_kernel, cdiv(h_counts[0], 256), 256, 0, W, (const uint32_t*)items_n.get(), h_counts[0], (const int32_t*)h.score.get(), sk0.get());
                    const int w = radix_sort_bits<uint32_t, uint32_t>(sk0.get(), sk1.get(), items_n.get(), si1.get(), h_counts[0], 8, 24);
                    it_n = w ? si1.get() : items_n.get();
                }
                {
                    ProfScope pf("gp_forward");
                    if (h_counts[0]) {
                        auto go = [&](auto kern, int per_sm) {
                            launch(kern, std::min<uint32_t>(h_counts[0], std::min<uint32_t>(conc, (uint32_t)(cx.sm_count * per_sm))), 32, 0, tv, qv, W, it_n, h_counts[0],
                                   next_item.get(), h.tile.get(), prm, d_same.get(), pool, res.get(), counters, lay_narrow);
                        };
                        if (occ >= 20) go(gp_forward_kernel<32, 20>, 20);
                        else go(gp_forward_kernel<32, 16>, 16);
                    }
                    if (h_counts[1]) {
                        launch(gp_forward_kernel<64, 4>, std::min<uint32_t>(h_counts[1], std::min<uint32_t>(conc, (uint32_t)(cx.sm_count * 4))), 32, 0, tv, qv, W, (const uint32_t*)items_w.get(), h_counts[1],
                               next_item.get() + 1, h.tile.get(), prm, d_same.get(), pool_wide, res.get(), counters, lay_wide);
                    }
                }
                {
                    ProfScope pw("gp_walk");
                    if (h_counts[0]) launch(gp_walk_kernel, cdiv(h_counts[0], 4), 128, 0, tv, qv, W, it_n, h_counts[0], h.tile.get(), prm, pool, res.get(), counters);
                    if (h_counts[1]) launch(gp_walk_kernel, cdiv(h_counts[1], 4), 128, 0, tv, qv, W, (const uint32_t*)items_w.get(), h_counts[1], h.tile.get(), prm, pool, res.get(), counters);
                }
                if (h_counts[1]) {                 // only the wide kernel hands out ST_BAND items; rounds with wide items are rare
                    uint32_t h_full = 0;
                    MB2_CUDA(cudaMemcpyAsync(&h_full, counts.get() + 2, sizeof(uint32_t), cudaMemcpyDeviceToHost, cx.stream));
                    MB2_CUDA(cudaStreamSynchronize(cx.stream));
                    if (h_full) {
                        ProfScope pfull("gp_full");
                        if (!full_rows.get()) full_rows.alloc((size_t)GP_FULL_WARPS * 3 * GP_FULL_CAP);
                        launch(gp_full_kernel, std::min<uint32_t>(h_full, GP_FULL_WARPS), 32, 0, tv, qv, W, next_item.get() + 2, h.tile.get(), prm,
                               full_rows.get(), res.get(), counters);
                    }
                }
                if (dbg) cudaEventRecord(ev1, cx.stream);
            }
            if (dbg) { cudaEventDestroy(ev0); cudaEventDestroy(ev1); }
        }
    }
    exclusive_scan_u32(keep.get(), keep_off.get(), n, d_nout.get());
    uint32_t h_nout = 0; unsigned long long h_err = 0;
    MB2_CUDA(cudaMemcpyAsync(&h_nout, d_nout.get(), sizeof(uint32_t), cudaMemcpyDeviceToHost, cx.stream));
    MB2_CUDA(cudaMemcpyAsync(&h_err, counters + CNT_ERR, sizeof(h_err), cudaMemcpyDeviceToHost, cx.stream));
    MB2_CUDA(cudaStreamSynchronize(cx.stream));
    MB2_REQUIRE(h_err == 0, -5, "gapped stage: an extension failed (an anti-diagonal wider than 65536 cells, or an inconsistent trace)");
    out.n = h_nout;
    if (h_nout == 0) return;
    out.tile.alloc(h_nout); out.s1.alloc(h_nout); out.e1.alloc(h_nout); out.s2.alloc(h_nout); out.e2.alloc(h_nout);
    out.score.alloc(h_nout); out.nmatch.alloc(h_nout); out.ncols.alloc(h_nout);
    launch(aln_gather_kernel, cdiv(n, 256), 256, 0, keep.get(), keep_off.get(), n, r_tile.get(), r_s1.get(), r_e1.get(), r_s2.get(),
           r_e2.get(), r_score.get(), r_nm.get(), r_nc.get(), out.tile.get(), out.s1.get(), out.e1.get(), out.s2.get(), out.e2.get(),
           out.score.get(), out.nmatch.get(), out.ncols.get());
}

}  // namespace mb2
