// xdrop_table.cuh -- exact gap-free x-drop at three columns per shared-memory table lookup (used by the thread-per-diagonal
// HSP extension of hsp.cu; the first-stage filter of seed.cu has a table of the same size indexed by merged 4-bit codes).
//
// Entry for target bases t0 t1 t2 / query bases q0 q1 q2 (index = q6 << 6 | t6, first column in the low bits; the shared-memory
// bank comes from the TARGET bases: the 32 hits of a seed-scan batch mostly share one query position, so with the query bits in
// the bank they collided 7.75 ways per lookup (ncu, profiles/r2_seed_scan_c4_ncu_summary.txt)):
//   bits 22..31 = s0+s1+s2 (signed), bits 18..19 = index (0..2) of the FIRST column that reaches the maximum prefix sum,
//   bits 9..17 = 125 + max prefix sum, bits 0..8 = 375 + min prefix sum.
// Exactness of the chunked rule: prefix sums inside a chunk differ by at most 2*125 < xdrop (callers require
// xdrop > 250), so a column can only terminate the extension against the maximum reached BEFORE the chunk; hence
// "terminates in this chunk" is run + min_prefix < best - X (and then no column of the chunk has raised best),
// otherwise best = max(best, run + max_prefix), first reached at the recorded column.
// The state is kept as (best, D) with D = (best - run) + 375 - X, the deficit to the running maximum in the bias of the
// min-prefix field, so a chunk is: terminate iff min_field < D; DM = max(D, max_field + 250 - X); best += DM - D;
// D = DM - sum.
#pragma once
#include "seq.cuh"

namespace mb2 {

constexpr int XT_SIZE = 4096;
constexpr int XT_MIN_XDROP = 251;

// 16 HOXD70 scores as int8 in two 64-bit registers, index t*4+q
__device__ __forceinline__ int sub_lut(uint32_t idx) {
    // {91,-114,-31,-123, -114,100,-125,-31} , {-31,-125,100,-114, -123,-31,-114,91}
    const uint64_t lo = 0xE183648E85E18E5Bull, hi = 0x5B8EE1858E6483E1ull;
    const uint64_t v = (idx & 8) ? hi : lo;
    return (int)(int8_t)(v >> ((idx & 7) * 8));
}

__device__ __forceinline__ uint32_t xt_entry(uint32_t idx) {
    const uint32_t q6 = idx >> 6, t6 = idx & 63;
    int sum = 0, mx = INT_MIN, mn = INT_MAX, at = 0;
    for (int c = 0; c < 3; c++) {
        sum += sub_lut((((t6 >> (2 * c)) & 3u) << 2) | ((q6 >> (2 * c)) & 3u));
        if (sum > mx) { mx = sum; at = c; }
        mn = min(mn, sum);
    }
    return ((uint32_t)sum << 22) | ((uint32_t)at << 18) | ((uint32_t)(mx + 125) << 9) | (uint32_t)(mn + 375);
}
__device__ __forceinline__ int xt_sum(uint32_t e) { return (int)e >> 22; }
__device__ __forceinline__ int xt_argmax(uint32_t e) { return (int)((e >> 18) & 3u); }
__device__ __forceinline__ int xt_maxf(uint32_t e) { return (int)((e >> 9) & 511u); }
__device__ __forceinline__ int xt_minf(uint32_t e) { return (int)(e & 511u); }

// reverse the order of the 32 two-bit groups of a word
__device__ __forceinline__ uint64_t rev2groups(uint64_t x) {
    x = __brevll(x);
    return ((x & 0xAAAAAAAAAAAAAAAAull) >> 1) | ((x & 0x5555555555555555ull) << 1);
}
// table index of chunk k (columns 3k..3k+2) of two 32-base windows; k is a compile-time constant after unrolling
__device__ __forceinline__ uint32_t xt_index(uint32_t tl, uint32_t th, uint32_t ql, uint32_t qh, int k) {
    const int sh = 6 * k;
    uint32_t t6, q6;
    if (sh + 6 <= 32) { t6 = (tl >> sh) & 63u; q6 = (ql >> sh) & 63u; }
    else if (sh >= 32) { t6 = (th >> (sh - 32)) & 63u; q6 = (qh >> (sh - 32)) & 63u; }
    else { t6 = __funnelshift_r(tl, th, sh) & 63u; q6 = __funnelshift_r(ql, qh, sh) & 63u; }
    return (q6 << 6) | t6;
}

}  // namespace mb2
