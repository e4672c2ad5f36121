// seq.cuh -- device genome layout and sequence access helpers.
//
// A genome is one concatenated coordinate space. Every scaffold starts at a multiple of 64 bases
// and is surrounded by at least 64 pad bases (2048 at both ends of the genome) that are flagged non-ACGT, so that
//   * a 19-mer seed window can never span two scaffolds,
//   * gap-free x-drop extension needs no bounds checks: a pad column scores -100 like any
//     non-ACGT character, so the 64 columns of the narrowest pad lose 6400 and end every extension whose
//     x-drop is below that (GF_MAX_XDROP) without changing its maximum,
//   * unaligned 64-bit window reads one word past a scaffold are always in bounds.
// Storage: pk  = 2 bits/base, 32 bases per uint64 word, base p in bits [2(p%32), 2(p%32)+1];
//          nm  = 1 bit/base, 32 bases per uint32 word, 1 = not A/C/G/T (N, IUPAC, pad): scores -100 in every extension;
//          sm  = nm | soft-mask: lower-case input is excluded from SEEDING on both sequences, as LASTZ does without
//                [unmask] (a 19-mer window holding such a base is no seed word), but is extended through by its base;
//          nb  = 4 bits/base, 8 bases per uint32 word, base p in bits [4(p%8), 4(p%8)+3]: base | parity << 2 (parity = C or G)
//                for A/C/G/T, 8 for anything else (N, IUPAC, pad). The seed scan merges a target and a query word of it into one
//                code per column (seed.cu: nib_merge) that indexes its x-drop table directly.
#pragma once
#include "common.cuh"

namespace mb2 {

constexpr int SEED_SPAN = 19;
constexpr uint32_t GENOME_PAD = 64;       // between scaffolds
constexpr uint32_t GENOME_END_PAD = 2048;  // before the first and after the last scaffold: wide x-drop steps read 1024 columns ahead

struct Genome {
    int nscaf = 0;
    std::vector<uint32_t> off, len;   // host copies: scaffold start (padded coords) and length
    uint64_t G = 0;                   // padded total length, multiple of 64
    uint64_t nbases = 0;              // sum of scaffold lengths
    DevBuf<uint64_t> pk;              // G/32 + 2 words
    DevBuf<uint32_t> nm;              // G/32 + 2 words
    DevBuf<uint32_t> sm;              // G/32 + 2 words: 1 = not seedable (non-ACGT, pad, or soft-masked = lower case in the input)
    bool has_soft = false;            // false: no lower-case base anywhere, sm == nm bit for bit and kernels are handed nm (one plane to gather from)
    DevBuf<uint32_t> nb;              // G/8 + 8 words: 4-bit codes (see above)
    DevBuf<uint8_t> codes;            // 1 byte/base for the gapped DP: base | parity << 2, 8 = other, 12 = pad (genome.cu:code_byte)
    DevBuf<uint32_t> d_off, d_len;
    DevBuf<uint32_t> d_nfree;         // per scaffold: 1 = every base is A/C/G/T
    bool is_rc = false;
    // identity bookkeeping for the trivial self-alignment shortcut: scaffolds [0, nfwd) of this genome are byte-identical
    // to the scaffolds of the genome whose id is fwd_src_id (a genome is its own source)
    uint64_t id = 0, fwd_src_id = 0;
    int nfwd = 0;
};
uint64_t next_genome_id();

struct GenomeView {   // what kernels receive
    const uint64_t* __restrict__ pk;
    const uint32_t* __restrict__ nm;
    const uint32_t* __restrict__ sm;
    const uint32_t* __restrict__ nb;
    const uint8_t* __restrict__ codes;
    const uint32_t* __restrict__ off;
    const uint32_t* __restrict__ len;
    const uint32_t* __restrict__ nfree;
    int nscaf;
    uint32_t G;
};
inline GenomeView view(const Genome& g) { return GenomeView{g.pk.get(), g.nm.get(), g.has_soft ? g.sm.get() : g.nm.get(), g.nb.get(), g.codes.get(), g.d_off.get(), g.d_len.get(), g.d_nfree.get(), g.nscaf, (uint32_t)g.G}; }

// HOXD70 as LASTZ's default, row = target base, col = query base (index t*4+q)
static __constant__ int c_sub[16] = {91, -114, -31, -123, -114, 100, -125, -31, -31, -125, 100, -114, -123, -31, -114, 91};
constexpr int SCORE_N = -100;
// largest x-drop a gap-free extension may use: with 6400 or more it could walk through a 64-column pad into the next scaffold
constexpr int GF_MAX_XDROP = -SCORE_N * (int)GENOME_PAD - 1;

__device__ __forceinline__ uint32_t base_at(const uint64_t* __restrict__ pk, uint32_t p) {
    return (uint32_t)(pk[p >> 5] >> ((p & 31) * 2)) & 3u;
}
__device__ __forceinline__ uint32_t isn_at(const uint32_t* __restrict__ nm, uint32_t p) {
    return (nm[p >> 5] >> (p & 31)) & 1u;
}
// 32 bases starting at p (unaligned), base p+c in bits [2c, 2c+1]
__device__ __forceinline__ uint64_t window32(const uint64_t* __restrict__ pk, uint32_t p) {
    const uint32_t w = p >> 5, s = (p & 31) * 2;
    const uint64_t lo = pk[w];
    if (s == 0) return lo;
    return (lo >> s) | (pk[w + 1] << (64 - s));
}
// 32 N-flags starting at p
__device__ __forceinline__ uint32_t nwindow32(const uint32_t* __restrict__ nm, uint32_t p) {
    const uint32_t w = p >> 5, s = p & 31;
    return __funnelshift_r(nm[w], nm[w + 1], s);
}
// 32 bases ENDING at p (inclusive), base p-c in bits [2c, 2c+1] (i.e. reversed order) is awkward to build;
// leftward walks instead fetch the aligned window that contains p and index into it.

// nb code of one base (see above)
__device__ __forceinline__ uint32_t nib_code(uint32_t base, uint32_t bad) {
    return bad ? 8u : (base | (((base ^ (base >> 1)) & 1u) << 2));
}

__device__ __forceinline__ int sub_score(uint32_t tb, uint32_t qb, uint32_t anyn) {
    return anyn ? SCORE_N : c_sub[(tb << 2) | qb];
}

// 12-of-19 spaced seed 1110100110010101111: care offsets {0,1,2,4,7,8,11,13,15,16,17,18}
constexpr uint32_t SEED_WINDOW_MASK19 = (1u << SEED_SPAN) - 1u;

__device__ __forceinline__ uint32_t seed_key(uint64_t w) {
    return (uint32_t)(w & 0x3F) | ((uint32_t)(w >> 8) & 3u) << 6 | ((uint32_t)(w >> 14) & 0xFu) << 8 |
           ((uint32_t)(w >> 22) & 3u) << 12 | ((uint32_t)(w >> 26) & 3u) << 14 | ((uint32_t)(w >> 30) & 0xFFu) << 16;
}
}  // namespace mb2
