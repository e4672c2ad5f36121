// align.cu -- host driver of the alignment half: target table -> seed scan -> HSPs -> chain -> gapped.
//
// The target genome is indexed once; the (strand-oriented) query genome is processed in chunks of whole scaffolds so
// that the survivor / HSP buffers stay bounded no matter how repeat-rich the input is. A chunk never splits a query
// scaffold, so every (target scaffold, query scaffold, strand) tile -- the scope of LASTZ's --chain and of the gapped
// stage -- is complete inside one chunk and the results are identical to a single pass (tests/test_gpu_align.py forces
// tiny chunks and compares). Chunk size: MB2_CHUNK_MBP (default 128 Mbp of query per chunk).
#include <algorithm>
#include <cstdlib>

#include "primitives.cuh"
#include "seq.cuh"
#include "internal.cuh"

namespace mb2 {

static const uint64_t MAX_SURVIVORS = 1500000000ull;   // 12 GB of keys (x2 for the sort ping-pong)

struct QChunk { int s_lo, s_hi; };   // query scaffolds [s_lo, s_hi)

static uint64_t default_chunk_bases() {
    uint64_t chunk_bases = 128ull << 20;
    if (const char* e = getenv("MB2_CHUNK_MBP")) { const double v = atof(e); if (v > 0) chunk_bases = (uint64_t)(v * 1e6); }
    return chunk_bases;
}
// the next chunk: whole scaffolds from s_lo on, at most `limit` bases (but at least one scaffold)
static QChunk next_chunk(const Genome& Q, int s_lo, uint64_t limit) {
    uint64_t acc = 0;
    int s = s_lo;
    while (s < Q.nscaf && (s == s_lo || acc + Q.len[s] <= limit)) { acc += Q.len[s]; s++; }
    return {s_lo, s};
}

// query position range of scaffolds [s_lo, s_hi): from the first base of s_lo to the last base of s_hi-1 (windows that
// start in the pad are invalid by construction)
static void chunk_range(const Genome& Q, const QChunk& c, uint32_t& q_lo, uint32_t& q_hi) {
    q_lo = Q.off[c.s_lo];
    q_hi = Q.off[c.s_hi - 1] + Q.len[c.s_hi - 1];
}

// Seed scan of one chunk into a survivor buffer; grows the buffer once if it overflowed; returns false if the chunk must
// be split because even MAX_SURVIVORS is not enough.
static bool scan_chunk(const Genome& T, const Genome& Q, const SeedTable& tab, uint32_t q_lo, uint32_t q_hi, const AlignParams& p,
                       DevBuf<uint64_t>& s0, uint64_t& cap, unsigned long long* counters, unsigned long long& nsurv,
                       unsigned long long* stat_acc) {
    Ctx& cx = ctx();
    for (int attempt = 0; attempt < 2; attempt++) {
        if (s0.n < cap) s0.alloc(cap);
        MB2_CUDA(cudaMemsetAsync(counters, 0, 4 * sizeof(unsigned long long), cx.stream));
        MB2_CUDA(cudaMemsetAsync(counters + CNT_WORK, 0, sizeof(unsigned long long), cx.stream));      // the scan's round dispenser
        seed_scan(T, Q, tab, q_lo, q_hi, p, s0.get(), (uint32_t)std::min<uint64_t>(cap, 0xffffffffull), counters);
        unsigned long long h[4];
        MB2_CUDA(cudaMemcpyAsync(h, counters, sizeof(h), cudaMemcpyDeviceToHost, cx.stream));
        MB2_CUDA(cudaStreamSynchronize(cx.stream));
        nsurv = h[CNT_SURV];
        if (nsurv <= cap) {
            stat_acc[CNT_SURV] += h[CNT_SURV]; stat_acc[CNT_SEED_HITS] += h[CNT_SEED_HITS];
            stat_acc[CNT_LEADERS] += h[CNT_LEADERS]; stat_acc[CNT_S1_CELLS] += h[CNT_S1_CELLS];
            return true;
        }
        if (nsurv > MAX_SURVIVORS) return false;
        cap = nsurv;
    }
    return false;
}

std::vector<int32_t> same_scaffold_map(const Genome& T, const Genome& Q, const int32_t* h_same_q) {
    std::vector<int32_t> same(T.nscaf, -1);
    for (int t = 0; t < T.nscaf; t++) {
        if (h_same_q) same[t] = h_same_q[t];
        else if (Q.fwd_src_id != 0 && Q.fwd_src_id == T.id && t < Q.nfwd) same[t] = t;
    }
    return same;
}

// Test hook (stage a+b only): kept HSPs of every tile of T x Q in canonical order, single chunk.
void align_hsps(const Genome& T, const Genome& Q, const AlignParams& p, HspSet& hsps, unsigned long long* h_counters) {
    Ctx& cx = ctx();
    MB2_REQUIRE(T.G + Q.G < 0xffffffffull, -3, "align: target + query exceed 2^32 padded positions");
    DevBuf<unsigned long long> counters(CNT_N);
    MB2_CUDA(cudaMemsetAsync(counters.get(), 0, CNT_N * sizeof(unsigned long long), cx.stream));
    SeedTable tab;
    build_seed_table(T, 0, (uint32_t)T.G, tab);
    uint64_t cap = std::max<uint64_t>(1u << 20, (T.nbases + Q.nbases) / 2);
    DevBuf<uint64_t> s0, s1;
    unsigned long long nsurv = 0, acc[CNT_N] = {0};
    const bool ok = scan_chunk(T, Q, tab, GENOME_END_PAD, (uint32_t)Q.G - GENOME_END_PAD, p, s0, cap, counters.get(), nsurv, acc);
    MB2_REQUIRE(ok, -3, "align: too many surviving seed hits for one pass");
    s1.alloc(nsurv ? nsurv : 1);
    const std::vector<int32_t> same = same_scaffold_map(T, Q, nullptr);
    DevBuf<int32_t> d_same(T.nscaf);
    MB2_CUDA(cudaMemcpyAsync(d_same.get(), same.data(), T.nscaf * sizeof(int32_t), cudaMemcpyHostToDevice, cx.stream));
    MB2_CUDA(cudaStreamSynchronize(cx.stream));
    find_hsps(T, Q, s0.get(), s1.get(), (uint32_t)nsurv, p, hsps, counters.get(), d_same.get());
    if (h_counters) {
        MB2_CUDA(cudaMemcpyAsync(h_counters, counters.get(), CNT_N * sizeof(unsigned long long), cudaMemcpyDeviceToHost, cx.stream));
        MB2_CUDA(cudaStreamSynchronize(cx.stream));
        for (int k = 0; k < 4; k++) h_counters[k] = acc[k];
    }
}

// Test hook (stage a only): the survivors of one scan of the whole query, through scan_chunk (and so through its overflow and
// rescan when init_cap is too small). The query range is that of align_strand's chunks: first to last base.
void scan_survivors(const Genome& T, const Genome& Q, const AlignParams& p, uint64_t init_cap, std::vector<uint64_t>& surv,
                    unsigned long long* h_counters) {
    Ctx& cx = ctx();
    MB2_REQUIRE(T.G + Q.G < 0xffffffffull, -3, "scan: target + query exceed 2^32 padded positions");
    DevBuf<unsigned long long> counters(CNT_N);
    SeedTable tab;
    build_seed_table(T, 0, (uint32_t)T.G, tab);
    uint64_t cap = init_cap ? init_cap : std::max<uint64_t>(1u << 20, (T.nbases + Q.nbases) / 2);
    DevBuf<uint64_t> s0;
    unsigned long long nsurv = 0, acc[CNT_N] = {0};
    uint32_t q_lo, q_hi;
    chunk_range(Q, QChunk{0, Q.nscaf}, q_lo, q_hi);
    const bool ok = scan_chunk(T, Q, tab, q_lo, q_hi, p, s0, cap, counters.get(), nsurv, acc);
    MB2_REQUIRE(ok, -3, "scan: too many surviving seed hits for one pass");
    surv.resize(nsurv);
    if (nsurv) MB2_CUDA(cudaMemcpyAsync(surv.data(), s0.get(), nsurv * sizeof(uint64_t), cudaMemcpyDeviceToHost, cx.stream));
    MB2_CUDA(cudaStreamSynchronize(cx.stream));
    for (int k = 0; k < 4; k++) h_counters[k] = acc[k];
}

// Full pipeline for one strand-oriented query genome; the alignments of every query chunk are appended to the device hit
// table `out` in LASTZ's output columns.
void align_strand(const Genome& T, const Genome& Q, const AlignParams& p, const int32_t* h_same_q, DevHits& out, int nq, int strands,
                  unsigned long long* h_counters) {
    Ctx& cx = ctx();
    MB2_REQUIRE(T.G + Q.G < 0xffffffffull, -3, "align: target + query exceed 2^32 padded positions");
    // tile ids (target scaffold * query scaffolds + query scaffold) are 32-bit throughout the stage
    MB2_REQUIRE((uint64_t)T.nscaf * (uint64_t)Q.nscaf < (1ull << 32), -3,
                "align: target scaffolds x query scaffolds (both strands) must stay below 2^32 tiles; align the target in scaffold groups");
    unsigned long long acc[CNT_N] = {0};
    uint32_t maxlen = 0;
    for (int s = 0; s < T.nscaf; s++) maxlen = std::max(maxlen, T.len[s]);
    for (int s = 0; s < Q.nscaf; s++) maxlen = std::max(maxlen, Q.len[s]);
    int lb = 1; while (lb < 32 && (maxlen >> lb)) lb++;
    lb += 1;   // e = s + len can reach maxlen exactly
    int tb = 1; while (tb < 33 && (((uint64_t)T.nscaf * (uint64_t)Q.nscaf) >> tb)) tb++;

    SeedTable tab;
    build_seed_table(T, 0, (uint32_t)T.G, tab);
    DevBuf<unsigned long long> counters(CNT_N);
    DevBuf<uint64_t> s0, s1;
    const std::vector<int32_t> same = same_scaffold_map(T, Q, h_same_q);
    // scores are 32-bit (as LASTZ's score type): the trivial alignment of a scaffold with itself scores up to 100 per base
    for (int t = 0; t < T.nscaf; t++)
        MB2_REQUIRE(same[t] < 0 || T.len[t] < 21000000u, -3,
                    "align: a scaffold of 21 Mbp or more aligned to itself: the score of the trivial self-alignment does not fit 32 bits");
    DevBuf<int32_t> d_same(T.nscaf);
    MB2_CUDA(cudaMemcpyAsync(d_same.get(), same.data(), T.nscaf * sizeof(int32_t), cudaMemcpyHostToDevice, cx.stream));
    MB2_CUDA(cudaStreamSynchronize(cx.stream));

    // Chunks are formed on the fly: the survivor density (survivors per query base) seen so far sizes the next chunk and
    // its buffer, so that a repeat-rich genome costs at most one scan that overflows (the first), not one per chunk.
    const uint64_t chunk_default = default_chunk_bases();
    double dens = 0.0;                               // highest survivors-per-query-base observed so far
    int s_next = 0;
    while (s_next < Q.nscaf) {
        uint64_t limit = chunk_default;
        if (dens > 0.0) limit = std::min<uint64_t>(limit, std::max<uint64_t>(1, (uint64_t)(0.7 * (double)MAX_SURVIVORS / dens)));
        const QChunk c = next_chunk(Q, s_next, limit);
        uint32_t q_lo, q_hi;
        chunk_range(Q, c, q_lo, q_hi);
        uint64_t cbases = 0;
        for (int s = c.s_lo; s < c.s_hi; s++) cbases += Q.len[s];
        uint64_t cap = std::max<uint64_t>(1u << 20, std::min<uint64_t>(MAX_SURVIVORS, std::max<uint64_t>((T.nbases + cbases) / 2, (uint64_t)(1.3 * dens * (double)cbases))));
        unsigned long long nsurv = 0;
        MB2_CUDA(cudaMemsetAsync(counters.get(), 0, CNT_N * sizeof(unsigned long long), cx.stream));
        const bool ok = scan_chunk(T, Q, tab, q_lo, q_hi, p, s0, cap, counters.get(), nsurv, acc);
        if (cbases) dens = std::max(dens, (double)nsurv / (double)cbases);
        if (!ok) {
            MB2_REQUIRE(c.s_hi - c.s_lo > 1, -3, "align: one query scaffold alone produces more surviving seed hits than fit in memory");
            continue;                                // the same scaffolds again, in a smaller chunk sized by the density just measured
        }
        s_next = c.s_hi;
        if (nsurv == 0) continue;
        if (s1.n < nsurv) s1.alloc(nsurv);
        HspSet hsps;
        find_hsps(T, Q, s0.get(), s1.get(), (uint32_t)nsurv, p, hsps, counters.get(), d_same.get());
        DevBuf<uint8_t> in_chain;
        if (p.chain) chain_hsps(hsps, lb, tb, in_chain);
        else {
            in_chain.alloc(hsps.n ? hsps.n : 1);
            if (hsps.n) MB2_CUDA(cudaMemsetAsync(in_chain.get(), 1, hsps.n, cx.stream));
        }
        AlnSet a;
        gapped_extend(T, Q, hsps, in_chain, p, h_same_q, a, counters.get());
        unsigned long long c2[CNT_N];
        MB2_CUDA(cudaMemcpyAsync(c2, counters.get(), sizeof(c2), cudaMemcpyDeviceToHost, cx.stream));
        MB2_CUDA(cudaStreamSynchronize(cx.stream));
        acc[CNT_HSPS] += hsps.n; acc[CNT_EXTENDED] += c2[CNT_EXTENDED]; acc[CNT_S2_CELLS] += c2[CNT_S2_CELLS];
        acc[CNT_GAPPED_CELLS] += c2[CNT_GAPPED_CELLS]; acc[CNT_ANCHORS] += c2[CNT_ANCHORS]; acc[CNT_ALNS] += a.n;
        out.append(a, Q, nq, strands);
    }
    if (h_counters) for (int k = 0; k < CNT_N; k++) h_counters[k] = acc[k];
}

}  // namespace mb2
