// genome.cu -- build the device genome (2-bit pack, N mask, 4-bit codes) from ASCII, and its reverse complement.
// Replaces the FASTA -> per-scaffold files -> LASTZ sequence loading of the reference
// (utils.py:274-309 splitFasta, LASTZ's own reader) for the hot path.
#include "seq.cuh"
#include "internal.cuh"

namespace mb2 {

// `codes` mirror (1 byte per base, read by the gapped DP, ydrop_warp.cuh): base | parity(base) << 2 for A,C,G,T (0,5,6,3);
// 8 = any other character; 12 = pad (outside every scaffold): a DP cell that would consume it does not exist
__device__ __forceinline__ uint32_t code_byte(uint32_t base, uint32_t bad, uint32_t pad) {
    return pad ? 12u : (bad ? 8u : (base | (((base ^ (base >> 1)) & 1u) << 2)));
}

// the four nb words of 32 bases (2-bit codes `bits`, non-ACGT flags `nflag`)
__device__ __forceinline__ void store_nibbles(uint32_t* __restrict__ nb, uint32_t w, uint64_t bits, uint32_t nflag) {
    uint32_t v[4] = {0, 0, 0, 0};
#pragma unroll
    for (int c = 0; c < 32; c++) v[c >> 3] |= nib_code((uint32_t)(bits >> (2 * c)) & 3u, (nflag >> c) & 1u) << (4 * (c & 7));
    reinterpret_cast<uint4*>(nb)[w] = make_uint4(v[0], v[1], v[2], v[3]);
}

// one thread packs 32 bases -> one uint64 of 2-bit codes + one uint32 of N flags (+ soft-mask flags, 4-bit codes, code bytes)
__global__ void __launch_bounds__(256)
pack_kernel(const uint8_t* __restrict__ ascii, uint32_t nwords, uint64_t* __restrict__ pk, uint32_t* __restrict__ nm,
            uint32_t* __restrict__ sm, uint32_t* __restrict__ nb, uint8_t* __restrict__ codes, int* __restrict__ any_soft) {
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nwords) return;
    const uint4* src = reinterpret_cast<const uint4*>(ascii + (size_t)w * 32);
    uint64_t bits = 0;
    uint32_t nflag = 0, padflag = 0, lowflag = 0;
#pragma unroll
    for (int v = 0; v < 2; v++) {
        const uint4 x = src[v];
        const uint32_t words[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
        for (int k = 0; k < 4; k++) {
#pragma unroll
            for (int b = 0; b < 4; b++) {
                const uint32_t raw = (words[k] >> (8 * b)) & 0xFFu;
                const uint32_t c = raw & 0xDFu;   // fold to upper case (soft-masking ignored)
                uint32_t code = 0, bad = 0;
                if (c == 'A') code = 0; else if (c == 'C') code = 1; else if (c == 'G') code = 2; else if (c == 'T') code = 3; else bad = 1;
                const int idx = v * 16 + k * 4 + b;
                bits |= (uint64_t)code << (2 * idx);
                nflag |= bad << idx;
                padflag |= (raw == 0u ? 1u : 0u) << idx;                      // pad positions of the ASCII image are NUL bytes
                lowflag |= ((raw >= 'a' && raw <= 'z') ? 1u : 0u) << idx;        // soft-masked: not seeded, still extended through
            }
        }
    }
    pk[w] = bits;
    nm[w] = nflag;
    sm[w] = nflag | lowflag;
    store_nibbles(nb, w, bits, nflag);
    if (lowflag & ~nflag) atomicOr(any_soft, 1);      // rare: only soft-masked assemblies take this
    uint32_t out[8];
#pragma unroll
    for (int k = 0; k < 8; k++) {
        uint32_t v = 0;
#pragma unroll
        for (int b = 0; b < 4; b++) {
            const int idx = k * 4 + b;
            v |= code_byte((uint32_t)((bits >> (2 * idx)) & 3u), (nflag >> idx) & 1u, (padflag >> idx) & 1u) << (8 * b);
        }
        out[k] = v;
    }
    uint4* dst = reinterpret_cast<uint4*>(codes + (size_t)w * 32);
    dst[0] = make_uint4(out[0], out[1], out[2], out[3]);
    dst[1] = make_uint4(out[4], out[5], out[6], out[7]);
}

// reverse complement every scaffold in place of its own slot (same offsets, same lengths)
__global__ void __launch_bounds__(256)
revcomp_kernel(GenomeView src, uint64_t* __restrict__ pk, uint32_t* __restrict__ nm, uint32_t* __restrict__ sm, uint32_t* __restrict__ nb,
               uint8_t* __restrict__ codes, uint32_t nwords) {
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nwords) return;
    const uint32_t p0 = w * 32;
    // find the scaffold containing (or following) p0: last s with off[s] <= p0 + 31
    int lo = 0, hi = src.nscaf;
    while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (src.off[mid] <= p0 + 31) lo = mid; else hi = mid; }
    const uint32_t so = src.off[lo], sl = src.len[lo];
    uint64_t bits = 0;
    uint32_t nflag = 0, sflag = 0;
    for (int c = 0; c < 32; c++) {
        const uint32_t p = p0 + c;
        uint32_t code = 0, bad = 1, soft = 1;
        if (p >= so && p < so + sl) {
            const uint32_t sp = so + (sl - 1 - (p - so));
            bad = isn_at(src.nm, sp);
            soft = isn_at(src.sm, sp);
            code = bad ? 0u : 3u - base_at(src.pk, sp);
        }
        bits |= (uint64_t)code << (2 * c);
        nflag |= bad << c;
        sflag |= soft << c;
        codes[(size_t)p0 + c] = (uint8_t)code_byte(code, bad, (p >= so && p < so + sl) ? 0u : 1u);
    }
    pk[w] = bits;
    nm[w] = nflag;
    sm[w] = sflag;
    store_nibbles(nb, w, bits, nflag);
}

// nfree[s] = 1 iff scaffold s has no non-ACGT base (one CTA per scaffold scans its mask words)
__global__ void __launch_bounds__(256)
nfree_kernel(const uint32_t* __restrict__ nm, const uint32_t* __restrict__ off, const uint32_t* __restrict__ len, uint32_t* __restrict__ nfree) {
    const uint32_t s = blockIdx.x;
    const uint32_t o = off[s], l = len[s];
    const uint32_t w0 = o >> 5, nw = (l + 31) >> 5;          // scaffolds start word-aligned (multiple of 64 bases)
    int bad = 0;
    for (uint32_t w = threadIdx.x; w < nw; w += blockDim.x) {
        uint32_t m = nm[w0 + w];
        if (w == nw - 1 && (l & 31)) m &= (1u << (l & 31)) - 1u;
        bad |= m != 0;
    }
    bad = __syncthreads_or(bad);
    if (threadIdx.x == 0) nfree[s] = bad ? 0u : 1u;
}

uint64_t next_genome_id() { static uint64_t c = 0; return ++c; }

static void layout(Genome& g, const uint64_t* lens, int n) {
    g.nscaf = n;
    g.off.resize(n); g.len.resize(n);
    uint64_t pos = GENOME_END_PAD;
    g.nbases = 0;
    for (int s = 0; s < n; s++) {
        MB2_REQUIRE(lens[s] < 0x7fffffffull, -3, "scaffold longer than 2^31-1 bases");
        g.off[s] = (uint32_t)pos; g.len[s] = (uint32_t)lens[s];
        g.nbases += lens[s];
        pos = (pos + lens[s] + GENOME_PAD + 63) & ~63ull;
        MB2_REQUIRE(pos < 0xfff00000ull, -3, "genome exceeds 2^32 padded positions; load it as several genomes");
    }
    g.G = pos + GENOME_END_PAD;
}

Genome* genome_from_ascii(const uint8_t* const* seqs, const uint64_t* lens, int n) {
    MB2_REQUIRE(n > 0, -2, "genome: need at least one scaffold");
    Genome* g = new Genome();
    try {
        layout(*g, lens, n);
        Ctx& cx = ctx();
        // ASCII image of the padded coordinate space on the device: pads are 'N' (device memset), every scaffold is copied
        // straight from the caller's buffer to its offset (DMA when that buffer is pinned; the driver stages pageable
        // memory itself), then packed on the device
        const size_t nbytes = g->G + 64;   // = (G/32 + 2) * 32
        DevBuf<uint8_t> d_ascii(nbytes);
        MB2_CUDA(cudaMemsetAsync(d_ascii.get(), 0, nbytes, cx.stream));   // NUL = pad (pack_kernel flags it non-ACGT and codes it 12)
        for (int s = 0; s < n; s++)
            if (lens[s]) MB2_CUDA(cudaMemcpyAsync(d_ascii.get() + g->off[s], seqs[s], lens[s], cudaMemcpyHostToDevice, cx.stream));
        const uint32_t nwords = (uint32_t)(g->G / 32) + 2;
        g->pk.alloc(nwords); g->nm.alloc(nwords); g->sm.alloc(nwords); g->nb.alloc((size_t)nwords * 4); g->codes.alloc((size_t)nwords * 32);
        g->d_off.alloc(n); g->d_len.alloc(n);
        MB2_CUDA(cudaMemcpyAsync(g->d_off.get(), g->off.data(), n * sizeof(uint32_t), cudaMemcpyHostToDevice, cx.stream));
        MB2_CUDA(cudaMemcpyAsync(g->d_len.get(), g->len.data(), n * sizeof(uint32_t), cudaMemcpyHostToDevice, cx.stream));
        DevBuf<int> d_soft(1);
        MB2_CUDA(cudaMemsetAsync(d_soft.get(), 0, sizeof(int), cx.stream));
        launch(pack_kernel, cdiv(nwords, 256), 256, 0, d_ascii.get(), nwords, g->pk.get(), g->nm.get(), g->sm.get(), g->nb.get(), g->codes.get(), d_soft.get());
        int h_soft = 0;
        MB2_CUDA(cudaMemcpyAsync(&h_soft, d_soft.get(), sizeof(int), cudaMemcpyDeviceToHost, cx.stream));
        g->d_nfree.alloc(n);
        launch(nfree_kernel, n, 256, 0, g->nm.get(), g->d_off.get(), g->d_len.get(), g->d_nfree.get());
        MB2_CUDA(cudaStreamSynchronize(cx.stream));      // the caller's buffers are free again after this
        g->has_soft = h_soft != 0;
        if (!g->has_soft) g->sm.release();               // identical to nm: view() hands kernels nm
        g->id = next_genome_id(); g->fwd_src_id = g->id; g->nfwd = n;
    } catch (...) { delete g; throw; }
    return g;
}

Genome* genome_revcomp(const Genome& src) {
    Genome* g = new Genome();
    try {
        g->nscaf = src.nscaf; g->off = src.off; g->len = src.len; g->G = src.G; g->nbases = src.nbases; g->is_rc = !src.is_rc;
        g->has_soft = src.has_soft;
        const uint32_t nwords = (uint32_t)(g->G / 32) + 2;
        g->pk.alloc(nwords); g->nm.alloc(nwords); g->sm.alloc(nwords); g->nb.alloc((size_t)nwords * 4); g->codes.alloc((size_t)nwords * 32);
        g->d_off.alloc(src.nscaf); g->d_len.alloc(src.nscaf);
        Ctx& cx = ctx();
        MB2_CUDA(cudaMemcpyAsync(g->d_off.get(), src.d_off.get(), src.nscaf * sizeof(uint32_t), cudaMemcpyDeviceToDevice, cx.stream));
        MB2_CUDA(cudaMemcpyAsync(g->d_len.get(), src.d_len.get(), src.nscaf * sizeof(uint32_t), cudaMemcpyDeviceToDevice, cx.stream));
        g->d_nfree.alloc(src.nscaf);
        MB2_CUDA(cudaMemcpyAsync(g->d_nfree.get(), src.d_nfree.get(), src.nscaf * sizeof(uint32_t), cudaMemcpyDeviceToDevice, cx.stream));
        launch(revcomp_kernel, cdiv(nwords, 256), 256, 0, view(src), g->pk.get(), g->nm.get(), g->sm.get(), g->nb.get(), g->codes.get(), nwords);
        g->id = next_genome_id(); g->fwd_src_id = 0; g->nfwd = 0;
    } catch (...) { delete g; throw; }
    return g;
}

// Both strands in one genome: scaffolds [0,n) = src, scaffolds [n,2n) = their reverse complements. Lets one pass of the
// alignment pipeline cover --strand=both (tile = target x (scaffold, strand)), so the two strands share every launch.
__global__ void __launch_bounds__(256)
both_strands_kernel(GenomeView src, const uint32_t* __restrict__ noff, const uint32_t* __restrict__ nlen, int n2,
                    uint64_t* __restrict__ pk, uint32_t* __restrict__ nm, uint32_t* __restrict__ sm, uint32_t* __restrict__ nb,
                    uint8_t* __restrict__ codes, uint32_t nwords) {
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nwords) return;
    const uint32_t p0 = w * 32;
    int lo = 0, hi = n2;                         // scaffold of the new layout containing (or preceding) this word
    while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (noff[mid] <= p0 + 31) lo = mid; else hi = mid; }
    const uint32_t so = noff[lo], sl = nlen[lo];
    const int n = n2 >> 1;
    const bool rc = lo >= n;
    const uint32_t srco = src.off[rc ? lo - n : lo];
    uint64_t bits = 0; uint32_t nflag = 0, sflag = 0;
    uint32_t cw[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int c = 0; c < 32; c++) {
        const uint32_t p = p0 + c;
        uint32_t code = 0, bad = 1, soft = 1;
        if (p >= so && p < so + sl) {
            const uint32_t k = p - so;
            const uint32_t sp = srco + (rc ? sl - 1 - k : k);
            bad = isn_at(src.nm, sp);
            soft = isn_at(src.sm, sp);
            code = bad ? 0u : (rc ? 3u - base_at(src.pk, sp) : base_at(src.pk, sp));
        }
        bits |= (uint64_t)code << (2 * c);
        nflag |= bad << c;
        sflag |= soft << c;
        cw[c >> 2] |= code_byte(code, bad, (p >= so && p < so + sl) ? 0u : 1u) << (8 * (c & 3));
    }
    pk[w] = bits; nm[w] = nflag; sm[w] = sflag;
    store_nibbles(nb, w, bits, nflag);
    uint4* dst = reinterpret_cast<uint4*>(codes + (size_t)w * 32);
    dst[0] = make_uint4(cw[0], cw[1], cw[2], cw[3]);
    dst[1] = make_uint4(cw[4], cw[5], cw[6], cw[7]);
}

Genome* genome_both_strands(const Genome& src) {
    Genome* g = new Genome();
    try {
        const int n = src.nscaf;
        std::vector<uint64_t> lens(2 * n);
        for (int s = 0; s < n; s++) lens[s] = lens[n + s] = src.len[s];
        layout(*g, lens.data(), 2 * n);
        g->has_soft = src.has_soft;
        const uint32_t nwords = (uint32_t)(g->G / 32) + 2;
        g->pk.alloc(nwords); g->nm.alloc(nwords); g->sm.alloc(nwords); g->nb.alloc((size_t)nwords * 4); g->codes.alloc((size_t)nwords * 32);
        g->d_off.alloc(2 * n); g->d_len.alloc(2 * n); g->d_nfree.alloc(2 * n);
        Ctx& cx = ctx();
        MB2_CUDA(cudaMemcpyAsync(g->d_off.get(), g->off.data(), 2 * n * sizeof(uint32_t), cudaMemcpyHostToDevice, cx.stream));
        MB2_CUDA(cudaMemcpyAsync(g->d_len.get(), g->len.data(), 2 * n * sizeof(uint32_t), cudaMemcpyHostToDevice, cx.stream));
        MB2_CUDA(cudaMemcpyAsync(g->d_nfree.get(), src.d_nfree.get(), n * sizeof(uint32_t), cudaMemcpyDeviceToDevice, cx.stream));
        MB2_CUDA(cudaMemcpyAsync(g->d_nfree.get() + n, src.d_nfree.get(), n * sizeof(uint32_t), cudaMemcpyDeviceToDevice, cx.stream));
        launch(both_strands_kernel, cdiv(nwords, 256), 256, 0, view(src), g->d_off.get(), g->d_len.get(), 2 * n, g->pk.get(), g->nm.get(),
               g->sm.get(), g->nb.get(), g->codes.get(), nwords);
        MB2_CUDA(cudaStreamSynchronize(cx.stream));   // g->off/len host vectors were copy sources
        g->id = next_genome_id(); g->fwd_src_id = src.fwd_src_id == src.id ? src.id : 0; g->nfwd = src.fwd_src_id == src.id ? n : 0;
    } catch (...) { delete g; throw; }
    return g;
}

// test hook: decode a range back to codes 0..3 / 4
__global__ void decode_kernel(GenomeView g, uint32_t p0, uint32_t n, uint8_t* __restrict__ out) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const uint32_t p = p0 + k;
    out[k] = isn_at(g.nm, p) ? 4 : (uint8_t)base_at(g.pk, p);
}
void genome_decode(const Genome& g, int scaf, uint8_t* h_out) {
    MB2_REQUIRE(scaf >= 0 && scaf < g.nscaf, -2, "decode: scaffold index out of range");
    const uint32_t n = g.len[scaf];
    DevBuf<uint8_t> d(n);
    if (n) launch(decode_kernel, cdiv(n, 256), 256, 0, view(g), g.off[scaf], n, d.get());
    if (n) MB2_CUDA(cudaMemcpyAsync(h_out, d.get(), n, cudaMemcpyDeviceToHost, ctx().stream));
    MB2_CUDA(cudaStreamSynchronize(ctx().stream));
}

}  // namespace mb2
