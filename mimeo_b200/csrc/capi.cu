// capi.cu -- extern "C" boundary of libmimeo_b200.so (see include/mimeo_b200.h).
#include <algorithm>
#include <cstring>
#include <map>
#include <vector>

#include "primitives.cuh"
#include "internal.cuh"
#include "seq.cuh"
#include "xdrop_table.cuh"
#include "mimeo_b200.h"

namespace mb2 {

static Ctx g_ctx;
static thread_local std::string g_err;

Ctx& ctx() { return g_ctx; }

void ensure_init() {
    if (!g_ctx.ready) throw Error(MB2_ERR_INVALID_ARG, "mb2_init() has not been called");
    // other CUDA users in the process (torch, NCCL) may have changed the calling thread's current device
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess || cur != g_ctx.device) MB2_CUDA(cudaSetDevice(g_ctx.device));
}

// ---- scratch allocator (common.cuh)
namespace {
struct Slab { char* base; size_t size; };
struct ScratchState {
    std::vector<Slab> slabs;
    std::map<char*, size_t> free_blocks;     // address -> size, coalesced
    std::map<char*, size_t> used;            // address -> size
    size_t reserved = 0;
};
ScratchState g_scratch;
constexpr size_t SCRATCH_ALIGN = 512;
constexpr size_t SCRATCH_MIN_SLAB = (size_t)1 << 30;
}  // namespace

void* scratch_alloc(size_t bytes) {
    bytes = (bytes + SCRATCH_ALIGN - 1) / SCRATCH_ALIGN * SCRATCH_ALIGN;
    ScratchState& st = g_scratch;
    auto best = st.free_blocks.end();
    for (auto it = st.free_blocks.begin(); it != st.free_blocks.end(); ++it)
        if (it->second >= bytes && (best == st.free_blocks.end() || it->second < best->second)) best = it;
    if (best == st.free_blocks.end()) {
        // grow: a slab of at least 1 GiB (and at least half of what is reserved so far, so growth stays geometric)
        size_t want = std::max(bytes, std::max(SCRATCH_MIN_SLAB, st.reserved / 2));
        char* p = nullptr;
        cudaError_t e = cudaMalloc((void**)&p, want);
        if (e != cudaSuccess && want > bytes) { cudaGetLastError(); want = bytes; e = cudaMalloc((void**)&p, want); }
        if (e != cudaSuccess) {
            cudaGetLastError();
            throw Error(MB2_ERR_TOO_LARGE, "device memory exhausted: cannot reserve " + std::to_string(bytes >> 20) + " MiB of scratch (" +
                                               std::to_string(st.reserved >> 20) + " MiB reserved)");
        }
        st.slabs.push_back({p, want});
        st.reserved += want;
        best = st.free_blocks.emplace(p, want).first;
    }
    char* p = best->first;
    const size_t sz = best->second;
    st.free_blocks.erase(best);
    if (sz > bytes) st.free_blocks.emplace(p + bytes, sz - bytes);
    st.used.emplace(p, bytes);
    return p;
}

void scratch_free(void* ptr) {
    ScratchState& st = g_scratch;
    char* p = static_cast<char*>(ptr);
    auto u = st.used.find(p);
    if (u == st.used.end()) return;          // not ours (never happens), or released by scratch_release_all
    size_t sz = u->second;
    st.used.erase(u);
    auto nx = st.free_blocks.lower_bound(p);
    // coalesce with the following and the preceding free block when they touch AND lie in the same slab
    auto same_slab = [&](char* a, char* b) {
        for (const Slab& s : st.slabs) if (a >= s.base && a < s.base + s.size) return b >= s.base && b < s.base + s.size;
        return false;
    };
    if (nx != st.free_blocks.end() && p + sz == nx->first && same_slab(p, nx->first)) { sz += nx->second; nx = st.free_blocks.erase(nx); }
    if (nx != st.free_blocks.begin()) {
        auto pv = std::prev(nx);
        if (pv->first + pv->second == p && same_slab(pv->first, p)) { p = pv->first; sz += pv->second; st.free_blocks.erase(pv); }
    }
    st.free_blocks.emplace(p, sz);
}

void scratch_release_all() {
    ScratchState& st = g_scratch;
    for (const Slab& s : st.slabs) cudaFree(s.base);
    st = ScratchState();
}
size_t scratch_reserved_bytes() { return g_scratch.reserved; }

template <typename F>
static int guarded(F&& f) {
    try {
        f();
        return MB2_OK;
    } catch (const Error& e) {
        g_err = e.what();
        return e.code;
    } catch (const std::exception& e) {
        g_err = e.what();
        return MB2_ERR_INTERNAL;
    }
}

}  // namespace mb2

using namespace mb2;

template <typename K>
static void test_sort(K* keys, uint32_t* vals, uint64_t n, int b0, int b1) {
    ensure_init();
    DevBuf<K> k0(n), k1(n);
    DevBuf<uint32_t> v0(vals ? n : 0), v1(vals ? n : 0);
    if (n == 0) return;
    MB2_CUDA(cudaMemcpyAsync(k0.get(), keys, n * sizeof(K), cudaMemcpyHostToDevice, g_ctx.stream));
    int w;
    if (vals) {
        MB2_CUDA(cudaMemcpyAsync(v0.get(), vals, n * sizeof(uint32_t), cudaMemcpyHostToDevice, g_ctx.stream));
        w = radix_sort_bits<K, uint32_t>(k0.get(), k1.get(), v0.get(), v1.get(), n, b0, b1);
        MB2_CUDA(cudaMemcpyAsync(vals, w ? v1.get() : v0.get(), n * sizeof(uint32_t), cudaMemcpyDeviceToHost, g_ctx.stream));
    } else {
        NoVal* nv = nullptr;
        w = radix_sort_bits<K, NoVal>(k0.get(), k1.get(), nv, nv, n, b0, b1);
    }
    MB2_CUDA(cudaMemcpyAsync(keys, w ? k1.get() : k0.get(), n * sizeof(K), cudaMemcpyDeviceToHost, g_ctx.stream));
    MB2_CUDA(cudaStreamSynchronize(g_ctx.stream));
}

extern "C" {

int mb2_init(int device) {
    return guarded([&] {
        if (g_ctx.ready && g_ctx.device == device) return;
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || ndev == 0)
            throw Error(MB2_ERR_CUDA, std::string("no CUDA device available: ") + cudaGetErrorString(e) +
                                          " -- libmimeo_b200 has no CPU fallback");
        MB2_REQUIRE(device >= 0 && device < ndev, MB2_ERR_INVALID_ARG, "mb2_init: device index out of range");
        MB2_CUDA(cudaSetDevice(device));
        cudaDeviceProp prop;
        MB2_CUDA(cudaGetDeviceProperties(&prop, device));
        MB2_REQUIRE(prop.major >= 10, MB2_ERR_CUDA,
                    std::string("libmimeo_b200 is built for sm_100a only; found ") + prop.name);
        g_ctx.device = device;
        g_ctx.sm_count = prop.multiProcessorCount;
        MB2_CUDA(cudaStreamCreateWithFlags(&g_ctx.stream, cudaStreamNonBlocking));
        cudaMemPool_t pool;
        MB2_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
        uint64_t thresh = UINT64_MAX;   // keep freed scratch cached in the pool between calls
        MB2_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thresh));
        g_ctx.launches = 0;
        g_ctx.debug_sync = getenv("MB2_DEBUG_SYNC") != nullptr;
        g_ctx.ready = true;
    });
}

void mb2_shutdown(void) {
    if (g_ctx.ready) {
        cudaStreamSynchronize(g_ctx.stream);
        coverage_release_scratch();
        gapped_release_scratch();
        scratch_release_all();
        cudaStreamDestroy(g_ctx.stream);
        g_ctx.stream = nullptr;
        g_ctx.ready = false;
    }
}

const char* mb2_last_error(void) { return g_err.c_str(); }
void* mb2_stream(void) { return (void*)g_ctx.stream; }
unsigned long long mb2_launch_count(void) { return g_ctx.launches; }
int mb2_sm_count(void) { return g_ctx.sm_count; }
int mb2_sync(void) {
    return guarded([&] { ensure_init(); MB2_CUDA(cudaStreamSynchronize(g_ctx.stream)); });
}

static void prof_drain() {
    if (g_ctx.prof_recs.empty()) return;
    MB2_CUDA(cudaStreamSynchronize(g_ctx.stream));
    for (auto& r : g_ctx.prof_recs) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, r.a, r.b);
        auto& acc = g_ctx.prof_acc[r.tag];
        acc.first += ms; acc.second += 1;
        cudaEventDestroy(r.a); cudaEventDestroy(r.b);
    }
    g_ctx.prof_recs.clear();
}

int mb2_prof_enable(int on) {
    return guarded([&] { ensure_init(); prof_drain(); g_ctx.prof = on != 0; });
}
int mb2_prof_get(const char* tag, double* ms_total, unsigned long long* count) {
    return guarded([&] {
        ensure_init();
        prof_drain();
        auto it = g_ctx.prof_acc.find(tag ? tag : "");
        if (ms_total) *ms_total = it == g_ctx.prof_acc.end() ? 0.0 : it->second.first;
        if (count) *count = it == g_ctx.prof_acc.end() ? 0ull : it->second.second;
    });
}
int mb2_prof_reset(void) {
    return guarded([&] { ensure_init(); prof_drain(); g_ctx.prof_acc.clear(); });
}

// ------------------------------------------------------------------------------------------ coverage
int mb2_coverage_segments_dev(const int32_t* d_chrom, const int32_t* d_start, const int32_t* d_end, uint64_t nhits,
                              const int64_t* chrom_sizes, int nchrom, int min_cov, int min_len, mb2_segments* out) {
    return guarded([&] {
        ensure_init();
        MB2_REQUIRE(out != nullptr && chrom_sizes != nullptr, MB2_ERR_INVALID_ARG, "coverage: null argument");
        MB2_REQUIRE(nhits == 0 || (d_chrom && d_start && d_end), MB2_ERR_INVALID_ARG, "coverage: null hit arrays");
        std::memset(out, 0, sizeof(*out));
        CoverageResult res;
        coverage_segments_device(d_chrom, d_start, d_end, nhits, chrom_sizes, nchrom, min_cov, min_len, res);
        MB2_CUDA(cudaStreamSynchronize(g_ctx.stream));
        out->n = res.n;
        out->on_device = 1;
        // hand the buffers over to the caller (freed by mb2_free_segments)
        out->chrom = res.chrom.p; res.chrom.p = nullptr;
        out->start = res.start.p; res.start.p = nullptr;
        out->end = res.end.p; res.end.p = nullptr;
    });
}

int mb2_coverage_segments(const int32_t* chrom, const int32_t* start, const int32_t* end, uint64_t nhits,
                          const int64_t* chrom_sizes, int nchrom, int min_cov, int min_len, mb2_segments* out) {
    return guarded([&] {
        ensure_init();
        MB2_REQUIRE(out != nullptr && chrom_sizes != nullptr, MB2_ERR_INVALID_ARG, "coverage: null argument");
        MB2_REQUIRE(nhits == 0 || (chrom && start && end), MB2_ERR_INVALID_ARG, "coverage: null hit arrays");
        std::memset(out, 0, sizeof(*out));
        DevBuf<int32_t> dc(nhits), ds(nhits), de(nhits);
        if (nhits) {
            MB2_CUDA(cudaMemcpyAsync(dc.get(), chrom, nhits * sizeof(int32_t), cudaMemcpyHostToDevice, g_ctx.stream));
            MB2_CUDA(cudaMemcpyAsync(ds.get(), start, nhits * sizeof(int32_t), cudaMemcpyHostToDevice, g_ctx.stream));
            MB2_CUDA(cudaMemcpyAsync(de.get(), end, nhits * sizeof(int32_t), cudaMemcpyHostToDevice, g_ctx.stream));
        }
        CoverageResult res;
        coverage_segments_device(dc.get(), ds.get(), de.get(), nhits, chrom_sizes, nchrom, min_cov, min_len, res);
        out->n = res.n;
        out->on_device = 0;
        if (res.n) {
            out->chrom = (int32_t*)malloc(res.n * sizeof(int32_t));
            out->start = (int32_t*)malloc(res.n * sizeof(int32_t));
            out->end = (int32_t*)malloc(res.n * sizeof(int32_t));
            MB2_REQUIRE(out->chrom && out->start && out->end, MB2_ERR_INTERNAL, "coverage: host allocation failed");
            MB2_CUDA(cudaMemcpyAsync(out->chrom, res.chrom.get(), res.n * sizeof(int32_t), cudaMemcpyDeviceToHost, g_ctx.stream));
            MB2_CUDA(cudaMemcpyAsync(out->start, res.start.get(), res.n * sizeof(int32_t), cudaMemcpyDeviceToHost, g_ctx.stream));
            MB2_CUDA(cudaMemcpyAsync(out->end, res.end.get(), res.n * sizeof(int32_t), cudaMemcpyDeviceToHost, g_ctx.stream));
        }
        MB2_CUDA(cudaStreamSynchronize(g_ctx.stream));
    });
}

int mb2_coverage_segments_into(const int32_t* d_chrom, const int32_t* d_start, const int32_t* d_end, uint64_t nhits,
                               const int64_t* chrom_sizes, int nchrom, int min_cov, int min_len, int32_t* d_out_chrom,
                               int32_t* d_out_start, int32_t* d_out_end, uint64_t capacity, uint64_t* n_out) {
    CoverageResult res;
    const int rc = guarded([&] {
        ensure_init();
        MB2_REQUIRE(n_out != nullptr && chrom_sizes != nullptr, MB2_ERR_INVALID_ARG, "coverage: null argument");
        *n_out = 0;
        MB2_REQUIRE(nhits == 0 || (d_chrom && d_start && d_end), MB2_ERR_INVALID_ARG, "coverage: null hit arrays");
        MB2_REQUIRE(capacity > 0 && d_out_chrom && d_out_start && d_out_end, MB2_ERR_INVALID_ARG, "coverage: null or empty output arrays");
        res.ext_chrom = d_out_chrom; res.ext_start = d_out_start; res.ext_end = d_out_end; res.ext_cap = capacity;
        coverage_segments_device(d_chrom, d_start, d_end, nhits, chrom_sizes, nchrom, min_cov, min_len, res);
        MB2_CUDA(cudaStreamSynchronize(g_ctx.stream));
        *n_out = res.n;
    });
    if (rc == MB2_ERR_CAPACITY && n_out) *n_out = res.n;
    return rc;
}

void mb2_free_segments(mb2_segments* seg) {
    if (!seg) return;
    if (seg->on_device) {
        if (seg->chrom) scratch_free(seg->chrom);
        if (seg->start) scratch_free(seg->start);
        if (seg->end) scratch_free(seg->end);
    } else {
        free(seg->chrom); free(seg->start); free(seg->end);
    }
    std::memset(seg, 0, sizeof(*seg));
}

// ------------------------------------------------------------------------------------------ genomes
struct mb2_genome { Genome* g; };

int mb2_genome_create(const uint8_t* const* seqs, const uint64_t* lens, int n, mb2_genome** out) {
    return guarded([&] {
        ensure_init();
        MB2_REQUIRE(seqs && lens && out, MB2_ERR_INVALID_ARG, "genome_create: null argument");
        Genome* g = genome_from_ascii(seqs, lens, n);
        *out = new mb2_genome{g};
    });
}
int mb2_genome_revcomp(const mb2_genome* g, mb2_genome** out) {
    return guarded([&] {
        ensure_init();
        MB2_REQUIRE(g && g->g && out, MB2_ERR_INVALID_ARG, "genome_revcomp: null argument");
        *out = new mb2_genome{genome_revcomp(*g->g)};
    });
}
int mb2_genome_both_strands(const mb2_genome* g, mb2_genome** out) {
    return guarded([&] {
        ensure_init();
        MB2_REQUIRE(g && g->g && out, MB2_ERR_INVALID_ARG, "genome_both_strands: null argument");
        *out = new mb2_genome{genome_both_strands(*g->g)};
    });
}
void mb2_genome_free(mb2_genome* g) {
    if (!g) return;
    delete g->g;
    delete g;
}
int mb2_genome_decode(const mb2_genome* g, int scaf, uint8_t* out) {
    return guarded([&] {
        ensure_init();
        MB2_REQUIRE(g && g->g && out, MB2_ERR_INVALID_ARG, "genome_decode: null argument");
        genome_decode(*g->g, scaf, out);
    });
}
int mb2_test_genome_nibbles(const mb2_genome* g, uint32_t* out, uint64_t cap, uint64_t* nwords) {
    return guarded([&] {
        ensure_init();
        MB2_REQUIRE(g && g->g && nwords && (out || cap == 0), MB2_ERR_INVALID_ARG, "test_genome_nibbles: null argument");
        const uint64_t n = g->g->G / 8 + 8;
        *nwords = n;
        const uint64_t k = cap < n ? cap : n;
        if (k) MB2_CUDA(cudaMemcpyAsync(out, g->g->nb.get(), k * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx().stream));
        MB2_CUDA(cudaStreamSynchronize(ctx().stream));
    });
}

void mb2_default_align_params(mb2_align_params* p) {
    if (!p) return;
    AlignParams d;
    p->hspthresh = d.hspthresh; p->xdrop = d.xdrop; p->ydrop = d.ydrop; p->gap_open = d.gap_open; p->gap_extend = d.gap_extend;
    p->gappedthresh = d.gappedthresh; p->entropy = d.entropy; p->chain = d.chain; p->gapped = d.gapped; p->transition = d.transition;
}
static AlignParams to_params(const mb2_align_params* p) {
    AlignParams a;
    if (p) {
        a.hspthresh = p->hspthresh; a.xdrop = p->xdrop; a.ydrop = p->ydrop; a.gap_open = p->gap_open; a.gap_extend = p->gap_extend;
        a.gappedthresh = p->gappedthresh; a.entropy = p->entropy; a.chain = p->chain; a.gapped = p->gapped; a.transition = p->transition;
    }
    MB2_REQUIRE(a.hspthresh > 0, MB2_ERR_INVALID_ARG, "align params: hspthresh must be positive");
    MB2_REQUIRE(a.xdrop >= XT_MIN_XDROP, MB2_ERR_INVALID_ARG,
                "align params: x-drop below 251 is not supported (the three-column extension table needs x-drop > 250)");
    MB2_REQUIRE(a.xdrop <= GF_MAX_XDROP, MB2_ERR_INVALID_ARG,
                "align params: x-drop of 6400 or more is not supported (a gap-free extension could cross the 64-column pad "
                "between two scaffolds, which loses only 6400)");
    MB2_REQUIRE(a.ydrop >= YDROP_MIN && a.ydrop <= YDROP_MAX && a.gap_open >= 0 && a.gap_open <= GAP_OPEN_MAX &&
                    a.gap_extend >= GAP_EXTEND_MIN && a.gap_extend <= GAP_EXTEND_MAX,
                MB2_ERR_INVALID_ARG,
                "align params: y-drop must lie in 1000..20000, gap open in 0..2000 and gap extend in 10..60 "
                "(the range of the 16-bit gapped extension kernel)");
    return a;
}

}  // extern "C"
template <typename Tp>
static Tp* to_host(const DevBuf<Tp>& d, size_t n) {
    Tp* h = (Tp*)malloc((n ? n : 1) * sizeof(Tp));
    MB2_REQUIRE(h != nullptr, MB2_ERR_INTERNAL, "host allocation failed");
    if (n) MB2_CUDA(cudaMemcpyAsync(h, d.get(), n * sizeof(Tp), cudaMemcpyDeviceToHost, g_ctx.stream));
    return h;
}
extern "C" {

void mb2_free_hsps(mb2_hsps* h) {
    if (!h) return;
    free(h->tile); free(h->s1); free(h->s2); free(h->len); free(h->score);
    std::memset(h, 0, sizeof(*h));
}

int mb2_test_hsps(const mb2_genome* T, const mb2_genome* Q, const mb2_align_params* p, mb2_hsps* out, uint64_t* stats) {
    return guarded([&] {
        ensure_init();
        MB2_REQUIRE(T && Q && out, MB2_ERR_INVALID_ARG, "test_hsps: null argument");
        std::memset(out, 0, sizeof(*out));
        HspSet h;
        unsigned long long cnt[CNT_N];
        align_hsps(*T->g, *Q->g, to_params(p), h, cnt);
        out->n = h.n;
        out->tile = to_host(h.tile, h.n); out->s1 = to_host(h.s1, h.n); out->s2 = to_host(h.s2, h.n);
        out->len = to_host(h.len, h.n); out->score = to_host(h.score, h.n);
        MB2_CUDA(cudaStreamSynchronize(g_ctx.stream));
        if (stats) for (int k = 0; k < CNT_N; k++) stats[k] = cnt[k];
    });
}

void mb2_free_seed_survivors(mb2_seed_survivors* s) {
    if (!s) return;
    free(s->t_pos); free(s->q_pos); free(s->t_off); free(s->q_off);
    std::memset(s, 0, sizeof(*s));
}

int mb2_test_seed_scan(const mb2_genome* T, const mb2_genome* Q, const mb2_align_params* p, uint64_t init_cap,
                       mb2_seed_survivors* out) {
    return guarded([&] {
        ensure_init();
        MB2_REQUIRE(T && Q && T->g && Q->g && out, MB2_ERR_INVALID_ARG, "test_seed_scan: null argument");
        std::memset(out, 0, sizeof(*out));
        std::vector<uint64_t> surv;
        unsigned long long cnt[4];
        scan_survivors(*T->g, *Q->g, to_params(p), init_cap, surv, cnt);
        const size_t n = surv.size();
        const uint32_t qG = (uint32_t)Q->g->G;
        out->t_pos = (uint32_t*)malloc((n ? n : 1) * sizeof(uint32_t));
        out->q_pos = (uint32_t*)malloc((n ? n : 1) * sizeof(uint32_t));
        out->t_off = (uint32_t*)malloc(T->g->nscaf * sizeof(uint32_t));
        out->q_off = (uint32_t*)malloc(Q->g->nscaf * sizeof(uint32_t));
        MB2_REQUIRE(out->t_pos && out->q_pos && out->t_off && out->q_off, MB2_ERR_INTERNAL, "test_seed_scan: host allocation failed");
        for (size_t k = 0; k < n; k++) {
            const uint32_t qj = (uint32_t)surv[k];
            out->q_pos[k] = qj;
            out->t_pos[k] = (uint32_t)(surv[k] >> 32) - qG + qj;      // survivors hold (diagonal + Q.G, query position)
        }
        out->n = n;
        std::memcpy(out->t_off, T->g->off.data(), T->g->nscaf * sizeof(uint32_t));
        std::memcpy(out->q_off, Q->g->off.data(), Q->g->nscaf * sizeof(uint32_t));
        out->t_nscaf = T->g->nscaf; out->q_nscaf = Q->g->nscaf;
        for (int k = 0; k < 4; k++) out->counters[k] = cnt[k];
    });
}

void mb2_free_hits(mb2_hits* h) {
    if (!h) return;
    free(h->t_id); free(h->q_id); free(h->strand); free(h->start1); free(h->end1); free(h->start2); free(h->end2);
    free(h->score); free(h->nmatch); free(h->ncols);
    std::memset(h, 0, sizeof(*h));
}

}  // extern "C"

struct mb2_hits_dev { DevHits h; int nt = 0, nq = 0; };

// every `lastz T Q` of the job: rows of all (target scaffold, query scaffold, strand) tiles appended to a device table
static void align_into(const mb2_genome* T, const mb2_genome* Q, const mb2_genome* Q_aux, const mb2_align_params* p, int strands,
                       const int32_t* t_same_q, mb2_hits_dev& out) {
    MB2_REQUIRE(T && Q && T->g && Q->g, MB2_ERR_INVALID_ARG, "align: null argument");
    MB2_REQUIRE(strands >= 1 && strands <= 3, MB2_ERR_INVALID_ARG, "align: strands must be 1, 2 or 3");
    const AlignParams ap = to_params(p);
    const int nq = Q->g->nscaf;
    // the query actually aligned: Q (+), revcomp(Q) (-), or both strands as one 2n-scaffold genome
    const Genome* q = Q->g;
    Genome* own = nullptr;
    if (strands != 1) {
        if (Q_aux && Q_aux->g) {
            q = Q_aux->g;
            MB2_REQUIRE(q->nscaf == (strands == 3 ? 2 * nq : nq), MB2_ERR_INVALID_ARG, "align: Q_aux does not match Q and strands");
        } else {
            own = strands == 3 ? genome_both_strands(*Q->g) : genome_revcomp(*Q->g);
            q = own;
        }
    }
    try {
        align_strand(*T->g, *q, ap, (strands & 1) ? t_same_q : nullptr, out.h, nq, strands, out.h.stats);
        MB2_CUDA(cudaStreamSynchronize(g_ctx.stream));     // `own` is free to go
    } catch (...) { delete own; throw; }
    delete own;
    out.nt = T->g->nscaf; out.nq = nq;
}

static void download_hits(const DevHits& h, mb2_hits* out) {
    std::memset(out, 0, sizeof(*out));
    const size_t n = h.n;
    out->n = n;
    for (int k = 0; k < CNT_N; k++) out->stats[k] = h.stats[k];
    int32_t** dst[10] = {&out->t_id, &out->q_id, &out->strand, &out->start1, &out->end1, &out->start2, &out->end2,
                         &out->score, &out->nmatch, &out->ncols};
    for (int c = 0; c < 10; c++) {
        *dst[c] = (int32_t*)malloc((n ? n : 1) * sizeof(int32_t));
        MB2_REQUIRE(*dst[c] != nullptr, MB2_ERR_INTERNAL, "align: host allocation failed");
        if (n) MB2_CUDA(cudaMemcpyAsync(*dst[c], h.col[c].get(), n * sizeof(int32_t), cudaMemcpyDeviceToHost, g_ctx.stream));
    }
    MB2_CUDA(cudaStreamSynchronize(g_ctx.stream));
}

extern "C" {

int mb2_align(const mb2_genome* T, const mb2_genome* Q, const mb2_genome* Q_aux, const mb2_align_params* p, int strands,
              const int32_t* t_same_q, mb2_hits* out) {
    return guarded([&] {
        ensure_init();
        MB2_REQUIRE(out != nullptr, MB2_ERR_INVALID_ARG, "align: null argument");
        std::memset(out, 0, sizeof(*out));
        mb2_hits_dev d;
        align_into(T, Q, Q_aux, p, strands, t_same_q, d);
        download_hits(d.h, out);
    });
}

int mb2_align_dev(const mb2_genome* T, const mb2_genome* Q, const mb2_genome* Q_aux, const mb2_align_params* p, int strands,
                  const int32_t* t_same_q, mb2_hits_dev** out) {
    return guarded([&] {
        ensure_init();
        MB2_REQUIRE(out != nullptr, MB2_ERR_INVALID_ARG, "align_dev: null argument");
        *out = nullptr;
        mb2_hits_dev* d = new mb2_hits_dev();
        try { align_into(T, Q, Q_aux, p, strands, t_same_q, *d); } catch (...) { delete d; throw; }
        *out = d;
    });
}
void mb2_hits_dev_free(mb2_hits_dev* h) { delete h; }
uint64_t mb2_hits_dev_count(const mb2_hits_dev* h) { return h ? (uint64_t)h->h.n : 0; }

int mb2_filter_sort(mb2_hits_dev* h, double min_len, double min_idt, int map_rule, uint64_t* n_kept) {
    return guarded([&] {
        ensure_init();
        MB2_REQUIRE(h != nullptr, MB2_ERR_INVALID_ARG, "filter_sort: null argument");
        hits_filter_sort(h->h, min_len, min_idt, map_rule != 0, h->nt, h->nq);
        if (n_kept) *n_kept = h->h.n;
    });
}

int mb2_hits_dev_coverage(const mb2_hits_dev* h, int which, const int64_t* chrom_sizes, int nchrom, int min_cov, int min_len, mb2_segments* out) {
    return guarded([&] {
        ensure_init();
        MB2_REQUIRE(h && out && chrom_sizes, MB2_ERR_INVALID_ARG, "hits_dev_coverage: null argument");
        MB2_REQUIRE(which >= 0 && which <= 2, MB2_ERR_INVALID_ARG, "hits_dev_coverage: which must be 0 (all), 1 (t != q) or 2 (t == q)");
        std::memset(out, 0, sizeof(*out));
        CoverageResult res;
        hits_coverage(h->h, which, chrom_sizes, nchrom, min_cov, min_len, res);
        out->n = res.n;
        out->on_device = 0;
        if (res.n) {
            out->chrom = (int32_t*)malloc(res.n * sizeof(int32_t));
            out->start = (int32_t*)malloc(res.n * sizeof(int32_t));
            out->end = (int32_t*)malloc(res.n * sizeof(int32_t));
            MB2_REQUIRE(out->chrom && out->start && out->end, MB2_ERR_INTERNAL, "coverage: host allocation failed");
            MB2_CUDA(cudaMemcpyAsync(out->chrom, res.chrom.get(), res.n * sizeof(int32_t), cudaMemcpyDeviceToHost, g_ctx.stream));
            MB2_CUDA(cudaMemcpyAsync(out->start, res.start.get(), res.n * sizeof(int32_t), cudaMemcpyDeviceToHost, g_ctx.stream));
            MB2_CUDA(cudaMemcpyAsync(out->end, res.end.get(), res.n * sizeof(int32_t), cudaMemcpyDeviceToHost, g_ctx.stream));
        }
        MB2_CUDA(cudaStreamSynchronize(g_ctx.stream));
    });
}

int mb2_hits_dev_upload(const mb2_hits* in, int nt, int nq, mb2_hits_dev** out) {
    return guarded([&] {
        ensure_init();
        MB2_REQUIRE(in && out, MB2_ERR_INVALID_ARG, "hits_dev_upload: null argument");
        *out = nullptr;
        mb2_hits_dev* d = new mb2_hits_dev();
        try {
            const int32_t* src[10] = {in->t_id, in->q_id, in->strand, in->start1, in->end1, in->start2, in->end2, in->score, in->nmatch, in->ncols};
            d->h.reserve(in->n ? in->n : 1);
            for (int c = 0; c < 10 && in->n; c++) {
                MB2_REQUIRE(src[c] != nullptr, MB2_ERR_INVALID_ARG, "hits_dev_upload: null column");
                MB2_CUDA(cudaMemcpyAsync(d->h.col[c].get(), src[c], in->n * sizeof(int32_t), cudaMemcpyHostToDevice, g_ctx.stream));
            }
            d->h.n = in->n; d->nt = nt; d->nq = nq;
            MB2_CUDA(cudaStreamSynchronize(g_ctx.stream));
        } catch (...) { delete d; throw; }
        *out = d;
    });
}

int mb2_hits_dev_download(const mb2_hits_dev* h, mb2_hits* out) {
    return guarded([&] {
        ensure_init();
        MB2_REQUIRE(h && out, MB2_ERR_INVALID_ARG, "hits_dev_download: null argument");
        download_hits(h->h, out);
    });
}

// ------------------------------------------------------------------------------------------ tandem mask
void mb2_default_tandem_params(mb2_tandem_params* p) {
    if (!p) return;
    TandemParams d;
    p->match = d.match; p->mismatch = d.mismatch; p->delta = d.delta; p->minscore = d.minscore; p->maxperiod = d.maxperiod;
}
static TandemParams to_tandem(const mb2_tandem_params* p) {
    TandemParams t;
    if (p) { t.match = p->match; t.mismatch = p->mismatch; t.delta = p->delta; t.minscore = p->minscore; t.maxperiod = p->maxperiod; }
    return t;
}
int mb2_tandem_mask(const mb2_genome* g, const int32_t* scaf, const int64_t* start, const int64_t* len, uint64_t n,
                    const mb2_tandem_params* p, uint64_t* masked) {
    return guarded([&] {
        MB2_REQUIRE(g && g->g, MB2_ERR_INVALID_ARG, "tandem_mask: null genome");
        tandem_mask(*g->g, scaf, start, len, n, to_tandem(p), 0, masked, nullptr);
    });
}
// copies the merged runs of every span into the library-owned arrays of `runs`
static void fill_runs(const std::vector<std::vector<std::pair<int64_t, int64_t>>>& iv, uint64_t n, mb2_tandem_runs* runs) {
    size_t total = 0;
    for (const auto& v : iv) total += v.size();
    runs->off = (uint64_t*)malloc((n + 1) * sizeof(uint64_t));
    runs->start = (int64_t*)malloc((total ? total : 1) * sizeof(int64_t));
    runs->end = (int64_t*)malloc((total ? total : 1) * sizeof(int64_t));
    MB2_REQUIRE(runs->off && runs->start && runs->end, MB2_ERR_INTERNAL, "tandem_mask_runs: host allocation failed");
    runs->n = n;
    runs->off[0] = 0;
    for (uint64_t k = 0; k < n; k++) {
        for (size_t t = 0; t < iv[k].size(); t++) {
            runs->start[runs->off[k] + t] = iv[k][t].first;
            runs->end[runs->off[k] + t] = iv[k][t].second;
        }
        runs->off[k + 1] = runs->off[k] + iv[k].size();
    }
}
static int tandem_mask_runs(const mb2_genome* g, const int32_t* scaf, const int64_t* start, const int64_t* len, uint64_t n,
                            const mb2_tandem_params* p, uint64_t store_budget, uint64_t* masked, mb2_tandem_runs* runs) {
    return guarded([&] {
        MB2_REQUIRE(g && g->g && runs, MB2_ERR_INVALID_ARG, "tandem_mask_runs: null argument");
        std::memset(runs, 0, sizeof(*runs));
        std::vector<std::vector<std::pair<int64_t, int64_t>>> iv;
        tandem_mask(*g->g, scaf, start, len, n, to_tandem(p), (size_t)store_budget, masked, &iv);
        fill_runs(iv, n, runs);
    });
}
int mb2_tandem_mask_runs(const mb2_genome* g, const int32_t* scaf, const int64_t* start, const int64_t* len, uint64_t n,
                         const mb2_tandem_params* p, uint64_t* masked, mb2_tandem_runs* runs) {
    return tandem_mask_runs(g, scaf, start, len, n, p, 0, masked, runs);
}
int mb2_test_tandem_mask(const mb2_genome* g, const int32_t* scaf, const int64_t* start, const int64_t* len, uint64_t n,
                         const mb2_tandem_params* p, uint64_t store_budget, uint64_t* masked, mb2_tandem_runs* runs) {
    return tandem_mask_runs(g, scaf, start, len, n, p, store_budget, masked, runs);
}
void mb2_free_tandem_runs(mb2_tandem_runs* r) {
    if (!r) return;
    free(r->off); free(r->start); free(r->end);
    std::memset(r, 0, sizeof(*r));
}
int mb2_tandem_report(const mb2_genome* g, const int32_t* scaf, const int64_t* start, const int64_t* len, uint64_t n,
                      const mb2_tandem_params* p, uint64_t* masked, mb2_tandem_runs* runs, mb2_tandem_repeats* rep) {
    return guarded([&] {
        MB2_REQUIRE(g && g->g && runs && rep, MB2_ERR_INVALID_ARG, "tandem_report: null argument");
        std::memset(runs, 0, sizeof(*runs));
        std::memset(rep, 0, sizeof(*rep));
        std::vector<std::vector<std::pair<int64_t, int64_t>>> iv;
        TandemReport tr;
        tandem_report(*g->g, scaf, start, len, n, to_tandem(p), masked, iv, tr);
        fill_runs(iv, n, runs);
        const size_t nr = tr.period.size();
        rep->period = (int32_t*)malloc((nr ? nr : 1) * sizeof(int32_t));
        rep->score = (int64_t*)malloc((nr ? nr : 1) * sizeof(int64_t));
        rep->matches = (uint64_t*)malloc((nr ? nr : 1) * sizeof(uint64_t));
        rep->count = (uint64_t*)malloc((nr ? 4 * nr : 1) * sizeof(uint64_t));
        rep->cons_off = (uint64_t*)malloc((nr + 1) * sizeof(uint64_t));
        rep->consensus = (char*)malloc(tr.consensus.size() + 1);
        MB2_REQUIRE(rep->period && rep->score && rep->matches && rep->count && rep->cons_off && rep->consensus, MB2_ERR_INTERNAL,
                    "tandem_report: host allocation failed");
        rep->n = nr;
        std::copy(tr.period.begin(), tr.period.end(), rep->period);
        std::copy(tr.score.begin(), tr.score.end(), rep->score);
        std::copy(tr.matches.begin(), tr.matches.end(), rep->matches);
        std::copy(tr.count.begin(), tr.count.end(), rep->count);
        std::copy(tr.cons_off.begin(), tr.cons_off.end(), rep->cons_off);
        std::copy(tr.consensus.begin(), tr.consensus.end(), rep->consensus);
    });
}
void mb2_free_tandem_report(mb2_tandem_repeats* r) {
    if (!r) return;
    free(r->period); free(r->score); free(r->matches); free(r->count); free(r->cons_off); free(r->consensus);
    std::memset(r, 0, sizeof(*r));
}

// ------------------------------------------------------------------------------------------ test hooks
int mb2_test_sort_u32(uint32_t* keys, uint32_t* vals, uint64_t n, int begin_bit, int end_bit) {
    return guarded([&] { test_sort<uint32_t>(keys, vals, n, begin_bit, end_bit); });
}
int mb2_test_sort_u64(uint64_t* keys, uint32_t* vals, uint64_t n, int begin_bit, int end_bit) {
    return guarded([&] { test_sort<uint64_t>(keys, vals, n, begin_bit, end_bit); });
}
int mb2_test_sort_u32_pair(uint32_t* keys_a, uint32_t* keys_b, uint64_t n, int begin_bit, int end_bit) {
    return guarded([&] {
        ensure_init();
        if (n == 0) return;
        MB2_REQUIRE(keys_a && keys_b, MB2_ERR_INVALID_ARG, "sort pair: null argument");
        DevBuf<uint32_t> a0(n), a1(n), b0(n), b1(n);
        MB2_CUDA(cudaMemcpyAsync(a0.get(), keys_a, n * sizeof(uint32_t), cudaMemcpyHostToDevice, g_ctx.stream));
        MB2_CUDA(cudaMemcpyAsync(b0.get(), keys_b, n * sizeof(uint32_t), cudaMemcpyHostToDevice, g_ctx.stream));
        NoVal* nv = nullptr;
        const int w = radix_sort_bits<uint32_t, NoVal>(a0.get(), a1.get(), nv, nv, n, begin_bit, end_bit, b0.get(), b1.get());
        MB2_CUDA(cudaMemcpyAsync(keys_a, w ? a1.get() : a0.get(), n * sizeof(uint32_t), cudaMemcpyDeviceToHost, g_ctx.stream));
        MB2_CUDA(cudaMemcpyAsync(keys_b, w ? b1.get() : b0.get(), n * sizeof(uint32_t), cudaMemcpyDeviceToHost, g_ctx.stream));
        MB2_CUDA(cudaStreamSynchronize(g_ctx.stream));
    });
}
int mb2_test_scan_u32(uint32_t* data, uint64_t n, uint32_t* total) {
    return guarded([&] {
        ensure_init();
        DevBuf<uint32_t> d(n), t(1);
        if (n) MB2_CUDA(cudaMemcpyAsync(d.get(), data, n * sizeof(uint32_t), cudaMemcpyHostToDevice, g_ctx.stream));
        exclusive_scan_u32(d.get(), d.get(), n, t.get());
        if (n) MB2_CUDA(cudaMemcpyAsync(data, d.get(), n * sizeof(uint32_t), cudaMemcpyDeviceToHost, g_ctx.stream));
        if (total) MB2_CUDA(cudaMemcpyAsync(total, t.get(), sizeof(uint32_t), cudaMemcpyDeviceToHost, g_ctx.stream));
        MB2_CUDA(cudaStreamSynchronize(g_ctx.stream));
    });
}


static char** dup_strings(const std::vector<std::string>& v) {
    char** a = (char**)malloc(sizeof(char*) * (v.size() + 1));
    for (size_t k = 0; k < v.size(); k++) {
        a[k] = (char*)malloc(v[k].size() + 1);
        memcpy(a[k], v[k].data(), v[k].size());
        a[k][v[k].size()] = 0;
    }
    a[v.size()] = nullptr;
    return a;
}
static void free_strings(char** a, size_t n) {
    if (!a) return;
    for (size_t k = 0; k < n; k++) free(a[k]);
    free(a);
}

int mb2_tab_project(const char* path, int nthreads, mb2_tab_hits* out) {
    return guarded([&] {
        MB2_REQUIRE(path && out, MB2_ERR_INVALID_ARG, "mb2_tab_project: null argument");
        memset(out, 0, sizeof(*out));
        TabHits t;
        tab_project_file(path, nthreads, t);
        const size_t n = t.chrom.size();
        out->n = n;
        out->nnames = (int32_t)t.names.size();
        out->names = dup_strings(t.names);
        if (n) {
            out->chrom = (int32_t*)malloc(n * sizeof(int32_t)); out->start = (int64_t*)malloc(n * sizeof(int64_t)); out->end = (int64_t*)malloc(n * sizeof(int64_t));
            MB2_REQUIRE(out->chrom && out->start && out->end, MB2_ERR_INTERNAL, "mb2_tab_project: out of memory");
            memcpy(out->chrom, t.chrom.data(), n * sizeof(int32_t));
            memcpy(out->start, t.start.data(), n * sizeof(int64_t));
            memcpy(out->end, t.end.data(), n * sizeof(int64_t));
        }
    });
}
void mb2_free_tab_hits(mb2_tab_hits* h) {
    if (!h) return;
    free(h->chrom); free(h->start); free(h->end);
    free_strings(h->names, (size_t)h->nnames);
    memset(h, 0, sizeof(*h));
}

int mb2_fasta_read(const char* path, int nthreads, mb2_fasta* out) {
    return guarded([&] {
        MB2_REQUIRE(path && out, MB2_ERR_INVALID_ARG, "mb2_fasta_read: null argument");
        memset(out, 0, sizeof(*out));
        FastaData f;
        fasta_read_file(path, nthreads, f);
        out->n = (int32_t)f.ids.size();
        out->ids = dup_strings(f.ids);
        out->headers = dup_strings(f.headers);
        out->off = (uint64_t*)malloc((f.off.size() + 1) * sizeof(uint64_t));
        if (f.off.empty()) out->off[0] = 0; else memcpy(out->off, f.off.data(), f.off.size() * sizeof(uint64_t));
        MB2_REQUIRE(out->off, MB2_ERR_INTERNAL, "mb2_fasta_read: out of memory");
        out->seq = f.seq ? f.seq : (uint8_t*)malloc(1);      // ownership moves to the caller-visible struct
        f.seq = nullptr;
    });
}
int mb2_fasta_split(const char* path, const char* outdir, int unique, int width, int nthreads, uint64_t* nfiles) {
    return guarded([&] {
        MB2_REQUIRE(path && outdir, MB2_ERR_INVALID_ARG, "mb2_fasta_split: null argument");
        if (nfiles) *nfiles = 0;
        const uint64_t k = fasta_split_file(path, outdir, unique != 0, width, nthreads);
        if (nfiles) *nfiles = k;
    });
}
void mb2_free_fasta(mb2_fasta* f) {
    if (!f) return;
    free_strings(f->ids, (size_t)f->n); free_strings(f->headers, (size_t)f->n);
    free(f->off); free(f->seq);
    memset(f, 0, sizeof(*f));
}

int mb2_format_tab(const int32_t* t_id, const int32_t* q_id, const int32_t* strand, const int32_t* start1, const int32_t* end1,
                   const int32_t* start2, const int32_t* end2, const int32_t* score, const int32_t* nmatch, const int32_t* ncols,
                   uint64_t n, const char* const* tnames, int nt, const char* const* qnames, int nq, double min_len, double min_idt,
                   mb2_tab_text* out) {
    return guarded([&] {
        MB2_REQUIRE(out && tnames && qnames, MB2_ERR_INVALID_ARG, "mb2_format_tab: null argument");
        memset(out, 0, sizeof(*out));
        TabText t;
        format_tab_blocks(t_id, q_id, strand, start1, end1, start2, end2, score, nmatch, ncols, n, tnames, nt, qnames, nq, min_len, min_idt, t);
        const size_t nb = t.t_id.size();
        out->nblocks = nb; out->nbytes = t.text.size();
        out->text = (char*)malloc(t.text.size() + 1);
        out->t_id = (int32_t*)malloc((nb + 1) * sizeof(int32_t)); out->q_id = (int32_t*)malloc((nb + 1) * sizeof(int32_t));
        out->off = (uint64_t*)malloc((nb + 1) * sizeof(uint64_t)); out->nrows = (uint32_t*)malloc((nb + 1) * sizeof(uint32_t));
        MB2_REQUIRE(out->text && out->t_id && out->q_id && out->off && out->nrows, MB2_ERR_INTERNAL, "mb2_format_tab: out of memory");
        memcpy(out->text, t.text.data(), t.text.size()); out->text[t.text.size()] = 0;
        if (nb) {
            memcpy(out->t_id, t.t_id.data(), nb * sizeof(int32_t)); memcpy(out->q_id, t.q_id.data(), nb * sizeof(int32_t));
            memcpy(out->nrows, t.nrows.data(), nb * sizeof(uint32_t));
        }
        memcpy(out->off, t.off.data(), t.off.size() * sizeof(uint64_t));
    });
}
void mb2_free_tab_text(mb2_tab_text* t) {
    if (!t) return;
    free(t->text); free(t->t_id); free(t->q_id); free(t->off); free(t->nrows);
    memset(t, 0, sizeof(*t));
}

int mb2_map_gff(const char* tab_path, const char* prefix, double min_len, double min_idt, const char* ftype, int nthreads, mb2_text* out) {
    return guarded([&] {
        MB2_REQUIRE(tab_path && out, MB2_ERR_INVALID_ARG, "mb2_map_gff: null argument");
        memset(out, 0, sizeof(*out));
        std::string text;
        out->nrows = map_gff_rows(tab_path, prefix, min_len, min_idt, ftype, nthreads, text);
        out->nbytes = text.size();
        out->text = (char*)malloc(text.size() + 1);
        MB2_REQUIRE(out->text, MB2_ERR_INTERNAL, "mb2_map_gff: out of memory");
        memcpy(out->text, text.data(), text.size()); out->text[text.size()] = 0;
    });
}
int mb2_format_gff(const int32_t* chrom, const int32_t* start, const int32_t* end, uint64_t n, const char* const* names,
                   int nnames, const char* source, const char* label, const char* prefix, uint64_t first_id, int nthreads, mb2_text* out) {
    return guarded([&] {
        MB2_REQUIRE(out && source && label && prefix && (nnames == 0 || names), MB2_ERR_INVALID_ARG, "mb2_format_gff: null argument");
        MB2_REQUIRE(n == 0 || (chrom && start && end), MB2_ERR_INVALID_ARG, "mb2_format_gff: null segment arrays");
        memset(out, 0, sizeof(*out));
        std::string text;
        out->nrows = format_segment_gff(chrom, start, end, n, names, nnames, source, label, prefix, first_id, nthreads, text);
        out->nbytes = text.size();
        out->text = (char*)malloc(text.size() + 1);
        MB2_REQUIRE(out->text, MB2_ERR_INTERNAL, "mb2_format_gff: out of memory");
        memcpy(out->text, text.data(), text.size()); out->text[text.size()] = 0;
    });
}
void mb2_free_text(mb2_text* t) {
    if (!t) return;
    free(t->text);
    memset(t, 0, sizeof(*t));
}
}  // extern "C"
