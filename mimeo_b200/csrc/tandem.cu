// tandem.cu -- the tandem-repeat mask of `mimeo map --maxtandem` (DESIGN §2 T1-T4, kernel in tandem_warp.cuh): span
// validation, dedupe, scheduling (one warp per distinct span, longest first) and the storage bound; and the report of
// `--reportTRF` on the masked runs (DESIGN §2 R1-R6, kernel in tandem_report_warp.cuh), with the same scheduling per
// distinct run.
#include <algorithm>
#include <numeric>
#include <tuple>

#include "internal.cuh"
#include "seq.cuh"
#include "tandem_report_warp.cuh"
#include "tandem_warp.cuh"
#include "mimeo_b200.h"

namespace mb2 {

namespace {
constexpr int WARPS = 4;
constexpr size_t DEFAULT_STORE_BUDGET = (size_t)512 << 20;

template <int K, typename ST>
__global__ void __launch_bounds__(WARPS * 32) tandem_mask_kernel(const uint8_t* __restrict__ codes, const uint64_t* __restrict__ gstart,
                                                                 const int32_t* __restrict__ len, const uint64_t* __restrict__ store_off,
                                                                 uint32_t nspans, tw::Params p, ST* store, uint64_t* masked,
                                                                 const uint64_t* __restrict__ iv_off, int64_t* iv_start, int64_t* iv_end,
                                                                 uint32_t* iv_n, uint32_t* next) {
    __shared__ int ring[WARPS][tw::RING];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (;;) {
        uint32_t k = 0;
        if (lane == 0) k = atomicAdd(next, 1u);
        k = __shfl_sync(0xffffffffu, k, 0);
        if (k >= nspans) break;
        tw::Out o;
        o.masked = masked + k;
        o.iv_start = iv_start ? iv_start + iv_off[k] : nullptr;
        o.iv_end = iv_end ? iv_end + iv_off[k] : nullptr;
        o.iv_cap = iv_start ? (uint32_t)(iv_off[k + 1] - iv_off[k]) : 0u;
        o.iv_n = iv_n ? iv_n + k : nullptr;
        tw::tandem_warp<K, ST>(codes + gstart[k], len[k], p, store + store_off[k], ring[w], o);
    }
}

template <int K, typename ST>
void launch_batch(const Genome& g, const std::vector<uint64_t>& gs, const std::vector<int32_t>& ln, const std::vector<uint64_t>& so,
                  size_t store_elems, const tw::Params& p, uint64_t* h_masked, const std::vector<uint64_t>* iv_off,
                  std::vector<int64_t>* iv_s, std::vector<int64_t>* iv_e, std::vector<uint32_t>* iv_n) {
    const size_t n = gs.size();
    cudaStream_t s = ctx().stream;
    DevBuf<uint64_t> d_gs(n), d_so(n), d_m(n);
    DevBuf<int32_t> d_len(n);
    DevBuf<ST> d_store(store_elems ? store_elems : 1);
    DevBuf<uint32_t> d_next(1), d_ivn(iv_off ? n : 0);
    DevBuf<uint64_t> d_ivoff(iv_off ? n + 1 : 0);
    const size_t niv = iv_off ? (*iv_off)[n] : 0;
    DevBuf<int64_t> d_ivs(niv ? niv : (iv_off ? 1 : 0)), d_ive(niv ? niv : (iv_off ? 1 : 0));
    MB2_CUDA(cudaMemcpyAsync(d_gs.get(), gs.data(), n * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    MB2_CUDA(cudaMemcpyAsync(d_so.get(), so.data(), n * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    MB2_CUDA(cudaMemcpyAsync(d_len.get(), ln.data(), n * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    MB2_CUDA(cudaMemsetAsync(d_next.get(), 0, sizeof(uint32_t), s));
    if (iv_off) MB2_CUDA(cudaMemcpyAsync(d_ivoff.get(), iv_off->data(), (n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    const unsigned blocks = std::min<unsigned>(cdiv(n, WARPS), (unsigned)ctx().sm_count * 16u);
    {
        ProfScope prof("tandem_mask");
        launch(tandem_mask_kernel<K, ST>, dim3(blocks), dim3(WARPS * 32), 0, g.codes.get(), d_gs.get(), d_len.get(), d_so.get(), (uint32_t)n, p,
               d_store.get(), d_m.get(), iv_off ? d_ivoff.get() : nullptr, iv_off ? d_ivs.get() : nullptr, iv_off ? d_ive.get() : nullptr,
               iv_off ? d_ivn.get() : nullptr, d_next.get());
    }
    MB2_CUDA(cudaMemcpyAsync(h_masked, d_m.get(), n * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    if (iv_off) {
        iv_s->resize(niv); iv_e->resize(niv); iv_n->resize(n);
        if (niv) {
            MB2_CUDA(cudaMemcpyAsync(iv_s->data(), d_ivs.get(), niv * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
            MB2_CUDA(cudaMemcpyAsync(iv_e->data(), d_ive.get(), niv * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
        }
        MB2_CUDA(cudaMemcpyAsync(iv_n->data(), d_ivn.get(), n * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    }
    MB2_CUDA(cudaStreamSynchronize(s));
}

template <int K, typename ST>
void run_layout(const Genome& g, const std::vector<uint64_t>& ugs, const std::vector<int32_t>& ulen, const std::vector<size_t>& order,
                const tw::Params& p, size_t budget, std::vector<uint64_t>& um, std::vector<std::vector<std::pair<int64_t, int64_t>>>* uiv) {
    // batches of the spans in `order` (longest first) whose stored anti-diagonals fit the budget; a span larger than the
    // budget alone is a batch of its own
    size_t b0 = 0;
    while (b0 < order.size()) {
        std::vector<uint64_t> gs, so, ivoff{0};
        std::vector<int32_t> ln;
        size_t elems = 0, b1 = b0;
        while (b1 < order.size()) {
            const int32_t n = ulen[order[b1]];
            const size_t e = (size_t)(2 * (int64_t)n - 3) * 16 * K;
            if (b1 > b0 && (elems + e) * sizeof(ST) > budget) break;
            gs.push_back(ugs[order[b1]]); ln.push_back(n); so.push_back(elems);
            ivoff.push_back(ivoff.back() + (uint64_t)n / 2 + 1);
            elems += e;
            b1++;
        }
        std::vector<uint64_t> m(b1 - b0);
        std::vector<int64_t> ivs, ive;
        std::vector<uint32_t> ivn;
        launch_batch<K, ST>(g, gs, ln, so, elems, p, m.data(), uiv ? &ivoff : nullptr, &ivs, &ive, &ivn);
        for (size_t x = b0; x < b1; x++) {
            um[order[x]] = m[x - b0];
            if (uiv) {
                auto& v = (*uiv)[order[x]];
                const uint64_t o = ivoff[x - b0];
                MB2_REQUIRE(ivn[x - b0] <= ivoff[x - b0 + 1] - o, MB2_ERR_INTERNAL, "tandem_mask: interval capacity exceeded");
                for (uint32_t t = 0; t < ivn[x - b0]; t++) v.emplace_back(ivs[o + t], ive[o + t]);
            }
        }
        b0 = b1;
    }
}
template <int NT>
__global__ void __launch_bounds__(WARPS * 32) tandem_report_kernel(const uint8_t* __restrict__ codes, const uint64_t* __restrict__ gstart,
                                                                   const int32_t* __restrict__ len, uint32_t nruns, tr::Params p,
                                                                   tr::Out o, uint32_t* next) {
    __shared__ tr::Scratch sh[WARPS];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (;;) {
        uint32_t k = 0;
        if (lane == 0) k = atomicAdd(next, 1u);
        k = __shfl_sync(0xffffffffu, k, 0);
        if (k >= nruns) break;
        tr::report_warp<NT>(codes + gstart[k], len[k], p, sh[w], o, k);
    }
}
}  // namespace

void tandem_mask(const Genome& g, const int32_t* scaf, const int64_t* start, const int64_t* len, uint64_t n, const TandemParams& tp,
                 size_t store_budget, uint64_t* masked, std::vector<std::vector<std::pair<int64_t, int64_t>>>* intervals) {
    MB2_REQUIRE(tp.match >= 1 && tp.mismatch >= 0 && tp.delta >= 0 && tp.minscore >= 1, MB2_ERR_INVALID_ARG,
                "tandem_mask: need match >= 1, mismatch >= 0, delta >= 0, minscore >= 1");
    MB2_REQUIRE(tp.maxperiod >= 1 && tp.maxperiod <= tw::MAX_P, MB2_ERR_INVALID_ARG,
                "tandem_mask: maxperiod must be in 1.." + std::to_string(tw::MAX_P));
    MB2_REQUIRE((int64_t)tp.minscore + tp.mismatch <= 65535, MB2_ERR_INVALID_ARG,
                "tandem_mask: minscore + mismatch must be at most 65535 (16-bit storage of the clamped backward scores)");
    MB2_REQUIRE(n == 0 || (scaf && start && len && masked), MB2_ERR_INVALID_ARG, "tandem_mask: null argument");
    // distinct spans (map hits of many B loci share A spans); key order, then longest first
    std::vector<size_t> idx(n);
    std::iota(idx.begin(), idx.end(), 0);
    int64_t maxlen = 0;
    for (uint64_t k = 0; k < n; k++) {
        MB2_REQUIRE(scaf[k] >= 0 && scaf[k] < g.nscaf, MB2_ERR_INVALID_ARG, "tandem_mask: scaffold index out of range (span " + std::to_string(k) + ")");
        MB2_REQUIRE(start[k] >= 0 && len[k] >= 0 && start[k] + len[k] <= (int64_t)g.len[scaf[k]], MB2_ERR_INVALID_ARG,
                    "tandem_mask: span " + std::to_string(k) + " is not inside its scaffold");
        maxlen = std::max(maxlen, len[k]);
    }
    MB2_REQUIRE((int64_t)tp.match * (maxlen + 1) + tp.minscore + tp.mismatch < ((int64_t)1 << 31), MB2_ERR_INVALID_ARG,
                "tandem_mask: match * span length overflows the 32-bit scores");
    auto key = [&](size_t k) { return std::make_tuple(scaf[k], start[k], len[k]); };
    std::sort(idx.begin(), idx.end(), [&](size_t a, size_t b) { return key(a) < key(b); });
    std::vector<uint64_t> ugs;
    std::vector<int32_t> ulen;
    std::vector<size_t> uof(n);
    for (size_t x = 0; x < n; x++) {
        if (x == 0 || key(idx[x]) != key(idx[x - 1])) {
            ugs.push_back((uint64_t)g.off[scaf[idx[x]]] + (uint64_t)start[idx[x]]);
            ulen.push_back((int32_t)len[idx[x]]);
        }
        uof[idx[x]] = ugs.size() - 1;
    }
    const size_t nu = ugs.size();
    std::vector<size_t> order;
    for (size_t u = 0; u < nu; u++) if (ulen[u] >= 2) order.push_back(u);        // shorter spans hold no pair
    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return ulen[a] > ulen[b]; });
    std::vector<uint64_t> um(nu, 0);
    std::vector<std::vector<std::pair<int64_t, int64_t>>> uiv(intervals ? nu : 0);
    auto* uivp = intervals ? &uiv : nullptr;
    const tw::Params p{tp.match, tp.mismatch, tp.delta, tp.minscore, tp.maxperiod};
    const bool wide = tp.minscore + tp.mismatch > 255;
    const size_t budget = store_budget ? store_budget : DEFAULT_STORE_BUDGET;
    if (!order.empty()) {
        ensure_init();
        if (tp.maxperiod <= 64) {
            if (wide) run_layout<2, uint16_t>(g, ugs, ulen, order, p, budget, um, uivp); else run_layout<2, uint8_t>(g, ugs, ulen, order, p, budget, um, uivp);
        } else if (tp.maxperiod <= 128) {
            if (wide) run_layout<4, uint16_t>(g, ugs, ulen, order, p, budget, um, uivp); else run_layout<4, uint8_t>(g, ugs, ulen, order, p, budget, um, uivp);
        } else {
            if (wide) run_layout<8, uint16_t>(g, ugs, ulen, order, p, budget, um, uivp); else run_layout<8, uint8_t>(g, ugs, ulen, order, p, budget, um, uivp);
        }
    }
    if (intervals) intervals->assign(n, {});
    for (uint64_t k = 0; k < n; k++) {
        masked[k] = um[uof[k]];
        if (intervals) (*intervals)[k] = uiv[uof[k]];
    }
}

void tandem_report(const Genome& g, const int32_t* scaf, const int64_t* start, const int64_t* len, uint64_t n, const TandemParams& tp,
                   uint64_t* masked, std::vector<std::vector<std::pair<int64_t, int64_t>>>& intervals, TandemReport& rep) {
    tandem_mask(g, scaf, start, len, n, tp, 0, masked, &intervals);
    // rows = runs in span order; distinct runs by (genome offset, length), longest first
    std::vector<std::pair<uint64_t, int32_t>> key;
    for (uint64_t k = 0; k < n; k++)
        for (const auto& r : intervals[k]) {
            MB2_REQUIRE(r.second - r.first >= 1, MB2_ERR_INTERNAL, "tandem_report: masked run shorter than 2");
            key.emplace_back((uint64_t)g.off[scaf[k]] + (uint64_t)(start[k] + r.first), (int32_t)(r.second - r.first + 1));
        }
    const size_t nrow = key.size();
    std::vector<size_t> idx(nrow);
    std::iota(idx.begin(), idx.end(), 0);
    std::sort(idx.begin(), idx.end(), [&](size_t a, size_t b) { return key[a] < key[b]; });
    std::vector<uint64_t> ugs;
    std::vector<int32_t> ulen;
    std::vector<size_t> uof(nrow);
    for (size_t x = 0; x < nrow; x++) {
        if (x == 0 || key[idx[x]] != key[idx[x - 1]]) { ugs.push_back(key[idx[x]].first); ulen.push_back(key[idx[x]].second); }
        uof[idx[x]] = ugs.size() - 1;
    }
    const size_t nu = ugs.size();
    std::vector<size_t> order(nu);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return ulen[a] > ulen[b]; });
    std::vector<uint64_t> gs(nu), coff(nu + 1, 0);
    std::vector<int32_t> ln(nu);
    for (size_t x = 0; x < nu; x++) {
        gs[x] = ugs[order[x]];
        ln[x] = ulen[order[x]];
        coff[x + 1] = coff[x] + (uint64_t)std::min(tp.maxperiod, ln[x] - 1);
    }
    std::vector<int32_t> per(nu);
    std::vector<int64_t> sc(nu);
    std::vector<uint64_t> mt(nu), cnt(4 * nu);
    std::string cons(coff[nu], 'N');
    if (nu) {
        ensure_init();
        cudaStream_t s = ctx().stream;
        DevBuf<uint64_t> d_gs(nu), d_coff(nu), d_mt(nu), d_cnt(4 * nu);
        DevBuf<int32_t> d_len(nu), d_per(nu);
        DevBuf<int64_t> d_sc(nu);
        DevBuf<char> d_cons(coff[nu]);
        DevBuf<uint32_t> d_next(1);
        MB2_CUDA(cudaMemcpyAsync(d_gs.get(), gs.data(), nu * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
        MB2_CUDA(cudaMemcpyAsync(d_coff.get(), coff.data(), nu * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
        MB2_CUDA(cudaMemcpyAsync(d_len.get(), ln.data(), nu * sizeof(int32_t), cudaMemcpyHostToDevice, s));
        MB2_CUDA(cudaMemsetAsync(d_next.get(), 0, sizeof(uint32_t), s));
        const tr::Params p{tp.match, tp.mismatch, tp.maxperiod};
        const unsigned blocks = std::min<unsigned>(cdiv(nu, WARPS), (unsigned)ctx().sm_count * 16u);
        {
            ProfScope prof("tandem_report");
            auto* kernel = tp.maxperiod <= 32 ? tandem_report_kernel<1> : tp.maxperiod <= 64 ? tandem_report_kernel<2>
                         : tp.maxperiod <= 128 ? tandem_report_kernel<4> : tandem_report_kernel<8>;
            const tr::Out o{d_per.get(), d_sc.get(), d_mt.get(), d_cnt.get(), d_coff.get(), d_cons.get()};
            launch(kernel, dim3(blocks), dim3(WARPS * 32), 0, g.codes.get(), d_gs.get(), d_len.get(), (uint32_t)nu, p, o, d_next.get());
        }
        MB2_CUDA(cudaMemcpyAsync(per.data(), d_per.get(), nu * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        MB2_CUDA(cudaMemcpyAsync(sc.data(), d_sc.get(), nu * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
        MB2_CUDA(cudaMemcpyAsync(mt.data(), d_mt.get(), nu * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
        MB2_CUDA(cudaMemcpyAsync(cnt.data(), d_cnt.get(), 4 * nu * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
        MB2_CUDA(cudaMemcpyAsync(&cons[0], d_cons.get(), coff[nu], cudaMemcpyDeviceToHost, s));
        MB2_CUDA(cudaStreamSynchronize(s));
    }
    std::vector<size_t> slot(nu);                      // distinct run -> its launch slot
    for (size_t x = 0; x < nu; x++) slot[order[x]] = x;
    rep = TandemReport{};
    rep.cons_off.push_back(0);
    for (size_t r = 0; r < nrow; r++) {
        const size_t x = slot[uof[r]];
        MB2_REQUIRE(per[x] >= 1 && per[x] <= ln[x] - 1 && per[x] <= tp.maxperiod, MB2_ERR_INTERNAL, "tandem_report: period out of range");
        rep.period.push_back(per[x]);
        rep.score.push_back(sc[x]);
        rep.matches.push_back(mt[x]);
        for (int b = 0; b < 4; b++) rep.count.push_back(cnt[4 * x + b]);
        rep.consensus.append(cons, coff[x], (size_t)per[x]);
        rep.cons_off.push_back(rep.consensus.size());
    }
}

}  // namespace mb2
