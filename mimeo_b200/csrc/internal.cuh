// internal.cuh -- declarations shared between the translation units of libmimeo_b200.
#pragma once
#include <vector>

#include "common.cuh"

namespace mb2 {

constexpr int CNT_N_DECL = 16;

// ---- coverage.cu
struct CoverageResult {
    DevBuf<int32_t> chrom, start, end;   // library-owned result (unused when the caller supplies its own arrays)
    uint64_t n = 0;
    // caller-owned device arrays of ext_cap elements each: the result is written there instead; more segments than that
    // -> Error(-6) with n = the number needed and nothing written
    int32_t *ext_chrom = nullptr, *ext_start = nullptr, *ext_end = nullptr;
    uint64_t ext_cap = 0;
};
void coverage_segments_device(const int32_t* d_chrom, const int32_t* d_start, const int32_t* d_end, uint64_t nhits,
                              const int64_t* h_sizes, int nchrom, int min_cov, int min_len, CoverageResult& res);

void coverage_release_scratch();   // frees the stage's grow-only device scratch (kept between calls)
void gapped_release_scratch();     // frees the gapped stage's trace pool (kept between calls)

// ---- alignment half
struct Genome;
struct AlignParams {   // LASTZ defaults for mimeo's command line (SURVEY 9.1)
    int hspthresh = 3000, xdrop = 910, ydrop = 9400, gap_open = 400, gap_extend = 30, gappedthresh = 3000;
    int entropy = 1, chain = 1, gapped = 1, transition = 1;
};
// y-drop and gap penalties the 16-bit gapped extension kernel supports (ydrop_warp.cuh)
constexpr int YDROP_MIN = 1000, YDROP_MAX = 20000, GAP_OPEN_MAX = 2000, GAP_EXTEND_MIN = 10, GAP_EXTEND_MAX = 60;

// genome.cu
Genome* genome_from_ascii(const uint8_t* const* seqs, const uint64_t* lens, int n);
Genome* genome_revcomp(const Genome& src);
Genome* genome_both_strands(const Genome& src);
void genome_decode(const Genome& g, int scaf, uint8_t* h_out);

// seed.cu
struct SeedTable {
    DevBuf<uint32_t> off;   // 2^24+1 bucket offsets
    DevBuf<uint32_t> pos;   // target positions sorted by seed key
    uint32_t p_lo = 0, p_hi = 0;
};
void build_seed_table(const Genome& T, uint32_t p_lo, uint32_t p_hi, SeedTable& tab);
void seed_scan(const Genome& T, const Genome& Q, const SeedTable& tab, uint32_t q_lo, uint32_t q_hi, const AlignParams& p,
               uint64_t* surv, uint32_t surv_cap, unsigned long long* counters);

// hsp.cu : survivors -> kept HSPs in canonical order (tile, s1, s2, len); coordinates local to the scaffolds
struct HspSet {
    DevBuf<uint32_t> tile;              // tscaf * nQ + qscaf
    DevBuf<int32_t> s1, s2, len, score;
    uint32_t n = 0;
};
// d_same_q (device, may be null): per target scaffold the query scaffold holding the identical sequence, or -1; enables
// the closed form of the trivial self-diagonal HSP (results do not depend on it)
void find_hsps(const Genome& T, const Genome& Q, uint64_t* surv0, uint64_t* surv1, uint32_t nsurv, const AlignParams& p,
               HspSet& out, unsigned long long* counters, const int32_t* d_same_q = nullptr);
// host map target scaffold -> identical query scaffold (-1 if none): explicit hint, or inferred when Q was built from T
std::vector<int32_t> same_scaffold_map(const Genome& T, const Genome& Q, const int32_t* h_same_q);

// chain.cu : flags the members of the best collinear chain of every tile
void chain_hsps(const HspSet& h, int len_bits, int tile_bits, DevBuf<uint8_t>& in_chain);

// gapped.cu
struct AlnSet {   // strand-local, scaffold-local, 0-based half-open
    DevBuf<uint32_t> tile;
    DevBuf<int32_t> s1, e1, s2, e2, score, nmatch, ncols;
    uint32_t n = 0;
};
void gapped_extend(const Genome& T, const Genome& Q, const HspSet& h, const DevBuf<uint8_t>& in_chain, const AlignParams& p,
                   const int32_t* h_same_q, AlnSet& out, unsigned long long* counters);

// hits.cu : the hit table in HBM (LASTZ's output columns, one row per alignment)
struct HitCols { int32_t* c[10]; };     // t_id, q_id, strand, start1, end1, start2+, end2+, score, nmatch, ncols
struct DevHits {
    DevBuf<int32_t> col[10];
    size_t n = 0, cap = 0;
    unsigned long long stats[CNT_N_DECL] = {0};
    void reserve(size_t want);
    HitCols view() const;
    void append(const AlnSet& a, const Genome& Q, int nq, int strands);    // strand-local alignments -> output columns
};
void hits_filter_sort(DevHits& h, double min_len, double min_idt, bool map_rule, int nt, int nq);
void hits_coverage(const DevHits& h, int which, const int64_t* h_sizes, int nchrom, int min_cov, int min_len, CoverageResult& res);

// align.cu
void align_hsps(const Genome& T, const Genome& Q, const AlignParams& p, HspSet& hsps, unsigned long long* h_counters);
// test hook (stage a only): survivors of one scan of the whole query as (diagonal + Q.G) << 32 | query position, in scan
// order; init_cap = initial survivor capacity (0 = default); h_counters[0..3] = survivors, seed hits, leaders, stage-1 cells
void scan_survivors(const Genome& T, const Genome& Q, const AlignParams& p, uint64_t init_cap, std::vector<uint64_t>& surv,
                    unsigned long long* h_counters);

// whole pipeline for one (strand-oriented) query genome; rows are appended to `out` (nq, strands: see DevHits::append)
void align_strand(const Genome& T, const Genome& Q, const AlignParams& p, const int32_t* h_same_q, DevHits& out, int nq, int strands,
                  unsigned long long* h_counters);

// hostio.cu : native text ingest (no device work)
struct TabHits {                       // BED projection of a .tab file: columns 1, 3, 4 of every non-'#' line
    std::vector<int32_t> chrom;        // index into names
    std::vector<int64_t> start, end;
    std::vector<std::string> names;    // distinct column-1 values in order of first appearance
};
void tab_project_file(const char* path, int nthreads, TabHits& out);
struct FastaData {
    std::vector<std::string> ids, headers;
    std::vector<uint64_t> off;         // record r = seq[off[r], off[r+1])
    uint8_t* seq = nullptr;            // all sequences, line breaks and blanks removed (malloc; the caller takes it or it is freed)
    uint64_t total = 0;
    FastaData() = default;
    FastaData(const FastaData&) = delete;
    FastaData& operator=(const FastaData&) = delete;
    ~FastaData() { free(seq); }
};
void fasta_read_file(const char* path, int nthreads, FastaData& out);
// one <outdir>/<id>.fa per record (splitFasta, utils.py:274-309); returns the number of files written; Error(-7, id) on a repeated id
uint64_t fasta_split_file(const char* path, const char* outdir, bool unique, int width, int nthreads);

struct TabText {                       // filtered, sorted .tab rows grouped by (t_id, q_id) block
    std::string text;                  // all rows, blocks back to back
    std::vector<int32_t> t_id, q_id;   // per block
    std::vector<uint64_t> off;         // nblocks + 1 byte offsets into text
    std::vector<uint32_t> nrows;       // per block
};
void format_tab_blocks(const int32_t* t_id, const int32_t* q_id, const int32_t* strand, const int32_t* start1, const int32_t* end1,
                       const int32_t* start2, const int32_t* end2, const int32_t* score, const int32_t* nmatch, const int32_t* ncols,
                       uint64_t n, const char* const* tnames, int nt, const char* const* qnames, int nq, double min_len, double min_idt,
                       TabText& out);

// GFF3 feature rows of `mimeo map` straight from the .tab file; returns the number of rows
uint64_t map_gff_rows(const char* path, const char* prefix, double min_len, double min_idt, const char* ftype, int nthreads, std::string& out);

// GFF3 feature rows of one coverage block (the awk formatter of wrappers.py:1166-1173); returns the number of rows
uint64_t format_segment_gff(const int32_t* chrom, const int32_t* start, const int32_t* end, uint64_t n, const char* const* names,
                            int nnames, const char* source, const char* label, const char* prefix, uint64_t first_id, int nthreads,
                            std::string& out);

// tandem.cu : the tandem-repeat mask of `mimeo map --maxtandem` (m per span; intervals: merged masked runs, span-local
// and closed, for the test hook). store_budget: bytes of stored backward scores per launch, 0 = default.
struct TandemParams { int match = 2, mismatch = 7, delta = 7, minscore = 50, maxperiod = 50; };
void tandem_mask(const Genome& g, const int32_t* scaf, const int64_t* start, const int64_t* len, uint64_t n, const TandemParams& p,
                 size_t store_budget, uint64_t* masked, std::vector<std::vector<std::pair<int64_t, int64_t>>>* intervals);
// the report of `--reportTRF` (DESIGN §2, R1-R6): tandem_mask with intervals, then one row per run of every span, in span
// order and ascending within a span; row r's consensus is consensus[cons_off[r], cons_off[r+1])
struct TandemReport {
    std::vector<int32_t> period;
    std::vector<int64_t> score;
    std::vector<uint64_t> matches, count, cons_off;    // count: 4 per row (A, C, G, T); cons_off: rows + 1
    std::string consensus;
};
void tandem_report(const Genome& g, const int32_t* scaf, const int64_t* start, const int64_t* len, uint64_t n, const TandemParams& p,
                   uint64_t* masked, std::vector<std::vector<std::pair<int64_t, int64_t>>>& intervals, TandemReport& rep);

// counters layout (device, unsigned long long[16])
enum { CNT_SURV = 0, CNT_SEED_HITS = 1, CNT_LEADERS = 2, CNT_S1_CELLS = 3, CNT_HSPS = 4, CNT_EXTENDED = 5, CNT_S2_CELLS = 6,
       CNT_GAPPED_CELLS = 7, CNT_ALNS = 8, CNT_ANCHORS = 9, CNT_ERR = 10, CNT_WORK = 11, CNT_N = 16 };

}  // namespace mb2
