/*
 * mimeo_b200.h -- C ABI of libmimeo_b200.so, the B200 (sm_100a) implementation of mimeo's
 * alignment-to-annotation hot path.
 *
 * The reference (Adamtaranto/mimeo) has NO FFI for this path: its "plugin interface" is two
 * executable-path flags whose argv contracts are literal strings inside generated bash
 *   --lzpath   -> `lastz T.fa Q.fa --entropy --format=general:... --chain --gapped ...`
 *                 (src/mimeo/wrappers.py:1025-1037 self, 786-798 x, 645-653 map)
 *   --bedtools -> `bedtools genomecov -bg -i BED -g LENS` / `bedtools merge -i BED`
 *                 (src/mimeo/wrappers.py:1131-1150, 847-866, 1223-1250)
 * executed by utils.run_cmd (src/mimeo/utils.py:213-254). Each entry point below names the piece
 * of that script it replaces. Plain pointers and sizes only; no torch types. All functions return
 * 0 on success or a negative error code, with the message available from mb2_last_error().
 *
 * Threading: one process per GPU, calls are not re-entrant; every kernel is launched on the
 * library's own stream (mb2_stream()).
 */
#ifndef MIMEO_B200_H
#define MIMEO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define MB2_API __attribute__((visibility("default")))
#else
#define MB2_API
#endif

#define MB2_OK 0
#define MB2_ERR_INVALID_ARG (-2)
#define MB2_ERR_TOO_LARGE (-3)
#define MB2_ERR_BAD_HIT (-4)
#define MB2_ERR_INTERNAL (-5)
#define MB2_ERR_CAPACITY (-6)   /* caller-provided output buffers too small; the needed size is reported */
#define MB2_ERR_CUDA (-100)

/* ---- library / device -------------------------------------------------------------------- */
/* Bind the calling process to one CUDA device and create the library stream + memory pool.
 * Replaces nothing in the reference (it has no device); called once by the host layer that
 * replaces utils.run_cmd (utils.py:213). */
MB2_API int mb2_init(int device);
MB2_API void mb2_shutdown(void);
MB2_API const char* mb2_last_error(void);
/* cudaStream_t of the library as an opaque pointer (for CUDA-event timing by the caller). */
MB2_API void* mb2_stream(void);
/* Number of kernels of this library launched since mb2_init (the bench's `gpu_launches`). */
MB2_API unsigned long long mb2_launch_count(void);
MB2_API int mb2_sm_count(void);
/* Block the host until the library stream is idle. */
MB2_API int mb2_sync(void);

/* Per-kernel timing with CUDA events on the library stream (used by bench.py for the roofline
 * of the dominant kernel). mb2_prof_enable(1) starts recording; mb2_prof_get() synchronises and
 * returns accumulated milliseconds and launch count for a kernel tag (e.g. "cov_tile"), 0/0 if
 * the tag never ran; mb2_prof_reset() clears the accumulators. */
MB2_API int mb2_prof_enable(int on);
MB2_API int mb2_prof_get(const char* tag, double* ms_total, unsigned long long* count);
MB2_API int mb2_prof_reset(void);

/* ---- (d) coverage -> threshold -> merged segments ----------------------------------------- */
/* Output of the coverage stage: merged runs of depth >= min_cov with end-start >= min_len, ordered
 * by scaffold index then start. Coordinates are the raw BED-style numbers the reference prints into
 * GFF3 columns 4/5 (wrappers.py:1169-1171). Arrays are owned by the library; free with
 * mb2_free_segments. `on_device` tells whether the three arrays are host or device memory. */
typedef struct mb2_segments {
    int32_t* chrom;
    int32_t* start;
    int32_t* end;
    uint64_t n;
    int on_device;
} mb2_segments;

/* Replaces: awk BED projection + sort + `bedtools genomecov -bg` + awk '0+$4 >= cov' + sort +
 * `bedtools merge` + awk minLen filter  (wrappers.py:1120-1167; x: 827-885; self intra: 1201-1258).
 * Inputs are HOST arrays: one (scaffold index, start1, end1) triple per non-'#' line of the .tab file
 * (columns 1,3,4), scaffold sizes as in A_gen_lens.txt (utils.py:552-555), indexed in the byte order
 * `sort -k 1,1` produces. Host->device and device->host copies happen inside the call. */
MB2_API int mb2_coverage_segments(const int32_t* chrom, const int32_t* start, const int32_t* end, uint64_t nhits,
                          const int64_t* chrom_sizes, int nchrom, int min_cov, int min_len, mb2_segments* out);

/* Same computation with the three hit arrays already resident in device memory (e.g. torch
 * tensors' data_ptr()); the result arrays stay on the device (out->on_device = 1). */
MB2_API int mb2_coverage_segments_dev(const int32_t* d_chrom, const int32_t* d_start, const int32_t* d_end, uint64_t nhits,
                              const int64_t* chrom_sizes, int nchrom, int min_cov, int min_len, mb2_segments* out);

/* Same again, writing straight into CALLER-OWNED device arrays of `capacity` elements each (a pipeline that keeps its
 * tables in HBM, e.g. preallocated torch tensors): no allocation handed over, no copy. *n_out receives the number of
 * segments; if that exceeds `capacity` nothing is written, the call returns MB2_ERR_CAPACITY and *n_out says how many
 * elements a retry needs. */
MB2_API int mb2_coverage_segments_into(const int32_t* d_chrom, const int32_t* d_start, const int32_t* d_end, uint64_t nhits,
                               const int64_t* chrom_sizes, int nchrom, int min_cov, int min_len, int32_t* d_out_chrom,
                               int32_t* d_out_start, int32_t* d_out_end, uint64_t capacity, uint64_t* n_out);

MB2_API void mb2_free_segments(mb2_segments* seg);

/* ---- genomes --------------------------------------------------------------------------- */
/* A genome resident in HBM: every scaffold 2-bit packed + a non-ACGT mask, one padded coordinate
 * space. Replaces the per-scaffold FASTA files mimeo writes for LASTZ (utils.py:274-309) and
 * LASTZ's own sequence loading. `seqs[i]` is the ASCII sequence of scaffold i (no header, no
 * newlines), `lens[i]` its length; scaffold order defines the scaffold index used everywhere. */
typedef struct mb2_genome mb2_genome;
MB2_API int mb2_genome_create(const uint8_t* const* seqs, const uint64_t* lens, int n, mb2_genome** out);
/* Reverse complement of every scaffold (what LASTZ aligns for strand2 = '-'). */
MB2_API int mb2_genome_revcomp(const mb2_genome* g, mb2_genome** out);
/* Scaffolds [0,n) of g followed by their reverse complements as scaffolds [n,2n): one pass of the pipeline then covers
 * --strand=both. mb2_align accepts such a genome as Q_both. */
MB2_API int mb2_genome_both_strands(const mb2_genome* g, mb2_genome** out);
MB2_API void mb2_genome_free(mb2_genome* g);
/* Test hook: scaffold `scaf` decoded back to codes 0..3 = ACGT, 4 = other (HOST buffer of its length). */
MB2_API int mb2_genome_decode(const mb2_genome* g, int scaf, uint8_t* out);
/* Test hook: the 4-bit code plane of the whole padded coordinate space (8 codes per word). Sets *nwords to its length in
 * words and copies min(cap, *nwords) words to the HOST buffer out (out may be null when cap is 0). */
MB2_API int mb2_test_genome_nibbles(const mb2_genome* g, uint32_t* out, uint64_t cap, uint64_t* nwords);

/* ---- alignment parameters --------------------------------------------------------------- */
/* The knobs of the one LASTZ command line mimeo issues (wrappers.py:1031): --hspthresh is the only
 * one mimeo exposes (run_self.py:142-147); the rest are LASTZ defaults (SURVEY.md 9.1). */
typedef struct mb2_align_params {
    int32_t hspthresh, xdrop, ydrop, gap_open, gap_extend, gappedthresh;
    int32_t entropy, chain, gapped, transition;
} mb2_align_params;
MB2_API void mb2_default_align_params(mb2_align_params* p);

/* Ungapped HSPs (stage b), canonical order (tile, s1, s2, len); tile = t_scaffold * nQ + q_scaffold;
 * coordinates 0-based, local to the scaffolds, on the strand Q is oriented in. HOST arrays. */
typedef struct mb2_hsps {
    uint32_t* tile;
    int32_t *s1, *s2, *len, *score;
    uint64_t n;
} mb2_hsps;
MB2_API void mb2_free_hsps(mb2_hsps* h);
/* Test hook: stage (a)+(b) only. `stats` (may be NULL) receives 16 counters:
 * [0] survivors [1] seed hits [2] run leaders [3] stage-1 cells [4] HSPs [5] extensions [6] stage-2 cells. */
MB2_API int mb2_test_hsps(const mb2_genome* T, const mb2_genome* Q, const mb2_align_params* p, mb2_hsps* out, uint64_t* stats);

/* Test hook: stage (a) only. The seed hits of T x Q that the bounded first-stage x-drop could not rule out (one scan of the
 * whole query), as PADDED positions: the seed of survivor k starts at t_pos[k] in T and q_pos[k] in Q, in the order the scan
 * wrote them. t_off / q_off: padded start of every scaffold of T / Q. counters: [0] survivors [1] seed hits [2] run leaders
 * [3] stage-1 cells. init_cap = initial survivor capacity (0 = default); a smaller value forces the overflow and rescan.
 * HOST arrays owned by the library; free with mb2_free_seed_survivors. */
typedef struct mb2_seed_survivors {
    uint32_t *t_pos, *q_pos;
    uint64_t n;
    uint32_t *t_off, *q_off;
    int32_t t_nscaf, q_nscaf;
    uint64_t counters[4];
} mb2_seed_survivors;
MB2_API int mb2_test_seed_scan(const mb2_genome* T, const mb2_genome* Q, const mb2_align_params* p, uint64_t init_cap,
                               mb2_seed_survivors* out);
MB2_API void mb2_free_seed_survivors(mb2_seed_survivors* s);

/* ---- (a)+(b)+(b')+(c): the whole LASTZ stage ------------------------------------------------ */
/* One row per gapped alignment, i.e. per line of LASTZ's --format=general output before mimeo's
 * awk filters (wrappers.py:1044-1056). start1/end1/start2/end2 are what LASTZ prints: origin-one,
 * closed, start2/end2 on the query's + strand (start2+/end2+); strand: 0 = '+', 1 = '-';
 * length1 = end1-start1+1; identity = nmatch/ncols. HOST arrays owned by the library.
 * stats: [0] survivors [1] seed hits [2] run leaders [3] stage-1 cells [4] HSPs [5] stage-2 extensions
 * [6] stage-2 cells [7] gapped DP cells [8] alignments [9] anchors extended (summed over strands). */
typedef struct mb2_hits {
    int32_t *t_id, *q_id, *strand, *start1, *end1, *start2, *end2, *score, *nmatch, *ncols;
    uint64_t n;
    uint64_t stats[16];
} mb2_hits;
/* Replaces every `lastz T Q ...` process of mimeo's script (wrappers.py:1025-1037, 1070-1082, 786-798,
 * 645-653): aligns every scaffold of T against every scaffold of Q, both strands when strands == 3
 * (1 = plus only, 2 = minus only). Q_aux may be NULL; otherwise it is a prebuilt companion of Q that saves
 * rebuilding it per call: for strands == 3 the mb2_genome_both_strands(Q) genome, for strands == 2 mb2_genome_revcomp(Q).
 * Multi-GPU: each rank passes its own subset of target scaffolds as T.
 * t_same_q (may be NULL): for every target scaffold the index of the query scaffold holding the IDENTICAL sequence, or -1.
 * It only enables the exact closed form of the trivial self-alignment (DESIGN.md); results do not depend on it. When NULL
 * the identity is inferred if Q (or the genome Q_aux was built from) is the very genome object T. */
MB2_API int mb2_align(const mb2_genome* T, const mb2_genome* Q, const mb2_genome* Q_aux, const mb2_align_params* p, int strands,
                      const int32_t* t_same_q, mb2_hits* out);
MB2_API void mb2_free_hits(mb2_hits* h);

/* ---- the hit table kept in HBM between the stages ------------------------------------------------ */
/* mb2_align with the rows left on the device (same columns, same coordinates); the handle owns them. */
typedef struct mb2_hits_dev mb2_hits_dev;
MB2_API int mb2_align_dev(const mb2_genome* T, const mb2_genome* Q, const mb2_genome* Q_aux, const mb2_align_params* p, int strands,
                          const int32_t* t_same_q, mb2_hits_dev** out);
MB2_API void mb2_hits_dev_free(mb2_hits_dev* h);
MB2_API uint64_t mb2_hits_dev_count(const mb2_hits_dev* h);
/* Kernel (d) part 1, in place on the device table. Replaces the filter that follows every LASTZ call in the reference's
 * script (wrappers.py:1044-1056; map: 665-675; x: 805-817): keep length1 >= min_len and the PRINTED identity ('%.1f' of
 * 100*nmatch/ncols, as awk compares it) >= min_idt; map_rule != 0 adds import_Align's own test end1 - start1 >= min_len
 * (wrappers.py:76). Survivors are compacted and sorted by (t_id, q_id, start1, end1) -- the order of `sort -k 1,1 -k 3n,4n`
 * inside every scaffold-pair block; rows equal in all four keys keep their order (the text formatter breaks those ties). */
MB2_API int mb2_filter_sort(mb2_hits_dev* h, double min_len, double min_idt, int map_rule, uint64_t* n_kept);
/* Coverage stage straight from the device table (no host round trip of the BED projection, wrappers.py:1120-1128):
 * which = 0 every row, 1 rows with t_id != q_id (the .tab of --strictSelf), 2 rows with t_id == q_id (_intra.tab,
 * wrappers.py:1016). Segments are returned in HOST arrays (free with mb2_free_segments). */
MB2_API int mb2_hits_dev_coverage(const mb2_hits_dev* h, int which, const int64_t* chrom_sizes, int nchrom, int min_cov, int min_len,
                                  mb2_segments* out);
/* A device table from HOST columns (e.g. the rows of a recycled .tab, or a table gathered from other ranks); nt / nq = number of
 * target / query scaffolds the ids refer to. */
MB2_API int mb2_hits_dev_upload(const mb2_hits* in, int nt, int nq, mb2_hits_dev** out);
/* The (surviving) rows as HOST arrays, e.g. for the .tab text (free with mb2_free_hits). */
MB2_API int mb2_hits_dev_download(const mb2_hits_dev* h, mb2_hits* out);

/* ---- native text ingest (host side, no GPU needed) --------------------------------------------- */
/* The BED projection of a LASTZ-style .tab file, i.e. what `awk '!/^#/ {print $1,$3,$4;}'` hands to
 * sort | bedtools genomecov (wrappers.py:1120-1128, x: 827-835, self intra: 1201-1220): one (name, start1, end1)
 * triple per line that does not start with '#', fields split on blanks/tabs. Names are dictionary-encoded in order of
 * first appearance. The file is mmapped and parsed by `nthreads` threads (0 = all cores). Arrays owned by the library. */
typedef struct mb2_tab_hits {
    int32_t* chrom;      /* index into names */
    int64_t* start;
    int64_t* end;
    uint64_t n;
    char** names;        /* nnames NUL-terminated strings */
    int32_t nnames;
} mb2_tab_hits;
MB2_API int mb2_tab_project(const char* path, int nthreads, mb2_tab_hits* out);
MB2_API void mb2_free_tab_hits(mb2_tab_hits* h);

/* Every record of a FASTA file: id = first word of the header, header = the whole '>' line, sequence with line breaks
 * and blanks removed. Replaces Biopython's SeqIO.parse in chromlens / splitFasta (utils.py:301-309, 530-546).
 * seq holds all sequences back to back; record r is seq[off[r] .. off[r+1]). Arrays owned by the library. */
typedef struct mb2_fasta {
    int32_t n;
    char** ids;
    char** headers;
    uint64_t* off;       /* n + 1 entries */
    uint8_t* seq;
} mb2_fasta;
MB2_API int mb2_fasta_read(const char* path, int nthreads, mb2_fasta* out);
MB2_API void mb2_free_fasta(mb2_fasta* f);

/* splitFasta (utils.py:274-309): one `<outdir>/<id>.fa` per record of a multi-FASTA file, header line kept whole, sequence
 * wrapped at `width` columns (Biopython writes 60), files written by `nthreads` workers (0 = all cores). With `unique` a
 * repeated id stops the split at that record, as the reference does: the call returns MB2_ERR_DUPLICATE_ID and
 * mb2_last_error() is the id. *nfiles receives the number of files written. */
#define MB2_ERR_DUPLICATE_ID (-7)
MB2_API int mb2_fasta_split(const char* path, const char* outdir, int unique, int width, int nthreads, uint64_t* nfiles);

/* The filter + projection + sort that follows every LASTZ call in the reference's script (wrappers.py:1044-1056):
 * rows with length1 >= min_len and printed identity ('%.1f' of 100*nmatch/ncols) >= min_idt, as 10 tab-separated columns,
 * grouped by (t_id, q_id) block (ascending), each block sorted by start1 and then by the whole line's bytes
 * (`sort -k 1,1 -k 3n,4n`). Input: the columns of mb2_hits as HOST arrays. Block b is text[off[b] .. off[b+1]). */
typedef struct mb2_tab_text {
    char* text;
    uint64_t nbytes;
    int32_t* t_id;
    int32_t* q_id;
    uint64_t* off;       /* nblocks + 1 entries */
    uint32_t* nrows;
    uint64_t nblocks;
} mb2_tab_text;
MB2_API int mb2_format_tab(const int32_t* t_id, const int32_t* q_id, const int32_t* strand, const int32_t* start1, const int32_t* end1,
                           const int32_t* start2, const int32_t* end2, const int32_t* score, const int32_t* nmatch, const int32_t* ncols,
                           uint64_t n, const char* const* tnames, int nt, const char* const* qnames, int nq, double min_len, double min_idt,
                           mb2_tab_text* out);
MB2_API void mb2_free_tab_text(mb2_tab_text* t);

/* `mimeo map` post-processing: import_Align + writeGFFlines of the reference (wrappers.py:33-117, 443-522) in one pass over
 * the .tab file. Keeps rows with int(end1) - int(start1) >= min_len and float(identity) >= min_idt, sorts them (stable) by the
 * STRING values of (name1, start1, end1, strand1), numbers them prefix_0001.. (zero-filled to the width of the row count;
 * prefix NULL or "" = "BHit") and returns one GFF3 feature line per row:
 * name1, mimeo-map, ftype, start1, end1, score, strand1, ., ID=..;identity=..;B_locus=name2_strand2_start2_end2.
 * The header lines (##gff-version, ##sequence-region, ##seqid) are the caller's. Text owned by the library. */
typedef struct mb2_text {
    char* text;
    uint64_t nbytes;
    uint64_t nrows;
} mb2_text;
MB2_API int mb2_map_gff(const char* tab_path, const char* prefix, double min_len, double min_idt, const char* ftype, int nthreads,
                        mb2_text* out);
MB2_API void mb2_free_text(mb2_text* t);

/* The awk that ends every coverage block of the reference's script (wrappers.py:1166-1173; x: 885-891; intra: 1257-1264):
 * one GFF3 feature row per segment (HOST arrays, e.g. an mb2_segments result),
 *   names[chrom] \t source \t label \t start \t end \t . \t + \t . \t ID=<prefix>_%05d \n
 * numbered from first_id (the reference restarts at 1 in every block). Header lines are the caller's. */
MB2_API int mb2_format_gff(const int32_t* chrom, const int32_t* start, const int32_t* end, uint64_t n, const char* const* names,
                           int nnames, const char* source, const char* label, const char* prefix, uint64_t first_id, int nthreads,
                           mb2_text* out);

/* ---- tandem-repeat mask of `mimeo map --maxtandem` and `mimeo filter` ------------------------------------ */
/* The reference runs Tandem Repeats Finder on every A-genome hit span; this build computes its own mask (DESIGN §2,
 * T1-T4; not TRF): local self-alignment of the span within diagonals 1..maxperiod, +match / -mismatch (N never matches),
 * -delta per indel; a position is masked iff it lies between the two aligned positions of a column of some such
 * alignment scoring >= minscore. Defaults = mimeo's --tmatch 2 --tmismatch 7 --tdelta 7 --tminscore 50 --tmaxperiod 50. */
typedef struct mb2_tandem_params {
    int32_t match, mismatch, delta, minscore, maxperiod;
} mb2_tandem_params;
MB2_API void mb2_default_tandem_params(mb2_tandem_params* p);
/* masked[k] = number of masked positions of span k = scaffold scaf[k] of g, bases [start[k], start[k] + len[k]) (0-based;
 * len 0 allowed). HOST arrays. Identical spans are computed once. Parameters out of range (match < 1, mismatch or delta < 0,
 * minscore < 1, maxperiod outside 1..256, minscore + mismatch > 65535) or a span outside its scaffold: MB2_ERR_INVALID_ARG. */
MB2_API int mb2_tandem_mask(const mb2_genome* g, const int32_t* scaf, const int64_t* start, const int64_t* len, uint64_t n,
                            const mb2_tandem_params* p, uint64_t* masked);
/* mb2_tandem_mask that also returns the merged masked runs of every span (span-local, closed [start, end]): run r of span k
 * is (start[r], end[r]) for off[k] <= r < off[k+1], runs in increasing order. Arrays owned by the library; free with
 * mb2_free_tandem_runs (also after an error). What `mimeo filter --writeTRF` replaces by N. */
typedef struct mb2_tandem_runs {
    uint64_t* off;       /* n + 1 entries */
    int64_t* start;
    int64_t* end;
    uint64_t n;
} mb2_tandem_runs;
MB2_API int mb2_tandem_mask_runs(const mb2_genome* g, const int32_t* scaf, const int64_t* start, const int64_t* len, uint64_t n,
                                 const mb2_tandem_params* p, uint64_t* masked, mb2_tandem_runs* runs);
/* Test hook: mb2_tandem_mask_runs with store_budget = bytes of device storage per launch (0 = default; small values force
 * many launches). */
MB2_API int mb2_test_tandem_mask(const mb2_genome* g, const int32_t* scaf, const int64_t* start, const int64_t* len, uint64_t n,
                                 const mb2_tandem_params* p, uint64_t store_budget, uint64_t* masked, mb2_tandem_runs* runs);
MB2_API void mb2_free_tandem_runs(mb2_tandem_runs* r);
/* The tandem-repeat report of `--reportTRF` (DESIGN §2, R1-R6; not TRF's .dat): mb2_tandem_mask_runs, and in the same call
 * one entry per run r of `runs` (span order, runs ascending) describing the tandem array in that run: period (R2), score
 * (R6, may be negative), matches to the consensus (R4), count[4r .. 4r+3] of A, C, G, T (R5), and the consensus (R3),
 * consensus[cons_off[r] .. cons_off[r+1]), period[r] bytes of A/C/G/T/N without a terminator. Identical runs are computed
 * once. Arrays owned by the library; free rep with mb2_free_tandem_report and runs with mb2_free_tandem_runs (both also
 * after an error). Parameter checks are mb2_tandem_mask's. */
typedef struct mb2_tandem_repeats {
    int32_t* period;
    int64_t* score;
    uint64_t* matches;
    uint64_t* count;     /* 4 per run */
    uint64_t* cons_off;  /* n + 1 entries */
    char* consensus;
    uint64_t n;          /* number of runs */
} mb2_tandem_repeats;
MB2_API int mb2_tandem_report(const mb2_genome* g, const int32_t* scaf, const int64_t* start, const int64_t* len, uint64_t n,
                              const mb2_tandem_params* p, uint64_t* masked, mb2_tandem_runs* runs, mb2_tandem_repeats* rep);
MB2_API void mb2_free_tandem_report(mb2_tandem_repeats* r);

/* ---- device primitives exposed for parity tests ------------------------------------------- */
/* Stable LSD radix sort of HOST arrays on bits [begin_bit, end_bit) (vals may be NULL). */
MB2_API int mb2_test_sort_u32(uint32_t* keys, uint32_t* vals, uint64_t n, int begin_bit, int end_bit);
MB2_API int mb2_test_sort_u64(uint64_t* keys, uint32_t* vals, uint64_t n, int begin_bit, int end_bit);
/* Two independent key arrays of the same length sorted by the same launches (how the coverage stage bins its +1 and -1
   event arrays). */
MB2_API int mb2_test_sort_u32_pair(uint32_t* keys_a, uint32_t* keys_b, uint64_t n, int begin_bit, int end_bit);
/* Exclusive prefix sum of a HOST array, in place; *total receives the grand total. */
MB2_API int mb2_test_scan_u32(uint32_t* data, uint64_t n, uint32_t* total);

#ifdef __cplusplus
}
#endif
#endif /* MIMEO_B200_H */
