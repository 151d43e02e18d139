// hb_internal.h -- structures shared by the kernels and the host side of libhaplo_b200.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

namespace hb {

// Tile geometry shared by the tokenizer (checkpoints) and the GT decoder (sample tiles).
constexpr int kCP = 128;          // one column checkpoint every kCP samples
constexpr int kTS = 128;          // samples per decode tile (== kCP)
constexpr int kTV = 64;           // records (rows) per decode tile
constexpr uint64_t kNoCp = ~0ull; // "no checkpoint written"

// Allele bit planes, written by the GT decoder next to the byte planes and read by the frame encoder (hb_store.cu):
// per sample kBitGroupWords-word groups of 128 rows, [sample][group][array][4 words], array 0/1 = bit 0 of the phase1 /
// phase2 byte ("B"), array 2/3 = "the byte is neither 0 nor 1" ("N").  Row r of a sample: group r >> 7, word (r >> 5) & 3,
// bit r & 31.  A frame's rows are one contiguous byte range of every sample: one TMA bulk copy.
constexpr int kBitGroupWords = 16;

// Per kept record, produced by the site kernel, consumed by the GT decoder.
struct RowInfo {
    uint64_t samp_abs;   // offset of the TAB that precedes sample 0
    uint32_t samp_len;   // bytes from samp_abs to end of line (exclusive of '\n' / "\r\n")
    uint32_t cp_row;     // row of the checkpoint table (general path only)
    uint32_t misc;       // [7:0] GT index in FORMAT, bit 8 uniform ("\tX|Y" x n_samples), bit 9 has samples
    uint32_t pad;
};
constexpr uint32_t kRowUniform = 1u << 8;
constexpr uint32_t kRowHasSamples = 1u << 9;

// Device-side counters / results, one per parse handle.
struct DevStatus {
    unsigned long long n_lines;        // tokenizer: number of '\n'
    unsigned long long n_records;      // site kernel: rows kept
    unsigned long long n_nonuniform;   // kept rows that need the general decode path
    unsigned long long n_bad_gt;       // alleles neither digits nor '.'
    unsigned long long n_bad_cols;     // records whose column count != 9 + n_samples (or < 8 fields)
    unsigned long long n_nogt;         // kept records without a GT key / sample columns
    unsigned long long n_chrom_runs;
    unsigned long long n_nu_count;     // walker count pass: kept rows that will need the general decode path
    unsigned long long n_verify;       // walker: jumped-over spans the decoder will not validate
    unsigned int ticket;               // tile tickets of the site kernel
    unsigned int walk_broken;          // walker: a chain did not land on the next walker's start
    unsigned int index_invalid;        // a newline was found inside a span taken for one record's samples
    unsigned long long bcf_fail;       // BCF locator: least of 2k (segment k's start is not segment k - 1's exit) and
                                       // 2k + 1 (segment k's chain met a record that fails the header test); ~0 = none
    unsigned long long bcf_records;    // BCF locator: records that start in the segments
    unsigned long long bcf_bad_fmt;    // BCF sites: kept records whose FORMAT fields run past the record
};

// Per tokenizer CTA (one contiguous byte range each).
struct CtaTok {
    uint32_t n_newlines;   // '\n' bytes in the range
    uint32_t tail_tabs;    // tabs after the last newline of the range (all tabs if it has none)
};

// Staged line index: record starts as written by the tokenizer CTAs + prefix sums of their counts.
struct LineIndex {
    const uint64_t *nl_after;   // [n_cta * stage_cap]
    const uint64_t *base;       // [n_cta + 1] exclusive prefix sum of CtaTok::n_newlines
    uint32_t n_cta, stage_cap;
};

struct RegionArg {
    char chrom[240];
    uint32_t chrom_len;
    int has_region;
    long long beg0, end0;
};

struct Launch {   // filled by the host, one per parse
    cudaStream_t stream;
    int sm_count;
};

// ---- launchers (definitions in the .cu files) ----
void launch_tokenize(bool with_tabs, const uint8_t *d_text, uint64_t nbytes, uint32_t n_cta, uint64_t tiles_per_cta,
                     uint64_t *d_nl_after, uint32_t stage_cap, uint64_t *d_cp, uint32_t ncp, CtaTok *d_cta,
                     const Launch &L);
uint64_t tokenize_tile_bytes();
void launch_index_columns(const uint8_t *d_text, const RowInfo *d_rowinfo, const uint32_t *d_nu_rows,
                          uint64_t n_nu, uint64_t *d_cp, uint32_t ncp, const Launch &L);
void launch_sites(const uint8_t *d_text, const LineIndex &li, uint64_t n_lines, uint32_t n_samples,
                  const RegionArg &rg, int end_is_int, int want_gt, bool cp_by_line, uint32_t *d_start,
                  uint32_t *d_stop, uint8_t *d_ref, uint8_t *d_alt, uint64_t *d_chrom_abs, uint8_t *d_chrom_len,
                  uint64_t *d_chrom5, RowInfo *d_rowinfo, uint32_t *d_nu_rows, uint64_t *d_tile_state, DevStatus *d_st,
                  const Launch &L);
// index-free record location for GT-only text (hb_walk.cu)
uint32_t walk_plan(uint64_t nbytes, uint64_t first_line_len, uint32_t lines_per_walker, uint64_t *range_bytes);
// walker (hb_walk.cu): padded site rows, kWalkSlots per walker, compacted to dense rows after the prefix sum
constexpr uint32_t kWalkSlots = 24;
struct WalkPad {
    uint32_t *start = nullptr, *stop = nullptr;
    uint8_t *ref = nullptr, *alt = nullptr, *chrom_len = nullptr;
    uint64_t *chrom_abs = nullptr, *chrom5 = nullptr;
    RowInfo *rowinfo = nullptr;
    uint64_t cap = 0;                        // rows
};
void launch_walk(const uint8_t *d_text, uint64_t nbytes, uint32_t n_samples, uint64_t range_bytes, uint32_t n_walkers,
                 const RegionArg &rg, int end_is_int, uint64_t *d_wstart, void *d_wcount, uint64_t *d_wrow, const WalkPad &pad,
                 uint64_t *d_verify, uint64_t verify_cap, DevStatus *d_st, const Launch &L);
void launch_walk_compact(const uint8_t *d_text, uint64_t nbytes, uint32_t n_samples, uint32_t n_walkers, void *d_wcount,
                         uint64_t *d_wrow, const WalkPad &pad, uint32_t *d_start, uint32_t *d_stop, uint8_t *d_ref, uint8_t *d_alt,
                         uint64_t *d_chrom_abs, uint8_t *d_chrom_len, uint64_t *d_chrom5, RowInfo *d_rowinfo,
                         uint32_t *d_nu_rows, uint64_t *d_verify, uint64_t verify_cap, DevStatus *d_st, const Launch &L);
void launch_chrom_runs(const uint8_t *d_text, const uint64_t *d_chrom_abs, const uint8_t *d_chrom_len,
                       uint64_t n_rows, uint64_t *d_run_rows, uint64_t max_runs, DevStatus *d_st,
                       const Launch &L);
void launch_decode_gt(const uint8_t *d_text, const RowInfo *d_rowinfo, uint64_t n_rows, uint32_t n_samples,
                      const uint64_t *d_cp, uint32_t ncp, int8_t *d_gt0, int8_t *d_gt1, uint64_t gt_stride,
                      uint32_t *d_bits, uint64_t bits_stride, uint32_t *d_ploidy_err, uint32_t *d_badgt_err, DevStatus *d_st,
                      const Launch &L);

void launch_bits_from_planes(const int8_t *d_gt0, const int8_t *d_gt1, uint64_t gt_stride, uint64_t n_rows, uint32_t n_samples,
                             uint32_t *d_bits, uint64_t bits_stride, const Launch &L);

// ---- BCF 2.2 input (hb_bcf.cu): kernel 1b locates records by chaining their lengths, kernel 3b decodes typed GT values.
// BCF rows use RowInfo as: samp_abs = offset of the GT values of sample 0, samp_len = values per sample, misc [7:0] = value
// type (1 int8, 2 int16, 3 int32; 255 = no GT) | kRowHasSamples.
struct BcfContig {                 // one entry of the header's contig dictionary
    uint64_t name5;                // first 5 name bytes, NUL padded (the S5 field)
    uint64_t name_off;             // offset of the name in the parse's name buffer: what d_chrom_abs holds for BCF rows
    uint32_t name_len;             // min(length, 255)
    uint32_t pad;
};
constexpr uint64_t kBcfNone = ~0ull;
struct BcfSegs {                   // the locator's segments, [k * bytes, (k + 1) * bytes) of the body
    uint64_t n = 0, bytes = 0, cap = 0;
    uint64_t *start = nullptr;     // first record start at or past the segment's begin (kBcfNone: none found)
    uint64_t *exit = nullptr;      // first record start at or past its end, from chaining `start`
    uint64_t *bad = nullptr;       // 0, or reason << 56 | offset of the record that failed the header test
    uint64_t *base = nullptr;      // exclusive prefix sums of count
    uint32_t *count = nullptr;     // records that start in the segment
    uint32_t *flag = nullptr;      // chain the segment (again)
};
// header-test failures (BcfSegs::bad >> 56)
constexpr uint32_t kBcfTruncated = 1, kBcfNSample = 2, kBcfContig = 3, kBcfHead = 4;
struct BcfSiteArgs {
    const uint8_t *text;
    const uint64_t *rec_off;       // [n_rec] record starts
    uint64_t n_rec;
    uint32_t n_samples, n_contigs;
    const BcfContig *contigs;
    int gt_key;                    // string-dictionary index of GT, -1 = not declared
    int rid;                       // region: -1 none, -2 contig not in the dictionary, else its index
    long long beg0, end0;
    int want_gt;
    uint32_t *start, *stop;
    uint8_t *ref, *alt, *chrom_len;
    uint64_t *chrom_abs, *chrom5;
    RowInfo *rowinfo;
    uint32_t *blk_count;           // [ceil(n_rec / 256)] kept records per block of 256
    uint64_t *blk_base;
    DevStatus *st;
};
// find (round 0: every segment's first start) and chain the flagged segments
void launch_bcf_chain(const uint8_t *d_text, uint64_t nbytes, uint32_t n_samples, uint32_t n_contigs, const BcfSegs &sg, bool find,
                      const Launch &L);
void launch_bcf_verify(const BcfSegs &sg, DevStatus *d_st, const Launch &L);
void launch_bcf_emit(const uint8_t *d_text, uint64_t nbytes, const BcfSegs &sg, uint64_t *d_rec_off, const Launch &L);
void launch_bcf_sites(const BcfSiteArgs &a, const Launch &L);
void launch_bcf_decode(const uint8_t *d_text, const RowInfo *d_rowinfo, uint64_t n_rows, uint32_t n_samples, int8_t *d_gt0,
                       int8_t *d_gt1, uint64_t gt_stride, uint32_t *d_bits, uint64_t bits_stride, uint32_t *d_ploidy_err,
                       uint32_t *d_badgt_err, DevStatus *d_st, const Launch &L);

void count_launch(uint64_t n = 1);

// pooled big device buffers (hb_api.cu): cudaMalloc / cudaFree of GB-sized buffers are slow and erratic on these hosts
cudaError_t dev_pool_alloc(void **out, uint64_t bytes);
void dev_pool_free(void *p);
void dev_pool_flush();
uint64_t dev_pool_idle_bytes();

// device -> host memory of any kind, synchronous: pinned destinations directly, pageable ones through pinned staging
bool host_is_pinned(const void *p);
cudaError_t d2h_copy(void *dst, const void *src, uint64_t bytes, cudaStream_t stream);
cudaError_t d2h_copy_2d(void *dst, uint64_t dpitch, const void *src, uint64_t spitch, uint64_t width, uint64_t height, cudaStream_t stream);

// BGZF slab streaming (hb_inflate.cu): device tables of one slot, enqueue-only inflate, last newline of a text range
struct InflateScratch {
    uint8_t *d_comp = nullptr;
    uint64_t comp_cap = 0;
    uint64_t *d_coff = nullptr, *d_ooff = nullptr;
    uint32_t *d_clen = nullptr, *d_olen = nullptr;
    int *d_status = nullptr;
    unsigned long long *d_last_nl = nullptr;
    uint32_t n_cap = 0;
};
int inflate_scratch_alloc(InflateScratch &sc, uint64_t comp_cap, uint32_t n_cap);
void inflate_scratch_free(InflateScratch &sc);
int inflate_bgzf_enqueue(InflateScratch &sc, const uint8_t *comp, uint64_t comp_bytes, const uint64_t *coff, const uint32_t *clen,
                         const uint64_t *ooff, const uint32_t *olen, uint32_t n, uint8_t *d_out, cudaStream_t stream);
// hb_set_bgzf_crc_check: kernel 0 compares each member's CRC32 with its trailer, and so does the host for the header members
bool bgzf_crc_check();
constexpr int kInflateCrcMismatch = 19;   // kernel 0 status of a member whose text does not match its CRC32
std::string bgzf_crc_message(const uint8_t *raw, uint64_t coff);
void launch_last_newline(const uint8_t *d_buf, uint64_t begin, uint64_t end, unsigned long long *d_res, cudaStream_t stream);

}  // namespace hb
