// hb_parse_struct.h -- the device-resident parse handle, shared by hb_api.cu and hb_store.cu.
#pragma once
#include <string>
#include <vector>

#include "hb_internal.h"

namespace hb {
int api_fail(int code, const std::string &msg);    // sets the thread-local hb_last_error() text
}

struct hb_parse {
    int device = 0;
    cudaStream_t stream = nullptr;
    int sm_count = 148;
    const uint8_t *d_text = nullptr;
    uint8_t *d_text_owned = nullptr;
    bool text_released = false;         // hb_parse_release_text: the results stay, a re-run is no longer possible
    uint64_t nbytes = 0;
    // n_cols: sample columns of every record of the file (what locates records and checks their column counts);
    // n_samples: genotype planes -- the subset's size under a sample subset, else n_cols
    uint32_t n_cols = 0, n_samples = 0;
    std::vector<uint32_t> sel_cols;     // sample subset (hb_parse_*_subset): the selected columns, ascending; empty = every one
    uint4 *d_sel_mask = nullptr;        // its device tables (hb::SampleSel), one entry per 128-column block
    uint32_t *d_sel_base = nullptr;
    hb::RegionArg rg;
    int end_is_int = 0, want_gt = 1, tokenizer = 0;
    bool with_tabs = false;
    bool use_walker = false;            // records located by walking heads (hb_walk.cu) instead of tokenizing
    uint32_t n_walkers = 0, walk_cap = 0;
    uint64_t walk_range = 0;
    uint64_t *d_wstart = nullptr, *d_wrow = nullptr, *d_verify = nullptr, *d_wcount = nullptr;
    uint64_t verify_cap = 0;
    hb::SiteRows walk_pad;               // padded site rows of the walk, kWalkSlots per walker (compacted into rows)
    int walker_fallbacks = 0;
    int index_used = 0;                 // 1 newline tokenizer, 2 newline+tab tokenizer, 3 walker, 4 BCF records
    struct Bcf {                        // BCF input: the header's dictionaries and the locator's buffers (hb_bcf.cu)
        std::vector<std::string> contigs;
        std::vector<uint64_t> name_off;  // of each contig name in d_names (ascending)
        int gt_key = -1;                 // string-dictionary index of GT, -1 = not declared
        hb::BcfContig *d_contigs = nullptr;
        uint8_t *d_names = nullptr;      // the contig names, NUL-separated: the "text" of the CHROM runs
        uint64_t first_len = 0;          // bytes of the first record
        hb::BcfSegs seg;
        uint64_t *d_rec_off = nullptr, rec_cap = 0;
        uint32_t *d_blk_count = nullptr;
        uint64_t *d_blk_base = nullptr, blk_cap = 0;
    };
    Bcf *bcf = nullptr;
    uint32_t ncp = 0;

    uint64_t *d_nl_after = nullptr; uint64_t nl_after_cap = 0;
    uint32_t stage_cap = 0, n_cta = 0;
    uint64_t tiles_per_cta = 0;
    bool probed = false;
    uint64_t n_lines = 0;
    uint64_t first_line_len = 0;
    hb::CtaTok *d_cta = nullptr;
    uint64_t *d_cbase = nullptr;
    uint64_t *d_cp = nullptr; uint64_t cp_cap = 0;   // column checkpoints, ncp per row
    hb::DevStatus *d_st = nullptr;
    hb::DevStatus h_st;
    hb::DevStatus *h_st_pin = nullptr;       // pinned landing buffer of h_st
    hb::SiteRows rows;                  // one per kept record; chrom5 = first 5 CHROM bytes (the S5 field of the 35-byte record)
    uint32_t *d_nu_rows = nullptr;      // text paths only: the rows that need the general decode path
    uint64_t *d_sites_state = nullptr;  // tokenizer path only: tile state of the site kernel
    int8_t *d_gt[2] = {nullptr, nullptr};
    uint64_t gt_stride = 0, gt_bytes = 0;
    uint32_t *d_bits = nullptr;         // the same alleles as bit planes (hb_common.cuh, kBitGroupWords): what kernel 4b reads
    uint64_t bits_stride = 0;           // words per sample = gt_stride / 128 * kBitGroupWords
    uint32_t *d_ploidy = nullptr, *d_badgt = nullptr;
    uint64_t *d_run_rows = nullptr;
    static constexpr uint64_t kMaxRuns = 4096;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaStream_t side = nullptr;         // the CHROM-run kernel runs here, next to the GT decoder
    cudaEvent_t ev_runs = nullptr;
    float ms_tok = 0, ms_sites = 0, ms_decode = 0, ms_inflate = 0;
    uint64_t compressed_bytes = 0;      // BGZF bytes shipped over PCIe when the file was inflated on the GPU
    // region query through a .tbi / .csi (hb_parse_index_info): used, compressed bytes read, merged chunks of the query
    int idx_used = 0;
    uint64_t idx_bytes_read = 0, idx_chunks = 0;
    // chrom runs (host)
    std::vector<uint64_t> run_rows;
    std::vector<std::string> run_names;
    uint64_t run_seq = 0;                // counts run_parse calls (frames launched early belong to one of them)
    bool runs_valid = false;             // run_rows / run_names hold the runs of the last parse (fetched on demand)
    std::vector<std::string> samples;   // sample names when the parse was made from a file
    void *attached_frames = nullptr;    // hb_frames whose site templates are made while the GT decoder runs (hb_store.cu)
};


namespace hb {
// hb_store.cu: start the site-template kernel of the attached frames on their side stream (called by run_parse)
void frames_early_site_pass(void *frames, hb_parse *p);
void frames_early_launch(void *frames, hb_parse *p);
void frames_buffer_cache_clear();       // hb_store.cu: release the kept frame buffers
}
