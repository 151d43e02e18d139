// hb_index.h -- building a tabix (.tbi) or CSI (.csi) index on the GPU (hb_index.cu, kernels 7a / 7b).
#pragma once
#include <stdint.h>

#include <string>
#include <vector>

#include "hb_internal.h"

namespace hb {

// One inflated BGZF file whose records were located by a parse: every line of a VCF body (the newline tokenizer's line
// index) or every record of a BCF body (the BCF locator's record offsets), on the device.
struct IndexJob {
    const uint8_t *d_text = nullptr;     // the body: records only
    uint64_t text_base = 0;              // offset of d_text[0] in the file's text (where the header ends)
    uint64_t total = 0;                  // bytes of the file's text
    uint64_t n_rec = 0;
    bool bcf = false;
    LineIndex li{};                      // VCF
    const uint64_t *d_rec_off = nullptr; // BCF
    uint32_t n_contigs = 0;              // BCF: the header's contig dictionary (the index has one sequence per contig)
    // the BGZF members that hold text: block address, block end (the next block's address), text offset and length
    std::vector<uint64_t> boff, bend, ooff;
    std::vector<uint32_t> olen;
    bool csi = false;
    int min_shift = 14, n_lvls = 5;
    cudaStream_t stream = nullptr;
};

struct IndexTimes { float ms_keys = 0, ms_chunks = 0; double ms_host = 0; };

// the uncompressed bytes of the index (hts-specs layout, bins in ascending order)
int build_index(const IndexJob &job, std::vector<uint8_t> &out, IndexTimes *times);

}  // namespace hb
