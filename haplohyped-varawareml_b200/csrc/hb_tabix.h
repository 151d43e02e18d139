// hb_tabix.h -- tabix (.tbi) and CSI (.csi) indexes as the hts-specs define them: load one, and list the BGZF chunks a
// region query has to read (htslib's hts_itr_query for one interval).
#pragma once
#include <stdint.h>

#include <map>
#include <string>
#include <utility>
#include <vector>

namespace hb {

struct TabixIndex {
    bool csi = false;
    int min_shift = 14, n_lvls = 5;
    std::vector<std::string> names;              // sequence names (TBI, and CSI with tabix meta); empty for a BCF CSI
    struct Bin {
        uint64_t loff = 0;                       // CSI: smallest virtual offset of a record that starts in the bin's span
        std::vector<std::pair<uint64_t, uint64_t>> chunks;   // [begin, end) virtual offsets
    };
    struct Ref {
        std::map<uint32_t, Bin> bins;
        std::vector<uint64_t> lidx;              // TBI linear index: smallest virtual offset per 16 kb window
    };
    std::vector<Ref> refs;
};

// the bytes of an index file (BGZF, inflated here with zlib) -> idx; false with `why` when they are not a readable index
bool tabix_load(const uint8_t *bytes, uint64_t n, TabixIndex &idx, std::string &why);
// merged chunks that may hold records of sequence tid overlapping [beg, end) (0-based, half open), in file order
std::vector<std::pair<uint64_t, uint64_t>> tabix_query(const TabixIndex &idx, int tid, int64_t beg, int64_t end);

}  // namespace hb
