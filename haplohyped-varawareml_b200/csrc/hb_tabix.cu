// hb_tabix.cu -- host side of region queries through an index: read a tabix (.tbi) or CSI (.csi) file and restate
// htslib's hts_itr_query for one interval.  The chunks it returns only narrow the bytes a parse inflates; the GPU region
// filter still decides which records are kept.
#include <zlib.h>

#include <algorithm>
#include <cstring>

#include "hb_tabix.h"

namespace hb {
namespace {

// every gzip member of a BGZF file, one after another
bool inflate_members(const uint8_t *in, uint64_t n, std::vector<uint8_t> &out) {
    z_stream zs;
    memset(&zs, 0, sizeof zs);
    if (inflateInit2(&zs, 15 + 16) != Z_OK) return false;
    zs.next_in = const_cast<Bytef *>(in);
    zs.avail_in = (uInt)n;
    out.resize(std::max<uint64_t>(4 * n, 1 << 16));
    uint64_t produced = 0;
    bool ok = n > 0;
    while (ok) {
        if (out.size() - produced < (1 << 16)) out.resize(out.size() * 2);
        zs.next_out = out.data() + produced;
        zs.avail_out = (uInt)(out.size() - produced);
        const uInt before = zs.avail_out;
        const int rc = inflate(&zs, Z_NO_FLUSH);
        produced += before - zs.avail_out;
        if (rc == Z_STREAM_END) {
            if (zs.avail_in == 0) break;
            if (inflateReset(&zs) != Z_OK) ok = false;
        } else if (rc != Z_OK && rc != Z_BUF_ERROR) {
            ok = false;
        } else if (zs.avail_in == 0 && zs.avail_out != 0) {
            ok = false;                                   // truncated member
        }
    }
    inflateEnd(&zs);
    out.resize(produced);
    return ok;
}

struct Cursor {
    const uint8_t *p, *e;
    bool ok = true;
    bool take(void *dst, uint64_t k) {
        if (!ok || (uint64_t)(e - p) < k) return ok = false;
        memcpy(dst, p, k);
        p += k;
        return true;
    }
    int32_t i32() { int32_t v = 0; take(&v, 4); return v; }
    uint32_t u32() { uint32_t v = 0; take(&v, 4); return v; }
    uint64_t u64() { uint64_t v = 0; take(&v, 8); return v; }
};

// the tabix conf (format, col_seq, col_beg, col_end, meta, skip) and the NUL-separated sequence names
bool read_tabix_meta(Cursor &c, std::vector<std::string> &names) {
    for (int k = 0; k < 6; ++k) c.i32();
    const int32_t l_nm = c.i32();
    if (!c.ok || l_nm < 0 || (int64_t)(c.e - c.p) < l_nm) return false;
    const char *s = (const char *)c.p, *end = s + l_nm;
    while (s < end) {
        const char *z = (const char *)memchr(s, 0, (size_t)(end - s));
        if (!z) return false;
        names.emplace_back(s, z);
        s = z + 1;
    }
    c.p += l_nm;
    return true;
}

int bin_first(int l) { return ((1 << (3 * l)) - 1) / 7; }
int bin_parent(int b) { return (b - 1) >> 3; }
int bin_bot(int bin, int n_lvls) {                      // hts_bin_bot: first bottom-level window the bin covers
    int l = 0;
    for (int b = bin; b; b = bin_parent(b)) ++l;
    return (bin - bin_first(l)) << (n_lvls - l) * 3;
}

}  // namespace

bool tabix_load(const uint8_t *bytes, uint64_t n, TabixIndex &idx, std::string &why) {
    std::vector<uint8_t> raw;
    if (!inflate_members(bytes, n, raw)) { why = "the index does not inflate"; return false; }
    Cursor c{raw.data(), raw.data() + raw.size()};
    char magic[4] = {0, 0, 0, 0};
    c.take(magic, 4);
    idx = TabixIndex();
    if (memcmp(magic, "TBI\1", 4) == 0) {
        const int32_t n_ref = c.i32();
        if (!c.ok || n_ref < 0 || !read_tabix_meta(c, idx.names)) { why = "truncated TBI header"; return false; }
        idx.refs.resize((size_t)n_ref);
    } else if (memcmp(magic, "CSI\1", 4) == 0) {
        idx.csi = true;
        idx.min_shift = c.i32();
        idx.n_lvls = c.i32();
        const int32_t l_aux = c.i32();
        if (!c.ok || idx.min_shift < 1 || idx.min_shift > 30 || idx.n_lvls < 1 || idx.n_lvls > 9 || l_aux < 0 ||
            (int64_t)(c.e - c.p) < l_aux) { why = "bad CSI header"; return false; }
        if (l_aux >= 28) {                              // tabix meta: the sequence names
            Cursor a{c.p, c.p + l_aux};
            if (!read_tabix_meta(a, idx.names)) idx.names.clear();
        }
        c.p += l_aux;
        const int32_t n_ref = c.i32();
        if (!c.ok || n_ref < 0) { why = "truncated CSI header"; return false; }
        idx.refs.resize((size_t)n_ref);
    } else {
        why = "bad magic";
        return false;
    }
    for (TabixIndex::Ref &r : idx.refs) {
        const int32_t n_bin = c.i32();
        if (!c.ok || n_bin < 0) { c.ok = false; break; }
        for (int32_t b = 0; b < n_bin && c.ok; ++b) {
            const uint32_t bin = c.u32();
            TabixIndex::Bin &x = r.bins[bin];
            if (idx.csi) x.loff = c.u64();
            const int32_t n_chunk = c.i32();
            if (!c.ok || n_chunk < 0 || (uint64_t)(c.e - c.p) < 16ull * (uint64_t)n_chunk) { c.ok = false; break; }
            x.chunks.resize((size_t)n_chunk);
            for (auto &ch : x.chunks) { ch.first = c.u64(); ch.second = c.u64(); }
        }
        if (!idx.csi) {
            const int32_t n_intv = c.i32();
            if (!c.ok || n_intv < 0 || (uint64_t)(c.e - c.p) < 8ull * (uint64_t)n_intv) { c.ok = false; break; }
            r.lidx.resize((size_t)n_intv);
            for (auto &o : r.lidx) o = c.u64();
            // htslib gives a TBI's bins the loff of their first window, as CSI stores it
            const int n_bins = ((1 << (3 * idx.n_lvls + 3)) - 1) / 7;
            for (auto &kv : r.bins) {
                const int bot = (int)kv.first < n_bins ? bin_bot((int)kv.first, idx.n_lvls) : -1;
                kv.second.loff = bot >= 0 && (size_t)bot < r.lidx.size() ? r.lidx[(size_t)bot] : 0;
            }
        }
    }
    if (!c.ok) { why = "truncated index"; return false; }
    if (!idx.names.empty() && idx.names.size() != idx.refs.size()) { why = "sequence names do not match n_ref"; return false; }
    return true;
}

std::vector<std::pair<uint64_t, uint64_t>> tabix_query(const TabixIndex &idx, int tid, int64_t beg, int64_t end) {
    std::vector<std::pair<uint64_t, uint64_t>> off;
    const int64_t max_pos = 1ll << (idx.min_shift + 3 * idx.n_lvls);
    if (beg < 0) beg = 0;
    if (end > max_pos) end = max_pos;
    if (tid < 0 || (size_t)tid >= idx.refs.size() || beg >= end) return off;
    const auto &bins = idx.refs[(size_t)tid].bins;
    if (bins.empty()) return off;
    // min_off: the loff of the bottom-level bin of beg, or of the nearest bin present to its left or above it
    int bin = bin_first(idx.n_lvls) + (int)(beg >> idx.min_shift);
    auto it = bins.end();
    do {
        it = bins.find((uint32_t)bin);
        if (it != bins.end()) break;
        const int first = (bin_parent(bin) << 3) + 1;
        bin = bin > first ? bin - 1 : bin_parent(bin);
    } while (bin);
    if (bin == 0) it = bins.find(0);
    const uint64_t min_off = it != bins.end() ? it->second.loff : 0;
    // reg2bins: every bin of every level that overlaps [beg, end)
    int64_t e = end - 1;
    for (int l = 0, t = 0, s = idx.min_shift + 3 * idx.n_lvls; l <= idx.n_lvls; s -= 3, t += 1 << (3 * l), ++l) {
        for (int64_t b = t + (beg >> s); b <= t + (e >> s); ++b) {
            auto f = bins.find((uint32_t)b);
            if (f == bins.end()) continue;
            for (const auto &ch : f->second.chunks)
                if (ch.second > min_off) off.push_back(ch);
        }
    }
    if (off.empty()) return off;
    std::sort(off.begin(), off.end());
    size_t l = 0;
    for (size_t i = 1; i < off.size(); ++i)             // drop chunks contained in the one before
        if (off[l].second < off[i].second) off[++l] = off[i];
    off.resize(l + 1);
    for (size_t i = 1; i < off.size(); ++i)             // trim overlaps left by the index's own merging
        if (off[i - 1].second >= off[i].first) off[i - 1].second = off[i].first;
    l = 0;
    for (size_t i = 1; i < off.size(); ++i) {           // merge chunks that meet in one BGZF block
        if (off[l].second >> 16 == off[i].first >> 16) off[l].second = off[i].second;
        else off[++l] = off[i];
    }
    off.resize(l + 1);
    return off;
}

}  // namespace hb
