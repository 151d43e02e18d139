// hb_index.cu -- kernel 7: a tabix (.tbi) or CSI (.csi) index of an inflated BGZF file, built on the GPU.
//
// The text is already in HBM and its records located (kernel 0 inflated it; the newline tokenizer gives the start of every
// VCF line, the BCF locator every BCF record).  Then:
//   7a  index_keys_kernel / bcf_index_keys_kernel, one thread per record: [beg, end) as tabix reads it (POS - 1 and
//       POS - 1 + len(REF), or INFO/END when it is greater; BCF: pos and pos + rlen), the record's BGZF virtual offset
//       and its bin; records whose CHROM differs from the record before are appended to a short list (contig runs).
//   7b  index_chunks_kernel, one thread per record: a record whose (tid, bin) differs from the one before opens a chunk,
//       where htslib's hts_idx_push closes one; those few records are appended to a list.  Each record lowers the linear
//       index of every 16 kb window it touches to its offset (atomicMin: the first record in file order has the smallest),
//       and a position that goes down inside a contig is reported.
// The host sorts the short lists and does the O(chunks) rest htslib's hts_idx_finish does: chunk ends, the meta
// pseudo-bin, the linear index's gaps, bin loff, compress_binning and the merge of chunks in one BGZF block.
#include <algorithm>
#include <chrono>
#include <cstring>
#include <map>

#include "hb_index.h"

namespace hb {
int api_fail(int code, const std::string &msg);
}
#include "../../include/haplo_b200.h"

namespace hb {
namespace {

constexpr uint32_t kMaxIndexRuns = 1u << 16;      // contig runs (distinct CHROM blocks) an index may have
constexpr uint64_t kNone = ~0ull;

struct MemberTab {
    const uint64_t *ooff, *boff, *bend;
    const uint32_t *olen;
    uint32_t n;
};

struct Keys {
    int64_t *beg, *end;
    uint64_t *voff;
    uint32_t *bin;
};

struct Counters {                   // device, zeroed / set to kNone before each kernel
    unsigned long long n_runs, n_chunks, bad_line, bad_range, unsorted, max_end;
};

struct RunRec { uint64_t rec, key; };                    // key: line start (VCF) or rid (BCF)
struct ChunkRec { uint64_t rec, voff; uint32_t tid, bin; };

// the virtual offset of text position t: a position at the end of a member's text is (next block, 0), where
// bgzf_getline / bgzf_read leave a reader that has read the member's last byte
__host__ __device__ inline uint64_t voff_of(const uint64_t *ooff, const uint64_t *boff, const uint64_t *bend, const uint32_t *olen,
                                            uint32_t n, uint64_t t) {
    if (t == 0 || n == 0) return n ? boff[0] << 16 : 0;
    uint32_t lo = 0, hi = n;                              // members whose text starts before t
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (ooff[mid] < t) lo = mid + 1; else hi = mid;
    }
    const uint32_t k = lo - 1;
    const uint64_t u = t - ooff[k];
    return u == olen[k] ? bend[k] << 16 : (boff[k] << 16 | u);
}

__host__ __device__ inline int reg2bin(int64_t beg, int64_t end, int min_shift, int n_lvls) {
    int l, s = min_shift, t = ((1 << (3 * n_lvls)) - 1) / 7;
    for (--end, l = n_lvls; l > 0; --l, s += 3, t -= 1 << (3 * l))
        if (beg >> s == end >> s) return t + (int)(beg >> s);
    return 0;
}

__device__ __forceinline__ uint64_t line_end(const LineIndex &li, uint64_t k) {      // byte after the k-th newline
    uint32_t lo = 0, hi = li.n_cta;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (li.base[mid] <= k) lo = mid; else hi = mid;
    }
    return li.nl_after[(uint64_t)lo * li.stage_cap + (k - li.base[lo])];
}

__device__ __forceinline__ uint8_t ld(const uint8_t *p) { return __ldcg(p); }

__device__ __forceinline__ void store_key(const Keys &k, uint64_t r, int64_t beg, int64_t end, uint64_t voff, int min_shift,
                                          int n_lvls, int64_t max_pos, Counters *c) {
    if (beg < 0) beg = 0;
    if (end <= beg) end = beg + 1;
    if (beg > max_pos || end > max_pos) atomicMin(&c->bad_range, (unsigned long long)r);
    atomicMax(&c->max_end, (unsigned long long)end);
    k.beg[r] = beg; k.end[r] = end; k.voff[r] = voff;
    k.bin[r] = (uint32_t)reg2bin(beg, end, min_shift, n_lvls);
}

__device__ __forceinline__ void add_run(Counters *c, RunRec *runs, uint32_t cap, uint64_t r, uint64_t key) {
    const unsigned long long i = atomicAdd(&c->n_runs, 1ull);
    if (i < cap) runs[i] = RunRec{r, key};
}

// kernel 7a, VCF: one thread per line of the body
__global__ void __launch_bounds__(256) index_keys_kernel(const uint8_t *__restrict__ text, uint64_t text_base, LineIndex li,
                                                         uint64_t n, MemberTab mt, int min_shift, int n_lvls, int64_t max_pos,
                                                         Keys k, RunRec *runs, uint32_t run_cap, Counters *c) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const uint64_t ls = r ? line_end(li, r - 1) : 0, le = line_end(li, r) - 1;      // le: the '\n'
    // CHROM, POS, REF, INFO
    int col = 0;
    uint64_t chrom_end = ls, info_b = le, info_e = le;
    int64_t pos = 0;
    int pos_digits = 0;
    int64_t ref_len = 0;
    for (uint64_t i = ls; i < le && col < 8; ++i) {
        const uint8_t ch = ld(text + i);
        if (ch == '\t') {
            if (col == 0) chrom_end = i;
            if (col == 6) info_b = i + 1;
            if (col == 7) info_e = i;
            ++col;
            continue;
        }
        if (col == 1 && ch >= '0' && ch <= '9') { pos = pos * 10 + (ch - '0'); ++pos_digits; }
        else if (col == 3) ++ref_len;
    }
    if (col == 7) info_e = le > ls && ld(text + le - 1) == '\r' ? le - 1 : le;
    if (col < 4 || pos_digits == 0 || ld(text + ls) == '#') { atomicMin(&c->bad_line, (unsigned long long)r); return; }
    const int64_t beg = pos - 1 < 0 ? 0 : pos - 1;
    int64_t end = beg + ref_len;
    if (col >= 7) {                                       // INFO/END, the first "END=" at the start or after a ';'
        for (uint64_t i = info_b; i + 4 <= info_e; ++i) {
            if ((i == info_b || ld(text + i - 1) == ';') && ld(text + i) == 'E' && ld(text + i + 1) == 'N' &&
                ld(text + i + 2) == 'D' && ld(text + i + 3) == '=') {
                int64_t v = 0;
                int d = 0;
                for (uint64_t q = i + 4; q < info_e; ++q, ++d) {
                    const uint8_t ch = ld(text + q);
                    if (ch < '0' || ch > '9') break;
                    v = v * 10 + (ch - '0');
                }
                if (d && v > beg) end = v;
                break;
            }
        }
    }
    store_key(k, r, beg, end, voff_of(mt.ooff, mt.boff, mt.bend, mt.olen, mt.n, text_base + ls), min_shift, n_lvls, max_pos, c);
    // a contig run starts here when CHROM differs from the line before
    bool differs = r == 0;
    if (!differs) {
        const uint64_t ps = r > 1 ? line_end(li, r - 2) : 0;
        for (uint64_t i = 0;; ++i) {
            const uint8_t a = ld(text + ls + i), b = ld(text + ps + i);
            if (a != b) { differs = true; break; }
            if (ls + i == chrom_end) break;
        }
    }
    if (differs) add_run(c, runs, run_cap, r, ls);
}

__device__ __forceinline__ uint32_t ld32(const uint8_t *p) {
    return (uint32_t)ld(p) | (uint32_t)ld(p + 1) << 8 | (uint32_t)ld(p + 2) << 16 | (uint32_t)ld(p + 3) << 24;
}

// kernel 7a, BCF: one thread per record located by the BCF locator
__global__ void __launch_bounds__(256) bcf_index_keys_kernel(const uint8_t *__restrict__ text, uint64_t text_base,
                                                             const uint64_t *__restrict__ rec_off, uint64_t n, MemberTab mt,
                                                             int min_shift, int n_lvls, int64_t max_pos, Keys k, RunRec *runs,
                                                             uint32_t run_cap, Counters *c) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const uint64_t o = rec_off[r];
    const int32_t rid = (int32_t)ld32(text + o + 8), pos = (int32_t)ld32(text + o + 12), rlen = (int32_t)ld32(text + o + 16);
    store_key(k, r, pos, (int64_t)pos + rlen, voff_of(mt.ooff, mt.boff, mt.bend, mt.olen, mt.n, text_base + o), min_shift, n_lvls,
              max_pos, c);
    if (r == 0 || (int32_t)ld32(text + rec_off[r - 1] + 8) != rid) add_run(c, runs, run_cap, r, (uint64_t)(uint32_t)rid);
}

// kernel 7b: chunk openings, the linear index, sortedness
__global__ void __launch_bounds__(256) index_chunks_kernel(uint64_t n, Keys k, const uint64_t *__restrict__ run_rec,
                                                           const uint32_t *__restrict__ run_tid, uint32_t n_runs, int min_shift,
                                                           unsigned long long *lidx, uint64_t W, ChunkRec *chunks, uint64_t cap,
                                                           Counters *c) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    uint32_t lo = 0, hi = n_runs;                         // the run of r: run_rec[lo] <= r < run_rec[lo + 1]
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (run_rec[mid] <= r) lo = mid; else hi = mid;
    }
    const uint32_t tid = run_tid[lo];
    const int64_t beg = k.beg[r], end = k.end[r];
    const uint64_t voff = k.voff[r];
    const bool opens_run = run_rec[lo] == r;
    if (!opens_run && beg < k.beg[r - 1]) atomicMin(&c->unsorted, (unsigned long long)r);
    if (opens_run || k.bin[r] != k.bin[r - 1]) {
        const unsigned long long i = atomicAdd(&c->n_chunks, 1ull);
        if (i < cap) chunks[i] = ChunkRec{r, voff, tid, k.bin[r]};
    }
    unsigned long long *l = lidx + (uint64_t)tid * W;
    for (int64_t w = beg >> min_shift; w <= (end - 1) >> min_shift; ++w) atomicMin(l + w, (unsigned long long)voff);
}

// ---- host: hts_idx_finish and the hts-specs layout
int bin_first(int l) { return ((1 << (3 * l)) - 1) / 7; }
int bin_parent(int b) { return (b - 1) >> 3; }
int bin_bot(int bin, int n_lvls) {
    int l = 0;
    for (int b = bin; b; b = bin_parent(b)) ++l;
    return (bin - bin_first(l)) << (n_lvls - l) * 3;
}

struct Ref {
    std::map<uint32_t, std::vector<std::pair<uint64_t, uint64_t>>> bins;
    std::map<uint32_t, uint64_t> loff;
    std::vector<uint64_t> lidx;
};

void put32(std::vector<uint8_t> &o, uint32_t v) { for (int i = 0; i < 4; ++i) o.push_back((uint8_t)(v >> (8 * i))); }
void put64(std::vector<uint8_t> &o, uint64_t v) { for (int i = 0; i < 8; ++i) o.push_back((uint8_t)(v >> (8 * i))); }

void finish_ref(Ref &r, int n_lvls) {
    const uint32_t n_bins = ((1u << (3 * n_lvls + 3)) - 1) / 7;
    for (auto &kv : r.bins) {                             // update_loff: before the bins move
        if (kv.first >= n_bins) { r.loff[kv.first] = 0; continue; }
        const int bot = bin_bot((int)kv.first, n_lvls);
        r.loff[kv.first] = (size_t)bot < r.lidx.size() ? r.lidx[(size_t)bot] : 0;
    }
    for (int l = n_lvls; l > 0; --l) {                    // compress_binning: a bin spanning < 64 KiB of file moves up
        std::vector<uint32_t> keys;
        for (auto &kv : r.bins) if (kv.first >= (uint32_t)bin_first(l) && kv.first < n_bins) keys.push_back(kv.first);
        for (uint32_t b : keys) {
            auto &ch = r.bins[b];
            if (l < n_lvls) std::sort(ch.begin(), ch.end());
            if ((ch.back().second >> 16) - (ch.front().first >> 16) < 0x10000) {
                auto parent = r.bins.find((uint32_t)bin_parent((int)b));
                if (parent == r.bins.end()) continue;
                parent->second.insert(parent->second.end(), ch.begin(), ch.end());
                r.bins.erase(b);
            }
        }
    }
    if (r.bins.count(0)) std::sort(r.bins[0].begin(), r.bins[0].end());
    for (auto &kv : r.bins) {                             // chunks that start in the block where the one before ends
        if (kv.first >= n_bins) continue;
        auto &ch = kv.second;
        size_t m = 0;
        for (size_t i = 1; i < ch.size(); ++i) {
            if (ch[m].second >> 16 >= ch[i].first >> 16) ch[m].second = std::max(ch[m].second, ch[i].second);
            else ch[++m] = ch[i];
        }
        ch.resize(m + 1);
    }
}

template <class T>
cudaError_t upload(T **d, const std::vector<T> &h, cudaStream_t st) {
    cudaError_t e = dev_pool_alloc((void **)d, std::max<size_t>(1, h.size()) * sizeof(T));
    if (e == cudaSuccess && !h.empty()) e = cudaMemcpyAsync(*d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, st);
    return e;
}

struct DevBufs {                     // everything build_index puts on the device, freed on every return
    std::vector<void *> p;
    ~DevBufs() { for (void *x : p) dev_pool_free(x); }
    template <class T> cudaError_t alloc(T **d, uint64_t n) {
        cudaError_t e = dev_pool_alloc((void **)d, std::max<uint64_t>(1, n) * sizeof(T));
        if (e == cudaSuccess) p.push_back(*d);
        return e;
    }
    template <class T> cudaError_t put(T **d, const std::vector<T> &h, cudaStream_t st) {
        cudaError_t e = upload(d, h, st);
        if (e == cudaSuccess) p.push_back(*d);
        return e;
    }
};

int cuda_fail(cudaError_t e) { return api_fail(HB_ERR_CUDA, std::string("CUDA: ") + cudaGetErrorString(e)); }
#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return cuda_fail(e_); } while (0)

}  // namespace

int build_index(const IndexJob &j, std::vector<uint8_t> &out, IndexTimes *times) {
    cudaStream_t st = j.stream;
    const uint64_t n = j.n_rec;
    const int64_t max_pos = 1ll << (j.min_shift + 3 * j.n_lvls);
    const uint32_t nm = (uint32_t)j.ooff.size();
    const uint64_t *h_ooff = j.ooff.data(), *h_boff = j.boff.data(), *h_bend = j.bend.data();
    const uint32_t *h_olen = j.olen.data();
    DevBufs db;
    MemberTab mt{};
    mt.n = nm;
    {
        uint64_t *a, *b, *c;
        uint32_t *d;
        CK(db.put(&a, j.ooff, st)); CK(db.put(&b, j.boff, st)); CK(db.put(&c, j.bend, st)); CK(db.put(&d, j.olen, st));
        mt.ooff = a; mt.boff = b; mt.bend = c; mt.olen = d;
    }
    Keys k{};
    Counters *d_c = nullptr;
    CK(db.alloc(&k.beg, n)); CK(db.alloc(&k.end, n)); CK(db.alloc(&k.voff, n)); CK(db.alloc(&k.bin, n));
    CK(db.alloc(&d_c, 1));
    Counters hc;
    auto reset = [&]() -> cudaError_t {
        Counters z{0, 0, kNone, kNone, kNone, 0};
        return cudaMemcpyAsync(d_c, &z, sizeof z, cudaMemcpyHostToDevice, st);
    };
    auto fetch = [&]() -> cudaError_t {
        cudaError_t e = cudaMemcpyAsync(&hc, d_c, sizeof hc, cudaMemcpyDeviceToHost, st);
        return e == cudaSuccess ? cudaStreamSynchronize(st) : e;
    };
    cudaEvent_t ev[4];
    for (auto &e : ev) CK(cudaEventCreate(&e));
    struct EvFree { cudaEvent_t *e; ~EvFree() { for (int i = 0; i < 4; ++i) cudaEventDestroy(e[i]); } } ev_free{ev};
    const uint32_t grid = (uint32_t)std::max<uint64_t>(1, (n + 255) / 256);

    // ---- 7a
    RunRec *d_runs = nullptr;
    CK(db.alloc(&d_runs, kMaxIndexRuns));
    CK(reset());
    CK(cudaEventRecord(ev[0], st));
    if (n && j.bcf)
        bcf_index_keys_kernel<<<grid, 256, 0, st>>>(j.d_text, j.text_base, j.d_rec_off, n, mt, j.min_shift, j.n_lvls, max_pos, k,
                                                    d_runs, kMaxIndexRuns, d_c);
    else if (n)
        index_keys_kernel<<<grid, 256, 0, st>>>(j.d_text, j.text_base, j.li, n, mt, j.min_shift, j.n_lvls, max_pos, k, d_runs,
                                                kMaxIndexRuns, d_c);
    count_launch();
    CK(cudaEventRecord(ev[1], st));
    CK(cudaGetLastError());
    CK(fetch());
    if (hc.bad_line != kNone)
        return api_fail(HB_ERR_FORMAT, "line " + std::to_string(hc.bad_line + 1) + " of the body is not a VCF record");
    if (hc.bad_range != kNone)
        return api_fail(HB_ERR_FORMAT, "record " + std::to_string(hc.bad_range + 1) + " cannot be stored in a " +
                                           (j.csi ? "csi index with these parameters" : "tbi index: use a csi index"));
    if (hc.n_runs > kMaxIndexRuns) return api_fail(HB_ERR_FORMAT, "chromosome blocks not continuous (too many CHROM runs)");

    // ---- contig runs -> tids: VCF in order of first appearance, BCF the header's contig index
    std::vector<RunRec> runs(hc.n_runs);
    if (!runs.empty()) CK(d2h_copy(runs.data(), d_runs, runs.size() * sizeof(RunRec), st));
    std::sort(runs.begin(), runs.end(), [](const RunRec &a, const RunRec &b) { return a.rec < b.rec; });
    std::vector<std::string> names;
    std::vector<uint32_t> run_tid;
    std::vector<uint64_t> run_rec;
    std::vector<bool> seen;
    for (const RunRec &rr : runs) {
        uint32_t tid;
        if (j.bcf) {
            tid = (uint32_t)rr.key;
            if (tid >= j.n_contigs) return api_fail(HB_ERR_FORMAT, "BCF record with a contig outside the header's dictionary");
        } else {
            char buf[256];
            const uint64_t avail = std::min<uint64_t>(sizeof buf, j.total - j.text_base - rr.key);
            CK(d2h_copy(buf, j.d_text + rr.key, avail, st));
            const size_t len = (size_t)(std::find(buf, buf + avail, '\t') - buf);
            const std::string name(buf, len);
            const auto it = std::find(names.begin(), names.end(), name);
            tid = (uint32_t)(it - names.begin());
            if (it == names.end()) names.push_back(name);
        }
        if (tid >= seen.size()) seen.resize(tid + 1, false);
        if (seen[tid]) return api_fail(HB_ERR_FORMAT, "chromosome blocks not continuous");
        seen[tid] = true;
        run_tid.push_back(tid);
        run_rec.push_back(rr.rec);
    }
    const uint32_t n_ref = j.bcf ? j.n_contigs : (uint32_t)names.size();

    // ---- 7b
    const uint64_t W = hc.max_end ? ((hc.max_end - 1) >> j.min_shift) + 1 : 1;
    uint64_t *d_run_rec = nullptr;
    uint32_t *d_run_tid = nullptr;
    unsigned long long *d_lidx = nullptr;
    CK(db.put(&d_run_rec, run_rec, st));
    CK(db.put(&d_run_tid, run_tid, st));
    CK(db.alloc(&d_lidx, std::max<uint64_t>(1, n_ref) * W));
    uint64_t cap = std::min<uint64_t>(std::max<uint64_t>(n, 1), 1ull << 20);
    std::vector<ChunkRec> chunks;
    for (int attempt = 0; attempt < 2; ++attempt) {
        ChunkRec *d_chunks = nullptr;
        CK(db.alloc(&d_chunks, cap));
        CK(cudaMemsetAsync(d_lidx, 0xff, std::max<uint64_t>(1, n_ref) * W * 8, st));
        CK(reset());
        CK(cudaEventRecord(ev[2], st));
        if (n)
            index_chunks_kernel<<<grid, 256, 0, st>>>(n, k, d_run_rec, d_run_tid, (uint32_t)run_rec.size(), j.min_shift, d_lidx, W,
                                                      d_chunks, cap, d_c);
        count_launch();
        CK(cudaEventRecord(ev[3], st));
        CK(cudaGetLastError());
        CK(fetch());
        if (hc.unsorted != kNone)
            return api_fail(HB_ERR_FORMAT, "unsorted positions (record " + std::to_string(hc.unsorted + 1) + " of the body)");
        if (hc.n_chunks <= cap) {
            chunks.resize(hc.n_chunks);
            if (!chunks.empty()) CK(d2h_copy(chunks.data(), d_chunks, chunks.size() * sizeof(ChunkRec), st));
            break;
        }
        cap = hc.n_chunks;                                // exact count known: once more with room for all
    }
    std::vector<uint64_t> lidx(std::max<uint64_t>(1, n_ref) * W);
    CK(d2h_copy(lidx.data(), d_lidx, lidx.size() * 8, st));
    if (times) {
        cudaEventElapsedTime(&times->ms_keys, ev[0], ev[1]);
        cudaEventElapsedTime(&times->ms_chunks, ev[2], ev[3]);
    }
    const auto t_host = std::chrono::steady_clock::now();

    // ---- host: chunk ends, meta pseudo-bin, linear index, hts_idx_finish
    std::sort(chunks.begin(), chunks.end(), [](const ChunkRec &a, const ChunkRec &b) { return a.rec < b.rec; });
    const uint64_t final_off = voff_of(h_ooff, h_boff, h_bend, h_olen, nm, j.total);
    const uint32_t meta_bin = ((1u << (3 * j.n_lvls + 3)) - 1) / 7;
    std::vector<Ref> refs(n_ref);
    for (size_t i = 0; i < chunks.size(); ++i) {
        const uint64_t v = i + 1 < chunks.size() ? chunks[i + 1].voff : final_off;
        refs[chunks[i].tid].bins[chunks[i].bin].push_back({chunks[i].voff, v});
    }
    for (size_t i = 0; i < run_rec.size(); ++i) {
        const uint64_t first = run_rec[i], last = i + 1 < run_rec.size() ? run_rec[i + 1] : n;
        const auto at = std::lower_bound(chunks.begin(), chunks.end(), first, [](const ChunkRec &c, uint64_t r) { return c.rec < r; });
        const auto nx = i + 1 < run_rec.size()
                            ? std::lower_bound(chunks.begin(), chunks.end(), last, [](const ChunkRec &c, uint64_t r) { return c.rec < r; })
                            : chunks.end();
        const uint64_t off_beg = at->voff, off_end = nx == chunks.end() ? final_off : nx->voff;
        Ref &r = refs[run_tid[i]];
        r.bins[meta_bin] = {{off_beg, off_end}, {last - first, 0}};
        const uint64_t *l = lidx.data() + (uint64_t)run_tid[i] * W;
        uint64_t nl = W;
        while (nl && l[nl - 1] == kNone) --nl;
        r.lidx.assign(l, l + nl);
        for (uint64_t w = 0; w < nl; ++w)
            if (r.lidx[w] == kNone) r.lidx[w] = w ? r.lidx[w - 1] : off_beg;
        finish_ref(r, j.n_lvls);
    }
    // ---- the hts-specs layout
    std::string meta;                                     // tabix conf + sequence names (TBI; CSI of a VCF as l_aux)
    if (!j.bcf) {
        std::vector<uint8_t> m;
        for (int v : {2, 1, 2, 0, (int)'#', 0}) put32(m, (uint32_t)v);
        std::string nmb;
        for (const std::string &s : names) { nmb += s; nmb.push_back('\0'); }
        put32(m, (uint32_t)nmb.size());
        meta.assign(m.begin(), m.end());
        meta += nmb;
    }
    out.clear();
    if (!j.csi) {
        out.insert(out.end(), {'T', 'B', 'I', 1});
        put32(out, n_ref);
        out.insert(out.end(), meta.begin(), meta.end());
    } else {
        out.insert(out.end(), {'C', 'S', 'I', 1});
        put32(out, (uint32_t)j.min_shift); put32(out, (uint32_t)j.n_lvls); put32(out, (uint32_t)meta.size());
        out.insert(out.end(), meta.begin(), meta.end());
        put32(out, n_ref);
    }
    for (const Ref &r : refs) {
        put32(out, (uint32_t)r.bins.size());
        for (const auto &kv : r.bins) {
            put32(out, kv.first);
            if (j.csi) put64(out, r.loff.count(kv.first) ? r.loff.at(kv.first) : 0);
            put32(out, (uint32_t)kv.second.size());
            for (const auto &c : kv.second) { put64(out, c.first); put64(out, c.second); }
        }
        if (!j.csi) {
            put32(out, (uint32_t)r.lidx.size());
            for (uint64_t o : r.lidx) put64(out, o);
        }
    }
    put64(out, 0);                                        // n_no_coor
    if (times) times->ms_host = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_host).count();
    return HB_OK;
}

}  // namespace hb
