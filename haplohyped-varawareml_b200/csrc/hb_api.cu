// hb_api.cu -- host side of libhaplo_b200: the C ABI of include/haplo_b200.h sections A and B.
//
// Mirrors the reference's native layer (cpp/parse_vcf.cpp + the BcfReader of cpp/vcfpp.h) above
// the kernels: open a .vcf / .vcf.gz (BGZF or plain gzip), read the header (sample names,
// INFO/END type; vcfpp.h:1378-1385), ship the decompressed body to HBM, run tokenize -> sites ->
// GT decode once for ALL samples, and answer load_vcf(sample) / load_vcf_without_sample calls
// from that device-resident result.  No CPU parsing path exists: without a CUDA device every
// entry point fails with HB_ERR_CUDA.
#include <zlib.h>

#include <algorithm>
#include <chrono>
#include <atomic>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>
#include <thread>
#include <vector>

#include "../../include/haplo_b200.h"
#include "hb_internal.h"
#include "hb_parse_struct.h"
#include "hb_index.h"
#include "hb_tabix.h"

namespace hb {

static thread_local std::string g_err;
static std::atomic<uint64_t> g_launches{0};
static std::atomic<uint64_t> g_text_limit{0};        // hb_parse_set_text_limit: 0 = from free device memory
static std::atomic<uint32_t> g_walker_lines{16};   // hb_set_walker_lines
static std::atomic<uint64_t> g_bcf_segment{0};     // hb_set_bcf_segment_bytes: 0 = max(64 KiB, 8 x the first record)
static const char *const kBcfNoStream =
    "BCF streaming is not supported: read a .bcf with hb_parse_file, hb_parse_vcf_bytes or hb_load_vcf";
void count_launch(uint64_t n) { g_launches += n; }

static int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}
int api_fail(int code, const std::string &msg) { return fail(code, msg); }
static int fail_cuda(cudaError_t e, const char *where = "") {
    return fail(HB_ERR_CUDA, std::string("CUDA: ") + cudaGetErrorString(e) + where);
}
#define CU(expr)                                                   \
    do {                                                           \
        cudaError_t e_ = (expr);                                   \
        if (e_ != cudaSuccess) return fail_cuda(e_, " at " #expr); \
    } while (0)

static double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

static int ensure_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(HB_ERR_CUDA, "no CUDA device: libhaplo_b200 has no CPU fallback (" +
                                     std::string(e == cudaSuccess ? "0 devices" : cudaGetErrorString(e)) + ")");
    if (device < 0 || device >= n) return fail(HB_ERR_ARG, "bad device ordinal");
    CU(cudaSetDevice(device));
    // cudaGetDeviceProperties takes tens of milliseconds when the GPU is busy: two attributes, looked up once per device
    static std::atomic<int> cc_major[64];
    int major = device < 64 ? cc_major[device].load() : 0, minor = 0;
    if (!major) {
        CU(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
        CU(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device));
        if (major != 10) return fail(HB_ERR_CUDA, "libhaplo_b200 is built for sm_100a only; device is sm_" +
                                                      std::to_string(major) + std::to_string(minor));
        if (device < 64) cc_major[device].store(major);
    }
    return HB_OK;
}

static void parse_region(const char *s, RegionArg &rg) {
    memset(&rg, 0, sizeof rg);
    rg.beg0 = 0;
    rg.end0 = INT64_MAX;
    if (!s || !*s) return;
    rg.has_region = 1;
    const char *colon = strrchr(s, ':');
    size_t nlen = colon ? (size_t)(colon - s) : strlen(s);
    if (nlen >= sizeof rg.chrom) nlen = sizeof rg.chrom - 1;
    memcpy(rg.chrom, s, nlen);
    rg.chrom_len = (uint32_t)nlen;
    if (colon) {
        long long v = 0;
        bool any = false;
        const char *p = colon + 1;
        for (; *p && *p != '-'; ++p)
            if (*p >= '0' && *p <= '9') { v = v * 10 + (*p - '0'); any = true; }
        if (any && v > 0) rg.beg0 = v - 1;
        if (*p == '-') {
            v = 0; any = false;
            for (++p; *p; ++p)
                if (*p >= '0' && *p <= '9') { v = v * 10 + (*p - '0'); any = true; }
            if (any) rg.end0 = v;
        }
    }
}

}  // namespace hb

using namespace hb;

// =============================================================================================
// hb_parse: one device-resident parse
// =============================================================================================

// ---- big device buffers are pooled.  cudaMalloc / cudaFree of GB-sized buffers take anything from 10 to 500 ms on these
// hosts (measured inside the streaming entry points); a converter that walks 22 chromosome files, or a caller that makes a
// parse handle per file, would pay that for the text buffer, both allele planes and every column every time -- and the SMALL
// ones are no cheaper: r02's trace of the conversion step showed calls stalling 0.2-1.1 s in phases whose only driver work
// was a handful of cudaMalloc / cudaFree of KB-sized tables.  Every buffer that is freed goes to an idle list (at most 512 per
// process; sizes are rounded up to 512 bytes) and is handed out again to requests it fits with at most 50 % (or 64 KB) of
// slack; when a cudaMalloc fails the list is emptied and the call retried; hb_cache_clear() empties it too.
namespace {
struct DevPool {
    static constexpr uint64_t kMin = 1;
    static constexpr size_t kMaxIdle = 512;
    struct Item { void *p; uint64_t bytes; int device; };
    std::mutex mu;
    std::map<void *, Item> live;                 // big allocations handed out
    std::vector<Item> idle;
} g_pool;
}
namespace hb {
uint64_t dev_pool_idle_bytes() {                 // on the current device
    int cur = 0;
    cudaGetDevice(&cur);
    std::lock_guard<std::mutex> lk(g_pool.mu);
    uint64_t sum = 0;
    for (const auto &it : g_pool.idle) if (it.device == cur) sum += it.bytes;
    return sum;
}
void dev_pool_flush() {
    std::vector<DevPool::Item> items;
    {
        std::lock_guard<std::mutex> lk(g_pool.mu);
        items.swap(g_pool.idle);
    }
    int cur = 0;
    cudaGetDevice(&cur);
    for (auto &it : items) { cudaSetDevice(it.device); cudaFree(it.p); }
    cudaSetDevice(cur);
}
cudaError_t dev_pool_alloc(void **out, uint64_t bytes) {
    *out = nullptr;
    if (bytes == 0) bytes = 1;
    bytes = (bytes + 511) & ~511ull;
    int device = 0;
    cudaGetDevice(&device);
    if (bytes >= DevPool::kMin) {
        std::lock_guard<std::mutex> lk(g_pool.mu);
        size_t best = (size_t)-1;
        for (size_t i = 0; i < g_pool.idle.size(); ++i) {
            const auto &it = g_pool.idle[i];
            if (it.device == device && it.bytes >= bytes && it.bytes <= bytes + std::max<uint64_t>(bytes / 2, 65536) &&
                (best == (size_t)-1 || it.bytes < g_pool.idle[best].bytes)) best = i;
        }
        if (best != (size_t)-1) {
            DevPool::Item it = g_pool.idle[best];
            g_pool.idle.erase(g_pool.idle.begin() + (long)best);
            g_pool.live[it.p] = it;
            *out = it.p;
            return cudaSuccess;
        }
    }
    cudaError_t e = cudaMalloc(out, bytes);
    if (e != cudaSuccess) {                      // memory held by idle buffers may be what is missing
        cudaGetLastError();
        dev_pool_flush();
        e = cudaMalloc(out, bytes);
    }
    if (e == cudaSuccess && bytes >= DevPool::kMin) {
        std::lock_guard<std::mutex> lk(g_pool.mu);
        g_pool.live[*out] = DevPool::Item{*out, bytes, device};
    }
    return e;
}
void dev_pool_free(void *p) {
    if (!p) return;
    DevPool::Item it{nullptr, 0, 0};
    {
        std::lock_guard<std::mutex> lk(g_pool.mu);
        auto f = g_pool.live.find(p);
        if (f != g_pool.live.end()) { it = f->second; g_pool.live.erase(f); }
    }
    if (!it.p) { cudaFree(p); return; }
    cudaDeviceSynchronize();                     // what cudaFree would have done: nothing in flight still uses the buffer
    {
        std::lock_guard<std::mutex> lk(g_pool.mu);
        if (g_pool.idle.size() < DevPool::kMaxIdle) { g_pool.idle.push_back(it); return; }
    }
    cudaFree(p);
}
void dev_pool_release(void *p) {
    {
        std::lock_guard<std::mutex> lk(g_pool.mu);
        g_pool.live.erase(p);
    }
    cudaFree(p);
}
}  // namespace hb

static void free_dev(void *p) { hb::dev_pool_free(p); }

// ---- device -> host memory of any kind.  A pinned destination gets one asynchronous copy.  A pageable one is served
// through two pinned staging buffers (the D2H of piece k + 1 overlaps the memcpy of piece k): the driver's own pageable
// path ran at 3.7 GB/s on these hosts and stalled at random.  Both return when the data is in place.
namespace {
struct D2HStage {
    size_t cap = 32ull << 20;                    // HB_D2H_STAGE_KB overrides (the tests use a small one to walk every piece shape)
    std::mutex mu;
    uint8_t *buf[2] = {nullptr, nullptr};
    cudaEvent_t ev[64][2] = {};                  // per device: an event is recorded on streams of its own device only
    bool tried = false, ok = false;
} g_d2h;
bool is_pinned(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}
bool d2h_stage_ready() {                        // g_d2h.mu held
    if (!g_d2h.tried) {
        g_d2h.tried = true;
        if (const char *e = getenv("HB_D2H_STAGE_KB")) { const long v = atol(e); if (v >= 4 && v <= (1 << 22)) g_d2h.cap = (size_t)v << 10; }
        g_d2h.ok = cudaMallocHost((void **)&g_d2h.buf[0], g_d2h.cap) == cudaSuccess &&
                   cudaMallocHost((void **)&g_d2h.buf[1], g_d2h.cap) == cudaSuccess;
        if (!g_d2h.ok) cudaGetLastError();
    }
    return g_d2h.ok;
}
cudaEvent_t *d2h_events() {                     // g_d2h.mu held; the two events of the current device, or nullptr
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); return nullptr; }
    if (!g_d2h.ev[dev][0]) {
        if (cudaEventCreateWithFlags(&g_d2h.ev[dev][0], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&g_d2h.ev[dev][1], cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    }
    return g_d2h.ev[dev];
}
}  // namespace
namespace hb {
bool host_is_pinned(const void *p) { return is_pinned(p); }
// height rows of width bytes, spitch apart on the device, dpitch apart on the host
cudaError_t d2h_copy_2d(void *dst, uint64_t dpitch, const void *src, uint64_t spitch, uint64_t width, uint64_t height, cudaStream_t stream) {
    if (!width || !height) return cudaSuccess;
    cudaError_t e;
    std::unique_lock<std::mutex> lk(g_d2h.mu, std::defer_lock);
    cudaEvent_t *ev = nullptr;
    if (!is_pinned(dst)) {
        lk.lock();
        ev = d2h_stage_ready() ? d2h_events() : nullptr;
    }
    if (!ev) {                                  // a pinned destination, or no pinned memory to be had: the plain path
        e = height == 1 ? cudaMemcpyAsync(dst, src, width, cudaMemcpyDeviceToHost, stream)
                        : cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, height, cudaMemcpyDeviceToHost, stream);
        return e == cudaSuccess ? cudaStreamSynchronize(stream) : e;
    }
    // pieces: whole rows when a row fits the staging buffer, else parts of one row
    struct Piece { uint64_t row, col, rows, bytes; };
    auto land = [&](const Piece &pc, int b) {
        if (pc.rows == 0) return;
        if (pc.col == 0 && pc.bytes == width && dpitch == width) memcpy((uint8_t *)dst + pc.row * dpitch, g_d2h.buf[b], pc.rows * width);
        else if (pc.bytes == width) for (uint64_t r = 0; r < pc.rows; ++r) memcpy((uint8_t *)dst + (pc.row + r) * dpitch, g_d2h.buf[b] + r * width, width);
        else memcpy((uint8_t *)dst + pc.row * dpitch + pc.col, g_d2h.buf[b], pc.bytes);
    };
    Piece prev{0, 0, 0, 0};
    int k = 0;
    uint64_t row = 0, col = 0;
    while (row < height) {
        Piece pc;
        if (width <= g_d2h.cap) { pc = Piece{row, 0, std::min<uint64_t>(height - row, g_d2h.cap / width), width}; }
        else { pc = Piece{row, col, 1, std::min<uint64_t>(width - col, g_d2h.cap)}; }
        const int b = k & 1;
        const uint8_t *sp = (const uint8_t *)src + pc.row * spitch + pc.col;
        if (pc.bytes == width && pc.rows > 1) e = cudaMemcpy2DAsync(g_d2h.buf[b], width, sp, spitch, width, pc.rows, cudaMemcpyDeviceToHost, stream);
        else e = cudaMemcpyAsync(g_d2h.buf[b], sp, pc.bytes, cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaEventRecord(ev[b], stream);
        if (e != cudaSuccess) return e;
        if (k > 0) {                            // the piece before is complete: put it in place while this one is in flight
            e = cudaEventSynchronize(ev[b ^ 1]);
            if (e != cudaSuccess) return e;
            land(prev, b ^ 1);
        }
        prev = pc;
        ++k;
        if (pc.bytes == width) { row += pc.rows; col = 0; }
        else { col += pc.bytes; if (col >= width) { col = 0; ++row; } }
    }
    e = cudaEventSynchronize(ev[(k - 1) & 1]);
    if (e != cudaSuccess) return e;
    land(prev, (k - 1) & 1);
    return cudaSuccess;
}
cudaError_t d2h_copy(void *dst, const void *src, uint64_t bytes, cudaStream_t stream) {
    return d2h_copy_2d(dst, bytes, src, bytes, bytes, 1, stream);
}
}  // namespace hb

namespace { void pin_slot_release(hb::DevStatus *s); }

template <typename T>
static int dev_alloc(T **p, uint64_t n) {
    if (*p) { free_dev(*p); *p = nullptr; }
    if (n == 0) n = 1;
    cudaError_t e = hb::dev_pool_alloc((void **)p, n * sizeof(T));
    if (e != cudaSuccess) return fail(HB_ERR_MEM, std::string("cudaMalloc: ") + cudaGetErrorString(e));
    return HB_OK;
}
#define TRY(expr) do { int rc_ = (expr); if (rc_ != HB_OK) return rc_; } while (0)

// the capacity a buffer of n elements is made with: exact the first time, with room to grow when it had to grow before
static uint64_t regrown(uint64_t n, bool had) { return had ? n + n / 8 + 1024 : n; }

// a buffer that only grows: reallocated to exactly `need` elements when it holds fewer or is not there
template <class T>
static int grow(T *&p, uint64_t &cap, uint64_t need) {
    if (cap < need || !p) {
        TRY(dev_alloc(&p, need));
        cap = need;
    }
    return HB_OK;
}

static int alloc_rows(SiteRows &r, uint64_t cap) {
    TRY(dev_alloc(&r.start, cap)); TRY(dev_alloc(&r.stop, cap)); TRY(dev_alloc(&r.ref, cap)); TRY(dev_alloc(&r.alt, cap));
    TRY(dev_alloc(&r.chrom_abs, cap)); TRY(dev_alloc(&r.chrom_len, cap)); TRY(dev_alloc(&r.chrom5, cap));
    TRY(dev_alloc(&r.rowinfo, cap));
    r.cap = cap;
    return HB_OK;
}

static void free_rows(SiteRows &r) {
    free_dev(r.start); free_dev(r.stop); free_dev(r.ref); free_dev(r.alt);
    free_dev(r.chrom_len); free_dev(r.chrom_abs); free_dev(r.chrom5); free_dev(r.rowinfo);
    r = SiteRows();
}

void hb_parse_free(hb_parse *p) {
    if (!p) return;
    const double t_free0 = getenv("HB_TRACE") ? now_ms() : 0;
    cudaSetDevice(p->device);
    if (p->side) cudaStreamSynchronize(p->side);
    free_dev(p->d_text_owned); free_dev(p->d_nl_after); free_dev(p->d_cta); free_dev(p->d_cbase); free_dev(p->d_cp);
    free_dev(p->d_st); free_rows(p->rows); free_dev(p->d_nu_rows);
    free_dev(p->d_sites_state); free_dev(p->d_gt[0]); free_dev(p->d_gt[1]); free_dev(p->d_bits); free_dev(p->d_ploidy);
    free_dev(p->d_badgt); free_dev(p->d_run_rows);
    free_dev(p->d_wstart); free_dev(p->d_wrow); free_dev(p->d_verify); free_dev(p->d_wcount);
    free_rows(p->walk_pad);
    free_dev(p->d_sel_mask); free_dev(p->d_sel_base);
    if (hb_parse::Bcf *b = p->bcf) {
        free_dev(b->d_contigs); free_dev(b->d_names); free_dev(b->d_rec_off); free_dev(b->d_blk_count); free_dev(b->d_blk_base);
        free_dev(b->seg.start); free_dev(b->seg.exit); free_dev(b->seg.bad); free_dev(b->seg.base); free_dev(b->seg.count);
        free_dev(b->seg.flag);
        delete b;
    }
    for (auto &e : p->ev) if (e) cudaEventDestroy(e);
    if (p->side) { cudaStreamSynchronize(p->side); cudaStreamDestroy(p->side); }
    if (p->ev_runs) cudaEventDestroy(p->ev_runs);
    pin_slot_release(p->h_st_pin);
    if (t_free0 > 0) fprintf(stderr, "[hb_parse_free] %.1f ms\n", now_ms() - t_free0);
    delete p;
}

// device status -> host, through PINNED memory: a D2H copy into pageable memory is staged by the driver and was seen to
// wait behind the 256 MiB H2D copy of the next slab that streams on another stream (hb_parse_stream_host)
// pinned landing slots for the status words: cudaMallocHost / cudaFreeHost per handle cost up to 170 ms each on these hosts,
// so one pinned block is made per process and its slots are handed out and taken back
namespace {
struct PinSlots {
    static constexpr int kSlots = 256;
    static constexpr size_t kStride = 16896;     // DevStatus (256 B reserved) + 1024 CtaTok + 1025 prefix sums of the tokenizer path
    static constexpr size_t kCtaOff = 256, kBaseOff = 256 + 8192;
    std::mutex mu;
    uint8_t *base = nullptr;
    bool tried = false;
    std::vector<int> free_list;
} g_pin;
DevStatus *pin_slot_acquire() {
    std::lock_guard<std::mutex> lk(g_pin.mu);
    if (!g_pin.tried) {
        g_pin.tried = true;
        static_assert(sizeof(DevStatus) <= PinSlots::kCtaOff, "status words fit their reserve");
        if (cudaMallocHost((void **)&g_pin.base, PinSlots::kStride * PinSlots::kSlots) != cudaSuccess) { cudaGetLastError(); g_pin.base = nullptr; }
        else for (int i = PinSlots::kSlots - 1; i >= 0; --i) g_pin.free_list.push_back(i);
    }
    if (!g_pin.base || g_pin.free_list.empty()) return nullptr;
    const int i = g_pin.free_list.back();
    g_pin.free_list.pop_back();
    return reinterpret_cast<DevStatus *>(g_pin.base + (size_t)i * PinSlots::kStride);
}
void pin_slot_release(DevStatus *s) {
    if (!s) return;
    std::lock_guard<std::mutex> lk(g_pin.mu);
    g_pin.free_list.push_back((int)((reinterpret_cast<uint8_t *>(s) - g_pin.base) / PinSlots::kStride));
}
}  // namespace

static int fetch_status(hb_parse *p) {
    if (!p->h_st_pin) p->h_st_pin = pin_slot_acquire();
    DevStatus *land = p->h_st_pin ? p->h_st_pin : &p->h_st;      // no pinned slot left: the pageable copy still works
    cudaError_t e = cudaMemcpyAsync(land, p->d_st, sizeof(DevStatus), cudaMemcpyDeviceToHost, p->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(p->stream);
    if (e != cudaSuccess) return fail_cuda(e);
    if (land != &p->h_st) p->h_st = *land;
    return HB_OK;
}

// look at the first record of the body: FORMAT == "GT" -> newline-only tokenizer is enough;
// and exactly 4 bytes per sample after the 9th tab -> the walker (hb_walk.cu) applies
static void probe_head(const uint8_t *h, size_t n, uint32_t n_samples, bool &gt_only, bool &uniform,
                       uint64_t &first_line_len) {
    gt_only = false;
    uniform = false;
    first_line_len = 0;
    size_t i = 0, tab9 = 0;
    int f = 0;
    size_t fs = 0;
    for (; i < n; ++i) {
        if (h[i] == '\t' || h[i] == '\n') {
            if (f == 8) { gt_only = (i - fs == 2 && h[fs] == 'G' && h[fs + 1] == 'T'); tab9 = i; }
            if (h[i] == '\n') break;
            ++f;
            fs = i + 1;
        }
    }
    if (i < n) {
        first_line_len = i + 1;
        size_t e = i;
        if (e > 0 && h[e - 1] == '\r') --e;
        uniform = gt_only && f >= 9 && e - tab9 == 4ull * n_samples;
    }
}

// ---- records located by the tokenizer (any text): kernels 1 and 2
static int index_by_tokenizer(hb_parse *p, const Launch &L) {
    const uint64_t tile = tokenize_tile_bytes();
    const uint64_t n_tiles = (p->nbytes + tile - 1) / tile;
    {
        // one contiguous range of tiles per persistent CTA, 2 CTAs per SM (re-planned per run: a handle may
        // be re-run on text of another length, see hb_parse_stream_host)
        uint64_t want = std::min<uint64_t>((uint64_t)p->sm_count * 2, n_tiles);
        if (want > 1024) want = 1024;
        p->tiles_per_cta = (n_tiles + want - 1) / want;
        p->n_cta = (uint32_t)((n_tiles + p->tiles_per_cta - 1) / p->tiles_per_cta);
        uint64_t est = p->tiles_per_cta * tile / p->first_line_len;
        p->stage_cap = std::max<uint32_t>(p->stage_cap, (uint32_t)std::min<uint64_t>(est + est / 2 + 64, 0x7fffffffull));
        if (!p->d_cta) {
            TRY(dev_alloc(&p->d_cta, 1024));
            TRY(dev_alloc(&p->d_cbase, 1024 + 1));
        }
    }
    // per-CTA counts come back, and their prefix sums go out, through the handle's pinned block when it has one
    // (copies from / to pageable memory stall behind the big DMA transfers of a streaming caller)
    std::vector<CtaTok> v_cta;
    std::vector<uint64_t> v_base;
    if (!p->h_st_pin) p->h_st_pin = pin_slot_acquire();
    CtaTok *h_cta;
    uint64_t *h_base;
    if (p->h_st_pin && p->n_cta <= 1024) {
        h_cta = reinterpret_cast<CtaTok *>(reinterpret_cast<uint8_t *>(p->h_st_pin) + PinSlots::kCtaOff);
        h_base = reinterpret_cast<uint64_t *>(reinterpret_cast<uint8_t *>(p->h_st_pin) + PinSlots::kBaseOff);
    } else {
        v_cta.resize(p->n_cta); v_base.resize(p->n_cta + 1);
        h_cta = v_cta.data(); h_base = v_base.data();
    }
    for (int attempt = 0; attempt < 2; ++attempt) {
        uint64_t need = (uint64_t)p->n_cta * p->stage_cap;
        TRY(grow(p->d_nl_after, p->nl_after_cap, need));
        if (p->with_tabs) {
            TRY(grow(p->d_cp, p->cp_cap, need * p->ncp));
            CU(cudaMemsetAsync(p->d_cp, 0xff, p->cp_cap * sizeof(uint64_t), p->stream));
        }
        CU(cudaEventRecord(p->ev[0], p->stream));
        launch_tokenize(p->with_tabs, p->d_text, p->nbytes, p->n_cta, p->tiles_per_cta, p->d_nl_after, p->stage_cap,
                        p->d_cp, p->ncp, p->d_cta, L);
        CU(cudaEventRecord(p->ev[1], p->stream));
        CU(cudaMemcpyAsync(h_cta, p->d_cta, p->n_cta * sizeof(CtaTok), cudaMemcpyDeviceToHost, p->stream));
        CU(cudaStreamSynchronize(p->stream));
        CU(cudaGetLastError());
        uint32_t mx = 0;
        h_base[0] = 0;
        for (uint32_t c = 0; c < p->n_cta; ++c) {
            mx = std::max(mx, h_cta[c].n_newlines);
            h_base[c + 1] = h_base[c] + h_cta[c].n_newlines;
        }
        if ((uint64_t)mx + 1 <= p->stage_cap) break;
        if (attempt == 1) return fail(HB_ERR_MEM, "line index overflow");
        p->stage_cap = mx + 2;                 // exact counts are known even when the index overflowed
    }
    CU(cudaMemcpyAsync(p->d_cbase, h_base, (p->n_cta + 1) * 8ull, cudaMemcpyHostToDevice, p->stream));
    const uint64_t n_lines = h_base[p->n_cta];
    p->n_lines = n_lines;
    LineIndex li{p->d_nl_after, p->d_cbase, p->n_cta, p->stage_cap};

    SiteRows &r = p->rows;
    // (a side buffer whose allocation failed is null: the next run allocates the rows again)
    if (r.cap < n_lines || !r.start || !p->d_nu_rows || !p->d_sites_state) {
        const uint64_t cap = std::max(regrown(n_lines, r.start), r.cap);
        TRY(alloc_rows(r, cap));
        TRY(dev_alloc(&p->d_nu_rows, cap));
        TRY(dev_alloc(&p->d_sites_state, (cap + 255) / 256 + 1));
    }
    launch_sites(p->d_text, li, n_lines, p->n_cols, p->rg, p->end_is_int, p->want_gt, p->with_tabs, r, p->d_nu_rows,
                 p->d_sites_state, p->d_st, L);
    CU(cudaEventRecord(p->ev[2], p->stream));
    TRY(fetch_status(p));
    CU(cudaGetLastError());
    p->index_used = p->with_tabs ? 2 : 1;
    return HB_OK;
}

// ---- records located by walking heads (uniform GT-only text): hb_walk.cu
static int index_by_walker(hb_parse *p, const Launch &L) {
    {
        const uint32_t k = g_walker_lines.load();      // lines per walker: 16 (one-pass walker, r02u: 10 / 12 / 14 / 16 give 0.61 / 0.49 / 0.51 / 0.42 ms for locate)
        p->n_walkers = walk_plan(p->nbytes, p->first_line_len, k, &p->walk_range);
        if (!p->d_wstart || p->n_walkers > p->walk_cap) {
            TRY(dev_alloc(&p->d_wstart, (uint64_t)p->n_walkers + 1));
            TRY(dev_alloc(&p->d_wrow, p->n_walkers));
            TRY(dev_alloc(&p->d_wcount, p->n_walkers));
            p->walk_cap = p->n_walkers;
        }
    }
    {   // padded rows of the walk and the list of spans to verify: sized by the walkers, known before anything runs
        const uint64_t cap = (uint64_t)p->n_walkers * kWalkSlots;
        if (p->walk_pad.cap < cap) TRY(alloc_rows(p->walk_pad, cap));
        TRY(grow(p->d_verify, p->verify_cap, cap));
    }
    CU(cudaEventRecord(p->ev[0], p->stream));
    launch_walk(p->d_text, p->nbytes, p->n_cols, p->walk_range, p->n_walkers, p->rg, p->end_is_int, p->d_wstart, p->d_wcount,
                p->d_wrow, p->walk_pad, p->d_verify, p->verify_cap, p->d_st, L);
    CU(cudaEventRecord(p->ev[1], p->stream));
    TRY(fetch_status(p));
    CU(cudaGetLastError());
    const uint64_t n_lines = p->h_st.n_lines, n_rec = p->h_st.n_records;
    p->n_lines = n_lines;
    SiteRows &r = p->rows;
    if (r.cap < n_rec || !r.start || !p->d_nu_rows) {
        const uint64_t cap = std::max(regrown(n_rec, r.start), r.cap);
        TRY(alloc_rows(r, cap));
        TRY(dev_alloc(&p->d_nu_rows, cap));
        // the tokenizer sizes its tile state by the rows: a fallback to it on this handle makes it again
        free_dev(p->d_sites_state);
        p->d_sites_state = nullptr;
    }
    launch_walk_compact(p->d_text, p->nbytes, p->n_cols, p->n_walkers, p->d_wcount, p->d_wrow, p->walk_pad, r, p->d_nu_rows,
                        p->d_verify, p->verify_cap, p->d_st, L);
    CU(cudaEventRecord(p->ev[2], p->stream));
    p->index_used = 3;
    return HB_OK;
}

static int bcf_malformed(uint64_t bad, uint32_t n_samples, uint32_t n_contigs) {
    const std::string at = "BCF record at byte " + std::to_string(bad & ((1ull << 56) - 1)) + " of the body";
    switch ((uint32_t)(bad >> 56)) {
        case kBcfTruncated: return fail(HB_ERR_FORMAT, at + " is truncated: its length runs past the end of the data");
        case kBcfNSample: return fail(HB_ERR_FORMAT, at + ": n_sample differs from the header's " + std::to_string(n_samples) + " samples");
        case kBcfContig: return fail(HB_ERR_FORMAT, at + ": CHROM is not an index of the header's " + std::to_string(n_contigs) + " contigs");
        default: return fail(HB_ERR_FORMAT, at + " has a malformed record header");
    }
}

// ---- BCF records located by chaining their lengths, proven exact segment by segment: hb_bcf.cu
static int index_bcf(hb_parse *p, const Launch &L) {
    hb_parse::Bcf &b = *p->bcf;
    const uint32_t nc = (uint32_t)b.contigs.size();
    if (!b.first_len) {
        uint32_t h[2] = {0, 0};
        if (p->nbytes >= 8) {
            CU(cudaMemcpyAsync(h, p->d_text, 8, cudaMemcpyDeviceToHost, p->stream));
            CU(cudaStreamSynchronize(p->stream));
        }
        b.first_len = 8ull + h[0] + h[1];
    }
    // segments of several records each: the warp that finds a segment's first record scans at most about one record
    BcfSegs &sg = b.seg;
    const uint64_t knob = g_bcf_segment.load();
    sg.bytes = knob ? knob : std::max<uint64_t>(64ull << 10, std::min<uint64_t>(8 * b.first_len, 1ull << 40));
    sg.n = (p->nbytes + sg.bytes - 1) / sg.bytes;
    if (sg.cap < sg.n || !sg.start) {
        TRY(dev_alloc(&sg.start, sg.n)); TRY(dev_alloc(&sg.exit, sg.n)); TRY(dev_alloc(&sg.bad, sg.n));
        TRY(dev_alloc(&sg.base, sg.n)); TRY(dev_alloc(&sg.count, sg.n)); TRY(dev_alloc(&sg.flag, sg.n));
        sg.cap = sg.n;
    }
    CU(cudaEventRecord(p->ev[0], p->stream));
    launch_bcf_chain(p->d_text, p->nbytes, p->n_cols, nc, sg, true, L);
    for (;;) {                                   // until every segment's start is the exit of the segment before it
        CU(cudaMemsetAsync(&p->d_st->bcf_fail, 0xff, 8, p->stream));
        CU(cudaMemsetAsync(&p->d_st->bcf_records, 0, 8, p->stream));
        launch_bcf_verify(sg, p->d_st, L);
        TRY(fetch_status(p));
        CU(cudaGetLastError());
        const uint64_t f = p->h_st.bcf_fail;
        if (f == ~0ull) break;
        if (f & 1) {                             // a proven chain met a record that fails the header test
            uint64_t bad = 0;
            CU(cudaMemcpy(&bad, sg.bad + (f >> 1), 8, cudaMemcpyDeviceToHost));
            return bcf_malformed(bad, p->n_cols, nc);
        }
        launch_bcf_chain(p->d_text, p->nbytes, p->n_cols, nc, sg, false, L);
    }
    const uint64_t n_all = p->h_st.bcf_records;
    p->n_lines = n_all;
    TRY(grow(b.d_rec_off, b.rec_cap, n_all));
    launch_bcf_emit(p->d_text, p->nbytes, sg, b.d_rec_off, L);
    CU(cudaEventRecord(p->ev[1], p->stream));
    SiteRows &r = p->rows;
    if (r.cap < n_all || !r.start) TRY(alloc_rows(r, std::max(regrown(n_all, r.start), r.cap)));
    const uint64_t blocks = (n_all + 255) / 256;
    if (b.blk_cap < blocks || !b.d_blk_count) {
        TRY(dev_alloc(&b.d_blk_count, blocks)); TRY(dev_alloc(&b.d_blk_base, blocks));
        b.blk_cap = blocks;
    }
    BcfSiteArgs a;
    a.text = p->d_text; a.rec_off = b.d_rec_off; a.n_rec = n_all; a.n_samples = p->n_cols; a.n_contigs = nc;
    a.contigs = b.d_contigs; a.gt_key = b.gt_key;
    a.rid = -1;
    if (p->rg.has_region) {
        const std::string want(p->rg.chrom, p->rg.chrom_len);
        a.rid = -2;
        for (uint32_t i = 0; i < nc; ++i) if (b.contigs[i] == want) { a.rid = (int)i; break; }
    }
    a.beg0 = p->rg.beg0; a.end0 = p->rg.end0; a.want_gt = p->want_gt;
    a.start = r.start; a.stop = r.stop; a.ref = r.ref; a.alt = r.alt; a.chrom_len = r.chrom_len;
    a.chrom_abs = r.chrom_abs; a.chrom5 = r.chrom5; a.rowinfo = r.rowinfo;
    a.blk_count = b.d_blk_count; a.blk_base = b.d_blk_base; a.st = p->d_st;
    launch_bcf_sites(a, L);
    CU(cudaEventRecord(p->ev[2], p->stream));
    TRY(fetch_status(p));
    CU(cudaGetLastError());
    if (p->h_st.bcf_bad_fmt)
        return fail(HB_ERR_FORMAT, "BCF record whose alleles or FORMAT fields run past its length (" +
                                       std::to_string(p->h_st.bcf_bad_fmt) + " records)");
    p->index_used = 4;
    return HB_OK;
}

// the CHROM runs of the last run_parse, on the host (needs the text: hb_parse_release_text calls it first)
static int ensure_runs(hb_parse *p) {
    if (p->runs_valid) return HB_OK;
    CU(cudaSetDevice(p->device));
    p->run_rows.clear(); p->run_names.clear();
    const uint64_t n_runs = std::min<uint64_t>(p->h_st.n_chrom_runs, hb_parse::kMaxRuns);
    if (n_runs && p->d_run_rows && (p->d_text || p->bcf)) {
        p->run_rows.resize(n_runs);
        CU(cudaMemcpy(p->run_rows.data(), p->d_run_rows, n_runs * 8, cudaMemcpyDeviceToHost));
        std::sort(p->run_rows.begin(), p->run_rows.end());
        for (uint64_t r : p->run_rows) {
            uint64_t abs; uint8_t len; char name[256];
            CU(cudaMemcpy(&abs, p->rows.chrom_abs + r, 8, cudaMemcpyDeviceToHost));
            if (p->bcf) {                        // BCF rows point into the contig names: the name from the dictionary
                const auto &off = p->bcf->name_off;
                const size_t i = (size_t)(std::lower_bound(off.begin(), off.end(), abs) - off.begin());
                p->run_names.push_back(i < off.size() ? p->bcf->contigs[i] : std::string());
                continue;
            }
            CU(cudaMemcpy(&len, p->rows.chrom_len + r, 1, cudaMemcpyDeviceToHost));
            CU(cudaMemcpy(name, p->d_text + abs, len, cudaMemcpyDeviceToHost));
            p->run_names.emplace_back(name, name + len);
        }
    }
    p->runs_valid = true;
    return HB_OK;
}

// kernel 2b: the column checkpoints of the n_nu kept records that need the general decode path
static int index_nonuniform(hb_parse *p, uint64_t n_nu, const Launch &L) {
    TRY(grow(p->d_cp, p->cp_cap, n_nu * p->ncp));
    CU(cudaMemsetAsync(p->d_cp, 0xff, p->cp_cap * sizeof(uint64_t), p->stream));
    launch_index_columns(p->d_text, p->rows.rowinfo, p->d_nu_rows, n_nu, p->d_cp, p->ncp, L);
    return HB_OK;
}

static int run_parse(hb_parse *p) {
    ++p->run_seq;
    CU(cudaSetDevice(p->device));
    Launch L{p->stream, p->sm_count};
    if (!p->d_st) TRY(dev_alloc(&p->d_st, 1));
    CU(cudaMemsetAsync(p->d_st, 0, sizeof(DevStatus), p->stream));
    memset(&p->h_st, 0, sizeof p->h_st);
    p->ncp = (p->n_cols + kCP - 1) / kCP;
    if (p->nbytes == 0) return HB_OK;

    // ---- how to locate the records, from the first one
    if (!p->probed && !p->bcf) {
        // the whole first record: 4 bytes per sample when it is GT-only (800 KB at 200,000 samples) + its head
        std::vector<uint8_t> head((size_t)std::min<uint64_t>(4ull * p->n_cols + 65536, p->nbytes));
        const size_t hn = head.size();
        CU(cudaMemcpyAsync(head.data(), p->d_text, hn, cudaMemcpyDeviceToHost, p->stream));
        CU(cudaStreamSynchronize(p->stream));
        bool gt_only, uniform; uint64_t l0;
        probe_head(head.data(), hn, p->n_cols, gt_only, uniform, l0);
        p->with_tabs = p->tokenizer == 2 || ((p->tokenizer == 0 || p->tokenizer == 3) && !gt_only);
        if (!p->want_gt) p->with_tabs = false;
        // walking pays when a record is much longer than its head (and needs the decoder to validate the jumps)
        p->use_walker = p->want_gt && p->n_cols > 0 &&
                        (p->tokenizer == 3 || (p->tokenizer == 0 && uniform && p->n_cols >= 256));
        p->first_line_len = l0 ? l0 : hn;
        p->probed = true;
    }
    if (!p->d_ploidy) {
        TRY(dev_alloc(&p->d_ploidy, p->n_samples)); TRY(dev_alloc(&p->d_badgt, p->n_samples));
        TRY(dev_alloc(&p->d_run_rows, hb_parse::kMaxRuns));
    }
    CU(cudaMemsetAsync(p->d_ploidy, 0, std::max<uint64_t>(1, p->n_samples) * 4, p->stream));
    CU(cudaMemsetAsync(p->d_badgt, 0, std::max<uint64_t>(1, p->n_samples) * 4, p->stream));
    if (p->bcf) TRY(index_bcf(p, L));
    else if (p->use_walker) TRY(index_by_walker(p, L));
    else TRY(index_by_tokenizer(p, L));
    const uint64_t n_rec = p->h_st.n_records;
    if (p->attached_frames && n_rec) frames_early_site_pass(p->attached_frames, p);
    {   // CHROM runs need the site columns only: on a side stream, next to the decoder; the status fetch waits for them
        if (!p->side) CU(cudaStreamCreateWithFlags(&p->side, cudaStreamNonBlocking));
        if (!p->ev_runs) CU(cudaEventCreateWithFlags(&p->ev_runs, cudaEventDisableTiming));
        CU(cudaEventRecord(p->ev_runs, p->stream));
        CU(cudaStreamWaitEvent(p->side, p->ev_runs, 0));
        Launch Ls = L;
        Ls.stream = p->side;
        launch_chrom_runs(p->bcf ? p->bcf->d_names : p->d_text, p->rows.chrom_abs, p->rows.chrom_len, n_rec, p->d_run_rows, hb_parse::kMaxRuns, p->d_st, Ls);
        CU(cudaEventRecord(p->ev_runs, p->side));
    }

    // ---- GT decode
    if (p->want_gt && n_rec && p->n_samples) {
        if (p->index_used == 1 && p->h_st.n_nonuniform) TRY(index_nonuniform(p, p->h_st.n_nonuniform, L));
        // the planes are re-used (with their stride) whenever the rows fit: a handle that is re-run on slabs of
        // slightly different length must not re-allocate -- cudaFree synchronises the whole device
        if (!p->d_gt[0] || n_rec > p->gt_stride) {
            const uint64_t want = regrown(n_rec, p->d_gt[0]);
            const uint64_t stride = (want + 127) / 128 * 128;         // whole 128-row groups of the bit planes
            const uint64_t bytes = stride * p->n_samples;
            TRY(dev_alloc(&p->d_gt[0], bytes)); TRY(dev_alloc(&p->d_gt[1], bytes));
            p->gt_bytes = bytes; p->gt_stride = stride;
            p->bits_stride = stride / 128 * kBitGroupWords;
            TRY(dev_alloc(&p->d_bits, p->bits_stride * p->n_samples));
            // rows between the last decode tile and the end of its group are never written: they read as "no allele"
            CU(cudaMemsetAsync(p->d_bits, 0, p->bits_stride * p->n_samples * 4, p->stream));
        }
        // walker: the count pass told the host how many kept records are not plain "\tX|Y" columns
        if (p->index_used == 3 && p->h_st.n_nu_count) TRY(index_nonuniform(p, p->h_st.n_nu_count, L));
        // the decoders run over the file's columns; a subset picks which of them are decoded and into which planes
        const SampleSel sel{p->d_sel_mask, p->d_sel_base};
        if (p->bcf)
            launch_bcf_decode(p->d_text, p->rows.rowinfo, n_rec, p->n_cols, p->d_gt[0], p->d_gt[1], p->gt_stride, p->d_bits,
                              p->bits_stride, p->d_ploidy, p->d_badgt, p->d_st, sel, L);
        else
            launch_decode_gt(p->d_text, p->rows.rowinfo, n_rec, p->n_cols, p->d_cp, p->ncp, p->d_gt[0], p->d_gt[1],
                             p->gt_stride, p->d_bits, p->bits_stride, p->d_ploidy, p->d_badgt, p->d_st, sel, L);
    }
    CU(cudaEventRecord(p->ev[3], p->stream));
    // frames attached to this parse: their kernel is queued right behind the decoder now (the host waits for the templates
    // only), instead of after this function's status fetch + the caller's next call
    if (p->attached_frames && n_rec && p->want_gt && p->n_samples) frames_early_launch(p->attached_frames, p);
    CU(cudaStreamWaitEvent(p->stream, p->ev_runs, 0));       // the CHROM runs (side stream) are part of the status
    TRY(fetch_status(p));
    CU(cudaGetLastError());
    cudaEventElapsedTime(&p->ms_tok, p->ev[0], p->ev[1]);
    cudaEventElapsedTime(&p->ms_sites, p->ev[1], p->ev[2]);
    cudaEventElapsedTime(&p->ms_decode, p->ev[2], p->ev[3]);

    if (p->index_used == 3 && (p->h_st.walk_broken || p->h_st.index_invalid)) {
        // the text is not what the walker can prove exact: locate the records the plain way
        p->use_walker = false;
        ++p->walker_fallbacks;
        return run_parse(p);
    }

    // ---- CHROM runs -> names: fetched when somebody asks (ensure_runs): a handful of tiny synchronous D2H copies that a
    // step which goes on to compress the records does not need to wait for (~60 us of idle GPU per step, r02n)
    p->run_rows.clear(); p->run_names.clear();
    p->runs_valid = false;
    if (p->h_st.n_chrom_runs > hb_parse::kMaxRuns) return fail(HB_ERR_FORMAT, "more than 4096 CHROM runs (unsorted VCF?)");
    if (p->h_st.n_bad_cols)
        return fail(HB_ERR_FORMAT, "Number of columns does not match the number of samples (" +
                                       std::to_string(p->h_st.n_bad_cols) + " records)");
    return HB_OK;
}

// a handle under construction: every early return frees it and what it holds, until the caller releases it
using ParsePtr = std::unique_ptr<hb_parse, void (*)(hb_parse *)>;

static ParsePtr new_parse(const hb_parse_opts *o, int &rc) {
    ParsePtr p(nullptr, hb_parse_free);
    rc = o ? ensure_device(o->device) : fail(HB_ERR_ARG, "null argument");
    if (rc != HB_OK) return p;
    p.reset(new hb_parse());
    p->device = o->device;
    p->stream = (cudaStream_t)o->stream;
    cudaDeviceGetAttribute(&p->sm_count, cudaDevAttrMultiProcessorCount, o->device);
    p->n_cols = p->n_samples = o->n_samples;
    parse_region(o->region, p->rg);
    p->end_is_int = o->end_is_int;
    p->want_gt = o->want_gt;
    p->tokenizer = o->tokenizer;
    for (auto &e : p->ev) cudaEventCreate(&e);
    return p;
}

// ---- sample subsets (hb_parse_*_subset)
// cols[0..n) of records with n_cols sample columns: at least one, ascending, each once, all in range
static int check_cols(const uint32_t *cols, uint32_t n, uint32_t n_cols) {
    if (!cols || n == 0) return fail(HB_ERR_ARG, "a sample subset names at least one column");
    for (uint32_t i = 0; i < n; ++i) {
        if (cols[i] >= n_cols)
            return fail(HB_ERR_ARG, "sample column " + std::to_string(cols[i]) + " is out of range (" + std::to_string(n_cols) + " samples)");
        if (i && cols[i] <= cols[i - 1]) return fail(HB_ERR_ARG, "sample columns must be ascending and distinct");
    }
    return HB_OK;
}

// The subset cols (checked; empty = every sample) on a handle that has not run yet: its planes are cols.size() wide, plane j
// is column cols[j].  A subset of every column is the ordinary parse and changes nothing.
static int set_subset(hb_parse *p, const std::vector<uint32_t> &cols) {
    if (cols.empty() || cols.size() == p->n_cols) return HB_OK;
    const uint32_t nb = (p->n_cols + kTS - 1) / kTS;
    std::vector<uint32_t> mask(4ull * nb, 0), base(nb, 0);          // mask: 4 words per block, word c / 32 holds column c
    for (uint32_t c : cols) mask[c / 32] |= 1u << (c % 32);
    for (uint32_t b = 1; b < nb; ++b) {
        uint32_t in_block = 0;
        for (int q = 0; q < 4; ++q) in_block += (uint32_t)__builtin_popcount(mask[4 * (b - 1) + q]);
        base[b] = base[b - 1] + in_block;
    }
    TRY(dev_alloc(&p->d_sel_mask, nb));
    TRY(dev_alloc(&p->d_sel_base, nb));
    CU(cudaMemcpy(p->d_sel_mask, mask.data(), 16ull * nb, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(p->d_sel_base, base.data(), 4ull * nb, cudaMemcpyHostToDevice));
    p->sel_cols = cols;
    p->n_samples = (uint32_t)cols.size();
    return HB_OK;
}

// zero bytes behind the text of every parse: kernels that read it in whole 16-byte words find zeros past its end
constexpr uint64_t kTextPad = 256;

// n bytes of host text (+ '\n' when add_newline) become the parse's own device text
static int upload_text(hb_parse *p, const uint8_t *text, uint64_t n, bool add_newline) {
    const uint64_t total = n + (add_newline ? 1 : 0);
    TRY(dev_alloc(&p->d_text_owned, total + kTextPad));
    cudaError_t e = cudaMemcpyAsync(p->d_text_owned, text, n, cudaMemcpyHostToDevice, p->stream);
    if (e == cudaSuccess && add_newline) e = cudaMemsetAsync(p->d_text_owned + n, '\n', 1, p->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(p->d_text_owned + total, 0, kTextPad, p->stream);
    if (e != cudaSuccess) return fail_cuda(e);
    p->d_text = p->d_text_owned;
    p->nbytes = total;
    return HB_OK;
}

// cols: the sample subset (empty = every sample)
static int device_text(const uint8_t *d_text, uint64_t nbytes, const hb_parse_opts *opts, const std::vector<uint32_t> &cols,
                       hb_parse **out) {
    int rc;
    ParsePtr p = new_parse(opts, rc);
    if (!p) return rc;
    if (((uintptr_t)d_text & 15) != 0) return fail(HB_ERR_ARG, "d_text must be 16-byte aligned");
    TRY(set_subset(p.get(), cols));
    p->d_text = d_text;
    p->nbytes = nbytes;
    TRY(run_parse(p.get()));
    *out = p.release();
    return HB_OK;
}

static int host_text(const uint8_t *text, uint64_t nbytes, const hb_parse_opts *opts, const std::vector<uint32_t> &cols,
                     hb_parse **out) {
    int rc;
    ParsePtr p = new_parse(opts, rc);
    if (!p) return rc;
    TRY(set_subset(p.get(), cols));
    TRY(upload_text(p.get(), text, nbytes, nbytes && text[nbytes - 1] != '\n'));
    TRY(run_parse(p.get()));
    *out = p.release();
    return HB_OK;
}

int hb_parse_device_text(const uint8_t *d_text, uint64_t nbytes, const hb_parse_opts *opts, hb_parse **out) {
    return device_text(d_text, nbytes, opts, {}, out);
}

int hb_parse_host_text(const uint8_t *text, uint64_t nbytes, const hb_parse_opts *opts, hb_parse **out) {
    return host_text(text, nbytes, opts, {}, out);
}

int hb_parse_device_text_subset(const uint8_t *d_text, uint64_t nbytes, const hb_parse_opts *opts, const uint32_t *cols,
                                uint32_t n_cols, hb_parse **out) {
    TRY(ensure_device(opts ? opts->device : 0));
    if (!opts) return fail(HB_ERR_ARG, "null argument");
    TRY(check_cols(cols, n_cols, opts->n_samples));
    return device_text(d_text, nbytes, opts, std::vector<uint32_t>(cols, cols + n_cols), out);
}

int hb_parse_host_text_subset(const uint8_t *text, uint64_t nbytes, const hb_parse_opts *opts, const uint32_t *cols,
                              uint32_t n_cols, hb_parse **out) {
    TRY(ensure_device(opts ? opts->device : 0));
    if (!opts) return fail(HB_ERR_ARG, "null argument");
    TRY(check_cols(cols, n_cols, opts->n_samples));
    return host_text(text, nbytes, opts, std::vector<uint32_t>(cols, cols + n_cols), out);
}

// ---------------------------------------------------------------------------------------------
// Streaming form of hb_parse_host_text + hb_parse_fetch_matrix + hb_parse_fetch_sites: the text is cut
// into slabs at line boundaries and two device slots alternate, so that the H2D copy of slab k+1, the
// kernels of slab k and the D2H copy of slab k-1 run at the same time (PCIe is full duplex: the 2 bytes
// per call going back hide behind the 4 bytes per call coming in).  Device memory is O(slab), so the
// text may be far larger than HBM.
// ---------------------------------------------------------------------------------------------
// ---- the two device slots of the streaming entry points.  Making and freeing them costs little on a good day and
// hundreds of milliseconds on a bad one (cudaMalloc / cudaFree of the slab buffers: 150 ms setup, 340-520 ms cleanup were
// measured inside otherwise 225 ms calls), so a finished call leaves them in a per-process cache for the next call with the
// same options; hb_cache_clear() frees them.
namespace {
struct StreamSlot {
    hb_parse *p = nullptr;                        // parses the slab text in buf; owns no text
    cudaStream_t compute = nullptr, d2h = nullptr;
    cudaEvent_t fetched = nullptr;
    uint8_t *buf = nullptr;                       // [carry_cap + 32 | slab text | '\n' + 256]; host text (no carry) sits at buf + 0
    // BGZF streaming only
    hb::InflateScratch sc;
    unsigned long long *h_pin = nullptr;          // pinned: [last newline | inflate status of every member]
    uint64_t x = 0, end = 0, begin = 0;           // slab text at buf + x .. buf + end; the parse starts at buf + begin
};
struct StreamSlots {
    StreamSlot slot[2];
    size_t n_slots = 0;
    int device = -1, want_gt = 0, end_is_int = 0, tokenizer = 0;
    uint32_t n_samples = 0;
    std::vector<uint32_t> cols;                   // the slot parses' sample subset (empty = every sample)
    std::string region;
    uint64_t text_cap = 0, comp_cap = 0, carry_cap = 0;
    uint32_t n_cap = 0;
    void destroy() {
        if (device >= 0) cudaSetDevice(device);
        for (auto &s : slot) {
            if (s.compute) cudaStreamSynchronize(s.compute);
            if (s.d2h) cudaStreamSynchronize(s.d2h);
            if (s.p) hb_parse_free(s.p);
            free_dev(s.buf);
            if (s.h_pin) cudaFreeHost(s.h_pin);
            hb::inflate_scratch_free(s.sc);
            if (s.fetched) cudaEventDestroy(s.fetched);
            if (s.compute) cudaStreamDestroy(s.compute);
            if (s.d2h) cudaStreamDestroy(s.d2h);
            s = StreamSlot();
        }
        n_slots = 0;
    }
    bool same_options(const hb_parse_opts &o, const std::vector<uint32_t> &c) const {
        return device == o.device && n_samples == o.n_samples && want_gt == (o.want_gt ? 1 : 0) && end_is_int == (o.end_is_int ? 1 : 0) &&
               tokenizer == o.tokenizer && region == (o.region ? o.region : "") && cols == c;
    }
};
struct SlotCache { std::mutex mu; StreamSlots *kept = nullptr; bool in_use = false; };
SlotCache g_text_slots, g_bgzf_slots;

// the cached slots when they were made with these options and sample subset and are free, else fresh (empty) ones
StreamSlots *acquire_slots(SlotCache &c, const hb_parse_opts &o, const std::vector<uint32_t> &cols, size_t n_slots) {
    std::lock_guard<std::mutex> lk(c.mu);
    if (c.kept && !c.in_use) {
        if (c.kept->same_options(o, cols) && c.kept->n_slots >= n_slots) { c.in_use = true; return c.kept; }
        c.kept->destroy();
        delete c.kept;
        c.kept = nullptr;
    }
    StreamSlots *ss = new StreamSlots();
    ss->device = o.device; ss->n_samples = o.n_samples; ss->want_gt = o.want_gt ? 1 : 0; ss->end_is_int = o.end_is_int ? 1 : 0;
    ss->tokenizer = o.tokenizer; ss->region = o.region ? o.region : "";
    ss->cols = cols;
    return ss;
}
void release_slots(SlotCache &c, StreamSlots *ss, bool keep) {
    if (keep) for (auto &s : ss->slot) { if (s.compute) cudaStreamSynchronize(s.compute); if (s.d2h) cudaStreamSynchronize(s.d2h); }
    std::lock_guard<std::mutex> lk(c.mu);
    if (ss == c.kept) {
        c.in_use = false;
        if (!keep) { ss->destroy(); delete ss; c.kept = nullptr; }
        return;
    }
    if (keep && !c.kept) { c.kept = ss; return; }
    ss->destroy();
    delete ss;
}
void clear_slot_cache(SlotCache &c) {
    std::lock_guard<std::mutex> lk(c.mu);
    if (c.kept && !c.in_use) { c.kept->destroy(); delete c.kept; c.kept = nullptr; }
}

// the slots of one streaming call from cache c: streams, event and parse are made for a slot that has none, and the buffers of
// every slot grow together when a capacity is short (the carry offset is part of the layout).  text_cap: text of one slab;
// carry_cap, comp_cap, n_cap: BGZF only -- host text (all 0) has no inflate scratch and no pinned tables.  cols: the sample
// subset of the slot parses (empty = every sample).
int open_slots(SlotCache &c, const hb_parse_opts &opts, const std::vector<uint32_t> &cols, size_t n_slots, uint64_t text_cap,
               uint64_t carry_cap, uint64_t comp_cap, uint32_t n_cap, StreamSlots **out) {
    StreamSlots *ss = acquire_slots(c, opts, cols, n_slots);
    int rc = HB_OK;
    for (size_t i = ss->n_slots; i < n_slots && rc == HB_OK; ++i) {
        StreamSlot &s = ss->slot[i];
        if (cudaStreamCreateWithFlags(&s.compute, cudaStreamNonBlocking) != cudaSuccess ||
            cudaStreamCreateWithFlags(&s.d2h, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&s.fetched, cudaEventDisableTiming) != cudaSuccess) { rc = fail(HB_ERR_CUDA, "cannot create streams"); break; }
        hb_parse_opts o = opts;
        o.stream = s.compute;
        s.p = new_parse(&o, rc).release();
        if (rc == HB_OK) rc = set_subset(s.p, cols);
        if (rc == HB_OK) ss->n_slots = i + 1;
    }
    const bool grow = ss->text_cap < text_cap || ss->carry_cap < carry_cap || ss->comp_cap < comp_cap || ss->n_cap < n_cap;
    if (grow) {
        ss->text_cap = std::max(ss->text_cap, text_cap + text_cap / 16);
        ss->carry_cap = std::max(ss->carry_cap, carry_cap);
        ss->comp_cap = std::max(ss->comp_cap, comp_cap + comp_cap / 8);
        if (n_cap) ss->n_cap = std::max<uint32_t>(ss->n_cap, n_cap + n_cap / 8 + 16);
    }
    for (size_t i = 0; i < ss->n_slots && rc == HB_OK; ++i) {
        StreamSlot &s = ss->slot[i];
        s.p->probed = false;                         // this call's text may have another shape than the last one's
        if (s.buf && !grow) continue;
        rc = dev_alloc(&s.buf, ss->carry_cap + 32 + ss->text_cap + 1 + 256);
        if (rc != HB_OK || !ss->n_cap) continue;
        if (s.h_pin) { cudaFreeHost(s.h_pin); s.h_pin = nullptr; }
        inflate_scratch_free(s.sc);
        rc = inflate_scratch_alloc(s.sc, ss->comp_cap, ss->n_cap);
        // pinned: [last newline 8 | status 4n | coff 8n | ooff 8n | clen 4n | olen 4n] -- copies from / to pageable memory stall here
        if (rc == HB_OK && cudaMallocHost((void **)&s.h_pin, 8 + 28ull * ss->n_cap + 8) != cudaSuccess) rc = fail(HB_ERR_MEM, "cudaMallocHost failed");
    }
    if (rc != HB_OK) { release_slots(c, ss, false); return rc; }
    *out = ss;
    return HB_OK;
}

// the end of a streaming call: the D2H copies of every slot are waited for, a CUDA error becomes the return code, and the slots
// go back to cache c, kept for the next call when all went well
int close_slots(SlotCache &c, StreamSlots *ss, int rc, cudaError_t e) {
    for (size_t i = 0; i < ss->n_slots && rc == HB_OK && e == cudaSuccess; ++i) e = cudaStreamSynchronize(ss->slot[i].d2h);
    if (e != cudaSuccess && rc == HB_OK) rc = fail_cuda(e);
    release_slots(c, ss, rc == HB_OK);
    return rc;
}

// where the rows of a parsed slab go: host arrays (HostSink) or the growing planes of ONE resident parse (ResidentSink).
// deliver() enqueues copies on s.d2h (the slot's compute stream is idle by then).  The per-sample error counts of all
// slabs are summed into ploidy_err / badgt_err, each [n_samples], when set.
struct SlabSink {
    hb_parse_opts opts{};
    uint32_t *ploidy_err = nullptr, *badgt_err = nullptr;
    std::vector<uint32_t> pl, bg;                 // the counts of one slab
    virtual ~SlabSink() {}
    virtual int begin(const hb_parse_opts &o, const std::vector<std::string> &samples, uint64_t total_text) {
        (void)samples; (void)total_text;
        opts = o;
        if (ploidy_err) memset(ploidy_err, 0, 4ull * o.n_samples);
        if (badgt_err) memset(badgt_err, 0, 4ull * o.n_samples);
        pl.resize(o.n_samples); bg.resize(o.n_samples);
        return HB_OK;
    }
    virtual int deliver(StreamSlot &s, uint64_t R, uint64_t n, uint64_t slab_text, cudaError_t &e) = 0;
    void add_errors(const StreamSlot &s, cudaError_t &e) {      // waits for s.d2h
        if (!(ploidy_err || badgt_err) || !opts.want_gt || !opts.n_samples || e != cudaSuccess) return;
        e = cudaMemcpyAsync(pl.data(), s.p->d_ploidy, 4ull * opts.n_samples, cudaMemcpyDeviceToHost, s.d2h);
        if (e == cudaSuccess) e = cudaMemcpyAsync(bg.data(), s.p->d_badgt, 4ull * opts.n_samples, cudaMemcpyDeviceToHost, s.d2h);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s.d2h);
        for (uint32_t i = 0; i < opts.n_samples && e == cudaSuccess; ++i) {
            if (ploidy_err) ploidy_err[i] += pl[i];
            if (badgt_err) badgt_err[i] += bg[i];
        }
    }
};

// rows into the caller's host arrays: planes [n_samples][out_stride], columns of out_stride records; any of them may be NULL
struct HostSink : SlabSink {
    int8_t *gt0, *gt1; uint64_t out_stride; uint32_t *start, *stop; char *ref, *alt;
    HostSink(int8_t *gt0, int8_t *gt1, uint64_t out_stride, uint32_t *start, uint32_t *stop, char *ref, char *alt, uint32_t *pl, uint32_t *bg)
        : gt0(gt0), gt1(gt1), out_stride(out_stride), start(start), stop(stop), ref(ref), alt(alt) { ploidy_err = pl; badgt_err = bg; }
    int deliver(StreamSlot &s, uint64_t R, uint64_t n, uint64_t, cudaError_t &e) override {
        if (R + n > out_stride && (gt0 || gt1 || start || stop || ref || alt)) return fail(HB_ERR_ARG, "more records than the output arrays hold");
        if (opts.want_gt && opts.n_samples && s.p->d_gt[0]) {
            if (gt0) e = cudaMemcpy2DAsync(gt0 + R, out_stride, s.p->d_gt[0], s.p->gt_stride, n, opts.n_samples, cudaMemcpyDeviceToHost, s.d2h);
            if (gt1 && e == cudaSuccess) e = cudaMemcpy2DAsync(gt1 + R, out_stride, s.p->d_gt[1], s.p->gt_stride, n, opts.n_samples, cudaMemcpyDeviceToHost, s.d2h);
        }
        if (start && e == cudaSuccess) e = cudaMemcpyAsync(start + R, s.p->rows.start, n * 4, cudaMemcpyDeviceToHost, s.d2h);
        if (stop && e == cudaSuccess) e = cudaMemcpyAsync(stop + R, s.p->rows.stop, n * 4, cudaMemcpyDeviceToHost, s.d2h);
        if (ref && e == cudaSuccess) e = cudaMemcpyAsync(ref + R, s.p->rows.ref, n, cudaMemcpyDeviceToHost, s.d2h);
        if (alt && e == cudaSuccess) e = cudaMemcpyAsync(alt + R, s.p->rows.alt, n, cudaMemcpyDeviceToHost, s.d2h);
        return HB_OK;
    }
};

// the nbytes of slab text at s.buf + begin: parsed once the slot's previous rows have left, its rows handed to the sink behind
// the R rows before them.  Returns with the slot's compute stream idle; a CUDA error is left in e.
int parse_slab(StreamSlot &s, uint64_t begin, uint64_t nbytes, SlabSink &sink, uint64_t &R, cudaError_t &e) {
    uint64_t n = 0;
    if (nbytes) {
        e = cudaStreamWaitEvent(s.compute, s.fetched, 0);     // (putting the text in place did not need to wait for that)
        if (e != cudaSuccess) return HB_OK;
        s.p->d_text = s.buf + begin;
        s.p->nbytes = nbytes;
        TRY(run_parse(s.p));
        n = s.p->h_st.n_records;
    }
    if (n) {
        TRY(sink.deliver(s, R, n, nbytes, e));
        sink.add_errors(s, e);
    }
    if (e == cudaSuccess) e = cudaEventRecord(s.fetched, s.d2h);
    R += n;
    return HB_OK;
}
}  // namespace

int hb_parse_stream_host(const uint8_t *text, uint64_t nbytes, const hb_parse_opts *opts, uint64_t slab_bytes,
                         int8_t *gt0, int8_t *gt1, uint64_t out_stride, uint32_t *start, uint32_t *stop, char *ref,
                         char *alt, uint32_t *ploidy_err, uint32_t *badgt_err, uint64_t *n_records, uint32_t *n_slabs) {
    if (!opts || !n_records || (nbytes && !text)) return fail(HB_ERR_ARG, "null argument");
    if (nbytes >= 4 && memcmp(text, "BCF\2", 4) == 0) return fail(HB_ERR_ARG, kBcfNoStream);
    *n_records = 0;
    if (n_slabs) *n_slabs = 0;
    HostSink sink(gt0, gt1, out_stride, start, stop, ref, alt, ploidy_err, badgt_err);
    TRY(sink.begin(*opts, {}, nbytes));
    if (nbytes == 0) return HB_OK;
    if (text[nbytes - 1] != '\n') return fail(HB_ERR_ARG, "the text must end with a newline");
    if (slab_bytes == 0) slab_bytes = 1ull << 30;
    std::vector<std::pair<uint64_t, uint64_t>> slabs;
    uint64_t cap = 0;
    for (uint64_t off = 0; off < nbytes;) {
        uint64_t end = std::min(nbytes, off + slab_bytes);
        if (end < nbytes) {
            const void *q = memrchr(text + off, '\n', end - off);
            if (q) end = (uint64_t)((const uint8_t *)q - text) + 1;
            else {                                   // one line longer than a slab: take the whole line
                const void *f = memchr(text + end, '\n', nbytes - end);
                end = f ? (uint64_t)((const uint8_t *)f - text) + 1 : nbytes;
            }
        }
        slabs.emplace_back(off, end - off);
        cap = std::max(cap, end - off);
        off = end;
    }
    TRY(ensure_device(opts->device));
    const double t_begin = now_ms();
    StreamSlots *ss = nullptr;
    TRY(open_slots(g_text_slots, *opts, {}, std::min<size_t>(2, slabs.size()), cap, 0, 0, 0, &ss));
    StreamSlot *slot = ss->slot;
    auto h2d = [&](size_t k) -> cudaError_t {
        StreamSlot &s = slot[k & 1];
        cudaError_t e = cudaMemcpyAsync(s.buf, text + slabs[k].first, slabs[k].second, cudaMemcpyHostToDevice, s.compute);
        if (e == cudaSuccess) e = cudaMemsetAsync(s.buf + slabs[k].second, 0, 256, s.compute);
        return e;
    };
    const double t_setup = now_ms() - t_begin;
    double t_parse = 0;
    int rc = HB_OK;
    cudaError_t e = h2d(0);
    uint64_t R = 0;
    for (size_t k = 0; k < slabs.size() && rc == HB_OK && e == cudaSuccess; ++k) {
        if (k + 1 < slabs.size()) e = h2d(k + 1);
        if (e != cudaSuccess) break;
        const double t0 = now_ms();
        rc = parse_slab(slot[k & 1], 0, slabs[k].second, sink, R, e);
        t_parse += now_ms() - t0;
    }
    const double t_loop_end = now_ms();
    rc = close_slots(g_text_slots, ss, rc, e);
    if (getenv("HB_TRACE"))
        fprintf(stderr, "[hb_parse_stream_host] %zu slabs: setup %.1f ms, loop %.1f ms (parse + deliver %.1f ms), D2H tail + release %.1f ms\n",
                slabs.size(), t_setup, t_loop_end - t_begin - t_setup, t_parse, now_ms() - t_loop_end);
    if (rc != HB_OK) return rc;
    *n_records = R;
    if (n_slabs) *n_slabs = (uint32_t)slabs.size();
    return HB_OK;
}

int hb_parse_release_text(hb_parse *p) {
    if (!p) return fail(HB_ERR_ARG, "null handle");
    if (p->d_text_owned) {
        TRY(ensure_runs(p));                     // the CHROM names are read from the text
        CU(cudaSetDevice(p->device));
        dev_pool_release(p->d_text_owned);       // the caller wants the HBM back: not into the idle pool
        p->d_text_owned = nullptr;
        p->d_text = nullptr;
        p->nbytes = 0;
        p->text_released = true;
    }
    return HB_OK;
}

int hb_parse_rerun(hb_parse *p) {
    if (!p) return fail(HB_ERR_ARG, "null handle");
    if (p->text_released) return fail(HB_ERR_ARG, "the text of this parse was released");
    return run_parse(p);
}

int hb_parse_rerun_bytes(hb_parse *p, uint64_t nbytes) {
    if (!p) return fail(HB_ERR_ARG, "null handle");
    if (p->d_text_owned) return fail(HB_ERR_ARG, "hb_parse_rerun_bytes is for handles made by hb_parse_device_text");
    p->nbytes = nbytes;
    return run_parse(p);
}

int hb_parse_get_info(const hb_parse *p, hb_parse_info *info) {
    if (!p || !info) return fail(HB_ERR_ARG, "null argument");
    memset(info, 0, sizeof *info);
    info->text_bytes = p->nbytes;
    info->n_lines = p->n_lines;
    info->n_records = p->h_st.n_records;
    info->n_samples = p->n_samples;
    info->gt_stride = p->gt_stride;
    info->d_gt[0] = p->d_gt[0];
    info->d_gt[1] = p->d_gt[1];
    info->d_start = p->rows.start; info->d_stop = p->rows.stop; info->d_ref = p->rows.ref; info->d_alt = p->rows.alt;
    info->n_nonuniform = p->h_st.n_nonuniform;
    info->n_bad_gt = p->h_st.n_bad_gt;
    info->n_bad_cols = p->h_st.n_bad_cols;
    info->n_nogt = p->h_st.n_nogt;
    info->tokenizer_used = p->index_used;
    info->walker_fallbacks = p->walker_fallbacks;
    info->ms_tokenize = p->ms_tok; info->ms_sites = p->ms_sites; info->ms_decode = p->ms_decode;
    info->ms_inflate = p->ms_inflate; info->compressed_bytes = p->compressed_bytes;
    return HB_OK;
}

int hb_parse_fetch_sites(hb_parse *p, uint32_t *start, uint32_t *stop, char *ref, char *alt) {
    if (!p) return fail(HB_ERR_ARG, "null handle");
    CU(cudaSetDevice(p->device));
    uint64_t n = p->h_st.n_records;
    if (!n) return HB_OK;
    if (start) CU(d2h_copy(start, p->rows.start, n * 4, p->stream));
    if (stop) CU(d2h_copy(stop, p->rows.stop, n * 4, p->stream));
    if (ref) CU(d2h_copy(ref, p->rows.ref, n, p->stream));
    if (alt) CU(d2h_copy(alt, p->rows.alt, n, p->stream));
    return HB_OK;
}

int hb_parse_fetch_sample(hb_parse *p, uint32_t s, int8_t *gt0, int8_t *gt1) {
    if (!p) return fail(HB_ERR_ARG, "null handle");
    if (s >= p->n_samples) return fail(HB_ERR_SAMPLE, "sample index out of range");
    CU(cudaSetDevice(p->device));
    uint64_t n = p->h_st.n_records;
    if (!n) return HB_OK;
    if (!p->d_gt[0]) return fail(HB_ERR_NOGT, "parse was made without genotypes");
    if (gt0) CU(d2h_copy(gt0, p->d_gt[0] + (uint64_t)s * p->gt_stride, n, p->stream));
    if (gt1) CU(d2h_copy(gt1, p->d_gt[1] + (uint64_t)s * p->gt_stride, n, p->stream));
    return HB_OK;
}

int hb_parse_fetch_matrix(hb_parse *p, int8_t *gt0, int8_t *gt1) {
    if (!p) return fail(HB_ERR_ARG, "null handle");
    CU(cudaSetDevice(p->device));
    uint64_t n = p->h_st.n_records;
    if (!n || !p->n_samples) return HB_OK;
    if (!p->d_gt[0]) return fail(HB_ERR_NOGT, "parse was made without genotypes");
    if (gt0 && gt1 && is_pinned(gt0) && is_pinned(gt1)) {        // both planes in flight together
        CU(cudaMemcpy2DAsync(gt0, n, p->d_gt[0], p->gt_stride, n, p->n_samples, cudaMemcpyDeviceToHost, p->stream));
        CU(cudaMemcpy2DAsync(gt1, n, p->d_gt[1], p->gt_stride, n, p->n_samples, cudaMemcpyDeviceToHost, p->stream));
        CU(cudaStreamSynchronize(p->stream));
        return HB_OK;
    }
    if (gt0) CU(d2h_copy_2d(gt0, n, p->d_gt[0], p->gt_stride, n, p->n_samples, p->stream));
    if (gt1) CU(d2h_copy_2d(gt1, n, p->d_gt[1], p->gt_stride, n, p->n_samples, p->stream));
    return HB_OK;
}

int hb_parse_fetch_sample_errors(hb_parse *p, uint32_t *ploidy, uint32_t *badgt) {
    if (!p) return fail(HB_ERR_ARG, "null handle");
    CU(cudaSetDevice(p->device));
    if (!p->n_samples || !p->d_ploidy) return HB_OK;
    if (ploidy) CU(cudaMemcpy(ploidy, p->d_ploidy, p->n_samples * 4ull, cudaMemcpyDeviceToHost));
    if (badgt) CU(cudaMemcpy(badgt, p->d_badgt, p->n_samples * 4ull, cudaMemcpyDeviceToHost));
    return HB_OK;
}

int hb_parse_chrom_runs(hb_parse *p, uint64_t *n_runs, uint64_t *row_begin, uint64_t max_runs, char *names,
                        uint64_t names_cap, uint64_t *names_len) {
    if (!p || !n_runs) return fail(HB_ERR_ARG, "null argument");
    TRY(ensure_runs(p));
    *n_runs = p->run_rows.size();
    uint64_t used = 0;
    for (size_t i = 0; i < p->run_rows.size(); ++i) {
        if (row_begin && i < max_runs) row_begin[i] = p->run_rows[i];
        const std::string &s = p->run_names[i];
        if (names && used + s.size() + 1 <= names_cap) memcpy(names + used, s.c_str(), s.size() + 1);
        used += s.size() + 1;
    }
    if (names_len) *names_len = used;
    return HB_OK;
}

// =============================================================================================
// File level: .vcf / .vcf.gz reader (BGZF members inflate in parallel on the GPU) + per-(file, region) cache
// =============================================================================================
namespace hb {
bool bgzf_index(const uint8_t *raw, uint64_t size, std::vector<uint64_t> &coff, std::vector<uint32_t> &clen,
                std::vector<uint64_t> &ooff, std::vector<uint32_t> &olen, uint64_t &total, std::vector<uint64_t> *boff = nullptr);
int inflate_bgzf_to_device(const uint8_t *raw, uint64_t size, const std::vector<uint64_t> &coff,
                           const std::vector<uint32_t> &clen, const std::vector<uint64_t> &ooff,
                           const std::vector<uint32_t> &olen, uint8_t *d_out, cudaStream_t stream, float *ms);
}

namespace {

struct FileText {
    std::vector<uint8_t> data;   // whole decompressed file
    uint64_t body = 0;           // offset of the first record
    std::vector<std::string> samples;
    int end_is_int = 0;
    bool bcf = false;            // BCF 2.2: body = the records after the header text
    std::vector<std::string> contigs;   // BCF contig dictionary
    std::vector<uint64_t> contig_len;   // BCF: their ##contig length= (0: not given)
    int gt_key = -1;             // BCF string-dictionary index of GT (-1: not declared)
};

int read_all(const char *path, std::vector<uint8_t> &raw) {
    FILE *f = fopen(path, "rb");
    if (!f) return fail(HB_ERR_IO, std::string("cannot open ") + path);
    fseek(f, 0, SEEK_END);
    long sz = ftell(f);
    fseek(f, 0, SEEK_SET);
    raw.resize((size_t)sz);
    size_t got = sz ? fread(raw.data(), 1, (size_t)sz, f) : 0;
    fclose(f);
    if (got != (size_t)sz) return fail(HB_ERR_IO, std::string("short read on ") + path);
    return HB_OK;
}

// what parse_bytes_common does not inflate on the GPU: plain text as it is, and any gzip input that is not bgzip-conformant
// BGZF (e.g. the reference's own test fixture) through zlib, member after member, each checked against its CRC
int inflate_all(const std::vector<uint8_t> &raw, std::vector<uint8_t> &out) {
    if (raw.size() < 2 || raw[0] != 0x1f || raw[1] != 0x8b) { out = raw; return HB_OK; }   // plain text
    z_stream zs;
    memset(&zs, 0, sizeof zs);
    if (inflateInit2(&zs, 15 + 32) != Z_OK) return fail(HB_ERR_IO, "inflateInit2 failed");
    zs.next_in = const_cast<Bytef *>(raw.data());
    uint64_t in_left = raw.size();
    out.resize(std::max<size_t>(raw.size() * 4, 1 << 16));
    uint64_t produced = 0;
    for (;;) {
        if (out.size() - produced < (1 << 16)) out.resize(out.size() * 2);
        zs.avail_in = (uInt)std::min<uint64_t>(in_left, 1u << 30);
        uInt ain = zs.avail_in;
        zs.next_out = out.data() + produced;
        zs.avail_out = (uInt)std::min<uint64_t>(out.size() - produced, 1u << 30);
        uInt aout = zs.avail_out;
        int rc = inflate(&zs, Z_NO_FLUSH);
        produced += aout - zs.avail_out;
        in_left -= ain - zs.avail_in;
        if (rc == Z_STREAM_END) {
            if (in_left == 0) break;
            if (inflateReset(&zs) != Z_OK) { inflateEnd(&zs); return fail(HB_ERR_IO, "gzip member reset failed"); }
            continue;
        }
        if (rc != Z_OK && rc != Z_BUF_ERROR) { inflateEnd(&zs); return fail(HB_ERR_IO, "gzip inflate failed"); }
        if (rc == Z_BUF_ERROR && in_left == 0 && zs.avail_out != 0) { inflateEnd(&zs); return fail(HB_ERR_IO, "truncated gzip"); }
    }
    inflateEnd(&zs);
    out.resize(produced);
    return HB_OK;
}

// header lines of decompressed VCF text: sample names, INFO/END type, where the records start.
// complete = the #CHROM line (with its newline, or the end of the text when `whole`) lies inside [d, d + n)
bool parse_header(const uint8_t *d, uint64_t n, bool whole, FileText &ft) {
    ft.samples.clear();
    ft.end_is_int = 0;
    uint64_t p = 0;
    while (p < n && d[p] == '#') {
        const uint8_t *e = (const uint8_t *)memchr(d + p, '\n', n - p);
        if (!e && !whole) return false;                    // the line continues in text not inflated yet
        uint64_t le = e ? (uint64_t)(e - d) : n;
        if (p + 1 < n && d[p + 1] == '#') {
            std::string line((const char *)d + p, (const char *)d + le);
            if (line.compare(0, 15, "##INFO=<ID=END,") == 0 && line.find("Type=Integer") != std::string::npos) ft.end_is_int = 1;
        } else {
            uint64_t ce = le;
            if (ce > p && d[ce - 1] == '\r') --ce;
            uint64_t q = p; int col = 0;
            while (q <= ce) {
                const uint8_t *t = (const uint8_t *)memchr(d + q, '\t', ce - q);
                uint64_t te = t ? (uint64_t)(t - d) : ce;
                if (col >= 9) ft.samples.emplace_back((const char *)d + q, (const char *)d + te);
                ++col;
                if (!t) break;
                q = te + 1;
            }
            ft.body = e ? le + 1 : n;
            return true;
        }
        p = e ? le + 1 : n;
    }
    if (p >= n && !whole) return false;
    ft.body = p;
    return false;                                          // text without a #CHROM line
}

// attribute `key` of a structured header line "##X=<ID=...,key=value,...>" (values may be quoted)
bool hrec_attr(const std::string &line, const std::string &key, std::string &val) {
    size_t p = line.find('<');
    if (p == std::string::npos) return false;
    ++p;
    while (p < line.size()) {
        const size_t eq = line.find('=', p);
        if (eq == std::string::npos) return false;
        const std::string k = line.substr(p, eq - p);
        size_t q = eq + 1;
        std::string v;
        if (q < line.size() && line[q] == '"') {
            for (++q; q < line.size() && line[q] != '"'; ++q) {
                if (line[q] == '\\' && q + 1 < line.size()) ++q;
                v.push_back(line[q]);
            }
            ++q;
        } else {
            while (q < line.size() && line[q] != ',' && line[q] != '>') v.push_back(line[q++]);
        }
        if (k == key) { val = v; return true; }
        if (q >= line.size() || line[q] != ',') return false;
        p = q + 1;
    }
    return false;
}

// The header of a BCF 2.2 file (VCF v4.3 specification, section 6.3): magic "BCF\2\2", uint32 l_text, then l_text bytes of
// NUL-terminated VCF header text.  complete = false while [d, d + n) does not hold all of it.  Sample names come from the
// #CHROM line as for text.  Dictionaries, as htslib builds them: IDX= attributes (which htslib writes into BCF headers)
// win; without them the string dictionary is PASS = 0, then the FILTER / INFO / FORMAT IDs in order of first appearance
// (an ID shared by several lines gets one index), and the contig dictionary is the ##contig lines in order.
int bcf_header(const uint8_t *d, uint64_t n, FileText &ft, bool &complete) {
    complete = false;
    if (n < 5) return HB_OK;
    if (d[3] != 2 || d[4] != 2)
        return fail(HB_ERR_FORMAT, "BCF version " + std::to_string(d[3]) + "." + std::to_string(d[4]) +
                                       " is not supported: only BCF 2.2 is read");
    if (n < 9) return HB_OK;
    const uint32_t l_text = d[5] | d[6] << 8 | d[7] << 16 | (uint32_t)d[8] << 24;
    if (n < 9ull + l_text) return HB_OK;
    uint64_t len = l_text;
    while (len && d[9 + len - 1] == 0) --len;
    if (!parse_header(d + 9, len, true, ft)) return fail(HB_ERR_HEADER, "no #CHROM header line");
    std::map<std::string, int> strs{{"PASS", 0}};
    int next = 1, cnext = 0;
    std::vector<std::pair<int, std::string>> ctg;
    for (uint64_t p = 0; p < len;) {
        const uint8_t *e = (const uint8_t *)memchr(d + 9 + p, '\n', len - p);
        const uint64_t le = e ? (uint64_t)(e - d - 9) : len;
        const std::string line((const char *)d + 9 + p, (const char *)d + 9 + le);
        p = le + 1;
        const bool dict = line.rfind("##FILTER=<", 0) == 0 || line.rfind("##INFO=<", 0) == 0 || line.rfind("##FORMAT=<", 0) == 0;
        const bool contig = line.rfind("##contig=<", 0) == 0;
        std::string id, idx;
        if ((!dict && !contig) || !hrec_attr(line, "ID", id)) continue;
        const bool has_idx = hrec_attr(line, "IDX", idx) && !idx.empty() && idx.find_first_not_of("0123456789") == std::string::npos;
        const int i = has_idx ? std::atoi(idx.c_str()) : -1;
        if (contig) {
            const int c = i >= 0 ? i : cnext;
            cnext = std::max(cnext, c + 1);
            ctg.emplace_back(c, id);
            std::string len;
            if (hrec_attr(line, "length", len)) {
                if ((size_t)c >= ft.contig_len.size()) ft.contig_len.resize((size_t)c + 1, 0);
                ft.contig_len[(size_t)c] = strtoull(len.c_str(), nullptr, 10);
            }
        } else if (i >= 0) {
            strs[id] = i;
            next = std::max(next, i + 1);
        } else if (!strs.count(id)) strs[id] = next++;
    }
    ft.contigs.assign((size_t)cnext, std::string());
    ft.contig_len.resize((size_t)cnext, 0);
    for (auto &c : ctg) ft.contigs[(size_t)c.first] = c.second;
    const auto gt = strs.find("GT");
    ft.gt_key = gt == strs.end() ? -1 : gt->second;
    ft.bcf = true;
    ft.body = 9ull + l_text;
    complete = true;
    return HB_OK;
}

bool is_bcf(const uint8_t *d, uint64_t n) { return n >= 3 && memcmp(d, "BCF", 3) == 0; }

// the sample names of hb_parse_file_subset / hb_parse_vcf_bytes_subset
struct Subset {
    const char *const *names;
    uint32_t n;
};

// The columns of subset ss among the header's samples, ascending: the planes come out in header order whatever the order of
// the names, as htslib's bcf_hdr_set_samples gives them.  samples becomes the names of the planes.  ss == nullptr: every
// sample, cols stays empty.
int resolve_subset(const Subset *ss, std::vector<std::string> &samples, std::vector<uint32_t> &cols) {
    cols.clear();
    if (!ss) return HB_OK;
    if (!ss->names || ss->n == 0) return fail(HB_ERR_ARG, "a sample subset names at least one sample");
    std::map<std::string, uint32_t> at;
    for (uint32_t i = 0; i < samples.size(); ++i) at.emplace(samples[i], i);
    std::vector<uint8_t> taken(samples.size(), 0);
    for (uint32_t k = 0; k < ss->n; ++k) {
        if (!ss->names[k]) return fail(HB_ERR_ARG, "null sample name");
        const auto it = at.find(ss->names[k]);
        if (it == at.end()) return fail(HB_ERR_SAMPLE, std::string("sample ") + ss->names[k] + " is not in the VCF header");
        if (taken[it->second]) return fail(HB_ERR_ARG, std::string("sample ") + ss->names[k] + " is named twice");
        taken[it->second] = 1;
        cols.push_back(it->second);
    }
    std::sort(cols.begin(), cols.end());
    std::vector<std::string> picked;
    for (uint32_t c : cols) picked.push_back(samples[c]);
    samples.swap(picked);
    return HB_OK;
}

int read_vcf(const std::vector<uint8_t> &raw, FileText &ft) {
    TRY(inflate_all(raw, ft.data));
    if (is_bcf(ft.data.data(), ft.data.size())) {
        bool complete = false;
        TRY(bcf_header(ft.data.data(), ft.data.size(), ft, complete));
        return complete ? HB_OK : fail(HB_ERR_FORMAT, "BCF header is truncated");
    }
    if (!ft.data.empty() && ft.data.back() != '\n') ft.data.push_back('\n');
    if (!parse_header(ft.data.data(), ft.data.size(), true, ft)) return fail(HB_ERR_HEADER, "no #CHROM header line");
    return HB_OK;
}

// One .vcf / .vcf.gz -> device-resident parse.  BGZF files (what bgzip writes, what the reference's tabix path
// reads) travel over PCIe COMPRESSED and are inflated on the GPU (hb_inflate.cu) straight into the text buffer;
// only the header members are also inflated on the host, to learn the sample names.  Any other gzip input (plain
// gzip, or BGZF that bgzip would not have written) and plain text go through zlib / as they are.
// hb_parse_stream_bgzf_resident with the sample subset cols (empty = every sample)
int stream_resident(const uint8_t *bgzf, uint64_t nbytes, const char *region, int want_gt, int device, uint64_t slab_bytes,
                    hb_parse **out, uint32_t *n_slabs, const std::vector<uint32_t> &cols);

// ss: a sample subset (nullptr = every sample); samples: the names of the parse's planes
int parse_bytes_common(std::vector<uint8_t> &raw_owned, const uint8_t *raw_p, uint64_t raw_n, const char *region, bool want_gt,
                       int device, hb_parse **out, std::vector<std::string> &samples, const Subset *ss);

// a region query of a file with a usable .tbi / .csi next to it: HB_OK with used = false when the index is not usable
int parse_file_indexed(const char *path, const char *region, bool want_gt, int device, hb_parse **out,
                       std::vector<std::string> &samples, bool &used, const Subset *ss);

int parse_file_common(const char *path, const char *region, bool want_gt, int device, hb_parse **out,
                      std::vector<std::string> &samples, const Subset *ss = nullptr) {
    bool used = false;
    TRY(parse_file_indexed(path, region, want_gt, device, out, samples, used, ss));
    if (used) return HB_OK;
    std::vector<uint8_t> raw;
    TRY(read_all(path, raw));
    return parse_bytes_common(raw, raw.data(), raw.size(), region, want_gt, device, out, samples, ss);
}

// a BGZF file: its member table, then its header
struct BgzfFile {
    std::vector<uint64_t> coff, ooff;
    std::vector<uint32_t> clen, olen;
    uint64_t total = 0;          // bytes of text
    FileText ft;
};

// false: the bytes are not BGZF (each caller has its own answer to that)
bool index_bgzf(const uint8_t *raw, uint64_t n, BgzfFile &f) { return bgzf_index(raw, n, f.coff, f.clen, f.ooff, f.olen, f.total); }

// the VCF header of a BGZF file: leading members are inflated on the host (zlib) until the #CHROM line is complete; with
// hb_set_bgzf_crc_check on, each is checked against its CRC32 as kernel 0 checks the others.  more != NULL: f holds only the
// leading members of the file, and *more = true asks for more of them when the header does not end inside those
int bgzf_header(const uint8_t *raw, BgzfFile &f, bool *more = nullptr) {
    std::vector<uint8_t> head;
    bool have = false;
    const bool check_crc = bgzf_crc_check();
    for (size_t i = 0; i < f.coff.size() && !have; ++i) {
        const size_t at = head.size();
        head.resize(at + f.olen[i]);
        z_stream zs;
        memset(&zs, 0, sizeof zs);
        if (inflateInit2(&zs, -15) != Z_OK) return fail(HB_ERR_IO, "inflateInit2 failed");
        zs.next_in = const_cast<Bytef *>(raw + f.coff[i]);
        zs.avail_in = f.clen[i];
        zs.next_out = head.data() + at;
        zs.avail_out = f.olen[i];
        const int zr = inflate(&zs, Z_FINISH);
        inflateEnd(&zs);
        if (zr != Z_STREAM_END || zs.avail_out != 0) return fail(HB_ERR_IO, "BGZF inflate failed (header)");
        if (check_crc) {
            const uint8_t *tr = raw + f.coff[i] + f.clen[i];
            const uint32_t want = tr[0] | tr[1] << 8 | tr[2] << 16 | (uint32_t)tr[3] << 24;
            if ((uint32_t)crc32(crc32(0L, Z_NULL, 0), head.data() + at, f.olen[i]) != want) return fail(HB_ERR_IO, bgzf_crc_message(raw, f.coff[i]));
        }
        if (is_bcf(head.data(), head.size())) TRY(bcf_header(head.data(), head.size(), f.ft, have));
        else have = parse_header(head.data(), head.size(), !more && i + 1 == f.coff.size(), f.ft);
    }
    if (more) *more = !have;
    if (!have && more) return HB_OK;
    if (!have && is_bcf(head.data(), head.size())) return fail(HB_ERR_FORMAT, "BCF header is truncated");
    if (!have) return fail(HB_ERR_HEADER, "no #CHROM header line");
    return HB_OK;
}

// text bytes a whole-file parse may hold in HBM (hb_parse_set_text_limit, else from free device memory); slab: the slab
// size of the streamed route
uint64_t text_limit(uint64_t &slab) {
    uint64_t limit = g_text_limit.load();
    slab = limit ? std::max<uint64_t>(limit / 2, 1 << 16) : 0;      // two slabs of text are resident at a time
    if (!limit) {
        size_t fr = 0, tot = 0;
        if (cudaMemGetInfo(&fr, &tot) != cudaSuccess) { cudaGetLastError(); fr = 0; }
        // GT-only text is ~4 bytes per call, the planes + bit planes it leaves 2.125: text + 0.55 x text must fit
        limit = (uint64_t)(0.9 * (double)(fr + hb::dev_pool_idle_bytes()) / 1.55);
    }
    return limit;
}

// a BCF's contig table and names on the device, and the dictionaries on the handle
int bcf_attach(hb_parse *p, const FileText &ft) {
    hb_parse::Bcf *b = p->bcf = new hb_parse::Bcf();
    b->contigs = ft.contigs;
    b->gt_key = ft.gt_key;
    std::string names;
    std::vector<BcfContig> tab;
    for (const std::string &c : ft.contigs) {
        BcfContig x{0, names.size(), (uint32_t)std::min<size_t>(c.size(), 255), 0};
        for (size_t k = 0; k < 5 && k < c.size(); ++k) x.name5 |= (uint64_t)(uint8_t)c[k] << (8 * k);
        b->name_off.push_back(names.size());
        tab.push_back(x);
        names += c;
        names.push_back('\0');
    }
    TRY(dev_alloc(&b->d_contigs, tab.size()));
    TRY(dev_alloc(&b->d_names, names.size() + 1));
    if (!tab.empty()) CU(cudaMemcpy(b->d_contigs, tab.data(), tab.size() * sizeof(BcfContig), cudaMemcpyHostToDevice));
    if (!names.empty()) CU(cudaMemcpy(b->d_names, names.data(), names.size(), cudaMemcpyHostToDevice));
    return HB_OK;
}

int bcf_too_big(uint64_t body) {
    return fail(HB_ERR_ARG, "BCF body of " + std::to_string(body) + " bytes exceeds the text limit and BCF streaming is not supported");
}

// the body of an uncompressed or plain-gzip BCF, inflated on the host
int parse_bcf_host(const FileText &ft, const hb_parse_opts &o, const std::vector<uint32_t> &cols, hb_parse **out) {
    const uint64_t n = ft.data.size() - ft.body;
    uint64_t slab;
    TRY(ensure_device(o.device));
    if (n > text_limit(slab)) return bcf_too_big(n);
    int rc;
    ParsePtr p = new_parse(&o, rc);
    if (!p) return rc;
    TRY(set_subset(p.get(), cols));
    TRY(upload_text(p.get(), ft.data.data() + ft.body, n, false));
    TRY(bcf_attach(p.get(), ft));
    TRY(run_parse(p.get()));
    *out = p.release();
    return HB_OK;
}

hb_parse_opts opts_for(const FileText &ft, const char *region, bool want_gt, int device) {
    hb_parse_opts o;
    memset(&o, 0, sizeof o);
    o.region = region;
    o.want_gt = want_gt ? 1 : 0;
    o.device = device;
    o.n_samples = (uint32_t)ft.samples.size();
    o.end_is_int = ft.end_is_int;
    return o;
}

// raw_p[0..raw_n): the bytes of a .vcf / .vcf.gz / .bcf; raw_owned: the vector that holds them when the caller read a file
// (released early on the zlib path), empty when they belong to the caller
int parse_bytes_common(std::vector<uint8_t> &raw_owned, const uint8_t *raw_p, uint64_t raw_n, const char *region, bool want_gt,
                       int device, hb_parse **out, std::vector<std::string> &samples, const Subset *ss) {
    BgzfFile bz;
    std::vector<uint32_t> cols;
    const bool gpu_inflate = raw_n >= 28 && raw_p[0] == 0x1f && raw_p[1] == 0x8b && index_bgzf(raw_p, raw_n, bz) && bz.total > 0;
    if (!gpu_inflate) {
        FileText ft;
        if (raw_owned.empty()) raw_owned.assign(raw_p, raw_p + raw_n);
        TRY(read_vcf(raw_owned, ft));
        raw_owned.clear(); raw_owned.shrink_to_fit();
        samples = ft.samples;
        TRY(resolve_subset(ss, samples, cols));
        const hb_parse_opts o = opts_for(ft, region, want_gt, device);
        if (ft.bcf) return parse_bcf_host(ft, o, cols, out);
        return host_text(ft.data.data() + ft.body, ft.data.size() - ft.body, &o, cols, out);
    }
    // ---- header: inflate leading members on the host until the #CHROM line is complete
    TRY(bgzf_header(raw_p, bz));
    const FileText &ft = bz.ft;
    const uint64_t total = bz.total;
    samples = ft.samples;
    TRY(resolve_subset(ss, samples, cols));
    {   // a file whose text does not fit HBM next to its genotype planes passes through in slabs instead: same rows, same
        // handle minus the text (hb_parse_stream_bgzf_resident)
        TRY(ensure_device(device));
        uint64_t slab;
        const uint64_t limit = text_limit(slab);
        if (total > limit && ft.bcf) return bcf_too_big(total - ft.body);
        if (total > limit) return stream_resident(raw_p, raw_n, region, want_gt ? 1 : 0, device, slab, out, nullptr, cols);
    }
    const hb_parse_opts o = opts_for(ft, region, want_gt, device);
    const bool trace = getenv("HB_TRACE") != nullptr;
    const double t0 = now_ms();
    int rc;
    ParsePtr p = new_parse(&o, rc);
    if (!p) return rc;
    TRY(set_subset(p.get(), cols));
    const uint64_t pad = (16 - ft.body % 16) % 16;         // the records must start on a 16-byte boundary
    TRY(dev_alloc(&p->d_text_owned, pad + total + 1 + kTextPad));
    const double t1 = now_ms();
    TRY(inflate_bgzf_to_device(raw_p, raw_n, bz.coff, bz.clen, bz.ooff, bz.olen, p->d_text_owned + pad, p->stream, &p->ms_inflate));
    uint8_t last = 0;
    cudaError_t e = cudaMemcpy(&last, p->d_text_owned + pad + total - 1, 1, cudaMemcpyDeviceToHost);
    uint64_t end = pad + total;
    if (e == cudaSuccess && last != '\n' && !ft.bcf) { e = cudaMemset(p->d_text_owned + end, '\n', 1); ++end; }
    if (e == cudaSuccess) e = cudaMemset(p->d_text_owned + end, 0, kTextPad);
    if (e != cudaSuccess) return fail_cuda(e);
    p->d_text = p->d_text_owned + pad + ft.body;
    p->nbytes = end - pad - ft.body;
    p->compressed_bytes = raw_n;
    const double t2 = now_ms();
    rc = ft.bcf ? bcf_attach(p.get(), ft) : HB_OK;
    if (rc == HB_OK) rc = run_parse(p.get());
    if (trace) fprintf(stderr, "[parse_bytes_common] text buffer %.1f ms, H2D + inflate %.1f ms, parse %.1f ms\n", t1 - t0, t2 - t1, now_ms() - t2);
    TRY(rc);
    *out = p.release();
    return HB_OK;
}

// ---- region queries through a tabix / CSI index: only the BGZF members of the query's span are read and inflated
std::atomic<int> g_use_index{1};                  // hb_set_use_index

void index_not_used(const std::string &why) {
    if (getenv("HB_TRACE")) fprintf(stderr, "[index] not used: %s\n", why.c_str());
}

// the bytes of a file (pread) or of a caller's buffer
struct ByteSource {
    const uint8_t *mem = nullptr;
    int fd = -1;
    uint64_t size = 0;
    const uint8_t *get(uint64_t off, uint64_t n, std::vector<uint8_t> &buf) const {
        if (off > size || n > size - off) return nullptr;
        if (mem) return mem + off;
        buf.resize(n);
        for (uint64_t got = 0; got < n;) {
            const ssize_t r = pread(fd, buf.data() + got, n - got, (off_t)(off + got));
            if (r <= 0) return nullptr;
            got += (uint64_t)r;
        }
        return buf.data();
    }
};

// bytes of the BGZF member that starts at h (avail bytes readable there), 0 when none starts there
uint64_t bgzf_member_size(const uint8_t *h, uint64_t avail) {
    if (avail < 18 || h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || !(h[3] & 4)) return 0;
    const uint64_t xe = 12ull + (h[10] | h[11] << 8);
    if (xe > avail) return 0;
    for (uint64_t q = 12; q + 4 <= xe; q += 4 + (h[q + 2] | h[q + 3] << 8))
        if (h[q] == 'B' && h[q + 1] == 'C' && (h[q + 2] | h[q + 3] << 8) == 2 && q + 6 <= xe) return (h[q + 4] | h[q + 5] << 8) + 1ull;
    return 0;
}

// The parse of `region` from the members of src that hold the records the index lists for it.  The region filter runs
// as on a full scan, so the rows are the same.  used = false (with `why`): the index cannot serve this query and the
// caller takes the full-scan route; nothing has been parsed then.
// The header of BGZF input, from its leading members only: twice as many bytes of them each round until the header ends
// inside them (the rounds re-inflate what the round before inflated: at most twice the header's members in all).  false
// (with `why`): the input is not BGZF or its header does not read.  head_read: the compressed bytes read.
bool leading_bgzf_header(const ByteSource &src, FileText &ft, uint64_t &head_read, std::string &why) {
    std::vector<uint8_t> hbuf;
    {
        const uint8_t *h = src.get(0, std::min<uint64_t>(src.size, 18), hbuf);
        if (!h || !bgzf_member_size(h, std::min<uint64_t>(src.size, 18))) { why = "the input is not BGZF"; return false; }
    }
    BgzfFile bz;
    head_read = 0;
    std::vector<uint8_t> head;                              // bytes [0, head_read) of a file source
    for (bool more = true; more;) {
        const uint64_t target = std::min(src.size, std::max<uint64_t>(2 * head_read, 1));
        const uint64_t avail = std::min<uint64_t>(src.size, target + 65536) - head_read;
        const uint8_t *b = src.get(head_read, avail, hbuf);
        uint64_t w = 0;
        for (uint64_t s; b && head_read + w < target && (s = bgzf_member_size(b + w, avail - w)) != 0 && s <= avail - w;) w += s;
        if (!w) { why = "the input is not BGZF"; return false; }
        if (!src.mem) head.insert(head.end(), b, b + w);
        head_read += w;
        const uint8_t *all = src.mem ? src.mem : head.data();
        bz = BgzfFile();
        if (!index_bgzf(all, head_read, bz)) { why = "the input is not BGZF"; return false; }
        const std::string err = g_err;
        if (bgzf_header(all, bz, head_read < src.size ? &more : nullptr) != HB_OK) { g_err = err; why = "the header does not read"; return false; }
        if (head_read == src.size) more = false;
    }
    ft = bz.ft;
    return true;
}

int parse_indexed(const ByteSource &src, const uint8_t *ix, uint64_t ix_n, const char *region, bool want_gt, int device,
                  hb_parse **out, std::vector<std::string> &samples, bool &used, std::string &why, const Subset *ss) {
    used = false;
    std::vector<uint8_t> sbuf;
    {
        std::vector<uint8_t> hbuf;
        const uint8_t *h = src.get(0, std::min<uint64_t>(src.size, 18), hbuf);
        if (!h || !bgzf_member_size(h, std::min<uint64_t>(src.size, 18))) { why = "the input is not BGZF"; return HB_OK; }
    }
    TabixIndex idx;
    if (!tabix_load(ix, ix_n, idx, why)) return HB_OK;
    FileText ft;
    uint64_t head_read = 0;
    if (!leading_bgzf_header(src, ft, head_read, why)) return HB_OK;
    if (ft.bcf && !idx.csi) { why = "a BCF is queried through a CSI index only"; return HB_OK; }
    if (!ft.bcf && idx.names.empty()) { why = "the index names no sequences"; return HB_OK; }
    RegionArg rg;
    parse_region(region, rg);
    const std::vector<std::string> &names = ft.bcf ? ft.contigs : idx.names;
    const auto at = std::find(names.begin(), names.end(), std::string(rg.chrom, rg.chrom_len));
    const auto chunks = at == names.end() ? std::vector<std::pair<uint64_t, uint64_t>>()
                                          : tabix_query(idx, (int)(at - names.begin()), rg.beg0, rg.end0);
    // the span [first chunk begin, last chunk end): its members, read in one piece
    BgzfFile sp;
    const uint8_t *sb = nullptr;
    uint64_t t0 = 0, t1 = 0, span_comp = 0;
    if (!chunks.empty()) {
        const uint64_t c0 = chunks.front().first >> 16, c1 = chunks.back().second >> 16;
        const uint64_t u0 = chunks.front().first & 0xffff, u1 = chunks.back().second & 0xffff;
        if (c1 < c0 || c1 > src.size) { why = "the index points past the end of the file"; return HB_OK; }
        const uint64_t n = std::min<uint64_t>(src.size, c1 + (u1 ? 65536 : 0)) - c0;
        sb = src.get(c0, n, sbuf);
        if (!sb) { why = "read error"; return HB_OK; }
        uint64_t w = 0, last = 0;
        while (c0 + w < c1 || (u1 && c0 + w == c1)) {
            const uint64_t s = bgzf_member_size(sb + w, n - w);
            if (!s || s > n - w) break;
            last = w;
            w += s;
        }
        if (c0 + w < c1 || (u1 && c0 + last != c1) || !index_bgzf(sb, w, sp) || sp.total == 0) {
            why = "the index's offsets do not fall on BGZF members of the file";
            return HB_OK;
        }
        t0 = u0;
        t1 = u1 ? sp.total - sp.olen.back() + u1 : sp.total;
        if (t0 > t1 || u0 > sp.olen.front() || (u1 && u1 > sp.olen.back())) { why = "the index's offsets do not fall on BGZF members of the file"; return HB_OK; }
        span_comp = w;
    }
    TRY(ensure_device(device));
    uint64_t slab;
    if (t1 - t0 > text_limit(slab)) { why = "the region's span is above the text limit"; return HB_OK; }
    used = true;
    samples = ft.samples;
    std::vector<uint32_t> cols;
    TRY(resolve_subset(ss, samples, cols));
    const hb_parse_opts o = opts_for(ft, region, want_gt, device);
    const double ta = now_ms();
    int rc;
    ParsePtr p = new_parse(&o, rc);
    if (!p) return rc;
    TRY(set_subset(p.get(), cols));
    const uint64_t pad = (16 - t0 % 16) % 16;           // the records start on a 16-byte boundary
    TRY(dev_alloc(&p->d_text_owned, pad + sp.total + 1 + kTextPad));
    if (t1 > t0) TRY(inflate_bgzf_to_device(sb, span_comp, sp.coff, sp.clen, sp.ooff, sp.olen, p->d_text_owned + pad, p->stream, &p->ms_inflate));
    uint8_t *text = p->d_text_owned + pad + t0;
    uint64_t nb = t1 - t0;
    uint8_t last = '\n';
    cudaError_t e = nb ? cudaMemcpy(&last, text + nb - 1, 1, cudaMemcpyDeviceToHost) : cudaSuccess;
    if (e == cudaSuccess && last != '\n' && !ft.bcf) { e = cudaMemset(text + nb, '\n', 1); ++nb; }
    if (e == cudaSuccess) e = cudaMemset(text + nb, 0, kTextPad);
    if (e != cudaSuccess) return fail_cuda(e);
    p->d_text = text;
    p->nbytes = nb;
    p->compressed_bytes = span_comp;
    p->idx_used = 1;
    p->idx_bytes_read = head_read + span_comp;
    p->idx_chunks = chunks.size();
    const double tb = now_ms();
    rc = ft.bcf ? bcf_attach(p.get(), ft) : HB_OK;
    if (rc == HB_OK) rc = run_parse(p.get());
    if (getenv("HB_TRACE"))
        fprintf(stderr, "[index] %zu chunks, %llu of %llu compressed bytes read: H2D + inflate %.1f ms, parse %.1f ms\n", chunks.size(),
                (unsigned long long)p->idx_bytes_read, (unsigned long long)src.size, tb - ta, now_ms() - tb);
    TRY(rc);
    *out = p.release();
    return HB_OK;
}

// htslib's order: <path>.tbi then <path>.csi for a .vcf.gz, <path>.csi for a .bcf; an index older than the data is ignored
bool find_index(const char *path, std::vector<uint8_t> &ix, std::string &why) {
    const std::string base(path);
    const bool bcf = base.size() >= 4 && base.compare(base.size() - 4, 4, ".bcf") == 0;
    struct stat sd, si;
    if (stat(path, &sd) != 0) { why = "cannot stat the data file"; return false; }
    for (const char *ext : {".tbi", ".csi"}) {
        if (bcf && ext[1] == 't') continue;
        const std::string ip = base + ext;
        if (stat(ip.c_str(), &si) != 0) continue;
        if (si.st_mtime < sd.st_mtime) { why = ip + " is older than the data file"; return false; }
        const std::string err = g_err;
        if (read_all(ip.c_str(), ix) != HB_OK) { g_err = err; why = "cannot read " + ip; return false; }
        return true;
    }
    why = "no index next to the file";
    return false;
}

int parse_file_indexed(const char *path, const char *region, bool want_gt, int device, hb_parse **out,
                       std::vector<std::string> &samples, bool &used, const Subset *ss) {
    used = false;
    std::string why;
    std::vector<uint8_t> ix;
    if (!region || !*region) why = "the region is empty";
    else if (!g_use_index.load()) why = "hb_set_use_index(0)";
    else if (find_index(path, ix, why)) {
        const int fd = open(path, O_RDONLY);
        struct stat st;
        int rc = HB_OK;
        if (fd < 0 || fstat(fd, &st) != 0) why = std::string("cannot open ") + path;
        else rc = parse_indexed(ByteSource{nullptr, fd, (uint64_t)st.st_size}, ix.data(), ix.size(), region, want_gt, device, out,
                                samples, used, why, ss);
        if (fd >= 0) close(fd);
        if (rc != HB_OK || used) return rc;
    }
    index_not_used(why);
    return HB_OK;
}

struct CacheEntry {
    std::mutex mu;
    std::condition_variable cv;
    bool done = false;
    int rc = HB_OK;
    std::string err;
    hb_parse *parse = nullptr;
    std::vector<std::string> samples;
    std::vector<uint32_t> start, stop, chrom_off;
    std::vector<char> ref, alt;
    std::string chrom_pool;
    std::vector<uint32_t> ploidy_err, badgt_err;
    bool want_gt = true;
    uint64_t hbm_bytes = 0;            // device memory the entry pins (genotype planes + bit planes)
    uint64_t last_use = 0;             // LRU tick (g_cache_mu)
    ~CacheEntry() { if (parse) hb_parse_free(parse); }
};

// The per-sample reference API (one load_vcf call per donor and chromosome, vcf_to_h5.py:150-152) is served from
// device-resident parses kept here.  Key = path + file identity (size, mtime, inode: a file rewritten in place is a
// different key) + region.  Entries are dropped least-recently-used first once they pin more than g_cache_limit bytes
// of HBM (default 40 % of the device), and all idle ones go when a parse runs out of device memory.  An entry that is
// still referenced by records handed out lives on until they are freed.
std::mutex g_cache_mu;
std::map<std::string, std::shared_ptr<CacheEntry>> g_cache;
uint64_t g_cache_tick = 0, g_cache_limit = 0;

std::string file_identity(const char *path) {
    struct stat st;
    if (stat(path, &st) != 0) return "?";
    return std::to_string((unsigned long long)st.st_size) + ":" + std::to_string((long long)st.st_mtim.tv_sec) + "." +
           std::to_string((long)st.st_mtim.tv_nsec) + ":" + std::to_string((unsigned long long)st.st_ino);
}

uint64_t cache_limit_bytes() {           // g_cache_mu held
    if (g_cache_limit) return g_cache_limit;
    size_t fr = 0, tot = 0;
    if (cudaMemGetInfo(&fr, &tot) != cudaSuccess) { cudaGetLastError(); return 64ull << 30; }
    return (uint64_t)(0.4 * (double)tot);
}

// drop finished entries, least recently used first, until the rest pins at most `limit` bytes; `keep` stays
void cache_evict(uint64_t limit, const CacheEntry *keep) {      // g_cache_mu held
    for (;;) {
        uint64_t sum = 0;
        auto victim = g_cache.end();
        for (auto it = g_cache.begin(); it != g_cache.end(); ++it) {
            CacheEntry *ce = it->second.get();
            sum += ce->hbm_bytes;
            if (ce == keep || !ce->done) continue;                  // (done is set under ce->mu before the entry is used again)
            if (victim == g_cache.end() || ce->last_use < victim->second->last_use) victim = it;
        }
        if (sum <= limit || victim == g_cache.end()) return;
        g_cache.erase(victim);
    }
}

int env_device() {
    const char *e = getenv("HB_DEVICE");
    if (e && *e) return atoi(e);
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess) d = 0;
    return d;
}

int build_entry(CacheEntry &ce, const char *path, const char *region, bool want_gt) {
    ce.want_gt = want_gt;
    TRY(parse_file_common(path, region, want_gt, env_device(), &ce.parse, ce.samples));
    const uint32_t n_samples = (uint32_t)ce.samples.size();
    hb_parse *p = ce.parse;
    uint64_t n = p->h_st.n_records;
    ce.start.resize(n); ce.stop.resize(n); ce.ref.resize(n); ce.alt.resize(n); ce.chrom_off.resize(n);
    TRY(hb_parse_fetch_sites(p, ce.start.data(), ce.stop.data(), ce.ref.data(), ce.alt.data()));
    TRY(ensure_runs(p));
    for (size_t i = 0; i < p->run_rows.size(); ++i) {
        uint32_t off = (uint32_t)ce.chrom_pool.size();
        ce.chrom_pool.append(p->run_names[i]);
        ce.chrom_pool.push_back('\0');
        uint64_t b = p->run_rows[i], e = i + 1 < p->run_rows.size() ? p->run_rows[i + 1] : n;
        for (uint64_t r = b; r < e; ++r) ce.chrom_off[r] = off;
    }
    if (want_gt) {
        ce.ploidy_err.resize(n_samples); ce.badgt_err.resize(n_samples);
        TRY(hb_parse_fetch_sample_errors(p, ce.ploidy_err.data(), ce.badgt_err.data()));
    }
    // the text is no longer needed once names are resolved: give the HBM back
    if (p->d_text_owned) { free_dev(p->d_text_owned); p->d_text_owned = nullptr; p->d_text = nullptr; }
    ce.hbm_bytes = want_gt ? 2 * p->gt_bytes + 4 * p->bits_stride * p->n_samples : 0;
    return HB_OK;
}

std::shared_ptr<CacheEntry> get_entry(const char *path, const char *region, bool want_gt, int &rc) {
    // a parse made without the BGZF CRC check must not answer a call made with it
    const std::string base = std::string(path) + "\x01" + file_identity(path) + "\x01" + (region ? region : "") +
                             (bgzf_crc_check() ? "\x01crc" : "");
    const std::string key = base + (want_gt ? "\x01g" : "\x01s");
    std::shared_ptr<CacheEntry> ce;
    bool builder = false;
    {
        std::lock_guard<std::mutex> lk(g_cache_mu);
        auto it = g_cache.find(key);
        if (it == g_cache.end() && !want_gt) {   // a genotype parse also answers site queries
            auto it2 = g_cache.find(base + "\x01g");
            if (it2 != g_cache.end()) it = it2;
        }
        if (it == g_cache.end()) {
            ce = std::make_shared<CacheEntry>(); g_cache[key] = ce; builder = true;
            // an older parse of the same path (the file was rewritten since) can never be asked for again
            const std::string any_id = std::string(path) + "\x01", this_id = any_id + file_identity(path) + "\x01";
            for (auto jt = g_cache.begin(); jt != g_cache.end();) {
                const bool same_path = jt->first.compare(0, any_id.size(), any_id) == 0;
                const bool same_file = jt->first.compare(0, this_id.size(), this_id) == 0;
                if (same_path && !same_file && jt->second->done) jt = g_cache.erase(jt);
                else ++jt;
            }
        } else ce = it->second;
        ce->last_use = ++g_cache_tick;
    }
    if (builder) {
        int r = build_entry(*ce, path, region, want_gt);
        if (r == HB_ERR_MEM || r == HB_ERR_CUDA) {          // out of device memory? drop every idle entry and try once more
            { std::lock_guard<std::mutex> lk(g_cache_mu); cache_evict(0, ce.get()); }
            hb::dev_pool_flush();
            cudaGetLastError();
            if (ce->parse) { hb_parse_free(ce->parse); ce->parse = nullptr; }
            ce->samples.clear(); ce->chrom_pool.clear();
            r = build_entry(*ce, path, region, want_gt);
        }
        {
            std::lock_guard<std::mutex> lk(ce->mu);
            ce->rc = r; ce->err = g_err; ce->done = true;
        }
        ce->cv.notify_all();
        std::lock_guard<std::mutex> lk(g_cache_mu);
        if (r != HB_OK) g_cache.erase(key);
        else cache_evict(cache_limit_bytes(), ce.get());
    } else {
        std::unique_lock<std::mutex> lk(ce->mu);
        ce->cv.wait(lk, [&] { return ce->done; });
    }
    rc = ce->rc;
    if (rc != HB_OK) g_err = ce->err;
    return ce;
}

struct RecOwner {
    std::shared_ptr<CacheEntry> ce;
    std::vector<int8_t> gt0, gt1;
};

void fill_records(hb_records *out, RecOwner *ow) {
    CacheEntry &ce = *ow->ce;
    out->n = ce.start.size();
    out->n_samples = (uint32_t)ce.samples.size();
    out->start = ce.start.data(); out->stop = ce.stop.data();
    out->ref = ce.ref.data(); out->alt = ce.alt.data();
    out->chrom_off = ce.chrom_off.data();
    out->chrom_pool = ce.chrom_pool.data();
    out->chrom_pool_len = ce.chrom_pool.size();
    out->gt0 = ow->gt0.empty() ? nullptr : ow->gt0.data();
    out->gt1 = ow->gt1.empty() ? nullptr : ow->gt1.data();
    out->owner_ = ow;
}

}  // namespace

int hb_load_vcf(const char *in_vcf, const char *sample, const char *chrom, hb_records *out) {
    if (!in_vcf || !sample || !out) return fail(HB_ERR_ARG, "null argument");
    memset(out, 0, sizeof *out);
    if (!*sample) return fail(HB_ERR_SAMPLE, "load_vcf needs a sample name (hb_load_vcf_without_sample answers site queries)");
    int rc;
    auto ce = get_entry(in_vcf, chrom, true, rc);
    if (rc != HB_OK) return rc;
    auto it = std::find(ce->samples.begin(), ce->samples.end(), std::string(sample));
    if (it == ce->samples.end())
        return fail(HB_ERR_SAMPLE, "the 1-th sample are not in the VCF.\nparameter samples:" + std::string(sample));
    uint32_t s = (uint32_t)(it - ce->samples.begin());
    uint64_t n = ce->start.size();
    if (n && ce->parse->h_st.n_nogt)
        return fail(HB_ERR_NOGT, "genotypes not present. make sure you initilized the variant object first\n");
    if (ce->badgt_err[s]) return fail(HB_ERR_GT, "Couldn't read GT data: value not a number or '.'");
    if (ce->ploidy_err[s])
        return fail(HB_ERR_PLOIDY, "ploidy != 2 (reference: assert(var.ploidy() == 2), parse_vcf.cpp:46)");
    auto *ow = new RecOwner();
    ow->ce = ce;
    ow->gt0.resize(n ? n : 1); ow->gt1.resize(n ? n : 1);
    rc = hb_parse_fetch_sample(ce->parse, s, ow->gt0.data(), ow->gt1.data());
    if (rc != HB_OK) { delete ow; return rc; }
    fill_records(out, ow);
    return HB_OK;
}

int hb_load_vcf_without_sample(const char *in_vcf, const char *chrom, hb_records *out) {
    if (!in_vcf || !out) return fail(HB_ERR_ARG, "null argument");
    memset(out, 0, sizeof *out);
    int rc;
    auto ce = get_entry(in_vcf, chrom, false, rc);
    if (rc != HB_OK) return rc;
    auto *ow = new RecOwner();
    ow->ce = ce;
    fill_records(out, ow);
    out->gt0 = out->gt1 = nullptr;
    return HB_OK;
}

void hb_records_free(hb_records *r) {
    if (!r || !r->owner_) return;
    delete static_cast<RecOwner *>(r->owner_);
    memset(r, 0, sizeof *r);
}

void hb_cache_set_limit(uint64_t hbm_bytes) {
    std::lock_guard<std::mutex> lk(g_cache_mu);
    g_cache_limit = hbm_bytes;
    if (hbm_bytes) cache_evict(hbm_bytes, nullptr);
}

void hb_parse_set_text_limit(uint64_t text_bytes) { g_text_limit.store(text_bytes); }
void hb_set_walker_lines(uint32_t lines) { g_walker_lines.store(lines == 0 ? 16u : std::min(lines, 20u)); }
void hb_set_bcf_segment_bytes(uint64_t bytes) { g_bcf_segment.store(bytes == 0 ? 0 : std::max<uint64_t>(bytes, 64)); }

void hb_cache_clear(void) {
    {
        std::lock_guard<std::mutex> lk(g_cache_mu);
        g_cache.clear();
    }
    hb::frames_buffer_cache_clear();
    clear_slot_cache(g_text_slots);
    clear_slot_cache(g_bgzf_slots);
    hb::dev_pool_flush();
}

const char *hb_last_error(void) { return g_err.c_str(); }
const char *hb_version(void) { return "haplo_b200 0.1 (sm_100a)"; }
uint64_t hb_kernel_launches(void) { return g_launches.load(); }

// ---------------------------------------------------------------------------------------------
// File-level parse without the per-sample cache: what the converter (vcf_to_h5 mirror) drives.
// ---------------------------------------------------------------------------------------------
int hb_parse_file(const char *in_vcf, const char *region, int want_gt, int device, hb_parse **out) {
    if (!in_vcf || !out) return fail(HB_ERR_ARG, "null argument");
    std::vector<std::string> samples;
    TRY(parse_file_common(in_vcf, region, want_gt != 0, device, out, samples));
    (*out)->samples = samples;
    return HB_OK;
}

int hb_parse_file_subset(const char *in_vcf, const char *region, const char *const *names, uint32_t n, int device, hb_parse **out) {
    if (!in_vcf || !out) return fail(HB_ERR_ARG, "null argument");
    std::vector<std::string> samples;
    const Subset ss{names, n};
    TRY(parse_file_common(in_vcf, region, true, device, out, samples, &ss));
    (*out)->samples = samples;
    return HB_OK;
}

// header of the BGZF bytes of a .vcf.gz: sample count, decompressed size, offset of the first record in it
int hb_bgzf_vcf_info(const uint8_t *bgzf, uint64_t nbytes, uint32_t *n_samples, uint64_t *text_bytes, uint64_t *body_offset) {
    if (!bgzf) return fail(HB_ERR_ARG, "null argument");
    BgzfFile bz;
    if (!index_bgzf(bgzf, nbytes, bz)) return fail(HB_ERR_IO, "not a BGZF file");
    TRY(bgzf_header(bgzf, bz));
    if (bz.ft.bcf) return fail(HB_ERR_ARG, kBcfNoStream);
    if (n_samples) *n_samples = (uint32_t)bz.ft.samples.size();
    if (text_bytes) *text_bytes = bz.total;
    if (body_offset) *body_offset = bz.ft.body;
    return HB_OK;
}

// BGZF bytes in host memory -> results in host memory, streamed: slabs of whole BGZF members cross PCIe compressed,
// are inflated on the GPU behind the unfinished last line of the slab before, parsed up to their own last newline and
// fetched -- H2D + inflate of slab k + 1 and the D2H of slab k - 1 run while slab k is parsed.
// cols: the sample subset of the slab parses (empty = every sample); the sink gets planes of the subset's width
static int stream_bgzf(const char *entry, const uint8_t *bgzf, uint64_t nbytes, const char *region, int want_gt, int device,
                       uint64_t slab_bytes, SlabSink &sink, uint64_t *n_records, uint32_t *n_slabs,
                       const std::vector<uint32_t> &cols = {}) {
    if (!bgzf || !n_records) return fail(HB_ERR_ARG, "null argument");
    *n_records = 0;
    if (n_slabs) *n_slabs = 0;
    const double t_begin = now_ms();
    double t_wait = 0, t_parse = 0, t_enq = 0;
    BgzfFile bz;
    if (!index_bgzf(bgzf, nbytes, bz)) return fail(HB_ERR_IO, "not a BGZF file");
    TRY(bgzf_header(bgzf, bz));
    const std::vector<uint64_t> &coff = bz.coff, &ooff = bz.ooff;
    const std::vector<uint32_t> &clen = bz.clen, &olen = bz.olen;
    const FileText &ft = bz.ft;
    if (ft.bcf) return fail(HB_ERR_ARG, kBcfNoStream);
    const double t_index = now_ms() - t_begin;
    const hb_parse_opts opts = opts_for(ft, region, want_gt != 0, device);
    TRY(ensure_device(device));
    {
        hb_parse_opts planes = opts;
        std::vector<std::string> names;
        for (uint32_t c : cols) names.push_back(ft.samples[c]);
        if (!cols.empty()) planes.n_samples = (uint32_t)cols.size();
        TRY(sink.begin(planes, cols.empty() ? ft.samples : names, bz.total));
    }
    if (bz.total <= ft.body) return HB_OK;
    if (slab_bytes == 0) slab_bytes = 1ull << 30;
    // slabs of whole members, about slab_bytes of text each
    struct Slab { size_t m0, m1; uint64_t text; uint64_t comp0, comp; };
    std::vector<Slab> slabs;
    uint64_t text_cap = 0, comp_cap = 0;
    size_t n_cap = 0;
    for (size_t m = 0; m < coff.size();) {
        Slab sl{m, m, 0, coff[m], 0};
        while (sl.m1 < coff.size() && (sl.text == 0 || sl.text + olen[sl.m1] <= slab_bytes)) { sl.text += olen[sl.m1]; ++sl.m1; }
        sl.comp = coff[sl.m1 - 1] + clen[sl.m1 - 1] + 8 - sl.comp0;   // through the last member's trailer (CRC32, ISIZE)
        if (sl.text) slabs.push_back(sl);
        text_cap = std::max(text_cap, sl.text); comp_cap = std::max(comp_cap, sl.comp); n_cap = std::max(n_cap, sl.m1 - sl.m0);
        m = sl.m1;
    }
    if (slabs.empty()) return HB_OK;
    if (ft.body >= slabs[0].text) return fail(HB_ERR_ARG, "the VCF header is longer than a slab: raise slab_bytes");
    const uint64_t carry_cap = std::min<uint64_t>((text_cap + 15) & ~15ull, 256ull << 20);   // longest unfinished line carried over
    StreamSlots *ss = nullptr;
    TRY(open_slots(g_bgzf_slots, opts, cols, std::min<size_t>(2, slabs.size()), text_cap, carry_cap, comp_cap, (uint32_t)n_cap, &ss));
    StreamSlot *slot = ss->slot;
    const uint64_t carry_base = ss->carry_cap;                 // offset of a slab's text when nothing is carried
    int rc = HB_OK;
    cudaError_t e = cudaSuccess;
    // H2D + inflate of slab k behind a carry of carry_len bytes, then the search for its last newline
    auto enqueue = [&](size_t k, uint64_t carry_len) -> int {
        StreamSlot &s = slot[k & 1];
        const Slab &sl = slabs[k];
        const uint64_t skip = k == 0 ? ft.body : 0;            // slab 0 starts with the header
        s.x = carry_base + (k == 0 ? (16 - ft.body % 16) % 16 : carry_len % 16);   // the parse starts on a 16-byte boundary
        s.begin = s.x + skip - carry_len;
        s.end = s.x + sl.text;
        const uint32_t n = (uint32_t)(sl.m1 - sl.m0);
        const uint64_t nc = ss->n_cap + (ss->n_cap & 1);        // keeps the 8-byte tables aligned behind the status words
        uint64_t *pc = reinterpret_cast<uint64_t *>(s.h_pin + 1 + nc / 2), *po = pc + ss->n_cap;
        uint32_t *pcl = reinterpret_cast<uint32_t *>(po + ss->n_cap), *pol = pcl + ss->n_cap;
        for (uint32_t i = 0; i < n; ++i) {
            pc[i] = coff[sl.m0 + i] - sl.comp0; po[i] = s.x + (ooff[sl.m0 + i] - ooff[sl.m0]);
            pcl[i] = clen[sl.m0 + i]; pol[i] = olen[sl.m0 + i];
        }
        int r = inflate_bgzf_enqueue(s.sc, bgzf + sl.comp0, sl.comp, pc, pcl, po, pol, n, s.buf, s.compute);
        if (r != HB_OK) return r;
        if (k + 1 == slabs.size()) {                           // a file that does not end with a newline
            cudaError_t ee = cudaMemsetAsync(s.buf + s.end, '\n', 1, s.compute);
            if (ee != cudaSuccess) return fail(HB_ERR_CUDA, "cudaMemsetAsync failed");
        }
        launch_last_newline(s.buf, s.x + skip, s.end, s.sc.d_last_nl, s.compute);
        cudaError_t ee = cudaMemcpyAsync(s.h_pin, s.sc.d_last_nl, 8, cudaMemcpyDeviceToHost, s.compute);
        if (ee == cudaSuccess) ee = cudaMemcpyAsync(s.h_pin + 1, s.sc.d_status, 4ull * n, cudaMemcpyDeviceToHost, s.compute);
        if (ee != cudaSuccess) return fail_cuda(ee);
        return HB_OK;
    };
    const double t_setup = now_ms() - t_begin - t_index;
    rc = enqueue(0, 0);
    uint64_t R = 0;
    for (size_t k = 0; k < slabs.size() && rc == HB_OK && e == cudaSuccess; ++k) {
        StreamSlot &s = slot[k & 1];
        { const double t0 = now_ms();
        e = cudaStreamSynchronize(s.compute);                  // slab k is inflated, its last newline is known
        t_wait += now_ms() - t0; }
        if (e != cudaSuccess) break;
        const unsigned long long last_nl = s.h_pin[0];
        const int *status = reinterpret_cast<const int *>(s.h_pin + 1);
        for (size_t i = 0; i < slabs[k].m1 - slabs[k].m0; ++i) {
            if (status[i] == kInflateCrcMismatch) { rc = fail(HB_ERR_IO, bgzf_crc_message(bgzf, coff[slabs[k].m0 + i])); break; }
            if (status[i]) { rc = fail(HB_ERR_IO, "BGZF inflate failed (member " + std::to_string(slabs[k].m0 + i) + ", code " + std::to_string(status[i]) + ")"); break; }
        }
        if (rc != HB_OK) break;
        const bool last = k + 1 == slabs.size();
        uint64_t parse_end;                                     // one past the last newline of the slab's text
        if (last_nl == ~0ull) {
            if (!last) { rc = fail(HB_ERR_ARG, "a line is longer than a slab: raise slab_bytes"); break; }
            parse_end = s.begin;
        } else parse_end = last_nl + 1;
        if (last && parse_end < s.end) parse_end = s.end + 1;   // no newline at the end of the file: the one appended ends the last line
        const uint64_t carry_len = last ? 0 : s.end - parse_end;
        if (carry_len > carry_base) { rc = fail(HB_ERR_ARG, "a line is longer than the carry buffer: raise slab_bytes"); break; }
        if (!last) {
            StreamSlot &nx = slot[(k + 1) & 1];
            // the unfinished line goes in front of the next slab's text (that buffer's last parse has returned)
            const uint64_t nx_x = carry_base + carry_len % 16;
            if (carry_len) e = cudaMemcpyAsync(nx.buf + nx_x - carry_len, s.buf + parse_end, carry_len, cudaMemcpyDeviceToDevice, s.compute);
            if (e != cudaSuccess) break;
        }
        e = cudaMemsetAsync(s.buf + parse_end, 0, 256, s.compute);
        if (e != cudaSuccess) break;
        if (!last) { const double t0 = now_ms(); rc = enqueue(k + 1, carry_len); t_enq += now_ms() - t0; if (rc != HB_OK) break; }
        const double t0 = now_ms();
        rc = parse_slab(s, s.begin, parse_end > s.begin ? parse_end - s.begin : 0, sink, R, e);
        t_parse += now_ms() - t0;
    }
    const double t_loop_end = now_ms();
    rc = close_slots(g_bgzf_slots, ss, rc, e);
    if (getenv("HB_TRACE"))
        fprintf(stderr, "[%s] %zu slabs: index+header %.1f ms, setup %.1f ms, waits for inflate %.1f ms, enqueue %.1f ms, "
                        "parse + deliver %.1f ms, loop %.1f ms, D2H tail + release %.1f ms\n", entry, slabs.size(), t_index, t_setup,
                t_wait, t_enq, t_parse, t_loop_end - t_begin - t_index - t_setup, now_ms() - t_loop_end);
    if (rc != HB_OK) return rc;
    *n_records = R;
    if (n_slabs) *n_slabs = (uint32_t)slabs.size();
    return HB_OK;
}

namespace {
// The rows of every slab appended to ONE resident parse: genotype planes and site columns grow in HBM (2.5 bytes per call),
// the text never holds more than two slabs.  The result is the handle a whole-file parse would have given (without its
// text): same rows, so hb_compress_records cuts it into the same HDF5 chunks -- chunk boundaries do not see slab boundaries.
struct ResidentSink : SlabSink {
    ParsePtr big{nullptr, hb_parse_free};
    uint64_t total_text = 0, text_seen = 0, cap = 0;
    std::vector<uint32_t> ploidy, badgt;       // per-sample error counts, summed on the host and put on the device at the end
    int begin(const hb_parse_opts &o, const std::vector<std::string> &samples, uint64_t total) override {
        ploidy.assign(std::max<uint32_t>(o.n_samples, 1), 0); badgt.assign(std::max<uint32_t>(o.n_samples, 1), 0);
        ploidy_err = ploidy.data(); badgt_err = badgt.data();
        TRY(SlabSink::begin(o, samples, total));
        total_text = total;
        hb_parse_opts oo = o;
        oo.stream = nullptr;
        int rc;
        big = new_parse(&oo, rc);
        if (!big) return rc;
        big->samples = samples;
        big->text_released = true;             // there is no text to re-run on
        big->runs_valid = true;                // its CHROM runs are put together from the slabs'
        return HB_OK;
    }
    int grow(uint64_t need, cudaStream_t st, uint64_t R) {          // capacity for `need` rows, the R rows present are kept
        const uint32_t S = big->n_samples;
        const uint64_t stride = (need + 127) / 128 * 128;
        struct { SiteRows rows; int8_t *gt[2]; uint32_t *bits; uint64_t gt_stride; } old =
            {big->rows, {big->d_gt[0], big->d_gt[1]}, big->d_bits, big->gt_stride};
        cudaDeviceSynchronize();                   // (rare) copies of the other slot into the old planes are done
        big->rows = SiteRows();                    // only the columns of the stored record are kept
        big->d_gt[0] = big->d_gt[1] = nullptr; big->d_bits = nullptr;
        SiteRows &r = big->rows;
        int rc = dev_alloc(&r.start, stride);
        if (rc == HB_OK) rc = dev_alloc(&r.stop, stride);
        if (rc == HB_OK) rc = dev_alloc(&r.ref, stride);
        if (rc == HB_OK) rc = dev_alloc(&r.alt, stride);
        if (rc == HB_OK) rc = dev_alloc(&r.chrom5, stride);
        if (rc == HB_OK && big->want_gt && S) {
            rc = dev_alloc(&big->d_gt[0], stride * S);
            if (rc == HB_OK) rc = dev_alloc(&big->d_gt[1], stride * S);
            if (rc == HB_OK) rc = dev_alloc(&big->d_bits, stride / 128 * kBitGroupWords * S);
        }
        cudaError_t e = cudaSuccess;
        if (rc == HB_OK && R) {
            e = cudaMemcpyAsync(r.start, old.rows.start, R * 4, cudaMemcpyDeviceToDevice, st);
            if (e == cudaSuccess) e = cudaMemcpyAsync(r.stop, old.rows.stop, R * 4, cudaMemcpyDeviceToDevice, st);
            if (e == cudaSuccess) e = cudaMemcpyAsync(r.ref, old.rows.ref, R, cudaMemcpyDeviceToDevice, st);
            if (e == cudaSuccess) e = cudaMemcpyAsync(r.alt, old.rows.alt, R, cudaMemcpyDeviceToDevice, st);
            if (e == cudaSuccess) e = cudaMemcpyAsync(r.chrom5, old.rows.chrom5, R * 8, cudaMemcpyDeviceToDevice, st);
            if (e == cudaSuccess && old.gt[0]) e = cudaMemcpy2DAsync(big->d_gt[0], stride, old.gt[0], old.gt_stride, R, S, cudaMemcpyDeviceToDevice, st);
            if (e == cudaSuccess && old.gt[1]) e = cudaMemcpy2DAsync(big->d_gt[1], stride, old.gt[1], old.gt_stride, R, S, cudaMemcpyDeviceToDevice, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        }
        free_rows(old.rows); free_dev(old.gt[0]); free_dev(old.gt[1]); free_dev(old.bits);
        if (rc != HB_OK) return rc;
        if (e != cudaSuccess) return fail_cuda(e);
        big->gt_stride = stride; big->gt_bytes = stride * S; big->bits_stride = stride / 128 * kBitGroupWords; r.cap = stride;
        cap = stride;
        return HB_OK;
    }
    int deliver(StreamSlot &s, uint64_t R, uint64_t n, uint64_t slab_text, cudaError_t &e) override {
        text_seen += slab_text;
        if (R + n > cap) {
            // rows per byte seen so far, extrapolated to the whole file (+ 3 %): the planes are allocated once for most files
            const double per = (double)(R + n) / (double)std::max<uint64_t>(1, text_seen);
            uint64_t need = (uint64_t)(per * (double)total_text * 1.03) + 4096;
            need = std::max(need, R + n);
            e = cudaStreamSynchronize(s.d2h);
            if (e != cudaSuccess) return HB_OK;
            TRY(grow(need, s.d2h, R));
        }
        const uint32_t S = big->n_samples;
        if (big->want_gt && S && s.p->d_gt[0]) {
            e = cudaMemcpy2DAsync(big->d_gt[0] + R, big->gt_stride, s.p->d_gt[0], s.p->gt_stride, n, S, cudaMemcpyDeviceToDevice, s.d2h);
            if (e == cudaSuccess) e = cudaMemcpy2DAsync(big->d_gt[1] + R, big->gt_stride, s.p->d_gt[1], s.p->gt_stride, n, S, cudaMemcpyDeviceToDevice, s.d2h);
        }
        const SiteRows &to = big->rows, &from = s.p->rows;
        if (e == cudaSuccess) e = cudaMemcpyAsync(to.start + R, from.start, n * 4, cudaMemcpyDeviceToDevice, s.d2h);
        if (e == cudaSuccess) e = cudaMemcpyAsync(to.stop + R, from.stop, n * 4, cudaMemcpyDeviceToDevice, s.d2h);
        if (e == cudaSuccess) e = cudaMemcpyAsync(to.ref + R, from.ref, n, cudaMemcpyDeviceToDevice, s.d2h);
        if (e == cudaSuccess) e = cudaMemcpyAsync(to.alt + R, from.alt, n, cudaMemcpyDeviceToDevice, s.d2h);
        if (e == cudaSuccess) e = cudaMemcpyAsync(to.chrom5 + R, from.chrom5, n * 8, cudaMemcpyDeviceToDevice, s.d2h);
        // CHROM runs of the slab continue the file's
        TRY(ensure_runs(s.p));
        for (size_t i = 0; i < s.p->run_rows.size(); ++i) {
            if (!big->run_names.empty() && big->run_names.back() == s.p->run_names[i]) continue;
            big->run_rows.push_back(R + s.p->run_rows[i]);
            big->run_names.push_back(s.p->run_names[i]);
        }
        big->n_lines += s.p->n_lines;
        big->h_st.n_nonuniform += s.p->h_st.n_nonuniform; big->h_st.n_bad_gt += s.p->h_st.n_bad_gt;
        big->h_st.n_nogt += s.p->h_st.n_nogt;
        big->index_used = s.p->index_used;
        big->walker_fallbacks += s.p->walker_fallbacks;
        big->ms_tok += s.p->ms_tok; big->ms_sites += s.p->ms_sites; big->ms_decode += s.p->ms_decode;
        return HB_OK;
    }
};
}  // namespace

int hb_parse_stream_bgzf_host(const uint8_t *bgzf, uint64_t nbytes, const char *region, int want_gt, int device,
                              uint64_t slab_bytes, int8_t *gt0, int8_t *gt1, uint64_t out_stride, uint32_t *start,
                              uint32_t *stop, char *ref, char *alt, uint32_t *ploidy_err, uint32_t *badgt_err,
                              uint64_t *n_records, uint32_t *n_slabs) {
    HostSink sink(gt0, gt1, out_stride, start, stop, ref, alt, ploidy_err, badgt_err);
    return stream_bgzf("hb_parse_stream_bgzf_host", bgzf, nbytes, region, want_gt, device, slab_bytes, sink, n_records, n_slabs);
}

int hb_parse_stream_bgzf_resident(const uint8_t *bgzf, uint64_t nbytes, const char *region, int want_gt, int device,
                                  uint64_t slab_bytes, hb_parse **out, uint32_t *n_slabs) {
    return stream_resident(bgzf, nbytes, region, want_gt, device, slab_bytes, out, n_slabs, {});
}

namespace {
int stream_resident(const uint8_t *bgzf, uint64_t nbytes, const char *region, int want_gt, int device, uint64_t slab_bytes,
                    hb_parse **out, uint32_t *n_slabs, const std::vector<uint32_t> &cols) {
    if (!out) return fail(HB_ERR_ARG, "null argument");
    *out = nullptr;
    ResidentSink sink;
    uint64_t n = 0;
    TRY(stream_bgzf("hb_parse_stream_bgzf_resident", bgzf, nbytes, region, want_gt, device, slab_bytes, sink, &n, n_slabs, cols));
    hb_parse *p = sink.big.get();
    if (!p) return fail(HB_ERR_IO, "empty input");
    const uint32_t S = p->n_samples;
    cudaError_t e = cudaSuccess;
    if (want_gt && S) {
        int rc = dev_alloc(&p->d_ploidy, S);
        if (rc == HB_OK) rc = dev_alloc(&p->d_badgt, S);
        if (rc != HB_OK) return rc;
        e = cudaMemcpy(p->d_ploidy, sink.ploidy.data(), 4ull * S, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMemcpy(p->d_badgt, sink.badgt.data(), 4ull * S, cudaMemcpyHostToDevice);
        if (e == cudaSuccess && n && p->d_gt[0]) {                 // the allele bit planes kernel 4b reads, from the assembled byte planes
            Launch L{p->stream, p->sm_count};
            launch_bits_from_planes(p->d_gt[0], p->d_gt[1], p->gt_stride, n, S, p->d_bits, p->bits_stride, L);
            e = cudaStreamSynchronize(p->stream);
        }
    }
    if (e != cudaSuccess) return fail_cuda(e);
    p->h_st.n_records = n;
    p->compressed_bytes = nbytes;
    *out = sink.big.release();
    return HB_OK;
}
}  // namespace

// Host utility (tests, bench): text -> BGZF with stock zlib on all host threads -- what `bgzip -@` does.
// Not part of the product path (the path READS BGZF); it exists so that BGZF inputs of bench size can be made
// here without htslib.  out == NULL: *len is set to a sufficient capacity.
int hb_bgzf_compress_host(const uint8_t *text, uint64_t nbytes, int level, uint8_t *out, uint64_t cap, uint64_t *len) {
    if (!len || (nbytes && !text)) return fail(HB_ERR_ARG, "null argument");
    const uint64_t blk = 0xff00;
    const uint64_t n_blocks = (nbytes + blk - 1) / blk;
    const uint64_t worst = 18 + 8 + blk + blk / 1000 + 64;
    if (!out) { *len = n_blocks * worst + 28; return HB_OK; }
    if (cap < n_blocks * worst + 28) return fail(HB_ERR_ARG, "buffer too small");
    std::vector<uint32_t> sizes(n_blocks);
    std::atomic<uint64_t> next{0};
    std::atomic<int> bad{0};
    auto work = [&]() {
        for (;;) {
            const uint64_t i = next.fetch_add(1);
            if (i >= n_blocks) break;
            const uint8_t *src = text + i * blk;
            const uint32_t n = (uint32_t)std::min<uint64_t>(blk, nbytes - i * blk);
            uint8_t *dst = out + i * worst;
            z_stream zs;
            memset(&zs, 0, sizeof zs);
            if (deflateInit2(&zs, level, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) { bad = 1; break; }
            zs.next_in = const_cast<Bytef *>(src); zs.avail_in = n;
            zs.next_out = dst + 18; zs.avail_out = (uInt)(worst - 26);
            const int zr = deflate(&zs, Z_FINISH);
            const uint32_t clen = (uint32_t)zs.total_out;
            deflateEnd(&zs);
            if (zr != Z_STREAM_END || clen + 26 > 65536) { bad = 1; break; }
            const uint8_t hdr[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
            memcpy(dst, hdr, 16);
            const uint32_t bs = clen + 25;
            dst[16] = (uint8_t)bs; dst[17] = (uint8_t)(bs >> 8);
            const uint32_t crc = (uint32_t)crc32(crc32(0L, Z_NULL, 0), src, n);
            uint8_t *tr = dst + 18 + clen;
            for (int k = 0; k < 4; ++k) { tr[k] = (uint8_t)(crc >> (8 * k)); tr[4 + k] = (uint8_t)(n >> (8 * k)); }
            sizes[i] = clen + 26;
        }
    };
    unsigned nt = std::max(1u, std::min(std::thread::hardware_concurrency(), 64u));
    std::vector<std::thread> th;
    for (unsigned t = 1; t < nt; ++t) th.emplace_back(work);
    work();
    for (auto &t : th) t.join();
    if (bad) return fail(HB_ERR_IO, "deflate failed");
    uint64_t o = 0;
    for (uint64_t i = 0; i < n_blocks; ++i) { memmove(out + o, out + i * worst, sizes[i]); o += sizes[i]; }
    const uint8_t eof[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    memcpy(out + o, eof, 28);
    *len = o + 28;
    return HB_OK;
}

int hb_parse_vcf_bytes(const uint8_t *data, uint64_t nbytes, const char *region, int want_gt, int device, hb_parse **out) {
    if (!data || !out) return fail(HB_ERR_ARG, "null argument");
    std::vector<std::string> samples;
    std::vector<uint8_t> none;
    TRY(parse_bytes_common(none, data, nbytes, region, want_gt != 0, device, out, samples, nullptr));
    (*out)->samples = samples;
    return HB_OK;
}

int hb_parse_samples(hb_parse *p, uint32_t *n, char *names, uint64_t cap, uint64_t *len) {
    if (!p) return fail(HB_ERR_ARG, "null handle");
    if (n) *n = (uint32_t)p->samples.size();
    uint64_t used = 0;
    for (const std::string &s : p->samples) {
        if (names && used + s.size() + 1 <= cap) memcpy(names + used, s.c_str(), s.size() + 1);
        used += s.size() + 1;
    }
    if (len) *len = used;
    return HB_OK;
}

namespace {
// The header of a .vcf, .vcf.gz (BGZF or plain gzip) or .bcf from its leading bytes only.  BGZF: the leading members, as a
// region query reads them.  Anything else: read in rounds that double the bytes read, inflated as a stream when it is gzip,
// until the #CHROM line (or the BCF header text) is complete.
int leading_header(const ByteSource &src, FileText &ft) {
    {
        uint64_t head_read = 0;
        std::string why;
        if (leading_bgzf_header(src, ft, head_read, why)) return HB_OK;   // (else the stream below gives the reason)
    }
    std::vector<uint8_t> buf, text;
    const uint8_t *h = src.get(0, std::min<uint64_t>(src.size, 2), buf);
    const bool gz = h && src.size >= 2 && h[0] == 0x1f && h[1] == 0x8b;
    struct Z {
        z_stream zs;
        bool on = false;
        ~Z() { if (on) inflateEnd(&zs); }
    } z;
    if (gz) {
        memset(&z.zs, 0, sizeof z.zs);
        if (inflateInit2(&z.zs, 15 + 32) != Z_OK) return fail(HB_ERR_IO, "inflateInit2 failed");
        z.on = true;
    }
    for (uint64_t off = 0, chunk = 1 << 16;; chunk *= 2) {
        const uint64_t n = std::min<uint64_t>(chunk, src.size - off);
        const uint8_t *b = src.get(off, n, buf);
        if (!b) return fail(HB_ERR_IO, "read error");
        off += n;
        const bool eof = off == src.size;
        if (!gz) text.insert(text.end(), b, b + n);
        else {
            z.zs.next_in = const_cast<Bytef *>(b);
            z.zs.avail_in = (uInt)n;
            while (z.zs.avail_in) {
                const size_t at = text.size();
                text.resize(at + (1 << 16));
                z.zs.next_out = text.data() + at;
                z.zs.avail_out = 1 << 16;
                const int zr = inflate(&z.zs, Z_NO_FLUSH);
                text.resize(at + (1 << 16) - z.zs.avail_out);
                if (zr == Z_STREAM_END) { if (inflateReset(&z.zs) != Z_OK) return fail(HB_ERR_IO, "gzip member reset failed"); }
                else if (zr != Z_OK) return fail(HB_ERR_IO, "gzip inflate failed");
            }
        }
        if (is_bcf(text.data(), text.size())) {
            bool complete = false;
            TRY(bcf_header(text.data(), text.size(), ft, complete));
            if (complete) return HB_OK;
            if (eof) return fail(HB_ERR_FORMAT, "BCF header is truncated");
        } else if (parse_header(text.data(), text.size(), eof, ft)) {
            return HB_OK;
        } else if (eof) {
            return fail(HB_ERR_HEADER, "no #CHROM header line");
        }
    }
}
}  // namespace

int hb_file_samples(const char *path, uint32_t *n, char *names, uint64_t cap, uint64_t *len) {
    if (!path) return fail(HB_ERR_ARG, "null argument");
    const int fd = open(path, O_RDONLY);
    struct stat st;
    if (fd < 0 || fstat(fd, &st) != 0) {
        if (fd >= 0) close(fd);
        return fail(HB_ERR_IO, std::string("cannot open ") + path);
    }
    FileText ft;
    const int rc = leading_header(ByteSource{nullptr, fd, (uint64_t)st.st_size}, ft);
    close(fd);
    TRY(rc);
    if (n) *n = (uint32_t)ft.samples.size();
    uint64_t used = 0;
    for (const std::string &s : ft.samples) {
        if (names && used + s.size() + 1 <= cap) memcpy(names + used, s.c_str(), s.size() + 1);
        used += s.size() + 1;
    }
    if (len) *len = used;
    return HB_OK;
}

// ---- region queries through a .tbi / .csi index
void hb_set_use_index(int on) { g_use_index.store(on ? 1 : 0); }
int hb_get_use_index(void) { return g_use_index.load(); }

static int vcf_bytes_indexed(const uint8_t *data, uint64_t nbytes, const uint8_t *index, uint64_t index_n, const char *region,
                             int want_gt, int device, hb_parse **out, const Subset *ss) {
    if (!data || !out || (index_n && !index)) return fail(HB_ERR_ARG, "null argument");
    std::vector<std::string> samples;
    std::string why;
    bool used = false;
    if (!region || !*region) why = "the region is empty";
    else if (!g_use_index.load()) why = "hb_set_use_index(0)";
    else if (!index_n) why = "no index given";
    else TRY(parse_indexed(ByteSource{data, -1, nbytes}, index, index_n, region, want_gt != 0, device, out, samples, used, why, ss));
    if (!used) {
        index_not_used(why);
        std::vector<uint8_t> none;
        TRY(parse_bytes_common(none, data, nbytes, region, want_gt != 0, device, out, samples, ss));
    }
    (*out)->samples = samples;
    return HB_OK;
}

int hb_parse_vcf_bytes_indexed(const uint8_t *data, uint64_t nbytes, const uint8_t *index, uint64_t index_n, const char *region,
                               int want_gt, int device, hb_parse **out) {
    return vcf_bytes_indexed(data, nbytes, index, index_n, region, want_gt, device, out, nullptr);
}

int hb_parse_vcf_bytes_subset(const uint8_t *data, uint64_t nbytes, const uint8_t *index, uint64_t index_n, const char *region,
                              const char *const *names, uint32_t n, int device, hb_parse **out) {
    const Subset ss{names, n};
    return vcf_bytes_indexed(data, nbytes, index, index ? index_n : 0, region, 1, device, out, &ss);
}

int hb_parse_index_info(const hb_parse *p, int *used, uint64_t *compressed_bytes_read, uint64_t *n_chunks) {
    if (!p) return fail(HB_ERR_ARG, "null handle");
    if (used) *used = p->idx_used;
    if (compressed_bytes_read) *compressed_bytes_read = p->idx_bytes_read;
    if (n_chunks) *n_chunks = p->idx_chunks;
    return HB_OK;
}

// ---- building an index (kernel 7, hb_index.cu): kernel 0 inflates, the newline tokenizer or the BCF locator finds every
// record through a parse without a region or genotypes, then kernels 7a / 7b and the host assembly
int hb_index_bgzf(const uint8_t *data, uint64_t n, int fmt, int min_shift, int device, uint8_t *out, uint64_t cap, uint64_t *len) {
    if (!data || !len) return fail(HB_ERR_ARG, "null argument");
    if (fmt != HB_INDEX_TBI && fmt != HB_INDEX_CSI) return fail(HB_ERR_ARG, "fmt is HB_INDEX_TBI or HB_INDEX_CSI");
    if (fmt == HB_INDEX_CSI && (min_shift < 1 || min_shift > 30)) return fail(HB_ERR_ARG, "min_shift must be 1..30");
    const bool trace = getenv("HB_TRACE") != nullptr;
    const double t0 = now_ms();
    BgzfFile bz;
    std::vector<uint64_t> boff;
    if (n < 28 || data[0] != 0x1f || data[1] != 0x8b || !bgzf_index(data, n, bz.coff, bz.clen, bz.ooff, bz.olen, bz.total, &boff) ||
        bz.total == 0)
        return fail(HB_ERR_ARG, "an index needs BGZF input (bgzip / bcftools -Ob), not plain gzip or uncompressed bytes");
    TRY(bgzf_header(data, bz));
    const FileText &ft = bz.ft;
    if (ft.bcf && fmt == HB_INDEX_TBI) return fail(HB_ERR_ARG, "a BCF is indexed with CSI only");
    TRY(ensure_device(device));
    uint64_t slab;
    if (bz.total > text_limit(slab)) return fail(HB_ERR_ARG, "the text is above the text limit: slab-wise indexing is not supported");
    hb_parse *raw = nullptr;
    std::vector<std::string> samples;
    std::vector<uint8_t> none;
    TRY(parse_bytes_common(none, data, n, "", false, device, &raw, samples, nullptr));
    ParsePtr p(raw, hb_parse_free);
    const double t1 = now_ms();
    IndexJob j;
    j.d_text = p->d_text;
    j.text_base = ft.body;
    j.total = bz.total;
    j.n_rec = p->n_lines;
    j.bcf = ft.bcf;
    if (ft.bcf) {
        j.d_rec_off = p->bcf->d_rec_off;
        j.n_contigs = (uint32_t)ft.contigs.size();
    } else {
        if (p->index_used != 1) return fail(HB_ERR_ARG, "internal: the index needs the newline tokenizer's line index");
        j.li = LineIndex{p->d_nl_after, p->d_cbase, p->n_cta, p->stage_cap};
    }
    j.ooff = bz.ooff; j.olen = bz.olen; j.boff = boff;
    for (size_t i = 0; i < bz.coff.size(); ++i) j.bend.push_back(bz.coff[i] + bz.clen[i] + 8);
    j.csi = fmt == HB_INDEX_CSI;
    if (!j.csi) { j.min_shift = 14; j.n_lvls = 5; }                            // tabix -p vcf
    else if (!ft.bcf) { j.min_shift = min_shift; j.n_lvls = (31 - min_shift + 2) / 3; }   // tabix -C: TBX_MAX_SHIFT 31
    else {                                                                   // bcftools index: the longest contig + 256
        uint64_t longest = 0;
        for (uint64_t l : ft.contig_len) longest = std::max(longest, l);
        longest = (longest ? longest : (1ull << 31) - 1) + 256;
        j.min_shift = min_shift; j.n_lvls = 0;
        for (uint64_t s = 1ull << min_shift; longest > s; s <<= 3) ++j.n_lvls;
    }
    j.stream = p->stream;
    std::vector<uint8_t> idx;
    IndexTimes tm;
    TRY(build_index(j, idx, &tm));
    uint64_t need = 0;
    TRY(hb_bgzf_compress_host(idx.data(), idx.size(), 6, nullptr, 0, &need));
    std::vector<uint8_t> z(need);
    TRY(hb_bgzf_compress_host(idx.data(), idx.size(), 6, z.data(), z.size(), &need));
    *len = need;
    if (trace)
        fprintf(stderr, "[hb_index_bgzf] %llu records: parse (H2D + inflate + locate) %.1f ms, kernel 7a %.3f ms, 7b %.3f ms, "
                        "host assembly %.1f ms, total %.1f ms\n", (unsigned long long)j.n_rec, t1 - t0, tm.ms_keys, tm.ms_chunks,
                tm.ms_host, now_ms() - t0);
    if (!out) return HB_OK;
    if (cap < need) return fail(HB_ERR_ARG, "buffer too small: " + std::to_string(need) + " bytes needed");
    memcpy(out, z.data(), need);
    return HB_OK;
}

int hb_index_file(const char *path, int fmt, int min_shift, int device, const char *out_path) {
    if (!path) return fail(HB_ERR_ARG, "null argument");
    std::vector<uint8_t> raw;
    TRY(read_all(path, raw));
    uint64_t len = 0;
    TRY(hb_index_bgzf(raw.data(), raw.size(), fmt, min_shift, device, nullptr, 0, &len));
    std::vector<uint8_t> z(len);
    TRY(hb_index_bgzf(raw.data(), raw.size(), fmt, min_shift, device, z.data(), z.size(), &len));
    const std::string dst = out_path ? std::string(out_path) : std::string(path) + (fmt == HB_INDEX_TBI ? ".tbi" : ".csi");
    FILE *f = fopen(dst.c_str(), "wb");
    if (!f) return fail(HB_ERR_IO, "cannot write " + dst);
    const bool ok = fwrite(z.data(), 1, len, f) == len;
    if (fclose(f) != 0 || !ok) return fail(HB_ERR_IO, "cannot write " + dst);
    return HB_OK;
}
