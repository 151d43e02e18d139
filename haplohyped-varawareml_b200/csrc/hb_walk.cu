// hb_walk.cu -- kernel 1+2, index-free variant: locate the records of GT-only text by WALKING
// from record head to record head instead of reading every byte to find the newlines.
//
// Replaces the same reference code as hb_tokenize.cu + hb_sites.cu (BcfReader::getNextVariant,
// cpp/vcfpp.h:1455-1484, and the accessors behind cpp/parse_vcf.cpp:41-61) for the common shape of a
// cohort VCF: FORMAT == "GT" and every call 3 characters wide, so a record is
//     <head: 9 tab-terminated columns> { '\t' a sep b } x S '\n'
// and its end is at (9th tab) + 4*S.  A walker reads a head (~60 bytes), jumps 4*S bytes, checks
// that a newline is there, and is at the next head: ~2 % of the text is touched instead of 100 %.
//
// Nothing is assumed, everything is checked -- the result is exact or the caller falls back:
//   * the text is cut into byte ranges; a warp finds the first record start of each range by a
//     plain newline search (walk_sync_kernel); thread w then walks [start_w, start_{w+1}) and must
//     land EXACTLY on start_{w+1} (DevStatus::walk_broken otherwise);
//   * a jump is accepted only if the byte at (9th tab)+4*S is the newline; otherwise the walker
//     searches the newline byte by byte (records of any other shape stay exact, just slower);
//   * that no newline hides INSIDE a jumped-over span is proven by whoever reads the span: the GT
//     decoder validates every 4-byte group of the records it decodes (hb_gt.cu raises
//     DevStatus::index_invalid on a newline), and the spans nobody decodes (records dropped by
//     the SNP / region filter, or not plain-GT) are scanned by walk_verify_kernel.
// ONE pass over the heads (r02): a walker writes the rows it keeps into its own kWalkSlots slots of padded site arrays and
// counts them, one small prefix sum gives every walker its dense row base, and a compaction kernel moves the rows (54
// bytes each) to their dense places -- the second head-parsing pass of r01 (0.25 ms, instruction-bound at 14 warps per SM)
// became a 50 MB copy.
#include <algorithm>
#include <cstring>

#include "hb_common.cuh"
#include "hb_head.cuh"
#include "hb_internal.h"

namespace hb {

constexpr int WK_THREADS = 128;

struct WalkArgs {
    const uint8_t *text;
    uint64_t nbytes;
    uint32_t n_samples;
    uint64_t range_bytes;
    uint32_t n_walkers;
    RegionArg rg;
    int end_is_int;
    uint64_t *wstart;        // [n_walkers + 1] first record start at/after w * range_bytes; [n_walkers] = nbytes
    uint2 *wcount;           // [n_walkers] (lines, kept rows)
    uint64_t *wrow;          // [n_walkers] exclusive prefix sum of kept rows
    SiteOut out;             // dense rows (compaction) 
    SiteOut pad;             // [n_walkers * kWalkSlots] padded rows (walk)
    uint64_t *verify;        // spans (offset of their 9th tab) that the decoder will not validate
    uint64_t verify_cap;
    DevStatus *st;
};

__device__ __forceinline__ uint4 ld_chunk(const uint8_t *text, uint64_t off, uint64_t nbytes) {
    if (off >= nbytes) return make_uint4(0, 0, 0, 0);
    return __ldg(reinterpret_cast<const uint4 *>(text + off));
}

// 0x80 flags of the '\n' bytes of a 16-byte chunk, as a 16-bit mask (bit i = byte i)
__device__ __forceinline__ uint32_t nl_bits(const uint4 &v) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t m = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint32_t f = eq_mask(w[q], kNl4);      // 0x80 per matching byte
        // gather bits 7,15,23,31 -> 4 bits
        m |= (((f >> 7) & 1u) | ((f >> 14) & 2u) | ((f >> 21) & 4u) | ((f >> 28) & 8u)) << (4 * q);
    }
    return m;
}

// ------------------------------------------------------------------------------------------
// Pass 0: first record start of every range.  One warp per range, 2 KB per round trip.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) walk_sync_kernel(const WalkArgs a) {
    const int lane = threadIdx.x & 31;
    const uint32_t w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (w > a.n_walkers) return;
    if (w == a.n_walkers) { if (lane == 0) a.wstart[w] = a.nbytes; return; }
    if (w == 0) { if (lane == 0) a.wstart[0] = 0; return; }
    const uint64_t from = (uint64_t)w * a.range_bytes - 1;      // a newline here makes w*range_bytes a record start
    uint64_t found = a.nbytes;                                  // "none": the range holds no record start
    for (uint64_t base = from & ~15ull; base < a.nbytes; base += 2048) {
        uint4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = ld_chunk(a.text, base + (uint64_t)(u * 32 + lane) * 16, a.nbytes);
        uint64_t mine = ~0ull;
#pragma unroll
        for (int u = 3; u >= 0; --u) {
            const uint64_t o = base + (uint64_t)(u * 32 + lane) * 16;
            uint32_t m = nl_bits(v[u]);
            if (o < from) m &= ~((1u << (from - o)) - 1u);     // bytes before `from` do not count
            if (m) mine = o + (__ffs(m) - 1);
        }
        // warp minimum
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) {
            const uint64_t other = __shfl_xor_sync(0xffffffffu, mine, d);
            mine = other < mine ? other : mine;
        }
        if (mine != ~0ull) { found = mine < a.nbytes ? mine + 1 : a.nbytes; break; }
    }
    if (lane == 0) a.wstart[w] = found;
}

// ------------------------------------------------------------------------------------------
// A forward-only byte reader over global memory, 16-byte chunks held in registers, two chunks
// prefetched ahead so a head costs about one memory round trip.
// ------------------------------------------------------------------------------------------
struct ByteStream {
    const uint8_t *text;
    uint64_t nbytes, next_off;     // next_off: offset of the chunk after n2
    uint4 cur, n1, n2;
    uint32_t left;                 // unread bytes in cur

    __device__ __forceinline__ void init(const uint8_t *t, uint64_t nb, uint64_t q) {
        text = t; nbytes = nb;
        const uint64_t a0 = q & ~15ull;
        cur = ld_chunk(t, a0, nb);
        n1 = ld_chunk(t, a0 + 16, nb);
        n2 = ld_chunk(t, a0 + 32, nb);
        next_off = a0 + 48;
        const uint32_t k = (uint32_t)(q & 15ull);
        left = 16 - k;
        if (k & 8) { cur.x = cur.z; cur.y = cur.w; cur.z = 0; cur.w = 0; }
        if (k & 4) { cur.x = cur.y; cur.y = cur.z; cur.z = cur.w; cur.w = 0; }
        const uint32_t s = (k & 3) * 8;
        cur.x = __funnelshift_r(cur.x, cur.y, s);
        cur.y = __funnelshift_r(cur.y, cur.z, s);
        cur.z = __funnelshift_r(cur.z, cur.w, s);
        cur.w >>= s;
    }
    __device__ __forceinline__ uint8_t peek() const { return (uint8_t)(cur.x & 0xffu); }
    __device__ __forceinline__ void advance() {
        if (--left == 0) {
            cur = n1; n1 = n2;
            n2 = ld_chunk(text, next_off, nbytes);
            next_off += 16;
            left = 16;
        } else {
            cur.x = __funnelshift_r(cur.x, cur.y, 8);
            cur.y = __funnelshift_r(cur.y, cur.z, 8);
            cur.z = __funnelshift_r(cur.z, cur.w, 8);
            cur.w >>= 8;
        }
    }
};

// offset of the first '\n' at or after `from` (nbytes if none): one thread, 128 bytes per round trip
__device__ __noinline__ uint64_t find_newline(const uint8_t *text, uint64_t nbytes, uint64_t from) {
    for (uint64_t base = from & ~15ull; base < nbytes; base += 128) {
        uint4 v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = ld_chunk(text, base + 16 * u, nbytes);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const uint64_t o = base + 16 * u;
            uint32_t m = nl_bits(v[u]);
            if (o < from) m &= ~((1u << (from - o)) - 1u);
            if (m) { const uint64_t p = o + (__ffs(m) - 1); return p < nbytes ? p : nbytes; }
        }
    }
    return nbytes;
}

// ------------------------------------------------------------------------------------------
// Fast head.  The byte reader above costs ~45 instructions per byte of a head, and the walk is instruction-bound (80 M
// warp instructions at 14 warps per SM, r02u ncu).  When the 9th TAB of the record lies within 96 bytes of its start and
// no line end comes before it -- every ordinary record -- the window is loaded with seven 16-byte loads, the TAB and
// line-end bytes are found with word-wide compares, and the SAME state machine (HeadState::feed) is fed from a private
// shared-memory copy in a plain counted loop.  Anything else returns false before a byte is fed and takes the byte reader.
// ------------------------------------------------------------------------------------------
constexpr int kHeadWin = 112;                               // staged bytes per thread (7 chunks)
__device__ __forceinline__ uint32_t byte_bits(const uint4 &v, uint32_t c4) {       // bit i = (byte i == c)
    return pack_lsb4(eq_mask(v.x, c4) >> 7) | (pack_lsb4(eq_mask(v.y, c4) >> 7) << 4) |
           (pack_lsb4(eq_mask(v.z, c4) >> 7) << 8) | (pack_lsb4(eq_mask(v.w, c4) >> 7) << 12);
}
__device__ __forceinline__ bool fast_head(const uint8_t *__restrict__ text, uint64_t nbytes, uint64_t p, uint8_t *slot,
                                          HeadState &h, const RegionArg &rg) {
    const uint64_t base = p & ~15ull;
    if (base + kHeadWin > nbytes) return false;
    uint4 v[7];
#pragma unroll
    for (int i = 0; i < 7; ++i) v[i] = __ldg(reinterpret_cast<const uint4 *>(text + base + 16 * i));
    uint64_t tlo = 0, thi = 0, elo = 0, ehi = 0;              // TABs / line ends ('\n', '\r') of the window, bit i = byte i
#pragma unroll
    for (int i = 0; i < 7; ++i) {
        const uint64_t t = byte_bits(v[i], kTab4), e = byte_bits(v[i], kNl4) | byte_bits(v[i], 0x0D0D0D0Du);
        if (i < 4) { tlo |= t << (16 * i); elo |= e << (16 * i); }
        else { thi |= t << (16 * (i - 4)); ehi |= e << (16 * (i - 4)); }
    }
    const uint32_t k = (uint32_t)(p & 15ull);
    tlo &= ~0ull << k; elo &= ~0ull << k;
    uint32_t pos = 0;                                         // window offset of the 9th TAB
#pragma unroll 1
    for (int n = 0; n < 9; ++n) {
        if (tlo) { pos = (uint32_t)__ffsll((long long)tlo) - 1; tlo &= tlo - 1; }
        else if (thi) { pos = 64u + (uint32_t)__ffsll((long long)thi) - 1; thi &= thi - 1; }
        else return false;
    }
    if (pos < 64 ? (elo & ((1ull << pos) - 1ull)) != 0 : (elo != 0 || (ehi & ((1ull << (pos - 64)) - 1ull)) != 0)) return false;
#pragma unroll
    for (int i = 0; i < 7; ++i) reinterpret_cast<uint4 *>(slot)[i] = v[i];
    for (uint32_t i = k; i <= pos; ++i) h.feed(slot[i], base + i, rg);     // (returns true at the 9th TAB, the last byte fed)
    return true;
}

// ------------------------------------------------------------------------------------------
// The walk: lines and kept rows per walker are counted, kept rows written to the walker's padded slots.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(WK_THREADS) walk_kernel(const WalkArgs a) {
    __shared__ __align__(16) uint8_t heads[WK_THREADS][kHeadWin];
    const uint32_t w = blockIdx.x * WK_THREADS + threadIdx.x;
    if (w >= a.n_walkers) return;
    uint64_t p = a.wstart[w];
    const uint64_t end = a.wstart[w + 1];
    if (p >= end) { a.wcount[w] = make_uint2(0, 0); return; }
    uint32_t lines = 0, kept = 0;
    const uint64_t row0 = (uint64_t)w * kWalkSlots;
    const uint64_t span = 4ull * a.n_samples;
    ByteStream bs;
    bs.init(a.text, a.nbytes, p);
    while (p < end) {
        const uint64_t ls = p;
        HeadState h;
        h.init();
        uint64_t q = p, le = 0, nl = 0;
        bool ended = false, fast = false, skip = false;
        {
            const uint8_t c0 = bs.peek();
            if (c0 == '#') skip = true;
        }
        if (!skip && !fast_head(a.text, a.nbytes, p, heads[threadIdx.x], h, a.rg)) {
            for (;;) {
                if (q >= a.nbytes) { nl = a.nbytes; le = a.nbytes; ended = true; break; }
                const uint8_t c = bs.peek();
                if (c == '\n') { nl = q; le = q; ended = true; break; }
                bs.advance();
                if (c == '\r' && q + 1 < a.nbytes && bs.peek() == '\n') { nl = q + 1; le = q; ended = true; break; }
                const bool done = h.feed(c, q, a.rg);
                ++q;
                if (done) break;
            }
        }
        if (ended) {
            if (nl >= a.nbytes) break;                        // text without a final newline: not a record
            h.finish_short();
            // position the reader after the newline (it sits on '\n' now)
            bs.advance();
            p = nl + 1;
        } else {
            // q - 1 == samp_abs (or the '#' line): where does the record end?
            bool found = false;
            if (!skip) {
                const uint64_t e = h.samp_abs + span;
                if (e < a.nbytes) {
                    bs.init(a.text, a.nbytes, e);
                    const uint8_t c = bs.peek();
                    if (c == '\n') { le = e; nl = e; found = true; fast = true; }
                    else if (c == '\r') {
                        bs.advance();
                        if (e + 1 < a.nbytes && bs.peek() == '\n') { le = e; nl = e + 1; found = true; fast = true; }
                    }
                }
            }
            if (!found) {
                nl = find_newline(a.text, a.nbytes, skip ? ls : h.samp_abs);
                if (nl >= a.nbytes) break;
                le = (nl > ls && a.text[nl - 1] == '\r') ? nl - 1 : nl;
                bs.init(a.text, a.nbytes, nl);
            }
            bs.advance();                                     // consume the '\n'
            p = nl + 1;
        }
        ++lines;
        if (skip || le == ls) continue;                       // '#' line or empty line: ignored
        const HeadVerdict v = judge_head(h, le, a.n_samples, a.rg, a.end_is_int);
        if (v.malformed) atomicAdd(&a.st->n_bad_cols, 1ull);
        if (v.keep) {
            if (kept < kWalkSlots) write_site_row(a.pad, a.text, row0 + kept, ls, le, h, v, 1, kNoCpRow);
            else a.st->walk_broken = 1u;                     // more kept lines in a range than slots: the caller falls back
        }
        if (fast && !(v.keep && v.uniform)) {
            const unsigned long long k = atomicAdd(&a.st->n_verify, 1ull);
            if (k < a.verify_cap) a.verify[k] = h.samp_abs;
            else a.st->index_invalid = 1u;                   // cannot be proven: make the caller fall back
        }
        if (v.keep && h.has_samples && h.g >= 0 && !v.uniform) atomicAdd(&a.st->n_nu_count, 1ull);
        if (v.keep) ++kept;
    }
    if (p != end) a.st->walk_broken = 1u;
    a.wcount[w] = make_uint2(lines, kept < kWalkSlots ? kept : kWalkSlots);
}

// single CTA: exclusive prefix sum of kept rows over the walkers + totals.  1024 walkers per round, read coalesced (the
// next round's counts are requested before this round is scanned): 27 us for 69 K walkers, where one contiguous block of
// walkers per thread (strided reads, two passes) took 92.
__global__ void __launch_bounds__(1024) walk_scan_kernel(const WalkArgs a) {
    __shared__ uint32_t s_rows[32], s_lines[32];
    const uint32_t t = threadIdx.x, lane = t & 31, warp = t >> 5, n = a.n_walkers;
    uint64_t carry_rows = 0, carry_lines = 0;
    uint2 nxt = t < n ? a.wcount[t] : make_uint2(0, 0);
    for (uint32_t base = 0; base < n; base += 1024) {
        const uint2 c = nxt;
        nxt = base + 1024 + t < n ? a.wcount[base + 1024 + t] : make_uint2(0, 0);
        uint32_t r = c.y, l = c.x;                          // (a walker holds a handful of lines)
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, r, d);
            if (lane >= (uint32_t)d) r += v;
            l += __shfl_xor_sync(0xffffffffu, l, d);
        }
        if (lane == 31) { s_rows[warp] = r; s_lines[warp] = l; }
        __syncthreads();
        uint32_t wr = s_rows[lane], wl = s_lines[lane];     // every warp scans the 32 warp totals
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, wr, d);
            if (lane >= (uint32_t)d) wr += v;
            wl += __shfl_xor_sync(0xffffffffu, wl, d);
        }
        const uint32_t before = __shfl_sync(0xffffffffu, wr, warp) - s_rows[warp];      // rows of the warps in front
        const uint32_t total = __shfl_sync(0xffffffffu, wr, 31);
        if (base + t < n) a.wrow[base + t] = carry_rows + before + (r - c.y);
        carry_rows += total;
        carry_lines += wl;
        __syncthreads();                                    // s_rows / s_lines are rewritten by the next round
    }
    if (t == 0) { a.st->n_records = carry_rows; a.st->n_lines = carry_lines; }
}

// padded rows -> dense rows: thread = (walker, slot); a row that needs the general decode path registers its dense index
// under the checkpoint-table slot it was given during the walk
__global__ void __launch_bounds__(256) walk_compact_kernel(const WalkArgs a) {
    const uint64_t t = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    const uint32_t w = (uint32_t)(t / kWalkSlots), j = (uint32_t)(t - (uint64_t)w * kWalkSlots);
    if (w >= a.n_walkers || j >= a.wcount[w].y) return;
    const uint64_t dst = a.wrow[w] + j;
    a.out.start[dst] = a.pad.start[t];
    a.out.stop[dst] = a.pad.stop[t];
    a.out.ref[dst] = a.pad.ref[t];
    a.out.alt[dst] = a.pad.alt[t];
    a.out.chrom_abs[dst] = a.pad.chrom_abs[t];
    a.out.chrom_len[dst] = a.pad.chrom_len[t];
    a.out.chrom5[dst] = a.pad.chrom5[t];
    const RowInfo ri = a.pad.rowinfo[t];
    a.out.rowinfo[dst] = ri;
    const uint32_t gi = ri.misc & 0xffu;
    if ((ri.misc & kRowHasSamples) && gi != 255u && !(ri.misc & kRowUniform)) a.out.nu_rows[ri.cp_row] = (uint32_t)dst;
}

// The jumped-over spans nobody decodes: [tab9, tab9 + 4*S) must not hold a newline.
__global__ void __launch_bounds__(256) walk_verify_kernel(const WalkArgs a, uint32_t pieces_per_span) {
    const uint64_t nv = a.st->n_verify;
    const uint64_t n = nv < a.verify_cap ? nv : a.verify_cap;
    const uint64_t total = n * pieces_per_span;
    const uint64_t span = 4ull * a.n_samples;
    for (uint64_t item = blockIdx.x; item < total; item += gridDim.x) {
        const uint64_t b = a.verify[item / pieces_per_span];
        const uint64_t pb = b + (item % pieces_per_span) * 4096ull;
        const uint64_t pe = (b + span) < (pb + 4096ull) ? (b + span) : (pb + 4096ull);
        const uint64_t o = (pb & ~15ull) + 16ull * threadIdx.x;       // 256 threads x 16 B >= 4096 + 15
        for (uint64_t oo = o; oo < pe; oo += 4096) {
            uint32_t m = nl_bits(ld_chunk(a.text, oo, a.nbytes));
            if (oo < pb) m &= ~((1u << (pb - oo)) - 1u);
            if (oo + 16 > pe) m &= (1u << (pe - oo)) - 1u;
            if (m) a.st->index_invalid = 1u;
        }
    }
}

uint32_t walk_plan(uint64_t nbytes, uint64_t first_line_len, uint32_t lines_per_walker, uint64_t *range_bytes) {
    uint64_t r = std::max<uint64_t>(first_line_len, 64) * lines_per_walker;
    r = (r + 15) & ~15ull;
    uint64_t n = (nbytes + r - 1) / r;
    if (n > 0x3fffffffull) n = 0x3fffffffull;
    if (n == 0) n = 1;
    *range_bytes = r;
    return (uint32_t)n;
}

static WalkArgs make_args(const uint8_t *d_text, uint64_t nbytes, uint32_t n_samples, uint64_t range_bytes,
                          uint32_t n_walkers, const RegionArg &rg, int end_is_int, uint64_t *d_wstart, uint2 *d_wcount,
                          uint64_t *d_wrow, DevStatus *d_st) {
    WalkArgs a;
    memset(&a, 0, sizeof a);
    a.text = d_text; a.nbytes = nbytes; a.n_samples = n_samples; a.range_bytes = range_bytes; a.n_walkers = n_walkers;
    a.rg = rg; a.end_is_int = end_is_int; a.wstart = d_wstart; a.wcount = d_wcount; a.wrow = d_wrow; a.st = d_st;
    a.out.st = d_st;
    return a;
}

void launch_walk(const uint8_t *d_text, uint64_t nbytes, uint32_t n_samples, uint64_t range_bytes, uint32_t n_walkers,
                 const RegionArg &rg, int end_is_int, uint64_t *d_wstart, void *d_wcount, uint64_t *d_wrow, const SiteRows &pad,
                 uint64_t *d_verify, uint64_t verify_cap, DevStatus *d_st, const Launch &L) {
    WalkArgs a = make_args(d_text, nbytes, n_samples, range_bytes, n_walkers, rg, end_is_int, d_wstart,
                           (uint2 *)d_wcount, d_wrow, d_st);
    a.pad.start = pad.start; a.pad.stop = pad.stop; a.pad.ref = pad.ref; a.pad.alt = pad.alt;
    a.pad.chrom_abs = pad.chrom_abs; a.pad.chrom_len = pad.chrom_len; a.pad.chrom5 = pad.chrom5; a.pad.rowinfo = pad.rowinfo;
    a.pad.nu_rows = nullptr;                 // (the dense index is registered by the compaction)
    a.pad.st = d_st;
    a.verify = d_verify; a.verify_cap = verify_cap;
    walk_sync_kernel<<<(n_walkers + 1 + 7) / 8, 256, 0, L.stream>>>(a);
    walk_kernel<<<(n_walkers + WK_THREADS - 1) / WK_THREADS, WK_THREADS, 0, L.stream>>>(a);
    walk_scan_kernel<<<1, 1024, 0, L.stream>>>(a);
    count_launch(3);
}

void launch_walk_compact(const uint8_t *d_text, uint64_t nbytes, uint32_t n_samples, uint32_t n_walkers, void *d_wcount,
                         uint64_t *d_wrow, const SiteRows &pad, const SiteRows &rows, uint32_t *d_nu_rows, uint64_t *d_verify,
                         uint64_t verify_cap, DevStatus *d_st, const Launch &L) {
    RegionArg rg;
    memset(&rg, 0, sizeof rg);
    WalkArgs a = make_args(d_text, nbytes, n_samples, 0, n_walkers, rg, 0, nullptr, (uint2 *)d_wcount, d_wrow, d_st);
    a.pad.start = pad.start; a.pad.stop = pad.stop; a.pad.ref = pad.ref; a.pad.alt = pad.alt;
    a.pad.chrom_abs = pad.chrom_abs; a.pad.chrom_len = pad.chrom_len; a.pad.chrom5 = pad.chrom5; a.pad.rowinfo = pad.rowinfo;
    a.out.start = rows.start; a.out.stop = rows.stop; a.out.ref = rows.ref; a.out.alt = rows.alt;
    a.out.chrom_abs = rows.chrom_abs; a.out.chrom_len = rows.chrom_len; a.out.chrom5 = rows.chrom5; a.out.rowinfo = rows.rowinfo;
    a.out.nu_rows = d_nu_rows;
    a.verify = d_verify; a.verify_cap = verify_cap;
    const uint64_t n = (uint64_t)n_walkers * kWalkSlots;
    walk_compact_kernel<<<(unsigned)((n + 255) / 256), 256, 0, L.stream>>>(a);
    const uint32_t pieces = (uint32_t)((4ull * n_samples + 4095) / 4096);
    walk_verify_kernel<<<L.sm_count * 4, 256, 0, L.stream>>>(a, pieces ? pieces : 1);
    count_launch(2);
}

}  // namespace hb
