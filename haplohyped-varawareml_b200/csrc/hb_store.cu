// hb_store.cu -- kernel 4: Blosc byte-shuffle + LZ4 block encoder + Blosc chunk framing, and the read side.
//
// Replaces what h5py + hdf5plugin do for every HDF5 chunk of
//   create_dataset('snp_data', data=<35-byte records>, compression=32001,
//                  compression_opts=(2,2,0,0,5,1,2), chunks=True)        (vcf_to_h5.py:119-135)
// Filter 32001 is hdf5-blosc, i.e. c-blosc 1.x: shuffle(typesize 35) + an LZ4-family codec, one bare Blosc1 chunk
// per HDF5 chunk (the opts are [filter rev 2, Blosc format 2, typesize, chunk bytes, clevel 5, shuffle 1, compcode 2 =
// LZ4HC]).  LZ4 and LZ4HC share one block format and one Blosc codec-format id, so a stock decoder cannot tell
// which encoder wrote a stream.
//
// The byte-shuffled image of one (sample, chunk) is 35 planes of `cr` bytes.  Planes 0..32 hold
// site bytes and are IDENTICAL for every sample; only planes 33/34 (the two allele planes, which
// the GT decoder already wrote in exactly this planar layout) differ.  So the 33 site planes are encoded once per
// chunk (site_template_kernel) and every donor continues that LZ4 block with its own 2 * cr allele bytes
// (donor_frames_kernel).  The site encoder is a warp-cooperative greedy matcher: 32 candidate positions per step are
// hashed in parallel, the first hit is extended with ballots, literals are copied 32 bytes per step.
#include <emmintrin.h>
#include <sched.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <condition_variable>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "../../include/haplo_b200.h"
#include "hb_common.cuh"
#include "hb_internal.h"
#include "hb_parse_struct.h"

namespace hb {

extern __shared__ __align__(128) uint8_t smem[];     // the dynamic shared memory of the encoder kernels

__device__ __forceinline__ uint32_t rd32(const uint8_t *p) {     // unaligned 4-byte read (shared memory)
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const uint32_t *w = reinterpret_cast<const uint32_t *>(a & ~uintptr_t(3));
    return __funnelshift_r(w[0], w[1], (uint32_t)(a & 3) * 8u);
}

// extension bytes of an LZ4 literal length (or of a match length - 4)
__device__ __forceinline__ int lit_ext(int lit) { return lit >= 15 ? 1 + (lit - 15) / 255 : 0; }

// one LZ4 sequence, written by the whole warp; returns the new output offset
__device__ int warp_emit_seq(uint8_t *dst, int o, const uint8_t *lit, int litlen, int off, int ml) {
    const int lane = threadIdx.x & 31;
    if (lane == 0) dst[o] = (uint8_t)((min(litlen, 15) << 4) | min(ml - 4, 15));
    ++o;
    if (litlen >= 15) {
        int rem = litlen - 15;
        while (rem >= 255) { if (lane == 0) dst[o] = 255; ++o; rem -= 255; }
        if (lane == 0) dst[o] = (uint8_t)rem;
        ++o;
    }
    for (int i = lane; i < litlen; i += 32) dst[o + i] = lit[i];
    o += litlen;
    if (lane == 0) { dst[o] = (uint8_t)off; dst[o + 1] = (uint8_t)(off >> 8); }
    o += 2;
    if (ml - 4 >= 15) {
        int rem = ml - 19;
        while (rem >= 255) { if (lane == 0) dst[o] = 255; ++o; rem -= 255; }
        if (lane == 0) dst[o] = (uint8_t)rem;
        ++o;
    }
    return o;
}

// Warp-cooperative LZ4 encoder of one SEGMENT src[0..n) of a block whose earlier bytes (`hist` of them) sit right
// in front of src.  32 positions are examined per step; each lane tests three candidates for its position -- `far`
// bytes back (0 = none), the last position with the same 4-byte hash (own segment only), one byte back -- the first
// lane with a hit wins and the match is extended with ballots.  Only complete sequences are emitted and no match
// crosses the end of the segment.  The first sequence assumes that its literal run starts at src[0]: its header
// (token + literal-length bytes) occupies dst[0..*first_hdr) and announces *first_lit literals, so that a caller
// which carries literals in from the previous segment can re-write just that header.  *pending = trailing bytes of
// the segment not covered by a sequence.  deep: the hash table holds buckets of 4 (the last position of each p mod 4)
// and the candidate with the longest match over the next 8 bytes is taken -- about 6 % smaller output on random
// A/C/G/T planes for about twice the time.  table: 1 << hashlog uint16 entries (position + 1), cleared here;
// n < 65535.  Returns the bytes written to dst; all lanes return the same values.
// The site planes pass far = 4*cr: the stop column is the start column + 1, so bytes 1..3 of `stop` (planes 10-12)
// repeat bytes 1..3 of `start` (planes 6-8) almost everywhere.
__device__ int warp_lz4_segment(const uint8_t *src, int n, int hist, uint8_t *dst, uint16_t *table, int hashlog,
                                int far, bool deep, int *first_lit, int *first_hdr, int *pending) {
    const int lane = threadIdx.x & 31;
    for (int i = lane; i < (1 << hashlog); i += 32) table[i] = 0;
    __syncwarp();
    int op = 0, anchor = 0, pos = 0;
    const int mflimit = n - 4;                       // last position a match may start at
    *first_lit = 0; *first_hdr = 0;
    while (pos <= mflimit) {
        const int p = pos + lane;
        const bool valid = p <= mflimit;
        uint32_t v = 0, h = 0;
        int cand = -0x40000000;
        if (valid) {
            v = rd32(src + p);
            h = deep ? ((v * 2654435761u) >> (34 - hashlog)) << 2      // bucket of 4: the last position of each p mod 4
                     : (v * 2654435761u) >> (32 - hashlog);
            if (far && p + hist >= far && rd32(src + p - far) == v) cand = p - far;
            else if (!deep) {
                const int c = (int)table[h] - 1;
                if (c >= 0 && c < p && rd32(src + c) == v) cand = c;   // c == p: left by a re-examined window
                else if (p + hist >= 1 && rd32(src + p - 1) == v) cand = p - 1;      // run of one byte
            } else {
                // longest of the bucket's candidates, measured over the next 8 bytes (ties: the nearest)
                const uint2 b4 = *reinterpret_cast<const uint2 *>(table + h);
                const int cs[4] = {(int)(b4.x & 0xffffu) - 1, (int)(b4.x >> 16) - 1, (int)(b4.y & 0xffffu) - 1, (int)(b4.y >> 16) - 1};
                int best = -1;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int c = cs[k];
                    if (c >= 0 && c < p && rd32(src + c) == v) {                 // c == p: left by a re-examined window
                        const uint32_t x1 = rd32(src + p + 4) ^ rd32(src + c + 4);
                        int ex;
                        if (x1) ex = (__ffs(x1) - 1) >> 3;
                        else { const uint32_t x2 = rd32(src + p + 8) ^ rd32(src + c + 8); ex = 4 + (x2 ? (__ffs(x2) - 1) >> 3 : 4); }
                        const int key = (ex << 16) | c;                          // longer first, then nearer (larger c)
                        if (key > best) best = key;
                    }
                }
                if (best >= 0) cand = best & 0xffff;
                else if (p + hist >= 1 && rd32(src + p - 1) == v) cand = p - 1;  // run of one byte
            }
        }
        __syncwarp();
        if (valid) table[deep ? h + (p & 3) : h] = (uint16_t)(p + 1);
        __syncwarp();
        const unsigned hit = __ballot_sync(0xffffffffu, cand > -0x40000000);
        if (!hit) { pos += 32; continue; }
        const int f = __ffs(hit) - 1;
        const int m = pos + f;
        const int c = __shfl_sync(0xffffffffu, cand, f);
        int ml = 4;
        for (;;) {
            const int i = ml + lane;
            const bool same = (m + i < n) && src[m + i] == src[c + i];
            const unsigned bal = __ballot_sync(0xffffffffu, same);
            if (bal == 0xffffffffu) { ml += 32; continue; }
            ml += __ffs(~bal) - 1;
            break;
        }
        const int litlen = m - anchor;
        if (op == 0) { *first_lit = litlen; *first_hdr = op + 1 + lit_ext(litlen); }
        op = warp_emit_seq(dst, op, src + anchor, litlen, m - c, ml);
        anchor = pos = m + ml;
    }
    *pending = n - anchor;
    __syncwarp();
    return op;
}

// ------------------------------------------------------------------------------------------
// Chunk anatomy.  HDF5 filter 32001 is hdf5-blosc (c-blosc 1.x): one HDF5 chunk of one donor is stored as ONE
// bare Blosc1 chunk (blosc_compress output), little-endian:
//   [0,16)   header: version 2 (BLOSC_VERSION_FORMAT), versionlz 1 (LZ4 format), flags 0x31 (byte-shuffle |
//            don't-split | LZ4 codec format << 5), typesize 35, nbytes, blocksize (= nbytes: one block),
//            cbytes @12 (whole chunk incl. this header)                          -- cbytes depends on the donor
//   [16,20)  bstarts[0] = 20
//   [20,24)  csize of the block's single (no-split) stream, LE32                 -- depends on the donor
//   [24,24+plen)   LZ4 sequences of the 33 site planes    -- identical for every donor
//   [.., +dlen)    LZ4 sequences of the 2 allele planes   -- the donor's own
// typesize 35 > 16, so c-blosc itself never splits such a block either; the decoder (blosc_d) reads
// "int32 csize + stream" per block, csize == blocksize meaning "stored raw".
// Kernels:
//   site_template_kernel   one CTA per chunk: site planes -> LZ4; writes the chunk TEMPLATE (header with the two
//                          donor-dependent fields left zero + shared LZ4 head), 16-byte aligned.
//   donor_frames_kernel    one CTA per (chunk, group of samples), one warp per frame at a time.  The chunk's
//                          template is pulled into shared memory ONCE per CTA (TMA bulk copy); every frame's allele
//                          bits arrive by TMA one frame ahead; the warp encodes the allele planes as the LZ4 tail of
//                          the block (bit-parallel matcher, below) into shared memory; the frame then leaves as two
//                          TMA bulk stores (template body from the shared copy, own tail) + two 16-byte header
//                          vectors with the size fields filled in.  C_out is written exactly once.
//   site_template_large_kernel / donor_frames_large_kernel   the same frames for chunks of 2,731 - 7,489 records (still ONE
//                          Blosc block), built by the same encoder helpers (site_encode_chunk; build_bit_strings,
//                          parse_lane, scan_offsets, emit_lane, closing_literals).  What differs: site planes in a global
//                          scratch, allele tails in passes, template read from global memory.  The host picks the pair
//                          from cr.
// Output: ONE buffer of slots in [sample][chunk] order.  The slot of (sample s, chunk c) starts at
// s * row_stride + slot_off[c]; slot_off is the running sum of round16(template_len[c] + worst-case
// allele tail), so every frame's address is known before it is encoded (no scan, no look-back) and the
// layout is deterministic.  A frame fills the front of its slot; its true length is recorded.
// ------------------------------------------------------------------------------------------
constexpr int BLOSC_HDR = 16;
constexpr int TMPL_HDR = BLOSC_HDR + 8;        // 24 bytes of a chunk precede its LZ4 block

__device__ __forceinline__ void put_le32(uint8_t *p, uint32_t v) {
    p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); p[2] = (uint8_t)(v >> 16); p[3] = (uint8_t)(v >> 24);
}

// the 24 header bytes of a chunk of `nbytes` uncompressed bytes; the donor-dependent fields are zero
__device__ void write_frame_head(uint8_t *h, uint32_t nbytes) {
    for (int i = 0; i < TMPL_HDR; ++i) h[i] = 0;
    h[0] = 2; h[1] = 1; h[2] = 0x31; h[3] = 35;
    put_le32(h + 4, nbytes); put_le32(h + 8, nbytes);        // cbytes @12: patched
    put_le32(h + 16, BLOSC_HDR + 4);                         // bstarts[0]
}                                                            // csize @20: patched

// byte offsets of the fields of a 35-byte record (plane f of a shuffled chunk holds byte f of every record): CHROM's
// first 5 bytes at 0, start and stop as LE32, REF and ALT as the first bytes of their 10-byte fields, the two alleles
constexpr uint32_t kRecStart = 5, kRecStop = 9, kRecRef = 13, kRecAlt = 23, kRecP1 = 33, kRecP2 = 34;

struct SiteArgs4 {
    const uint64_t *chrom5;      // per record: first 5 CHROM bytes, NUL padded, in the low 40 bits
    const uint32_t *start, *stop;
    const uint8_t *ref, *alt;
    uint64_t n_records;
    uint32_t cr;                 // records per chunk
    uint8_t *tmpl;               // [n_chunks][tmpl_cap], 16-byte aligned rows
    uint32_t tmpl_cap;
    uint32_t *tmpl_len;          // [n_chunks] = TMPL_HDR + LZ4 bytes of the site planes
    int deep;                    // 4-way bucket matcher (hb_set_site_matcher(1)): smaller templates, slower kernel
};

constexpr int kSiteSegs = 18;                    // = warps of the CTA
constexpr int kSiteHashLog = 10;
__host__ __device__ inline uint32_t site_seg_cap(uint32_t len) { return (len + len / 255 + 24 + 15) & ~15u; }
// Segment s of the encoded part [0, 24*cr+1) of the site planes covers [site_seg_begin(s), site_seg_begin(s+1)).
// The cuts follow where the work is.  r01 gave the random REF and ALT planes three warps each and the nine planes in
// front of them ONE: the r02v ncu capture showed 69 % of the stall samples at the barrier behind the encode -- seven
// warps waiting for the one that walks start's byte 1 (a short run every few records) after five constant planes.
// The cuts below equalise the per-segment cycle counts measured with clock64() (0.57 -> 0.23 -> 0.14 ms).
__host__ __device__ inline uint32_t site_seg_begin(int s, uint32_t cr) {
    switch (s) {                                   // (cycles of a warp on its segment, r02w, at cr = 1075)
        case 0: return 0;                          // CHROM bytes: five constant planes                           38 K
        case 1: return 5 * cr;                     // start, byte 0: literals                                     27 K
        case 2: return 6 * cr;                     // start, byte 1: a short run every few records -- the most
        case 3: return 6 * cr + cr / 5;            //   expensive bytes of the block (180 cycles each): in fifths  39 K
        case 4: return 6 * cr + 2 * cr / 5;
        case 5: return 6 * cr + 3 * cr / 5;
        case 6: return 6 * cr + 4 * cr / 5;
        case 7: return 7 * cr;                     // start, bytes 2-3                                            17 K
        case 8: return 9 * cr;                     // stop: matches 4 * cr back, in halves                        25 K
        case 9: return 11 * cr;
        case 10: return 13 * cr;                   // REF in thirds                                               33 K
        case 11: return 13 * cr + cr / 3;
        case 12: return 13 * cr + 2 * cr / 3;
        case 13: return 14 * cr;                   // the nine zero planes behind REF, in halves                  29 K
        case 14: return 18 * cr + cr / 2;
        case 15: return 23 * cr;                   // ALT in thirds                                               33 K
        case 16: return 23 * cr + cr / 3;
        case 17: return 23 * cr + 2 * cr / 3;
        default: return 24 * cr + 1;
    }
}

// ---- The site-template encoder shared by site_template_kernel and site_template_large_kernel.

// site planes 0..23 of chunk c: CHROM, start, stop, REF and its nine zero planes, ALT's first byte.  Planes 24..32 (ALT
// bytes 1..9) are zero too; the caller clears them.
__device__ __forceinline__ void site_planes_fill(const SiteArgs4 &a, uint64_t c, uint8_t *planes) {
    const uint32_t cr = a.cr;
    const uint64_t r0 = c * cr;
    for (uint32_t i = threadIdx.x; i < cr; i += blockDim.x) {
        const uint64_t r = r0 + i;
        uint64_t ch = 0;
        uint32_t st = 0, sp = 0;
        uint8_t rf = 0, al = 0;
        if (r < a.n_records) { ch = a.chrom5[r]; st = a.start[r]; sp = a.stop[r]; rf = a.ref[r]; al = a.alt[r]; }
#pragma unroll
        for (int k = 0; k < 5; ++k) planes[k * cr + i] = (uint8_t)(ch >> (8 * k));
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            planes[(kRecStart + k) * cr + i] = (uint8_t)(st >> (8 * k));
            planes[(kRecStop + k) * cr + i] = (uint8_t)(sp >> (8 * k));
        }
        planes[kRecRef * cr + i] = rf;
        planes[kRecAlt * cr + i] = al;
#pragma unroll
        for (int k = 1; k < 10; ++k) planes[(kRecRef + k) * cr + i] = 0;
    }
}

// per-segment results and the stitch of one chunk (static shared memory of both site kernels)
struct SiteStitch {
    int len[kSiteSegs], pend[kSiteSegs], flit[kSiteSegs], fhdr[kSiteSegs];     // warp_lz4_segment's, per segment
    int dst[kSiteSegs], carry[kSiteSegs];        // where the segment's output goes; literals carried into it
    int final_off, final_carry;                  // end of the stitched head; literals left behind it
    uint8_t head[TMPL_HDR];                      // write_frame_head's bytes
};

// Chunk c's planes (16 zero bytes of history in front of them, planes 24..32 zero) -> its template and tmpl_len[c];
// `head` is written and the CTA synchronised before the call.  Planes 24..32 (ALT bytes 1..9) are all zero: the head
// is encoded up to the first of those zeros, then ONE offset-1 match covers the other 9*cr-1 -- so the site part always
// ends on a sequence boundary and every donor continues the block with nothing pending and zeros behind it.  The head
// is cut into kSiteSegs segments, one per warp, encoded independently into the warp's region of `outs` (own hash
// table; the fixed-distance candidates reach back across segments) and then stitched back to back.
__device__ __forceinline__ void site_encode_chunk(const SiteArgs4 &a, uint64_t c, const uint8_t *planes, uint8_t *outs,
                                                  uint16_t *table, SiteStitch &S) {
    const uint32_t cr = a.cr, n = 33u * cr;
    const int n1 = 24 * (int)cr + 1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sb = (int)site_seg_begin(warp, cr), se = (int)site_seg_begin(warp + 1, cr);
    uint32_t out_off = 0;
    for (int w = 0; w < warp; ++w) out_off += site_seg_cap(site_seg_begin(w + 1, cr) - site_seg_begin(w, cr));
    uint8_t *my_out = outs + out_off;
    {
        int flit, fhdr, pend;
        const int len = warp_lz4_segment(planes + sb, se - sb, sb, my_out, table, kSiteHashLog, 4 * (int)cr, a.deep != 0, &flit, &fhdr, &pend);
        if (lane == 0) { S.len[warp] = len; S.pend[warp] = pend; S.flit[warp] = flit; S.fhdr[warp] = fhdr; }
    }
    __syncthreads();
    if (threadIdx.x == 0) {                       // stitch: literals left over by a segment open the next one's first sequence
        int carry = 0, off = 0;
        for (int w = 0; w < kSiteSegs; ++w) {
            S.dst[w] = off; S.carry[w] = carry;
            if (S.len[w] == 0) { carry += S.pend[w]; continue; }
            off += 1 + lit_ext(S.flit[w] + carry) + carry + (S.len[w] - S.fhdr[w]);
            carry = S.pend[w];
        }
        S.final_off = off; S.final_carry = carry;
    }
    __syncthreads();
    uint8_t *g = a.tmpl + c * a.tmpl_cap;
    uint8_t *lz = g + TMPL_HDR;
    if (S.len[warp] > 0) {                        // the segment's first sequence, re-written with the carried literals
        const int carry = S.carry[warp], lit = S.flit[warp] + carry;
        int o = S.dst[warp];
        if (lane == 0) lz[o] = (uint8_t)((min(lit, 15) << 4) | (my_out[0] & 15));
        ++o;
        if (lit >= 15) {
            int rem = lit - 15;
            while (rem >= 255) { if (lane == 0) lz[o] = 255; ++o; rem -= 255; }
            if (lane == 0) lz[o] = (uint8_t)rem;
            ++o;
        }
        for (int i = lane; i < carry; i += 32) lz[o + i] = planes[sb - carry + i];
        o += carry;
        const int rest = S.len[warp] - S.fhdr[warp];
        for (int i = lane; i < rest; i += 32) lz[o + i] = my_out[S.fhdr[warp] + i];
    }
    const int fl = S.final_carry;
    int o = S.final_off;
    if (warp == 0) o = warp_emit_seq(lz, o, planes + n1 - fl, fl, 1, (int)n - n1);
    else o += 1 + lit_ext(fl) + fl + 2 + lit_ext((int)n - n1 - 4);
    const uint32_t tl = TMPL_HDR + (uint32_t)o;
    for (uint32_t i = threadIdx.x; i < TMPL_HDR; i += blockDim.x) g[i] = S.head[i];
    for (uint32_t i = tl + threadIdx.x; i < ((tl + 15) & ~15u); i += blockDim.x) g[i] = 0;
    if (threadIdx.x == 0) a.tmpl_len[c] = tl;
}

__global__ void __launch_bounds__(kSiteSegs * 32) site_template_kernel(const SiteArgs4 a) {
    __shared__ SiteStitch S;
    const uint32_t cr = a.cr;
    const uint32_t n = 33u * cr;
    const int warp = threadIdx.x >> 5;
    uint8_t *planes = smem + 16;                            // 16 zero bytes of history in front
    uint8_t *outs = planes + ((n + 19) & ~15u);             // per-segment output regions, then the hash tables
    uint16_t *table = reinterpret_cast<uint16_t *>(outs + ((site_seg_cap(24 * cr + 1) + kSiteSegs * 48 + 15) & ~15u)) + ((size_t)warp << kSiteHashLog);
    const uint64_t c = blockIdx.x;
    site_planes_fill(a, c, planes);
    for (uint32_t i = 24 * cr + threadIdx.x; i < n; i += blockDim.x) planes[i] = 0;
    if (threadIdx.x < 16) smem[threadIdx.x] = 0;
    if (threadIdx.x == 0) write_frame_head(S.head, 35u * cr);
    __syncthreads();
    // Chunks of fewer than 6 records cannot honour LZ4's end-of-block rules (last match >= 12 bytes
    // before the end) once the 2*cr allele bytes follow: such blocks are stored raw (csize == size).
    if (cr < 6) {
        uint8_t *g = a.tmpl + c * a.tmpl_cap;
        for (uint32_t i = threadIdx.x; i < TMPL_HDR; i += blockDim.x) g[i] = S.head[i];
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) g[TMPL_HDR + i] = planes[i];
        const uint32_t tl = TMPL_HDR + n;
        for (uint32_t i = tl + threadIdx.x; i < ((tl + 15) & ~15u); i += blockDim.x) g[i] = 0;
        if (threadIdx.x == 0) a.tmpl_len[c] = tl;
        return;
    }
    site_encode_chunk(a, c, planes, outs, table, S);
}

// ------------------------------------------------------------------------------------------
// Kernel 4a-L: the site templates of chunks of kSmallChunkMax < cr <= kMaxChunkRecords records.  Up to 7,489 records
// such a chunk is still ONE Blosc block with ONE LZ4 stream (c-blosc 1.x cuts blocks of 262,115 bytes for typesize 35
// at clevel 5 with LZ4HC), so the template has exactly the layout of site_template_kernel's, and both kernels encode it
// with site_planes_fill and site_encode_chunk: the same segments, matcher, stitch and closing offset-1 match over
// planes 24-32.  What differs is where the bytes live: 33 * cr bytes of planes no longer fit shared memory, so the head
// [0, 24 * cr + 1) that is encoded and the per-segment outputs sit in a per-CTA global scratch (L2-resident:
// ~2 * 24 * cr bytes per CTA), and only the hash tables stay in shared memory.  The 16-bit table entries still hold:
// positions are relative to a segment, and the longest segment (the five CHROM planes) is 5 * 7,489 < 65,535 bytes;
// far = 4 * cr and 2 * cr are legal LZ4 offsets.  The grid is smaller than the chunk count (the scratch is per CTA):
// CTA b encodes chunks b, b + gridDim.x, ...
// ------------------------------------------------------------------------------------------
constexpr uint32_t kSmallChunkMax = 2730;        // largest chunk of site_template_kernel / donor_frames_kernel
constexpr uint32_t kMaxChunkRecords = 7489;      // largest chunk that is ONE c-blosc 1.x block at typesize 35
constexpr uint32_t kSitePad = 48;                // zero bytes behind the head: look-ahead reads of the last segment
__host__ __device__ inline uint32_t site_large_head_bytes(uint32_t cr) { return (16 + 24 * cr + 1 + kSitePad + 15) & ~15u; }
__host__ __device__ inline uint32_t site_large_scratch(uint32_t cr) {
    return site_large_head_bytes(cr) + ((site_seg_cap(24 * cr + 1) + kSiteSegs * 48 + 15) & ~15u);
}

__global__ void __launch_bounds__(kSiteSegs * 32) site_template_large_kernel(const SiteArgs4 a, uint8_t *scratch) {
    __shared__ SiteStitch S;
    const uint32_t cr = a.cr;
    const int warp = threadIdx.x >> 5;
    uint8_t *planes = scratch + (size_t)blockIdx.x * site_large_scratch(cr) + 16;   // 16 zero bytes of history in front
    uint8_t *outs = planes - 16 + site_large_head_bytes(cr);
    uint16_t *table = reinterpret_cast<uint16_t *>(smem) + ((size_t)warp << kSiteHashLog);
    const uint64_t n_chunks = (a.n_records + cr - 1) / cr;
    if (threadIdx.x < 16) planes[(int)threadIdx.x - 16] = 0;
    for (uint32_t i = 24 * cr + threadIdx.x; i < 24 * cr + 1 + kSitePad; i += blockDim.x) planes[i] = 0;   // planes 24.. are zero
    if (threadIdx.x == 0) write_frame_head(S.head, 35u * cr);
    for (uint64_t c = blockIdx.x; c < n_chunks; c += gridDim.x) {
        site_planes_fill(a, c, planes);
        __syncthreads();
        site_encode_chunk(a, c, planes, outs, table, S);
        __syncthreads();                          // the scratch and the stitch table are re-used by the next chunk
    }
}

// ------------------------------------------------------------------------------------------
// Allele-plane encoder, bit-parallel.  After the SNP filter the allele bytes are 0 / 1 (rarely -9), and the GT
// decoder leaves them as bit planes too (B = bit 0 of the byte, N = "neither 0 nor 1"; hb_internal.h), so LZ4
// matches are found with word-wide logic instead of byte-wise hashing.  Two match sources:
//   Z  a zero byte: matches the all-zero site plane two planes back      (offset 2*cr),  Z = ~B & ~N
//   C  plane 1 only: equal to the same record's byte in plane 0           (offset cr),    C = ~(B1^B0) & ~(N1|N0)
// A byte with N set never matches, so the stream is exact for ANY byte values; it just compresses
// best on genotype data.  Runs of >= 5 Z positions become matches first, then runs of >= 4 C positions
// in what is left; everything else is literal.  Lanes 0-15 own 16 segments of plane 0, lanes 16-31 the
// same segments of plane 1 (a match never crosses a segment); trailing literals of a segment are
// carried into the next lane's first sequence.  The size of every lane's output follows from popcounts
// (3 bytes per match + literals + one extension byte per literal run >= 15 / match >= 19, counted with
// shifted-OR windows), one warp scan turns the sizes into output offsets, and every lane then walks its
// matches ONCE, emitting token, literals (bits -> bytes, four per step) and offset through a 4-byte
// register accumulator into the frame's tail buffer in shared memory.
// ------------------------------------------------------------------------------------------
constexpr int kMinZ = 5, kMinC = 4;
constexpr uint32_t kSlack = 128;
constexpr int kWpc = 8;                       // warps per CTA
constexpr int kFramesPerWarp = 8;             // frames (samples of one chunk) a warp encodes one after the other

__device__ __forceinline__ uint32_t low_mask(int n) { return n <= 0 ? 0u : (n >= 32 ? 0xFFFFFFFFu : ((1u << n) - 1u)); }
__device__ __forceinline__ int ctz32(uint32_t v) { return __clz(__brev(v)); }       // 32 for 0
// bits 0..3 of b -> bytes 0..3 (0 / 1)
__device__ __forceinline__ uint32_t spread4(uint32_t b) { return ((b & 0xFu) * 0x00204081u) & 0x01010101u; }

// R = the positions of X that lie inside a run of at least MINRUN consecutive ones (multi-word, LSB first)
template <int NW, int MINRUN>
__device__ __forceinline__ void runs_cover(const uint32_t (&X)[NW], uint32_t (&R)[NW]) {
    uint32_t S[NW];
#pragma unroll
    for (int k = 0; k < NW; ++k) {
        const uint32_t nxt = k + 1 < NW ? X[k + 1] : 0u;
        uint32_t s = X[k];
#pragma unroll
        for (int d = 1; d < MINRUN; ++d) s &= __funnelshift_r(X[k], nxt, d);
        S[k] = s;
    }
#pragma unroll
    for (int k = 0; k < NW; ++k) {
        const uint32_t prv = k > 0 ? S[k - 1] : 0u;
        uint32_t r = S[k];
#pragma unroll
        for (int d = 1; d < MINRUN; ++d) r |= __funnelshift_l(prv, S[k], d);
        R[k] = r;
    }
}
// Y = X | (X >> d): bit i of Y = X(i) | X(i + d) (multi-word, LSB first, 0 < d < 32)
template <int NW>
__device__ __forceinline__ void or_shr(const uint32_t (&X)[NW], int d, uint32_t (&Y)[NW]) {
    uint32_t T[NW];
#pragma unroll
    for (int k = 0; k < NW; ++k) T[k] = X[k] | __funnelshift_r(X[k], k + 1 < NW ? X[k + 1] : 0u, d);
#pragma unroll
    for (int k = 0; k < NW; ++k) Y[k] = T[k];
}
template <int NW>
__device__ __forceinline__ uint32_t shr_word(const uint32_t (&X)[NW], int k, int d) {
    return __funnelshift_r(X[k], k + 1 < NW ? X[k + 1] : 0u, d);
}

__device__ __forceinline__ void sts32(uint32_t addr, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ void sts64(uint32_t addr, uint64_t v) { asm volatile("st.shared.u64 [%0], %1;" ::"r"(addr), "l"(v) : "memory"); }
__device__ __forceinline__ void sts_or32(uint32_t addr, uint32_t v) { asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }

struct FusedArgs {
    const int8_t *gt0, *gt1;             // byte planes: read only where an allele is neither 0 nor 1 (and for raw blocks)
    uint64_t gt_stride, n_records;
    const uint32_t *bits;                // allele bit planes (hb_internal.h)
    uint64_t bits_stride;                // words per sample
    uint32_t cr, n_samples, s0;          // samples [s0, s0 + n_samples)
    uint64_t n_chunks;
    const uint8_t *tmpl; uint32_t tmpl_cap; const uint32_t *tmpl_len;
    uint8_t *frames;
    const uint64_t *slot_off;            // [n_chunks + 1] offset of chunk c's slot inside a sample row; [n_chunks] = row stride
    uint32_t *size;                      // [n_samples * n_chunks] true length of each frame
    uint32_t strw;       // words of one seamless bit string (B, N)
    uint32_t stg_bytes;  // bytes of a warp's staging area for the bit-plane slices of one frame
    uint32_t outcap;     // bytes of a warp's tail buffer
    uint32_t tmpl_smem;  // bytes reserved for the chunk's template
    uint32_t warp_smem;  // bytes per warp
    uint32_t groups, gs; // sample groups per chunk (= CTAs per chunk), samples per group
    uint32_t seg;        // block positions per lane.  Normally ceil(2 * cr / 32); when one mask word less per lane leaves at
                         // most kSlack positions of the block without an owner, those become part of the block's closing
                         // literals instead (cr 1075: 64 instead of 68 per lane, 102 of 2150 positions; +0.5 % frame size)
};

// ---- The allele-tail encoder shared by donor_frames_kernel and donor_frames_large_kernel: steps 1, 2, 3 and 5 and the
//      closing literals of one frame, run by one warp.

// One frame's allele bytes: block position x (0 .. 2 * cr) is bit alpha + x of the bit strings B and N; a byte with N set
// is read from the byte planes, row grow + x of gt0 for x < cr and row grow + x - cr of gt1 otherwise.
struct AlleleBits {
    const uint32_t *strB, *strN;
    bool any_n;                          // some allele of the frame is neither 0 nor 1: strN is valid
    int alpha, cr;
    const int8_t *gt0, *gt1;
    uint64_t grow;
    __device__ __forceinline__ uint32_t byte(int x) const { return (uint8_t)(x < cr ? gt0 : gt1)[grow + (x < cr ? x : x - cr)]; }
};

// ---- 1. this frame's slices of the bit planes (staged by TMA, words [0, nwst) of each array) -> ONE bit string each for
//         B and N over both planes, so the parse and the literal emission walk from plane 0 into plane 1 without a seam.
//         Rows outside [r0, r0 + valid) belong to other chunks (or to nobody) and are masked off in the staging area.
//         Returns any_n; strN is written only when it is set.
__device__ __forceinline__ bool build_bit_strings(uint32_t *stage, uint32_t *strB, uint32_t *strN, int nwst, int strw, int alpha,
                                                  int valid, int cr) {
    const int lane = threadIdx.x & 31;
    const int sh = cr & 31, wsh = cr >> 5;       // plane 1 sits cr bits above plane 0 in the strings
    uint32_t nacc = 0;
    for (int w = lane; w < nwst; w += 32) {
        const uint32_t mk = low_mask(alpha + valid - 32 * w) & ~low_mask(alpha - 32 * w);
        uint32_t *gq = stage + (w >> 2) * kBitGroupWords + (w & 3);
        if (mk != 0xFFFFFFFFu) { gq[0] &= mk; gq[4] &= mk; gq[8] &= mk; gq[12] &= mk; }
        nacc |= gq[8] | gq[12];
    }
    const bool any_n = __any_sync(0xffffffffu, nacc != 0);
    __syncwarp();
    for (int k = lane; k < strw; k += 32) {
        const int j = k - wsh;
        uint32_t b = 0, b1lo = 0, b1hi = 0;
        if (k < nwst) b = stage[(k >> 2) * kBitGroupWords + (k & 3)];
        if (j >= 1 && j <= nwst) b1lo = stage[((j - 1) >> 2) * kBitGroupWords + 4 + ((j - 1) & 3)];
        if (j >= 0 && j < nwst) b1hi = stage[(j >> 2) * kBitGroupWords + 4 + (j & 3)];
        strB[k] = b | __funnelshift_l(b1lo, b1hi, sh);
        if (any_n) {
            uint32_t x = 0, x1lo = 0, x1hi = 0;
            if (k < nwst) x = stage[(k >> 2) * kBitGroupWords + 8 + (k & 3)];
            if (j >= 1 && j <= nwst) x1lo = stage[((j - 1) >> 2) * kBitGroupWords + 12 + ((j - 1) & 3)];
            if (j >= 0 && j < nwst) x1hi = stage[(j >> 2) * kBitGroupWords + 12 + (j & 3)];
            strN[k] = x | __funnelshift_l(x1lo, x1hi, sh);
        }
    }
    fence_proxy_async();                        // the staging area was masked in place: order that before the copy engine's writes
    __syncwarp();
    return any_n;
}

// what the parse of a lane's segment leaves for the scans and the emission
template <int NW>
struct LaneParse {
    uint32_t Rp[NW], K[NW];              // match cover without the last position of each run; C-run cover (match type)
    int m;                               // matches that start in the segment
    int matched;                         // positions covered by them
    int prev_end;                        // end of the last match (0: none)
    int first_lit;                       // literals in front of the first match
    int n_ext;                           // extension bytes of literal runs >= 15 and matches >= 19
    int trail;                           // literals behind the last match (carried into the next sequence)
};

// ---- 2. per-lane parse of the segment [x0, x0 + seg) of the block, position-parallel
template <int NW>
__device__ __forceinline__ void parse_lane(const AlleleBits &ab, int x0, int seg, LaneParse<NW> &P) {
    const uint32_t *strB = ab.strB, *strN = ab.strN;
    const bool any_n = ab.any_n;
    const int cr = ab.cr, n = 2 * cr;
    const int seglen = max(0, min(seg, n - x0));
    const int mlim = min(seglen, n - 11 - x0);                    // the last 11 bytes of the block stay literals
    const int bi = ab.alpha + x0, j0 = bi >> 5, shb = bi & 31;
    const int ci = bi - cr, jc = ci >> 5, shc = ci & 31;          // the same rows in plane 0 (positions >= cr only)
    uint32_t Z[NW], C[NW], ZR[NW], S[NW], E[NW];
#pragma unroll
    for (int k = 0; k < NW; ++k) {
        const uint32_t bw = __funnelshift_r(strB[j0 + k], strB[j0 + k + 1], shb);
        const uint32_t nw = any_n ? __funnelshift_r(strN[j0 + k], strN[j0 + k + 1], shb) : 0u;
        const uint32_t vm = low_mask(mlim - 32 * k);
        Z[k] = ~(bw | nw) & vm;
        C[k] = 0;
        const uint32_t cm = vm & ~low_mask(cr - x0 - 32 * k);     // the word's positions in plane 1
        if (cm) {                                                 // (then jc + k >= -1: the zero words in front)
            const uint32_t b0w = __funnelshift_r(strB[jc + k], strB[jc + k + 1], shc);
            const uint32_t n0w = any_n ? __funnelshift_r(strN[jc + k], strN[jc + k + 1], shc) : 0u;
            C[k] = ~((bw ^ b0w) | nw | n0w) & cm;
        }
    }
    runs_cover<NW, kMinZ>(Z, ZR);
#pragma unroll
    for (int k = 0; k < NW; ++k) C[k] &= ~ZR[k];
    runs_cover<NW, kMinC>(C, P.K);        // K = the C-run cover: a match that starts on a K bit copies from plane 0
    int m = 0, matched = 0;
#pragma unroll
    for (int k = 0; k < NW; ++k) {
        const uint32_t zp = k > 0 ? ZR[k - 1] : 0u, zn = k + 1 < NW ? ZR[k + 1] : 0u;
        const uint32_t cp = k > 0 ? P.K[k - 1] : 0u, cn = k + 1 < NW ? P.K[k + 1] : 0u;
        S[k] = (ZR[k] & ~__funnelshift_l(zp, ZR[k], 1)) | (P.K[k] & ~__funnelshift_l(cp, P.K[k], 1));
        E[k] = (ZR[k] & ~__funnelshift_r(ZR[k], zn, 1)) | (P.K[k] & ~__funnelshift_r(P.K[k], cn, 1));
        m += __popc(S[k]);
        matched += __popc(ZR[k] | P.K[k]);
    }
    // size of the lane's output from popcounts: 3 bytes per match + its literals + one extension byte per
    // literal run >= 15 (runs inside a segment are < 270) and per match >= 19 (a match is < 274 long)
    int prev_end = 0, first_lit = 0, n_ext = 0;
    if (m > 0) {
        bool f = false;
#pragma unroll
        for (int k = NW - 1; k >= 0; --k)
            if (!f && E[k]) { prev_end = 32 * k + 32 - __clz(E[k]); f = true; }
        f = false;
#pragma unroll
        for (int k = 0; k < NW; ++k)
            if (!f && S[k]) { first_lit = 32 * k + ctz32(S[k]); f = true; }
        // a match [st, en] is >= 19 long iff no end bit lies in [st, st + 17]
        uint32_t e1[NW], w[NW];
        or_shr<NW>(E, 1, e1);
        or_shr<NW>(e1, 2, w);
        or_shr<NW>(w, 4, w);
        or_shr<NW>(w, 8, w);
#pragma unroll
        for (int k = 0; k < NW; ++k) n_ext += __popc(S[k] & ~(w[k] | shr_word<NW>(e1, k, 16)));
        // the literal run after end bit e (not the last one: that run is carried) is >= 15 long iff no start
        // bit lies in [e + 1, e + 15]
        uint32_t s1[NW], s2[NW], s3[NW];
        or_shr<NW>(S, 1, s1);
        or_shr<NW>(s1, 2, s2);
        or_shr<NW>(s2, 4, s3);
#pragma unroll
        for (int k = 0; k < NW; ++k) {
            uint32_t ek = E[k];
            if (32 * k <= prev_end - 1 && prev_end - 1 < 32 * k + 32) ek &= ~(1u << ((prev_end - 1) & 31));
            const uint32_t near = shr_word<NW>(s3, k, 1) | shr_word<NW>(s2, k, 9) | shr_word<NW>(s1, k, 13) | shr_word<NW>(S, k, 15);
            n_ext += __popc(ek & ~near);
        }
    }
    P.m = m; P.matched = matched; P.prev_end = prev_end; P.first_lit = first_lit; P.n_ext = n_ext;
    P.trail = seglen - prev_end;
    // runs of Rp are separated by at least one zero even where a Z run touches a C run, so "lowest run" arithmetic
    // enumerates the matches in step 5
#pragma unroll
    for (int k = 0; k < NW; ++k) P.Rp[k] = (ZR[k] | P.K[k]) & ~E[k];
}

// ---- 3. carry trailing literals forward (lane 0 takes carry_in, the literals in front of the warp's first segment);
//         scan: output offsets.  Gives this lane's carried literals, the literals the warp leaves behind its last
//         match (carry_out), where the lane's output starts and the bytes the whole warp writes.
template <int NW>
__device__ __forceinline__ void scan_offsets(const LaneParse<NW> &P, int carry_in, int &carry, int &carry_out, int &out_base,
                                             int &total) {
    const int lane = threadIdx.x & 31;
    int val = P.trail + (lane == 0 && P.m == 0 ? carry_in : 0), flag = P.m > 0;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int v2 = __shfl_up_sync(0xffffffffu, val, d), f2 = __shfl_up_sync(0xffffffffu, flag, d);
        if (lane >= d && !flag) { val += v2; flag = f2; }
    }
    carry = __shfl_up_sync(0xffffffffu, val, 1);
    if (lane == 0) carry = carry_in;
    carry_out = __shfl_sync(0xffffffffu, val, 31);
    const int mysize = P.m > 0 ? 3 * P.m + (P.prev_end - P.matched) + carry + lit_ext(P.first_lit + carry) + P.n_ext : 0;
    int inc = mysize;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int t1 = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += t1;
    }
    total = __shfl_sync(0xffffffffu, inc, 31);
    out_base = inc - mysize;
}

// ---- 5. emission of the lane's sequences at shared address waddr.  Every lane walks its own byte stream -- per
//         sequence: token [+ length bytes], literals (rebuilt from the bits), offset [+ length byte] -- in passes of at
//         most 8 bytes, all lanes in step: a flat state machine, so a lane with a long literal run does not hold up the
//         others' next sequence.  The bytes of a pass are gathered in a 64-bit value and appended to the lane's region of
//         the tail buffer through a 64-bit accumulator; a lane's first and last 8-byte word may be shared with its
//         neighbours: those two are OR-ed into the zeroed buffer at the end, everything between is stored plainly.
//         `closes`: this lane also writes the token and length bytes of the block's last, literals-only sequence of
//         final_lit literals (>= 11 of them); the literals themselves are written by closing_literals.
template <int NW>
__device__ __forceinline__ void emit_lane(uint32_t waddr, LaneParse<NW> &P, int x0, int carry, bool closes, int final_lit,
                                          const AlleleBits &ab) {
    uint32_t (&Rp)[NW] = P.Rp;
    uint32_t (&K)[NW] = P.K;
    const int cr = ab.cr;
    uint32_t fill = waddr & 7u;                      // bytes of the accumulator in use
    waddr &= ~7u;
    const uint32_t faddr = waddr;
    uint64_t acc = 0, fw = 0;
    uint32_t first = 1;                              // the first word is still being filled: nothing stored yet
    auto put = [&](uint64_t v, uint32_t nb) {        // append the low nb (<= 8) bytes of v; the bytes above must be zero
        const uint32_t sh = 8u * fill;
        acc |= v << sh;
        const uint64_t spill = (v >> 1) >> (63u - sh);            // = v >> (64 - sh), 0 for sh == 0
        fill += nb;
        const bool full = fill >= 8u;
        if (full && !first) sts64(waddr, acc);
        fw = (full && first) ? acc : fw;
        first = full ? 0u : first;
        waddr += full ? 8u : 0u;
        acc = full ? spill : acc;
        fill -= full ? 8u : 0u;
    };
    // up to 8 literal bytes of block positions x .. x + nb - 1
    auto lit8 = [&](int x, int nb) -> uint64_t {
        const int G = ab.alpha + x;
        const uint32_t keep = (1u << nb) - 1u;
        const uint32_t bits = __funnelshift_r(ab.strB[G >> 5], ab.strB[(G >> 5) + 1], G) & keep;
        uint64_t v = (uint64_t)spread4(bits) | ((uint64_t)spread4(bits >> 4) << 32);
        if (ab.any_n) {
            uint32_t nb8 = __funnelshift_r(ab.strN[G >> 5], ab.strN[(G >> 5) + 1], G) & keep;
#pragma unroll 1
            while (nb8) {                            // an allele other than 0 / 1: the byte itself
                const int i = ctz32(nb8);
                nb8 &= nb8 - 1;
                const uint64_t byte = ab.byte(x + i);
                v = (v & ~(0xFFull << (8 * i))) | (byte << (8 * i));
            }
        }
        return v;
    };
    int pos = x0 - carry;                            // next block position that has not been emitted
    int base = x0;                                   // block position of bit 0 of Rp[0]
    int left = P.m;                                  // matches still to start
    uint32_t fin = closes ? 1u : 0u;
    int litrem = 0, cur_ml = 0;
    uint32_t cur_off = 0, pend = 0;                  // pend: the current sequence's offset has not been emitted yet
    while ((left | litrem | (int)pend | (int)fin) != 0) {
        uint64_t v = 0;
        uint32_t nb = 0;
        if ((litrem | (int)pend) == 0) {             // the next sequence starts
            int lit;
            uint32_t tok;
            if (left > 0) {
                // matches are taken in order: whole words that are used up move out (at most NW - 1 times)
#pragma unroll
                for (int r = 0; r + 1 < NW; ++r) {
                    const bool z = Rp[0] == 0u;
#pragma unroll
                    for (int k = 0; k + 1 < NW; ++k) { Rp[k] = z ? Rp[k + 1] : Rp[k]; K[k] = z ? K[k + 1] : K[k]; }
                    Rp[NW - 1] = z ? 0u : Rp[NW - 1];
                    base += z ? 32 : 0;
                }
                // lowest run of Rp: low = its first bit, Rp + low carries through the run (and on into the next words)
                const uint32_t low = Rp[0] & (0u - Rp[0]);
                const int ts = __popc(low - 1u);
                const bool is_k = (K[0] & low) != 0u;
                uint64_t cy = low;
                int ml = 1;
#pragma unroll
                for (int k = 0; k < NW; ++k) {
                    cy += Rp[k];
                    const uint32_t t = (uint32_t)cy;
                    cy >>= 32;
                    ml += __popc(Rp[k] & ~t);
                    Rp[k] &= t;
                }
                lit = base + ts - pos;
                cur_ml = ml;
                cur_off = is_k ? (uint32_t)cr : 2u * (uint32_t)cr;
                pend = 1;
                --left;
                tok = (uint32_t)((min(lit, 15) << 4) | min(ml - 4, 15));
            } else {                                 // the last sequence of the block: literals only
                lit = final_lit;
                fin = 0;
                tok = (uint32_t)(min(lit, 15) << 4);
            }
            v = tok; nb = 1;
            if (lit >= 15) {
                int rem = lit - 15;
#pragma unroll 1
                while (rem >= 255) { put(v, nb); v = 255u; nb = 1; rem -= 255; }
                v |= (uint64_t)(uint32_t)rem << (8u * nb);
                ++nb;
            }
            litrem = pend ? lit : 0;
        }
        const int take = min(litrem, 8 - (int)nb);
        if (take > 0) {
            v |= lit8(pos, take) << (8u * nb);
            nb += (uint32_t)take; pos += take; litrem -= take;
        }
        if (pend != 0 && litrem == 0) {
            const uint32_t ob = cur_ml >= 19 ? 3u : 2u;
            if (nb + ob <= 8u) {
                v |= (uint64_t)(cur_off | (cur_ml >= 19 ? (uint32_t)(cur_ml - 19) << 16 : 0u)) << (8u * nb);
                nb += ob; pend = 0; pos += cur_ml;
            }
        }
        put(v, nb);
    }
    const uint64_t fv = first ? acc : fw;
    if ((uint32_t)fv) sts_or32(faddr, (uint32_t)fv);
    if ((uint32_t)(fv >> 32)) sts_or32(faddr + 4u, (uint32_t)(fv >> 32));
    if (!first) {
        if ((uint32_t)acc) sts_or32(waddr, (uint32_t)acc);
        if ((uint32_t)(acc >> 32)) sts_or32(waddr + 4u, (uint32_t)(acc >> 32));
    }
}

// the block's closing literals -- its last final_lit positions (>= 11, and all the positions no lane owns) -- to fdst:
// one byte per lane and step
__device__ __forceinline__ void closing_literals(uint8_t *fdst, int final_lit, const AlleleBits &ab) {
    const int fx = 2 * ab.cr - final_lit;
    for (int i = threadIdx.x & 31; i < final_lit; i += 32) {
        const int x = fx + i, G = ab.alpha + x;
        uint32_t byte = (ab.strB[G >> 5] >> (G & 31)) & 1u;
        if (ab.any_n && ((ab.strN[G >> 5] >> (G & 31)) & 1u)) byte = ab.byte(x);
        fdst[i] = (uint8_t)byte;
    }
}

template <int NW>
__global__ void __launch_bounds__(kWpc * 32) donor_frames_kernel(const FusedArgs A) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t c = blockIdx.x / A.groups, grp = blockIdx.x - c * A.groups;
    const int cr = (int)A.cr, n = 2 * cr;
    uint64_t *tbar = reinterpret_cast<uint64_t *>(smem);
    uint8_t *tmpl_s = smem + 16;
    uint8_t *wbase = smem + 16 + A.tmpl_smem + (size_t)warp * A.warp_smem;
    uint64_t *wbar = reinterpret_cast<uint64_t *>(wbase);
    uint32_t *stage = reinterpret_cast<uint32_t *>(wbase + 16);
    uint32_t *strB = reinterpret_cast<uint32_t *>(wbase + 16 + A.stg_bytes) + 4;      // 4 zero words in front of each string:
    uint32_t *strN = strB + A.strw + 4;                                                //   word -1 may be read (step 2)
    uint8_t *outb = reinterpret_cast<uint8_t *>(strN + A.strw);

    const uint32_t tl = A.tmpl_len[c];
    const uint32_t tl16 = tl & ~15u, sh16 = tl & 15u;
    if (threadIdx.x == 0) mbar_init(tbar, 1);
    if (lane == 0) mbar_init(wbar, 1);
    if (lane < 4) { strB[lane - 4] = 0; strN[lane - 4] = 0; }
    mbar_fence_init();
    __syncthreads();
    if (threadIdx.x == 0) {            // the chunk's template: once per CTA, by TMA
        const uint32_t bytes = (tl + 15u) & ~15u;
        mbar_expect_tx(tbar, bytes);
        tma_load_1d(tmpl_s, A.tmpl + (size_t)c * A.tmpl_cap, bytes, tbar);
    }
    const uint32_t s_end = min(A.n_samples, (grp + 1) * A.gs);
    uint32_t s = grp * A.gs + warp;
    if (s >= s_end) return;

    const uint64_t r0 = (uint64_t)c * (uint64_t)cr;
    const int valid = (int)min((uint64_t)cr, A.n_records - r0);       // rows past n_records read as zero (HDF5 edge chunk)
    const int alpha = (int)(r0 & 127);                                 // block position x is bit alpha + x of the strings
    const bool raw = cr < 6;                                           // see site_template_kernel
    // the 128-row groups of the bit planes that hold rows [r0, r0 + valid)
    const uint32_t g0 = (uint32_t)(r0 >> 7);
    const uint32_t ngrp = (uint32_t)((r0 + (uint64_t)valid - 1) >> 7) - g0 + 1;
    const uint32_t stg = ngrp * (kBitGroupWords * 4);
    const int nwst = 4 * (int)ngrp;                                    // staged words per array
    if (!raw && lane == 0) {
        mbar_expect_tx(wbar, stg);
        tma_load_1d(stage, A.bits + (uint64_t)(A.s0 + s) * A.bits_stride + (uint64_t)g0 * kBitGroupWords, stg, wbar);
    }
    uint32_t phase = 0;
    bool tmpl_ready = false;
    const unsigned long long row_stride = A.slot_off[A.n_chunks], slot = A.slot_off[c];

    for (; s < s_end; s += kWpc) {
        // read per frame, not hoisted out of the loop: kept live across it they cost NW >= 5 some 40 registers
        const int seg = (int)A.seg;                  // block positions per lane: lane i owns [i * seg, (i + 1) * seg)
        const int x0 = lane * seg;
        AlleleBits ab{strB, strN, false, alpha, cr, A.gt0, A.gt1, (uint64_t)(A.s0 + s) * A.gt_stride + r0};
        LaneParse<NW> P;
        int dlen = n, carry = 0, out_base = 0, final_lit = 0;
        if (!raw) {
            mbar_wait(wbar, phase);
            phase ^= 1;
            ab.any_n = build_bit_strings(stage, strB, strN, nwst, (int)A.strw, alpha, valid, cr);
            if (lane == 0 && s + kWpc < s_end) {        // the next frame's slices: one TMA bulk copy, a whole frame ahead
                mbar_expect_tx(wbar, stg);
                tma_load_1d(stage, A.bits + (uint64_t)(A.s0 + s + kWpc) * A.bits_stride + (uint64_t)g0 * kBitGroupWords, stg, wbar);
            }
            parse_lane<NW>(ab, x0, seg, P);
            int total;
            scan_offsets<NW>(P, 0, carry, final_lit, out_base, total);
            final_lit += max(0, n - 32 * seg);           // + the positions no lane owns (FusedArgs::seg)
            dlen = total + 1 + lit_ext(final_lit) + final_lit;
        }

        // ---- 4. the tail buffer: zeroed (neighbouring lanes OR their shared boundary words together), lined up with
        //         the template's end modulo 16 so that the frame leaves as 16-byte aligned bulk copies
        if (lane == 0) tma_store_wait_read();           // the previous frame's bulk store has read the buffer
        __syncwarp();
        {
            const int nz = (int)((sh16 + (uint32_t)dlen + 15u) >> 4);
            for (int i = lane; i < nz; i += 32) reinterpret_cast<uint4 *>(outb)[i] = make_uint4(0, 0, 0, 0);
        }
        if (!tmpl_ready) { mbar_wait(tbar, 0); tmpl_ready = true; }
        __syncwarp();
        if ((uint32_t)lane < sh16) outb[lane] = tmpl_s[tl16 + lane];      // the template's last, partial 16 bytes
        __syncwarp();
        uint8_t *seq = outb + sh16;

        if (raw) {
            for (int i = lane; i < n; i += 32) {
                const int x = i < cr ? i : i - cr;
                seq[i] = x < valid ? (uint8_t)ab.byte(i) : (uint8_t)0;
            }
        } else {
            emit_lane<NW>(smem_u32(seq) + (uint32_t)out_base, P, x0, carry, lane == 31, final_lit, ab);
            __syncwarp();
            closing_literals(seq + (dlen - final_lit), final_lit, ab);
        }
        fence_proxy_async();                 // the tail buffer is read by the bulk-copy engine next
        __syncwarp();

        // ---- 6. the frame leaves: 2 header vectors (size fields filled in) + template body + own tail by TMA bulk stores
        const uint32_t flen = tl + (uint32_t)dlen;               // = cbytes of the Blosc chunk header
        const uint32_t lz = flen - TMPL_HDR;                     // = csize of the block's stream
        uint8_t *dst = A.frames + (unsigned long long)(s) * row_stride + slot;
        if (tl16 >= 32) {
            if (lane < 2) {
                uint4 v = reinterpret_cast<const uint4 *>(tmpl_s)[lane];
                if (lane == 0) v.w = flen; else v.y = lz;
                stg_stream(reinterpret_cast<uint4 *>(dst) + lane, v);
            }
            if (lane == 0) {
                if (tl16 > 32) tma_store_1d(dst + 32, tmpl_s + 32, tl16 - 32);
                tma_store_1d(dst + tl16, outb, (sh16 + (uint32_t)dlen + 15u) & ~15u);
                tma_store_commit();
            }
        } else {                             // a template shorter than its two header vectors (tiny chunks): byte by byte
            for (uint32_t i = lane; i < flen; i += 32) {
                uint32_t b = i < tl ? tmpl_s[i] : seq[i - tl];
                if (i >= 12 && i < 16) b = (flen >> (8 * (i - 12))) & 0xFFu;
                if (i >= 20 && i < 24) b = (lz >> (8 * (i - 20))) & 0xFFu;
                dst[i] = (uint8_t)b;
            }
        }
        if (lane == 0) A.size[(uint64_t)s * A.n_chunks + c] = flen;
    }
    if (lane == 0) tma_store_wait_read();    // shared memory must outlive the bulk stores that read it
}

// ------------------------------------------------------------------------------------------
// Kernel 4b-L: the allele tails of chunks of kSmallChunkMax < cr <= kMaxChunkRecords records.  Shared with
// donor_frames_kernel: the bit strings, the lane parse, the offset scans, the emission and the closing literals, so the
// frames are built by the same rules (Z and C match sources at offsets 2 * cr and cr, the same closing literals) and
// the slot bound (template + 2 cr + 2 cr / 255 + 24) still holds.  What differs:
//   - the parse, scans and emission run in PASSES of 32 lanes x 32 * NW block positions; the literals a pass leaves at
//     its end are carried into the first sequence of the next pass exactly as a lane carries them into the next lane's,
//     and lane 31 of the last pass closes the block;
//   - the template is NOT staged in shared memory (a chunk with high-entropy sites makes a template of up to ~24 * cr
//     bytes): the warp copies its body from global memory (L2-resident: every warp of the chunk reads the same bytes);
//   - shared memory per warp = bit-plane staging + the two bit strings + the whole tail buffer, zeroed up front because
//     the tail's length is known only after the last pass.
// ------------------------------------------------------------------------------------------
constexpr int kLargeNW = 4;                   // mask words per lane and pass: 4,096 block positions per pass
constexpr int kWpcL = 4;                      // warps per CTA: 2-6 CTAs per SM from cr 7,489 down to 2,731

// __maxnreg__(96) instead of __launch_bounds__: with the bounds alone ptxas settles on 64 registers and spills
template <int NW>
__global__ void __maxnreg__(96) donor_frames_large_kernel(const FusedArgs A) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t c = blockIdx.x / A.groups, grp = blockIdx.x - c * A.groups;
    const int cr = (int)A.cr, n = 2 * cr;
    uint8_t *wbase = smem + (size_t)warp * A.warp_smem;
    uint64_t *wbar = reinterpret_cast<uint64_t *>(wbase);
    uint32_t *stage = reinterpret_cast<uint32_t *>(wbase + 16);
    uint32_t *strB = reinterpret_cast<uint32_t *>(wbase + 16 + A.stg_bytes) + 4;      // 4 zero words in front of each string
    uint32_t *strN = strB + A.strw + 4;
    uint8_t *outb = reinterpret_cast<uint8_t *>(strN + A.strw);
    const uint8_t *tmpl = A.tmpl + (size_t)c * A.tmpl_cap;

    const uint32_t tl = A.tmpl_len[c];
    const uint32_t tl16 = tl & ~15u, sh16 = tl & 15u;                  // tl >= TMPL_HDR: tl16 >= 16
    const uint32_t s_end = min(A.n_samples, (grp + 1) * A.gs);
    uint32_t s = grp * A.gs + warp;
    if (s >= s_end) return;
    if (lane == 0) mbar_init(wbar, 1);
    if (lane < 4) { strB[lane - 4] = 0; strN[lane - 4] = 0; }
    mbar_fence_init();
    __syncwarp();

    const uint64_t r0 = (uint64_t)c * (uint64_t)cr;
    const int valid = (int)min((uint64_t)cr, A.n_records - r0);
    const int alpha = (int)(r0 & 127);
    const uint32_t g0 = (uint32_t)(r0 >> 7);
    const uint32_t ngrp = (uint32_t)((r0 + (uint64_t)valid - 1) >> 7) - g0 + 1;
    const uint32_t stg = ngrp * (kBitGroupWords * 4);
    const int nwst = 4 * (int)ngrp;
    if (lane == 0) {
        mbar_expect_tx(wbar, stg);
        tma_load_1d(stage, A.bits + (uint64_t)(A.s0 + s) * A.bits_stride + (uint64_t)g0 * kBitGroupWords, stg, wbar);
    }
    uint32_t phase = 0;
    const unsigned long long row_stride = A.slot_off[A.n_chunks], slot = A.slot_off[c];
    constexpr int seg = 32 * NW;                 // block positions per lane and pass
    const int npass = (n + 32 * seg - 1) / (32 * seg);

    for (; s < s_end; s += kWpcL) {
        AlleleBits ab{strB, strN, false, alpha, cr, A.gt0, A.gt1, (uint64_t)(A.s0 + s) * A.gt_stride + r0};
        mbar_wait(wbar, phase);
        phase ^= 1;
        ab.any_n = build_bit_strings(stage, strB, strN, nwst, (int)A.strw, alpha, valid, cr);
        if (lane == 0 && s + kWpcL < s_end) {
            mbar_expect_tx(wbar, stg);
            tma_load_1d(stage, A.bits + (uint64_t)(A.s0 + s + kWpcL) * A.bits_stride + (uint64_t)g0 * kBitGroupWords, stg, wbar);
        }
        // the tail buffer: zeroed whole, the template's last partial 16 bytes in front
        if (lane == 0) tma_store_wait_read();           // the previous frame's bulk store has read the buffer
        __syncwarp();
        for (uint32_t i = lane; i < A.outcap / 16u; i += 32) reinterpret_cast<uint4 *>(outb)[i] = make_uint4(0, 0, 0, 0);
        __syncwarp();
        if ((uint32_t)lane < sh16) outb[lane] = tmpl[tl16 + lane];
        __syncwarp();
        uint8_t *seq = outb + sh16;

        int carry_in = 0, pass_base = 0;             // carry_in: literals the passes so far leave behind their last match
        for (int q = 0; q < npass; ++q) {
            const int x0 = q * 32 * seg + lane * seg;
            LaneParse<NW> P;
            parse_lane<NW>(ab, x0, seg, P);
            int carry, out_base, total;
            scan_offsets<NW>(P, carry_in, carry, carry_in, out_base, total);
            emit_lane<NW>(smem_u32(seq) + (uint32_t)(pass_base + out_base), P, x0, carry, lane == 31 && q == npass - 1, carry_in, ab);
            pass_base += total;
        }
        const int final_lit = carry_in;
        const int dlen = pass_base + 1 + lit_ext(final_lit) + final_lit;
        __syncwarp();
        closing_literals(seq + (dlen - final_lit), final_lit, ab);
        // ---- 6. the frame leaves: header + template body from global memory (size fields filled in), own tail by a
        //         TMA bulk store.  A size field that lies behind tl16 sits in the tail buffer's first bytes.
        const uint32_t flen = tl + (uint32_t)dlen;
        const uint32_t lz = flen - TMPL_HDR;
        if (lane == 0 && tl16 < 24) for (int i = 0; i < 4; ++i) outb[20 - tl16 + i] = (uint8_t)(lz >> (8 * i));
        fence_proxy_async();
        __syncwarp();
        uint8_t *dst = A.frames + (unsigned long long)(s) * row_stride + slot;
        for (uint32_t k = lane; k < tl16 / 16u; k += 32) {
            uint4 v = __ldg(reinterpret_cast<const uint4 *>(tmpl) + k);
            if (k == 0) v.w = flen;
            if (k == 1) v.y = lz;
            stg_stream(reinterpret_cast<uint4 *>(dst) + k, v);
        }
        if (lane == 0) {
            tma_store_1d(dst + tl16, outb, (sh16 + (uint32_t)dlen + 15u) & ~15u);
            tma_store_commit();
            A.size[(uint64_t)s * A.n_chunks + c] = flen;
        }
    }
    if (lane == 0) tma_store_wait_read();    // shared memory must outlive the bulk stores that read it
}

__global__ void __launch_bounds__(256) sum_sizes_kernel(const uint32_t *__restrict__ size, uint64_t n, unsigned long long *__restrict__ total) {
    unsigned long long acc = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) acc += size[i];
#pragma unroll
    for (int d = 16; d; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(total, acc);
}

// Frames out of their slots, packed back to back (16-byte aligned) into one piece of the packed image: one warp per
// frame, 16-byte vectors.  slot of frame i = (i / n_chunks) * row_stride + slot_off[i % n_chunks]; packed_off = where the
// frame starts in the packed image, piece_base = where this piece starts.
__global__ void __launch_bounds__(256)
pack_frames_kernel(const uint8_t *__restrict__ frames, const uint64_t *__restrict__ slot_off, uint64_t n_chunks,
                   const uint32_t *__restrict__ size, const uint64_t *__restrict__ packed_off, uint64_t first, uint64_t count,
                   uint64_t piece_base, uint8_t *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const uint64_t w = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (w >= count) return;
    const uint64_t i = first + w;
    const uint64_t s = i / n_chunks, c = i - s * n_chunks;
    const uint4 *src = reinterpret_cast<const uint4 *>(frames + s * slot_off[n_chunks] + slot_off[c]);
    uint4 *dst = reinterpret_cast<uint4 *>(out + (packed_off[i] - piece_base));
    const uint32_t nv = (size[i] + 15u) >> 4;              // the slot is zero behind the frame up to the next 16-byte boundary
    for (uint32_t k = lane; k < nv; k += 32) stg_stream(dst + k, ldg_stream(src + k));
}

// The donor-specific bytes of frames [first, first + count): a stored chunk is the chunk's template with its first 32
// bytes patched (size fields) and its own tail behind it, so only the 32 header bytes and the tail -- from the last 16-byte
// boundary of the template on -- have to leave the GPU per donor; the template goes once per chunk.  Tails are packed
// back to back (16-byte units, tail_off), the headers follow them.  One warp per frame.
__global__ void __launch_bounds__(256)
pack_tails_kernel(const uint8_t *__restrict__ frames, const uint64_t *__restrict__ slot_off, uint64_t n_chunks,
                  const uint32_t *__restrict__ size, const uint32_t *__restrict__ tmpl_len, const uint64_t *__restrict__ tail_off,
                  uint64_t first, uint64_t count, uint64_t piece_base, uint8_t *__restrict__ out_tails, uint4 *__restrict__ out_hdr) {
    const int lane = threadIdx.x & 31;
    const uint64_t w = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (w >= count) return;
    const uint64_t i = first + w;
    const uint64_t s = i / n_chunks, c = i - s * n_chunks;
    const uint8_t *slot = frames + s * slot_off[n_chunks] + slot_off[c];
    const uint32_t tl16 = tmpl_len[c] & ~15u, sz = size[i];
    const uint32_t nv = sz > tl16 ? (sz - tl16 + 15u) >> 4 : 0u;       // the slot is zero behind the frame up to the next 16-byte boundary
    const uint4 *src = reinterpret_cast<const uint4 *>(slot + tl16);
    uint4 *dst = reinterpret_cast<uint4 *>(out_tails + (tail_off[i] - piece_base));
    for (uint32_t k = lane; k < nv; k += 32) stg_stream(dst + k, ldg_stream(src + k));
    if (lane < 2) out_hdr[2 * w + lane] = ldg_stream(reinterpret_cast<const uint4 *>(slot) + lane);
}

uint64_t guess_chunk_records(uint64_t n) {      // h5py/_hl/filters.py guess_chunk for shape (n,), 35-byte items
    const double CHUNK_BASE = 16 * 1024, CHUNK_MIN = 8 * 1024, CHUNK_MAX = 1024 * 1024;
    if (n == 0) return 1;
    double chunk = (double)n;
    const double dset_size = chunk * 35.0;
    double target = CHUNK_BASE * std::pow(2.0, std::log10(dset_size / (1024.0 * 1024.0)));
    if (target > CHUNK_MAX) target = CHUNK_MAX;
    else if (target < CHUNK_MIN) target = CHUNK_MIN;
    for (;;) {
        const double bytes = chunk * 35.0;
        if ((bytes < target || std::fabs(bytes - target) / target < 0.5) && bytes < CHUNK_MAX) break;
        if (chunk == 1) break;
        chunk = std::ceil(chunk / 2.0);
    }
    return (uint64_t)chunk;
}

}  // namespace hb

using namespace hb;

struct hb_frames {
    int device = 0;
    cudaStream_t stream = nullptr;
    uint64_t n_records = 0, n_chunks = 0, cr = 0;
    uint64_t chunk_cap = 0;                  // chunks the per-chunk arrays were allocated for
    bool cr_explicit = false;                // chunk_records was given by the caller (it does not follow n_records)
    uint32_t n_samples = 0, tmpl_cap = 0;    // n_samples: samples of the current window
    uint32_t s0 = 0, win_cap = 0;            // window = samples [s0, s0 + n_samples) of the parse; win_cap = allocated for
    size_t smem_site = 0;
    FusedArgs fa;                            // geometry of the fused kernel
    int nw = 1;
    bool large = false;                      // cr > kSmallChunkMax: kernels 4a-L / 4b-L
    uint8_t *d_site_scratch = nullptr;       // 4a-L: site_large_scratch(cr) bytes per CTA
    uint32_t site_ctas = 0;                  // 4a-L: CTAs the scratch was made for
    uint8_t *d_tmpl = nullptr, *d_frames = nullptr;
    uint32_t *d_tmpl_len = nullptr, *d_size = nullptr;
    uint64_t *d_slot_off = nullptr;
    unsigned long long *d_totals = nullptr;
    std::vector<uint64_t> h_slot_off;            // [n_chunks + 1]
    uint64_t frames_cap = 0;
    uint64_t total_bytes = 0, padded_bytes = 0;
    std::vector<uint32_t> h_tmpl_len;
    // host copies of the layout, fetched on demand
    bool layout_valid = false;
    std::vector<uint32_t> h_size;                // [n_samples][n_chunks]
    std::vector<uint8_t> h_row;                  // scratch for hb_frames_fetch_sample
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
    float ms_site = 0, ms_frames = 0;
    // the site templates only need the site columns, not the genotype planes: when the frames are attached to
    // their parse (hb_parse_attach_frames) the template kernel runs on `side`, concurrently with the GT decoder
    cudaStream_t side = nullptr;
    cudaEvent_t ev_sites = nullptr, ev_tmpl = nullptr, ev_side0 = nullptr;
    bool early_site = false;                     // the template pass of the current parse run is already in flight
    uint64_t last_d2h_bytes = 0;                 // bytes the last hb_frames_fetch_packed moved device -> host
    // frames launched from inside run_parse, right behind the GT decoder (frames_early_launch): hb_frames_rerun only collects
    bool launched = false;
    bool totals_valid = false;                   // total_bytes is summed when somebody asks (hb_frames_get_info)
    uint64_t launched_run = 0, pending_need = 0;
    bool pending_was_early = false;
};

// More than 48 KB of dynamic shared memory is opt-in per function AND per device.  The ceiling is always raised to the
// device maximum (never to the size of one launch), so that concurrent callers cannot shrink each other's limit, and on
// every launch (a microsecond), so that a process that moves to another device is served too.
static void raise_smem_limit(const void *func) {
    int dev = 0, smem_max = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max - 1024);
}

template <int NW>
static void launch_donor_frames(const FusedArgs &fa, uint64_t n_ctas, cudaStream_t st) {
    const size_t smem = 16 + (size_t)fa.tmpl_smem + (size_t)kWpc * fa.warp_smem;
    raise_smem_limit(reinterpret_cast<const void *>(donor_frames_kernel<NW>));
    donor_frames_kernel<NW><<<(unsigned)n_ctas, kWpc * 32, smem, st>>>(fa);
}

// The frame buffer is many GB and cudaMalloc / cudaFree of that size cost ~100 ms (and cudaFree synchronises the device):
// released buffers are kept, two per device, for the next frames handles of the process: a converter walks 22 chromosomes
// and parses + compresses one file ahead of the one whose frames are leaving, so two handles are alive at a time (with one
// kept buffer every file paid a cudaMalloc and a device-synchronising cudaFree of 18 GB: the stalls of r02j's trace).
// hb_cache_clear() gives them back.
namespace {
struct BufCache { uint8_t *p = nullptr; uint64_t cap = 0; };
constexpr int kKeptBuffers = 2;
std::mutex g_fb_mu;
BufCache g_fb[64][kKeptBuffers];
}
namespace hb {
void frames_buffer_cache_clear() {
    std::lock_guard<std::mutex> lk(g_fb_mu);
    for (int d = 0; d < 64; ++d)
        for (auto &c : g_fb[d])
            if (c.p) { cudaSetDevice(d); cudaFree(c.p); c = BufCache(); }
}
}

static std::atomic<int> g_site_deep{0};
extern "C" void hb_set_site_matcher(int deep) { g_site_deep.store(deep ? 1 : 0); }

// templates of all chunks.  early: launched from inside run_parse on the side stream, right after the site columns
// were written on the parse's stream; otherwise on the parse's stream itself.
static int frames_site_pass(hb_frames *f, hb_parse *p, bool early) {
    cudaError_t e;
#define CUF(x) do { e = (x); if (e != cudaSuccess) return api_fail(HB_ERR_CUDA, std::string("CUDA: ") + cudaGetErrorString(e) + " at " #x); } while (0)
    SiteArgs4 sa;
    sa.chrom5 = p->rows.chrom5; sa.start = p->rows.start; sa.stop = p->rows.stop; sa.ref = p->rows.ref; sa.alt = p->rows.alt;
    sa.n_records = f->n_records; sa.cr = (uint32_t)f->cr; sa.tmpl = f->d_tmpl; sa.tmpl_cap = f->tmpl_cap; sa.tmpl_len = f->d_tmpl_len;
    sa.deep = g_site_deep.load() ? 1 : 0;
    cudaStream_t st = early ? f->side : f->stream;
    if (early) {
        CUF(cudaEventRecord(f->ev_sites, p->stream));
        CUF(cudaStreamWaitEvent(f->side, f->ev_sites, 0));
    }
    CUF(cudaEventRecord(early ? f->ev_side0 : f->ev[0], st));
    if (f->large) {
        site_template_large_kernel<<<(unsigned)std::min<uint64_t>(f->n_chunks, f->site_ctas), kSiteSegs * 32, f->smem_site, st>>>(sa, f->d_site_scratch);
    } else {
        raise_smem_limit(reinterpret_cast<const void *>(site_template_kernel));
        site_template_kernel<<<(unsigned)f->n_chunks, kSiteSegs * 32, f->smem_site, st>>>(sa);
    }
    count_launch();
    CUF(cudaEventRecord(early ? f->ev_tmpl : f->ev[1], st));
    f->early_site = early;
#undef CUF
    return HB_OK;
}

namespace hb {
// called by run_parse (hb_api.cu) once the site columns of this run are on their way
void frames_early_site_pass(void *frames, hb_parse *p) {
    hb_frames *f = static_cast<hb_frames *>(frames);
    if (!f || !f->n_chunks || !f->n_samples || !f->side) return;
    if (p->h_st.n_records != f->n_records || p->device != f->device) return;     // shape changed: hb_frames_rerun will say so
    frames_site_pass(f, p, true);
}
}  // namespace hb

// everything up to the launch of the frame kernel.  early: called from inside run_parse with the template pass in flight on
// the side stream and the GT decoder queued on the main one -- the host waits for the TEMPLATES only (their lengths size the
// slots), then queues the frame kernel behind the decoder: no idle GPU between the two.
static int frames_prepare(hb_frames *f, hb_parse *p, bool early) {
    cudaError_t e;
#define CUF(x) do { e = (x); if (e != cudaSuccess) return api_fail(HB_ERR_CUDA, std::string("CUDA: ") + cudaGetErrorString(e) + " at " #x); } while (0)
    CUF(cudaSetDevice(f->device));
    const uint64_t n = f->n_records;
    const uint32_t cr = (uint32_t)f->cr;
    f->layout_valid = false;
    f->totals_valid = false;
    const bool was_early = f->early_site;
    if (was_early) {
        CUF(cudaStreamWaitEvent(f->stream, f->ev_tmpl, 0));       // the templates were made while the decoder ran
        CUF(cudaEventRecord(f->ev[1], f->stream));
    } else {
        int rc = frames_site_pass(f, p, false);
        if (rc != HB_OK) return rc;
    }
    f->early_site = false;
    f->launched = false;
    // the frame buffer is sized from the longest template: frame <= template + worst-case allele tail
    cudaStream_t lens = early && was_early ? f->side : f->stream;
    CUF(cudaMemcpyAsync(f->h_tmpl_len.data(), f->d_tmpl_len, f->n_chunks * 4, cudaMemcpyDeviceToHost, lens));
    CUF(cudaStreamSynchronize(lens));
    CUF(cudaGetLastError());
    // slots: frame <= template + worst-case allele tail, so every address is known before the encode
    uint64_t need = 0;
    {
        const uint64_t tail = 2ull * cr + 2ull * cr / 255 + 24;
        uint64_t run = 0;
        for (uint64_t c = 0; c < f->n_chunks; ++c) { f->h_slot_off[c] = run; run += (f->h_tmpl_len[c] + tail + 15) & ~15ull; }
        f->h_slot_off[f->n_chunks] = run;
        need = run * f->n_samples;
    }
    bool regrow = false;
    if (f->frames_cap < need) {
        regrow = f->d_frames != nullptr;
        if (f->d_frames) { cudaFree(f->d_frames); f->d_frames = nullptr; f->frames_cap = 0; }
        if (f->device >= 0 && f->device < 64) {            // a buffer left behind by an earlier handle?
            std::lock_guard<std::mutex> lk(g_fb_mu);
            BufCache *best = nullptr;                       // the smallest kept buffer that is large enough
            for (auto &c : g_fb[f->device])
                if (c.p && c.cap >= need && (!best || c.cap < best->cap)) best = &c;
            if (best) { f->d_frames = best->p; f->frames_cap = best->cap; *best = BufCache(); }
        }
    }
    if (f->frames_cap < need) {
        // head-room: a re-run on other data (slab streaming) has slightly different template lengths, and growing
        // means cudaFree + cudaMalloc of many GB (~100 ms)
        const uint64_t cap = regrow ? need + need / 16 + (64ull << 20) : need + need / 64 + (16ull << 20);
        e = cudaMalloc(&f->d_frames, cap);
        if (e != cudaSuccess) { cudaGetLastError(); dev_pool_flush(); e = cudaMalloc(&f->d_frames, cap); }     // idle pooled buffers may hold what is missing
        if (e != cudaSuccess) return api_fail(HB_ERR_MEM, std::string("cudaMalloc of the frame buffer (") + std::to_string(cap) + " bytes): " + cudaGetErrorString(e));
        f->frames_cap = cap;
    }
    CUF(cudaMemcpyAsync(f->d_slot_off, f->h_slot_off.data(), (f->n_chunks + 1) * 8, cudaMemcpyHostToDevice, f->stream));
    FusedArgs fa = f->fa;
    fa.gt0 = p->d_gt[0]; fa.gt1 = p->d_gt[1]; fa.gt_stride = p->gt_stride; fa.n_records = n;
    fa.cr = cr; fa.n_samples = f->n_samples; fa.s0 = f->s0; fa.n_chunks = f->n_chunks;
    fa.tmpl = f->d_tmpl; fa.tmpl_cap = f->tmpl_cap; fa.tmpl_len = f->d_tmpl_len;
    fa.frames = f->d_frames; fa.slot_off = f->d_slot_off; fa.size = f->d_size;
    fa.bits = p->d_bits; fa.bits_stride = p->bits_stride;
    {
        uint32_t mx = 0;
        for (uint64_t c = 0; c < f->n_chunks; ++c) mx = std::max(mx, f->h_tmpl_len[c]);
        fa.tmpl_smem = f->large ? 0u : (mx + 15u) & ~15u;            // 4b-L reads the template from global memory
        fa.gs = (f->large ? kWpcL : kWpc) * kFramesPerWarp;
        fa.groups = (f->n_samples + fa.gs - 1) / fa.gs;
        if (!f->large && 16 + (size_t)fa.tmpl_smem + (size_t)kWpc * fa.warp_smem > 227 * 1024)
            return api_fail(HB_ERR_ARG, "chunk too large for the allele encoder (template + tail buffers exceed shared memory)");
    }
    const uint64_t n_ctas = f->n_chunks * fa.groups;
    if (f->large) {
        raise_smem_limit(reinterpret_cast<const void *>(donor_frames_large_kernel<kLargeNW>));
        donor_frames_large_kernel<kLargeNW><<<(unsigned)n_ctas, kWpcL * 32, (size_t)kWpcL * fa.warp_smem, f->stream>>>(fa);
    } else switch (f->nw) {
        case 1: launch_donor_frames<1>(fa, n_ctas, f->stream); break;
        case 2: launch_donor_frames<2>(fa, n_ctas, f->stream); break;
        case 3: launch_donor_frames<3>(fa, n_ctas, f->stream); break;
        case 4: launch_donor_frames<4>(fa, n_ctas, f->stream); break;
        case 5: launch_donor_frames<5>(fa, n_ctas, f->stream); break;
        default: launch_donor_frames<6>(fa, n_ctas, f->stream); break;
    }
    count_launch(1);
    CUF(cudaEventRecord(f->ev[2], f->stream));
    f->pending_need = need;
    f->pending_was_early = was_early;
    f->launched = true;
    f->launched_run = p->run_seq;
#undef CUF
    return HB_OK;
}

static int frames_finish(hb_frames *f) {
    cudaError_t e;
#define CUF(x) do { e = (x); if (e != cudaSuccess) return api_fail(HB_ERR_CUDA, std::string("CUDA: ") + cudaGetErrorString(e) + " at " #x); } while (0)
    f->launched = false;
    CUF(cudaSetDevice(f->device));
    CUF(cudaStreamSynchronize(f->stream));
    CUF(cudaGetLastError());
    f->padded_bytes = f->pending_need;
    if (f->pending_was_early) cudaEventElapsedTime(&f->ms_site, f->ev_side0, f->ev_tmpl);
    else cudaEventElapsedTime(&f->ms_site, f->ev[0], f->ev[1]);
    cudaEventElapsedTime(&f->ms_frames, f->ev[1], f->ev[2]);
#undef CUF
    return HB_OK;
}

static int frames_run(hb_frames *f, hb_parse *p) {
    int rc = frames_prepare(f, p, false);
    return rc == HB_OK ? frames_finish(f) : rc;
}

namespace hb {
// called by run_parse (hb_api.cu) right after the GT decoder of this run was launched
void frames_early_launch(void *frames, hb_parse *p) {
    hb_frames *f = static_cast<hb_frames *>(frames);
    if (!f || !f->early_site || !f->n_chunks || !f->n_samples) return;      // no template pass in flight for this run
    if (frames_prepare(f, p, true) != HB_OK) f->launched = false;             // hb_frames_rerun will do (and report) it
}
}  // namespace hb

static int frames_layout(hb_frames *f) {
    if (f->layout_valid) return HB_OK;
    const uint64_t n_frames = f->n_chunks * f->n_samples;
    f->h_size.resize(n_frames);
    if (n_frames) {
        if (cudaSetDevice(f->device) != cudaSuccess) return api_fail(HB_ERR_CUDA, "cudaSetDevice failed");
        cudaError_t e = d2h_copy(f->h_size.data(), f->d_size, n_frames * 4, f->stream);      // pageable destination: staged (hb_api.cu)
        if (e != cudaSuccess) return api_fail(HB_ERR_CUDA, std::string("CUDA: ") + cudaGetErrorString(e));
    }
    f->layout_valid = true;
    return HB_OK;
}

extern "C" {

uint64_t hb_guess_chunk_records(uint64_t n_records) { return guess_chunk_records(n_records); }

void hb_frames_free(hb_frames *f) {
    if (!f) return;
    if (f->side) cudaStreamSynchronize(f->side);
    cudaSetDevice(f->device);
    if (f->d_frames && f->device >= 0 && f->device < 64) {     // keep the big buffer for the next handle (see g_fb)
        std::lock_guard<std::mutex> lk(g_fb_mu);
        BufCache *small = &g_fb[f->device][0];              // replace the smallest kept buffer if this one is larger
        for (auto &c : g_fb[f->device]) if (c.cap < small->cap) small = &c;
        if (small->cap < f->frames_cap) { std::swap(small->p, f->d_frames); std::swap(small->cap, f->frames_cap); }
    }
    dev_pool_free(f->d_tmpl); cudaFree(f->d_frames); dev_pool_free(f->d_tmpl_len); dev_pool_free(f->d_size);
    dev_pool_free(f->d_slot_off); dev_pool_free(f->d_totals); dev_pool_free(f->d_site_scratch);
    for (auto &x : f->ev) if (x) cudaEventDestroy(x);
    if (f->ev_sites) cudaEventDestroy(f->ev_sites);
    if (f->ev_tmpl) cudaEventDestroy(f->ev_tmpl);
    if (f->ev_side0) cudaEventDestroy(f->ev_side0);
    if (f->side) cudaStreamDestroy(f->side);
    delete f;
}

int hb_compress_records(hb_parse *p, uint64_t chunk_records, hb_frames **out) {
    if (!p) return api_fail(HB_ERR_ARG, "null argument");
    return hb_compress_sample_range(p, chunk_records, 0, p->n_samples, out);
}

int hb_compress_sample_range(hb_parse *p, uint64_t chunk_records, uint32_t s0, uint32_t ns, hb_frames **out) {
    if (!p || !out) return api_fail(HB_ERR_ARG, "null argument");
    *out = nullptr;
    if ((uint64_t)s0 + ns > p->n_samples) return api_fail(HB_ERR_ARG, "sample window outside the parse");
    if (cudaSetDevice(p->device) != cudaSuccess) return api_fail(HB_ERR_CUDA, "cudaSetDevice failed");
    const uint64_t n = p->h_st.n_records;
    if (!p->d_gt[0] && n) return api_fail(HB_ERR_NOGT, "parse was made without genotypes");
    hb_frames *f = new hb_frames();
    memset(&f->fa, 0, sizeof f->fa);
    f->device = p->device; f->stream = p->stream;
    f->n_records = n; f->n_samples = ns; f->s0 = s0; f->win_cap = ns;
    f->cr = chunk_records ? chunk_records : guess_chunk_records(n);
    f->cr_explicit = chunk_records != 0;
    f->n_chunks = n ? (n + f->cr - 1) / f->cr : 0;
    if (!f->n_chunks || !f->n_samples) { f->n_chunks = n ? f->n_chunks : 0; *out = f; return HB_OK; }
    if (f->cr > kMaxChunkRecords) {
        hb_frames_free(f);
        return api_fail(HB_ERR_ARG, "chunk_records too large (at most 7,489: a stored chunk must be ONE Blosc block, and c-blosc 1.x "
                                    "cuts blocks of 262,115 bytes = 7,489 records of 35 bytes at clevel 5 with LZ4HC)");
    }
    const uint32_t cr = (uint32_t)f->cr;
    const uint32_t n_site = 33u * cr, n_gt = 2u * cr;
    auto bound = [](uint32_t x) { return x + x / 255 + 64; };
    f->tmpl_cap = (TMPL_HDR + bound(n_site) + 15) & ~15u;
    f->large = cr > kSmallChunkMax;
    FusedArgs &fa = f->fa;
    if (f->large) {                          // kernels 4a-L / 4b-L: hash tables in shared memory, 4b-L in passes
        f->smem_site = ((size_t)kSiteSegs << kSiteHashLog) * 2;
        f->nw = kLargeNW;
        fa.seg = 32u * kLargeNW;
        const uint32_t span = 32u * fa.seg, npass = (n_gt + span - 1) / span;
        fa.strw = (((127 + npass * span) >> 5) + (uint32_t)f->nw + 3 + 3) & ~3u;   // every pass's words + look-ahead
    } else {
        f->smem_site = 16 + ((n_site + 19) & ~15u) + ((site_seg_cap(24 * cr + 1) + kSiteSegs * 48 + 15) & ~15u) +
                       ((size_t)kSiteSegs << kSiteHashLog) * 2;
        uint32_t seg = (n_gt + 31) / 32;
        f->nw = (int)((seg + 31) / 32);
        if (f->nw > 1 && 1024u * (uint32_t)(f->nw - 1) + kSlack >= n_gt) { f->nw -= 1; seg = 32u * (uint32_t)f->nw; }
        fa.seg = seg;
        fa.strw = (((127 + 2 * cr) >> 5) + (uint32_t)f->nw + 3 + 3) & ~3u;   // both planes from bit alpha <= 127 on, + look-ahead words
    }
    fa.stg_bytes = (((127 + cr - 1) >> 7) + 1) * (kBitGroupWords * 4);   // 128-row groups a chunk's rows can touch
    fa.outcap = (16 + n_gt + n_gt / 255 + 24 + 15) & ~15u;
    fa.warp_smem = 16 + fa.stg_bytes + 2 * (16 + 4 * fa.strw) + fa.outcap;
    f->chunk_cap = f->n_chunks + 4;          // a re-run on a slightly longer record set (streaming) still fits
    const uint64_t n_frames = f->chunk_cap * f->n_samples;
    f->h_tmpl_len.resize(f->n_chunks);
    f->h_slot_off.resize(f->n_chunks + 1);
    cudaError_t e = cudaSuccess;
    auto ck = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    ck(dev_pool_alloc((void **)&f->d_tmpl, f->chunk_cap * (uint64_t)f->tmpl_cap));       // pooled (hb_api.cu): cudaMalloc / cudaFree are slow here
    ck(dev_pool_alloc((void **)&f->d_tmpl_len, f->chunk_cap * 4));
    ck(dev_pool_alloc((void **)&f->d_size, n_frames * 4));
    ck(dev_pool_alloc((void **)&f->d_slot_off, (f->chunk_cap + 1) * 8));
    ck(dev_pool_alloc((void **)&f->d_totals, 8));
    if (f->large) {                          // 4a-L scratch: two CTAs per SM at most, each loops over its chunks
        int sms = 0;
        ck(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, f->device));
        f->site_ctas = (uint32_t)std::min<uint64_t>(f->chunk_cap, 2ull * (uint64_t)std::max(1, sms));
        ck(dev_pool_alloc((void **)&f->d_site_scratch, (uint64_t)f->site_ctas * site_large_scratch(cr)));
    }
    for (auto &x : f->ev) ck(cudaEventCreate(&x));
    {   // highest priority: its few long CTAs must get SM slots while the decoder's many short ones stream through
        int lo = 0, hi = 0;
        ck(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        ck(cudaStreamCreateWithPriority(&f->side, cudaStreamNonBlocking, hi));
    }
    ck(cudaEventCreateWithFlags(&f->ev_sites, cudaEventDisableTiming));
    ck(cudaEventCreate(&f->ev_tmpl)); ck(cudaEventCreate(&f->ev_side0));
    if (e != cudaSuccess) { hb_frames_free(f); return api_fail(HB_ERR_MEM, std::string("CUDA: ") + cudaGetErrorString(e)); }
    int rc = frames_run(f, p);
    if (rc != HB_OK) { hb_frames_free(f); return rc; }
    *out = f;
    return HB_OK;
}

int hb_parse_attach_frames(hb_parse *p, hb_frames *f) {
    if (!p) return api_fail(HB_ERR_ARG, "null handle");
    p->attached_frames = f;
    return HB_OK;
}

int hb_frames_rerun(hb_frames *f, hb_parse *p) {
    if (!f || !p) return api_fail(HB_ERR_ARG, "null argument");
    if ((uint64_t)f->s0 + f->n_samples > p->n_samples || p->device != f->device)
        return api_fail(HB_ERR_ARG, "hb_frames_rerun: the parse no longer has the shape these frames were made for");
    if (p->h_st.n_records != f->n_records) {
        // another record count is fine when the chunk size was fixed by the caller and the chunk arrays are large enough
        const uint64_t nc = p->h_st.n_records ? (p->h_st.n_records + f->cr - 1) / f->cr : 0;
        if (!f->cr_explicit || nc > f->chunk_cap || nc == 0)
            return api_fail(HB_ERR_ARG, "hb_frames_rerun: the parse no longer has the shape these frames were made for");
        f->n_records = p->h_st.n_records;
        f->n_chunks = nc;
        f->h_tmpl_len.resize(nc);
        f->h_slot_off.resize(nc + 1);
        f->early_site = false;                   // an early template pass (if any) was made for the old shape
    }
    if (!f->n_chunks || !f->n_samples) return HB_OK;
    if (f->launched && f->launched_run == p->run_seq) return frames_finish(f);     // launched behind the decoder of this very run
    return frames_run(f, p);
}

int hb_frames_set_window(hb_frames *f, uint32_t s0, uint32_t ns) {
    if (!f) return api_fail(HB_ERR_ARG, "null handle");
    if (ns == 0 || ns > f->win_cap) return api_fail(HB_ERR_ARG, "window larger than the one the frames were made for");
    f->s0 = s0;
    f->n_samples = ns;
    f->layout_valid = false;
    f->launched = false;
    return HB_OK;
}

int hb_frames_get_info(const hb_frames *f, hb_frames_info *info) {
    if (!f || !info) return api_fail(HB_ERR_ARG, "null argument");
    memset(info, 0, sizeof *info);
    info->n_records = f->n_records; info->n_chunks = f->n_chunks; info->chunk_records = f->cr;
    if (!f->totals_valid && f->n_chunks && f->n_samples && f->d_size) {       // sum of the frame sizes, on demand (18 us of kernel per step otherwise)
        hb_frames *w = const_cast<hb_frames *>(f);
        unsigned long long tot = 0;
        cudaError_t e = cudaSetDevice(f->device);
        if (e == cudaSuccess) e = cudaMemsetAsync(w->d_totals, 0, 8, w->stream);
        if (e == cudaSuccess) {
            sum_sizes_kernel<<<296, 256, 0, w->stream>>>(w->d_size, w->n_chunks * w->n_samples, w->d_totals);
            count_launch();
            e = cudaMemcpyAsync(&tot, w->d_totals, 8, cudaMemcpyDeviceToHost, w->stream);
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(w->stream);
        if (e != cudaSuccess) return api_fail(HB_ERR_CUDA, std::string("CUDA: ") + cudaGetErrorString(e));
        w->total_bytes = tot;
        w->totals_valid = true;
    }
    info->n_samples = f->n_samples; info->total_bytes = f->total_bytes;
    info->raw_bytes = 35ull * f->n_records * f->n_samples;
    info->ms_site = f->ms_site; info->ms_frames = f->ms_frames;
    info->padded_bytes = f->padded_bytes;
    info->d_frames = f->d_frames;
    uint64_t st = 0;
    for (uint32_t t : f->h_tmpl_len) st += t - TMPL_HDR;
    info->site_lz4_bytes = st;
    return HB_OK;
}

int hb_frames_layout(hb_frames *f, uint64_t *offsets, uint32_t *sizes) {
    if (!f) return api_fail(HB_ERR_ARG, "null handle");
    int rc = frames_layout(f);
    if (rc != HB_OK) return rc;
    const uint64_t n_frames = f->n_chunks * f->n_samples, nc = f->n_chunks;
    if (offsets)
        for (uint32_t s = 0; s < f->n_samples; ++s)
            for (uint64_t c = 0; c < nc; ++c) offsets[s * nc + c] = s * f->h_slot_off[nc] + f->h_slot_off[c];
    if (sizes && n_frames) memcpy(sizes, f->h_size.data(), n_frames * 4);
    return HB_OK;
}

int hb_frames_fetch_all(hb_frames *f, uint8_t *buf, uint64_t cap) {
    if (!f || !buf) return api_fail(HB_ERR_ARG, "null argument");
    if (cap < f->padded_bytes) return api_fail(HB_ERR_ARG, "buffer too small");
    if (!f->padded_bytes) return HB_OK;
    if (cudaSetDevice(f->device) != cudaSuccess) return api_fail(HB_ERR_CUDA, "cudaSetDevice failed");
    cudaError_t e = d2h_copy(buf, f->d_frames, f->padded_bytes, f->stream);      // pinned: one copy; pageable: staged
    if (e != cudaSuccess) return api_fail(HB_ERR_CUDA, std::string("CUDA: ") + cudaGetErrorString(e));
    return HB_OK;
}

// ---- hb_frames_fetch_packed, way 1: every frame gathered whole on the device (C_out bytes cross PCIe)
static int fetch_packed_gather(hb_frames *f, uint8_t *buf, const std::vector<uint64_t> &poff) {
    const uint64_t nc = f->n_chunks, n_frames = nc * f->n_samples;
    const uint64_t run = poff[n_frames];
    f->last_d2h_bytes = run + 4 * n_frames;
    if (cudaSetDevice(f->device) != cudaSuccess) return api_fail(HB_ERR_CUDA, "cudaSetDevice failed");
    constexpr uint64_t kPackPiece = 64ull << 20;
    cudaError_t e = cudaSuccess;
    auto ck = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    uint64_t *d_poff = nullptr;
    uint8_t *d_piece[2] = {nullptr, nullptr};
    cudaStream_t copy = nullptr;
    cudaEvent_t ev_g[2] = {nullptr, nullptr}, ev_c[2] = {nullptr, nullptr};
    const uint64_t piece_cap = std::min<uint64_t>(run, kPackPiece + (1ull << 20));
    ck(dev_pool_alloc((void **)&d_poff, (n_frames + 1) * 8));
    ck(dev_pool_alloc((void **)&d_piece[0], piece_cap));
    ck(dev_pool_alloc((void **)&d_piece[1], piece_cap));
    ck(cudaStreamCreateWithFlags(&copy, cudaStreamNonBlocking));
    // the gather kernels run on a stream of the highest priority: when another host thread is parsing the next file (the
    // converter does: one chromosome ahead), its 36-ms inflate kernel owns every SM, and a gather that waits for a free SM
    // leaves the D2H engine idle; with priority its CTAs take the first slots that retire
    cudaStream_t packs = nullptr;
    cudaEvent_t ev_ready = nullptr;
    {
        int lo = 0, hi = 0;
        ck(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        ck(cudaStreamCreateWithPriority(&packs, cudaStreamNonBlocking, hi));
        ck(cudaEventCreateWithFlags(&ev_ready, cudaEventDisableTiming));
    }
    for (int k = 0; k < 2; ++k) { ck(cudaEventCreateWithFlags(&ev_g[k], cudaEventDisableTiming)); ck(cudaEventCreateWithFlags(&ev_c[k], cudaEventDisableTiming)); }
    if (e == cudaSuccess) ck(cudaMemcpyAsync(d_poff, poff.data(), (n_frames + 1) * 8, cudaMemcpyHostToDevice, f->stream));
    if (e == cudaSuccess) { ck(cudaEventRecord(ev_ready, f->stream)); ck(cudaStreamWaitEvent(packs, ev_ready, 0)); }   // the frames are complete
    const bool pinned = host_is_pinned(buf);
    uint64_t first = 0;
    int k = 0;
    while (e == cudaSuccess && first < n_frames) {
        // frames [first, last) = the next piece: at most kPackPiece bytes (one frame is far smaller than that)
        const uint64_t base = poff[first];
        uint64_t last = std::upper_bound(poff.begin() + first, poff.begin() + n_frames + 1, base + kPackPiece) - poff.begin() - 1;
        if (last <= first) last = first + 1;
        const uint64_t bytes = poff[last] - base;
        const int b = k & 1;
        // the copy that read this buffer last is done.  Waited for on the HOST, so that at most two pieces are queued on the
        // D2H engine at any time: the engine serves copies in submission order, and with all 60 pieces queued up front the
        // 4-byte status reads of a parse running in another host thread sat behind 270 ms of frames (HB_TRACE, r02j)
        if (k >= 2) ck(cudaEventSynchronize(ev_c[b]));
        pack_frames_kernel<<<(unsigned)((last - first + 7) / 8), 256, 0, packs>>>(f->d_frames, f->d_slot_off, nc, f->d_size, d_poff,
                                                                                first, last - first, base, d_piece[b]);
        count_launch();
        ck(cudaGetLastError());
        ck(cudaEventRecord(ev_g[b], packs));
        if (pinned) {
            ck(cudaStreamWaitEvent(copy, ev_g[b], 0));
            ck(cudaMemcpyAsync(buf + base, d_piece[b], bytes, cudaMemcpyDeviceToHost, copy));
            ck(cudaEventRecord(ev_c[b], copy));
        } else {                                                                // pageable destination: staged copy, piece by piece
            ck(d2h_copy(buf + base, d_piece[b], bytes, packs));
        }
        first = last;
        ++k;
    }
    if (copy) { cudaError_t e2 = cudaStreamSynchronize(copy); if (e == cudaSuccess) e = e2; }
    if (packs) { cudaError_t e2 = cudaStreamSynchronize(packs); if (e == cudaSuccess) e = e2; }
    { cudaError_t e2 = cudaStreamSynchronize(f->stream); if (e == cudaSuccess) e = e2; }
    for (int q = 0; q < 2; ++q) { if (ev_g[q]) cudaEventDestroy(ev_g[q]); if (ev_c[q]) cudaEventDestroy(ev_c[q]); }
    if (ev_ready) cudaEventDestroy(ev_ready);
    if (packs) cudaStreamDestroy(packs);
    if (copy) cudaStreamDestroy(copy);
    dev_pool_free(d_poff); dev_pool_free(d_piece[0]); dev_pool_free(d_piece[1]);
    if (e != cudaSuccess) { cudaGetLastError(); return api_fail(HB_ERR_CUDA, std::string("CUDA: ") + cudaGetErrorString(e)); }
    return HB_OK;
}


// ---- way 2: the chunk templates cross PCIe once, per donor only the 32 header bytes and the tail; host threads put the
// frames together in buf (template body, tail, header: three memcpy per frame).  Config 2: 2.7 GB instead of 15.2 GB over
// PCIe; the assembly is a memory-bound copy that the host does at several times PCIe speed when it has a few cores.
namespace {
std::atomic<int> g_fetch_mode{0};        // 0 auto, 1 device gather, 2 host assembly
std::atomic<int> g_host_threads{0};      // 0 = the CPUs this process may run on, at most 16

int host_threads() {
    int n = g_host_threads.load();
    if (n > 0) return std::min(n, 64);
    cpu_set_t set;
    CPU_ZERO(&set);
    n = sched_getaffinity(0, sizeof set, &set) == 0 ? CPU_COUNT(&set) : (int)std::thread::hardware_concurrency();
    return std::max(1, std::min(n, 16));
}

// pinned staging buffers, kept between calls (cudaMallocHost of tens of MB costs milliseconds)
struct StagePool {
    std::mutex mu;
    std::vector<std::pair<uint8_t *, uint64_t>> idle;
    uint8_t *get(uint64_t bytes) {
        {
            std::lock_guard<std::mutex> lk(mu);
            for (size_t i = 0; i < idle.size(); ++i)
                if (idle[i].second >= bytes) { uint8_t *p = idle[i].first; sizes[p] = idle[i].second; idle.erase(idle.begin() + (long)i); return p; }
        }
        uint8_t *p = nullptr;
        if (cudaMallocHost((void **)&p, bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        std::lock_guard<std::mutex> lk(mu);
        sizes[p] = bytes;
        return p;
    }
    void put(uint8_t *p) {
        if (!p) return;
        std::lock_guard<std::mutex> lk(mu);
        const uint64_t b = sizes[p];
        if (idle.size() < 8) idle.push_back({p, b}); else { sizes.erase(p); cudaFreeHost(p); }
    }
    std::map<uint8_t *, uint64_t> sizes;
} g_stage_pool;

struct Piece {                            // frames [first, last) whose tails + headers sit in `stage`
    uint64_t first = 0, last = 0, tail_base = 0, hdr_at = 0;
    const uint8_t *stage = nullptr;
};

// fork-join over the frames of one piece at a time
struct Assembler {
    const hb_frames *f; uint8_t *buf; const uint64_t *poff; const uint64_t *tail_off; const uint8_t *tmpl;
    std::vector<std::thread> th;
    std::mutex mu;
    std::condition_variable cv_work, cv_done;
    Piece piece;
    uint64_t gen = 0, next = 0, grain = 1;
    int busy = 0;
    bool quit = false;
    // n bytes (a multiple of 16) to a 16-byte aligned destination with non-temporal stores: the image is written once and
    // not read again here, and ordinary stores would first READ every destination line (15 GB of extra DRAM traffic)
    static void stream16(uint8_t *dst, const uint8_t *src, size_t n) {
        for (size_t k = 0; k < n; k += 16)
            _mm_stream_si128(reinterpret_cast<__m128i *>(dst + k), _mm_loadu_si128(reinterpret_cast<const __m128i *>(src + k)));
    }
    void frame(uint64_t i) const {
        const uint64_t nc = f->n_chunks, c = i % nc;
        const uint32_t tl = f->h_tmpl_len[c], tl16 = tl & ~15u, sz = f->h_size[i];
        uint8_t *dst = buf + poff[i];
        const uint8_t *tp = tmpl + c * (uint64_t)f->tmpl_cap;
        const uint8_t *tail = piece.stage + (tail_off[i] - piece.tail_base), *hdr = piece.stage + piece.hdr_at + 32 * (i - piece.first);
        if (tl16 >= 32 && sz >= tl16 && (reinterpret_cast<uintptr_t>(buf) & 15) == 0) {     // (frames start on 16-byte boundaries of buf)
            stream16(dst, hdr, 32);                                       // header with this frame's size fields
            stream16(dst + 32, tp + 32, tl16 - 32);                       // template body
            stream16(dst + tl16, tail, ((size_t)(sz - tl16) + 15) & ~size_t(15));     // own tail from the template's last 16-byte boundary, zero pad included
            return;
        }
        memcpy(dst, tp, std::min(tl, sz));                                // tiny templates: the same three pieces, any overlap
        if (sz > tl16) memcpy(dst + tl16, tail, sz - tl16);
        memcpy(dst, hdr, std::min<uint32_t>(32, sz));
        const uint64_t pad = (16 - (sz & 15)) & 15;                       // the image is zero up to the next frame
        if (pad) memset(dst + sz, 0, pad);
    }
    void worker() {
        uint64_t seen = 0;
        for (;;) {
            std::unique_lock<std::mutex> lk(mu);
            cv_work.wait(lk, [&] { return quit || gen != seen; });
            if (quit) return;
            seen = gen;
            for (;;) {
                const uint64_t a = next;
                if (a >= piece.last) break;
                next = std::min(piece.last, a + grain);
                const uint64_t b = next;
                lk.unlock();
                for (uint64_t i = a; i < b; ++i) frame(i);
                _mm_sfence();
                lk.lock();
            }
            if (--busy == 0) cv_done.notify_all();
        }
    }
    void start(int n) { for (int k = 0; k < n; ++k) th.emplace_back([this] { worker(); }); }
    void run(const Piece &p) {                 // returns when the piece before has been assembled and this one is handed out
        std::unique_lock<std::mutex> lk(mu);
        cv_done.wait(lk, [&] { return busy == 0; });
        piece = p; next = p.first;
        grain = std::max<uint64_t>(64, (p.last - p.first) / (8 * std::max<uint64_t>(1, (uint64_t)th.size())));
        busy = (int)th.size(); ++gen;
        cv_work.notify_all();
    }
    void wait() { std::unique_lock<std::mutex> lk(mu); cv_done.wait(lk, [&] { return busy == 0; }); }
    void stop() {
        { std::lock_guard<std::mutex> lk(mu); quit = true; }
        cv_work.notify_all();
        for (auto &t : th) t.join();
        th.clear();
    }
};
}  // namespace

static int fetch_packed_assemble(hb_frames *f, uint8_t *buf, const std::vector<uint64_t> &poff, int n_threads) {
    const uint64_t nc = f->n_chunks, n_frames = nc * f->n_samples;
    if (cudaSetDevice(f->device) != cudaSuccess) return api_fail(HB_ERR_CUDA, "cudaSetDevice failed");
    // tails in frame order, 16-byte units
    std::vector<uint64_t> toff(n_frames + 1);
    {
        uint64_t run = 0;
        for (uint64_t i = 0; i < n_frames; ++i) {
            toff[i] = run;
            const uint32_t tl16 = f->h_tmpl_len[i % nc] & ~15u, sz = f->h_size[i];
            if (sz > tl16) run += ((uint64_t)(sz - tl16) + 15) & ~15ull;
        }
        toff[n_frames] = run;
    }
    constexpr uint64_t kTailPiece = 32ull << 20;
    // pieces: at most kTailPiece bytes of tails each
    std::vector<uint64_t> cut{0};
    while (cut.back() < n_frames) {
        const uint64_t a = cut.back();
        uint64_t b = std::upper_bound(toff.begin() + a, toff.begin() + n_frames + 1, toff[a] + kTailPiece) - toff.begin() - 1;
        if (b <= a) b = a + 1;
        b = std::min(b, a + (kTailPiece >> 5));              // and at most as many headers as fit the same room
        cut.push_back(b);
    }
    f->last_d2h_bytes = toff[n_frames] + 32 * n_frames + (uint64_t)nc * f->tmpl_cap + 4 * n_frames;    // tails, headers, templates, sizes
    uint64_t stage_bytes = 0;
    for (size_t k = 0; k + 1 < cut.size(); ++k)
        stage_bytes = std::max<uint64_t>(stage_bytes, ((toff[cut[k + 1]] - toff[cut[k]] + 15) & ~15ull) + 32ull * (cut[k + 1] - cut[k]));
    cudaError_t e = cudaSuccess;
    auto ck = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    uint64_t *d_toff = nullptr;
    uint8_t *d_piece[2] = {nullptr, nullptr}, *h_stage[2] = {nullptr, nullptr};
    cudaStream_t copy = nullptr, packs = nullptr;
    cudaEvent_t ev_g[2] = {nullptr, nullptr}, ev_c[2] = {nullptr, nullptr}, ev_ready = nullptr;
    std::vector<uint8_t> tmpl((uint64_t)nc * f->tmpl_cap);
    ck(dev_pool_alloc((void **)&d_toff, (n_frames + 1) * 8));
    ck(dev_pool_alloc((void **)&d_piece[0], stage_bytes));
    ck(dev_pool_alloc((void **)&d_piece[1], stage_bytes));
    h_stage[0] = g_stage_pool.get(stage_bytes); h_stage[1] = g_stage_pool.get(stage_bytes);
    if (!h_stage[0] || !h_stage[1]) ck(cudaErrorMemoryAllocation);
    ck(cudaStreamCreateWithFlags(&copy, cudaStreamNonBlocking));
    {
        int lo = 0, hi = 0;
        ck(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        ck(cudaStreamCreateWithPriority(&packs, cudaStreamNonBlocking, hi));     // see fetch_packed_gather
        ck(cudaEventCreateWithFlags(&ev_ready, cudaEventDisableTiming));
    }
    for (int k = 0; k < 2; ++k) { ck(cudaEventCreateWithFlags(&ev_g[k], cudaEventDisableTiming)); ck(cudaEventCreateWithFlags(&ev_c[k], cudaEventDisableTiming)); }
    if (e == cudaSuccess) {
        ck(cudaMemcpyAsync(d_toff, toff.data(), (n_frames + 1) * 8, cudaMemcpyHostToDevice, f->stream));
        ck(d2h_copy(tmpl.data(), f->d_tmpl, tmpl.size(), f->stream));            // the templates, once (a few MB)
        ck(cudaEventRecord(ev_ready, f->stream));
        ck(cudaStreamWaitEvent(packs, ev_ready, 0));                             // the frames are complete
    }
    Assembler as;
    as.f = f; as.buf = buf; as.poff = poff.data(); as.tail_off = toff.data(); as.tmpl = tmpl.data();
    if (e == cudaSuccess) as.start(n_threads);
    const size_t n_pieces = cut.size() - 1;
    std::vector<Piece> pieces(n_pieces);
    // piece k: gathered + copied into stage k & 1 while piece k - 1 is assembled; a stage is reused when the piece that
    // used it (k - 2) is done, which as.run(k - 1) has waited for
    for (size_t k = 0; e == cudaSuccess && k <= n_pieces; ++k) {
        if (k < n_pieces) {
            const int b = (int)(k & 1);
            Piece &pc = pieces[k];
            pc.first = cut[k]; pc.last = cut[k + 1]; pc.tail_base = toff[pc.first];
            pc.hdr_at = (toff[pc.last] - pc.tail_base + 15) & ~15ull;
            pc.stage = h_stage[b];
            if (k >= 2) { as.wait(); }                                           // (run(k - 1) below already waited for k - 2; this is the k - 1 hand-out)
            const uint64_t cnt = pc.last - pc.first;
            pack_tails_kernel<<<(unsigned)((cnt + 7) / 8), 256, 0, packs>>>(f->d_frames, f->d_slot_off, nc, f->d_size, f->d_tmpl_len, d_toff,
                                                                          pc.first, cnt, pc.tail_base, d_piece[b],
                                                                          reinterpret_cast<uint4 *>(d_piece[b] + pc.hdr_at));
            count_launch();
            ck(cudaGetLastError());
            ck(cudaEventRecord(ev_g[b], packs));
            ck(cudaStreamWaitEvent(copy, ev_g[b], 0));
            ck(cudaMemcpyAsync(h_stage[b], d_piece[b], pc.hdr_at + 32 * cnt, cudaMemcpyDeviceToHost, copy));
            ck(cudaEventRecord(ev_c[b], copy));
        }
        if (k >= 1 && e == cudaSuccess) {
            ck(cudaEventSynchronize(ev_c[(k - 1) & 1]));
            if (e == cudaSuccess) as.run(pieces[k - 1]);
        }
    }
    if (!as.th.empty()) { as.wait(); as.stop(); }
    if (copy) cudaStreamSynchronize(copy);
    if (packs) cudaStreamSynchronize(packs);
    for (int q = 0; q < 2; ++q) { if (ev_g[q]) cudaEventDestroy(ev_g[q]); if (ev_c[q]) cudaEventDestroy(ev_c[q]); }
    if (ev_ready) cudaEventDestroy(ev_ready);
    if (packs) cudaStreamDestroy(packs);
    if (copy) cudaStreamDestroy(copy);
    dev_pool_free(d_toff); dev_pool_free(d_piece[0]); dev_pool_free(d_piece[1]);
    g_stage_pool.put(h_stage[0]); g_stage_pool.put(h_stage[1]);
    if (e != cudaSuccess) { cudaGetLastError(); return api_fail(HB_ERR_CUDA, std::string("CUDA: ") + cudaGetErrorString(e)); }
    return HB_OK;
}

uint64_t hb_frames_last_d2h_bytes(const hb_frames *f) { return f ? f->last_d2h_bytes : 0; }
void hb_set_fetch_mode(int mode) { g_fetch_mode.store(mode < 0 || mode > 2 ? 0 : mode); }
void hb_set_host_threads(int n) { g_host_threads.store(n < 0 ? 0 : n); }

// All frames packed back to back (each starts on a 16-byte boundary of the image), [sample][chunk] order: what a
// converter writes into the HDF5 file with one write.  offsets [n_samples][n_chunks] = where each frame starts in buf;
// sizes as in hb_frames_layout; either may be NULL.  buf == NULL: only *total (bytes needed) is set.
int hb_frames_fetch_packed(hb_frames *f, uint8_t *buf, uint64_t cap, uint64_t *offsets, uint32_t *sizes, uint64_t *total) {
    if (!f) return api_fail(HB_ERR_ARG, "null handle");
    int rc = frames_layout(f);
    if (rc != HB_OK) return rc;
    const uint64_t nc = f->n_chunks, n_frames = nc * f->n_samples;
    std::vector<uint64_t> poff(n_frames + 1);
    uint64_t run = 0;
    for (uint64_t i = 0; i < n_frames; ++i) { poff[i] = run; run += ((uint64_t)f->h_size[i] + 15) & ~15ull; }
    poff[n_frames] = run;
    if (total) *total = run;
    if (offsets && n_frames) memcpy(offsets, poff.data(), n_frames * 8);
    if (sizes && n_frames) memcpy(sizes, f->h_size.data(), n_frames * 4);
    if (!buf || !n_frames) return HB_OK;
    if (cap < run) return api_fail(HB_ERR_ARG, "buffer too small");
    // host assembly needs a template that IS the head of every frame (not so for raw chunks, cr < 6) and pays when the
    // host has a few cores to copy with
    const int mode = g_fetch_mode.load(), nt = host_threads();
    const bool assemble = f->cr >= 6 && (mode == 2 || (mode == 0 && nt >= 4));
    return assemble ? fetch_packed_assemble(f, buf, poff, nt) : fetch_packed_gather(f, buf, poff);
}

int hb_frames_fetch_sample(hb_frames *f, uint32_t s, uint64_t *sizes, uint8_t *buf, uint64_t cap, uint64_t *total) {
    if (!f) return api_fail(HB_ERR_ARG, "null handle");
    if (s >= f->n_samples) return api_fail(HB_ERR_SAMPLE, "sample index out of range");
    int rc = frames_layout(f);
    if (rc != HB_OK) return rc;
    const uint64_t nc = f->n_chunks;
    uint64_t tot = 0;
    for (uint64_t c = 0; c < nc; ++c) {
        const uint32_t sz = f->h_size[s * nc + c];
        if (sizes) sizes[c] = sz;
        tot += sz;
    }
    if (total) *total = tot;
    if (!buf || !nc) return HB_OK;
    if (cap < tot) return api_fail(HB_ERR_ARG, "buffer too small");
    // one contiguous D2H of the sample's row of slots, then the frames are packed together on the host
    const uint64_t row0 = s * f->h_slot_off[nc];
    const uint64_t row = f->h_slot_off[nc - 1] + f->h_size[s * nc + nc - 1];
    f->h_row.resize(row);
    if (cudaSetDevice(f->device) != cudaSuccess) return api_fail(HB_ERR_CUDA, "cudaSetDevice failed");
    cudaError_t e = d2h_copy(f->h_row.data(), f->d_frames + row0, row, f->stream);
    if (e != cudaSuccess) return api_fail(HB_ERR_CUDA, std::string("D2H of frames failed: ") + cudaGetErrorString(e));
    uint64_t o = 0;
    for (uint64_t c = 0; c < nc; ++c) {
        const uint32_t sz = f->h_size[s * nc + c];
        memcpy(buf + o, f->h_row.data() + f->h_slot_off[c], sz);
        o += sz;
    }
    return HB_OK;
}

}  // extern "C"

// =============================================================================================
// Read side: Blosc chunk -> LZ4 -> un-shuffle, one warp per HDF5 chunk.
// Replaces, for VCFH5Reader.fetch_genotypes (src/utils/h5_reader.py:37-41), what h5py + the hdf5-blosc filter
// (32001, blosc_decompress of c-blosc 1.x) do when a `snp_data` dataset is read.  Accepts what stock c-blosc writes
// for this path too -- several blocks per chunk, LZ4 / LZ4HC streams, split and unsplit blocks, raw streams,
// memcpyed chunks -- and the extended (32-byte) header of a c-blosc2 chunk with byte-shuffle as its only filter;
// anything else, and every field that would make the kernel read or write outside the frame / its output, sets the
// frame's status to non-zero (a stored file is untrusted input).  The three decoders (decode_frames_kernel, kernels 6
// and 6-L) read the header with read_blosc_head and walk LZ4 with lz4_walk, so those checks exist once.
// =============================================================================================
namespace hb {

__device__ __forceinline__ uint32_t ld_le32(const uint8_t *p) {
    return p[0] | (p[1] << 8) | (p[2] << 16) | ((uint32_t)p[3] << 24);
}

// LZ4 block walk by one warp: sequences are walked in lock-step, every check on the untrusted stream is made here.  True
// iff the stream is well-formed and decodes to exactly cap bytes.  `out` says what happens to the bytes:
// out.lit(op, p, ll) receives the literals of positions [op, op + ll), out.match(op, off, ml) repeats ml bytes from off
// back (off <= op).
template <class Out>
__device__ bool lz4_walk(const uint8_t *__restrict__ src, uint32_t n, uint32_t cap, const Out &out) {
    uint32_t ip = 0, op = 0;
    if (n == 0) return false;
    for (;;) {
        if (ip >= n) return false;
        const uint32_t tok = src[ip++];
        uint32_t ll = tok >> 4;
        if (ll == 15) { uint32_t b; do { if (ip >= n) return false; b = src[ip++]; ll += b; } while (b == 255 && ll <= cap); }
        if (ll > n - ip || ll > cap - op) return false;
        out.lit(op, src + ip, ll);
        ip += ll; op += ll;
        if (ip == n) break;
        if (ip + 2 > n) return false;
        const uint32_t off = src[ip] | ((uint32_t)src[ip + 1] << 8);
        ip += 2;
        if (off == 0 || off > op) return false;
        uint32_t ml = tok & 15;
        if (ml == 15) { uint32_t b; do { if (ip >= n) return false; b = src[ip++]; ml += b; } while (b == 255 && ml <= cap); }
        ml += 4;
        if (ml > cap - op) return false;
        out.match(op, off, ml);
        op += ml;
    }
    __syncwarp();
    return op == cap;
}

__device__ __forceinline__ void warp_copy(uint8_t *dst, const uint8_t *src, uint32_t n) {
    for (uint32_t i = threadIdx.x & 31; i < n; i += 32) dst[i] = src[i];
}

// into global memory, written and re-read by different lanes: matches read through L2 (__ldcg)
struct Lz4ToGlobal {
    uint8_t *dst;
    __device__ void lit(uint32_t op, const uint8_t *p, uint32_t ll) const { warp_copy(dst + op, p, ll); }
    __device__ void match(uint32_t op, uint32_t off, uint32_t ml) const {
        __syncwarp();
        // periodic copy: dst[op+i] = dst[op-off + i % off] only reads bytes written before this match
        for (uint32_t i = threadIdx.x & 31; i < ml; i += 32) {
            const uint32_t k = off >= ml ? i : i % off;
            dst[op + i] = __ldcg(dst + op - off + k);
        }
        __syncwarp();
    }
};

// into shared memory
struct Lz4ToShared {
    uint8_t *dst;
    __device__ void lit(uint32_t op, const uint8_t *p, uint32_t ll) const { warp_copy(dst + op, p, ll); }
    __device__ void match(uint32_t op, uint32_t off, uint32_t ml) const {
        __syncwarp();
        if (off >= ml) {                                // source and destination do not overlap
            for (uint32_t i = threadIdx.x & 31; i < ml; i += 32) dst[op + i] = dst[op - off + i];
        } else {                                        // periodic: dst[op + i] = dst[op - off + i % off]; every source precedes op
            for (uint32_t i = threadIdx.x & 31; i < ml; i += 32) dst[op + i] = dst[op - off + i % off];
        }
        __syncwarp();
    }
};

// nowhere: the walk only checks the stream
struct Lz4Check {
    __device__ void lit(uint32_t, const uint8_t *, uint32_t) const {}
    __device__ void match(uint32_t, uint32_t, uint32_t) const {}
};

// A Blosc chunk's 16-byte header (c-blosc 1.x), or the 32-byte one of c-blosc2 (both shuffle bits set), read and checked.
struct BloscHead {
    uint32_t flags, ext, hdr, shuffle, typesize, cn, bs, ccb;   // shuffle: the stored bytes are byte-shuffled
    int err;
};
// Status codes, first failure wins: 1 shorter than a header; 2 format version or reserved bit; then the decoder's own size
// checks, `sizes(h)`, which returns its code or 0; 3 a c-blosc2 filter other than byte-shuffle; 6 a special chunk
// (runs of zeros / NaNs / uninit); 5 neither memcpyed nor LZ4 / LZ4HC.
template <class Sizes>
__device__ __forceinline__ BloscHead read_blosc_head(const uint8_t *c, uint64_t flen, Sizes sizes) {
    BloscHead h{0, 0, 16, 0, 1, 0, 0, 0, 0};
    if (flen < 16) { h.err = 1; return h; }
    h.flags = c[2]; h.typesize = c[3];
    h.cn = ld_le32(c + 4); h.bs = ld_le32(c + 8); h.ccb = ld_le32(c + 12);
    h.ext = (h.flags & 1) && (h.flags & 4);
    h.hdr = h.ext ? 32 : 16;
    h.shuffle = !h.ext && (h.flags & 1);
    if (c[0] < 2 || c[0] > 5 || (!h.ext && (c[0] != 2 || (h.flags & 0x08)))) h.err = 2;
    else h.err = sizes(h);
    if (!h.err && h.ext) {
        for (int i = 0; i < 6; ++i) { if (c[16 + i] == 1) h.shuffle = 1; else if (c[16 + i] != 0) h.err = 3; }
        if ((c[31] >> 4) & 7) h.err = 6;
    }
    if (h.flags & 2) h.shuffle = 0;                  // memcpyed: the bytes as they were given, never shuffled
    else if (!h.err && ((h.flags >> 5) != 1 || (!h.ext && c[1] != 1))) h.err = 5;
    return h;
}

constexpr uint32_t kBloscMaxSplits = 16, kBloscMinBuffer = 128;      // c-blosc: MAX_SPLITS, MIN_BUFFERSIZE

// frame i = frames[off[i], off[i] + len[i]) (len == nullptr: the frames are contiguous, off has n_frames + 1 entries)
// -> out + i * chunk_nbytes; tmp: n_frames * chunk_nbytes bytes of scratch (the shuffled image)
__global__ void __launch_bounds__(256)
decode_frames_kernel(const uint8_t *__restrict__ frames, const uint64_t *__restrict__ off, const uint32_t *__restrict__ len,
                     uint64_t n_frames, uint32_t chunk_nbytes, uint8_t *__restrict__ tmp, uint8_t *__restrict__ out,
                     int planar, int *__restrict__ status) {
    const int lane = threadIdx.x & 31;
    const uint64_t wid = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (wid >= n_frames) return;
    const uint8_t *c = frames + off[wid];
    const uint64_t flen = len ? (uint64_t)len[wid] : off[wid + 1] - off[wid];
    uint8_t *t = tmp + wid * (uint64_t)chunk_nbytes;
    uint8_t *o = out + wid * (uint64_t)chunk_nbytes;
    const BloscHead h = read_blosc_head(c, flen, [&](const BloscHead &x) {
        return x.cn != chunk_nbytes || x.ccb > flen || x.ccb < x.hdr || x.bs == 0 || x.bs > x.cn || x.typesize == 0 ? 4 : 0;
    });
    const uint32_t typesize = h.typesize, cn = h.cn, bs = h.bs, ccb = h.ccb, hdr = h.hdr;
    const bool shuffle = h.shuffle;
    int err = h.err;
    if (!err && (h.flags & 2)) {                             // memcpyed
        if ((uint64_t)hdr + cn > ccb) err = 7;
        else warp_copy(t, c + hdr, cn);
        planar = 1;                                          // nothing to undo
    } else if (!err) {
        const bool dont_split = h.flags & 0x10;
        const uint32_t nblocks = (cn + bs - 1) / bs;
        const uint64_t data0 = (uint64_t)hdr + 4ull * nblocks;        // first byte after bstarts
        if (data0 > ccb) err = 7;
        for (uint32_t b = 0; b < nblocks && !err; ++b) {
            const bool leftover = (b == nblocks - 1) && (cn % bs);
            const uint32_t bsize = leftover ? cn % bs : bs;
            const bool split = !dont_split && !leftover &&
                               (h.ext || (typesize <= kBloscMaxSplits && bs / typesize >= kBloscMinBuffer));
            const uint32_t nstreams = split ? typesize : 1;
            const uint32_t ne = bsize / nstreams;
            uint64_t ip = ld_le32(c + hdr + 4 * b);
            if (ip < data0 || ip > ccb) { err = 7; break; }
            for (uint32_t s = 0; s < nstreams && !err; ++s) {
                if (ip + 4 > ccb) { err = 7; break; }
                const int32_t cs = (int32_t)ld_le32(c + ip);
                ip += 4;
                uint8_t *d = t + (uint64_t)b * bs + (uint64_t)s * ne;
                if (cs == 0 && h.ext) { for (uint32_t i = lane; i < ne; i += 32) d[i] = 0; }        // c-blosc2: run of zeros
                else if (cs <= 0 || ip + (uint32_t)cs > ccb) err = 8;
                else if ((uint32_t)cs == ne) { warp_copy(d, c + ip, ne); ip += cs; }
                else { if (!lz4_walk(c + ip, (uint32_t)cs, ne, Lz4ToGlobal{d})) err = 9; ip += cs; }
                __syncwarp();
            }
        }
        if (!err && shuffle && nblocks != 1 && !planar) {
            // Blosc shuffles per block: un-shuffle each block on its own
            for (uint32_t b = 0; b < nblocks; ++b) {
                const uint32_t bsize = (b == nblocks - 1 && cn % bs) ? cn % bs : bs;
                const uint32_t ne = bsize / typesize;
                const uint8_t *sb = t + (uint64_t)b * bs;
                uint8_t *ob = o + (uint64_t)b * bs;
                for (uint32_t i = lane; i < ne * typesize; i += 32) ob[i] = __ldcg(sb + (i % typesize) * ne + i / typesize);
                for (uint32_t i = ne * typesize + lane; i < bsize; i += 32) ob[i] = __ldcg(sb + i);
            }
            if (lane == 0) status[wid] = 0;
            return;
        }
        if (!err && planar && shuffle && nblocks != 1) err = 10;     // the planar view exists for single-block chunks only
        if (!err && !shuffle) planar = 1;                            // nothing to undo
    }
    __syncwarp();
    if (!err) {
        if (planar) { for (uint32_t i = lane; i < chunk_nbytes; i += 32) o[i] = __ldcg(t + i); }
        else {
            const uint32_t ne = chunk_nbytes / typesize;
            for (uint32_t i = lane; i < ne * typesize; i += 32) o[i] = __ldcg(t + (i % typesize) * ne + i / typesize);
            for (uint32_t i = ne * typesize + lane; i < chunk_nbytes; i += 32) o[i] = __ldcg(t + i);
        }
    }
    if (lane == 0) status[wid] = err;
}

// ---------------------------------------------------------------------------------------------
// Read side, device in / device out (SURVEY 8 row f4): stored chunks that are RESIDENT in HBM -> record COLUMNS, only
// for the chunks a batch of windows touches.  One warp per chunk; the LZ4 block is decoded into SHARED memory (a chunk
// of the reference's layout is 8-100 KB), then the five columns the dataset reads leave as coalesced stores.
// chunk i = frames[off[i], off[i] + len[i]); its records go to rows [row[i], row[i] + cr) of the output columns.
// ---------------------------------------------------------------------------------------------
struct DecodeColsArgs {
    const uint8_t *frames; const uint64_t *off; const uint32_t *len; const uint64_t *row;
    uint64_t n; uint32_t cr;
    uint32_t *start, *stop; uint8_t *ref, *alt; int8_t *p1, *p2;
    int *status;
    uint32_t warp_smem;
};

// Where the one block of a chunk of `nbytes` bytes is, for kernels 6 and 6-L.  h.err = the status code; without an
// error: a c-blosc2 run of zeros (zero), or src = the block's bytes in place (memcpyed, or stored raw) or its LZ4 stream
// of cs bytes (lz).  (src is never compared with null: with absolute offsets the frame base is null.)  Code 11: several blocks per chunk, or a c-blosc2 block split into `typesize` streams (no
// dont-split flag 0x10); the host-pointer decoder reads those.
struct SingleBlock {
    BloscHead h;
    const uint8_t *src;
    uint32_t cs;
    bool zero, lz;
};
__device__ __forceinline__ SingleBlock locate_single_block(const uint8_t *c, uint32_t flen, uint32_t nbytes) {
    SingleBlock b{read_blosc_head(c, flen, [&](const BloscHead &x) {
                      if (x.typesize != 35 || x.cn != nbytes || x.ccb > flen || x.ccb < x.hdr) return 4;
                      return !(x.flags & 2) && (x.bs != x.cn || (x.ext && !(x.flags & 0x10))) ? 11 : 0;
                  }),
                  nullptr, 0, false, false};
    BloscHead &h = b.h;
    if (h.err) return b;
    if (h.flags & 2) {                                   // memcpyed: record-major
        if ((uint64_t)h.hdr + nbytes > h.ccb) h.err = 7;
        else b.src = c + h.hdr;
        return b;
    }
    const uint64_t data0 = (uint64_t)h.hdr + 4;
    if (data0 + 4 > h.ccb) { h.err = 7; return b; }
    uint64_t ip = ld_le32(c + h.hdr);
    if (ip < data0 || ip + 4 > h.ccb) { h.err = 7; return b; }
    const int32_t cs = (int32_t)ld_le32(c + ip);
    ip += 4;
    if (cs == 0 && h.ext) { b.zero = true; return b; }  // c-blosc2: run of zeros
    if (cs <= 0 || ip + (uint32_t)cs > h.ccb) { h.err = 8; return b; }
    b.src = c + ip;
    b.cs = (uint32_t)cs;
    b.lz = (uint32_t)cs != nbytes;
    return b;
}

// the six columns of records [0, cr) at rows row0 + r from B(r, f) = byte f of record r: one record per lane and step
template <class Byte>
__device__ __forceinline__ void write_columns(const DecodeColsArgs &a, uint64_t row0, Byte B) {
    for (uint32_t r = threadIdx.x & 31; r < a.cr; r += 32) {
        if (a.start) a.start[row0 + r] = B(r, kRecStart) | (B(r, kRecStart + 1) << 8) | (B(r, kRecStart + 2) << 16) | (B(r, kRecStart + 3) << 24);
        if (a.stop) a.stop[row0 + r] = B(r, kRecStop) | (B(r, kRecStop + 1) << 8) | (B(r, kRecStop + 2) << 16) | (B(r, kRecStop + 3) << 24);
        if (a.ref) a.ref[row0 + r] = (uint8_t)B(r, kRecRef);
        if (a.alt) a.alt[row0 + r] = (uint8_t)B(r, kRecAlt);
        if (a.p1) a.p1[row0 + r] = (int8_t)B(r, kRecP1);
        if (a.p2) a.p2[row0 + r] = (int8_t)B(r, kRecP2);
    }
}

__global__ void __launch_bounds__(128) decode_columns_kernel(const DecodeColsArgs a) {
    extern __shared__ __align__(16) uint8_t dsm[];
    const int warp = threadIdx.x >> 5;
    const uint64_t wid = (uint64_t)blockIdx.x * (blockDim.x >> 5) + warp;
    if (wid >= a.n) return;
    uint8_t *t = dsm + (size_t)warp * a.warp_smem;
    const uint32_t cr = a.cr, nbytes = 35u * cr;
    const SingleBlock blk = locate_single_block(a.frames + a.off[wid], a.len[wid], nbytes);
    int err = blk.h.err;
    if (!err) {
        if (blk.lz) { if (!lz4_walk(blk.src, blk.cs, nbytes, Lz4ToShared{t})) err = 9; }
        else if (blk.zero) for (uint32_t i = threadIdx.x & 31; i < nbytes; i += 32) t[i] = 0;
        else warp_copy(t, blk.src, nbytes);
    }
    __syncwarp();
    // byte f of record r: plane-major when the chunk was byte-shuffled, record-major otherwise
    const bool shuffle = blk.h.shuffle;
    if (!err) write_columns(a, a.row[wid], [&](uint32_t r, uint32_t f) -> uint32_t { return shuffle ? t[f * cr + r] : t[r * 35u + f]; });
    if ((threadIdx.x & 31) == 0) a.status[wid] = err;
}

// ---------------------------------------------------------------------------------------------
// Kernel 6-L: decode_columns_kernel for single-block chunks whose 35 * cr bytes do not fit a warp's shared memory (up to
// kMaxChunkRecords).  One warp (= one CTA) per chunk.  Shared with kernel 6: the header and block checks
// (locate_single_block, so the status codes are the same), the LZ4 checks (lz4_walk) and the column writer.  What
// differs: an LZ4 offset is at most 65,535, so the decoded block streams through a 64 KiB history ring in shared memory
// and every byte of the planes the columns need (5-13, 23, 33, 34) goes straight to its column.  The stream is first
// walked once without copying -- its checks are all structural -- so a chunk that fails writes no row, as in kernel 6.
// Stored-raw, memcpyed and zero-run chunks are read in place.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kHistRing = 1u << 16;

// byte f of record r -> its column (f outside the six columns: nothing)
__device__ __forceinline__ void put_column_byte(const DecodeColsArgs &a, uint64_t row, uint32_t f, uint8_t v) {
    if (f >= kRecStart && f < kRecStart + 4) { if (a.start) reinterpret_cast<uint8_t *>(a.start + row)[f - kRecStart] = v; }
    else if (f >= kRecStop && f < kRecStop + 4) { if (a.stop) reinterpret_cast<uint8_t *>(a.stop + row)[f - kRecStop] = v; }
    else if (f == kRecRef) { if (a.ref) a.ref[row] = v; }
    else if (f == kRecAlt) { if (a.alt) a.alt[row] = v; }
    else if (f == kRecP1) { if (a.p1) a.p1[row] = (int8_t)v; }
    else if (f == kRecP2) { if (a.p2) a.p2[row] = (int8_t)v; }
}

__global__ void __launch_bounds__(32) decode_columns_large_kernel(const DecodeColsArgs a) {
    extern __shared__ __align__(16) uint8_t ring[];
    const int lane = threadIdx.x;
    const uint64_t wid = blockIdx.x;
    const uint32_t cr = a.cr, nbytes = 35u * cr;
    SingleBlock blk = locate_single_block(a.frames + a.off[wid], a.len[wid], nbytes);
    if (!blk.h.err && blk.lz && !lz4_walk(blk.src, blk.cs, nbytes, Lz4Check{})) blk.h.err = 9;
    if (lane == 0) a.status[wid] = blk.h.err;
    if (blk.h.err) return;
    const uint64_t row0 = a.row[wid];
    const uint8_t *src = blk.src;
    const bool shuffle = blk.h.shuffle, zero = blk.zero;
    if (!blk.lz) {                                      // in place
        write_columns(a, row0, [&](uint32_t r, uint32_t f) -> uint32_t { return zero ? 0u : shuffle ? src[f * cr + r] : src[r * 35u + f]; });
        return;
    }
    // block position q -> (plane, record) when shuffled, (record, field) otherwise: q / d by a multiply-high, exact for
    // q < 2^18 and d < 2^13
    const uint32_t d = shuffle ? cr : 35u, magic = 0xFFFFFFFFu / d + 1u;
    auto put = [&](uint32_t q, uint8_t v) {
        const uint32_t hi = __umulhi(q, magic), lo = q - hi * d;
        if (shuffle) put_column_byte(a, row0 + lo, hi, v);
        else put_column_byte(a, row0 + hi, lo, v);
    };
    const uint32_t cs = blk.cs;
    uint32_t ip = 0, op = 0;
    for (;;) {                                        // the stream is valid: no bounds checks
        const uint32_t tok = src[ip++];
        uint32_t ll = tok >> 4;
        if (ll == 15) { uint32_t b; do { b = src[ip++]; ll += b; } while (b == 255); }
        for (uint32_t i = lane; i < ll; i += 32) {
            const uint8_t v = src[ip + i];
            ring[(op + i) & (kHistRing - 1)] = v;
            put(op + i, v);
        }
        ip += ll; op += ll;
        if (ip == cs) break;
        const uint32_t off = src[ip] | ((uint32_t)src[ip + 1] << 8);
        ip += 2;
        uint32_t ml = tok & 15;
        if (ml == 15) { uint32_t b; do { b = src[ip++]; ml += b; } while (b == 255); }
        ml += 4;
        __syncwarp();
        // step b copies positions [op + b, op + b + 32): position op + i repeats position op + i - k * off, k >= 1 the
        // smallest with a source written before this step (k = 1 unless off < 32).  Such a source is at most 65,535
        // bytes back, so its ring slot still holds it; reads and writes of a step are split by a barrier.
        for (uint32_t b = 0; b < ml; b += 32) {
            const uint32_t i = b + lane;
            uint8_t v = 0;
            if (i < ml) v = ring[(op + i - off * ((i - b + off) / off)) & (kHistRing - 1)];
            __syncwarp();
            if (i < ml) { ring[(op + i) & (kHistRing - 1)] = v; put(op + i, v); }
            __syncwarp();
        }
        op += ml;
    }
}

}  // namespace hb

// kernel 6 where a chunk fits a warp's shared memory; above that kernel 6-L when `large` allows it
static int decode_columns(const uint8_t *d_frames, const uint64_t *d_off, const uint32_t *d_len, const uint64_t *d_row,
                          uint64_t n_chunks, uint32_t chunk_records, uint32_t *d_start, uint32_t *d_stop, uint8_t *d_ref,
                          uint8_t *d_alt, int8_t *d_p1, int8_t *d_p2, int *d_status, void *stream, bool large) {
    if (!n_chunks) return HB_OK;
    if (!d_off || !d_len || !d_row || !d_status || !chunk_records) return api_fail(HB_ERR_ARG, "bad argument");
    const uint64_t nbytes = 35ull * chunk_records;
    const uint32_t warp_smem = (uint32_t)((nbytes + 15) & ~15ull);
    int dev = 0, smem_max = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return api_fail(HB_ERR_CUDA, "no CUDA device: libhaplo_b200 has no CPU fallback");
    cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    smem_max -= 1024;
    if (nbytes > (uint64_t)smem_max) {
        if (!large)
            return api_fail(HB_ERR_ARG, "chunk too large for the device-side decoder (hb_decode_columns_device_large reads up to "
                                        "7,489 records, hb_decode_frames any chunk)");
        if (chunk_records > kMaxChunkRecords)
            return api_fail(HB_ERR_ARG, "chunk too large for the device-side decoder (at most 7,489 records: ONE Blosc block of "
                                        "c-blosc 1.x at typesize 35; use hb_decode_frames)");
        DecodeColsArgs a{d_frames, d_off, d_len, d_row, n_chunks, chunk_records, d_start, d_stop, d_ref, d_alt, d_p1, d_p2, d_status, 0};
        cudaFuncSetAttribute(decode_columns_large_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kHistRing);
        decode_columns_large_kernel<<<(unsigned)n_chunks, 32, kHistRing, (cudaStream_t)stream>>>(a);
        count_launch();
        if (cudaGetLastError() != cudaSuccess) return api_fail(HB_ERR_CUDA, "decode_columns_large_kernel launch failed");
        return HB_OK;
    }
    const int warps = (int)std::max<uint64_t>(1, std::min<uint64_t>(4, (uint64_t)smem_max / warp_smem));
    DecodeColsArgs a{d_frames, d_off, d_len, d_row, n_chunks, chunk_records, d_start, d_stop, d_ref, d_alt, d_p1, d_p2, d_status, warp_smem};
    cudaFuncSetAttribute(decode_columns_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    decode_columns_kernel<<<(unsigned)((n_chunks + warps - 1) / warps), warps * 32, (size_t)warps * warp_smem, (cudaStream_t)stream>>>(a);
    count_launch();
    if (cudaGetLastError() != cudaSuccess) return api_fail(HB_ERR_CUDA, "decode_columns_kernel launch failed");
    return HB_OK;
}

extern "C" int hb_decode_columns_device(const uint8_t *d_frames, const uint64_t *d_off, const uint32_t *d_len, const uint64_t *d_row,
                                        uint64_t n_chunks, uint32_t chunk_records, uint32_t *d_start, uint32_t *d_stop, uint8_t *d_ref,
                                        uint8_t *d_alt, int8_t *d_p1, int8_t *d_p2, int *d_status, void *stream) {
    return decode_columns(d_frames, d_off, d_len, d_row, n_chunks, chunk_records, d_start, d_stop, d_ref, d_alt, d_p1, d_p2, d_status,
                          stream, false);
}

extern "C" int hb_decode_columns_device_large(const uint8_t *d_frames, const uint64_t *d_off, const uint32_t *d_len,
                                              const uint64_t *d_row, uint64_t n_chunks, uint32_t chunk_records, uint32_t *d_start,
                                              uint32_t *d_stop, uint8_t *d_ref, uint8_t *d_alt, int8_t *d_p1, int8_t *d_p2, int *d_status,
                                              void *stream) {
    return decode_columns(d_frames, d_off, d_len, d_row, n_chunks, chunk_records, d_start, d_stop, d_ref, d_alt, d_p1, d_p2, d_status,
                          stream, true);
}

extern "C" int hb_decode_frames(const uint8_t *frames, const uint64_t *offsets, uint64_t n_frames,
                                uint64_t chunk_nbytes, uint8_t *out, int planar, int device) {
    if (!n_frames) return HB_OK;
    if (!frames || !offsets || !out || chunk_nbytes == 0 || chunk_nbytes > 0x7fffffffull) return api_fail(HB_ERR_ARG, "bad argument");
    for (uint64_t i = 0; i < n_frames; ++i)
        if (offsets[i + 1] < offsets[i]) return api_fail(HB_ERR_ARG, "frame offsets must not decrease");
    int nd = 0;
    if (cudaGetDeviceCount(&nd) != cudaSuccess || nd == 0) return api_fail(HB_ERR_CUDA, "no CUDA device: libhaplo_b200 has no CPU fallback");
    if (cudaSetDevice(device) != cudaSuccess) return api_fail(HB_ERR_CUDA, "cudaSetDevice failed");
    const uint64_t total = offsets[n_frames];
    uint8_t *d_frames = nullptr, *d_tmp = nullptr, *d_out = nullptr;
    uint64_t *d_off = nullptr;
    int *d_status = nullptr;
    std::vector<int> status(n_frames);
    int rc = HB_OK;
    cudaError_t e = cudaSuccess;
    auto ck = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    ck(cudaMalloc(&d_frames, total + 64));
    ck(cudaMalloc(&d_off, (n_frames + 1) * 8));
    ck(cudaMalloc(&d_tmp, n_frames * chunk_nbytes));
    ck(cudaMalloc(&d_out, n_frames * chunk_nbytes));
    ck(cudaMalloc(&d_status, n_frames * sizeof(int)));
    if (e == cudaSuccess) {
        ck(cudaMemcpy(d_frames, frames, total, cudaMemcpyHostToDevice));
        ck(cudaMemcpy(d_off, offsets, (n_frames + 1) * 8, cudaMemcpyHostToDevice));
        decode_frames_kernel<<<(unsigned)((n_frames + 7) / 8), 256>>>(d_frames, d_off, nullptr, n_frames, (uint32_t)chunk_nbytes,
                                                                     d_tmp, d_out, planar, d_status);
        count_launch();
        ck(cudaGetLastError());
        ck(cudaMemcpy(out, d_out, n_frames * chunk_nbytes, cudaMemcpyDeviceToHost));
        ck(cudaMemcpy(status.data(), d_status, n_frames * sizeof(int), cudaMemcpyDeviceToHost));
    }
    cudaFree(d_frames); cudaFree(d_off); cudaFree(d_tmp); cudaFree(d_out); cudaFree(d_status);
    if (e != cudaSuccess) return api_fail(HB_ERR_CUDA, std::string("CUDA: ") + cudaGetErrorString(e));
    for (uint64_t i = 0; i < n_frames; ++i)
        if (status[i]) { rc = api_fail(HB_ERR_IO, "corrupt or unsupported Blosc chunk (chunk " + std::to_string(i) + ", code " + std::to_string(status[i]) + ")"); break; }
    return rc;
}
