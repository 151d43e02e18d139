// hb_inflate.cu -- BGZF -> text on the GPU: the step in front of the path (SURVEY.md 8f rank 1).
//
// In the reference every byte of VCF text comes out of htslib's BGZF reader (tbx_itr_next / bcf_read inside
// vcfpp.h:1455-1484): zlib inflate of <= 64 KiB gzip members, one core, once per (donor, chromosome) call.  BGZF
// members are independent DEFLATE streams (RFC 1951 inside RFC 1952 framing with a 'BC' extra subfield that
// carries the member size), so here the COMPRESSED file goes over PCIe (20-50x fewer bytes than the text) and
// one warp inflates one member straight into the HBM text buffer the tokenizer / walker reads:
//   * the warp builds the literal/length and distance decode tables of each DEFLATE block together
//     (canonical code assignment with match.any ranks, table entries filled 32 at a time),
//   * every lane then runs the same symbol loop on the same bit buffer (no divergence, no communication),
//   * LZ77 copies are done by all 32 lanes (sources always precede the current output position, so the
//     32-byte pieces of one match are independent), literals are stored by lane 0.
// Stored and fixed-Huffman blocks are handled too.  ISIZE is always checked.  CRC32 is checked when hb_set_bgzf_crc_check(1)
// is in force (inflate_bgzf_kernel<true>): after a clean decode each lane takes the CRC of a contiguous slice of the member's
// text, read back through L2 (slice-by-4 tables in shared memory), and a 5-level warp tree joins the 32 lane CRCs with
// zlib's crc32_combine operator (multiplication by x^(8 n) mod P); the result is compared with the member's trailer.
//
// Round 2 tried to remove the 32-fold redundant decode (profiles/r02g_inflate_experiments.txt): a thread per member with
// tables in shared memory and an aligned-word byte FIFO (bit-exact, 5 of 32 lanes active on average: copy paths diverge),
// and lanes decoding 32 members with the warp copying their matches round by round (bit-exact, 8x fewer instructions, but
// ~10 K cycles of latency per round on the critical path of the heaviest member: 16-20 ms per GB-sized slab against 4.5
// here).  Both lose to this kernel at the slab sizes the streaming path uses, so it stays; what was kept from them:
// one aligned word per refill, length / distance bases computed instead of looked up, runs copied without a per-byte
// modulo, loads of a match issued before its stores, 48 resident warps per SM.
#include <atomic>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/haplo_b200.h"
#include "hb_common.cuh"
#include "hb_internal.h"
#include "hb_parse_struct.h"

namespace hb {

constexpr int kLitBits = 10, kDistBits = 8;       // primary table widths; longer codes take the canonical slow path
constexpr int kInfWarps = 8;

// runs of period d < 32: D = d * (32 / d); lane / d == (lane * inv) >> 16 for lane < 32 with inv = 65536 / d + 1 (d = 1: lane % 1 == 0)
__constant__ uint8_t c_runD[32] = {0, 32, 32, 30, 32, 30, 30, 28, 32, 27, 30, 22, 24, 26, 28, 30, 32, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 29, 30, 31};
__constant__ uint32_t c_runInv[32] = {0, 65536, 32769, 21846, 16385, 13108, 10923, 9363, 8193, 7282, 6554, 5958, 5462, 5042, 4682, 4370, 4097, 3856, 3641, 3450, 3277, 3121, 2979, 2850, 2731, 2622, 2521, 2428, 2341, 2260, 2185, 2115};
__constant__ uint8_t c_clorder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

struct HuffTab {            // one canonical Huffman code, in shared memory
    uint16_t *tab;          // [1 << bits]: (symbol << 4) | length, 0 = longer than `bits` (or unused)
    uint16_t *sorted;       // symbols ordered by (length, symbol)
    uint16_t *count;        // [16] codes per length
    int bits;
};

struct BitReader {          // identical in every lane of the warp
    const uint32_t *wp;     // next aligned word of the payload
    uint32_t cur, sh;       // the word before it; bit offset of the stream inside a word
    uint32_t ip, n;         // payload bytes fetched / available
    uint64_t bb;
    int bc;
    __device__ __forceinline__ void seek(const uint8_t *src, uint32_t at) {
        const uintptr_t a = reinterpret_cast<uintptr_t>(src + at);
        wp = reinterpret_cast<const uint32_t *>(a & ~uintptr_t(3));
        sh = (uint32_t)(a & 3) * 8u;
        cur = __ldg(wp++);
        ip = at; bb = 0; bc = 0;
    }
    __device__ __forceinline__ void refill() {
        if (bc <= 32) {
            const uint32_t nxt = __ldg(wp++);                 // may read past n: the buffer has slack
            bb |= (uint64_t)__funnelshift_r(cur, nxt, sh) << bc;
            cur = nxt;
            bc += 32;
            ip += 4;
        }
    }
    __device__ __forceinline__ uint32_t take(int k) {
        const uint32_t v = (uint32_t)bb & ((1u << k) - 1u);
        bb >>= k;
        bc -= k;
        return v;
    }
    // bytes of the payload really consumed (bits still in the buffer were fetched, not used)
    __device__ __forceinline__ bool overrun() const { return (int64_t)ip * 8 - bc > (int64_t)n * 8; }
};

// canonical decode of one symbol whose code may be up to 15 bits (puff's loop); -1 on an invalid code
__device__ int decode_slow(const HuffTab &h, BitReader &br) {
    int code = 0, first = 0, index = 0;
    uint32_t bits = (uint32_t)br.bb;
    for (int len = 1; len <= 15; ++len) {
        code |= bits & 1;
        bits >>= 1;
        const int count = h.count[len];
        if (code - count < first) { br.take(len); return h.sorted[index + (code - first)]; }
        index += count;
        first += count;
        first <<= 1;
        code <<= 1;
    }
    return -1;
}
__device__ __forceinline__ int decode_sym(const HuffTab &h, BitReader &br) {
    const uint32_t e = h.tab[(uint32_t)br.bb & ((1u << h.bits) - 1u)];
    const int len = e & 15;
    if (len) { br.take(len); return (int)(e >> 4); }
    return decode_slow(h, br);
}

// lens[0..nsym) in shared memory -> count / sorted / primary table.  Returns false for an over-subscribed code and, as
// zlib does (inftrees.c), for an incomplete one, except a literal/length or distance code whose longest code is <= 1 bit
// (a single code, or none); the code-length code (`lengths_code`) must always be complete.
__device__ bool build_table(HuffTab &h, const uint8_t *lens, int nsym, uint16_t *cursor /* [16] scratch */, bool lengths_code) {
    const int lane = threadIdx.x & 31;
    if (lane < 16) h.count[lane] = 0;
    __syncwarp();
    for (int base = 0; base < nsym; base += 32) {
        const int s = base + lane;
        const int L = s < nsym ? lens[s] : 0;
        const unsigned peers = __match_any_sync(0xffffffffu, L);
        if (L && (peers & ((1u << lane) - 1u)) == 0) h.count[L] += (uint16_t)__popc(peers);
        __syncwarp();
    }
    // offsets of each length in `sorted`; Kraft check (every lane, redundantly)
    int left = 1, off = 0, longest = 0;
    bool ok = true;
    for (int len = 1; len <= 15; ++len) {
        left <<= 1;
        left -= h.count[len];
        if (left < 0) ok = false;
        if (h.count[len]) longest = len;
        if (lane == 0) cursor[len] = (uint16_t)off;
        off += h.count[len];
    }
    if (left > 0 && (lengths_code || longest > 1)) ok = false;
    __syncwarp();
    for (int base = 0; base < nsym; base += 32) {
        const int s = base + lane;
        const int L = s < nsym ? lens[s] : 0;
        const unsigned peers = __match_any_sync(0xffffffffu, L);
        const int rank = __popc(peers & ((1u << lane) - 1u));
        if (L) h.sorted[cursor[L] + rank] = (uint16_t)s;
        __syncwarp();
        if (L && rank == 0) cursor[L] += (uint16_t)__popc(peers);
        __syncwarp();
    }
    // primary table: entry idx holds the symbol whose code is a prefix of idx (bit 0 of idx = first bit read)
    for (int idx = lane; idx < (1 << h.bits); idx += 32) {
        int code = 0, first = 0, index = 0;
        uint16_t e = 0;
        for (int len = 1; len <= h.bits; ++len) {
            code |= (idx >> (len - 1)) & 1;
            const int count = h.count[len];
            if (code - count < first) { e = (uint16_t)((h.sorted[index + (code - first)] << 4) | len); break; }
            index += count;
            first += count;
            first <<= 1;
            code <<= 1;
        }
        h.tab[idx] = e;
    }
    __syncwarp();
    return ok;
}

struct InflateArgs {
    const uint8_t *comp;         // the whole compressed file in HBM
    const uint64_t *coff;        // [n] offset of each member's DEFLATE payload
    const uint32_t *clen;        // [n] payload bytes
    const uint64_t *ooff;        // [n] offset of the member's text in `out`
    const uint32_t *olen;        // [n] ISIZE
    uint8_t *out;
    uint32_t n_blocks;
    int *status;                 // [n] 0 = ok; 19 = the text's CRC32 is not the trailer's (inflate_bgzf_kernel<true>)
};

// ---- CRC32 of a member's text (zlib's: reflected polynomial 0xEDB88320, x^0 = bit 31), for inflate_bgzf_kernel<true>
constexpr uint32_t kCrcPoly = 0xEDB88320u;
// a * b mod P (zlib's multmodp), as a fixed 32-step loop
__host__ __device__ constexpr uint32_t crc_mulmod(uint32_t a, uint32_t b) {
    uint32_t p = 0;
    for (int k = 0; k < 32; ++k) {
        p ^= b & (0u - (a >> 31));
        a <<= 1;
        b = (b >> 1) ^ (kCrcPoly & (0u - (b & 1u)));
    }
    return p;
}
// x^(8 n) mod P = lo[n % 256] * hi[n / 256] for n <= 65,536: one multiplication instead of zlib's one per set bit of n
struct CrcShift { uint32_t lo[256], hi[257]; };
constexpr CrcShift crc_shift_tables() {
    CrcShift t{};
    t.lo[0] = 0x80000000u;                                  // x^0
    for (int n = 1; n < 256; ++n) t.lo[n] = crc_mulmod(t.lo[n - 1], 0x00800000u);   // * x^8
    const uint32_t x2048 = crc_mulmod(t.lo[255], 0x00800000u);
    t.hi[0] = 0x80000000u;
    for (int j = 1; j < 257; ++j) t.hi[j] = crc_mulmod(t.hi[j - 1], x2048);
    return t;
}
__device__ const CrcShift g_crc_shift = crc_shift_tables();
// crc * x^(8 n) mod P: a CRC register followed by n zero bytes, the shift of zlib's crc32_combine
__device__ __forceinline__ uint32_t crc_shift(uint32_t crc, uint32_t n) {
    return crc_mulmod(crc_mulmod(__ldg(&g_crc_shift.lo[n & 255]), __ldg(&g_crc_shift.hi[n >> 8])), crc);
}
// one 32-bit little-endian word into the register (slice-by-4: t[k][b] = the register after byte b and k zero bytes)
__device__ __forceinline__ uint32_t crc_word(uint32_t c, uint32_t w, const uint32_t (*t)[256]) {
    c ^= w;
    return t[3][c & 255] ^ t[2][(c >> 8) & 255] ^ t[1][(c >> 16) & 255] ^ t[0][c >> 24];
}
// CRC32 of out[0, olen), the warp together.  Lane L takes the bytes of [A0 + L S, A0 + (L + 1) S), A0 = out rounded down to 32
// bytes, S a multiple of 32: aligned 16-byte loads through L2, bytes before `out` read as zeros (which leave a register that
// starts at 0 unchanged), the last lane's ragged end byte by byte.  Lane registers start at 0 and are joined in a tree,
// crc(A B) = crc(A) x^(8 |B|) + crc(B); zlib's initial and final inversions are applied to the joined value.
__device__ uint32_t member_crc32(const uint8_t *out, uint32_t olen, const uint32_t (*t)[256]) {
    const int lane = threadIdx.x & 31;
    const uintptr_t a = reinterpret_cast<uintptr_t>(out), e = a + olen, a0 = a & ~uintptr_t(31);
    const uint32_t S = ((uint32_t)(e - a0) + 1023u) / 1024u * 32u;
    const uintptr_t lo = a0 + (uintptr_t)lane * S, hi = lo + S < e ? lo + S : e;
    uint32_t c = 0, n = 0;
    if (lo < e) {
        n = (uint32_t)(hi - (lo > a ? lo : a));
        for (uintptr_t p = lo; p < hi; p += 32) {
            const uint4 *q = reinterpret_cast<const uint4 *>(p);
            if (p >= a && p + 32 <= hi) {                  // whole chunk
                const uint4 v0 = __ldcg(q), v1 = __ldcg(q + 1);
                c = crc_word(c, v0.x, t); c = crc_word(c, v0.y, t); c = crc_word(c, v0.z, t); c = crc_word(c, v0.w, t);
                c = crc_word(c, v1.x, t); c = crc_word(c, v1.y, t); c = crc_word(c, v1.z, t); c = crc_word(c, v1.w, t);
                continue;
            }
            uint4 v[2] = {make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0)};
#pragma unroll
            for (int h = 0; h < 2; ++h)                    // only 16-byte pieces that hold member bytes are read
                if (p + 16 * h + 16 > a && p + 16 * h < hi) v[h] = __ldcg(q + h);
            const uint32_t w[8] = {v[0].x, v[0].y, v[0].z, v[0].w, v[1].x, v[1].y, v[1].z, v[1].w};
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const uintptr_t wa = p + 4 * j;
                if (wa >= hi) break;
                uint32_t x = w[j];
                if (wa + 4 <= a) x = 0;
                else if (wa < a) x &= 0xFFFFFFFFu << (8 * (uint32_t)(a - wa));
                if (wa + 4 <= hi) { c = crc_word(c, x, t); continue; }
                for (uint32_t b = 0; wa + b < hi; ++b) c = (c >> 8) ^ t[0][(c ^ (x >> (8 * b))) & 255];
            }
        }
    }
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t rc = __shfl_down_sync(0xffffffffu, c, d), rn = __shfl_down_sync(0xffffffffu, n, d);
        if ((lane & (2 * d - 1)) == 0 && rn) { c = crc_shift(c, rn) ^ rc; n += rn; }
    }
    c = __shfl_sync(0xffffffffu, c, 0);
    return ~(c ^ crc_shift(0xFFFFFFFFu, olen));
}

constexpr int kInfSmemPerWarp = 2 * (1 << kLitBits) + 2 * (1 << kDistBits) + 2 * 288 + 2 * 32 + 2 * 16 * 3 + 2 * 16 + 320 + 2 * 128 + 2 * 19 + 2 * 16 + 26;

// kCrc: also check each member's CRC32 (4 KiB more shared memory per CTA: still 6 CTAs = 48 warps per SM)
template <bool kCrc>
__global__ void __launch_bounds__(kInfWarps * 32, 6) inflate_bgzf_kernel(const InflateArgs a) {
    __shared__ __align__(16) uint8_t smem[kInfWarps][(kInfSmemPerWarp + 15) & ~15];
    __shared__ uint32_t crc_tab[kCrc ? 4 : 1][256];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t blk = blockIdx.x * kInfWarps + warp;
    if constexpr (kCrc) {                                  // slice-by-4 tables: thread i fills entry i of each
        uint32_t c = threadIdx.x;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
#pragma unroll
            for (int b = 0; b < 8; ++b) c = (c >> 1) ^ (kCrcPoly & (0u - (c & 1u)));
            crc_tab[k][threadIdx.x] = c;
        }
        __syncthreads();
    }
    if (blk >= a.n_blocks) return;
    uint8_t *sm = smem[warp];
    HuffTab lit, dist, cl;
    lit.tab = reinterpret_cast<uint16_t *>(sm); sm += 2 * (1 << kLitBits);
    dist.tab = reinterpret_cast<uint16_t *>(sm); sm += 2 * (1 << kDistBits);
    lit.sorted = reinterpret_cast<uint16_t *>(sm); sm += 2 * 288;
    dist.sorted = reinterpret_cast<uint16_t *>(sm); sm += 2 * 32;
    lit.count = reinterpret_cast<uint16_t *>(sm); sm += 2 * 16;
    dist.count = reinterpret_cast<uint16_t *>(sm); sm += 2 * 16;
    cl.count = reinterpret_cast<uint16_t *>(sm); sm += 2 * 16;
    uint16_t *cursor = reinterpret_cast<uint16_t *>(sm); sm += 2 * 16;
    cl.tab = reinterpret_cast<uint16_t *>(sm); sm += 2 * 128;
    cl.sorted = reinterpret_cast<uint16_t *>(sm); sm += 2 * 19 + 2;
    uint8_t *lens = sm;          // [320] code lengths: literal/length symbols then distance symbols
    lit.bits = kLitBits; dist.bits = kDistBits; cl.bits = 7;

    BitReader br;
    const uint8_t *src = a.comp + a.coff[blk];
    br.n = a.clen[blk];
    br.seek(src, 0);
    uint8_t *out = a.out + a.ooff[blk];
    const uint32_t olen = a.olen[blk];
    uint32_t op = 0;
    int err = 0;
    for (int last = 0; !last && !err;) {
        br.refill();
        last = (int)br.take(1);
        const int type = (int)br.take(2);
        if (type == 0) {                                   // stored
            br.take(br.bc & 7);                            // to the byte boundary
            br.refill();
            const uint32_t len = br.take(16), nlen = br.take(16);
            if ((len ^ nlen) != 0xFFFFu) { err = 1; break; }
            // bytes still in the bit buffer belong to the stored data
            const uint32_t pos = br.ip - (uint32_t)(br.bc >> 3);
            if (pos + len > br.n || op + len > olen) { err = 2; break; }
            for (uint32_t i = lane; i < len; i += 32) out[op + i] = src[pos + i];
            op += len;
            br.seek(src, pos + len);
            __syncwarp();
            continue;
        }
        if (type == 3) { err = 3; break; }
        int nlit, ndist;
        if (type == 1) {                                   // fixed code
            for (int s = lane; s < 288; s += 32) lens[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
            lens[288 + lane] = 5;                          // 32 distance codes, so the code is complete; 30 and 31 are rejected below
            nlit = 288; ndist = 32;
            __syncwarp();
        } else {                                           // dynamic code
            nlit = (int)br.take(5) + 257;
            ndist = (int)br.take(5) + 1;
            const int ncl = (int)br.take(4) + 4;
            if (nlit > 286 || ndist > 30) { err = 4; break; }
            if (lane < 19) lens[lane] = 0;
            __syncwarp();
            for (int i = 0; i < ncl; ++i) {
                br.refill();
                const uint32_t v = br.take(3);
                if (lane == 0) lens[c_clorder[i]] = (uint8_t)v;
            }
            __syncwarp();
            if (!build_table(cl, lens, 19, cursor, true)) { err = 5; break; }
            // the nlit + ndist code lengths, run-length coded (every lane decodes; lane 0 writes)
            int i = 0, prev = 0;
            while (i < nlit + ndist) {
                br.refill();
                const int sym = decode_sym(cl, br);
                if (sym < 0) { err = 6; break; }
                int rep = 1, val = sym;
                if (sym == 16) { if (i == 0) { err = 7; break; } val = prev; rep = 3 + (int)br.take(2); }
                else if (sym == 17) { val = 0; rep = 3 + (int)br.take(3); }
                else if (sym == 18) { val = 0; rep = 11 + (int)br.take(7); }
                if (i + rep > nlit + ndist) { err = 8; break; }
                // lens is laid out [0,288) literal/length, [288,320) distance
                for (int k = lane; k < rep; k += 32) { const int s = i + k; lens[s < nlit ? s : 288 + (s - nlit)] = (uint8_t)val; }
                prev = val;
                i += rep;
            }
            if (err) break;
            __syncwarp();
            if (lens[256] == 0) { err = 9; break; }
        }
        if (!build_table(lit, lens, nlit, cursor, false)) { err = 10; break; }
        if (!build_table(dist, lens + 288, ndist, cursor, false)) { err = 11; break; }
        // ---- symbols
        for (;;) {
            br.refill();
            int sym = decode_sym(lit, br);
            if (sym < 256) {
                if (sym < 0) { err = 12; break; }
                if (op >= olen) { err = 13; break; }
                if (lane == 0) out[op] = (uint8_t)sym;
                ++op;
                continue;
            }
            if (sym == 256) break;
            sym -= 257;
            if (sym >= 29) { err = 14; break; }
            uint32_t len;                                  // RFC 1951 3.2.5, computed instead of looked up
            if (sym < 8) len = 3 + sym;
            else if (sym == 28) len = 258;
            else { const int eb = (sym >> 2) - 1; len = 3 + ((4 + (sym & 3)) << eb) + br.take(eb); }
            br.refill();
            const int ds = decode_sym(dist, br);
            if (ds < 0 || ds >= 30) { err = 15; break; }
            uint32_t d;
            if (ds < 4) d = 1 + ds;
            else { const int eb = (ds >> 1) - 1; d = 1 + ((2 + (ds & 1)) << eb) + br.take(eb); }
            if (d > op || op + len > olen) { err = 16; break; }
            __syncwarp();                                  // earlier stores of the warp are visible to the loads below
            uint8_t *to = out + op;
            const uint8_t *from = to - d;
            if (d >= len) {                                // no overlap: independent 32-byte pieces, three loads in flight
                for (uint32_t base = 0; base < len; base += 96) {
                    uint8_t v[3];
#pragma unroll
                    for (int k = 0; k < 3; ++k) { const uint32_t i = base + 32 * k + lane; v[k] = i < len ? __ldcg(from + i) : (uint8_t)0; }
#pragma unroll
                    for (int k = 0; k < 3; ++k) { const uint32_t i = base + 32 * k + lane; if (i < len) to[i] = v[k]; }
                }
            } else if (d < 32) {                           // a run of period d (the "0|0\t" of genotype text is d = 4, len = 258):
                const uint32_t D = c_runD[d];              // a lane's byte repeats every D = the largest multiple of d <= 32
                if ((uint32_t)lane < D) {                  // (D and lane % d from tables: two divisions by a variable cost ~40 instructions)
                    const uint32_t r = (uint32_t)lane - (((uint32_t)lane * c_runInv[d]) >> 16) * d;
                    const uint8_t b = __ldcg(from + r);
                    for (uint32_t i = lane; i < len; i += D) to[i] = b;
                }
            } else {                                       // 32 <= d < len: each 32 bytes read what the ones before stored
                for (uint32_t r = 0; r < len; r += 32) {
                    const uint32_t i = r + lane;
                    if (i < len) to[i] = __ldcg(from + i);
                    __syncwarp();
                }
            }
            op += len;
        }
        if (br.overrun()) err = 17;
        __syncwarp();
    }
    if (!err && op != olen) err = 18;
    if constexpr (kCrc) {                                  // err is the same in every lane
        if (!err) {
            const uint8_t *tr = src + br.n;                // the trailer: CRC32, ISIZE
            const uint32_t want = (uint32_t)__ldg(tr) | (uint32_t)__ldg(tr + 1) << 8 | (uint32_t)__ldg(tr + 2) << 16 |
                                  (uint32_t)__ldg(tr + 3) << 24;
            if (member_crc32(out, olen, crc_tab) != want) err = kInflateCrcMismatch;
        }
    }
    if (lane == 0) a.status[blk] = err;
}

// hb_set_bgzf_crc_check: process-wide, off by default
std::atomic<int> g_bgzf_crc{0};
bool bgzf_crc_check() { return g_bgzf_crc.load() != 0; }

// "BGZF CRC32 mismatch (member i, compressed offset X)" for the member whose DEFLATE payload starts at raw[coff]: i counts
// every member of the file before it (empty ones too) and X is where its gzip header starts.  The headers up to it were
// validated by bgzf_index.
std::string bgzf_crc_message(const uint8_t *raw, uint64_t coff) {
    uint64_t p = 0, i = 0;
    for (;;) {
        const uint8_t *h = raw + p;
        const uint32_t xlen = h[10] | (h[11] << 8);
        if (p + 12 + xlen >= coff) break;
        uint32_t bsize = 0;
        for (uint64_t q = p + 12; q + 4 <= p + 12 + xlen; q += 4 + (raw[q + 2] | (raw[q + 3] << 8)))
            if (raw[q] == 'B' && raw[q + 1] == 'C') bsize = (raw[q + 4] | (raw[q + 5] << 8)) + 1;
        p += bsize;
        ++i;
    }
    return "BGZF CRC32 mismatch (member " + std::to_string(i) + ", compressed offset " + std::to_string(p) + ")";
}

static void launch_inflate(const InflateArgs &a, cudaStream_t stream) {
    const uint32_t grid = (a.n_blocks + kInfWarps - 1) / kInfWarps;
    if (bgzf_crc_check()) inflate_bgzf_kernel<true><<<grid, kInfWarps * 32, 0, stream>>>(a);
    else inflate_bgzf_kernel<false><<<grid, kInfWarps * 32, 0, stream>>>(a);
}

// BGZF member table of a whole file (host): false when the bytes are not BGZF; boff (may be NULL): each member's address
bool bgzf_index(const uint8_t *raw, uint64_t size, std::vector<uint64_t> &coff, std::vector<uint32_t> &clen,
                std::vector<uint64_t> &ooff, std::vector<uint32_t> &olen, uint64_t &total, std::vector<uint64_t> *boff) {
    uint64_t p = 0;
    total = 0;
    while (p < size) {
        if (p + 18 > size) return false;
        const uint8_t *h = raw + p;
        if (h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || !(h[3] & 4)) return false;
        const uint32_t xlen = h[10] | (h[11] << 8);
        uint32_t bsize = 0;
        bool found = false;
        uint64_t q = p + 12;
        const uint64_t xe = p + 12 + xlen;
        if (xe > size) return false;
        while (q + 4 <= xe) {
            const uint32_t slen = raw[q + 2] | (raw[q + 3] << 8);
            if (raw[q] == 'B' && raw[q + 1] == 'C' && slen == 2) { bsize = (raw[q + 4] | (raw[q + 5] << 8)) + 1; found = true; }
            q += 4 + slen;
        }
        if (!found || p + bsize > size || bsize < 12 + xlen + 8) return false;
        if (h[3] & ~4) return false;                       // FNAME / FCOMMENT / FHCRC: not what bgzip writes
        const uint8_t *tr = raw + p + bsize - 4;
        const uint32_t isize = tr[0] | (tr[1] << 8) | (tr[2] << 16) | ((uint32_t)tr[3] << 24);
        if (isize > 65536) return false;
        if (isize) {                                       // the 28-byte EOF marker (and any empty member) carries no text
            coff.push_back(p + 12 + xlen);
            clen.push_back(bsize - 12 - xlen - 8);
            ooff.push_back(total);
            olen.push_back(isize);
            if (boff) boff->push_back(p);
        }
        total += isize;
        p += bsize;
    }
    return true;
}

// pinned staging for the member tables and the status words of inflate_bgzf_to_device: copies from / to pageable memory
// were seen to stall for 100-1400 ms on these hosts; one pinned block per process, grown on demand, used under its lock
namespace {
std::mutex g_stage_mu;
uint8_t *g_stage = nullptr;
size_t g_stage_cap = 0;
}

// raw (host, BGZF) -> d_out (device, `total` bytes).  d_out must hold total bytes.
int inflate_bgzf_to_device(const uint8_t *raw, uint64_t size, const std::vector<uint64_t> &coff,
                           const std::vector<uint32_t> &clen, const std::vector<uint64_t> &ooff,
                           const std::vector<uint32_t> &olen, uint8_t *d_out, cudaStream_t stream, float *ms) {
    const uint32_t n = (uint32_t)coff.size();
    if (!n) return HB_OK;
    uint8_t *d_comp = nullptr;
    uint64_t *d_coff = nullptr, *d_ooff = nullptr;
    uint32_t *d_clen = nullptr, *d_olen = nullptr;
    int *d_status = nullptr;
    cudaError_t e = cudaSuccess;
    auto ck = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    ck(dev_pool_alloc((void **)&d_comp, size + 64));
    ck(dev_pool_alloc((void **)&d_coff, n * 8ull)); ck(dev_pool_alloc((void **)&d_ooff, n * 8ull));
    ck(dev_pool_alloc((void **)&d_clen, n * 4ull)); ck(dev_pool_alloc((void **)&d_olen, n * 4ull));
    ck(dev_pool_alloc((void **)&d_status, n * 4ull));
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::vector<int> status(n, 0);
    std::lock_guard<std::mutex> stage_lock(g_stage_mu);
    const size_t stage_need = 28ull * n;                 // coff, ooff (8 B), clen, olen, status (4 B)
    if (e == cudaSuccess && g_stage_cap < stage_need) {
        if (g_stage) cudaFreeHost(g_stage);
        g_stage = nullptr; g_stage_cap = 0;
        if (cudaMallocHost((void **)&g_stage, stage_need + stage_need / 4) == cudaSuccess) g_stage_cap = stage_need + stage_need / 4;
        else cudaGetLastError();
    }
    const bool staged = g_stage_cap >= stage_need;
    uint8_t *h_coff = g_stage, *h_ooff = g_stage + 8ull * n, *h_clen = g_stage + 16ull * n, *h_olen = g_stage + 20ull * n,
            *h_status = g_stage + 24ull * n;
    if (staged) {
        memcpy(h_coff, coff.data(), 8ull * n); memcpy(h_ooff, ooff.data(), 8ull * n);
        memcpy(h_clen, clen.data(), 4ull * n); memcpy(h_olen, olen.data(), 4ull * n);
    }
    if (e == cudaSuccess) {
        ck(cudaMemcpyAsync(d_comp, raw, size, cudaMemcpyHostToDevice, stream));
        ck(cudaMemsetAsync(d_comp + size, 0, 64, stream));
        ck(cudaMemcpyAsync(d_coff, staged ? (const void *)h_coff : (const void *)coff.data(), n * 8ull, cudaMemcpyHostToDevice, stream));
        ck(cudaMemcpyAsync(d_ooff, staged ? (const void *)h_ooff : (const void *)ooff.data(), n * 8ull, cudaMemcpyHostToDevice, stream));
        ck(cudaMemcpyAsync(d_clen, staged ? (const void *)h_clen : (const void *)clen.data(), n * 4ull, cudaMemcpyHostToDevice, stream));
        ck(cudaMemcpyAsync(d_olen, staged ? (const void *)h_olen : (const void *)olen.data(), n * 4ull, cudaMemcpyHostToDevice, stream));
        InflateArgs a{d_comp, d_coff, d_clen, d_ooff, d_olen, d_out, n, d_status};
        if (ms) { cudaEventCreate(&ev0); cudaEventCreate(&ev1); cudaEventRecord(ev0, stream); }
        launch_inflate(a, stream);
        count_launch();
        if (ms) cudaEventRecord(ev1, stream);
        ck(cudaGetLastError());
        ck(cudaMemcpyAsync(staged ? (void *)h_status : (void *)status.data(), d_status, n * 4ull, cudaMemcpyDeviceToHost, stream));
        ck(cudaStreamSynchronize(stream));
        if (staged && e == cudaSuccess) memcpy(status.data(), h_status, 4ull * n);
        if (ms && e == cudaSuccess) cudaEventElapsedTime(ms, ev0, ev1);
    }
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    dev_pool_free(d_comp); dev_pool_free(d_coff); dev_pool_free(d_ooff); dev_pool_free(d_clen); dev_pool_free(d_olen); dev_pool_free(d_status);
    if (e != cudaSuccess) return api_fail(HB_ERR_CUDA, std::string("CUDA: ") + cudaGetErrorString(e));
    for (uint32_t i = 0; i < n; ++i) {
        if (status[i] == kInflateCrcMismatch) return api_fail(HB_ERR_IO, bgzf_crc_message(raw, coff[i]));
        if (status[i]) return api_fail(HB_ERR_IO, "BGZF inflate failed (member " + std::to_string(i) + ", code " + std::to_string(status[i]) + ")");
    }
    return HB_OK;
}

// ---- slab streaming: pre-allocated tables, enqueue only (no allocation, no synchronisation)
int inflate_scratch_alloc(InflateScratch &sc, uint64_t comp_cap, uint32_t n_cap) {
    cudaError_t e = cudaSuccess;
    auto ck = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    sc.comp_cap = comp_cap; sc.n_cap = n_cap;
    ck(cudaMalloc(&sc.d_comp, comp_cap + 64));
    ck(cudaMalloc(&sc.d_coff, n_cap * 8ull)); ck(cudaMalloc(&sc.d_ooff, n_cap * 8ull));
    ck(cudaMalloc(&sc.d_clen, n_cap * 4ull)); ck(cudaMalloc(&sc.d_olen, n_cap * 4ull));
    ck(cudaMalloc(&sc.d_status, n_cap * 4ull));
    ck(cudaMalloc(&sc.d_last_nl, 8));
    if (e != cudaSuccess) return api_fail(HB_ERR_MEM, std::string("cudaMalloc (inflate tables): ") + cudaGetErrorString(e));
    return HB_OK;
}
void inflate_scratch_free(InflateScratch &sc) {
    cudaFree(sc.d_comp); cudaFree(sc.d_coff); cudaFree(sc.d_ooff); cudaFree(sc.d_clen); cudaFree(sc.d_olen);
    cudaFree(sc.d_status); cudaFree(sc.d_last_nl);
    sc = InflateScratch();
}
// comp[0 .. comp_bytes): the compressed bytes of n consecutive members; coff relative to comp, ooff relative to d_out
int inflate_bgzf_enqueue(InflateScratch &sc, const uint8_t *comp, uint64_t comp_bytes, const uint64_t *coff, const uint32_t *clen,
                         const uint64_t *ooff, const uint32_t *olen, uint32_t n, uint8_t *d_out, cudaStream_t stream) {
    if (!n) return HB_OK;
    if (comp_bytes > sc.comp_cap || n > sc.n_cap) return api_fail(HB_ERR_ARG, "inflate scratch too small");
    cudaError_t e = cudaSuccess;
    auto ck = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    ck(cudaMemcpyAsync(sc.d_comp, comp, comp_bytes, cudaMemcpyHostToDevice, stream));
    ck(cudaMemsetAsync(sc.d_comp + comp_bytes, 0, 64, stream));
    ck(cudaMemcpyAsync(sc.d_coff, coff, n * 8ull, cudaMemcpyHostToDevice, stream));
    ck(cudaMemcpyAsync(sc.d_ooff, ooff, n * 8ull, cudaMemcpyHostToDevice, stream));
    ck(cudaMemcpyAsync(sc.d_clen, clen, n * 4ull, cudaMemcpyHostToDevice, stream));
    ck(cudaMemcpyAsync(sc.d_olen, olen, n * 4ull, cudaMemcpyHostToDevice, stream));
    InflateArgs a{sc.d_comp, sc.d_coff, sc.d_clen, sc.d_ooff, sc.d_olen, d_out, n, sc.d_status};
    launch_inflate(a, stream);
    count_launch();
    ck(cudaGetLastError());
    if (e != cudaSuccess) return api_fail(HB_ERR_CUDA, std::string("CUDA: ") + cudaGetErrorString(e));
    return HB_OK;
}

// position of the last '\n' in buf[begin, end), or ~0: one CTA walks back from the end in 16 KiB steps
__global__ void __launch_bounds__(1024) last_newline_kernel(const uint8_t *__restrict__ buf, uint64_t begin, uint64_t end,
                                                            unsigned long long *__restrict__ res) {
    __shared__ unsigned long long best;
    if (threadIdx.x == 0) best = 0;
    __syncthreads();
    for (uint64_t hi = end; hi > begin;) {
        const uint64_t lo = hi - begin > 16384 ? hi - 16384 : begin;
        unsigned long long mine = 0;                        // position + 1
        for (uint64_t q = lo + 16ull * threadIdx.x; q < hi && q < lo + 16ull * threadIdx.x + 16; ++q)
            if (buf[q] == '\n') mine = q + 1;
        if (mine) atomicMax(&best, mine);
        __syncthreads();
        if (best) break;
        hi = lo;
    }
    if (threadIdx.x == 0) *res = best ? best - 1 : ~0ull;
}
void launch_last_newline(const uint8_t *d_buf, uint64_t begin, uint64_t end, unsigned long long *d_res, cudaStream_t stream) {
    last_newline_kernel<<<1, 1024, 0, stream>>>(d_buf, begin, end, d_res);
    count_launch();
}

}  // namespace hb

using namespace hb;

// host BGZF bytes -> host text, inflated on the GPU (tests; the file path keeps the text in HBM)
extern "C" int hb_bgzf_inflate(const uint8_t *bgzf, uint64_t nbytes, uint8_t *out, uint64_t cap, uint64_t *out_len,
                               int device, float *kernel_ms) {
    if (!bgzf || !out_len) return api_fail(HB_ERR_ARG, "null argument");
    int nd = 0;
    if (cudaGetDeviceCount(&nd) != cudaSuccess || nd == 0) return api_fail(HB_ERR_CUDA, "no CUDA device: libhaplo_b200 has no CPU fallback");
    if (cudaSetDevice(device) != cudaSuccess) return api_fail(HB_ERR_CUDA, "cudaSetDevice failed");
    std::vector<uint64_t> coff, ooff;
    std::vector<uint32_t> clen, olen;
    uint64_t total = 0;
    if (!bgzf_index(bgzf, nbytes, coff, clen, ooff, olen, total, nullptr)) return api_fail(HB_ERR_IO, "not a BGZF file");
    *out_len = total;
    if (!out) return HB_OK;
    if (cap < total) return api_fail(HB_ERR_ARG, "buffer too small");
    if (!total) return HB_OK;
    uint8_t *d_out = nullptr;
    if (cudaMalloc(&d_out, total) != cudaSuccess) return api_fail(HB_ERR_MEM, "cudaMalloc failed");
    int rc = inflate_bgzf_to_device(bgzf, nbytes, coff, clen, ooff, olen, d_out, nullptr, kernel_ms);
    if (rc == HB_OK && cudaMemcpy(out, d_out, total, cudaMemcpyDeviceToHost) != cudaSuccess) rc = api_fail(HB_ERR_CUDA, "D2H failed");
    cudaFree(d_out);
    return rc;
}

void hb_set_bgzf_crc_check(int on) { g_bgzf_crc.store(on ? 1 : 0); }
int hb_get_bgzf_crc_check(void) { return g_bgzf_crc.load(); }
