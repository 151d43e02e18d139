// hb_gt.cu -- kernel 3: GT-field decode into phased int8 allele planes, sample-major.
//
// Replaces BcfRecord::getGenotypes (reference cpp/vcfpp.h:546-588, over htslib's GT branch of
// vcf_parse_format) plus the int8 narrowing of cpp/parse_vcf.cpp:51-52 -- for ALL samples of a
// record at once instead of one sample per whole-file pass.
//
// Work unit: a 2-D tile of kTV records x kTS samples.  Variant-major text goes in, sample-major
// bytes come out, so every tile is a transpose:
//   * the per-record byte range of the tile's sample columns is known from the site kernel
//     (uniform "\tX|Y" records: arithmetic) or from the tokenizer's column checkpoints;
//   * uniform segments are staged into shared memory with one TMA bulk copy per record
//     (cp.async.bulk, mbarrier completion); each thread then decodes 1 sample x 16 records with
//     a SWAR compare per call and packs the 16 alleles of each plane into one 16-byte
//     shared-memory store of the transposed tile;
//   * anything else (GT:GQ:DP columns, multi-digit alleles, malformed text) is decoded by a
//     warp that streams the segment, ranks its tabs with popc + a warp scan, and parses each field;
//   * the tile is written out as 16-byte vectors, kTV contiguous bytes per (plane, sample).
// Output layout = the Blosc2 byte-shuffled layout of the reference's 35-byte records
// (planes 33 and 34 of every chunk), see DESIGN.md.
#include <cstdlib>

#include "hb_common.cuh"
#include "hb_internal.h"

namespace hb {

constexpr int GT_THREADS = 256;
constexpr int GT_WARPS = GT_THREADS / 32;
constexpr int SEG_PITCH = 4 * kTS + 16;   // staged bytes per record: 4*kTS + up to 15 bytes of misalignment
constexpr int OUT_PITCH = kTV + 16;       // bytes; (kTV+16)/16 odd => conflict-free 16-byte transposed stores
static_assert(kTV % 16 == 0 && ((OUT_PITCH / 16) & 1) == 1, "tile geometry");

struct GtSmem {
    alignas(128) uint8_t text[kTV][SEG_PITCH];
    alignas(16) uint8_t out[2][kTS][OUT_PITCH];
    alignas(16) uint32_t addr[kTV];       // byte offset (multiple of 4) of sample 0's column word inside text[][]
    alignas(16) uint32_t shft[kTV];       // 8 * (misalignment of that column, 0..3)
    alignas(16) uint32_t dummy[kTS + 4];  // "\t0|0" x kTS: what records off the fast path decode
    uint64_t seg_begin[kTV];
    uint32_t seg_len[kTV];
    uint32_t seg_g[kTV];
    int mode[kTV];                        // 0 nothing to decode (zeros), 1 staged fast path, 2 general path
    alignas(8) uint64_t bar;
    uint32_t any_general;                 // some record of the tile takes the general path (phase 2)
    uint32_t any_fast;                    // some record of the tile is staged for the fast path (phase 1)
};

// One sample column starting at p (first byte after the TAB).  Restates htslib's GT parse:
// '.' -> missing (-9), digits -> allele index (int8-narrowed), '|' or '/' continue.
// Returns ploidy, or -1 when an allele is neither digits nor '.'.
__device__ __noinline__ int decode_field(const uint8_t *__restrict__ t, uint64_t p, int g, int &a0, int &a1) {
    for (int k = 0; k < g; ++k) {
        for (;;) {
            uint8_t c = t[p];
            if (c == '\t' || c == '\n' || c == '\r') { a0 = -9; a1 = -9; return 0; }
            ++p;
            if (c == ':') break;
        }
    }
    int l = 0;
    a0 = 0; a1 = -128;
    for (;;) {
        uint8_t c = t[p];
        int val;
        if (c == '.') { ++p; val = -9; }
        else {
            uint32_t v = 0; int nd = 0;
            while (c >= '0' && c <= '9') { v = v * 10u + (uint32_t)(c - '0'); ++nd; c = t[++p]; }
            if (nd == 0) {
                if (l == 0 && (c == '\t' || c == '\n' || c == '\r' || c == ':')) { a0 = -9; a1 = -9; return 1; }
                return -1;
            }
            val = (int)(int8_t)(uint8_t)v;
        }
        if (l == 0) a0 = val; else if (l == 1) a1 = val;
        ++l;
        c = t[p];
        if (c == '|' || c == '/') { ++p; continue; }
        break;
    }
    return l;
}

// "\tXsY" with X,Y in [0-9.] and s in [|/] that is not the common "\t[01]|[01]".
// Returns (a0 & 0xff) << 8 | (a1 & 0xff) << 24.  A group that is not of that shape demotes its record
// (*mode = 2) to the general path, which redoes the whole segment; records that were never on the
// fast path (*mode != 1) just yield 0.
// A '\n' inside a group means the span was not one record's samples (possible only when the records
// were located by the walker, hb_walk.cu): the whole index is void and the caller falls back.
__device__ __noinline__ uint32_t decode_group_slow(uint32_t w, int *mode, uint32_t *any_general, DevStatus *st) {
    if (has_byte(w, kNl4)) st->index_invalid = 1u;           // (before the early return: another lane may have demoted the record already)
    if (*mode != 1) return 0;
    const uint32_t sep = (w >> 16) & 0xffu, x = (w >> 8) & 0xffu, y = w >> 24;
    bool ok = (w & 0xffu) == '\t' && (sep == '|' || sep == '/');
    uint32_t a0 = x - '0', a1 = y - '0';
    if (x == '.') a0 = (uint32_t)(-9) & 0xffu; else if (a0 > 9) ok = false;
    if (y == '.') a1 = (uint32_t)(-9) & 0xffu; else if (a1 > 9) ok = false;
    if (!ok) { *mode = 2; *any_general = 1u; return 0; }
    return (a0 << 8) | (a1 << 24);
}

// kSubset: only the columns of `sel` are decoded and written, to their planes.  Every column of every kept record is still
// staged and read as in the full decode: the shape check of phase 1, decode_group_slow's newline check and phase 2's TAB
// count see them all, so a record with too many or too few columns is still found, and so is a newline inside a span the
// head walker jumped over (DevStatus::index_invalid).  Per-sample decoding, per-sample error counts and output are for
// selected columns only.
template <bool kSubset>
__global__ void __launch_bounds__(GT_THREADS, 4)
decode_gt_kernel(const uint8_t *__restrict__ text, const RowInfo *__restrict__ rowinfo, uint64_t n_rows,
                 uint32_t n_samples, uint32_t n_stiles, const uint64_t *__restrict__ cp, uint32_t ncp,
                 int8_t *__restrict__ gt0, int8_t *__restrict__ gt1, uint64_t gt_stride,
                 uint32_t *__restrict__ bits, uint64_t bits_stride,
                 uint32_t *__restrict__ ploidy_err, uint32_t *__restrict__ badgt_err,
                 DevStatus *__restrict__ st, uint32_t pf_dist, SampleSel sel) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    GtSmem &sm = *reinterpret_cast<GtSmem *>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t tile = blockIdx.x;                      // (32-bit on purpose: a 64-bit divide is ~100 dependent instructions
    const uint32_t tile_r = tile / n_stiles;               //  at the head of every CTA's critical path)
    const uint32_t tile_s = tile - tile_r * n_stiles;
    const uint32_t s0 = tile_s * kTS;
    const uint32_t ns = min((uint32_t)kTS, n_samples - s0);
    const uint64_t r0 = (uint64_t)tile_r * kTV;
    const uint32_t nr = (uint32_t)min((uint64_t)kTV, n_rows - r0);
    uint4 msk = make_uint4(0, 0, 0, 0);                    // kSubset: the tile's selected columns and the plane of the first
    uint32_t sbase = 0;
    if constexpr (kSubset) { msk = sel.mask[tile_s]; sbase = sel.base[tile_s]; }

    if (tid == 0) {
        mbar_init(&sm.bar, kTV);                           // every record's thread arrives, with the bytes it requested
        mbar_fence_init();
        sm.any_general = 0;
        sm.any_fast = 0;
    }
    if (tid < kTS + 4) sm.dummy[tid] = 0x307C3009u;
    __syncthreads();

    // ---- phase 0: locate each record's segment; stage uniform ones with TMA
    uint64_t pf_addr = 0;
    uint32_t pf_bytes = 0;
    if (tid < kTV) {
        int mode = 0;
        uint64_t b = 0;
        uint32_t len = 0, g = 0;
        if ((uint32_t)tid < nr) {
            const RowInfo ri = rowinfo[r0 + tid];
            g = ri.misc & 0xffu;
            if ((ri.misc & kRowHasSamples) && g != 255u) {
                if (ri.misc & kRowUniform) {
                    b = ri.samp_abs + 4ull * s0;
                    len = 4u * ns;
                    mode = 1;
                } else {
                    const uint64_t *row = cp + (uint64_t)ri.cp_row * ncp;
                    uint64_t bb = row[tile_s];
                    uint64_t ee = (tile_s + 1 < n_stiles) ? row[tile_s + 1] : ri.samp_abs + ri.samp_len;
                    if (bb == kNoCp || ee == kNoCp || ee < bb || ee - bb > 0xffffffffull) {
                        atomicAdd(&st->n_bad_cols, 1ull);     // too few columns in this record
                    } else {
                        b = bb;
                        len = (uint32_t)(ee - bb);
                        mode = (len == 4u * ns && g == 0) ? 1 : 2;
                    }
                }
            }
        }
        sm.seg_begin[tid] = b;
        sm.seg_len[tid] = len;
        sm.seg_g[tid] = g;
        sm.mode[tid] = mode;
        if (mode == 2) sm.any_general = 1u;
        if (mode == 1) sm.any_fast = 1u;
        if (mode == 1) {
            sm.addr[tid] = (uint32_t)tid * SEG_PITCH + ((uint32_t)(b & 15ull) & ~3u);
            sm.shft[tid] = 8u * ((uint32_t)b & 3u);
            // the record's segment is requested the moment its RowInfo is here (no CTA barrier, no byte total first), and
            // BEFORE this thread reads the RowInfo of the tile it prefetches: that second load was on every tile's critical path
            const uint32_t bytes = (uint32_t)(((b & 15ull) + len + 15ull) & ~15ull);
            mbar_expect_tx(&sm.bar, bytes);
            tma_load_1d(sm.text[tid], text + (b & ~15ull), bytes, &sm.bar);
        } else {
            sm.addr[tid] = (uint32_t)(reinterpret_cast<const uint8_t *>(sm.dummy) - &sm.text[0][0]);
            sm.shft[tid] = 0;
            mbar_arrive(&sm.bar);
        }
        // The tile that will run in this CTA's slot once it retires (pf_dist tiles ahead = resident CTAs of the whole
        // GPU): its text is pulled into L2 now (UBLKPF), so that CTA's TMA loads find it there instead of in DRAM.
        const uint32_t tf = tile + pf_dist;
        if (pf_dist && tf < gridDim.x && tf > tile) {
            const uint32_t trf = tf / n_stiles;
            const uint32_t s0f = (tf - trf * n_stiles) * kTS;
            const uint64_t rf = (uint64_t)trf * kTV + tid;
            if (rf < n_rows) {
                const RowInfo rif = rowinfo[rf];
                if ((rif.misc & kRowHasSamples) && (rif.misc & kRowUniform) && (rif.misc & 0xffu) != 255u) {
                    const uint64_t bf = rif.samp_abs + 4ull * s0f;
                    const uint32_t nsf = min((uint32_t)kTS, n_samples - s0f);
                    pf_addr = bf & ~15ull;
                    pf_bytes = (uint32_t)(((bf & 15ull) + 4u * nsf + 15ull) & ~15ull);
                }
            }
        }
        if (pf_bytes) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(text + pf_addr), "r"(pf_bytes) : "memory");
    }
    // ONE thread waits for the bulk copies, the CTA barrier releases the rest: 256 threads spinning on try_wait were
    // 8.7 % of the kernel's instructions (r02a ncu), issue slots taken from the CTAs that share the SM
    if (tid == kTV) mbar_wait(&sm.bar, 0);                 // (a thread that has no record to locate first)
    __syncthreads();

    // ---- phase 1: fast path.  One thread = 1 sample x 16 records; lanes run along samples, so the
    //      two 4-byte loads per call and the 16-byte transposed stores are bank-conflict free.
    //      Records that are not on the fast path read a dummy row of "\t0|0" instead (-> zeros), and
    //      anything that is not "\t[01]|[01]" only raises a flag, so the hot loop has no branches;
    //      flagged threads then redo their few odd calls one by one.
    if (!sm.any_fast) {      // a tile of general-path records only (GT:GQ:DP text): nothing to decode here, the tile starts as zeros
        for (int i = tid; i < (int)(sizeof(sm.out) / 16); i += GT_THREADS) reinterpret_cast<uint4 *>(&sm.out[0][0][0])[i] = make_uint4(0, 0, 0, 0);
    } else
    for (int item = tid; item < kTS * (kTV / 16); item += GT_THREADS) {
        const int s = item % kTS, rg = item / kTS;
        uint32_t acc0[4] = {0, 0, 0, 0}, acc1[4] = {0, 0, 0, 0};
        uint32_t bad = 0;
        const uint8_t *tbase = &sm.text[0][0] + 4 * s;
        if ((uint32_t)s < ns) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const uint4 a4 = *reinterpret_cast<const uint4 *>(&sm.addr[16 * rg + 4 * q]);
                const uint4 h4 = *reinterpret_cast<const uint4 *>(&sm.shft[16 * rg + 4 * q]);
                const uint32_t aa[4] = {a4.x, a4.y, a4.z, a4.w}, hh[4] = {h4.x, h4.y, h4.z, h4.w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const uint32_t *colp = reinterpret_cast<const uint32_t *>(tbase + aa[k]);
                    const uint32_t x = __funnelshift_r(colp[0], colp[1], hh[k]) ^ 0x307C3009u;   // "\t0|0"
                    if (x & 0xFEFFFEFFu) bad |= 1u << (4 * q + k);   // anything but the two allele bits left? remember which call
                    // byte k of acc0 <- byte 1 of x, byte k of acc1 <- byte 3 of x
                    acc0[q] = __byte_perm(acc0[q], x, k == 0 ? 0x3215 : k == 1 ? 0x3250 : k == 2 ? 0x3510 : 0x5210);
                    acc1[q] = __byte_perm(acc1[q], x, k == 0 ? 0x3217 : k == 1 ? 0x3270 : k == 2 ? 0x3710 : 0x7210);
                }
            }
        }
        *reinterpret_cast<uint4 *>(&sm.out[0][s][16 * rg]) = make_uint4(acc0[0], acc0[1], acc0[2], acc0[3]);
        *reinterpret_cast<uint4 *>(&sm.out[1][s][16 * rg]) = make_uint4(acc1[0], acc1[1], acc1[2], acc1[3]);
        while (bad) {                                         // the thread's odd calls (a/b, '.', alleles >= 2), one by one
            const int i = __ffs(bad) - 1;
            bad &= bad - 1;
            const int r = 16 * rg + i;
            const uint32_t *colp = reinterpret_cast<const uint32_t *>(tbase + sm.addr[r]);
            const uint32_t w = __funnelshift_r(colp[0], colp[1], sm.shft[r]);
            const uint32_t x = decode_group_slow(w, &sm.mode[r], &sm.any_general, st);
            sm.out[0][s][r] = (uint8_t)(x >> 8);
            sm.out[1][s][r] = (uint8_t)(x >> 24);
        }
    }
    __syncthreads();

    // ---- phase 2: general path, one warp per record segment (skipped, with its barrier, when no record of the tile needs
    //      it: the empty loop over the tile's records was 7.6 % of the fast path's instructions)
    if (sm.any_general) {
    for (uint32_t r = warp; r < nr; r += GT_WARPS) {
        if (sm.mode[r] != 2) continue;
        const uint64_t b = sm.seg_begin[r], e = b + sm.seg_len[r];
        const int g = (int)sm.seg_g[r];
        uint32_t seen = 0;
        // the next 512 bytes are requested before these are decoded: a warp otherwise alternates between waiting for DRAM
        // and decoding, and 32 warps x 512 bytes in flight per SM bound the general path at ~0.7 TB/s (r01c, r02e)
        uint4 nxt = make_uint4(0, 0, 0, 0);
        if ((b & ~15ull) + 16ull * lane < e) nxt = *reinterpret_cast<const uint4 *>(text + (b & ~15ull) + 16ull * lane);
        for (uint64_t base = b & ~15ull; base < e; base += 512) {
            const uint64_t o = base + 16ull * lane;
            const uint4 v = nxt;
            nxt = make_uint4(0, 0, 0, 0);
            if (o + 512 < e + 4) nxt = *reinterpret_cast<const uint4 *>(text + o + 512);     // (+ 4: the look-ahead of a field that ends the segment; the buffer has slack)
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
            // the 512 bytes (+ 16 of look-ahead = lane 0's next piece) also go to this record's row of the staging buffer,
            // which the general path does not use otherwise: the common field shape "X|Y" + terminator is then decoded from
            // shared memory with one unaligned 4-byte read instead of a byte-wise parse over global memory
            uint8_t *row = sm.text[r];
            *reinterpret_cast<uint4 *>(row + 16 * lane) = make_uint4(w[0], w[1], w[2], w[3]);
            if (lane == 0) *reinterpret_cast<uint4 *>(row + 512) = nxt;
            __syncwarp();
            // one bit per byte of the lane's 16 that is a TAB inside [b, e): the lane walks ITS tabs (1-2 for "a|b:GQ:DP"
            // fields) in one loop -- per-word loops ran 4 passes per piece with a third of the lanes in each, and the
            // per-byte range test of the first / last piece (most pieces: a segment is 2-3 of them) was 22 % of the instructions
            uint32_t mm = pack_lsb4(eq_mask(w[0], kTab4) >> 7) | (pack_lsb4(eq_mask(w[1], kTab4) >> 7) << 4) |
                          (pack_lsb4(eq_mask(w[2], kTab4) >> 7) << 8) | (pack_lsb4(eq_mask(w[3], kTab4) >> 7) << 12);
            {
                const int64_t lo = (int64_t)b - (int64_t)o, hi = (int64_t)e - (int64_t)o;      // valid bytes of the lane: [lo, hi) within 0..16
                const uint32_t below_lo = lo <= 0 ? 0u : (lo >= 16 ? 0xFFFFu : (1u << lo) - 1u);
                const uint32_t below_hi = hi <= 0 ? 0u : (hi >= 16 ? 0xFFFFu : (1u << hi) - 1u);
                mm &= below_hi & ~below_lo;
            }
            const uint32_t cnt = __popc(mm);
            uint32_t inc = cnt;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
                if (lane >= d) inc += t;
            }
            uint32_t k = seen + inc - cnt;
            while (mm) {
                const int bit = __ffs(mm) - 1;                                   // byte of the TAB inside the lane's 16
                mm &= mm - 1;
                if (k < ns && (!kSubset || sel_has(msk, k))) {
                    int a0, a1, pl;
                    const int rel = 16 * lane + bit + 1;                         // first byte of the field, in `row`
                    const uint32_t *fw = reinterpret_cast<const uint32_t *>(row + (rel & ~3));
                    const uint32_t x = __funnelshift_r(fw[0], fw[1], (rel & 3) * 8);
                    const uint32_t X = x & 0xffu, sep = (x >> 8) & 0xffu, Y = (x >> 16) & 0xffu, T = x >> 24;
                    const uint32_t dx = X - '0', dy = Y - '0';
                    if (g == 0 && (sep == '|' || sep == '/') && (T == ':' || T == '\t' || T == '\n' || T == '\r') &&
                        (dx <= 9u || X == '.') && (dy <= 9u || Y == '.')) {
                        a0 = X == '.' ? -9 : (int)dx;
                        a1 = Y == '.' ? -9 : (int)dy;
                        pl = 2;
                    } else pl = decode_field(text, o + (uint64_t)bit + 1, g, a0, a1);
                    if (pl < 0) { atomicAdd(&st->n_bad_gt, 1ull); atomicAdd(&badgt_err[sel_plane<kSubset>(msk, sbase, s0, k)], 1u); a0 = 0; a1 = 0; }
                    else if (pl != 2) atomicAdd(&ploidy_err[sel_plane<kSubset>(msk, sbase, s0, k)], 1u);
                    sm.out[0][k][r] = (uint8_t)a0;
                    sm.out[1][k][r] = (uint8_t)a1;
                }
                ++k;
            }
            seen += __shfl_sync(0xffffffffu, inc, 31);
            __syncwarp();                                     // the row is overwritten by the next 512 bytes
        }
        if (seen != ns) {
            if (lane == 0) atomicAdd(&st->n_bad_cols, 1ull);
            for (uint32_t k = seen + lane; k < ns; k += 32) { sm.out[0][k][r] = 0; sm.out[1][k][r] = 0; }
        }
    }
    __syncthreads();
    }

    // ---- phase 3: kTV contiguous bytes per (plane, sample), 16-byte vector stores; and the same alleles as bit planes
    //      (B = bit 0 of the byte, N = "neither 0 nor 1") for the frame encoder: the 4 lanes that hold the 4 pieces of one
    //      (plane, sample) combine their 16-bit masks with shuffles and one of them stores 2 words of each array
    {
        constexpr int PIECES = kTV / 16;
        static_assert(PIECES == 4 && (2 * kTS * PIECES) % GT_THREADS == 0, "the 4 pieces of a row sit in 4 neighbouring lanes");
        // kSubset: a thread's items are columns tid / 4 and tid / 4 + 64 only (of both planes): their selection and their
        // planes are worked out once here, not per item
        static_assert(GT_THREADS * 2 == kTS * PIECES, "item >> 8 & 1 picks the column");
        bool take[2] = {true, true};
        uint32_t plane[2] = {0, 0};
        if constexpr (kSubset) {
            for (int h = 0; h < 2; ++h) {
                const uint32_t c = (uint32_t)(tid / PIECES) + 64u * h;
                take[h] = sel_has(msk, c);
                plane[h] = sbase + sel_rank(msk, c);
            }
        }
        for (int item = tid; item < 2 * kTS * PIECES; item += GT_THREADS) {
            const int piece = item % PIECES;
            const int ps = item / PIECES;       // plane * kTS + s
            const int s = ps % kTS, p = ps / kTS;
            const bool live = (uint32_t)s < ns && (!kSubset || take[(item >> 8) & 1]);
            uint4 v = make_uint4(0, 0, 0, 0);
            if (live) {
                v = *reinterpret_cast<const uint4 *>(&sm.out[p][s][16 * piece]);
                int8_t *dst = (p ? gt1 : gt0) + (uint64_t)(kSubset ? plane[(item >> 8) & 1] : s0 + s) * gt_stride + r0 + 16ull * piece;
                stg_stream(reinterpret_cast<uint4 *>(dst), v);
            }
            if (bits) {
                uint32_t t = pack_lsb4(v.x) | (pack_lsb4(v.y) << 4) | (pack_lsb4(v.z) << 8) | (pack_lsb4(v.w) << 12);
                if ((v.x | v.y | v.z | v.w) & 0xFEFEFEFEu)
                    t |= (pack_nz4(v.x) | (pack_nz4(v.y) << 4) | (pack_nz4(v.z) << 8) | (pack_nz4(v.w) << 12)) << 16;
                const uint32_t u = __shfl_down_sync(0xffffffffu, t, 1);
                const uint32_t bw = (t & 0xffffu) | (u << 16), nw = (t >> 16) | (u & 0xffff0000u);   // valid in even lanes
                const uint32_t bw1 = __shfl_down_sync(0xffffffffu, bw, 2), nw1 = __shfl_down_sync(0xffffffffu, nw, 2);
                if (live && piece == 0) {
                    uint32_t *row = bits + (uint64_t)(kSubset ? plane[(item >> 8) & 1] : s0 + s) * bits_stride + (r0 >> 7) * kBitGroupWords + ((r0 >> 5) & 3u);
                    *reinterpret_cast<uint2 *>(row + 4 * p) = make_uint2(bw, bw1);
                    *reinterpret_cast<uint2 *>(row + 4 * (2 + p)) = make_uint2(nw, nw1);
                }
            }
        }
    }
}

void launch_decode_gt(const uint8_t *d_text, const RowInfo *d_rowinfo, uint64_t n_rows, uint32_t n_samples,
                      const uint64_t *d_cp, uint32_t ncp, int8_t *d_gt0, int8_t *d_gt1, uint64_t gt_stride,
                      uint32_t *d_bits, uint64_t bits_stride, uint32_t *d_ploidy_err, uint32_t *d_badgt_err, DevStatus *d_st,
                      const SampleSel &sel, const Launch &L) {
    if (!n_rows || !n_samples) return;
    size_t smem = sizeof(GtSmem);
    const bool subset = sel.mask != nullptr;
    auto kernel = subset ? decode_gt_kernel<true> : decode_gt_kernel<false>;
    // > 48 KB of dynamic shared memory is opt-in per function AND per device: set on every launch (a microsecond), so a
    // process that moves to another device is served too
    cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    uint32_t n_stiles = (n_samples + kTS - 1) / kTS;
    uint64_t n_rtiles = (n_rows + kTV - 1) / kTV;
    uint64_t tiles = n_rtiles * n_stiles;
    const uint32_t pf_dist = 4u * (uint32_t)L.sm_count;      // 4 CTAs per SM are resident (__launch_bounds__)
    kernel<<<(unsigned)tiles, GT_THREADS, smem, L.stream>>>(d_text, d_rowinfo, n_rows, n_samples, n_stiles, d_cp, ncp, d_gt0,
                                                            d_gt1, gt_stride, d_bits, bits_stride, d_ploidy_err, d_badgt_err,
                                                            d_st, pf_dist, sel);
    count_launch();
}

// The allele bit planes (hb_internal.h, kBitGroupWords) of byte planes that were not written by the decoder above:
// the resident streamed parse assembles its planes from slabs with device copies.  One thread = 32 rows of one sample.
__global__ void __launch_bounds__(256)
bits_from_planes_kernel(const int8_t *__restrict__ gt0, const int8_t *__restrict__ gt1, uint64_t gt_stride, uint64_t n_rows,
                        uint32_t n_samples, uint32_t *__restrict__ bits, uint64_t bits_stride) {
    const uint64_t words = (n_rows + 31) / 32;                  // 32-row words per sample
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= words * n_samples) return;
    const uint64_t s = i / words, w = i - s * words;
    uint32_t out[4] = {0, 0, 0, 0};                             // B0, B1, N0, N1
#pragma unroll
    for (int p = 0; p < 2; ++p) {
        const uint4 *src = reinterpret_cast<const uint4 *>((p ? gt1 : gt0) + s * gt_stride + 32 * w);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const uint4 v = ldg_stream(src + h);
            const uint32_t b = pack_lsb4(v.x) | (pack_lsb4(v.y) << 4) | (pack_lsb4(v.z) << 8) | (pack_lsb4(v.w) << 12);
            const uint32_t nz = pack_nz4(v.x) | (pack_nz4(v.y) << 4) | (pack_nz4(v.z) << 8) | (pack_nz4(v.w) << 12);
            out[p] |= b << (16 * h);
            out[2 + p] |= nz << (16 * h);
        }
    }
    uint32_t *row = bits + s * bits_stride + (w >> 2) * kBitGroupWords + (w & 3);
    row[0] = out[0]; row[4] = out[1]; row[8] = out[2]; row[12] = out[3];
}

void launch_bits_from_planes(const int8_t *d_gt0, const int8_t *d_gt1, uint64_t gt_stride, uint64_t n_rows, uint32_t n_samples,
                             uint32_t *d_bits, uint64_t bits_stride, const Launch &L) {
    if (!n_rows || !n_samples) return;
    const uint64_t n = (n_rows + 31) / 32 * n_samples;
    bits_from_planes_kernel<<<(unsigned)((n + 255) / 256), 256, 0, L.stream>>>(d_gt0, d_gt1, gt_stride, n_rows, n_samples, d_bits, bits_stride);
    count_launch();
}

}  // namespace hb
