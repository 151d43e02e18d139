// hb_bcf.cu -- BCF 2.2 input: kernel 1b (record locator + site columns) and kernel 3b (GT decode).
//
// BCF is what `bcftools view -Ob` writes and what the reference's BcfReader reads through the same hts_open / bcf_read
// calls as a .vcf.gz (vcfpp.h:1381,1479).  A record (VCF v4.3 specification, section 6.3) is
//   uint32 l_shared, uint32 l_indiv, int32 CHROM, int32 POS (0-based), int32 rlen, float QUAL,
//   uint32 n_allele << 16 | n_info, uint32 n_fmt << 24 | n_sample,
//   ID (typed string), n_allele alleles (typed strings), FILTER (typed ints), INFO pairs     l_shared bytes from CHROM on
//   per FORMAT field: typed int key, type byte, n_sample x count values                      l_indiv bytes
// Records carry no sync marker: only the chain of lengths from the body's first byte says where one starts, and a
// serial walk of that chain is one dependent load per record.
//
// Locator.  The body is cut into segments of at least several records.  One warp per segment finds the first offset
// whose header passes a strict test and whose successor passes it too; one thread per segment chains from there to the
// first record start at or past the segment's end (its exit), counting records.  Segment 0 starts at the body's first
// byte, which the header's l_text makes known, so its chain is the true one; segment k's chain is true when its start
// is the exit of a true segment k - 1.  The verify kernel checks every pair; a start that differs is replaced by the
// exit before it and that segment is chained again, until every pair agrees.  Each round proves at least one more
// segment, so the loop ends, and a chain that meets a record failing the test inside the proven prefix is a malformed
// file, reported by the host.  Nothing is taken from a guess: a fake header inside genotype bytes costs a round.
//
// Sites.  One thread per record reads CHROM / POS / rlen / REF / ALT and the GT locator, applies the biallelic-SNP and
// region rules of the text path (hb_head.cuh) to the same fields, and kept records are compacted in file order.
//
// GT decode.  The tile of kernel 3: 64 records x 128 samples, a transpose.  A record's values for the tile's samples are
// one contiguous run at an arbitrary alignment; int8 x 2 runs are staged into shared memory with one TMA bulk copy per
// record, as kernel 3 stages its text, and every other type or count is read per sample by a slower branch.  The byte
// planes and the allele bit planes are written from the tile as kernel 3 writes them.
#include "hb_common.cuh"
#include "hb_internal.h"

namespace hb {

// 4 bytes at any offset of the body (the buffer has >= 64 readable bytes of slack after it)
__device__ __forceinline__ uint32_t ld_u32(const uint8_t *__restrict__ t, uint64_t o) {
    const uint32_t *w = reinterpret_cast<const uint32_t *>(t + (o & ~3ull));
    return __funnelshift_r(__ldg(w), __ldg(w + 1), 8u * (uint32_t)(o & 3));
}

// The strict header test of the record at o.  0 = passes (next = offset of the record after it), else a kBcf* reason.
__device__ __forceinline__ uint32_t bcf_check(const uint8_t *__restrict__ t, uint64_t o, uint64_t n, uint32_t n_samples,
                                              uint32_t n_contigs, uint64_t &next) {
    if (o + 33 > n) return kBcfTruncated;                             // 32 fixed bytes + the ID's type byte
    const uint32_t fs = ld_u32(t, o + 28);
    if ((fs & 0xffffffu) != n_samples) return kBcfNSample;
    if (ld_u32(t, o + 8) >= n_contigs) return kBcfContig;             // (a negative int32 is out of range too)
    const uint32_t ls = ld_u32(t, o), li = ld_u32(t, o + 4);
    next = o + 8 + (uint64_t)ls + li;
    if (next > n) return kBcfTruncated;
    const uint32_t n_allele = ld_u32(t, o + 24) >> 16;
    if (ls < 25 || n_allele == 0 || (li == 0) != ((fs >> 24) == 0) || (t[o + 32] & 0xfu) != 7u) return kBcfHead;
    return 0;
}

__global__ void __launch_bounds__(256) bcf_find_kernel(const uint8_t *__restrict__ t, uint64_t n, uint32_t n_samples,
                                                       uint32_t n_contigs, BcfSegs sg) {
    const uint64_t k = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31;
    if (k >= sg.n) return;
    uint64_t found = k == 0 ? 0 : kBcfNone;
    if (k) {
        const uint64_t b = k * sg.bytes, e = min(b + sg.bytes, n);
        for (uint64_t base = b; base < e; base += 32) {
            const uint64_t o = base + lane;
            uint64_t nx = 0, nx2 = 0;
            const bool ok = o < e && bcf_check(t, o, n, n_samples, n_contigs, nx) == 0 &&
                            (nx == n || bcf_check(t, nx, n, n_samples, n_contigs, nx2) == 0);
            const unsigned m = __ballot_sync(0xffffffffu, ok);
            if (m) { found = base + (uint64_t)(__ffs(m) - 1); break; }
        }
    }
    if (lane == 0) { sg.start[k] = found; sg.flag[k] = 1u; }
}

__global__ void __launch_bounds__(256) bcf_chain_kernel(const uint8_t *__restrict__ t, uint64_t n, uint32_t n_samples,
                                                        uint32_t n_contigs, BcfSegs sg) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= sg.n || !sg.flag[k]) return;
    const uint64_t e = min((k + 1) * sg.bytes, n);
    uint64_t s = sg.start[k], bad = 0;
    uint32_t cnt = 0;
    if (s != kBcfNone) {
        while (s < e) {
            uint64_t nx = 0;
            const uint32_t r = bcf_check(t, s, n, n_samples, n_contigs, nx);
            if (r) { bad = (uint64_t)r << 56 | s; break; }
            s = nx;
            ++cnt;
        }
    }
    sg.exit[k] = s;
    sg.count[k] = cnt;
    sg.bad[k] = bad;
    sg.flag[k] = 0u;
}

// every pair (exit of k - 1, start of k): a start that differs is replaced and its segment flagged for another chain
__global__ void __launch_bounds__(256) bcf_verify_kernel(BcfSegs sg, DevStatus *st) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t cnt = 0;
    if (k < sg.n) {
        unsigned long long code = ~0ull;
        if (k && sg.start[k] != sg.exit[k - 1]) {
            code = 2 * k;
            sg.start[k] = sg.exit[k - 1];
            sg.flag[k] = 1u;
        } else if (sg.bad[k]) code = 2 * k + 1;
        if (code != ~0ull) atomicMin(&st->bcf_fail, code);
        cnt = sg.count[k];
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(&st->bcf_records, (unsigned long long)cnt);
}

// exclusive prefix sums of n counts by one CTA (n is the number of segments or of 256-record blocks: at most a few 100 k)
__global__ void __launch_bounds__(1024) bcf_scan_kernel(const uint32_t *__restrict__ in, uint64_t n, uint64_t *__restrict__ out,
                                                        unsigned long long *total) {
    __shared__ uint64_t part[1024];
    const uint32_t tid = threadIdx.x;
    const uint64_t per = (n + 1023) / 1024, b = min(n, tid * per), e = min(n, b + per);
    uint64_t sum = 0;
    for (uint64_t i = b; i < e; ++i) sum += in[i];
    part[tid] = sum;
    __syncthreads();
    for (uint32_t d = 1; d < 1024; d <<= 1) {
        const uint64_t v = tid >= d ? part[tid - d] : 0;
        __syncthreads();
        part[tid] += v;
        __syncthreads();
    }
    uint64_t run = part[tid] - sum;
    for (uint64_t i = b; i < e; ++i) { out[i] = run; run += in[i]; }
    if (tid == 1023 && total) *total = part[1023];
}

__global__ void __launch_bounds__(256) bcf_emit_kernel(const uint8_t *__restrict__ t, uint64_t n, BcfSegs sg,
                                                       uint64_t *__restrict__ rec_off) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= sg.n) return;
    const uint64_t e = min((k + 1) * sg.bytes, n);
    uint64_t s = sg.start[k], r = sg.base[k];
    while (s < e) {                                                   // the proven chain: every header passed the test
        rec_off[r++] = s;
        s += 8 + (uint64_t)ld_u32(t, s) + ld_u32(t, s + 4);
    }
}

__device__ __forceinline__ uint32_t bcf_type_size(uint32_t ty) {
    return ty == 1 || ty == 7 ? 1u : ty == 2 ? 2u : ty == 3 || ty == 5 ? 4u : 0u;
}
// an integer of type ty (1 int8, 2 int16, 3 int32) at q
__device__ __forceinline__ int32_t bcf_int(const uint8_t *__restrict__ t, uint64_t q, uint32_t ty) {
    if (ty == 1) return (int8_t)t[q];
    if (ty == 2) return (int16_t)(t[q] | (t[q + 1] << 8));
    return (int32_t)ld_u32(t, q);
}
// a type byte at q (+ the typed int count that follows a count of 15); false when it runs past lim or is malformed
__device__ __forceinline__ bool bcf_typed(const uint8_t *__restrict__ t, uint64_t &q, uint64_t lim, uint32_t &ty, uint32_t &count) {
    if (q >= lim) return false;
    const uint8_t b = t[q++];
    ty = b & 0xfu;
    count = b >> 4;
    if (count == 15) {
        if (q >= lim) return false;
        const uint32_t ct = t[q++] & 0xfu, sz = bcf_type_size(ct);
        if (ct < 1 || ct > 3 || q + sz > lim) return false;
        const int32_t c = bcf_int(t, q, ct);
        q += sz;
        if (c < 0) return false;
        count = (uint32_t)c;
    }
    return ty == 0 ? count == 0 : bcf_type_size(ty) != 0;
}

struct BcfSite {
    bool keep, has_gt, bad_fmt;
    int32_t chrom;
    uint32_t start, stop, gt_count, gt_type;
    uint8_t ref0, alt0;
    uint64_t gt_off;
};

// the site columns and GT locator of the record at o (whose header passed the test)
__device__ __forceinline__ BcfSite bcf_site(const BcfSiteArgs &a, uint64_t o) {
    const uint8_t *__restrict__ t = a.text;
    BcfSite s;
    s.keep = s.has_gt = s.bad_fmt = false;
    s.gt_count = s.gt_type = 0;
    s.gt_off = 0;
    s.ref0 = s.alt0 = 0;
    const uint32_t ls = ld_u32(t, o), li = ld_u32(t, o + 4);
    s.chrom = (int32_t)ld_u32(t, o + 8);
    const int32_t pos = (int32_t)ld_u32(t, o + 12), rlen = (int32_t)ld_u32(t, o + 16);
    const uint32_t n_allele = ld_u32(t, o + 24) >> 16, n_fmt = ld_u32(t, o + 28) >> 24;
    const uint64_t shared_end = o + 8 + ls, end = shared_end + li;
    s.start = (uint32_t)pos;
    s.stop = (uint32_t)((long long)pos + rlen);
    uint64_t q = o + 32;
    uint32_t ty, c, ref_len = 0, alt_len = 0;
    bool ok = bcf_typed(t, q, shared_end, ty, c) && q + (uint64_t)c * bcf_type_size(ty) <= shared_end;   // ID
    q += (uint64_t)c * bcf_type_size(ty);
    if (ok) {                                                          // REF, then the first ALT
        ok = bcf_typed(t, q, shared_end, ty, c) && (ty == 7 || c == 0) && q + c <= shared_end;
        if (ok) { ref_len = c; if (c) s.ref0 = t[q]; q += c; }
    }
    if (ok && n_allele >= 2) {
        ok = bcf_typed(t, q, shared_end, ty, c) && (ty == 7 || c == 0) && q + c <= shared_end;
        if (ok) { alt_len = c; if (c) s.alt0 = t[q]; }
    }
    // the text path's rules on the same fields: a one-allele record is ALT ".", which is not a SNP
    const bool snp = ok && n_allele == 2 && ref_len <= 1 && alt_len == 1 &&
                     (s.alt0 == 'A' || s.alt0 == 'C' || s.alt0 == 'G' || s.alt0 == 'T');
    bool in_region = a.rid == -1;
    if (a.rid >= 0) in_region = s.chrom == a.rid && (long long)pos < a.end0 && (long long)pos + rlen > a.beg0;
    s.keep = snp && in_region;
    if (!ok) s.bad_fmt = s.keep = true;                               // (reported as a malformed file)
    if (!s.keep || !a.want_gt || a.gt_key < 0) return s;
    q = shared_end;
    for (uint32_t f = 0; f < n_fmt; ++f) {
        uint32_t kt, kc;
        if (!bcf_typed(t, q, end, kt, kc) || kc != 1 || kt < 1 || kt > 3 || q + bcf_type_size(kt) > end) { s.bad_fmt = true; break; }
        const int32_t key = bcf_int(t, q, kt);
        q += bcf_type_size(kt);
        if (!bcf_typed(t, q, end, ty, c)) { s.bad_fmt = true; break; }
        const uint64_t vals = q;
        q += (uint64_t)a.n_samples * c * bcf_type_size(ty);
        if (q > end) { s.bad_fmt = true; break; }
        if (key == a.gt_key) {
            if (ty < 1 || ty > 3) { s.bad_fmt = true; break; }
            s.has_gt = true;
            s.gt_off = vals;
            s.gt_count = c;
            s.gt_type = ty;
            break;
        }
    }
    return s;
}

// pass 0: kept records per block of 256; pass 1: the dense rows (blk_base = exclusive sums of pass 0)
template <int kPass>
__global__ void __launch_bounds__(256) bcf_sites_kernel(const BcfSiteArgs a) {
    __shared__ uint32_t s_warp[8];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint64_t r = (uint64_t)blockIdx.x * 256 + tid;
    BcfSite s;
    s.keep = false;
    if (r < a.n_rec) s = bcf_site(a, a.rec_off[r]);
    const unsigned bal = __ballot_sync(0xffffffffu, s.keep);
    if (lane == 0) s_warp[warp] = __popc(bal);
    __syncthreads();
    uint32_t before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) { const uint32_t c = s_warp[w]; if (w < warp) before += c; total += c; }
    if (kPass == 0) {
        if (tid == 0) a.blk_count[blockIdx.x] = total;
        return;
    }
    if (!s.keep) return;
    if (s.bad_fmt) { atomicAdd(&a.st->bcf_bad_fmt, 1ull); }
    const uint64_t row = a.blk_base[blockIdx.x] + before + __popc(bal & ((1u << lane) - 1u));
    a.start[row] = s.start;
    a.stop[row] = s.stop;
    a.ref[row] = s.ref0;
    a.alt[row] = s.alt0;
    const bool known = s.chrom >= 0 && (uint32_t)s.chrom < a.n_contigs;
    const BcfContig ct = known ? a.contigs[s.chrom] : BcfContig{0, 0, 0, 0};
    a.chrom_abs[row] = ct.name_off;
    a.chrom_len[row] = (uint8_t)ct.name_len;
    a.chrom5[row] = ct.name5;
    RowInfo ri;
    ri.samp_abs = s.gt_off;
    ri.samp_len = s.gt_count;
    ri.cp_row = 0;
    ri.pad = 0;
    const bool gt = s.has_gt && a.n_samples > 0;
    ri.misc = gt ? (s.gt_type | kRowHasSamples) : 255u;
    if (a.want_gt && !gt) atomicAdd(&a.st->n_nogt, 1ull);
    a.rowinfo[row] = ri;
}

void launch_bcf_chain(const uint8_t *d_text, uint64_t nbytes, uint32_t n_samples, uint32_t n_contigs, const BcfSegs &sg, bool find,
                      const Launch &L) {
    if (!sg.n) return;
    if (find) {
        bcf_find_kernel<<<(unsigned)((sg.n * 32 + 255) / 256), 256, 0, L.stream>>>(d_text, nbytes, n_samples, n_contigs, sg);
        count_launch();
    }
    bcf_chain_kernel<<<(unsigned)((sg.n + 255) / 256), 256, 0, L.stream>>>(d_text, nbytes, n_samples, n_contigs, sg);
    count_launch();
}

void launch_bcf_verify(const BcfSegs &sg, DevStatus *d_st, const Launch &L) {
    if (!sg.n) return;
    bcf_verify_kernel<<<(unsigned)((sg.n + 255) / 256), 256, 0, L.stream>>>(sg, d_st);
    count_launch();
}

void launch_bcf_emit(const uint8_t *d_text, uint64_t nbytes, const BcfSegs &sg, uint64_t *d_rec_off, const Launch &L) {
    if (!sg.n) return;
    bcf_scan_kernel<<<1, 1024, 0, L.stream>>>(sg.count, sg.n, sg.base, nullptr);
    bcf_emit_kernel<<<(unsigned)((sg.n + 255) / 256), 256, 0, L.stream>>>(d_text, nbytes, sg, d_rec_off);
    count_launch(2);
}

void launch_bcf_sites(const BcfSiteArgs &a, const Launch &L) {
    if (!a.n_rec) return;
    const uint64_t blocks = (a.n_rec + 255) / 256;
    bcf_sites_kernel<0><<<(unsigned)blocks, 256, 0, L.stream>>>(a);
    bcf_scan_kernel<<<1, 1024, 0, L.stream>>>(a.blk_count, blocks, a.blk_base, &a.st->n_records);
    bcf_sites_kernel<1><<<(unsigned)blocks, 256, 0, L.stream>>>(a);
    count_launch(3);
}

// ---------------------------------------------------------------------------------------------------------------- kernel 3b
constexpr int BD_THREADS = 256;
constexpr int BD_PITCH = kTV + 16;        // as kernel 3: (kTV + 16) / 16 odd => conflict-free 16-byte transposed stores
static_assert(((BD_PITCH / 16) & 1) == 1 && kTS % 2 == 0, "tile geometry");

constexpr int BD_STAGE = 2 * kTS + 16;   // staged bytes per record: 2 * kTS + up to 15 bytes of misalignment

struct BcfGtSmem {
    alignas(128) uint8_t stage[kTV][BD_STAGE];  // int8 x 2 records: sample s's two values at bytes shift + 2s, + 1
    alignas(16) uint8_t out[2][kTS][BD_PITCH];
    uint64_t off[kTV];                          // the tile's first value of the record
    uint32_t count[kTV], type[kTV], shift[kTV];
    int mode[kTV];                              // 0 no GT (zeros), 1 int8 x 2 (staged), 2 any other type or count
    alignas(8) uint64_t bar;
};

__device__ __forceinline__ int bcf_allele(int32_t v) {          // v >= 0
    return (v >> 1) == 0 ? -9 : (int)(int8_t)(uint8_t)((v >> 1) - 1);
}

// One sample's GT vector, count values of type ty at p: the alleles the text path reads from the same record's VCF text.
// A value is (allele + 1) << 1 | phased; 0 and 1 are a missing allele (-9); the allele index is narrowed to int8.
// Returns 0; 1 when the ploidy is not 2 (fewer or more than two values before vector_end, or a value after it); 2 when a
// value before vector_end is one a conforming writer never puts in GT (the type's missing value, a reserved value, any
// other negative one): the sample's alleles are then 0, as for an unreadable allele in text.
__device__ __noinline__ int bcf_gt_sample(const uint8_t *p, uint32_t ty, uint32_t count, int &a0, int &a1) {
    const int32_t vend = ty == 1 ? -127 : ty == 2 ? -32767 : (int32_t)0x80000001u;
    uint32_t pl = count;
    bool bad = false, tail = false;
    int32_t v0 = 0, v1 = 0;
    for (uint32_t i = 0; i < count; ++i) {
        int32_t v;
        if (ty == 1) v = (int8_t)p[i];
        else if (ty == 2) v = (int16_t)(p[2 * i] | (p[2 * i + 1] << 8));
        else v = (int32_t)(p[4 * i] | (p[4 * i + 1] << 8) | (p[4 * i + 2] << 16) | ((uint32_t)p[4 * i + 3] << 24));
        if (pl == count) {
            if (v == vend) pl = i;
            else {
                if (v < 0) bad = true;
                if (i == 0) v0 = v; else if (i == 1) v1 = v;
            }
        } else if (v != vend) tail = true;
    }
    if (bad) { a0 = 0; a1 = 0; return 2; }
    a0 = pl >= 1 ? bcf_allele(v0) : -9;
    a1 = pl >= 2 ? bcf_allele(v1) : -128;
    return pl != 2 || tail ? 1 : 0;
}

// kSubset: as kernel 3's, only the columns of `sel` are decoded, counted and written, to their planes.  Every sample's values
// sit at a fixed stride, so the records' column counts are known without reading the others.
template <bool kSubset>
__global__ void __launch_bounds__(BD_THREADS, 4)
bcf_decode_kernel(const uint8_t *__restrict__ text, const RowInfo *__restrict__ rowinfo, uint64_t n_rows, uint32_t n_samples,
                  uint32_t n_stiles, int8_t *__restrict__ gt0, int8_t *__restrict__ gt1, uint64_t gt_stride,
                  uint32_t *__restrict__ bits, uint64_t bits_stride, uint32_t *__restrict__ ploidy_err,
                  uint32_t *__restrict__ badgt_err, DevStatus *__restrict__ st, SampleSel sel) {
    __shared__ BcfGtSmem sm;
    const int tid = threadIdx.x;
    const uint32_t tile = blockIdx.x;
    const uint32_t tile_r = tile / n_stiles;
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
    }
    __syncthreads();

    // ---- phase 0: each record's run of values for the tile's samples; int8 x 2 runs are requested with TMA
    if (tid < kTV) {
        int mode = 0;
        uint64_t off = 0;
        uint32_t count = 0, ty = 0;
        if ((uint32_t)tid < nr) {
            const RowInfo ri = rowinfo[r0 + tid];
            ty = ri.misc & 0xffu;
            if ((ri.misc & kRowHasSamples) && ty != 255u) {
                count = ri.samp_len;
                off = ri.samp_abs + (uint64_t)s0 * count * (ty == 1 ? 1u : ty == 2 ? 2u : 4u);
                mode = ty == 1 && count == 2 ? 1 : 2;
            }
        }
        sm.off[tid] = off;
        sm.count[tid] = count;
        sm.type[tid] = ty;
        sm.mode[tid] = mode;
        sm.shift[tid] = (uint32_t)(off & 15ull);
        if (mode == 1) {                                   // [off & ~15, off + 2 ns) rounded up to 16 bytes (the body has slack)
            const uint32_t bytes = (uint32_t)(((off & 15ull) + 2u * ns + 15ull) & ~15ull);
            mbar_expect_tx(&sm.bar, bytes);
            tma_load_1d(sm.stage[tid], text + (off & ~15ull), bytes, &sm.bar);
        } else {
            mbar_arrive(&sm.bar);
        }
    }
    if (tid == kTV) mbar_wait(&sm.bar, 0);
    __syncthreads();

    // ---- phase 2: one thread = 1 sample x 16 records; lanes run along samples (broadcast reads of the staged words)
    for (int item = tid; item < kTS * (kTV / 16); item += BD_THREADS) {
        const int s = item % kTS, rg = item / kTS;
        uint32_t acc0[4] = {0, 0, 0, 0}, acc1[4] = {0, 0, 0, 0};
        if ((uint32_t)s < ns && (!kSubset || sel_has(msk, s))) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const int r = 16 * rg + i;
                const int mode = sm.mode[r];
                if (mode == 0) continue;
                int a0, a1, rc = 0;
                if (mode == 1) {
                    const uint8_t *v = &sm.stage[r][sm.shift[r] + 2 * s];
                    const uint32_t x = v[0] - 2u, y = v[1] - 2u;
                    if ((x | y) < 4u) { a0 = (int)(x >> 1); a1 = (int)(y >> 1); }           // 0 / 1 alleles, either phase
                    else rc = bcf_gt_sample(v, 1, 2, a0, a1);
                } else {
                    const uint32_t ty = sm.type[r], c = sm.count[r];
                    rc = bcf_gt_sample(text + sm.off[r] + (uint64_t)s * c * (ty == 1 ? 1u : ty == 2 ? 2u : 4u), ty, c, a0, a1);
                }
                if (rc == 2) { atomicAdd(&st->n_bad_gt, 1ull); atomicAdd(&badgt_err[sel_plane<kSubset>(msk, sbase, s0, s)], 1u); }
                else if (rc == 1) atomicAdd(&ploidy_err[sel_plane<kSubset>(msk, sbase, s0, s)], 1u);
                acc0[i >> 2] |= (uint32_t)(uint8_t)a0 << (8 * (i & 3));
                acc1[i >> 2] |= (uint32_t)(uint8_t)a1 << (8 * (i & 3));
            }
        }
        *reinterpret_cast<uint4 *>(&sm.out[0][s][16 * rg]) = make_uint4(acc0[0], acc0[1], acc0[2], acc0[3]);
        *reinterpret_cast<uint4 *>(&sm.out[1][s][16 * rg]) = make_uint4(acc1[0], acc1[1], acc1[2], acc1[3]);
    }
    __syncthreads();

    // ---- phase 3 (as kernel 3): kTV contiguous bytes per (plane, sample), and the same alleles as bit planes
    {
        constexpr int PIECES = kTV / 16;
        static_assert(PIECES == 4 && (2 * kTS * PIECES) % BD_THREADS == 0, "the 4 pieces of a row sit in 4 neighbouring lanes");
        for (int item = tid; item < 2 * kTS * PIECES; item += BD_THREADS) {
            const int piece = item % PIECES;
            const int ps = item / PIECES;
            const int s = ps % kTS, p = ps / kTS;
            const bool live = (uint32_t)s < ns && (!kSubset || sel_has(msk, s));
            uint4 v = make_uint4(0, 0, 0, 0);
            if (live) {
                v = *reinterpret_cast<const uint4 *>(&sm.out[p][s][16 * piece]);
                int8_t *dst = (p ? gt1 : gt0) + (uint64_t)sel_plane<kSubset>(msk, sbase, s0, s) * gt_stride + r0 + 16ull * piece;
                stg_stream(reinterpret_cast<uint4 *>(dst), v);
            }
            uint32_t t = pack_lsb4(v.x) | (pack_lsb4(v.y) << 4) | (pack_lsb4(v.z) << 8) | (pack_lsb4(v.w) << 12);
            if ((v.x | v.y | v.z | v.w) & 0xFEFEFEFEu)
                t |= (pack_nz4(v.x) | (pack_nz4(v.y) << 4) | (pack_nz4(v.z) << 8) | (pack_nz4(v.w) << 12)) << 16;
            const uint32_t u = __shfl_down_sync(0xffffffffu, t, 1);
            const uint32_t bw = (t & 0xffffu) | (u << 16), nw = (t >> 16) | (u & 0xffff0000u);
            const uint32_t bw1 = __shfl_down_sync(0xffffffffu, bw, 2), nw1 = __shfl_down_sync(0xffffffffu, nw, 2);
            if (live && piece == 0) {
                uint32_t *row = bits + (uint64_t)sel_plane<kSubset>(msk, sbase, s0, s) * bits_stride + (r0 >> 7) * kBitGroupWords + ((r0 >> 5) & 3u);
                *reinterpret_cast<uint2 *>(row + 4 * p) = make_uint2(bw, bw1);
                *reinterpret_cast<uint2 *>(row + 4 * (2 + p)) = make_uint2(nw, nw1);
            }
        }
    }
}

void launch_bcf_decode(const uint8_t *d_text, const RowInfo *d_rowinfo, uint64_t n_rows, uint32_t n_samples, int8_t *d_gt0,
                       int8_t *d_gt1, uint64_t gt_stride, uint32_t *d_bits, uint64_t bits_stride, uint32_t *d_ploidy_err,
                       uint32_t *d_badgt_err, DevStatus *d_st, const SampleSel &sel, const Launch &L) {
    if (!n_rows || !n_samples) return;
    const uint32_t n_stiles = (n_samples + kTS - 1) / kTS;
    const uint64_t tiles = (n_rows + kTV - 1) / kTV * n_stiles;
    auto kernel = sel.mask ? bcf_decode_kernel<true> : bcf_decode_kernel<false>;
    kernel<<<(unsigned)tiles, BD_THREADS, 0, L.stream>>>(d_text, d_rowinfo, n_rows, n_samples, n_stiles, d_gt0, d_gt1, gt_stride,
                                                         d_bits, bits_stride, d_ploidy_err, d_badgt_err, d_st, sel);
    count_launch();
}

}  // namespace hb
