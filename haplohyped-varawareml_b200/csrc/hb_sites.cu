// hb_sites.cu -- kernel 2: CHROM / POS / REF / ALT extraction, the biallelic-SNP predicate,
// the region filter, and stream compaction of the records that pass.
//
// Replaces, per record, what the reference reaches through vcfpp accessors after vcf_parse1:
//   isSNP   cpp/vcfpp.h:990-1000      CHROM :1076   Start/End :1118-1127   REF :1130   ALT :1142-1151
// and the loop body of VCFLoader::load_vcf (cpp/parse_vcf.cpp:41-61) up to the genotype read.
// One thread per line walks the nine fixed columns as a small state machine (a record head is
// 50-100 bytes; the sample columns -- kilobytes -- are never touched here).  Kept records get a
// dense row index from a ticketed single-pass decoupled look-back scan, so outputs are written
// directly in row order (file order), ready for the decoder and for the shuffle stage.
#include "hb_common.cuh"
#include "hb_head.cuh"
#include "hb_internal.h"

namespace hb {

constexpr int ST_THREADS = 256;

struct SiteArgs {
    const uint8_t *text;
    LineIndex li;
    uint64_t n_lines;
    uint32_t n_samples;
    RegionArg rg;
    int end_is_int, want_gt, cp_by_line;
    SiteOut out;
    uint64_t *tile_state;
    DevStatus *st;
};

// offset of the byte after the k-th newline of the text (k = global newline ordinal)
__device__ __forceinline__ uint64_t nl_after_global(const LineIndex &li, const uint64_t *s_base, uint64_t k) {
    uint32_t lo = 0, hi = li.n_cta;          // find b with base[b] <= k < base[b+1]
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (s_base[mid] <= k) lo = mid; else hi = mid;
    }
    return li.nl_after[(uint64_t)lo * li.stage_cap + (k - s_base[lo])];
}

constexpr int kMaxTokCta = 1024;

__global__ void __launch_bounds__(ST_THREADS) sites_kernel(const SiteArgs a) {
    __shared__ uint64_t s_cbase[kMaxTokCta + 1];
    __shared__ uint32_t s_tile;
    __shared__ uint32_t s_warp[ST_THREADS / 32];
    __shared__ uint64_t s_base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_tile = atomicAdd(&a.st->ticket, 1u);
    for (uint32_t k = tid; k <= a.li.n_cta; k += ST_THREADS) s_cbase[k] = a.li.base[k];
    __syncthreads();
    const uint64_t tile = s_tile;
    const uint64_t line = tile * ST_THREADS + tid;

    bool keep = false, malformed = false;
    HeadState h;
    HeadVerdict v;
    h.init();
    v.keep = v.uniform = v.malformed = false;
    v.start = v.stop = 0;
    uint64_t ls = 0, le = 0;

    if (line < a.n_lines) {
        ls = line ? nl_after_global(a.li, s_cbase, line - 1) : 0;
        le = nl_after_global(a.li, s_cbase, line) - 1;         // position of '\n'
        const uint8_t *t = a.text;
        if (le > ls && t[le - 1] == '\r') --le;
        if (le > ls && t[ls] != '#') {
            uint64_t q = ls;
            for (; q < le; ++q)
                if (h.feed(t[q], q, a.rg)) break;
            if (!h.has_samples) h.finish_short();
            v = judge_head(h, le, a.n_samples, a.rg, a.end_is_int);
            keep = v.keep;
            malformed = v.malformed;
        }
    }

    // ---- row index: CTA exclusive scan of keep + ticketed look-back across tiles
    unsigned bal = __ballot_sync(0xffffffffu, keep);
    uint32_t wcount = __popc(bal);
    if (lane == 0) s_warp[warp] = wcount;
    __syncthreads();
    uint32_t before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < ST_THREADS / 32; ++w) {
        uint32_t c = s_warp[w];
        if (w < warp) before += c;
        total += c;
    }
    if (warp == 0) {
        uint64_t excl = 0;
        if (tile == 0) {
            if (lane == 0) st_relaxed(&a.tile_state[0], kFlagPre | total);
        } else {
            if (lane == 0) st_relaxed(&a.tile_state[tile], kFlagAgg | total);
            int64_t base = (int64_t)tile - 1;
            for (;;) {
                int64_t idx = base - lane;
                uint64_t w = kFlagPre;
                if (idx >= 0) { do { w = ld_relaxed(&a.tile_state[idx]); } while ((w >> 62) == 0); }
                unsigned pre = __ballot_sync(0xffffffffu, (w >> 62) == 2);
                int P = pre ? (__ffs(pre) - 1) : 31;
                uint64_t v = lane <= P ? (w & kPayload) : 0;
#pragma unroll
                for (int d = 16; d >= 1; d >>= 1) v += __shfl_down_sync(0xffffffffu, v, d);
                excl += __shfl_sync(0xffffffffu, v, 0);
                if (pre) break;
                base -= 32;
            }
            if (lane == 0) st_relaxed(&a.tile_state[tile], kFlagPre | (excl + total));
        }
        if (lane == 0) {
            s_base = excl;
            if ((tile + 1) * ST_THREADS >= a.n_lines) a.st->n_records = excl + total;
        }
    }
    __syncthreads();
    if (malformed) atomicAdd(&a.st->n_bad_cols, 1ull);
    if (!keep) return;
    const uint64_t row = s_base + before + __popc(bal & ((1u << lane) - 1u));
    uint32_t cp_row = kNoCpRow;
    if (a.cp_by_line && a.want_gt && h.has_samples && h.g >= 0 && !v.uniform) {
        // staged id of the line: (tokenizer CTA, local line) -- see hb_tokenize.cu
        uint32_t cb = 0, jl = 0;
        if (line) {
            uint32_t lo = 0, hi = a.li.n_cta;
            while (hi - lo > 1) { uint32_t mid = (lo + hi) >> 1; if (s_cbase[mid] <= line - 1) lo = mid; else hi = mid; }
            cb = lo; jl = (uint32_t)(line - 1 - s_cbase[lo]) + 1;
        }
        cp_row = cb * a.li.stage_cap + jl;
    }
    write_site_row(a.out, a.text, row, ls, le, h, v, a.want_gt, cp_row);
}

void launch_sites(const uint8_t *d_text, const LineIndex &li, uint64_t n_lines, uint32_t n_samples,
                  const RegionArg &rg, int end_is_int, int want_gt, bool cp_by_line, const SiteRows &rows,
                  uint32_t *d_nu_rows, uint64_t *d_tile_state, DevStatus *d_st, const Launch &L) {
    if (!n_lines) return;
    uint64_t tiles = (n_lines + ST_THREADS - 1) / ST_THREADS;
    cudaMemsetAsync(d_tile_state, 0, tiles * sizeof(uint64_t), L.stream);
    SiteArgs a;
    a.text = d_text; a.li = li; a.n_lines = n_lines; a.n_samples = n_samples;
    a.rg = rg; a.end_is_int = end_is_int; a.want_gt = want_gt; a.cp_by_line = cp_by_line ? 1 : 0;
    a.out.start = rows.start; a.out.stop = rows.stop; a.out.ref = rows.ref; a.out.alt = rows.alt;
    a.out.chrom_abs = rows.chrom_abs; a.out.chrom_len = rows.chrom_len; a.out.chrom5 = rows.chrom5; a.out.rowinfo = rows.rowinfo;
    a.out.nu_rows = d_nu_rows; a.out.st = d_st;
    a.tile_state = d_tile_state; a.st = d_st;
    sites_kernel<<<(unsigned)tiles, ST_THREADS, 0, L.stream>>>(a);
    count_launch();
}

// rows whose CHROM differs from the previous row's start a new run (row 0 always does)
__global__ void chrom_runs_kernel(const uint8_t *__restrict__ text, const uint64_t *__restrict__ chrom_abs,
                                  const uint8_t *__restrict__ chrom_len, uint64_t n_rows,
                                  uint64_t *__restrict__ run_rows, uint64_t max_runs, DevStatus *st) {
    uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    bool is_new = r == 0;
    if (!is_new) {
        uint32_t la = chrom_len[r], lb = chrom_len[r - 1];
        if (la != lb) is_new = true;
        else {
            const uint8_t *pa = text + chrom_abs[r], *pb = text + chrom_abs[r - 1];
            for (uint32_t i = 0; i < la; ++i)
                if (pa[i] != pb[i]) { is_new = true; break; }
        }
    }
    if (is_new) {
        unsigned long long k = atomicAdd(&st->n_chrom_runs, 1ull);
        if (k < max_runs) run_rows[k] = r;
    }
}

void launch_chrom_runs(const uint8_t *d_text, const uint64_t *d_chrom_abs, const uint8_t *d_chrom_len,
                       uint64_t n_rows, uint64_t *d_run_rows, uint64_t max_runs, DevStatus *d_st,
                       const Launch &L) {
    if (!n_rows) return;
    uint64_t blocks = (n_rows + 255) / 256;
    chrom_runs_kernel<<<(unsigned)blocks, 256, 0, L.stream>>>(d_text, d_chrom_abs, d_chrom_len, n_rows, d_run_rows,
                                                              max_runs, d_st);
    count_launch();
}

}  // namespace hb
