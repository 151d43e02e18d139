/*
 * haplo_b200.h -- C ABI of libhaplo_b200.so: the B200-native VCF -> tensor hot path.
 *
 * Plain pointers and sizes only (no torch / pybind types).  Every entry point names the
 * reference interface it replaces (paths relative to the HaploHyped-VarAwareML checkout).
 * All functions return HB_OK (0) or an HB_ERR_* code; hb_last_error() gives the thread-local
 * message.  There is NO CPU fallback: every compute entry point needs a CUDA device of
 * compute capability 10.x and fails with HB_ERR_CUDA otherwise.
 */
#ifndef HAPLO_B200_H
#define HAPLO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HB_OK 0
#define HB_ERR_IO 1        /* cannot open / read / inflate the input */
#define HB_ERR_HEADER 2    /* no #CHROM line */
#define HB_ERR_SAMPLE 3    /* unknown sample (vcfpp.h:369-378 runtime_error) */
#define HB_ERR_PLOIDY 4    /* GT of the requested sample is not diploid (parse_vcf.cpp:46 assert) */
#define HB_ERR_GT 5        /* allele neither digits nor '.' (htslib "Couldn't read GT data") */
#define HB_ERR_FORMAT 6    /* wrong number of columns */
#define HB_ERR_NOGT 7      /* FORMAT has no GT (vcfpp.h:550-552 "genotypes not present") */
#define HB_ERR_MEM 8
#define HB_ERR_CUDA 9      /* no usable device / CUDA failure: the product never falls back to CPU */
#define HB_ERR_ARG 10

const char *hb_last_error(void);
const char *hb_version(void);
/* number of this library's kernels launched by the calling process so far (bench "gpu_launches") */
uint64_t hb_kernel_launches(void);

/* ------------------------------------------------------------------------------------------
 * A. Reference-facing entry points.  These are what the reference's pybind11 module binds:
 *      VCFLoader::load_vcf                cpp/parse_vcf.cpp:30-71   (bound at :120-121)
 *      VCFLoader::load_vcf_without_sample cpp/parse_vcf.cpp:80-113  (bound at :122-123)
 *    Same argument meaning (path, sample id, region string; "" = whole file), same filter
 *    (biallelic SNP, vcfpp.h:990-1000), same values (POS-1, POS-1+rlen, REF, ALT, int8 alleles,
 *    -9 = missing).  Results are columnar; the pybind11 shim turns them into the list of tuples.
 *    One (file, region) is parsed ONCE on the GPU for all samples and cached, so the reference's
 *    per-donor call pattern (vcf_to_h5.py:150-152) costs one parse, not n_samples parses.
 * ------------------------------------------------------------------------------------------ */
typedef struct hb_records {
    uint64_t n;                 /* records kept */
    uint32_t n_samples;         /* samples in the file header */
    const uint32_t *start;      /* [n] POS-1                       (vcfpp.h:1118-1121) */
    const uint32_t *stop;       /* [n] POS-1+rlen                  (vcfpp.h:1124-1127) */
    const char *ref;            /* [n] one char per record         (vcfpp.h:1130-1133) */
    const char *alt;            /* [n] one char per record         (vcfpp.h:1142-1151) */
    const uint32_t *chrom_off;  /* [n] offset of the NUL-terminated CHROM in chrom_pool (vcfpp.h:1076) */
    const char *chrom_pool;
    uint64_t chrom_pool_len;
    const int8_t *gt0;          /* [n] first allele index or -9; NULL without sample (parse_vcf.cpp:51) */
    const int8_t *gt1;          /* [n] second allele                                   (parse_vcf.cpp:52) */
    void *owner_;               /* private */
} hb_records;

/* in_vcf: a .vcf, .vcf.gz or .bcf, as the reference's hts_open reads all three (vcfpp.h:1381) */
int hb_load_vcf(const char *in_vcf, const char *sample, const char *chrom, hb_records *out);
int hb_load_vcf_without_sample(const char *in_vcf, const char *chrom, hb_records *out);
void hb_records_free(hb_records *r);
/* Device memory the cache behind hb_load_vcf may pin (genotype planes of the parsed files): entries go least recently
 * used first.  0 = the default, 40 % of the device.  A file whose size / mtime / inode changed is parsed again. */
void hb_cache_set_limit(uint64_t hbm_bytes);
void hb_cache_clear(void);      /* drop the per-(file, region) device-resident parse cache, the kept frame buffer and the
                                 * device slots the streaming entry points keep between calls */

/* ------------------------------------------------------------------------------------------
 * B. Text-level entry points: the kernels behind A, on a caller-supplied buffer of decompressed
 *    VCF *body* text (no header lines).  Replaces the hot loop parse_vcf.cpp:41-62 /
 *    vcfpp.h:1455-1484 (tokenise), :1076-1151 (site columns), :546-588 (GT decode) for ALL
 *    samples at once.  Output stays in HBM in the byte-shuffled (planar) layout:
 *        gt[plane][sample][row]  int8, row stride = gt_stride, plane 0 = phase1, 1 = phase2.
 * ------------------------------------------------------------------------------------------ */
typedef struct hb_parse hb_parse;

typedef struct hb_parse_opts {
    uint32_t n_samples;     /* sample columns per record (from the #CHROM line) */
    const char *region;     /* "" / NULL, "chr22" or "chr22:beg-end" (tabix syntax, vcfpp.h:1424-1451) */
    int end_is_int;         /* header declares INFO/END as Integer: END overrides rlen */
    int want_gt;            /* 0: sites only (load_vcf_without_sample) */
    int device;             /* CUDA device ordinal */
    int tokenizer;          /* 0 auto, 1 newline-only (GT-only text), 2 newline+tab checkpoints,
                               3 head walker (uniform GT-only text; falls back to 1/2 when it cannot prove itself exact) */
    void *stream;           /* cudaStream_t or NULL */
} hb_parse_opts;

typedef struct hb_parse_info {
    uint64_t text_bytes, n_lines, n_records;
    uint32_t n_samples;
    uint64_t gt_stride;             /* bytes between consecutive samples in a plane */
    const int8_t *d_gt[2];          /* device: plane base pointers */
    const uint32_t *d_start, *d_stop;
    const uint8_t *d_ref, *d_alt;
    uint64_t n_nonuniform;          /* records that took the general (tab-scan) decode path */
    uint64_t n_bad_gt, n_bad_cols;  /* malformed alleles / column-count mismatches */
    uint64_t n_nogt;                /* kept records without a GT key or without sample columns */
    int tokenizer_used;             /* 1 newline-only, 2 newline + tab checkpoints, 3 head walker, 4 BCF records (ms_tokenize
                                       = locate, ms_sites = site columns, ms_decode = GT decode) */
    float ms_tokenize, ms_sites, ms_decode;   /* CUDA-event kernel times of the last parse */
    int walker_fallbacks;           /* times the head walker could not prove itself exact and the tokenizer re-ran */
    float ms_inflate;               /* GPU BGZF inflate kernel time (file-level parses of BGZF input), else 0 */
    uint64_t compressed_bytes;      /* BGZF bytes that crossed PCIe instead of the text, else 0 */
} hb_parse_info;

/* text on the HOST (pageable or pinned): H2D copy + kernels.  body must end with '\n'. */
int hb_parse_host_text(const uint8_t *text, uint64_t nbytes, const hb_parse_opts *opts, hb_parse **out);
/* text already in HBM.  d_text must be 16-byte aligned with >= 64 readable bytes of slack after nbytes. */
int hb_parse_device_text(const uint8_t *d_text, uint64_t nbytes, const hb_parse_opts *opts, hb_parse **out);
/* Streaming form: host text -> genotype matrix + site columns in HOST memory, in one call.  The text is cut into
 * slabs of about slab_bytes (0 = 1 GiB) at line boundaries; H2D of the next slab, the kernels of the current one and
 * D2H of the previous one overlap, and device memory is O(slab_bytes) whatever the size of the text.  Use pinned
 * host buffers for the overlap to be real.  gt0/gt1: [n_samples][out_stride] (row = sample, as
 * hb_parse_fetch_matrix with out_stride instead of n_records); out_stride = capacity in records of every output
 * array (HB_ERR_ARG when exceeded; the number of lines is always enough).  Any output pointer may be NULL.
 * ploidy_err / badgt_err: [n_samples], see hb_parse_fetch_sample_errors.  Replaces, for one (file, region), the
 * n_samples calls of parse_vcf.cpp:30-71 that vcf_to_h5.py:150-152 makes. */
int hb_parse_stream_host(const uint8_t *text, uint64_t nbytes, const hb_parse_opts *opts, uint64_t slab_bytes,
                         int8_t *gt0, int8_t *gt1, uint64_t out_stride, uint32_t *start, uint32_t *stop, char *ref,
                         char *alt, uint32_t *ploidy_err, uint32_t *badgt_err, uint64_t *n_records, uint32_t *n_slabs);
/* a whole .vcf / .vcf.gz / .bcf (BGZF, plain gzip or uncompressed; BCF 2.2 is recognised by its magic): header + body,
 * all samples, no per-sample cache.  A BCF gives the rows the VCF text of the same records gives (tokenizer_used 4).
 * BCF is not streamed: a BCF body above the text limit (hb_parse_set_text_limit) fails with HB_ERR_ARG.
 * What the vcf_to_h5 converter drives (src/haplohyped/vcf_to_h5.py:98-101 without the per-donor re-scan). */
int hb_parse_file(const char *in_vcf, const char *region, int want_gt, int device, hb_parse **out);
/* the same for the bytes of a .vcf / .vcf.gz / .bcf already in host memory (BGZF bytes cross PCIe compressed and are
 * inflated on the GPU; pinned memory makes that copy asynchronous) */
int hb_parse_vcf_bytes(const uint8_t *data, uint64_t nbytes, const char *region, int want_gt, int device, hb_parse **out);
/* BGZF bytes of a .vcf.gz in (pinned) host memory -> the same results as hb_parse_stream_host, streamed: slabs of whole
 * BGZF members (about slab_bytes of text each, 0 = 1 GiB) cross PCIe compressed, are inflated on the GPU behind the
 * unfinished last line of the slab before, parsed and fetched; H2D + inflate of slab k + 1 and the D2H of slab k - 1
 * overlap the parse of slab k.  This is the reference's whole read path (tbx_itr_next + vcf_parse1 + getGenotypes,
 * vcfpp.h:1468-1472, :546-588) for all samples at once.  hb_bgzf_vcf_info gives what is needed to size the outputs. */
int hb_bgzf_vcf_info(const uint8_t *bgzf, uint64_t nbytes, uint32_t *n_samples, uint64_t *text_bytes, uint64_t *body_offset);
/* The streaming entry points (hb_parse_stream_host, hb_bgzf_vcf_info, hb_parse_stream_bgzf_host / _resident) read VCF text
 * only: BCF input fails with HB_ERR_ARG. */
int hb_parse_stream_bgzf_host(const uint8_t *bgzf, uint64_t nbytes, const char *region, int want_gt, int device,
                              uint64_t slab_bytes, int8_t *gt0, int8_t *gt1, uint64_t out_stride, uint32_t *start,
                              uint32_t *stop, char *ref, char *alt, uint32_t *ploidy_err, uint32_t *badgt_err,
                              uint64_t *n_records, uint32_t *n_slabs);
/* The same streamed read, but the rows of every slab are appended to ONE device-resident parse: genotype planes and site
 * columns grow in HBM (2.5 bytes per call) while the text never holds more than two slabs.  *out is the handle a whole-
 * file hb_parse_vcf_bytes would have given, minus its text (hb_parse_rerun is refused): the same rows, so
 * hb_compress_records cuts them into the same HDF5 chunks -- `chunks=True` on the whole dataset (vcf_to_h5.py:135) --
 * and chunk boundaries never see slab boundaries.  For files whose text does not fit HBM next to the planes. */
int hb_parse_stream_bgzf_resident(const uint8_t *bgzf, uint64_t nbytes, const char *region, int want_gt, int device,
                                  uint64_t slab_bytes, hb_parse **out, uint32_t *n_slabs);
/* hb_parse_file / hb_parse_vcf_bytes / hb_load_vcf take that streamed route by themselves when the text of a BGZF file
 * would not fit the device next to its planes (text > 0.9 x free / 1.55).  text_bytes != 0 sets the threshold explicitly
 * (bound the HBM a parse may take; tests); 0 = automatic. */
void hb_parse_set_text_limit(uint64_t text_bytes);
/* Lines per walker of the head walker (kernel 1a): 0 = the default (16), at most 20 (a walker has 24 row slots).  Tests
 * use 1-3 to put a walker boundary at every line. */
void hb_set_walker_lines(uint32_t lines);
/* Bytes per segment of the BCF record locator (kernel 1b): 0 = the default, max(64 KiB, 8 x the first record's length);
 * other values are raised to at least 64.  Tests use small segments to put segment boundaries at every offset of a
 * record and to make records longer than a segment. */
void hb_set_bcf_segment_bytes(uint64_t bytes);
/* sample names of a file-level parse, NUL-separated (under a sample subset: the subset's, in header order) */
int hb_parse_samples(hb_parse *p, uint32_t *n, char *names, uint64_t cap, uint64_t *len);
/* Sample subsets: only the listed samples' genotypes are decoded and kept, as htslib's bcf_hdr_set_samples does before it
 * parses.  Planes come out in header order whatever the order of the list: plane j is the j-th selected column of the
 * header, and n_samples (hb_parse_get_info, hb_parse_samples, the frame calls) is the subset's size.  For every selected
 * sample the result is what the full parse of the same bytes gives: the same rows, site columns, CHROM runs and planes,
 * the same per-sample error counts.  The columns of unselected samples are still counted, so a record with too many or
 * too few columns fails with HB_ERR_FORMAT as in the full parse, but their GT text is not parsed: a bad allele or a
 * haploid call there neither fails nor counts (n_bad_gt counts selected samples only).  A list of every sample is the
 * ordinary parse.  hb_parse_rerun repeats the subset.
 * Text level: cols[0..n_cols) are column indices into the opts->n_samples sample columns, ascending and distinct;
 * an empty list, an index out of range, unsorted or repeated fails with HB_ERR_ARG. */
int hb_parse_host_text_subset(const uint8_t *text, uint64_t nbytes, const hb_parse_opts *opts, const uint32_t *cols,
                              uint32_t n_cols, hb_parse **out);
int hb_parse_device_text_subset(const uint8_t *d_text, uint64_t nbytes, const hb_parse_opts *opts, const uint32_t *cols,
                                uint32_t n_cols, hb_parse **out);
/* File level (hb_parse_file / hb_parse_vcf_bytes_indexed with genotypes and a subset; every route they take -- BCF, an
 * index, the slab-streamed route -- takes the subset): names[0..n) in any order.  A name the header does not have fails
 * with HB_ERR_SAMPLE and names it; an empty list or a name given twice fails with HB_ERR_ARG.  index == NULL: what
 * hb_parse_vcf_bytes does. */
int hb_parse_file_subset(const char *in_vcf, const char *region, const char *const *names, uint32_t n, int device,
                         hb_parse **out);
int hb_parse_vcf_bytes_subset(const uint8_t *data, uint64_t nbytes, const uint8_t *index, uint64_t index_n, const char *region,
                              const char *const *names, uint32_t n, int device, hb_parse **out);
/* The header's sample names of a .vcf, .vcf.gz (BGZF or plain gzip) or .bcf, NUL-separated, read from the leading bytes
 * (BGZF members) of the file only; host only, no device needed.  As hb_parse_samples: the names that fit cap are written,
 * *len is what all of them need. */
int hb_file_samples(const char *path, uint32_t *n, char *names, uint64_t cap, uint64_t *len);
/* re-run the kernels of an existing handle on (new contents of) the same device buffer: no allocation */
int hb_parse_rerun(hb_parse *p);
/* the same for a handle made by hb_parse_device_text whose buffer now holds nbytes of (other) text: slab streaming */
int hb_parse_rerun_bytes(hb_parse *p, uint64_t nbytes);
/* give the text buffer of a host-text / file parse back (a 64 GB chromosome needs the HBM for its frames); every result
 * stays valid, only hb_parse_rerun is no longer possible */
int hb_parse_release_text(hb_parse *p);
int hb_parse_get_info(const hb_parse *p, hb_parse_info *info);
/* host copies.  Any pointer may be NULL.  chrom names: see hb_parse_chrom_runs. */
int hb_parse_fetch_sites(hb_parse *p, uint32_t *start, uint32_t *stop, char *ref, char *alt);
int hb_parse_fetch_sample(hb_parse *p, uint32_t sample_index, int8_t *gt0, int8_t *gt1);
int hb_parse_fetch_matrix(hb_parse *p, int8_t *gt0, int8_t *gt1); /* [n_samples][n_records] each */
/* per-sample counts [n_samples]: records whose GT was not diploid (the reference aborts there,
 * parse_vcf.cpp:46) and records whose GT had an unreadable allele (htslib "Couldn't read GT data") */
int hb_parse_fetch_sample_errors(hb_parse *p, uint32_t *ploidy, uint32_t *badgt);
/* CHROM runs: rows [row_begin[i], row_begin[i+1]) share names[i]; names are written NUL-separated.  The names are read
 * from the text on the first call after a parse: a caller that owns the text buffer (hb_parse_device_text) must ask
 * before it overwrites the buffer. */
int hb_parse_chrom_runs(hb_parse *p, uint64_t *n_runs, uint64_t *row_begin, uint64_t max_runs,
                        char *names, uint64_t names_cap, uint64_t *names_len);
void hb_parse_free(hb_parse *p);

/* BGZF (htslib's block gzip: what `bgzip` writes and tabix / vcfpp.h:1381,1468 read) inflated on the GPU, one warp per
 * <= 64 KiB member: host BGZF bytes -> host text.  out == NULL: only *out_len is set.  The file-level entry points
 * (hb_load_vcf, hb_parse_file) use the same kernel but leave the text in HBM.  kernel_ms may be NULL. */
int hb_bgzf_inflate(const uint8_t *bgzf, uint64_t nbytes, uint8_t *out, uint64_t cap, uint64_t *out_len, int device,
                    float *kernel_ms);

/* Host utility for tests and the bench (NOT on the product path, which only reads BGZF): text -> BGZF with stock
 * zlib on all host threads, as `bgzip -@` would.  out == NULL: *len = a sufficient capacity. */
int hb_bgzf_compress_host(const uint8_t *text, uint64_t nbytes, int level, uint8_t *out, uint64_t cap, uint64_t *len);

/* ------------------------------------------------------------------------------------------
 * C. Storage: Blosc byte-shuffle (typesize 35) + LZ4 block encoder + Blosc chunk framing, one
 *    frame (= one stored HDF5 chunk) per (sample, HDF5 chunk) -- what h5py + hdf5plugin produce for
 *    create_dataset('snp_data', compression=32001, compression_opts=(2,2,0,0,5,1,2), chunks=True)
 *    (src/haplohyped/vcf_to_h5.py:119-135).  Filter 32001 is hdf5-blosc, i.e. c-blosc 1.x: a stored
 *    chunk is the bare output of blosc_compress (16-byte header, bstarts, one LZ4 stream per block;
 *    the reference's docs call it "Blosc2", whose own filter id is 32026 -- c-blosc2 reads this
 *    format as well).  Frames stay in HBM until fetched.
 * ------------------------------------------------------------------------------------------ */
typedef struct hb_frames hb_frames;

typedef struct hb_frames_info {
    uint64_t n_records, n_chunks, chunk_records;
    uint32_t n_samples;
    uint64_t total_bytes;           /* all frames of all samples (C_out) */
    uint64_t raw_bytes;             /* 35 * n_records * n_samples */
    float ms_site, ms_frames;       /* kernel times: site templates; fused allele encode + frame assembly */
    uint64_t padded_bytes;          /* bytes of the device frame buffer in use: frames start on 16-byte boundaries */
    const uint8_t *d_frames;        /* device: frames in [sample][chunk] order, see hb_frames_layout */
    uint64_t site_lz4_bytes;        /* LZ4 bytes of the site planes, summed over chunks (shared by every sample) */
} hb_frames_info;

/* chunk_records = 0 -> h5py's auto-chunk heuristic for a 1-D dataset of 35-byte items (hb_guess_chunk_records; it is not
 * clamped, and stays <= 7,489 for every dataset below ~122.7 M records).  chunk_records may be at most 7,489: up to there
 * a stored chunk is ONE Blosc block with ONE LZ4 stream, as c-blosc 1.x cuts blocks of 262,115 bytes at typesize 35,
 * clevel 5, LZ4HC; larger values fail with HB_ERR_ARG.  Chunks above 2,730 records take kernels 4a-L / 4b-L.
 * All frames of all samples are produced in one pass and stay in HBM as ONE buffer, laid out
 * [sample][chunk] with every frame starting on a 16-byte boundary: a sample's dataset is one contiguous
 * byte range, and the whole buffer can be written to the HDF5 file with one write. */
int hb_compress_records(hb_parse *p, uint64_t chunk_records, hb_frames **out);
/* the same for samples [s0, s0 + ns) only: when all frames of a big chromosome do not fit in HBM next to the genotype
 * planes, the converter walks a window over the samples -- hb_frames_set_window(f, s0', ns' <= ns) + hb_frames_rerun.
 * Sample indices of hb_frames_layout / hb_frames_fetch_sample are relative to the window. */
int hb_compress_sample_range(hb_parse *p, uint64_t chunk_records, uint32_t s0, uint32_t ns, hb_frames **out);
int hb_frames_set_window(hb_frames *f, uint32_t s0, uint32_t ns);
/* Attach frames to the parse they were made from (NULL detaches): from then on every hb_parse_rerun of p also
 * starts the site-template kernel of f, on a side stream, as soon as the site columns exist -- it overlaps the GT
 * decoder instead of following it.  hb_frames_rerun then only runs what needs the genotype planes.  The frames must
 * outlive the attachment. */
int hb_parse_attach_frames(hb_parse *p, hb_frames *f);
/* run the kernels again on the (re-parsed) handle the frames were made from: no allocation unless C_out grew.  The
 * record count may differ from the first run when chunk_records was given explicitly (slab streaming: a few chunks
 * more than the first slab had are provided for). */
int hb_frames_rerun(hb_frames *f, hb_parse *p);
int hb_frames_get_info(const hb_frames *f, hb_frames_info *info);
/* offsets (into the frame buffer) and true sizes of every frame, [n_samples][n_chunks]; either may be NULL */
int hb_frames_layout(hb_frames *f, uint64_t *offsets, uint32_t *sizes);
/* the whole frame buffer (padded_bytes) in one D2H copy */
int hb_frames_fetch_all(hb_frames *f, uint8_t *buf, uint64_t cap);
/* All frames packed back to back, [sample][chunk] order, each starting on a 16-byte boundary of buf -- what a converter
 * writes into the HDF5 file with one write (replaces the per-dataset writes of vcf_to_h5.py:131-135).  The frames are
 * gathered out of their slots on the device in pieces and the D2H copy of one piece overlaps the gather of the next:
 * total_bytes (+ < 16 per frame) cross PCIe instead of padded_bytes.  offsets / sizes [n_samples][n_chunks] may be
 * NULL; buf == NULL only reports *total, the bytes buf must hold.  buf should be pinned memory. */
int hb_frames_fetch_packed(hb_frames *f, uint8_t *buf, uint64_t cap, uint64_t *offsets, uint32_t *sizes, uint64_t *total);
/* How hb_frames_fetch_packed moves the frames.  A stored chunk is its HDF5 chunk's template (the LZ4 stream of the 33 site
 * planes, the same for every donor) with 32 patched header bytes and the donor's own tail behind it, so by default
 * (mode 0, when the process may run on >= 4 CPUs) the templates cross PCIe once per chunk, only headers and tails per
 * donor (config 2: 2.7 GB instead of 15.2 GB), and host threads put the frames together in buf with memcpy.  mode 1:
 * every frame is gathered whole on the device and copied (what r01 / r02j did); mode 2: host assembly regardless of the
 * CPU count.  The bytes in buf are the same either way.  hb_set_host_threads: threads used for the assembly
 * (0 = the CPUs the process may run on, at most 16). */
void hb_set_fetch_mode(int mode);
void hb_set_host_threads(int n);
/* BGZF CRC32 check, process-wide, off by default.  On: every BGZF member (.vcf.gz and BGZF .bcf, on every route:
 * hb_parse_file, hb_parse_vcf_bytes, hb_load_vcf, the streamed routes, hb_bgzf_inflate) has the CRC32 of its text compared
 * with its gzip trailer, on the GPU inside the inflate kernel and on the host for the header members.  A mismatch fails
 * with HB_ERR_IO and "BGZF CRC32 mismatch (member i, compressed offset X)", i and X positions in the whole file.  This is
 * what htslib's BGZF reader does; off, a member whose DEFLATE stream is valid but whose bytes changed (any byte of a stored
 * block, many in Huffman-coded data) is accepted as it is.  ISIZE is checked either way; plain gzip input goes through
 * zlib, which always checks the CRC.  hb_load_vcf keeps parses made with the check on apart from those made with it off. */
void hb_set_bgzf_crc_check(int on);
int hb_get_bgzf_crc_check(void);
/* Region queries through a tabix or CSI index (process-wide, on by default).  When the region is not empty and the input
 * is BGZF, hb_parse_file, hb_load_vcf and hb_load_vcf_without_sample look for <path>.tbi, then <path>.csi (a .bcf:
 * <path>.csi only) and read and inflate only the BGZF members between the first and the last chunk the index lists for
 * the region; the GPU region filter still decides which records are kept, so the rows are those of a full scan.  The
 * index is ignored (HB_TRACE says why) when it is older than the data file, does not read, names no sequences, or when the
 * region's span is above the text limit: the file is then scanned whole, as with the setting off.  A contig the index
 * does not know gives a parse with no records. */
void hb_set_use_index(int on);
int hb_get_use_index(void);
/* hb_parse_vcf_bytes with the bytes of the data file's index (.tbi / .csi, as on disk) next to them; index_n == 0 or
 * hb_set_use_index(0): what hb_parse_vcf_bytes does */
int hb_parse_vcf_bytes_indexed(const uint8_t *data, uint64_t nbytes, const uint8_t *index, uint64_t index_n, const char *region,
                               int want_gt, int device, hb_parse **out);
/* whether the parse went through an index (used 1) or scanned the whole input (0); the compressed bytes it read from the
 * data (header members + the span) and the merged chunks of the query.  Any output pointer may be NULL. */
int hb_parse_index_info(const hb_parse *p, int *used, uint64_t *compressed_bytes_read, uint64_t *n_chunks);
/* Build the index of BGZF bytes on the GPU (kernel 7): what `tabix -p vcf` (HB_INDEX_TBI), `tabix -C -m min_shift -p vcf`
 * (HB_INDEX_CSI) or, for a BGZF .bcf, `bcftools index -m min_shift` (CSI only) writes, BGZF-compressed into out[0, *len).
 * min_shift is used by CSI only (TBI is 14 with 5 levels).  out == NULL: *len is set only; a cap below it fails with
 * HB_ERR_ARG and sets *len.  Plain gzip or uncompressed input, TBI for a BCF, and text above the text limit
 * (hb_parse_set_text_limit) fail with HB_ERR_ARG; records out of order ("unsorted positions"), a contig in two blocks
 * ("chromosome blocks not continuous") and a position TBI cannot hold fail with HB_ERR_FORMAT, as tabix does. */
#define HB_INDEX_TBI 0
#define HB_INDEX_CSI 1
int hb_index_bgzf(const uint8_t *data, uint64_t nbytes, int fmt, int min_shift, int device, uint8_t *out, uint64_t cap,
                  uint64_t *len);
/* the index of a file, written to out_path (NULL: <path>.tbi or <path>.csi) */
int hb_index_file(const char *path, int fmt, int min_shift, int device, const char *out_path);
/* bytes the last hb_frames_fetch_packed of this handle moved device -> host (frames or tails + headers + templates, + sizes) */
uint64_t hb_frames_last_d2h_bytes(const hb_frames *f);
/* sizes[n_chunks] of one sample's frames; then the frames themselves, concatenated without padding */
int hb_frames_fetch_sample(hb_frames *f, uint32_t sample_index, uint64_t *sizes, uint8_t *buf, uint64_t cap,
                           uint64_t *total);
void hb_frames_free(hb_frames *f);
uint64_t hb_guess_chunk_records(uint64_t n_records);   /* h5py guess_chunk restated for 35-byte items */
/* Site-plane matcher of the encoder, process-wide: 0 (default) = one hash candidate per position, 1 = 4-way hash
 * buckets (about 5 % smaller frames, the template kernel takes twice as long).  Same decoded bytes either way. */
void hb_set_site_matcher(int deep);
/* Read side (VCFH5Reader.fetch_genotypes, src/utils/h5_reader.py:37-41): n_frames stored HDF5 chunks
 * (bare Blosc chunks as filter 32001 stores them; frame i = frames[offsets[i] .. offsets[i+1])) ->
 * out[i * chunk_nbytes ...], decoded on the GPU (chunk -> LZ4 -> un-shuffle).  Reads what this library writes
 * and what stock c-blosc writes for the path (several blocks, LZ4 / LZ4HC, split streams, memcpyed chunks).
 * planar != 0 keeps the byte-shuffled plane layout (single-block chunks).  Host pointers. */
int hb_decode_frames(const uint8_t *frames, const uint64_t *offsets, uint64_t n_frames, uint64_t chunk_nbytes,
                     uint8_t *out, int planar, int device);
/* The same read, DEVICE in and DEVICE out, for the dataset (haplotype_dataset.py:71 reads a whole (donor, chromosome)
 * dataset per item; here only the chunks a window touches are decoded, and nothing crosses PCIe): n_chunks stored
 * `snp_data` chunks resident in device memory -- chunk i = d_frames[d_off[i] .. d_off[i] + d_len[i]); with d_frames == NULL
 * d_off[i] is the chunk's device address itself, so one call serves chunks of many datasets -- are decoded into
 * record COLUMNS: the chunk_records records of chunk i go to rows [d_row[i], d_row[i] + chunk_records) of d_start /
 * d_stop (uint32), d_ref / d_alt (first byte of the S10 field), d_p1 / d_p2 (int8); any column may be NULL.
 * 35 * chunk_records must fit a warp's shared memory (kernel 6: 6,612 records on a B200); larger values fail with
 * HB_ERR_ARG.
 * d_status[i] = 0 or a non-zero code (corrupt or unsupported chunk; 11 = several Blosc blocks per chunk, which
 * hb_decode_frames reads).  Asynchronous on `stream` (the current device's); all pointers are device pointers. */
int hb_decode_columns_device(const uint8_t *d_frames, const uint64_t *d_off, const uint32_t *d_len, const uint64_t *d_row,
                             uint64_t n_chunks, uint32_t chunk_records, uint32_t *d_start, uint32_t *d_stop, uint8_t *d_ref,
                             uint8_t *d_alt, int8_t *d_p1, int8_t *d_p2, int *d_status, void *stream);
/* The same call for every single-block chunk size, chunk_records <= 7,489 (one c-blosc 1.x block at typesize 35): kernel 6
 * where a chunk fits a warp's shared memory, above that kernel 6-L (one warp per chunk, the block streamed through a
 * 64 KiB history ring, a bad chunk writes no row).  Same arguments, statuses and untouched rows; larger values fail
 * with HB_ERR_ARG. */
int hb_decode_columns_device_large(const uint8_t *d_frames, const uint64_t *d_off, const uint32_t *d_len, const uint64_t *d_row,
                                   uint64_t n_chunks, uint32_t chunk_records, uint32_t *d_start, uint32_t *d_stop, uint8_t *d_ref,
                                   uint8_t *d_alt, int8_t *d_p1, int8_t *d_p2, int *d_status, void *stream);

/* ------------------------------------------------------------------------------------------
 * D. Dataset: batched on-the-fly haplotype construction, replacing
 *    RandomHaplotypeDataset.encode_haplotypes + encode_sequence
 *    (src/datasets/haplotype_dataset.py:86-110, src/utils/common_utils.py:84-103).
 *    All pointers are DEVICE pointers; the per-item arrays hold DEVICE ADDRESSES, so the items of
 *    one batch may come from different chromosomes and donors.  For batch item b:
 *      window  = item_len[b] ASCII bases (any case) at address item_seq[b]
 *      records = item_nrec[b] rows of the (donor, chrom) columns at item_start[b] (uint32, sorted),
 *                item_ref[b] / item_alt[b] (uint8) and item_p1[b] / item_p2[b] (int8 phases)
 *      out     = hap1/hap2 [B][L][C] float32 one-hot; positions >= item_len[b] are all-zero rows
 * ------------------------------------------------------------------------------------------ */
typedef struct hb_hap_batch {
    uint32_t B, L, C;
    const uint64_t *item_seq;        /* [B] address of window position 0 in the reference sequence */
    const uint32_t *item_len;        /* [B] window length (<= L) */
    const uint32_t *item_win_start;  /* [B] genomic coordinate of window position 0 */
    const uint64_t *item_start;      /* [B] address of the record start column */
    const uint64_t *item_ref, *item_alt, *item_p1, *item_p2;   /* [B] addresses of the other columns */
    const uint64_t *item_nrec;       /* [B] records in those columns */
    const int8_t *lut;               /* [256] base byte -> class index (encode_spec order), -1 = none */
    float *hap1, *hap2;              /* [B][L][C] */
    void *stream;
} hb_hap_batch;

int hb_encode_haplotypes(const hb_hap_batch *batch);

/* ------------------------------------------------------------------------------------------
 * E. Synthetic input (bench / tests): seeded, counter-based, identical bytes from the CUDA
 *    generator and from hb_synth_host (SURVEY.md section 8d configs 2-4).
 * ------------------------------------------------------------------------------------------ */
typedef struct hb_synth_spec {
    uint64_t n_variants;
    uint32_t n_samples;
    uint64_t seed;
    uint32_t first_pos, pos_step;   /* POS_i = first_pos + i*pos_step + hash(i) % pos_step */
    uint32_t mix;                   /* bits 0-7: 0 config 2/3 (biallelic SNP, a|b); 1 config 4 (multiallelic,
                                       indel, a/b, missing); bits 8-15: ALT-frequency skew, 0 = u^4 (mean 0.2, the
                                       bench workload), 1 = u^8 (mean 0.11, about Beta(0.2, 2)), 2 = u^16 (mean 0.06) */
    char chrom[16];
} hb_synth_spec;

uint64_t hb_synth_body_bytes(const hb_synth_spec *s);
int hb_synth_header(const hb_synth_spec *s, char *buf, uint64_t cap, uint64_t *len);
int hb_synth_device(const hb_synth_spec *s, uint8_t *d_text, uint64_t cap, int device, void *stream);
int hb_synth_host(const hb_synth_spec *s, uint64_t first_variant, uint64_t n, uint8_t *buf, uint64_t cap,
                  uint64_t *len);

#ifdef __cplusplus
}
#endif
#endif
