"""BCF 2.2 input on the GPU (kernels 1b and 3b): every BCF parse must give what the VCF path gives on the VCF text of the
same records, and what the oracle gives on that text."""
import gzip
import os
import struct
import sys
import tempfile

import numpy as np
import pytest

import bcf_writer
import oracle
import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def capi(built):
    from haplohyped_varawareml_b200 import capi as c
    return c


@pytest.fixture
def segment(capi):
    """hb_set_bcf_segment_bytes for one test."""
    def set_(n):
        capi.lib().hb_set_bcf_segment_bytes(int(n))
    yield set_
    capi.lib().hb_set_bcf_segment_bytes(0)


def _wrap(bcf, container):
    if container == "bgzf":
        return synth.bgzf_compress(bcf)
    if container == "bgzf_small":
        return synth.bgzf_compress(bcf, block=97)
    if container == "gzip":
        return gzip.compress(bcf)
    return bcf


def _compare(capi, text, bcf, region="", want_gt=True, container="bgzf", rerun=False):
    pb = capi.Parse.from_vcf_bytes(_wrap(bcf, container), region=region, want_gt=want_gt)
    if rerun:
        pb.rerun()
    pv = capi.Parse.from_vcf_bytes(synth.bgzf_compress(text), region=region, want_gt=want_gt)
    ib, iv = pb.info, pv.info
    assert iv.n_records == ib.n_records
    if ib.n_records or len(synth.body_of(text)):
        assert ib.tokenizer_used == 4
    assert pb.sample_names() == pv.sample_names()
    for a, b in zip(pb.sites(), pv.sites()):
        assert np.array_equal(a, b)
    assert pb.chrom_column() == pv.chrom_column()
    assert pb.chrom_runs() == pv.chrom_runs()
    assert ib.n_nogt == iv.n_nogt and ib.n_bad_gt == iv.n_bad_gt
    pl, bg = pv.sample_errors()
    if want_gt:
        for a, b in zip(pb.matrix(), pv.matrix()):
            assert np.array_equal(a, b)
        for a, b in zip(pb.sample_errors(), (pl, bg)):
            assert np.array_equal(a, b)
    if pl.sum() == 0 and bg.sum() == 0:
        ora = oracle.parse_text(text, "*" if want_gt else None, region)
        assert ib.n_records == ora["n"]
        start, stop, ref, alt = pb.sites()
        assert np.array_equal(start, ora["start"]) and np.array_equal(stop, ora["stop"])
        assert np.array_equal(ref, ora["ref"]) and np.array_equal(alt, ora["alt"])
        assert pb.chrom_column() == ora["chrom"]
        if want_gt and ora["n"]:
            g0, g1 = pb.matrix()
            assert np.array_equal(g0, ora["gt0"]) and np.array_equal(g1, ora["gt1"])
    return pb, pv


@pytest.mark.parametrize("fmt", ["GT", "GT:GQ:DP", "DP:GT"])
@pytest.mark.parametrize("container", ["bgzf", "bgzf_small", "gzip", "plain"])
def test_random_vcf(capi, fmt, container):
    text, _ = synth.random_vcf(300, 37, seed=7 * len(fmt) + len(container), fmt=fmt, info_end=True)
    _compare(capi, text, bcf_writer.vcf_to_bcf(text), container=container)


@pytest.mark.parametrize("gt_type", [None, bcf_writer.INT16, bcf_writer.INT32])
def test_multidigit_and_wide_types(capi, gt_type):
    text, _ = synth.random_vcf(400, 130, seed=5, fmt="GT:GQ", multidigit=True)
    pb, _ = _compare(capi, text, bcf_writer.vcf_to_bcf(text, gt_type=gt_type))
    assert pb.info.n_records > 0


def test_int32_alleles_and_later_gt_position(capi):
    text, samples = synth.random_vcf(200, 20, seed=8, fmt="GQ:GT:DP")
    lines = text.split(b"\n")
    k = next(i for i, ln in enumerate(lines) if ln and not ln.startswith(b"#") and b"\tA\tC\t" in ln)
    f = lines[k].split(b"\t")
    f[9] = b"5:20000|1:7"                    # (20001 << 1) needs int32; the text path narrows 20000 to int8 32
    lines[k] = b"\t".join(f)
    text = b"\n".join(lines)
    _compare(capi, text, bcf_writer.vcf_to_bcf(text, gt_pos=2))
    _compare(capi, text, bcf_writer.vcf_to_bcf(text, idx=False))


def test_ploidy_and_unreadable_values(capi):
    """Haploid, triploid and '.' calls are ploidy errors of their sample; the type's missing value in GT is badgt."""
    samples = synth.sample_names(4)
    body = ["chr22\t%d\t.\tA\tG\t.\tPASS\t.\tGT\t%s" % (100 + i, "\t".join(g)) for i, g in enumerate([
        ("0|1", "1", "0|0", "1|1"), ("0|1|1", "0/1", ".", "1|0"), ("./.", ".|1", "0|.", "1/1")])]
    text = (synth.header(samples) + "\n".join(body) + "\n").encode()
    bcf = bytearray(bcf_writer.vcf_to_bcf(text))
    pb, pv = _compare(capi, text, bytes(bcf))
    pl, _ = pb.sample_errors()
    assert pl.tolist() == [1, 1, 1, 0]
    # sample 3 of the last record: values (2, 2) -> int8 missing (0x80) in its first slot
    last = bytes(bcf).rfind(b"\x21")                   # the GT type byte of the last record (count 2, int8)
    bcf[last + 1 + 2 * 3] = 0x80
    p = capi.Parse.from_vcf_bytes(synth.bgzf_compress(bytes(bcf)))
    pl2, bg2 = p.sample_errors()
    assert bg2.tolist() == [0, 0, 0, 1] and p.info.n_bad_gt == 1
    g0, g1 = p.matrix()
    assert g0[3, 2] == 0 and g1[3, 2] == 0


@pytest.mark.parametrize("mix", [0, 1])
@pytest.mark.parametrize("S", [1, 3, 128, 129, 2504])
def test_synth_host(capi, mix, S):
    spec = capi.synth_spec(300 if S == 2504 else 1500, S, seed=S + mix, mix=mix)
    text = capi.synth_header(spec) + capi.synth_host(spec)
    _compare(capi, text, bcf_writer.vcf_to_bcf(text))


@pytest.mark.parametrize("region", ["", "chr22", "chr22:10020000-10060000", "chr21", "chrX"])
def test_regions_and_sites_only(capi, region):
    text, _ = synth.random_vcf(500, 9, seed=21, fmt="GT:GQ")
    bcf = bcf_writer.vcf_to_bcf(text)
    _compare(capi, text, bcf, region=region)
    _compare(capi, text, bcf, region=region, want_gt=False)


def test_header_only_and_no_records(capi):
    text = synth.header(synth.sample_names(3)).encode()
    for c in ("bgzf", "plain"):
        pb = capi.Parse.from_vcf_bytes(_wrap(bcf_writer.vcf_to_bcf(text), c))
        assert pb.info.n_records == 0 and pb.sample_names() == synth.sample_names(3)
    text2, _ = synth.random_vcf(50, 3, seed=2)
    lines = [ln for ln in text2.split(b"\n") if ln.startswith(b"#") or b"\tA\tC,G\t" in ln]   # no biallelic SNP kept
    _compare(capi, b"\n".join(lines) + b"\n", bcf_writer.vcf_to_bcf(b"\n".join(lines) + b"\n"))


def test_segment_boundaries_at_every_offset(capi, segment):
    """Segments of 64 + k bytes over records of varying length put a segment boundary at every offset of a record."""
    text, _ = synth.random_vcf(400, 5, seed=3, fmt="GT:GQ:DP", info_end=True)
    bcf = bcf_writer.vcf_to_bcf(text)
    for k in range(0, 80, 7):
        segment(64 + k)
        _compare(capi, text, bcf, rerun=k == 0)


def test_records_longer_than_a_segment(capi, segment):
    text, _ = synth.random_vcf(60, 300, seed=4, fmt="GT:GQ:DP")
    segment(100)                                    # a record is ~1.5 KB: 15 segments each
    _compare(capi, text, bcf_writer.vcf_to_bcf(text))


def test_fake_record_header_in_genotype_bytes(capi, segment):
    """DP values that spell two record headers which pass the strict test: the segment that starts at them chains off
    the true records, and only the repair from the exit before it gives the right rows."""
    samples = synth.sample_names(24)
    S = len(samples)
    rows = []
    for i in range(20):
        dp = [str(5 + j) for j in range(S)]
        if i == 2:
            # fake 1 at the DP of sample 2: l_shared 27 + l_indiv 1 -> fake 2 36 bytes on; fake 2 jumps 1000 bytes
            w1 = [27, 1, 0, 7, 1, 0x7F800001, 2 << 16, 1 << 24 | S]
            w2 = [27 + 1000, 1, 1, 9, 1, 0x7F800001, 2 << 16, 1 << 24 | S]
            words = w1 + [0x41414107] + w2 + [0x41414107]
            for j, w in enumerate(words):
                dp[2 + j] = str(w - (1 << 32) if w >= 1 << 31 else w)
        rows.append("chr22\t%d\t.\tA\tG\t.\tPASS\t.\tDP:GT\t%s" % (1000 + 10 * i, "\t".join(
            "%s:%d|%d" % (dp[j], j & 1, (i + j) & 1) for j in range(S))))
    text = (synth.header(samples) + "\n".join(rows) + "\n").encode()
    bcf = bcf_writer.vcf_to_bcf(text)
    l_text = struct.unpack("<I", bcf[5:9])[0]
    body = bcf[9 + l_text:]
    fake = body.index(struct.pack("<II", 27, 1) + struct.pack("<i", 0))
    segment(fake - 3)                               # segment 1 begins 3 bytes before the fake header
    _compare(capi, text, bcf)


@pytest.mark.parametrize("case", ["truncated", "n_sample", "past_end", "contig", "version"])
def test_malformed(capi, case):
    text, _ = synth.random_vcf(40, 4, seed=6)
    bcf = bytearray(bcf_writer.vcf_to_bcf(text))
    l_text = struct.unpack("<I", bcf[5:9])[0]
    body = 9 + l_text
    rec2 = body + 8 + sum(struct.unpack("<II", bcf[body:body + 8]))          # the second record
    if case == "truncated":
        bcf = bcf[:-5]
        want = "truncated"
    elif case == "n_sample":
        bcf[rec2 + 28] = 5
        want = "n_sample differs from the header's 4 samples"
    elif case == "past_end":
        bcf[rec2:rec2 + 4] = struct.pack("<I", 1 << 30)
        want = "truncated"
    elif case == "contig":
        bcf[rec2 + 8:rec2 + 12] = struct.pack("<i", 77)
        want = "CHROM is not an index"
    else:
        bcf[4] = 1
        want = "BCF version 2.1 is not supported"
    for c in ("bgzf", "plain"):
        with pytest.raises(capi.HaploError) as e:
            capi.Parse.from_vcf_bytes(_wrap(bytes(bcf), c))
        assert e.value.code == 6 and want in str(e.value)


def test_frames_identical_to_vcf(capi):
    spec = capi.synth_spec(6000, 131, seed=9, mix=0)
    text = capi.synth_header(spec) + capi.synth_host(spec)
    pb, pv = _compare(capi, text, bcf_writer.vcf_to_bcf(text))
    for cr in (0, 4883):
        fb, fv = pb.compress(cr), pv.compress(cr)
        assert fb.fetch_packed()[0].tobytes() == fv.fetch_packed()[0].tobytes()


def test_load_vcf_on_bcf(capi, built):
    sys.path.insert(0, os.path.join(ROOT, "haplohyped-varawareml_b200"))
    import parse_vcf
    text, samples = synth.random_vcf(300, 6, seed=12, fmt="GT:GQ")
    with tempfile.TemporaryDirectory() as d:
        vcf, bcf = os.path.join(d, "x.vcf.gz"), os.path.join(d, "x.bcf")
        open(vcf, "wb").write(synth.bgzf_compress(text))
        open(bcf, "wb").write(synth.bgzf_compress(bcf_writer.vcf_to_bcf(text)))
        for s in (samples[0], samples[-1]):
            assert parse_vcf.load_vcf(bcf, s, "chr22") == parse_vcf.load_vcf(vcf, s, "chr22")
        assert parse_vcf.load_vcf_without_sample(bcf, "chr22") == parse_vcf.load_vcf_without_sample(vcf, "chr22")
        assert parse_vcf.load_vcf_without_sample(bcf, "") == parse_vcf.load_vcf_without_sample(vcf, "")
        p = capi.Parse.from_file(bcf)
        assert p.info.tokenizer_used == 4


def test_full_shape(capi):
    spec = capi.synth_spec(60_000, 2504, seed=7, mix=0)
    text = capi.synth_header(spec) + capi.synth_host(spec)
    pv = capi.Parse.from_vcf_bytes(capi.bgzf_compress_host(text, 1))
    start, stop, ref, alt = pv.sites()
    g0, g1 = pv.matrix()
    bcf = bcf_writer.bcf_from_columns(capi.synth_header(spec), "chr22", start, ref, alt, g0, g1)
    pb = capi.Parse.from_vcf_bytes(capi.bgzf_compress_host(np.frombuffer(bcf, np.uint8), 1))
    assert pb.info.tokenizer_used == 4 and pb.info.n_records == pv.info.n_records
    for a, b in zip(pb.sites(), (start, stop, ref, alt)):
        assert np.array_equal(a, b)
    b0, b1 = pb.matrix()
    assert np.array_equal(b0, g0) and np.array_equal(b1, g1)
    pb.rerun()
    assert np.array_equal(pb.matrix()[0], g0)
    fb, fv = pb.compress(0), pv.compress(0)
    assert fb.fetch_packed()[0].tobytes() == fv.fetch_packed()[0].tobytes()


def test_streaming_entry_points_refuse_bcf(capi):
    text, _ = synth.random_vcf(30, 3, seed=1)
    bcf = bcf_writer.vcf_to_bcf(text)
    data = synth.bgzf_compress(bcf)
    for call in (lambda: capi.bgzf_vcf_info(data),
                 lambda: capi.parse_stream_bgzf_host(data, 100),
                 lambda: capi.Parse.from_vcf_bytes_streamed(data),
                 lambda: capi.parse_stream_host(bcf, 3, 100)):
        with pytest.raises(capi.HaploError) as e:
            call()
        assert e.value.code == 10 and "BCF streaming is not supported" in str(e.value)


def test_pysam_written_bcf(capi):
    pysam = pytest.importorskip("pysam")
    text, _ = synth.random_vcf(200, 5, seed=13, fmt="GT:GQ")
    with tempfile.TemporaryDirectory() as d:
        src, dst = os.path.join(d, "x.vcf"), os.path.join(d, "x.bcf")
        open(src, "wb").write(text)
        with pysam.VariantFile(src) as fi, pysam.VariantFile(dst, "wb", header=fi.header) as fo:
            for r in fi:
                fo.write(r)
        _compare(capi, text, open(dst, "rb").read(), container="plain")
