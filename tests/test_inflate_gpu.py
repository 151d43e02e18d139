"""GPU BGZF inflate (the step in front of the path, SURVEY.md 8f rank 1) against stock zlib: the members are
produced by Python's zlib (an independent, third-party DEFLATE encoder) in BGZF framing, inflated on the GPU
and compared byte for byte with the input.  Dynamic, fixed and stored DEFLATE blocks, all levels."""
import gzip
import os
import struct
import zlib

import numpy as np
import pytest

import oracle
import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def capi(built):
    from haplohyped_varawareml_b200 import capi as c
    return c


def _vcf_text(n=3000, s=60, fmt="GT", seed=1):
    text, samples = synth.random_vcf(n, s, seed=seed, fmt=fmt, kinds="mixed")
    return text, samples


@pytest.mark.parametrize("level", [1, 6, 9])
def test_vcf_text_roundtrip(capi, level):
    text, _ = _vcf_text(fmt="GT:GQ:DP" if level == 6 else "GT")
    assert len(text) > 200_000                                         # several members
    assert capi.bgzf_inflate(synth.bgzf_compress(text, level)) == text


def test_block_types_and_edges(capi):
    rng = np.random.default_rng(5)
    noise = rng.integers(0, 256, 150_000, dtype=np.uint8).tobytes()    # incompressible -> stored blocks
    assert capi.bgzf_inflate(synth.bgzf_compress(noise, 6)) == noise
    assert capi.bgzf_inflate(synth.bgzf_compress(noise, 0)) == noise   # level 0: stored only
    text, _ = _vcf_text(800, 20)
    assert capi.bgzf_inflate(synth.bgzf_compress(text, 6, strategy=zlib.Z_FIXED)) == text          # fixed Huffman
    assert capi.bgzf_inflate(synth.bgzf_compress(text, 6, strategy=zlib.Z_HUFFMAN_ONLY)) == text   # no matches at all
    assert capi.bgzf_inflate(synth.bgzf_compress(text, 6, strategy=zlib.Z_RLE)) == text            # distance-1 matches only
    runs = (b"A" * 70_000 + b"ab" * 40_000 + bytes(range(256)) * 300)                              # overlapping copies, long matches
    assert capi.bgzf_inflate(synth.bgzf_compress(runs, 9)) == runs
    skew = bytes(rng.choice(np.arange(256, dtype=np.uint8), 120_000, p=np.r_[0.6, 0.2, [0.2 / 254] * 254]))
    assert capi.bgzf_inflate(synth.bgzf_compress(skew, 9)) == skew     # very uneven code lengths (> 10-bit codes)
    assert capi.bgzf_inflate(synth.bgzf_compress(b"x", 6)) == b"x"
    assert capi.bgzf_inflate(synth.bgzf_compress(b"", 6)) == b""       # EOF member only
    small = synth.bgzf_compress(text, 6, block=777)                    # many tiny members
    assert capi.bgzf_inflate(small) == text


def test_corrupt_and_foreign_input_is_rejected(capi, golden_dir):
    text, _ = _vcf_text(500, 10)
    good = bytearray(synth.bgzf_compress(text, 6))
    bad = bytearray(good)
    bad[18 + 40] ^= 0x55                                               # inside the first DEFLATE payload
    try:
        out = capi.bgzf_inflate(bytes(bad))
        assert out != text                                             # (a flipped bit may still be a valid stream)
    except capi.HaploError:
        pass
    plain = open(os.path.join(golden_dir, "chr22.filtered.vcf.gz"), "rb").read()                    # plain gzip, not BGZF
    with pytest.raises(capi.HaploError):
        capi.bgzf_inflate(plain)


def test_bgzf_file_through_the_reference_api(capi, tmp_path, built):
    """A bgzipped VCF through parse_vcf.load_vcf / hb_parse_file: GPU inflate -> GPU parse, vs the oracle on the text."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "haplohyped-varawareml_b200"))
    import parse_vcf
    text, samples = _vcf_text(2500, 17, seed=9)
    path = str(tmp_path / "chr22.filtered.vcf.gz")
    open(path, "wb").write(synth.bgzf_compress(text, 6))
    gz = str(tmp_path / "same.vcf.gz")
    with gzip.open(gz, "wb") as f:
        f.write(text)
    for s in (samples[0], samples[9], samples[16]):
        exp = oracle.parse_text(text, s, "chr22")
        got = parse_vcf.load_vcf(path, s, "chr22")
        assert len(got) == exp["n"]
        assert [r[1] for r in got] == list(exp["start"]) and [r[5] for r in got] == list(exp["gt0"]) and [r[6] for r in got] == list(exp["gt1"])
        assert got == parse_vcf.load_vcf(gz, s, "chr22")                # plain gzip (CPU zlib) gives the same tuples
    p = capi.Parse.from_file(path, region="chr22")
    assert p.sample_names() == samples and p.info.compressed_bytes == os.path.getsize(path) and p.info.ms_inflate > 0
    pb = capi.Parse.from_vcf_bytes(open(path, "rb").read(), region="chr22")          # the same bytes from host memory
    assert pb.sample_names() == samples and np.array_equal(pb.matrix()[0], p.matrix()[0])
    pc = capi.Parse.from_file(gz, region="chr22")                                      # plain gzip: one zlib stream on the host
    assert pc.info.compressed_bytes == 0 and np.array_equal(pc.matrix()[1], p.matrix()[1])
    ora = oracle.parse_text(text, "*", "chr22")
    g0, g1 = p.matrix()
    assert np.array_equal(g0, ora["gt0"]) and np.array_equal(g1, ora["gt1"])


def test_gzip_members_with_a_file_name_are_read(capi):
    """Members that carry FNAME next to the BGZF 'BC' subfield (FLG = FEXTRA | FNAME) are valid gzip but not what bgzip
    writes: the GPU inflater refuses them and the host's zlib reads them, member by member, with their CRCs checked."""
    text, _ = _vcf_text(2000, 23, seed=4)
    name = b"chr22.vcf\0"
    members = []
    for i in range(0, len(text), 40_000):
        chunk = text[i:i + 40_000]
        c = zlib.compressobj(6, zlib.DEFLATED, -15)
        payload = c.compress(chunk) + c.flush()
        bsize = 12 + 6 + len(name) + len(payload) + 8
        head = struct.pack("<BBBBIBBH", 0x1f, 0x8b, 8, 4 | 8, 0, 0, 0xff, 6) + b"BC" + struct.pack("<HH", 2, bsize - 1)
        members.append(head + name + payload + struct.pack("<II", zlib.crc32(chunk), len(chunk)))
    data = b"".join(members)
    assert len(members) > 1 and gzip.decompress(data) == text
    ora = oracle.parse_text(text, "*", "chr22")
    p = capi.Parse.from_vcf_bytes(data, region="chr22")
    assert p.info.n_records == ora["n"]
    g0, g1 = p.matrix()
    assert np.array_equal(g0, ora["gt0"]) and np.array_equal(g1, ora["gt1"])
    start, stop, ref, alt = p.sites()
    assert np.array_equal(start, ora["start"]) and np.array_equal(stop, ora["stop"])
    assert np.array_equal(ref, ora["ref"]) and np.array_equal(alt, ora["alt"])


@pytest.mark.parametrize("fmt,kinds,slab,block", [("GT", "phased", 5000, 0xff00), ("GT", "mixed", 30000, 4000),
                                                  ("GT:GQ:DP", "mixed", 9000, 1500), ("GT", "mixed", 1 << 30, 0xff00)])
def test_stream_bgzf_host_equals_oracle(capi, fmt, kinds, slab, block):
    """hb_parse_stream_bgzf_host: BGZF members cross PCIe compressed in slabs, are inflated on the GPU behind the
    unfinished line of the slab before, parsed and fetched -- the same matrix as the oracle, whatever the slab and
    member sizes (lines straddle members and slabs)."""
    text, samples = synth.random_vcf(1500, 41, seed=78, fmt=fmt, kinds=kinds)
    ora = oracle.parse_text(text, "*", "chr22")
    gz = synth.bgzf_compress(text, block=block)
    ns, tb, body = capi.bgzf_vcf_info(gz)
    assert ns == len(samples) and tb == len(text) and body == len(text) - len(synth.body_of(text))
    r = capi.parse_stream_bgzf_host(gz, capacity=1500, region="chr22", slab_bytes=slab)
    assert r["n"] == ora["n"] and r["n_slabs"] >= 1
    if slab < len(text):
        assert r["n_slabs"] > 1
    assert np.array_equal(r["gt0"], ora["gt0"]) and np.array_equal(r["gt1"], ora["gt1"])
    assert np.array_equal(r["start"], ora["start"]) and np.array_equal(r["stop"], ora["stop"])
    assert np.array_equal(r["ref"], ora["ref"]) and np.array_equal(r["alt"], ora["alt"])
    assert r["ploidy_err"].sum() == 0 and r["badgt_err"].sum() == 0
    with pytest.raises(capi.HaploError):                               # capacity is checked, not overrun
        capi.parse_stream_bgzf_host(gz, capacity=ora["n"] - 1, region="chr22", slab_bytes=slab)


def test_stream_bgzf_host_edges(capi):
    # no newline at the end of the file; a slab smaller than one line is an error, not a wrong result
    text, samples = synth.random_vcf(300, 200, seed=9, fmt="GT", kinds="phased", site_mix=False)
    ora = oracle.parse_text(text, "*", "chr22")
    gz = synth.bgzf_compress(text[:-1], block=3000)
    r = capi.parse_stream_bgzf_host(gz, capacity=300, region="chr22", slab_bytes=20000)
    assert r["n"] == ora["n"] == 300 and r["n_slabs"] > 5
    assert np.array_equal(r["gt0"], ora["gt0"]) and np.array_equal(r["gt1"], ora["gt1"]) and np.array_equal(r["start"], ora["start"])
    with pytest.raises(capi.HaploError):
        capi.parse_stream_bgzf_host(synth.bgzf_compress(text, block=300), capacity=300, region="chr22", slab_bytes=500)
    # uniform GT-only text (walker path) in many slabs
    spec = capi.synth_spec(4000, 300, seed=3, mix=1)
    text = capi.synth_header(spec) + capi.synth_host(spec)
    ora = oracle.parse_text(text, "*", "chr22")
    r = capi.parse_stream_bgzf_host(synth.bgzf_compress(text), capacity=4000, region="chr22", slab_bytes=len(text) // 7)
    assert r["n"] == ora["n"] and r["n_slabs"] >= 7
    assert np.array_equal(r["gt0"], ora["gt0"]) and np.array_equal(r["gt1"], ora["gt1"]) and np.array_equal(r["start"], ora["start"])


def test_stream_bgzf_host_grows_every_cached_slot(capi):
    """A one-slab call grows the buffers of both cached slots, so a later two-slab call of that size finds room in each."""
    text, _ = synth.random_vcf(1500, 41, seed=79, fmt="GT", kinds="mixed")
    ora = oracle.parse_text(text, "*", "chr22")
    gz = synth.bgzf_compress(text, block=4000)
    capi.lib().hb_cache_clear()
    for slab in (8000, 1 << 30, len(text) // 2 + 4000):
        r = capi.parse_stream_bgzf_host(gz, capacity=1500, region="chr22", slab_bytes=slab)
        assert r["n"] == ora["n"] and np.array_equal(r["gt0"], ora["gt0"]) and np.array_equal(r["gt1"], ora["gt1"])
        assert np.array_equal(r["start"], ora["start"]) and np.array_equal(r["alt"], ora["alt"])
    assert r["n_slabs"] == 2
    capi.lib().hb_cache_clear()


def test_streamed_resident_parse_gives_the_whole_file_chunks(capi):
    """Chunk continuity across slabs: a .vcf.gz streamed through HBM in >= 5 slabs (hb_parse_stream_bgzf_resident) gives the
    same resident parse as the whole-file call -- same matrix, site columns, CHROM runs, per-sample errors -- and therefore
    byte-identical stored chunks with the whole file's h5py chunk geometry (vcf_to_h5.py:135, chunks=True on the whole
    dataset): no chunk boundary sees a slab boundary."""
    text, samples = synth.random_vcf(9000, 41, seed=23, fmt="GT", kinds="mixed")
    bg = capi.bgzf_compress_host(text, 6)
    whole = capi.Parse.from_vcf_bytes(bg, region="chr22")
    for slab in (len(text) // 7 + 1, 150_000):
        streamed, n_slabs = capi.Parse.from_vcf_bytes_streamed(bg, region="chr22", slab_bytes=slab)
        assert n_slabs >= 5
        assert streamed.info.n_records == whole.info.n_records and streamed.info.n_lines == whole.info.n_lines
        assert streamed.sample_names() == whole.sample_names() == samples
        for a, b in zip(streamed.matrix(), whole.matrix()):
            assert np.array_equal(a, b)
        for a, b in zip(streamed.sites(), whole.sites()):
            assert np.array_equal(a, b)
        assert streamed.chrom_column() == whole.chrom_column()
        for a, b in zip(streamed.sample_errors(), whole.sample_errors()):
            assert np.array_equal(a, b)
        for cr in (0, 100):
            fw, fs = whole.compress(cr), streamed.compress(cr)
            assert fs.info.chunk_records == fw.info.chunk_records and fs.info.n_chunks == fw.info.n_chunks
            bw, ow, zw = fw.fetch_packed()
            bs, os_, zs = fs.fetch_packed()
            assert np.array_equal(zw, zs) and np.array_equal(ow, os_) and np.array_equal(bw, bs)      # byte-identical frames
            fw.close(); fs.close()
        with pytest.raises(capi.HaploError):
            streamed.rerun()                                   # there is no text to parse again
        streamed.close()
    # no region filter, sites only
    s2, _ = capi.Parse.from_vcf_bytes_streamed(bg, region="", want_gt=False, slab_bytes=200_000)
    w2 = capi.Parse.from_vcf_bytes(bg, region="", want_gt=False)
    assert s2.info.n_records == w2.info.n_records and s2.chrom_column() == w2.chrom_column()
    for a, b in zip(s2.sites(), w2.sites()):
        assert np.array_equal(a, b)
