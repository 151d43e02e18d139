"""BGZF CRC32 check (hb_set_bgzf_crc_check): kernel 0's CRC epilogue and the host's check of the header members.

With the check on, every valid stream must inflate to zlib's bytes and the same bytes as with it off; a member whose
trailer CRC is off by one bit, or whose stored block has one byte changed (a valid DEFLATE stream with the right ISIZE,
which only the CRC can catch), must fail on every route that reads BGZF and name the member and its offset in the whole
file.  With the check off the same files are read as they always were."""
import logging
import os
import re
import struct
import sys
import zlib

import numpy as np
import pytest

import bcf_writer
import synth
import test_inflate_streams_gpu as streams

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BLOCK = 4000                       # text bytes per member of the test files: 16 members per 64 KiB slab


@pytest.fixture(scope="module")
def capi(built):
    from haplohyped_varawareml_b200 import capi as c
    return c


@pytest.fixture(scope="module")
def parse_vcf(built):
    sys.path.insert(0, os.path.join(ROOT, "haplohyped-varawareml_b200"))
    import parse_vcf as m
    return m


@pytest.fixture
def crc_off(capi):
    """every test starts and ends with the check off and an empty parse cache"""
    capi.set_bgzf_crc_check(False)
    capi.lib().hb_cache_clear()
    yield
    capi.set_bgzf_crc_check(False)
    capi.lib().hb_parse_set_text_limit(0)
    capi.lib().hb_cache_clear()


# ---------------------------------------------------------------------------------------------------------------------
# BGZF files with one bad member

def _member(chunk, level):
    c = zlib.compressobj(level, zlib.DEFLATED, -15)
    return streams.bgzf_member(c.compress(chunk) + c.flush(), chunk)


def bgzf_with_bad_member(data, bad, case, block=BLOCK):
    """data -> (BGZF bytes, offset of member `bad`).  Member `bad` is a stored block (level 0); case "trailer" flips bit 0
    of its CRC, case "stored" toggles one byte inside the stored block (in VCF text the first '0' / '1' allele followed by
    '|', so that the text still parses), case None leaves it intact."""
    chunks = [data[i:i + block] for i in range(0, len(data), block)]
    assert 0 <= bad < len(chunks)
    out, at = bytearray(), 0
    for k, ch in enumerate(chunks):
        m = bytearray(_member(ch, 0 if k == bad else 6))
        if k == bad:
            at = len(out)
            if case == "trailer":
                m[-8] ^= 1
            elif case == "stored":
                j = next((i for i in range(len(ch) - 1) if ch[i] in b"01" and ch[i + 1] == ord("|")), len(ch) // 2)
                m[18 + 5 + j] ^= 1 if ch[j] in b"01" else 0x20      # 18 header bytes, then BFINAL/BTYPE, LEN, NLEN
        out += m
    return bytes(out + streams.BGZF_EOF), at


def _positions(n_members):
    return {"first": 0, "middle": n_members // 2, "last": n_members - 1}


def _message(bad, at):
    return re.escape(f"BGZF CRC32 mismatch (member {bad}, compressed offset {at})")


@pytest.fixture(scope="module")
def vcf_text():
    text, samples = synth.random_vcf(3000, 24, seed=31, fmt="GT", kinds="phased", chrom="chr22", site_mix=False)
    assert len(text) > 48 * BLOCK
    return text, samples


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the corrupted files are what they claim to be


@pytest.mark.parametrize("case", ["trailer", "stored"])
def test_corruption_is_caught_by_crc_only(vcf_text, case):
    text = vcf_text[0]
    for bad in _positions((len(text) + BLOCK - 1) // BLOCK).values():
        data, at = bgzf_with_bad_member(text, bad, case)
        m = data[at:at + struct.unpack_from("<H", data, at + 16)[0] + 1]
        d = zlib.decompressobj(-15)
        got = d.decompress(m[18:-8]) + d.flush()
        assert d.eof and len(got) == struct.unpack_from("<I", m, len(m) - 4)[0]     # a valid stream, the right ISIZE
        assert zlib.crc32(got) != struct.unpack_from("<I", m, len(m) - 8)[0]       # and the wrong CRC
        with pytest.raises(zlib.error, match="incorrect data check"):
            zlib.decompress(data[at:at + len(m)], 31)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: valid streams inflate the same with the check on


@pytest.mark.gpu
@pytest.mark.parametrize("name,members", streams.VALID, ids=[n for n, _ in streams.VALID])
def test_valid_stream_inflates_with_check_on(capi, crc_off, name, members):
    want = b"".join(t for _, t in members)
    for fr in streams.framings_for(members):
        f = streams.bgzf_file(members, **fr)
        with capi.crc_check():
            assert capi.bgzf_inflate(f) == want, fr
        assert capi.bgzf_inflate(f) == want


SIZES = (1, 2, 3, 31, 32, 33, 63, 64, 65, 4095, 65535, 65536)


def _text_of(n, seed):
    rng = np.random.default_rng(seed)
    return bytes(rng.choice(np.frombuffer(b"0|1\t\n.ACGT", np.uint8), n).astype(np.uint8).tobytes())


def _payload(text, kind):
    if kind == "stored":
        c = zlib.compressobj(0, zlib.DEFLATED, -15)
    elif kind == "fixed":
        c = zlib.compressobj(6, zlib.DEFLATED, -15, 8, zlib.Z_FIXED)
    else:
        c = zlib.compressobj(9, zlib.DEFLATED, -15)
    return c.compress(text) + c.flush()


@pytest.mark.gpu
@pytest.mark.parametrize("residue", range(32))
def test_member_sizes_at_every_text_offset(capi, crc_off, residue):
    """members of every size and block type, each placed so that its text starts at `residue` mod 32 (odd-length filler
    members in between)"""
    members, off = [], 0
    for i, n in enumerate(SIZES):
        for kind in ("stored", "fixed", "dynamic"):
            if kind == "stored" and n > 65505:
                continue                                      # a stored block of more does not fit a BGZF member
            fill = (residue - off) % 32 or 32
            ft = _text_of(fill, 1000 + fill)
            members.append((_payload(ft, "dynamic"), ft))
            off += fill
            t = _text_of(n, 7 * n + residue)
            members.append((_payload(t, kind), t))
            off += n
    want = b"".join(t for _, t in members)
    f = streams.bgzf_file(members)
    with capi.crc_check():
        got_on = capi.bgzf_inflate(f)
    assert got_on == want == capi.bgzf_inflate(f)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: detection on every route


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["trailer", "stored"])
@pytest.mark.parametrize("where", ["first", "middle", "last"])
def test_whole_file_routes(capi, parse_vcf, crc_off, vcf_text, tmp_path, case, where):
    text, samples = vcf_text
    bad = _positions((len(text) + BLOCK - 1) // BLOCK)[where]
    data, at = bgzf_with_bad_member(text, bad, case)
    path = str(tmp_path / "x.vcf.gz")
    open(path, "wb").write(data)
    msg = _message(bad, at)
    # the check off: read as before
    assert len(capi.bgzf_inflate(data)) == len(text)
    n = capi.Parse.from_vcf_bytes(data).info.n_records
    assert capi.Parse.from_file(path).info.n_records == n == 3000
    ref = parse_vcf.load_vcf(path, samples[1], "chr22")
    capi.lib().hb_cache_clear()
    with capi.crc_check():
        with pytest.raises(capi.HaploError, match=msg):
            capi.bgzf_inflate(data)
        with pytest.raises(capi.HaploError, match=msg):
            capi.Parse.from_file(path)
        with pytest.raises(capi.HaploError, match=msg):
            capi.Parse.from_vcf_bytes(data)
        with pytest.raises(RuntimeError, match="Error parsing VCF file: " + msg):
            parse_vcf.load_vcf(path, samples[1], "chr22")
    assert parse_vcf.load_vcf(path, samples[1], "chr22") == ref


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["trailer", "stored"])
def test_streamed_routes(capi, crc_off, vcf_text, tmp_path, case):
    """bad member in the third of >= 3 slabs: the automatic streamed route of hb_parse_file / hb_parse_vcf_bytes and
    hb_parse_stream_bgzf_resident name its position in the whole file"""
    text, _ = vcf_text
    bad = 2 * 16 + 5                                          # 64 KiB slabs of 16 members of 4,000 bytes: slab 2
    data, at = bgzf_with_bad_member(text, bad, case)
    path = str(tmp_path / "x.vcf.gz")
    open(path, "wb").write(data)
    msg = _message(bad, at)
    whole = capi.Parse.from_vcf_bytes(data)
    p, n_slabs = capi.Parse.from_vcf_bytes_streamed(data, slab_bytes=64 << 10)
    assert n_slabs >= 3 and p.info.n_records == whole.info.n_records
    capi.lib().hb_parse_set_text_limit(128 << 10)             # slabs of 64 KiB inside the whole-file entry points
    h = capi.Parse.from_file(path)
    assert h.info.text_bytes == 0 and h.info.n_records == whole.info.n_records
    with capi.crc_check():
        with pytest.raises(capi.HaploError, match=msg):
            capi.Parse.from_file(path)
        with pytest.raises(capi.HaploError, match=msg):
            capi.Parse.from_vcf_bytes(data)
        capi.lib().hb_parse_set_text_limit(0)
        with pytest.raises(capi.HaploError, match=msg):
            capi.Parse.from_vcf_bytes_streamed(data, slab_bytes=64 << 10)
        ok = bgzf_with_bad_member(text, bad, None)[0]
        q, n_slabs = capi.Parse.from_vcf_bytes_streamed(ok, slab_bytes=64 << 10)
        assert n_slabs >= 3 and q.info.n_records == whole.info.n_records


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["first", "middle", "last"])
def test_bgzf_bcf(capi, parse_vcf, crc_off, vcf_text, tmp_path, where):
    """a BGZF .bcf goes through the same kernel and the same header check"""
    text, samples = vcf_text
    bcf = bcf_writer.vcf_to_bcf(text)
    bad = _positions((len(bcf) + BLOCK - 1) // BLOCK)[where]
    good = bgzf_with_bad_member(bcf, bad, None)[0]
    ref = capi.Parse.from_vcf_bytes(good)
    for case in ("trailer", "stored"):
        data, at = bgzf_with_bad_member(bcf, bad, case)
        path = str(tmp_path / f"{case}.bcf")
        open(path, "wb").write(data)
        if case == "trailer":                                 # the text is intact: the check off reads it unchanged
            p = capi.Parse.from_vcf_bytes(data)
            assert p.info.tokenizer_used == 4
            for a, b in zip(p.sites(), ref.sites()):
                assert np.array_equal(a, b)
            assert all(np.array_equal(a, b) for a, b in zip(p.matrix(), ref.matrix()))
        msg = _message(bad, at)
        with capi.crc_check():
            with pytest.raises(capi.HaploError, match=msg):
                capi.bgzf_inflate(data)
            with pytest.raises(capi.HaploError, match=msg):
                capi.Parse.from_vcf_bytes(data)
            with pytest.raises(capi.HaploError, match=msg):
                capi.Parse.from_file(path)
            with pytest.raises(RuntimeError, match="Error parsing VCF file: " + msg):
                parse_vcf.load_vcf(path, samples[0], "chr22")


# ---------------------------------------------------------------------------------------------------------------------
# GPU: valid data gives the same results either way


@pytest.mark.gpu
def test_results_identical_with_check_on(capi, crc_off):
    spec = capi.synth_spec(6000, 131, seed=9, mix=1)
    text = capi.synth_header(spec) + capi.synth_host(spec)
    for data in (synth.bgzf_compress(text), synth.bgzf_compress(bcf_writer.vcf_to_bcf(text))):
        got = []
        for on in (False, True):
            with capi.crc_check(on):
                p = capi.Parse.from_vcf_bytes(data)
                assert p.info.n_records > 5000
                got.append((p.sites(), p.matrix(), p.compress(0).fetch_packed()[0].tobytes()))
        (s0, m0, f0), (s1, m1, f1) = got
        assert all(np.array_equal(a, b) for a, b in zip(s0, s1))
        assert all(np.array_equal(a, b) for a, b in zip(m0, m1))
        assert f0 == f1


@pytest.mark.gpu
def test_setting_and_context_manager(capi, parse_vcf, crc_off):
    assert capi.get_bgzf_crc_check() is False
    with capi.crc_check():
        assert capi.get_bgzf_crc_check() is True
        with capi.crc_check(False):
            assert capi.get_bgzf_crc_check() is False
        assert capi.get_bgzf_crc_check() is True
    assert capi.get_bgzf_crc_check() is False
    parse_vcf.set_bgzf_crc_check(True)
    assert capi.lib().hb_get_bgzf_crc_check() == 1
    parse_vcf.set_bgzf_crc_check(False)
    assert capi.lib().hb_get_bgzf_crc_check() == 0


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the load_vcf cache keeps the two settings apart


@pytest.mark.gpu
def test_cache_does_not_answer_a_checked_call(capi, parse_vcf, crc_off, vcf_text, tmp_path):
    text, samples = vcf_text
    bad = 20
    data, at = bgzf_with_bad_member(text, bad, "stored")
    path = str(tmp_path / "x.vcf.gz")
    open(path, "wb").write(data)
    first = parse_vcf.load_vcf(path, samples[2], "chr22")
    assert len(first) == 3000
    capi.lib().hb_set_bgzf_crc_check(1)
    with pytest.raises(RuntimeError, match=_message(bad, at)):
        parse_vcf.load_vcf(path, samples[2], "chr22")
    capi.lib().hb_set_bgzf_crc_check(0)
    assert parse_vcf.load_vcf(path, samples[2], "chr22") == first


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the converter skips a file that fails the check


@pytest.mark.gpu
def test_converter_verify_crc(capi, crc_off, tmp_path, caplog):
    from haplohyped_varawareml_b200 import h5_reader, vcf_to_h5
    vdir = tmp_path / "vcf"
    vdir.mkdir()
    samples = None
    for c in (1, 2, 3):
        text, samples = synth.random_vcf(1500, 9, seed=40 + c, fmt="GT", kinds="phased", chrom=f"chr{c}", site_mix=False)
        data = bgzf_with_bad_member(text, 7, "stored" if c == 2 else None)[0]
        (vdir / f"chr{c}.filtered.vcf.gz").write_bytes(data)
    (tmp_path / "donors.txt").write_text("\n".join(samples))
    got = {}
    for verify in (False, True):
        out = tmp_path / f"o{int(verify)}"
        caplog.clear()
        with caplog.at_level(logging.ERROR):
            conv = vcf_to_h5.VCFtoHDF5Converter("c", str(vdir), str(out), str(tmp_path / "donors.txt"), 2, 4,
                                                chromosomes=[1, 2, 3], verify_crc=verify)
            conv.run()
        assert capi.get_bgzf_crc_check() is False
        rd = h5_reader.VCFH5Reader(str(out / "c.h5"))
        got[verify] = {c: rd.fetch_genotypes(samples[0], c).tobytes() for c in ((1, 3) if verify else (1, 2, 3))}
        rd.close()
        if verify:
            assert conv.stats["skipped_files"] == 1 and conv.stats["datasets"] == 2 * 9
            assert any("BGZF CRC32 mismatch (member 7" in r.getMessage() for r in caplog.records)
        else:
            assert conv.stats["skipped_files"] == 0 and conv.stats["datasets"] == 3 * 9
            assert not any("CRC32" in r.getMessage() for r in caplog.records)
            assert len(got[False][2]) > 0
    assert got[True][1] == got[False][1] and got[True][3] == got[False][3]
