"""Region queries through a tabix / CSI index: the parse reads and inflates only the BGZF members of the query's span, and
gives the rows, genotype planes, sample errors, CHROM runs and stored frames a full scan gives.  The indexes are written
by tests/index_writer.py (and by pysam when it is installed), not by this project's reader."""
import os
import sys
import tempfile

import pytest

import bcf_writer
import index_writer as iw
import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CONTIGS = ["chr1", "chr2", "chrX"]


@pytest.fixture(scope="module")
def capi(built):
    from haplohyped_varawareml_b200 import capi as c
    return c


def bgzf_at_lines(text: bytes, every: int) -> bytes:
    """BGZF whose members end on record ends: every `every` lines close a member."""
    lines = text.split(b"\n")
    out = []
    for i in range(0, len(lines), every):
        chunk = b"\n".join(lines[i:i + every]) + (b"\n" if i + every < len(lines) else b"")
        if chunk:
            out.append(synth.bgzf_compress(chunk)[:-28])
    return b"".join(out) + synth.bgzf_compress(b"")


def results(p):
    out = {"sites": [x.tobytes() for x in p.sites()], "names": p.sample_names(), "runs": p.chrom_runs(),
           "errors": [x.tobytes() for x in p.sample_errors()], "n": p.info.n_records}
    if p.info.n_records and p.info.n_samples:
        out["matrix"] = [x.tobytes() for x in p.matrix()]
    return out


def regions(text):
    """Regions that exercise the query: whole contig, open end, a range across members, one position, before the first and
    after the last record, an absent contig, and a deletion / INFO/END record that starts before the region."""
    vo = iw.VirtualOffsets([(0, 0, len(text), 1)])
    names, _, recs = iw.vcf_records(text, vo)
    on2 = [r for r in recs if r[0] == 1]
    mid = on2[len(on2) // 2]
    out = ["chr2", "chr2:%d" % (mid[1] + 1), "chr2:%d-%d" % (on2[100][1] + 1, on2[400][1] + 1),
           "chr2:%d-%d" % (mid[1] + 1, mid[1] + 1), "chr1:1-100", "chrX:%d-%d" % (on2[-1][2] + 10**7, on2[-1][2] + 2 * 10**7),
           "chr9", "chr9:1-1000"]
    long = [r for r in on2 if r[2] - r[1] > 4]
    if long:
        r = long[len(long) // 2]
        out.append("chr2:%d-%d" % (r[1] + 3, r[1] + 4))
    return out


def expected_read(data, index, text, region):
    """(header bytes, span bytes) the reader reads: the members through the one where the header ends, and the members
    from the first chunk's block through the block the last chunk ends in."""
    members = iw.bgzf_members(data)
    body = text.index(b"\n", text.index(b"#CHROM")) + 1
    head = next(a + size for a, off, n, size in members if off <= body - 1 < off + n)
    idx = iw.read(index)
    name, _, rng = region.partition(":")
    names = idx["names"] or CONTIGS
    b, _, e = rng.partition("-")
    beg, end = (int(b) - 1 if b else 0), (int(e) if e else 1 << 40)
    ch = iw.query(idx, names.index(name), beg, end) if name in names else []
    span = 0
    if ch:
        c0, c1, u1 = ch[0][0] >> 16, ch[-1][1] >> 16, ch[-1][1] & 0xffff
        span = c1 + (next(size for a, _, _, size in members if a == c1) if u1 else 0) - c0
    return head, span, head == members[0][3]


def check_parity(capi, path, data, index, regs, text=None):
    for region in regs:
        with capi.use_index(False):
            full = capi.Parse.from_file(path, region)
            assert full.index_info[0] is False
            want = results(full)
        with capi.use_index(True):
            p = capi.Parse.from_file(path, region)
            assert p.index_info[0] is True, region
            assert results(p) == want, region
            if text is not None:                          # no more than the header and the query's span
                head, span, one_member = expected_read(data, index, text, region)
                if one_member:
                    assert p.index_info[1] == head + span, region
                else:                                     # the header is read in rounds that double the bytes
                    assert head + span <= p.index_info[1] <= 2 * head + span, region
            q = capi.Parse.from_vcf_bytes(data, region, index=index)
            assert q.index_info[0] is True
            assert results(q) == want, region


def write_pair(d, name, data, index, ext):
    path = os.path.join(d, name)
    open(path, "wb").write(data)
    open(path + ext, "wb").write(index)
    return path


@pytest.mark.parametrize("fmt", ["tbi", "csi"])
@pytest.mark.parametrize("container", ["bgzf", "small_members", "member_ends"])
@pytest.mark.parametrize("kind", ["GT", "GT:GQ:DP"])
def test_query_parity_vcf(capi, fmt, container, kind):
    text = iw.multi_contig_vcf(CONTIGS, 1500, 7, seed=5, fmt=kind, info_end=True)
    data = {"bgzf": lambda: synth.bgzf_compress(text), "small_members": lambda: synth.bgzf_compress(text, block=300),
            "member_ends": lambda: bgzf_at_lines(text, 7)}[container]()
    index = iw.write(iw.index_vcf(text, data, fmt))
    with tempfile.TemporaryDirectory() as d:
        path = write_pair(d, "x.vcf.gz", data, index, "." + fmt)
        check_parity(capi, path, data, index, regions(text), text=text)


def test_query_parity_csi_high_positions(capi):
    text = iw.multi_contig_vcf(CONTIGS, 1000, 5, seed=8, info_end=True, first_pos=(1 << 29) + 12345)
    data = synth.bgzf_compress(text, block=4000)
    index = iw.write(iw.index_vcf(text, data, "csi"))
    with tempfile.TemporaryDirectory() as d:
        path = write_pair(d, "x.vcf.gz", data, index, ".csi")
        check_parity(capi, path, data, index, regions(text))


def test_query_parity_bcf(capi):
    text = iw.multi_contig_vcf(CONTIGS, 1200, 6, seed=9, fmt="GT:GQ")
    raw = bcf_writer.vcf_to_bcf(text)
    data = synth.bgzf_compress(raw, block=700)
    index = iw.write(iw.index_bcf(raw, data))
    with tempfile.TemporaryDirectory() as d:
        path = write_pair(d, "x.bcf", data, index, ".csi")
        check_parity(capi, path, data, index, regions(text))
        p = capi.Parse.from_file(path, "chr2")
        assert p.info.tokenizer_used == 4 and p.index_info[0]


def test_frames_and_load_vcf(capi, built):
    sys.path.insert(0, os.path.join(ROOT, "haplohyped-varawareml_b200"))
    import parse_vcf
    text = iw.multi_contig_vcf(CONTIGS, 3000, 40, seed=2)
    data = synth.bgzf_compress(text, block=5000)
    index = iw.write(iw.index_vcf(text, data, "tbi"))
    with tempfile.TemporaryDirectory() as d:
        path = write_pair(d, "x.vcf.gz", data, index, ".tbi")
        for region in ("chr2", "chr1:10100000-10300000"):
            got = {}
            for on in (False, True):
                with capi.use_index(on):
                    parse_vcf.cache_clear()
                    p = capi.Parse.from_file(path, region)
                    assert p.index_info[0] is on
                    got[on] = (p.compress(0).fetch_packed()[0].tobytes(),
                               parse_vcf.load_vcf(path, "s0000", region), parse_vcf.load_vcf(path, "s0039", region),
                               parse_vcf.load_vcf_without_sample(path, region))
            assert got[True] == got[False], region
    parse_vcf.cache_clear()


@pytest.mark.parametrize("case", ["stale", "bad_magic", "truncated", "plain_gzip"])
def test_ignored_index(capi, case):
    import gzip
    text = iw.multi_contig_vcf(CONTIGS, 600, 5, seed=4, info_end=True)
    data = synth.bgzf_compress(text, block=2000)
    raw = iw.index_vcf(text, data, "tbi")
    index = iw.write(raw)
    if case == "bad_magic":
        index = iw.write(b"TBX\1" + raw[4:])
    elif case == "truncated":
        index = iw.write(raw[:len(raw) // 2])
    elif case == "plain_gzip":
        data = gzip.compress(text)
    with tempfile.TemporaryDirectory() as d:
        path = write_pair(d, "x.vcf.gz", data, index, ".tbi")
        if case == "stale":
            st = os.stat(path)
            os.utime(path + ".tbi", (st.st_atime - 100, st.st_mtime - 100))
        for region in ("chr2", "chr2:10100000-10200000"):
            with capi.use_index(False):
                want = results(capi.Parse.from_file(path, region))
            p = capi.Parse.from_file(path, region)
            assert p.index_info[0] is False
            assert results(p) == want
            if case != "stale":
                q = capi.Parse.from_vcf_bytes(data, region, index=index)
                assert q.index_info[0] is False and results(q) == want


def test_bcf_above_text_limit(capi):
    text = iw.multi_contig_vcf(CONTIGS, 1500, 8, seed=6, fmt="GT:GQ:DP")
    raw = bcf_writer.vcf_to_bcf(text)
    data = synth.bgzf_compress(raw, block=0xff00)
    index = iw.write(iw.index_bcf(raw, data))
    vcf = capi.Parse.from_vcf_bytes(synth.bgzf_compress(text), "chr2:10100000-10150000")
    assert vcf.info.n_records > 0
    with tempfile.TemporaryDirectory() as d:
        path = write_pair(d, "x.bcf", data, index, ".csi")
        capi.lib().hb_parse_set_text_limit(len(raw) // 3)
        try:
            p = capi.Parse.from_file(path, "chr2:10100000-10150000")
            assert p.index_info[0] is True
            assert results(p) == results(vcf)
            with capi.use_index(False):
                with pytest.raises(capi.HaploError) as e:
                    capi.Parse.from_file(path, "chr2:10100000-10150000")
                assert e.value.code == 10 and "exceeds the text limit" in str(e.value)
        finally:
            capi.lib().hb_parse_set_text_limit(0)


def test_pysam_written_index(capi):
    pysam = pytest.importorskip("pysam")
    text = iw.multi_contig_vcf(CONTIGS, 1500, 5, seed=13, info_end=True)
    data = synth.bgzf_compress(text, block=3000)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "x.vcf.gz")
        open(path, "wb").write(data)
        pysam.tabix_index(path, preset="vcf", force=True)
        index = open(path + ".tbi", "rb").read()
        # htslib writes its bins in hash-table order: the same index, compared bin by bin
        ours = iw.read(capi.build_index(data, "tbi"))
        theirs = iw.read(index)
        assert theirs["names"] == ours["names"] and theirs["refs"] == ours["refs"]
        check_parity(capi, path, data, index, regions(text))
        open(path + ".tbi", "wb").write(capi.build_index(data, "tbi"))
        full = [str(r) for r in pysam.TabixFile(path).fetch("chr2")]
        assert full == [x.decode() for x in text.split(b"\n") if x.startswith(b"chr2\t")]
