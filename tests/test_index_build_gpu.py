"""Indexes built on the GPU (kernel 7): the inflated bytes equal those of the pure-Python restatement of the hts-specs
(tests/index_writer.py) for TBI and CSI of a .vcf.gz and CSI of a .bcf; the builder refuses what tabix refuses; the
vcf_index command line writes and keeps indexes."""
import gzip
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
    lines = text.split(b"\n")
    out = [synth.bgzf_compress(b"\n".join(lines[i:i + every]) + (b"\n" if i + every < len(lines) else b""))[:-28]
           for i in range(0, len(lines), every) if b"\n".join(lines[i:i + every])]
    return b"".join(out) + synth.bgzf_compress(b"")


@pytest.mark.parametrize("fmt", ["tbi", "csi"])
@pytest.mark.parametrize("container", ["bgzf", "block300", "member_ends"])
@pytest.mark.parametrize("kind", ["GT", "GT:GQ:DP"])
def test_vcf_index_equals_python(capi, fmt, container, kind):
    text = iw.multi_contig_vcf(CONTIGS, 1500, 7, seed=21, fmt=kind, info_end=True)
    data = {"bgzf": lambda: synth.bgzf_compress(text), "block300": lambda: synth.bgzf_compress(text, block=300),
            "member_ends": lambda: bgzf_at_lines(text, 5)}[container]()
    assert gzip.decompress(capi.build_index(data, fmt)) == iw.index_vcf(text, data, fmt)


@pytest.mark.parametrize("min_shift", [14, 12])
def test_csi_positions_above_2_29(capi, min_shift):
    text = iw.multi_contig_vcf(CONTIGS, 1000, 4, seed=22, info_end=True, first_pos=(1 << 29) + 777)
    data = synth.bgzf_compress(text, block=2000)
    assert gzip.decompress(capi.build_index(data, "csi", min_shift)) == iw.index_vcf(text, data, "csi", min_shift)
    with pytest.raises(capi.HaploError) as e:
        capi.build_index(data, "tbi")
    assert e.value.code == 6 and "tbi" in str(e.value)


@pytest.mark.parametrize("block", [0xff00, 300])
def test_bcf_index_equals_python(capi, block):
    text = iw.multi_contig_vcf(CONTIGS, 1200, 6, seed=23, fmt="GT:GQ", info_end=True)
    raw = bcf_writer.vcf_to_bcf(text)
    data = synth.bgzf_compress(raw, block=block)
    assert gzip.decompress(capi.build_index(data, "csi")) == iw.index_bcf(raw, data)
    with pytest.raises(capi.HaploError) as e:
        capi.build_index(data, "tbi")
    assert e.value.code == 10


def test_full_shape(capi):
    spec = capi.synth_spec(60_000, 2504, seed=7, mix=0)
    text = capi.synth_header(spec) + capi.synth_host(spec)
    data = capi.bgzf_compress_host(text, 1).tobytes()
    for fmt in ("tbi", "csi"):
        assert gzip.decompress(capi.build_index(data, fmt)) == iw.index_vcf(text, data, fmt)


def test_built_index_serves_queries(capi):
    text = iw.multi_contig_vcf(CONTIGS, 2000, 9, seed=24)
    data = synth.bgzf_compress(text, block=4000)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "x.vcf.gz")
        open(path, "wb").write(data)
        assert capi.index_file(path) == path + ".tbi"
        for region in ("chr2", "chrX:10050000-10100000"):
            p = capi.Parse.from_file(path, region)
            with capi.use_index(False):
                q = capi.Parse.from_file(path, region)
            assert p.index_info[0] and not q.index_info[0]
            assert [x.tobytes() for x in p.sites()] == [x.tobytes() for x in q.sites()]
            assert [x.tobytes() for x in p.matrix()] == [x.tobytes() for x in q.matrix()]


def test_builder_errors(capi):
    text = iw.multi_contig_vcf(CONTIGS, 300, 3, seed=25)
    lines = text.split(b"\n")
    head = [x for x in lines if x.startswith(b"#")]
    body = [x for x in lines if x and not x.startswith(b"#")]
    swapped = b"\n".join(head + body[:5] + [body[6], body[5]] + body[7:]) + b"\n"
    with pytest.raises(capi.HaploError) as e:
        capi.build_index(synth.bgzf_compress(swapped))
    assert e.value.code == 6 and "unsorted positions" in str(e.value)
    split = b"\n".join(head + body[:10] + body[400:410] + body[10:20]) + b"\n"
    with pytest.raises(capi.HaploError) as e:
        capi.build_index(synth.bgzf_compress(split), "csi")
    assert e.value.code == 6 and "not continuous" in str(e.value)
    for plain in (gzip.compress(text), text):
        with pytest.raises(capi.HaploError) as e:
            capi.build_index(plain)
        assert e.value.code == 10


def test_cli(capi, built):
    from click.testing import CliRunner
    sys.path.insert(0, os.path.join(ROOT, "haplohyped-varawareml_b200"))
    import vcf_index
    text = iw.multi_contig_vcf(CONTIGS, 500, 4, seed=26)
    raw = bcf_writer.vcf_to_bcf(text)
    with tempfile.TemporaryDirectory() as d:
        vcf, bcf = os.path.join(d, "x.vcf.gz"), os.path.join(d, "x.bcf")
        open(vcf, "wb").write(synth.bgzf_compress(text))
        open(bcf, "wb").write(synth.bgzf_compress(raw))
        r = CliRunner().invoke(vcf_index.main, [vcf])
        assert r.exit_code == 0, r.output
        assert gzip.decompress(open(vcf + ".tbi", "rb").read()) == iw.index_vcf(text, open(vcf, "rb").read(), "tbi")
        r = CliRunner().invoke(vcf_index.main, [vcf, "--csi"])
        assert r.exit_code == 0 and os.path.exists(vcf + ".csi")
        open(vcf + ".tbi", "wb").write(b"keep")
        r = CliRunner().invoke(vcf_index.main, [vcf])
        assert r.exit_code != 0 and "--force" in r.output
        assert open(vcf + ".tbi", "rb").read() == b"keep"
        r = CliRunner().invoke(vcf_index.main, [vcf, "--force"])
        assert r.exit_code == 0 and open(vcf + ".tbi", "rb").read() != b"keep"
        r = CliRunner().invoke(vcf_index.main, [bcf])
        assert r.exit_code == 0 and os.path.exists(bcf + ".csi")
