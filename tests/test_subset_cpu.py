"""Sample subsets without a GPU: the header's sample names come from the leading bytes of every file form the project reads,
and the subset entry points fail with HB_ERR_CUDA when there is no device (no CPU fallback)."""
import gzip

import numpy as np
import pytest

import bcf_writer
import synth


@pytest.fixture(scope="module")
def capi(built):
    from haplohyped_varawareml_b200 import capi as c
    return c


def _no_device():
    try:
        import torch
        return not torch.cuda.is_available()
    except ImportError:
        return True


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    d = tmp_path_factory.mktemp("subset")
    text, samples = synth.random_vcf(300, 45, seed=3, fmt="GT:GQ:DP", kinds="mixed")
    paths = {}
    for name, data in (("x.vcf", text), ("x.vcf.gz", synth.bgzf_compress(text, block=997)), ("x.gzip.vcf.gz", gzip.compress(text)),
                       ("x.bcf", synth.bgzf_compress(bcf_writer.vcf_to_bcf(text))), ("x.plain.bcf", bcf_writer.vcf_to_bcf(text))):
        (d / name).write_bytes(data)
        paths[name] = str(d / name)
    return paths, samples


@pytest.mark.parametrize("name", ["x.vcf", "x.vcf.gz", "x.gzip.vcf.gz", "x.bcf", "x.plain.bcf"])
def test_file_sample_names(capi, files, name):
    paths, samples = files
    assert capi.file_sample_names(paths[name]) == samples


def test_file_sample_names_of_a_wide_header(capi, tmp_path):
    """A header longer than the first read rounds (and than one BGZF member)."""
    samples = ["sample_with_a_long_name_%06d" % i for i in range(20000)]
    text = synth.header(samples).encode() + b"chr22\t100\t.\tA\tC\t.\tPASS\t.\tGT\t" + b"\t".join([b"0|1"] * 20000) + b"\n"
    for name, data in (("w.vcf", text), ("w.vcf.gz", synth.bgzf_compress(text)), ("w.gz", gzip.compress(text))):
        (tmp_path / name).write_bytes(data)
        assert capi.file_sample_names(str(tmp_path / name)) == samples


def test_file_sample_names_errors(capi, tmp_path):
    (tmp_path / "nohdr.vcf").write_bytes(b"chr22\t100\t.\tA\tC\t.\tPASS\t.\tGT\t0|1\n")
    with pytest.raises(capi.HaploError) as e:
        capi.file_sample_names(str(tmp_path / "nohdr.vcf"))
    assert e.value.code == capi.HB_ERR_HEADER
    with pytest.raises(capi.HaploError) as e:
        capi.file_sample_names(str(tmp_path / "missing.vcf"))
    assert e.value.code == capi.HB_ERR_IO


@pytest.mark.skipif(not _no_device(), reason="checks the no-device path")
def test_subset_entry_points_need_a_device(capi, files):
    paths, samples = files
    text = open(paths["x.vcf"], "rb").read()
    body = synth.body_of(text)
    with pytest.raises(capi.HaploError) as e:
        capi.Parse.from_host(body, len(samples), samples=[0, 3])
    assert e.value.code == capi.HB_ERR_CUDA
    with pytest.raises(capi.HaploError) as e:
        capi.Parse.from_device(0, 0, len(samples), samples=[0, 3])
    assert e.value.code == capi.HB_ERR_CUDA
    for name in ("x.vcf", "x.vcf.gz", "x.bcf"):
        with pytest.raises(capi.HaploError) as e:
            capi.Parse.from_file(paths[name], samples=[samples[4], samples[1]])
        assert e.value.code == capi.HB_ERR_CUDA
        with pytest.raises(capi.HaploError) as e:
            capi.Parse.from_vcf_bytes(np.fromfile(paths[name], np.uint8), samples=[samples[4]])
        assert e.value.code == capi.HB_ERR_CUDA
