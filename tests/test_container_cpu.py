"""CPU tests of the minimal HDF5 writer/reader (minih5): the file structures behind the reference's
`donor_{id}/chr_{N}/snp_data` layout (vcf_to_h5.py:131-135).  Payloads are opaque here (no codec, no
GPU): what is checked is that groups, the chunk index and the dataset metadata survive a round trip,
including group fan-outs that need several symbol-table nodes and B-tree levels."""
import struct

import numpy as np
import pytest

REC = np.dtype([("chrom", "S5"), ("start", np.uint32), ("stop", np.uint32), ("ref", "S10"), ("alt", "S10"),
                ("phase1", np.int8), ("phase2", np.int8)])


@pytest.fixture(scope="module")
def minih5():
    from haplohyped_varawareml_b200 import minih5 as m
    return m


def test_record_dtype_layout():
    assert REC.itemsize == 35 and [REC.fields[n][1] for n in REC.names] == [0, 5, 9, 13, 23, 33, 34]


def test_superblock_and_signature(tmp_path, minih5):
    p = str(tmp_path / "a.h5")
    with minih5.H5Writer(p) as w:
        w.create_dataset_contiguous("x", np.arange(10, dtype=np.uint32))
    raw = open(p, "rb").read()
    assert raw[:8] == b"\x89HDF\r\n\x1a\n" and raw[8] == 0 and raw[13] == 8 and raw[14] == 8
    eof = struct.unpack_from("<Q", raw, 40)[0]
    assert eof == len(raw)


@pytest.mark.parametrize("n_donors,n_chroms", [(1, 1), (3, 22), (70, 2), (600, 1)])
def test_group_tree_roundtrip(tmp_path, minih5, n_donors, n_chroms):
    rng = np.random.default_rng(n_donors)
    p = str(tmp_path / "g.h5")
    payloads = {}
    with minih5.H5Writer(p) as w:
        for d in range(n_donors):
            for c in range(1, n_chroms + 1):
                n = int(rng.integers(0, 2000))
                chunk = 250
                k = (n + chunk - 1) // chunk
                chunks = [rng.integers(0, 256, int(rng.integers(1, 400)), dtype=np.uint8).tobytes() for _ in range(k)]
                path = f"donor_{d:04d}-x/chr_{c}/snp_data"
                w.create_dataset_chunked(path, REC, n, chunk, chunks, filter_id=32001,
                                         cd_values=(2, 2, 35, chunk * 35, 5, 1, 2), filter_name="blosc")
                payloads[path] = (n, chunks)
    r = minih5.H5Reader(p)
    assert r.keys("/") == sorted({q.split("/")[0] for q in payloads})
    assert "donor_0000-x/chr_1" in r and "donor_0000-x/chr_99" not in r and "nobody" not in r
    for path, (n, chunks) in payloads.items():
        info = r.dataset_info(path)
        assert info.dtype == REC and info.shape == (n,) and info.layout == "chunked" and info.chunk == 250
        assert info.filters == [(32001, (2, 2, 35, 250 * 35, 5, 1, 2))]
        got = r.chunks(info)
        assert [o for o, _ in got] == [k * 250 for k in range(len(chunks))]
        assert [b for _, b in got] == chunks
    r.close()


def test_many_chunks_need_btree_levels(tmp_path, minih5):
    p = str(tmp_path / "c.h5")
    chunks = [bytes([k & 255]) * (1 + k % 7) for k in range(5000)]           # > 64 and > 64*64 leaves
    with minih5.H5Writer(p) as w:
        w.create_dataset_chunked("d/c/snp_data", REC, 5000 * 10 - 3, 10, chunks)
    r = minih5.H5Reader(p)
    info = r.dataset_info("d/c/snp_data")
    got = r.chunks(info)
    assert [b for _, b in got] == chunks and not info.filters
    r.close()


def test_contiguous_and_unfiltered_read(tmp_path, minih5):
    from haplohyped_varawareml_b200 import container
    p = str(tmp_path / "r.h5")
    seq = np.frombuffer(b"ACGTN" * 1000, "S1")
    with container.open_h5(p, "w", backend="minih5") as f:
        f.write_array("chr1", seq)
        f.write_array("chr2", np.zeros(0, "S1"))
    f = container.open_h5(p, "r", backend="minih5")
    assert "chr1" in f and f.keys() == ["chr1", "chr2"]
    assert np.array_equal(f.read_dataset("chr1"), seq) and len(f.read_dataset("chr2")) == 0
    f.close()


def test_duplicate_and_bad_paths(tmp_path, minih5):
    with minih5.H5Writer(str(tmp_path / "d.h5")) as w:
        w.create_dataset_contiguous("a/b", np.zeros(3, np.uint8))
        with pytest.raises(ValueError):
            w.create_dataset_contiguous("a/b", np.zeros(3, np.uint8))
        with pytest.raises(ValueError):
            w.create_dataset_contiguous("a/b/c", np.zeros(3, np.uint8))
    with pytest.raises(OSError):
        (tmp_path / "junk.h5").write_bytes(b"not hdf5" * 20)
        minih5.H5Reader(str(tmp_path / "junk.h5"))


@pytest.mark.parametrize("n_chunks", [1, 5, 64, 65, 300, 5000])
def test_bulk_blob_writer_equals_per_chunk_writer(tmp_path, minih5, n_chunks):
    """write_blob + create_dataset_chunked_at (one write for all stored chunks, numpy-built chunk B-tree, gaps between
    chunks allowed) must describe the same dataset as the per-chunk writer."""
    rng = np.random.default_rng(n_chunks)
    dt = np.dtype([("a", "S5"), ("b", "<u4")])
    chunks = [rng.integers(0, 256, int(rng.integers(1, 50)), dtype=np.uint8).tobytes() for _ in range(n_chunks)]
    cd = (2, 2, 9, 90, 5, 1, 2)
    with minih5.H5Writer(str(tmp_path / "a.h5")) as w:
        w.create_dataset_chunked("g/x/snp", dt, n_chunks * 10, 10, chunks, filter_id=32001, cd_values=cd, filter_name="blosc")
    offs, blob = [], bytearray()
    for c in chunks:
        blob += b"\xee" * int(rng.integers(0, 16))
        offs.append(len(blob))
        blob += c
    with minih5.H5Writer(str(tmp_path / "b.h5")) as w:
        base = w.write_blob(bytes(blob))
        assert base % 16 == 0
        w.create_dataset_chunked_at("g/x/snp", dt, n_chunks * 10, 10, base + np.array(offs, np.uint64),
                                    np.array([len(c) for c in chunks], np.uint32), filter_id=32001, cd_values=cd, filter_name="blosc")
    ra, rb = minih5.H5Reader(str(tmp_path / "a.h5")), minih5.H5Reader(str(tmp_path / "b.h5"))
    ia, ib = ra.dataset_info("g/x/snp"), rb.dataset_info("g/x/snp")
    assert [c for _, c in ra.chunks(ia)] == chunks and rb.chunks(ib) == ra.chunks(ia)
    assert ia.filters == ib.filters and ia.chunk == ib.chunk and ia.shape == ib.shape and ia.dtype == ib.dtype
    ra.close(); rb.close()


def test_chunk_filter_mask_roundtrip(tmp_path, minih5):
    """Per-chunk filter masks survive the chunk B-tree (one level and several); a chunk with mask bit 0 (the optional
    Blosc filter skipped, as HDF5 stores a chunk the filter could not shrink) keeps the dataset out of stored_chunks."""
    from haplohyped_varawareml_b200 import container
    rng = np.random.default_rng(3)
    cd = (2, 2, 35, 350, 5, 1, 2)
    p = str(tmp_path / "m.h5")
    small = [rng.integers(0, 256, 350, dtype=np.uint8).tobytes()]
    many = [rng.integers(0, 256, int(rng.integers(1, 60)), dtype=np.uint8).tobytes() for _ in range(300)]
    masks = [int(m) for m in rng.choice([0, 1, 2, 0xFFFFFFFF], 300)]
    with minih5.H5Writer(p) as w:
        w.create_dataset_chunked("d/chr_1/snp_data", REC, 2, 10, small, filter_id=32001, cd_values=cd,
                                 filter_name="blosc", masks=[1])
        w.create_dataset_chunked("d/chr_2/snp_data", REC, 3000, 10, many, filter_id=32001, cd_values=cd,
                                 filter_name="blosc", masks=masks)
        w.create_dataset_chunked("d/chr_3/snp_data", REC, 3000, 10, many, filter_id=32001, cd_values=cd,
                                 filter_name="blosc")
    r = minih5.H5Reader(p)
    assert r.chunks_with_masks(r.dataset_info("d/chr_1/snp_data")) == [(0, small[0], 1)]
    info2 = r.dataset_info("d/chr_2/snp_data")
    assert r.chunks_with_masks(info2) == [(10 * k, c, m) for k, (c, m) in enumerate(zip(many, masks))]
    assert r.chunks(info2) == [(10 * k, c) for k, c in enumerate(many)]
    assert [m for _, _, m in r.chunks_with_masks(r.dataset_info("d/chr_3/snp_data"))] == [0] * 300
    r.close()
    f = container.open_h5(p, "r", backend="minih5")
    assert f.stored_chunks("d/chr_1/snp_data") is None and f.stored_chunks("d/chr_2/snp_data") is None
    n, cr, dt, chunks = f.stored_chunks("d/chr_3/snp_data")
    assert (n, cr, dt, chunks) == (3000, 10, REC, many)
    # every chunk unfiltered: read without any codec, the records as stored (the tail past n dropped)
    rec = np.frombuffer(small[0], REC)
    assert f.read_dataset("d/chr_1/snp_data").tobytes() == rec[:2].tobytes()
    f.close()
