"""HDF5 chunks of 2,731 - 7,489 records: kernels 4a-L / 4b-L (site templates and allele tails of large chunks) and
kernel 6-L (device-side decode of chunks larger than a warp's shared memory).

Up to 7,489 records a chunk of 35-byte records is still ONE Blosc block with ONE LZ4 stream (c-blosc 1.x cuts blocks of
262,115 bytes at typesize 35, clevel 5, LZ4HC: oracle.cblosc1_blocksize), and h5py's unclamped auto-chunk reaches that
range for chromosomes above 2.8 M records.  Every stored chunk is decoded by the oracle's independent Blosc path and by
stock liblz4 and compared with the zero-padded 35-byte records the reference would have stored."""
import ctypes as C
import random
import string
import struct

import numpy as np
import pytest

import oracle
import synth

pytestmark = pytest.mark.gpu

LARGE = (2731, 3028, 3125, 4096, 4883, 6001, 7489)
SENT32, SENT8 = 0x5A5A5A5A, 0x5A
COLS = ("start", "stop", "ref", "alt", "p1", "p2")


@pytest.fixture(scope="module")
def capi(built):
    from haplohyped_varawareml_b200 import capi as c
    return c


def _expected_chunks(ora, s, cr):
    rec = oracle.records_from_columns(ora["chrom"], ora["start"], ora["stop"], ora["ref"], ora["alt"], ora["gt0"][s], ora["gt1"][s])
    n_chunks = (ora["n"] + cr - 1) // cr
    raw = rec.tobytes() + b"\0" * (n_chunks * cr * 35 - rec.nbytes)          # HDF5 edge chunks are zero-filled
    return [raw[k * cr * 35:(k + 1) * cr * 35] for k in range(n_chunks)]


def _check_frames(frames, exp):
    """each stored chunk: oracle decode, the header fields of a one-block Blosc1 chunk, stock liblz4 on the payload"""
    L = oracle.stock_lz4()
    assert len(frames) == len(exp)
    for f, e in zip(frames, exp):
        assert oracle.blosc_chunk_decode(f, len(e)).tobytes() == e, "decompressed chunk differs"
        assert f[:4] == bytes([2, 1, 0x31, 35])
        assert struct.unpack("<IIII", f[4:20]) == (len(e), len(e), len(f), 20)
        csize = struct.unpack("<i", f[20:24])[0]
        assert csize == len(f) - 24
        payload = f[24:]
        if csize == len(e):
            assert payload == oracle.shuffle(e, 35).tobytes()
            continue
        out = C.create_string_buffer(len(e))
        assert L.LZ4_decompress_safe(payload, out, len(payload), len(e)) == len(e), "stock liblz4 rejected the block"
        assert out.raw == oracle.shuffle(e, 35).tobytes()


def _roundtrip(capi, text, n_samples, region, cr, samples):
    ora = oracle.parse_text(text, "*", region)
    p = capi.Parse.from_host(synth.body_of(text), n_samples, region=region)
    fr = p.compress(cr)
    assert int(fr.info.chunk_records) == cr and fr.info.n_chunks == (ora["n"] + cr - 1) // cr
    for s in samples:
        _check_frames(fr.sample(s), _expected_chunks(ora, s, cr))
    info = fr.info
    fr.close()
    p.close()
    return ora, info


@pytest.mark.parametrize("cr", LARGE)
def test_large_chunks_roundtrip(capi, cr):
    """synthetic cohorts (biallelic SNPs; multiallelic / indel / missing) with a last partial chunk and with fewer
    records than one chunk, and the mixed-site random VCF without a region filter (several contigs)"""
    S = 6
    sp = capi.synth_spec(2 * cr + 123, S, seed=cr, mix=0)
    ora, info = _roundtrip(capi, capi.synth_header(sp) + capi.synth_host(sp), S, "chr22", cr, [0, 3, 5])
    assert ora["n"] % cr and ora["n"] > 2 * cr and info.total_bytes < info.raw_bytes
    sp = capi.synth_spec(cr - 77, S, seed=cr + 1, mix=1)
    ora, _ = _roundtrip(capi, capi.synth_header(sp) + capi.synth_host(sp), S, "chr22", cr, [0, 5])
    assert 0 < ora["n"] < cr
    text, samples = synth.random_vcf(cr + cr // 2, 5, seed=cr, fmt="GT", kinds="mixed")
    ora, _ = _roundtrip(capi, text, len(samples), "", cr, [0, 2, 4])
    assert len(set(ora["chrom"])) > 1 and ora["n"] > cr


def _adversarial_vcf(n, n_samples, seed):
    """random start gaps (up to 200,000), random REF letters and ALT bases (every record a SNP: all are kept), runs of 1-15
    records on 300 random contig names (at most 4,096 CHROM runs per file): every site plane that can be is high-entropy,
    so the chunk templates are large"""
    rng = random.Random(seed)
    samples = synth.sample_names(n_samples)
    contigs = ["".join(rng.choice("abcdefghijklmnopqrstuvwxyz0123456789_") for _ in range(rng.randint(1, 12))) for _ in range(300)]
    out = [synth.header(samples)]
    pos, run, contig = 1, 0, None
    for i in range(n):
        if run == 0:
            run, contig = rng.randint(1, 15), rng.choice(contigs)
        run -= 1
        pos += rng.randint(1, 200_000)
        ref = rng.choice(string.ascii_letters)
        alt = rng.choice("ACGT")
        gts = ["%d|%d" % (rng.random() < 0.3, rng.random() < 0.3) for _ in range(n_samples)]
        out.append("\t".join([contig, str(pos), ".", ref, alt, ".", "PASS", ".", "GT"] + gts) + "\n")
    return "".join(out).encode(), samples


def test_adversarial_sites_at_the_largest_chunk(capi):
    cr = 7489
    text, samples = _adversarial_vcf(2 * cr + 1000, 4, seed=3)
    try:
        for deep in (0, 1):
            capi.lib().hb_set_site_matcher(deep)
            ora, info = _roundtrip(capi, text, len(samples), "", cr, [0, 1, 2, 3])
            assert ora["n"] == 2 * cr + 1000
            assert info.site_lz4_bytes > 3 * 5 * cr                   # large templates: several random planes per chunk
    finally:
        capi.lib().hb_set_site_matcher(0)


@pytest.mark.parametrize("cr", [4883, 7489])
def test_layout_fetch_and_windows_at_large_chunks(capi, cr):
    """layout / fetch_all / fetch_packed (both ways, 1 and 3 host threads, pinned / pageable / unaligned destinations) /
    sample agree; rerun is deterministic; a sample window equals the same samples of the all-sample pass"""
    import torch
    S = 40
    sp = capi.synth_spec(3 * cr + 500, S, seed=cr + 7, mix=1)
    text = capi.synth_header(sp) + capi.synth_host(sp)
    p = capi.Parse.from_host(synth.body_of(text), S, region="chr22")
    fr = p.compress(cr)
    nc = int(fr.info.n_chunks)
    offs, sizes = fr.layout()
    buf = fr.fetch_all()
    assert offs.shape == (S, nc) and (offs % 16 == 0).all()
    assert (np.diff(offs.reshape(-1).astype(np.int64)) >= sizes.reshape(-1)[:-1]).all()
    assert int(sizes.sum()) == fr.info.total_bytes and len(buf) == fr.info.padded_bytes
    per_sample = {s: fr.sample(s) for s in (0, 17, S - 1)}
    for s, frames in per_sample.items():
        for k, f in enumerate(frames):
            assert buf[int(offs[s, k]):int(offs[s, k]) + int(sizes[s, k])].tobytes() == f
    pk, poffs, psizes = fr.fetch_packed()
    assert np.array_equal(psizes, sizes) and (poffs % 16 == 0).all()
    for s, frames in per_sample.items():
        for k, f in enumerate(frames):
            assert pk[int(poffs[s, k]):int(poffs[s, k]) + int(psizes[s, k])].tobytes() == f
    pin = torch.empty(len(pk) + 64, dtype=torch.uint8).pin_memory()
    try:
        for mode, threads in ((1, 0), (2, 1), (2, 3)):
            capi.lib().hb_set_fetch_mode(mode)
            capi.lib().hb_set_host_threads(threads)
            pin.fill_(0xEE)
            tot, o2, z2 = fr.fetch_packed(out=(pin.data_ptr(), pin.numel()))
            assert tot == len(pk) and np.array_equal(pin.numpy()[:tot], pk) and (pin.numpy()[tot:] == 0xEE).all()
            assert np.array_equal(o2, poffs) and np.array_equal(z2, psizes)
            got, _, _ = fr.fetch_packed()                                       # pageable
            assert np.array_equal(got, pk)
            odd = np.empty(len(pk) + 64, np.uint8)
            shift = (1 - odd.ctypes.data) % 16 or 16
            tot3, _, _ = fr.fetch_packed(out=(odd.ctypes.data + shift, len(pk)))
            assert tot3 == len(pk) and np.array_equal(odd[shift:shift + tot3], pk)
    finally:
        capi.lib().hb_set_fetch_mode(0)
        capi.lib().hb_set_host_threads(0)
    fr.rerun(p)
    assert np.array_equal(fr.fetch_all(), buf)
    # a window of 16 samples, moved to [11, 27) and re-run
    win = p.compress(cr, 0, 16)
    win.set_window(11, 16)
    win.rerun(p)
    for k in range(16):
        assert win.sample(k) == fr.sample(11 + k)
    win.close()
    fr.close()
    p.close()


def test_streamed_resident_parse_at_large_chunks(capi):
    """a .vcf.gz parsed through the streamed-resident route (hb_parse_set_text_limit forces it) gives byte-identical
    frames at cr 4,883 to the whole-file parse"""
    cr = 4883
    text, samples = synth.random_vcf(3 * cr + 700, 12, seed=41, fmt="GT", kinds="mixed")
    bg = capi.bgzf_compress_host(text, 6)
    whole = capi.Parse.from_vcf_bytes(bg, region="chr22")
    try:
        capi.lib().hb_parse_set_text_limit(64 << 10)
        streamed = capi.Parse.from_vcf_bytes(bg, region="chr22")
    finally:
        capi.lib().hb_parse_set_text_limit(0)
    assert streamed.info.text_bytes == 0 and streamed.info.n_records == whole.info.n_records > 2 * cr
    fw, fs = whole.compress(cr), streamed.compress(cr)
    assert fw.info.n_chunks == fs.info.n_chunks
    bw, ow, zw = fw.fetch_packed()
    bs, os_, zs = fs.fetch_packed()
    assert np.array_equal(zw, zs) and np.array_equal(ow, os_) and np.array_equal(bw, bs)
    ora = oracle.parse_text(text, "*", "chr22")
    _check_frames(fs.sample(7), _expected_chunks(ora, 7, cr))
    for h in (fw, fs, whole, streamed):
        h.close()


# ---------------------------------------------------------------------------------------------------------------------
# kernel 6-L through hb_decode_columns_device_large

def make_records(n, seed):
    rng = np.random.default_rng(seed)
    rec = np.zeros(n, oracle.RECORD_DTYPE)
    rec["chrom"] = b"chr22"
    start = np.sort(rng.integers(0, 2 ** 32, n, dtype=np.uint64)).astype(np.uint32)
    rec["start"] = start
    rec["stop"] = start + np.uint32(1)
    rec["ref"] = rng.choice(np.array([b"A", b"C", b"G", b"T", b"N", b"ACGT"]), n)
    rec["alt"] = rng.choice(np.array([b"A", b"C", b"G", b"T", b"<DEL>"]), n)
    rec["phase1"] = rng.choice(np.array([0, 1, -9, 127, -128], np.int8), n, p=[0.6, 0.3, 0.05, 0.03, 0.02])
    rec["phase2"] = rng.choice(np.array([0, 1, -9], np.int8), n, p=[0.6, 0.35, 0.05])
    return rec


def columns_of(raw):
    b = np.frombuffer(raw, np.uint8).reshape(-1, 35)
    return {"start": b[:, 5:9].copy().view("<u4")[:, 0], "stop": b[:, 9:13].copy().view("<u4")[:, 0], "ref": b[:, 13].copy(),
            "alt": b[:, 23].copy(), "p1": b[:, 33].view(np.int8).copy(), "p2": b[:, 34].view(np.int8).copy()}


def memcpyed_chunk(data):
    return bytes([2, 1, 0x02 | (1 << 5), 35]) + struct.pack("<III", len(data), len(data), 16 + len(data)) + data


def decode_columns(capi, chunks, cr, rows, rows_total, want=COLS, absolute=False, seed=0, entry="hb_decode_columns_device_large"):
    import torch
    rng = np.random.default_rng(seed)
    offs, blob = [], bytearray()
    for c in chunks:
        blob += bytes(rng.integers(0, 256, int(rng.integers(1, 16)), dtype=np.uint8))
        if len(blob) % 16 == 0:
            blob += b"\x00"                                                    # never 16-byte aligned
        offs.append(len(blob))
        blob += c
    blob += bytes(64)
    dev = torch.device("cuda:0")
    d_blob = torch.from_numpy(np.frombuffer(bytes(blob), np.uint8).copy()).to(dev)
    base = d_blob.data_ptr()
    offs = np.array(offs, np.uint64) + (np.uint64(base) if absolute else np.uint64(0))
    d_off = torch.from_numpy(offs.view(np.int64)).to(dev)
    d_len = torch.from_numpy(np.array([len(c) for c in chunks], np.int32)).to(dev)
    d_row = torch.from_numpy(np.asarray(rows, np.int64)).to(dev)
    status = torch.full((len(chunks),), -1, dtype=torch.int32, device=dev)
    types = {"start": torch.int32, "stop": torch.int32, "ref": torch.uint8, "alt": torch.uint8, "p1": torch.int8, "p2": torch.int8}
    out = {k: torch.full((rows_total,), SENT32 if k in ("start", "stop") else SENT8, dtype=t, device=dev) for k, t in types.items()}
    ptr = lambda k: out[k].data_ptr() if k in want else None
    capi.check(getattr(capi.lib(), entry)(None if absolute else base, d_off.data_ptr(), d_len.data_ptr(), d_row.data_ptr(),
                                                   len(chunks), cr, *[ptr(k) for k in COLS], status.data_ptr(), None))
    torch.cuda.synchronize()
    got = {k: v.cpu().numpy() for k, v in out.items()}
    got["start"] = got["start"].view(np.uint32)
    got["stop"] = got["stop"].view(np.uint32)
    return got, status.cpu().numpy()


def check_columns(got, status, expect, cr, rows, rows_total, want=COLS):
    """expect[i] = columns of chunk i, or None for a chunk that must fail; rows no good chunk wrote keep the sentinels"""
    written = np.zeros(rows_total, bool)
    for i, exp in enumerate(expect):
        r0 = int(rows[i])
        if exp is None:
            assert status[i] != 0, i
            continue
        assert status[i] == 0, (i, status[i])
        written[r0:r0 + cr] = True
        for k in want:
            assert np.array_equal(got[k][r0:r0 + cr], exp[k]), (i, k)
    for k in COLS:
        sent = SENT32 if k in ("start", "stop") else SENT8
        mask = ~written if k in want else np.ones(rows_total, bool)
        assert np.all(got[k][mask].astype(np.int64) & 0xFFFFFFFF == sent), k


def permuted_rows(n_chunks, cr, seed):
    slots = np.random.default_rng(seed).permutation(n_chunks + 3)[:n_chunks]
    return (slots * cr).astype(np.int64), (n_chunks + 3) * cr


def _optin_smem():
    import torch
    return int(torch.cuda.get_device_properties(0).shared_memory_per_block_optin)


def _kernel6_sizes():
    """above 2,730 records: the largest chunk kernel 6 holds in a warp's shared memory, the first one above it (kernel
    6-L) and more kernel 6-L sizes up to the limit"""
    last_6 = (_optin_smem() - 1024) // 35
    return sorted({2731, 6001, last_6, last_6 + 1, 7000, 7489})


def test_kernel6_large_chunks_from_every_producer(capi):
    for cr in _kernel6_sizes():
        n_chunks = 4
        n = n_chunks * cr - cr // 3
        rec = make_records(n, cr)
        raw = rec.tobytes() + bytes(n_chunks * cr * 35 - rec.nbytes)
        chunks, expect = [], []
        for i in range(n_chunks):
            data = raw[i * cr * 35:(i + 1) * cr * 35]
            ch = (oracle.reference_like_chunk, memcpyed_chunk, lambda d: oracle.blosc1_chunk_encode(d, 35))[i % 3](data)
            assert oracle.blosc_chunk_decode(ch, cr * 35).tobytes() == data
            chunks.append(ch)
            expect.append(columns_of(data))
        rows, total = permuted_rows(n_chunks, cr, cr)
        for absolute in (False, True):
            got, status = decode_columns(capi, chunks, cr, rows, total, absolute=absolute, seed=cr)
            check_columns(got, status, expect, cr, rows, total)
        want = ("stop", "alt", "p2")                                           # NULL columns stay untouched
        got, status = decode_columns(capi, chunks, cr, rows, total, want=want, seed=cr + 1)
        check_columns(got, status, expect, cr, rows, total, want=want)
        assert capi.decode_frames(chunks, cr * 35).tobytes() == raw            # the host-pointer decoder agrees


def test_kernel6_large_chunks_from_gpu_frames(capi):
    for cr in _kernel6_sizes():
        text, samples = synth.random_vcf(2 * cr + 211, 3, seed=cr, fmt="GT", kinds="mixed")
        ora = oracle.parse_text(text, "*", "")
        p = capi.Parse.from_host(synth.body_of(text), len(samples), region="")
        fr = p.compress(cr)
        for s in (0, 2):
            frames = fr.sample(s)
            exp = _expected_chunks(ora, s, cr)
            expect = [columns_of(e) for e in exp]
            rows, total = permuted_rows(len(frames), cr, s)
            got, status = decode_columns(capi, frames, cr, rows, total, absolute=bool(s))
            check_columns(got, status, expect, cr, rows, total)
            assert capi.decode_frames(frames, cr * 35).tobytes() == b"".join(exp)
        fr.close()
        p.close()


def test_kernel6_large_hostile_chunks_between_good_ones(capi):
    """each damaged chunk between good ones in ONE launch at cr 7,489: a chunk the oracle refuses gets a non-zero status
    and writes no row; a damage that still decodes (LZ4 payload bytes) gives exactly what the oracle decodes"""
    cr = 7489
    data = make_records(cr, 5).tobytes()
    good = oracle.reference_like_chunk(data)
    lz4_len = struct.unpack("<i", good[20:24])[0]
    assert lz4_len < cr * 35                                                # an LZ4 stream, not stored raw

    def mutated(at, value):
        b = bytearray(good)
        b[at:at + len(value)] = value
        return bytes(b)

    rng = np.random.default_rng(9)
    bad = [mutated(0, b"\x09"), mutated(2, bytes([good[2] | 0x08])), mutated(4, struct.pack("<I", cr * 35 + 35)),
           mutated(12, struct.pack("<I", len(good) + 1000)), mutated(16, struct.pack("<I", 0xfffffff0)),
           mutated(20, struct.pack("<i", -5)), mutated(20, struct.pack("<I", len(good))), good[:len(good) // 2],
           good[:len(good) - 1], mutated(len(good) - 40, b"\x00" * 8), mutated(24, b"\xff" * 8)]
    bad += [mutated(int(rng.integers(24, len(good) - 1)), bytes([int(rng.integers(0, 256))])) for _ in range(12)]
    several = oracle.blosc1_chunk_encode(data, 35, blocksize=35 * (cr // 3))
    assert oracle.blosc_chunk_decode(several, cr * 35).tobytes() == data   # well-formed, but several blocks: status 11
    bad.append(several)
    chunks, expect = [], []
    exp_good = columns_of(data)
    for h in bad:
        try:
            dec = None if h is several else oracle.blosc_chunk_decode(h, cr * 35).tobytes()
        except ValueError:
            dec = None
        chunks += [good, h]
        expect += [exp_good, None if dec is None else columns_of(dec)]
    chunks.append(good)
    expect.append(exp_good)
    assert sum(e is None for e in expect) >= 12
    rows, total = permuted_rows(len(chunks), cr, 4)
    got, status = decode_columns(capi, chunks, cr, rows, total)
    check_columns(got, status, expect, cr, rows, total)
    assert status[2 * (len(bad) - 1) + 1] == 11


def test_largest_chunk_the_kernels_accept(capi):
    """7,489 records (one c-blosc 1.x block) is the limit of the writer and of hb_decode_columns_device_large;
    hb_decode_columns_device keeps its limit (a chunk must fit a warp's shared memory)"""
    cr = 7489
    assert oracle.cblosc1_blocksize(35 * cr, 35) == 35 * cr == oracle.cblosc1_blocksize(35 * (cr + 1), 35)
    chunks = [oracle.reference_like_chunk(make_records(cr, 1).tobytes())]
    got, status = decode_columns(capi, chunks, cr, [0], cr)
    assert status[0] == 0
    with pytest.raises(capi.HaploError):
        decode_columns(capi, chunks, cr + 1, [0], cr + 1)
    last_6 = (_optin_smem() - 1024) // 35
    small = [oracle.reference_like_chunk(make_records(last_6, 2).tobytes())]
    for entry in ("hb_decode_columns_device", "hb_decode_columns_device_large"):
        got, status = decode_columns(capi, small, last_6, [0], last_6, entry=entry)
        assert status[0] == 0 and np.array_equal(got["p1"], columns_of(make_records(last_6, 2).tobytes())["p1"])
    for n in (last_6 + 1, cr):
        with pytest.raises(capi.HaploError):
            decode_columns(capi, chunks, n, [0], n, entry="hb_decode_columns_device")
    sp = capi.synth_spec(cr + 10, 3, seed=2)
    p = capi.Parse.from_host(synth.body_of(capi.synth_header(sp) + capi.synth_host(sp)), 3, region="chr22")
    with pytest.raises(capi.HaploError, match="7,489"):
        p.compress(cr + 1)
    p.close()


def test_guess_chunk_records_at_the_band_edges(capi):
    """h5py's auto-chunk is not clamped: above 2,730 records in the bands below; the C restatement equals the oracle's"""
    edges = [2_795_521, 2_825_217, 5_591_041, 7_616_513, 11_182_081, 20_533_249, 22_364_161, 122_699_777]
    for e in edges:
        for n in (e - 1, e, e + 1):
            assert int(capi.lib().hb_guess_chunk_records(n)) == oracle.guess_chunk_1d(n), n
    assert oracle.guess_chunk_1d(2_795_520) == 2730 and int(capi.lib().hb_guess_chunk_records(2_795_521)) == 2731
    assert int(capi.lib().hb_guess_chunk_records(122_699_776)) == 7489


def test_converter_end_to_end_above_2_8_million_records(capi, tmp_path):
    """a chromosome of 2,795,521 kept records (auto-chunk 2,731): the converter writes it, VCFH5Reader reads it back,
    and the dataset keeps it compressed in HBM and decodes windows of it on the device"""
    import torch
    from haplohyped_varawareml_b200 import h5_reader, haplotype_dataset, vcf_to_h5
    n = 2_795_521
    sp = capi.synth_spec(n, 2, seed=8, mix=0)
    text = capi.synth_header(sp) + capi.synth_host(sp)
    ora = oracle.parse_text(text, "*", "chr22")
    assert ora["n"] == n
    vdir = tmp_path / "vcf"
    vdir.mkdir()
    (vdir / "chr22.filtered.vcf.gz").write_bytes(capi.bgzf_compress_host(text, 1).tobytes())
    del text
    samples = capi.synth_sample_names(sp)
    (tmp_path / "donors.txt").write_text("\n".join(samples))
    conv = vcf_to_h5.VCFtoHDF5Converter("c", str(vdir), str(tmp_path / "out"), str(tmp_path / "donors.txt"), 2, 4, chromosomes=[22])
    conv.run()
    assert conv.stats["datasets"] == 2
    path = str(tmp_path / "out" / "c.h5")
    rd = h5_reader.VCFH5Reader(path)
    recs = {}
    for s, name in enumerate(samples):
        rec = oracle.records_from_columns(ora["chrom"], ora["start"], ora["stop"], ora["ref"], ora["alt"], ora["gt0"][s], ora["gt1"][s])
        assert rd.fetch_genotypes(name, 22).tobytes() == rec.tobytes()
        got = rd.stored_chunks(name, 22)
        assert got[0] == n and got[1] == 2731
        recs[name] = rec
    st = haplotype_dataset.GenotypeStore.from_reader(rd)
    start = ora["start"]
    rng = np.random.default_rng(1)
    picks = [int(i) for i in rng.integers(0, n, 6)] + [0, 2731 - 1, 2731, n - 1]
    items = [(samples[k % 2], 22, int(start[i]) - 50, int(start[i]) + 5000) for k, i in enumerate(picks)]
    cols, keep = st.window_columns(items)
    torch.cuda.synchronize()
    st.check_last()
    assert all(st._stored[(name, 22)] is not None for name in samples) and not st._cols     # no whole-dataset fallback
    assert len(keep) == 1                                                     # one chunk geometry: one launch
    dec = [t.cpu().numpy() for t in keep[0][:5]]                              # start, ref, alt, p1, p2 of the batch
    base = [t.data_ptr() for t in keep[0][:5]]
    whole = {}
    for name in samples:                                                      # the dataset decoded whole (`columns`)
        c = st.columns(name, 22)
        whole[name] = [t.cpu().numpy() for t in st._cols[(name, 22)][:5]]
        assert c[5] == n
    for (donor, _, ws, we), c in zip(items, cols):
        m = c[5]
        assert 0 < m < n
        o = (c[0] - base[0]) // 4
        assert all(c[k] - base[k] == o for k in range(1, 5))
        got = [d[o:o + m] for d in dec]
        ref = whole[donor]
        r0 = int(np.searchsorted(ref[0].view(np.uint32), got[0].view(np.uint32)[0], "left"))
        assert r0 % 2731 == 0                                                 # the span starts on a chunk
        for k in range(5):
            assert np.array_equal(got[k], ref[k][r0:r0 + m]), k
        inside = np.nonzero((start >= ws) & (start < we))[0]                  # every record of the window is covered
        assert inside.size == 0 or (inside[0] >= r0 and inside[-1] < r0 + m)
    del keep
    st.close()
