"""Kernel 6 (decode_columns_kernel, hb_decode_columns_device) and the read path around it, on stored chunks that other
writers produce: stock LZ4HC as the reference's writer stores it (c-blosc 1.x through hdf5-blosc), the oracle's greedy
Blosc1 writer, raw streams, memcpyed chunks, c-blosc2 extended headers, and this project's own GPU frames.  Every column
is compared with the numpy record array the chunk was made from; the oracle's Blosc decoder is the definition of the
format (oracle/vcf_oracle.c, orc_blosc_chunk_decode)."""
import ctypes as C
import struct

import numpy as np
import pytest

import oracle
import synth

pytestmark = pytest.mark.gpu

PHASES = np.array([-9, -56, -128, 0, 1, 127], np.int8)
SENT32, SENT8 = 0x5A5A5A5A, 0x5A
COLS = ("start", "stop", "ref", "alt", "p1", "p2")


@pytest.fixture(scope="module")
def mods(built):
    import torch
    from haplohyped_varawareml_b200 import capi, container, h5_reader, haplotype_dataset
    return capi, torch, container, h5_reader, haplotype_dataset


def make_records(n, seed):
    """start / stop with four different bytes (0 and 0xFFFFFFFF included), every phase value, random alleles"""
    rng = np.random.default_rng(seed)
    rec = np.zeros(n, oracle.RECORD_DTYPE)
    rec["chrom"] = b"chr22"
    start = rng.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32)
    k = min(n, 4)
    start[:k] = np.array([0, 0xFFFFFFFF, 0x01020304, 0xFFFEFDFC], np.uint32)[:k]
    rec["start"] = start
    rec["stop"] = start ^ np.uint32(0x80C0E0F0)
    rec["ref"] = rng.choice(np.array([b"A", b"C", b"G", b"T", b"N", b"ACGT"]), n)
    rec["alt"] = rng.choice(np.array([b"A", b"C", b"G", b"T", b"<DEL>"]), n)
    rec["phase1"] = PHASES[np.arange(n) % 6]
    rec["phase2"] = PHASES[(np.arange(n) * 5 + 1) % 6]
    return rec


def columns_of(rec):
    b = np.frombuffer(rec.tobytes(), np.uint8).reshape(-1, 35)
    return {"start": b[:, 5:9].copy().view("<u4")[:, 0], "stop": b[:, 9:13].copy().view("<u4")[:, 0], "ref": b[:, 13].copy(),
            "alt": b[:, 23].copy(), "p1": b[:, 33].view(np.int8).copy(), "p2": b[:, 34].view(np.int8).copy()}


# ---------------------------------------------------------------------------------------------------------------------
# chunk producers: records of one chunk (35 * cr bytes) -> stored chunk bytes

def _blosc_header(flags, nbytes, cbytes, version=2, versionlz=1):
    return bytes([version, versionlz, flags, 35]) + struct.pack("<III", nbytes, nbytes, cbytes)


def memcpyed_chunk(data):
    """flag 0x02: the bytes follow the header as they are (not shuffled)"""
    return _blosc_header(0x02 | (1 << 5), len(data), 16 + len(data)) + data


def blosc2_chunk(data, zero_run=False, split=False):
    """c-blosc2 extended 32-byte header (both shuffle bits), byte-shuffle as the only filter, one block of one stream
    (don't-split flag 0x10), LZ4 stream of the shuffled bytes or a zero run (csize 0).  split=True leaves out 0x10: the
    block then holds 35 streams, one per byte plane: plane 0 (must be zero) as a zero run, the others stored raw."""
    nbytes = len(data)
    if split:
        sh = oracle.shuffle(data, 35).tobytes()
        ne = nbytes // 35
        assert not any(sh[:ne])
        stream = struct.pack("<i", 0) + b"".join(struct.pack("<i", ne) + sh[j * ne:(j + 1) * ne] for j in range(1, 35))
    elif zero_run:
        assert not any(data)
        stream = struct.pack("<i", 0)
    else:
        sh = oracle.shuffle(data, 35).tobytes()
        L = oracle.stock_lz4()
        out = C.create_string_buffer(len(sh) + 64)
        cs = L.LZ4_compress_HC(sh, out, len(sh), len(sh) - 1, 5)
        stream = struct.pack("<i", cs) + out.raw[:cs] if cs > 0 else struct.pack("<i", len(sh)) + sh   # raw if LZ4 does not gain
    flags = 0x01 | 0x04 | (0 if split else 0x10) | (1 << 5)
    ext = bytes([0, 0, 0, 0, 0, 1, 0, 0]) + bytes(7) + bytes([0])          # filters [16,22): byte-shuffle last
    cbytes = 32 + 4 + len(stream)
    return bytes([5, 1, flags, 35]) + struct.pack("<III", nbytes, nbytes, cbytes) + ext + struct.pack("<I", 36) + stream


PRODUCERS = {
    "lz4hc": lambda d: oracle.reference_like_chunk(d),
    "greedy": lambda d: oracle.blosc1_chunk_encode(d, 35),
    "memcpyed": memcpyed_chunk,
    "blosc2_lz4": blosc2_chunk,
}


# ---------------------------------------------------------------------------------------------------------------------
# one call of hb_decode_columns_device

class Launch:
    def __init__(self, mods, chunks, cr, rows_total, rows, absolute=False, want=COLS, seed=0):
        capi, torch = mods[0], mods[1]
        rng = np.random.default_rng(seed)
        offs, blob = [], bytearray()
        for c in chunks:
            blob += bytes(rng.integers(0, 256, int(rng.integers(1, 16)), dtype=np.uint8))   # never 16-byte aligned
            if len(blob) % 16 == 0:
                blob += b"\x00"
            offs.append(len(blob))
            blob += c
        blob += bytes(64)
        dev = torch.device("cuda:0")
        self.blob = torch.from_numpy(np.frombuffer(bytes(blob), np.uint8).copy()).to(dev)
        base = self.blob.data_ptr()
        offs = np.array(offs, np.uint64) + (np.uint64(base) if absolute else np.uint64(0))
        self.off = torch.from_numpy(offs.view(np.int64)).to(dev)
        self.len = torch.from_numpy(np.array([len(c) for c in chunks], np.int32)).to(dev)
        self.row = torch.from_numpy(np.asarray(rows, np.int64)).to(dev)
        self.status = torch.full((len(chunks),), -1, dtype=torch.int32, device=dev)
        types = {"start": torch.int32, "stop": torch.int32, "ref": torch.uint8, "alt": torch.uint8, "p1": torch.int8, "p2": torch.int8}
        self.out = {k: torch.full((rows_total,), SENT32 if k in ("start", "stop") else SENT8, dtype=t, device=dev)
                    for k, t in types.items()}
        ptr = lambda k: self.out[k].data_ptr() if k in want else None
        capi.check(capi.lib().hb_decode_columns_device(None if absolute else base, self.off.data_ptr(), self.len.data_ptr(),
                                                       self.row.data_ptr(), len(chunks), cr, *[ptr(k) for k in COLS],
                                                       self.status.data_ptr(), None))
        torch.cuda.synchronize()

    def host(self):
        got = {k: v.cpu().numpy() for k, v in self.out.items()}
        got["start"] = got["start"].view(np.uint32)
        got["stop"] = got["stop"].view(np.uint32)
        return got, self.status.cpu().numpy()


def check_launch(got, status, expect, cr, rows, rows_total, want=COLS):
    """expect[i] = columns of chunk i (or None for a chunk that must fail); rows outside written chunks keep sentinels"""
    written = np.zeros(rows_total, bool)
    for i, exp in enumerate(expect):
        r0 = int(rows[i])
        if exp is None:
            assert status[i] != 0, i
            continue
        assert status[i] == 0, (i, status[i])
        written[r0:r0 + cr] = True
        for k in COLS:
            if k in want:
                assert np.array_equal(got[k][r0:r0 + cr], exp[k]), (i, k)
    for k in COLS:
        sent = SENT32 if k in ("start", "stop") else SENT8
        mask = ~written if k in want else np.ones(rows_total, bool)
        assert np.all(got[k][mask].astype(np.int64) & 0xFFFFFFFF == sent), k


def permuted_rows(n_chunks, cr, seed):
    """chunk i -> rows [slot_i * cr, slot_i * cr + cr): slots permuted, three unused slots as gaps"""
    rng = np.random.default_rng(seed)
    slots = rng.permutation(n_chunks + 3)[:n_chunks]
    return (slots * cr).astype(np.int64), (n_chunks + 3) * cr


def chunk_set(cr, n_chunks, seed, producers):
    """records of n_chunks chunks, producer k of chunk i = producers[i % len]; the last chunk half full (zero padding)"""
    n = n_chunks * cr - cr // 2
    rec = make_records(n, seed)
    raw = rec.tobytes() + bytes(n_chunks * cr * 35 - rec.nbytes)
    chunks, expect = [], []
    for i in range(n_chunks):
        data = raw[i * cr * 35:(i + 1) * cr * 35]
        ch = PRODUCERS[producers[i % len(producers)]](data)
        assert oracle.blosc_chunk_decode(ch, cr * 35).tobytes() == data           # the oracle agrees on the framing
        chunks.append(ch)
        expect.append(columns_of(np.frombuffer(data, oracle.RECORD_DTYPE)))
    return chunks, expect, raw


@pytest.mark.parametrize("absolute", [False, True], ids=["base+offsets", "absolute"])
@pytest.mark.parametrize("n_chunks", [1, 3, 4, 5, 257])
@pytest.mark.parametrize("cr", [1, 7, 64, 1075])
def test_columns_from_every_producer(mods, absolute, n_chunks, cr):
    chunks, expect, raw = chunk_set(cr, n_chunks, seed=n_chunks * 31 + cr, producers=list(PRODUCERS))
    rows, total = permuted_rows(n_chunks, cr, seed=cr)
    got, status = Launch(mods, chunks, cr, total, rows, absolute=absolute, seed=n_chunks).host()
    check_launch(got, status, expect, cr, rows, total)
    # only some columns asked for: the others stay untouched
    want = ("stop", "alt", "p2")
    got, status = Launch(mods, chunks, cr, total, rows, absolute=absolute, want=want, seed=n_chunks + 1).host()
    check_launch(got, status, expect, cr, rows, total, want=want)
    # the host-pointer decoder gives the same records
    capi = mods[0]
    assert capi.decode_frames(chunks, cr * 35).tobytes() == raw


def test_raw_stream_and_zero_run_chunks(mods):
    cr = 300
    rng = np.random.default_rng(4)
    noise = rng.integers(0, 256, cr * 35, dtype=np.uint8).tobytes()           # incompressible: LZ4 does not gain
    raw_chunk = oracle.reference_like_chunk(noise)
    assert struct.unpack_from("<i", raw_chunk, 20)[0] == cr * 35               # stored raw: csize == nbytes
    zeros = bytes(cr * 35)
    z2 = blosc2_chunk(zeros, zero_run=True)
    good, exp_good, _ = chunk_set(cr, 2, 9, ["lz4hc", "blosc2_lz4"])
    chunks = [raw_chunk, z2] + good
    for ch, data in zip(chunks[:2], (noise, zeros)):
        assert oracle.blosc_chunk_decode(ch, cr * 35).tobytes() == data
    expect = [columns_of(np.frombuffer(noise, oracle.RECORD_DTYPE)), columns_of(np.frombuffer(zeros, oracle.RECORD_DTYPE))] + exp_good
    rows, total = permuted_rows(len(chunks), cr, 5)
    for absolute in (False, True):
        got, status = Launch(mods, chunks, cr, total, rows, absolute=absolute).host()
        check_launch(got, status, expect, cr, rows, total)


@pytest.mark.parametrize("cr", [1, 2, 3, 6, 64, 1075, 2730])
def test_gpu_frames_at_every_geometry(mods, cr):
    """this project's own frames (Parse.compress): every column, the last chunk's zero padding decodes to zero records"""
    capi = mods[0]
    text, samples = synth.random_vcf(2900, 3, seed=cr, fmt="GT", kinds="mixed", site_mix=False)
    ora = oracle.parse_text(text, "*", "chr22")
    p = capi.Parse.from_host(synth.body_of(text), len(samples), region="chr22")
    fr = p.compress(cr)
    assert int(fr.info.chunk_records) == cr
    for s in (0, 2):
        frames = fr.sample(s)
        rec = oracle.records_from_columns(ora["chrom"], ora["start"], ora["stop"], ora["ref"], ora["alt"], ora["gt0"][s], ora["gt1"][s])
        raw = rec.tobytes() + bytes(len(frames) * cr * 35 - rec.nbytes)
        full = np.frombuffer(raw, oracle.RECORD_DTYPE)
        expect = [columns_of(full[k * cr:(k + 1) * cr]) for k in range(len(frames))]
        rows, total = permuted_rows(len(frames), cr, s)
        got, status = Launch(mods, frames, cr, total, rows, absolute=bool(s)).host()
        check_launch(got, status, expect, cr, rows, total)
        pad = len(frames) * cr - len(rec)
        if pad:
            r0 = int(rows[-1]) + cr - pad
            assert all(not got[k][r0:r0 + pad].any() for k in COLS)
        assert capi.decode_frames(frames, cr * 35).tobytes() == raw
    fr.close()
    p.close()


def _optin_smem(torch):
    return int(torch.cuda.get_device_properties(0).shared_memory_per_block_optin)


def test_largest_chunk_the_kernel_accepts(mods):
    capi, torch = mods[0], mods[1]
    cr = (_optin_smem(torch) - 1024) // 35
    chunks, expect, _ = chunk_set(cr, 3, 17, ["lz4hc", "greedy", "memcpyed"])
    rows, total = permuted_rows(3, cr, 1)
    got, status = Launch(mods, chunks, cr, total, rows).host()
    check_launch(got, status, expect, cr, rows, total)
    with pytest.raises(capi.HaploError):
        Launch(mods, chunks, cr + 1, total + 3, rows)


def test_hostile_chunks_in_one_launch(mods):
    """each bad chunk between good ones in ONE launch: its own non-zero status, every good chunk still exact"""
    capi = mods[0]
    cr = 500
    data = make_records(cr, 21).tobytes()
    good = oracle.reference_like_chunk(data)

    def mutated(at, value):
        b = bytearray(good)
        b[at:at + len(value)] = value
        return bytes(b)

    split_rec = make_records(cr, 8)
    split_rec["chrom"] = b""                                                   # byte plane 0 all zero
    split_data = split_rec.tobytes()
    hostile = [
        mutated(0, b"\x09"), mutated(2, bytes([good[2] | 0x08])), mutated(2, bytes([(good[2] & 0x1f) | (2 << 5)])),
        mutated(4, struct.pack("<I", cr * 35 + 35)), mutated(8, struct.pack("<I", 0)), mutated(8, struct.pack("<I", 1)),
        mutated(12, struct.pack("<I", len(good) + 1000)), mutated(16, struct.pack("<I", 0xfffffff0)),
        mutated(16, struct.pack("<I", 4)), mutated(20, struct.pack("<i", -5)), mutated(20, struct.pack("<I", len(good))),
        good[:len(good) // 2], mutated(24, b"\xff" * 8), mutated(len(good) - 40, b"\x00" * 8), good[:12],
        mutated(3, b"\x24"),                                                   # typesize 36
        mutated(4, struct.pack("<I", cr * 35 - 35)),                           # nbytes != 35 * cr
        mutated(16, struct.pack("<I", 12)),                                    # bstarts[0] inside the header
        oracle.blosc1_chunk_encode(data, 35, blocksize=35 * (cr // 3)),         # several Blosc blocks
        blosc2_chunk(split_data, split=True),                                  # c-blosc2 block split in 35 streams
    ]
    for h in hostile[:15]:                                                     # the oracle refuses them as well
        with pytest.raises(ValueError):
            oracle.blosc_chunk_decode(h, cr * 35)
    for h, want in ((hostile[-2], data), (hostile[-1], split_data)):           # well-formed, just not for kernel 6:
        assert oracle.blosc_chunk_decode(h, cr * 35).tobytes() == want        # the host-pointer decoder reads them
        assert capi.decode_frames([h], cr * 35).tobytes() == want
    chunks, expect = [], []
    exp_good = columns_of(np.frombuffer(data, oracle.RECORD_DTYPE))
    for h in hostile:
        chunks += [good, h]
        expect += [exp_good, None]
    chunks.append(good)
    expect.append(exp_good)
    rows, total = permuted_rows(len(chunks), cr, 3)
    for absolute in (False, True):
        got, status = Launch(mods, chunks, cr, total, rows, absolute=absolute).host()
        check_launch(got, status, expect, cr, rows, total)
        assert status[2 * (len(hostile) - 2) + 1] == 11 and status[2 * (len(hostile) - 1) + 1] == 11


# ---------------------------------------------------------------------------------------------------------------------
# the dataset on a file whose chunks the reference's writer would have stored

def _expected(items, seqs, records, L):
    """the oracle's one-hot haplotypes of each item (as in test_dataset_gpu)"""
    spec = oracle.parse_encode_dict(None)
    C_ = len(spec)
    h1 = np.zeros((len(items), L, C_), np.float32)
    h2 = np.zeros_like(h1)
    for b, (chrom, donor, ns, ne) in enumerate(items):
        win = seqs[f"chr{chrom}"][ns:ne]
        rec = records[(donor, chrom)]
        a, bb = oracle.encode_haplotypes(win, rec["start"], rec["ref"], rec["alt"], rec["phase1"], rec["phase2"], ns, ne, spec)
        n = min(len(win), L)
        h1[b, :n] = oracle.onehot(a[:n], C_)
        h2[b, :n] = oracle.onehot(bb[:n], C_)
    return h1, h2


def _positions(n, cr, rng):
    """sorted starts in [1000, ...): one value repeated across the boundary of chunks 1 and 2"""
    start = np.sort(rng.choice(np.arange(1000, 1000 + 40 * n), n, replace=False)).astype(np.uint32)
    if n > 2 * cr + 1:
        start[2 * cr - 1] = start[2 * cr] = start[2 * cr + 1] = start[2 * cr - 1]
    return np.sort(start)


def _cohort(tmp_path, mods, n, cr, encoder, name):
    capi, torch, container = mods[0], mods[1], mods[2]
    rng = np.random.default_rng(n + cr)
    donors = ["a", "b"]
    records = {}
    path = str(tmp_path / name)
    start = _positions(n, cr, rng)
    with container.open_h5(path, "w", backend="minih5") as f:
        for di, d in enumerate(donors):
            rec = np.zeros(n, oracle.RECORD_DTYPE)
            rec["chrom"] = b"chr22"
            rec["start"], rec["stop"] = start, start + 1
            rec["ref"] = rng.choice(np.array([b"A", b"C", b"G", b"T"]), n)
            rec["alt"] = rng.choice(np.array([b"A", b"C", b"G", b"T"]), n)
            rec["phase1"] = rng.choice(np.array([0, 1], np.int8), n)
            rec["phase2"] = rng.choice(np.array([0, 1, -9], np.int8), n)
            raw = rec.tobytes() + bytes((-n % cr) * 35)
            frames = [encoder(raw[k * cr * 35:(k + 1) * cr * 35]) for k in range((n + cr - 1) // cr)]
            f.write_chunked(f"donor_{d}/chr_22/snp_data", oracle.RECORD_DTYPE, n, cr, frames)
            records[(d, 22)] = rec
    return path, donors, records, start


def _run_dataset(mods, tmp_path, path, donors, records, start, cr, L=400):
    capi, torch, container, h5_reader, hd = mods
    seq = np.random.default_rng(1).choice(np.frombuffer(b"ACGT", np.uint8), size=int(start.max()) + 5000)
    seqs = {f"chr{c}": seq for c in range(1, 23)}
    (tmp_path / "samples.txt").write_text("\n".join(donors))
    bed = tmp_path / "r.bed"
    bed.write_text("chr22\t1000\t2000\n")
    ds = hd.RandomHaplotypeDataset(str(bed), path, None, str(tmp_path / "samples.txt"), batch_size=1, seq_length=L,
                                   reference_genome=hd.ReferenceGenome(sequences=seqs))
    n = len(start)
    firsts = [int(start[k * cr]) for k in range(0, (n + cr - 1) // cr)]
    ws = [int(start[n // 2]) - 7,                                              # inside a chunk
          firsts[min(1, len(firsts) - 1)] - L // 2,                            # across a chunk boundary
          firsts[min(1, len(firsts) - 1)],                                     # exactly at a chunk's first start
          int(start[min(2 * cr, n - 1)]) - 3,                                  # around the duplicated start
          int(start[min(2 * cr, n - 1)]),                                      # at it: chunk 2's first start = chunk 1's last
          max(0, int(start[0]) - L - 50),                                      # before the first record
          int(start[-1]) + 10]                                                 # after the last record
    items = [(22, d, w, w + L) for w in ws for d in donors]
    hap1, hap2 = ds.encode_items(items)
    e1, e2 = _expected(items, seqs, records, L)
    assert np.array_equal(hap1.cpu().numpy(), e1) and np.array_equal(hap2.cpu().numpy(), e2)
    store = ds.genotypes
    store.check_last()
    return ds, store


@pytest.mark.parametrize("n,cr", [(3000, oracle.guess_chunk_1d(3000)), (500, 7), (5000, 1075)])
def test_dataset_on_reference_written_file(mods, tmp_path, n, cr):
    path, donors, records, start = _cohort(tmp_path, mods, n, cr, oracle.reference_like_chunk, "ref.h5")
    ds, store = _run_dataset(mods, tmp_path, path, donors, records, start, cr)
    assert store._stored and all(v is not None for v in store._stored.values())     # compressed-resident
    assert not store._cols
    ds.close()


def test_dataset_on_multi_block_file_reads_whole(mods, tmp_path):
    cr = 300
    enc = lambda d: oracle.blosc1_chunk_encode(d, 35, blocksize=35 * 70)
    path, donors, records, start = _cohort(tmp_path, mods, 2000, cr, enc, "mb.h5")
    ds, store = _run_dataset(mods, tmp_path, path, donors, records, start, cr)
    assert store._cols and all(v is None for v in store._stored.values())            # whole-dataset fallback
    ds.close()


def test_unfiltered_chunk_reads_back(mods, tmp_path):
    """a 2-record dataset that HDF5 stored unfiltered (mask bit 0: the optional Blosc filter could not shrink it) reads
    through VCFH5Reader.fetch_genotypes and the dataset"""
    capi, torch, container, h5_reader, hd = mods
    from haplohyped_varawareml_b200 import minih5
    rec = np.zeros(2, oracle.RECORD_DTYPE)
    rec["chrom"] = b"chr22"
    rec["start"], rec["stop"] = [1100, 1200], [1101, 1201]
    rec["ref"], rec["alt"] = [b"A", b"C"], [b"G", b"T"]
    rec["phase1"], rec["phase2"] = [1, 0], [0, 1]
    cr = 2
    path = str(tmp_path / "tiny.h5")
    big = make_records(3 * 64, 2)
    big["start"] = np.arange(1000, 1000 + 3 * 64, dtype=np.uint32)
    with minih5.H5Writer(path) as w:
        cd = (2, 2, 35, cr * 35, 5, 1, 2)
        w.create_dataset_chunked("donor_a/chr_22/snp_data", oracle.RECORD_DTYPE, 2, cr, [rec.tobytes()], filter_id=32001,
                                 cd_values=cd, filter_name="blosc", masks=[1])
        # a mixed dataset: Blosc chunks and one stored unfiltered
        frames = [oracle.reference_like_chunk(big[k * 64:(k + 1) * 64].tobytes()) for k in range(3)]
        frames[1] = big[64:128].tobytes()
        w.create_dataset_chunked("donor_b/chr_22/snp_data", oracle.RECORD_DTYPE, 3 * 64, 64, frames, filter_id=32001,
                                 cd_values=(2, 2, 35, 64 * 35, 5, 1, 2), filter_name="blosc", masks=[0, 1, 0])
    rd = h5_reader.VCFH5Reader(path)
    assert rd.fetch_genotypes("a", 22).tobytes() == rec.tobytes()
    assert rd.fetch_genotypes("b", 22).tobytes() == big.tobytes()
    assert rd.stored_chunks("a", 22) is None and rd.stored_chunks("b", 22) is None
    rd.close()
    ds, store = _run_dataset(mods, tmp_path, path, ["a"], {("a", 22): rec}, rec["start"], cr)
    ds.close()
