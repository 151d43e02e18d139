"""Host-side mirror of the reference's src/datasets/haplotype_dataset.py.

`RandomHaplotypeDataset` keeps the reference's constructor arguments, `__len__`, `__getitem__(idx)
-> (hap1, hap2)` and `close()` (haplotype_dataset.py:30-114).  What changes is where the work runs:
the whole batch is built by ONE launch of the CUDA kernel behind `hb_encode_haplotypes`
(csrc/hb_hap.cu) from device-resident columns, and the tensors it returns are CUDA float32
`[batch_size, 2*(seq_length//2), C]`.

Kept literally from the reference (SURVEY.md 8a, A12-A14):
  * three `np.random.randint` draws per item, in the order region, donor, chromosome, from the
    global numpy RNG seeded once in `__init__` (:40,:49,:59-61); `idx` is ignored (:54);
  * the chromosome is drawn independently of the BED row, whose `chrom` column is never read;
  * window = calculate_midpoint_region(start, end, seq_length) (:11-16), i.e. 2*(L//2) bases,
    clamped at 0;
  * phase == 1 -> ALT index, anything else -> the record's REF index; last duplicate wins.
Repairs (the reference code cannot run as written, SURVEY.md D4-D10): R1 haplotypes start from the
encoded reference window, R2 only records inside the window are applied, R3 one-hot columns follow
encode_spec order, R4 records are read from `snp_data` with group key `chr_{N}` and the reference
sequence from key `chr{N}`.  Windows shortened by the clamp (or by the end of the chromosome) are
padded with all-zero rows so the batch stays rectangular.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch
from torch.utils.data import Dataset

from . import capi
from .common_utils import build_lut, parse_encode_dict


def calculate_midpoint_region(start, end, seq_length):
    """haplotype_dataset.py:11-16, verbatim."""
    midpt = (start + end) // 2
    half_seq_length = seq_length // 2
    new_start = max(0, midpt - half_seq_length)
    new_end = midpt + half_seq_length
    return new_start, new_end


# ------------------------------------------------------------------------------------------------
# device-resident sources
# ------------------------------------------------------------------------------------------------
class ReferenceGenome:
    """Reference bases per chromosome key (`chr{N}`), resident in HBM as uint8 ASCII.

    Mirrors the reference's local ReferenceGenome (haplotype_dataset.py:18-28): get_sequence(chrom,
    start, end) -> |S1 array; `device_sequence` is what the kernel reads."""

    def __init__(self, h5_file=None, encode_spec=None, sequences=None, device="cuda:0"):
        self.encode_spec = parse_encode_dict(encode_spec)
        self.device = torch.device(device)
        self._host = {}
        self._dev = {}
        self._h5 = None
        if sequences is not None:
            for k, v in sequences.items():
                self._host[k] = np.frombuffer(v, np.uint8) if isinstance(v, (bytes, bytearray)) else np.asarray(v).view(np.uint8)
        elif h5_file is not None:
            from .container import open_h5
            self._h5 = open_h5(h5_file, "r")

    def _host_seq(self, chrom):
        if chrom not in self._host:
            if self._h5 is None or chrom not in self._h5:
                raise KeyError(f"No reference sequence for {chrom}")
            self._host[chrom] = np.ascontiguousarray(self._h5.read_dataset(chrom)).view(np.uint8).reshape(-1)
        return self._host[chrom]

    def get_sequence(self, chrom, start, end):
        return self._host_seq(chrom)[start:end].view("|S1")

    def device_sequence(self, chrom) -> torch.Tensor:
        if chrom not in self._dev:
            self._dev[chrom] = torch.from_numpy(np.ascontiguousarray(self._host_seq(chrom))).to(self.device)
        return self._dev[chrom]

    def close(self):
        if self._h5 is not None:
            self._h5.close()


class _DevAddr:
    """A device address that is kept alive by something else (quacks like a tensor for data_ptr())."""

    def __init__(self, addr, owner):
        self._addr, self._owner = int(addr), owner

    def data_ptr(self):
        return self._addr


class _Stored:
    """One dataset as the file stores it, resident in HBM: blob (uint8 tensor) + per-chunk offsets / sizes (host)."""
    __slots__ = ("blob", "offs", "sizes", "n", "cr")

    def __init__(self, blob, offs, sizes, n, cr):
        self.blob, self.offs, self.sizes, self.n, self.cr = blob, offs, sizes, n, cr


class GenotypeStore:
    """(donor, chromosome) -> device columns (start u32 sorted, ref u8, alt u8, phase1 i8, phase2 i8).

    `from_reader` pulls record arrays through VCFH5Reader.fetch_genotypes (the reference's access
    path, h5_reader.py:23-43) and keeps the columns in HBM; `from_parse` points straight at the
    planes a device-resident parse already holds (no copy)."""

    def __init__(self, device="cuda:0"):
        self.device = torch.device(device)
        self._cols = {}
        self._reader = None
        self._parses = {}
        self._stored = {}          # (donor, chrom) -> _Stored | None
        self._first = {}           # (chrom, n_records, chunk_records) -> first start of every chunk
        self.last_status = []

    @classmethod
    def from_reader(cls, reader, device="cuda:0"):
        st = cls(device)
        st._reader = reader
        return st

    @classmethod
    def from_records(cls, records: dict, device="cuda:0"):
        """records: {(donor, chrom:int): structured array with start/ref/alt/phase1/phase2}."""
        st = cls(device)
        for key, rec in records.items():
            st._cols[key] = st._upload(rec)
        return st

    def add_parse(self, chrom: int, parse, sample_names):
        """Zero-copy: columns of a capi.Parse (kept alive by this store)."""
        self._parses[chrom] = (parse, {n: i for i, n in enumerate(sample_names)})

    def add_frames(self, chrom: int, frames, sample_names):
        """Zero-copy: the stored chunks of every sample of a capi.Frames handle (kept alive by this store) serve as the
        compressed-resident datasets of `chrom` -- converter output used straight from HBM."""
        i = frames.info
        offs, sizes = frames.layout()
        for s, name in enumerate(sample_names):
            self._stored[(name, chrom)] = _Stored(_DevAddr(i.d_frames, frames), offs[s].copy(), sizes[s].copy(), int(i.n_records), int(i.chunk_records))

    def _upload(self, rec):
        dev = self.device
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        ref = np.ascontiguousarray(rec["ref"]).view(np.uint8).reshape(len(rec), -1)[:, 0] if len(rec) else np.zeros(0, np.uint8)
        alt = np.ascontiguousarray(rec["alt"]).view(np.uint8).reshape(len(rec), -1)[:, 0] if len(rec) else np.zeros(0, np.uint8)
        return (t(rec["start"].astype(np.uint32).view(np.int32)), t(ref), t(alt),
                t(rec["phase1"].astype(np.int8)), t(rec["phase2"].astype(np.int8)), len(rec))

    # ---- compressed-resident datasets (SURVEY 8 row f4): the stored chunks of a (donor, chromosome) dataset stay in HBM as
    # they are in the file; a batch decodes, on the device, only the chunks its windows touch.  The reference reads and
    # decodes the whole dataset for every item (h5_reader.py:37-41, haplotype_dataset.py:71): O(chromosome) per item.
    def _compressed(self, donor, chrom: int):
        """-> _Stored of the dataset, uploading its stored chunks on first use; None when the file does not store it as
        single-block Blosc chunks (then `columns` decodes it whole, once)."""
        key = (donor, chrom)
        if key in self._stored:
            return self._stored[key]
        st = None
        got = self._reader.stored_chunks(donor, chrom) if (self._reader is not None and hasattr(self._reader, "stored_chunks")) else None
        if got is not None:
            n, cr, dtype, chunks = got
            # up to 7,489 records a chunk of the reference's writer is ONE Blosc block, which the device decoder reads;
            # chunks with several blocks make the first decode fail and the dataset is then read whole (_chunk_first)
            if dtype.itemsize == 35 and n > 0 and cr <= 7489:
                sizes = np.array([len(c) for c in chunks], np.uint32)
                offs = np.zeros(len(chunks), np.uint64)
                offs[1:] = np.cumsum((sizes[:-1].astype(np.uint64) + 15) // 16 * 16)
                blob = np.zeros(int(offs[-1]) + int(sizes[-1]) + 64, np.uint8)
                for o, c in zip(offs, chunks):
                    blob[int(o):int(o) + len(c)] = np.frombuffer(c, np.uint8)
                st = _Stored(torch.from_numpy(blob).to(self.device), offs, sizes, n, cr)
        self._stored[key] = st
        return st

    def _chunk_first(self, chrom: int, st):
        """First `start` of every chunk of the chromosome (host, sorted): built once per (chromosome, geometry) by decoding
        the start column of the first dataset seen -- every donor of a cohort file has the same sites (one VCF per
        chromosome, vcf_to_h5.py:182-207), so it serves all of them."""
        key = (chrom, st.n, st.cr)
        if key not in self._first:
            nck = len(st.sizes)
            start = torch.empty(nck * st.cr, dtype=torch.int32, device=self.device)
            status = self._decode(st, np.arange(nck), np.arange(nck, dtype=np.uint64) * st.cr, start=start)
            if bool(status.any().item()):         # e.g. several Blosc blocks per chunk: this file is read whole instead
                self._first[key] = None
            else:
                self._first[key] = start[::st.cr].cpu().numpy().view(np.uint32).astype(np.int64)
        return self._first[key]

    def _decode(self, st, chunk_ids, rows, start=None, ref=None, alt=None, p1=None, p2=None, frames=None, offs=None, lens=None):
        """hb_decode_columns_device_large (every single-block chunk size) on chunks `chunk_ids` of one stored dataset (or on
        pre-built device lists)."""
        dev = self.device
        n = len(chunk_ids)
        if offs is None:
            base = st.blob.data_ptr()
            offs = torch.from_numpy((st.offs[chunk_ids]).astype(np.int64)).to(dev)
            lens = torch.from_numpy(st.sizes[chunk_ids].view(np.int32)).to(dev)
            frames = base
        rows_t = torch.from_numpy(np.asarray(rows, np.uint64).view(np.int64)).to(dev)
        status = torch.empty(n, dtype=torch.int32, device=dev)
        ptr = lambda t: t.data_ptr() if t is not None else None
        capi.check(capi.lib().hb_decode_columns_device_large(frames, offs.data_ptr(), lens.data_ptr(), rows_t.data_ptr(), n, st.cr,
                                                       ptr(start), None, ptr(ref), ptr(alt), ptr(p1), ptr(p2), status.data_ptr(),
                                                       torch.cuda.current_stream(dev).cuda_stream))
        return status

    def window_columns(self, items):
        """items: [(donor, chrom, new_start, new_end)] -> per item (addr_start, addr_ref, addr_alt, addr_p1, addr_p2, n_records)
        covering at least every record with new_start <= start < new_end, decoded on the device from the resident
        stored chunks in ONE launch for the whole batch; `keep` (second result) must outlive the kernel that reads them.
        Items whose dataset is not kept compressed fall back to `columns`."""
        dev = self.device
        self.check_last()
        plan, out = [], [None] * len(items)
        for b, (donor, chrom, ws, we) in enumerate(items):
            st = None if chrom in self._parses or (donor, chrom) in self._cols else self._compressed(donor, chrom)
            if st is None:
                out[b] = self.columns(donor, chrom)
                continue
            first = self._chunk_first(chrom, st)
            if first is None:
                self._stored[(donor, chrom)] = None
                out[b] = self.columns(donor, chrom)
                continue
            c0 = max(0, int(np.searchsorted(first, ws, "left")) - 1)
            c1 = max(c0, int(np.searchsorted(first, we, "left")) - 1)
            plan.append((b, st, c0, c1))
        keep = None
        if plan:
            by_cr = {}
            for b, st, c0, c1 in plan:
                by_cr.setdefault(st.cr, []).append((b, st, c0, c1))
            keep = []
            for cr, group in by_cr.items():
                tot = sum(c1 - c0 + 1 for _, _, c0, c1 in group)
                addr = np.empty(tot, np.uint64); lens = np.empty(tot, np.uint32); rows = np.empty(tot, np.uint64)
                k = 0
                spans = []
                for b, st, c0, c1 in group:
                    m = c1 - c0 + 1
                    addr[k:k + m] = np.uint64(st.blob.data_ptr()) + st.offs[c0:c1 + 1]
                    lens[k:k + m] = st.sizes[c0:c1 + 1]
                    rows[k:k + m] = (np.arange(m, dtype=np.uint64) + np.uint64(k)) * np.uint64(cr)
                    spans.append((b, k, m, min(st.n - c0 * cr, m * cr)))
                    k += m
                start = torch.empty(tot * cr, dtype=torch.int32, device=dev)
                ref = torch.empty(tot * cr, dtype=torch.uint8, device=dev); alt = torch.empty_like(ref)
                p1 = torch.empty(tot * cr, dtype=torch.int8, device=dev); p2 = torch.empty_like(p1)
                # chunk addresses are absolute: frames base 0, offsets = device addresses
                offs_t = torch.from_numpy(addr.view(np.int64)).to(dev)
                lens_t = torch.from_numpy(lens.view(np.int32)).to(dev)
                status = self._decode(group[0][1], range(tot), rows, start, ref, alt, p1, p2, frames=0, offs=offs_t, lens=lens_t)
                keep.append((start, ref, alt, p1, p2, offs_t, lens_t, status))
                for b, k0, m, nrec in spans:
                    o = k0 * cr
                    out[b] = (start.data_ptr() + 4 * o, ref.data_ptr() + o, alt.data_ptr() + o, p1.data_ptr() + o, p2.data_ptr() + o, int(nrec))
            self.last_status = [t[-1] for t in keep]
        return out, keep

    def check_last(self):
        """Raise if a chunk of the previous batch did not decode (checked one batch late: no sync on the hot path)."""
        bad = [t for t in self.last_status if bool(t.any().item())]
        self.last_status = []
        if bad:
            raise OSError("corrupt or unsupported stored chunk in the genotype file (device decode status %d)" % int(bad[0].max().item()))

    def columns(self, donor, chrom: int):
        """-> (addr_start, addr_ref, addr_alt, addr_p1, addr_p2, n_records) device addresses."""
        if chrom in self._parses:
            parse, idx = self._parses[chrom]
            if donor not in idx:
                raise KeyError(f"No data found for donor_{donor}/chr_{chrom}")
            i = parse.info
            s = idx[donor]
            return (i.d_start, i.d_ref, i.d_alt, i.d_gt[0] + s * i.gt_stride, i.d_gt[1] + s * i.gt_stride,
                    int(i.n_records))
        key = (donor, chrom)
        if key not in self._cols:
            if self._reader is None:
                raise KeyError(f"No data found for donor_{donor}/chr_{chrom}")
            self._cols[key] = self._upload(self._reader.fetch_genotypes(donor, chrom))
        c = self._cols[key]
        return (c[0].data_ptr(), c[1].data_ptr(), c[2].data_ptr(), c[3].data_ptr(), c[4].data_ptr(), c[5])

    def close(self):
        if self._reader is not None:
            self._reader.close()
        self._cols.clear()
        self._parses.clear()
        self._stored.clear()
        self._first.clear()


# ------------------------------------------------------------------------------------------------
def _launch(B, L, Cn, seq_addr, lens, wstart, cols, lut, device, stream=None):
    """cols: list of (start, ref, alt, p1, p2, nrec) device-address tuples, one per item."""
    dev = torch.device(device)
    hap1 = torch.empty((B, L, Cn), dtype=torch.float32, device=dev)
    hap2 = torch.empty((B, L, Cn), dtype=torch.float32, device=dev)
    meta = np.zeros((9, B), dtype=np.uint64)
    meta[0] = seq_addr
    meta[1] = lens
    meta[2] = wstart
    for b, c in enumerate(cols):
        meta[3:9, b] = c
    m = torch.from_numpy(meta.view(np.int64)).to(dev)
    lens32 = torch.from_numpy(np.asarray(lens, np.uint32).view(np.int32)).to(dev)
    ws32 = torch.from_numpy(np.asarray(wstart, np.uint32).view(np.int32)).to(dev)
    lut_t = torch.from_numpy(lut.copy()).to(dev)
    hb = capi.HapBatch()
    hb.B, hb.L, hb.C = B, L, Cn
    hb.item_seq = m[0].data_ptr()
    hb.item_len = lens32.data_ptr()
    hb.item_win_start = ws32.data_ptr()
    hb.item_start, hb.item_ref, hb.item_alt = m[3].data_ptr(), m[4].data_ptr(), m[5].data_ptr()
    hb.item_p1, hb.item_p2, hb.item_nrec = m[6].data_ptr(), m[7].data_ptr(), m[8].data_ptr()
    hb.lut = lut_t.data_ptr()
    hb.hap1, hb.hap2 = hap1.data_ptr(), hap2.data_ptr()
    hb.stream = stream if stream is not None else torch.cuda.current_stream(dev).cuda_stream
    capi.check(capi.lib().hb_encode_haplotypes(C.byref(hb)))
    # m / lens32 / ws32 / lut_t must outlive the (stream-ordered) launch: torch's caching allocator
    # only reuses them for later work on the same stream, which is what we launched on
    return hap1, hap2


def onehot_windows(windows, L, encode_spec=None, ignore_case=True, device="cuda:0"):
    """One-hot of plain byte windows (no variants): the GPU form of encode_sequence."""
    spec = parse_encode_dict(encode_spec)
    lut = build_lut(spec, ignore_case)
    dev = torch.device(device)
    bufs = [torch.from_numpy(np.ascontiguousarray(w)).to(dev) for w in windows]
    B = len(windows)
    cols = [(0, 0, 0, 0, 0, 0)] * B
    h1, _ = _launch(B, L, len(spec), [b.data_ptr() for b in bufs], [len(w) for w in windows], [0] * B, cols, lut, dev)
    torch.cuda.synchronize(dev)
    return h1


class RandomHaplotypeDataset(Dataset):
    def __init__(self, bed_file, hdf5_genotype_file, hdf5_reference_file, samples_file, encode_spec=None, seed=42,
                 batch_size=1, seq_length=1000, device="cuda:0", genotype_store=None, reference_genome=None):
        # BED: tab separated, no header, columns chrom/start/end (haplotype_dataset.py:32)
        starts, ends = [], []
        with open(bed_file) as f:
            for line in f:
                if not line.strip():
                    continue
                c = line.rstrip("\n").split("\t")
                starts.append(int(c[1]))
                ends.append(int(c[2]))
        self.bed_start = np.asarray(starts, np.int64)
        self.bed_end = np.asarray(ends, np.int64)
        self.device = torch.device(device)
        if genotype_store is None:
            from .h5_reader import VCFH5Reader
            self.vcf_reader = VCFH5Reader(hdf5_genotype_file)
            genotype_store = GenotypeStore.from_reader(self.vcf_reader, device)
        self.genotypes = genotype_store
        self.reference_genome = reference_genome or ReferenceGenome(hdf5_reference_file, encode_spec, device=device)
        self.encode_spec = parse_encode_dict(encode_spec)
        self.lut = build_lut(self.encode_spec)
        self.donor_ids = self.read_samples(samples_file)
        self.chromosomes = np.arange(1, 23)
        self.batch_size = batch_size
        self.seq_length = seq_length
        self.set_random_seed(seed)
        self.num_samples = len(self.bed_start)

    def read_samples(self, samples_file):
        with open(samples_file, "r") as f:
            donors = [line.strip() for line in f]
        return donors

    def set_random_seed(self, seed):
        np.random.seed(seed)

    def __len__(self):
        return self.num_samples

    def draw(self):
        """The reference's sampling loop (:58-68) without the encoding: [(chrom, donor, new_start, new_end)]."""
        items = []
        for _ in range(self.batch_size):
            region_idx = np.random.randint(0, self.num_samples)
            donor_idx = np.random.randint(0, len(self.donor_ids))
            chrom_idx = np.random.randint(0, len(self.chromosomes))
            donor_id = self.donor_ids[donor_idx]
            chrom = int(self.chromosomes[chrom_idx])
            start, end = int(self.bed_start[region_idx]), int(self.bed_end[region_idx])
            new_start, new_end = calculate_midpoint_region(start, end, self.seq_length)
            items.append((chrom, donor_id, new_start, new_end))
        return items

    def encode_items(self, items):
        L = 2 * (self.seq_length // 2)
        B = len(items)
        seq_addr, lens, ws = [], [], []
        keep = []
        # record columns of every item: decoded on the device from the resident stored chunks, window-limited
        cols, keep_cols = self.genotypes.window_columns([(d, c, a, e) for c, d, a, e in items])
        keep.append(keep_cols)
        for chrom, donor_id, new_start, new_end in items:
            seq = self.reference_genome.device_sequence(f"chr{chrom}")
            keep.append(seq)
            n = int(seq.numel())
            ln = max(0, min(new_end, n) - new_start)
            seq_addr.append(seq.data_ptr() + min(new_start, n))
            lens.append(min(ln, L))
            ws.append(new_start)
        return _launch(B, L, len(self.encode_spec), seq_addr, lens, ws, cols, self.lut, self.device)

    def __getitem__(self, idx):
        return self.encode_items(self.draw())

    def close(self):
        self.genotypes.close()
        self.reference_genome.close()
