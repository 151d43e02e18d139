"""Tabix (.tbi) and CSI (.csi) indexes in pure Python, restated from the hts-specs (SAMv1 section 5, "Indexing BAM";
tabix.pdf; CSIv1.pdf), independently of the native reader:

- reg2bin / reg2bins, the binning scheme;
- a writer over the uncompressed text of a VCF (or the bytes of an uncompressed BCF) and the BGZF members of its
  compressed form: what `tabix -p vcf`, `tabix -C -p vcf` and `bcftools index` compute;
- a reader, and the query of one interval (the chunks a reader has to visit).

Bins are written in ascending order; the specs leave the order open (htslib writes its hash table's order)."""
import bisect
import gzip
import struct

import synth

MIN_MARKER_DIST = 0x10000        # compress_binning: a bin whose chunks span less than this many compressed bytes moves up
VCF_CONF = (2, 1, 2, 0, ord("#"), 0)   # tabix conf of a VCF: format, col_seq, col_beg, col_end, meta char, skip


def bin_first(level: int) -> int:
    return ((1 << (3 * level)) - 1) // 7


def bin_parent(b: int) -> int:
    return (b - 1) >> 3


def bin_level(b: int) -> int:
    level = 0
    while b:
        b = bin_parent(b)
        level += 1
    return level


def reg2bin(beg: int, end: int, min_shift: int = 14, depth: int = 5) -> int:
    """The smallest bin that holds [beg, end) (0-based, half open)."""
    end -= 1
    s, t = min_shift, bin_first(depth)
    for level in range(depth, 0, -1):
        if beg >> s == end >> s:
            return t + (beg >> s)
        s += 3
        t -= 1 << (3 * (level - 1))
    return 0


def reg2bins(beg: int, end: int, min_shift: int = 14, depth: int = 5):
    """Every bin that overlaps [beg, end), level by level."""
    if beg >= end:
        return []
    end = min(end, 1 << (min_shift + 3 * depth)) - 1
    out = []
    for level in range(depth + 1):
        s = min_shift + 3 * (depth - level)
        out.extend(range(bin_first(level) + (beg >> s), bin_first(level) + (end >> s) + 1))
    return out


# ---- BGZF geometry: virtual offsets of text positions
def bgzf_members(data: bytes):
    """[(compressed address, text offset, text length, member size)] of BGZF bytes."""
    out, p, t = [], 0, 0
    while p < len(data):
        xlen = struct.unpack_from("<H", data, p + 10)[0]
        q, bsize = p + 12, None
        while q < p + 12 + xlen:
            slen = struct.unpack_from("<H", data, q + 2)[0]
            if data[q:q + 2] == b"BC":
                bsize = struct.unpack_from("<H", data, q + 4)[0] + 1
            q += 4 + slen
        isize = struct.unpack_from("<I", data, p + bsize - 4)[0]
        out.append((p, t, isize, bsize))
        t += isize
        p += bsize
    return out


class VirtualOffsets:
    """Text position -> BGZF virtual offset (coffset << 16 | uoffset).  A position at the end of a member's text is the
    start of the next member, (its address, 0): where a reader stands after reading the member's last byte."""

    def __init__(self, members):
        self.m = [m for m in members if m[2]]
        self.starts = [m[1] for m in self.m]

    def __call__(self, t: int) -> int:
        if t == 0 or not self.m:
            return (self.m[0][0] if self.m else 0) << 16
        i = bisect.bisect_left(self.starts, t) - 1
        addr, off, n, size = self.m[i]
        return (addr + size) << 16 if t - off == n else addr << 16 | (t - off)


# ---- records: (tid, beg, end, start voff, end voff)
def vcf_records(text: bytes, vo: VirtualOffsets):
    """tabix's reading of a VCF: sequence names in order of first appearance, [POS - 1, POS - 1 + len(REF)), or INFO/END
    when it is greater than POS - 1.  Returns (names, offset after the header, records)."""
    names, tids, recs = [], {}, []
    p, off0, in_header = 0, 0, True
    while p < len(text):
        e = text.find(b"\n", p)
        e = len(text) if e < 0 else e + 1
        line = text[p:e].rstrip(b"\n").rstrip(b"\r")
        if line.startswith(b"#"):
            assert in_header, "header line after a record"
            off0 = vo(e)
        elif line:
            in_header = False
            f = line.split(b"\t", 8)
            chrom = f[0].decode()
            if chrom not in tids:
                tids[chrom] = len(names)
                names.append(chrom)
            beg = max(int(f[1]) - 1, 0)
            end = beg + len(f[3]) if len(f) > 3 else beg + 1
            info = f[7] if len(f) > 7 else b""
            at = 0 if info.startswith(b"END=") else (info.find(b";END=") + 1 or -1)
            if at >= 0 and info[at + 4:at + 5] != b".":
                digits = info[at + 4:]
                k = 0
                while k < len(digits) and digits[k:k + 1].isdigit():
                    k += 1
                if k and int(digits[:k]) > beg:
                    end = int(digits[:k])
            recs.append((tids[chrom], beg, max(end, 1), vo(p), vo(e)))
        p = e
    return names, off0, recs


def bcf_records(raw: bytes, vo: VirtualOffsets):
    """The records of an uncompressed BCF 2.2: [pos, pos + rlen).  Returns (offset after the header, records)."""
    l_text = struct.unpack_from("<I", raw, 5)[0]
    p = 9 + l_text
    off0, recs = vo(p), []
    while p < len(raw):
        l_shared, l_indiv, rid, pos, rlen = struct.unpack_from("<IIiii", raw, p)
        e = p + 8 + l_shared + l_indiv
        recs.append((rid, pos, pos + rlen, vo(p), vo(e)))
        p = e
    return off0, recs


def bcf_depth(raw: bytes, min_shift: int) -> int:
    """bcftools' CSI depth: enough levels for the longest ##contig length (2^31 - 1 when none is given) + 256."""
    l_text = struct.unpack_from("<I", raw, 5)[0]
    longest = 0
    for line in raw[9:9 + l_text].decode().split("\n"):
        if line.startswith("##contig=<") and "length=" in line:
            longest = max(longest, int(line.split("length=")[1].split(",")[0].split(">")[0]))
    longest = (longest or (1 << 31) - 1) + 256
    depth, s = 0, 1 << min_shift
    while longest > s:
        depth += 1
        s <<= 3
    return depth


# ---- the index: binning (chunks per bin), linear index, per-sequence meta
def build(n_ref, off0, recs, final_off, min_shift, depth):
    """Chunks close where the (tid, bin) of consecutive records changes; then bins too small to be worth a seek merge into
    their parents and chunks that share a BGZF block merge, as the specs' reference implementation does."""
    max_pos = 1 << (min_shift + 3 * depth)
    n_bins = ((1 << (3 * depth + 3)) - 1) // 7
    meta_bin = n_bins
    refs = [None] * n_ref               # {bin: [[u, v], ...]}, linear index, meta
    lin = [dict() for _ in range(n_ref)]
    seen, last_tid, last_beg = set(), None, -1
    cur = None                          # open chunk: [tid, bin, u]
    n_mapped, seq_beg = 0, off0
    prev_end = off0

    def close(v):
        tid, b, u = cur
        refs[tid].setdefault(b, []).append([u, v])

    for tid, beg, end, u, v in recs:
        if end > max_pos or beg > max_pos:
            raise ValueError("position %d cannot be stored in this index" % end)
        if tid != last_tid:
            if tid in seen:
                raise ValueError("chromosome blocks not continuous")
            if cur is not None:
                close(prev_end)
                refs[cur[0]].setdefault(meta_bin, []).extend([[seq_beg, prev_end], [n_mapped, 0]])
                n_mapped, seq_beg = 0, prev_end
                cur = None
            seen.add(tid)
            refs[tid] = {}
            last_tid, last_beg = tid, -1
        elif beg < last_beg:
            raise ValueError("unsorted positions")
        b = reg2bin(beg, end, min_shift, depth)
        if cur is None or cur[1] != b:
            if cur is not None:
                close(prev_end)
            cur = [tid, b, prev_end]
        for w in range(beg >> min_shift, ((end - 1) >> min_shift) + 1):
            lin[tid].setdefault(w, prev_end)
        n_mapped += 1
        last_beg = beg
        prev_end = v
    if cur is not None:
        close(final_off)
        refs[cur[0]].setdefault(meta_bin, []).extend([[seq_beg, final_off], [n_mapped, 0]])

    out = []
    for tid in range(n_ref):
        bins = refs[tid]
        if bins is None:
            out.append(({}, []))
            continue
        # linear index: gaps take the window before them; leading gaps the sequence's first offset
        n = max(lin[tid]) + 1 if lin[tid] else 0
        first = bins[meta_bin][0][0] if meta_bin in bins else 0
        lidx = []
        for w in range(n):
            lidx.append(lin[tid].get(w, lidx[-1] if lidx else first))
        loff = {b: (lidx[(b - bin_first(bin_level(b))) << 3 * (depth - bin_level(b))]
                    if b < n_bins and ((b - bin_first(bin_level(b))) << 3 * (depth - bin_level(b))) < n else 0)
                for b in bins}
        # merge small bins into their parents, bottom level first
        for level in range(depth, 0, -1):
            for b in sorted(k for k in bins if bin_first(level) <= k < n_bins):
                ch = bins[b]
                if level < depth:
                    ch.sort()
                if (ch[-1][1] >> 16) - (ch[0][0] >> 16) < MIN_MARKER_DIST and bin_parent(b) in bins:
                    bins[bin_parent(b)].extend(ch)
                    del bins[b]
        if 0 in bins:
            bins[0].sort()
        for b, ch in bins.items():
            if b >= n_bins:
                continue
            merged = [ch[0]]
            for c in ch[1:]:
                if merged[-1][1] >> 16 >= c[0] >> 16:
                    merged[-1][1] = max(merged[-1][1], c[1])
                else:
                    merged.append(c)
            bins[b] = merged
        out.append(({b: (loff.get(b, 0), [tuple(c) for c in bins[b]]) for b in sorted(bins)}, lidx))
    return out


def _tabix_meta(names) -> bytes:
    nm = b"".join(n.encode() + b"\0" for n in names)
    return struct.pack("<6i", *VCF_CONF) + struct.pack("<i", len(nm)) + nm


def serialise(refs, fmt: str, min_shift=14, depth=5, names=None) -> bytes:
    """The uncompressed bytes of a TBI (fmt "tbi") or CSI (fmt "csi") index."""
    if fmt == "tbi":
        out = [b"TBI\1", struct.pack("<i", len(refs)), _tabix_meta(names)]
    else:
        aux = _tabix_meta(names) if names is not None else b""
        out = [b"CSI\1", struct.pack("<3i", min_shift, depth, len(aux)), aux, struct.pack("<i", len(refs))]
    for bins, lidx in refs:
        out.append(struct.pack("<i", len(bins)))
        for b, (loff, ch) in bins.items():
            out.append(struct.pack("<I", b))
            if fmt == "csi":
                out.append(struct.pack("<Q", loff))
            out.append(struct.pack("<i", len(ch)))
            out.extend(struct.pack("<QQ", u, v) for u, v in ch)
        if fmt == "tbi":
            out.append(struct.pack("<i", len(lidx)))
            out.extend(struct.pack("<Q", o) for o in lidx)
    out.append(struct.pack("<Q", 0))    # n_no_coor
    return b"".join(out)


def index_vcf(text: bytes, bgzf: bytes, fmt: str = "tbi", min_shift: int = 14) -> bytes:
    """The uncompressed index of `bgzf`, the BGZF form of the VCF `text`."""
    vo = VirtualOffsets(bgzf_members(bgzf))
    names, off0, recs = vcf_records(text, vo)
    depth = 5 if fmt == "tbi" else (31 - min_shift + 2) // 3
    if fmt == "tbi":
        min_shift = 14
    refs = build(len(names), off0, recs, vo(len(text)), min_shift, depth)
    return serialise(refs, fmt, min_shift, depth, names)


def index_bcf(raw: bytes, bgzf: bytes, min_shift: int = 14) -> bytes:
    """The uncompressed CSI of `bgzf`, the BGZF form of the uncompressed BCF `raw`."""
    vo = VirtualOffsets(bgzf_members(bgzf))
    off0, recs = bcf_records(raw, vo)
    depth = bcf_depth(raw, min_shift)
    l_text = struct.unpack_from("<I", raw, 5)[0]
    n_ref = max(raw[9:9 + l_text].count(b"\n##contig=<"), max((r[0] for r in recs), default=-1) + 1)   # every header contig
    refs = build(n_ref, off0, recs, vo(len(raw)), min_shift, depth)
    return serialise(refs, "csi", min_shift, depth, None)


def write(index_bytes: bytes) -> bytes:
    """An index file: the index BGZF-compressed."""
    return synth.bgzf_compress(index_bytes)


# ---- reading and querying
def read(data: bytes):
    """dict(fmt, min_shift, depth, names, refs=[(bins {bin: (loff, [(u, v)])}, lidx)], n_no_coor) of an index file."""
    raw = gzip.decompress(data)
    p = 4
    out = {"fmt": raw[:4], "names": None}

    def i32():
        nonlocal p
        p += 4
        return struct.unpack_from("<i", raw, p - 4)[0]

    def u64():
        nonlocal p
        p += 8
        return struct.unpack_from("<Q", raw, p - 8)[0]

    def meta(end):
        nonlocal p
        p += 24
        l_nm = i32()
        names = raw[p:p + l_nm].split(b"\0")[:-1]
        p += l_nm
        return [n.decode() for n in names]

    if raw[:4] == b"TBI\1":
        out["min_shift"], out["depth"] = 14, 5
        n_ref = i32()
        out["names"] = meta(None)
    elif raw[:4] == b"CSI\1":
        out["min_shift"], out["depth"] = i32(), i32()
        l_aux = i32()
        if l_aux:
            q = p
            out["names"] = meta(None)
            p = q + l_aux
        n_ref = i32()
    else:
        raise ValueError("bad magic")
    csi = raw[:4] == b"CSI\1"
    refs = []
    for _ in range(n_ref):
        bins = {}
        for _ in range(i32()):
            p += 4
            b = struct.unpack_from("<I", raw, p - 4)[0]
            loff = u64() if csi else 0
            bins[b] = (loff, [(u64(), u64()) for _ in range(i32())])
        lidx = [] if csi else [u64() for _ in range(i32())]
        refs.append((bins, lidx))
    out["refs"] = refs
    out["n_no_coor"] = u64() if p + 8 <= len(raw) else None
    return out


def query(idx, tid: int, beg: int, end: int):
    """Merged [(u, v)] chunks that may hold records of tid overlapping [beg, end), in file order."""
    ms, depth = idx["min_shift"], idx["depth"]
    beg, end = max(beg, 0), min(end, 1 << (ms + 3 * depth))
    if tid < 0 or tid >= len(idx["refs"]) or beg >= end:
        return []
    bins, lidx = idx["refs"][tid]
    if not bins:
        return []
    n_bins = ((1 << (3 * depth + 3)) - 1) // 7

    def loff(b):
        if idx["fmt"] == b"CSI\1":
            return bins[b][0]
        if b >= n_bins:
            return 0
        level = bin_level(b)
        w = (b - bin_first(level)) << 3 * (depth - level)
        return lidx[w] if w < len(lidx) else 0

    b = bin_first(depth) + (beg >> ms)
    while b and b not in bins:
        first = (bin_parent(b) << 3) + 1
        b = b - 1 if b > first else bin_parent(b)
    min_off = loff(b) if b in bins else 0
    off = sorted(c for k in reg2bins(beg, end, ms, depth) if k in bins for c in bins[k][1] if c[1] > min_off)
    if not off:
        return []
    kept = [list(off[0])]
    for c in off[1:]:
        if kept[-1][1] < c[1]:
            kept.append(list(c))
    for i in range(1, len(kept)):
        if kept[i - 1][1] >= kept[i][0]:
            kept[i - 1][1] = kept[i][0]
    merged = [kept[0]]
    for c in kept[1:]:
        if merged[-1][1] >> 16 == c[0] >> 16:
            merged[-1][1] = c[1]
        else:
            merged.append(c)
    return [tuple(c) for c in merged]


# ---- test data
def multi_contig_vcf(contigs, n_per: int, n_samples: int, seed: int = 0, fmt: str = "GT", info_end: bool = False,
                     first_pos: int = 0) -> bytes:
    """A sorted VCF of synth.random_vcf records on several contigs, one block each (the rows random_vcf puts on other
    contigs are moved to the block's own).  first_pos shifts every position."""
    out = []
    for k, c in enumerate(contigs):
        text, _ = synth.random_vcf(n_per, n_samples, seed=seed + k, fmt=fmt, chrom=c, info_end=info_end)
        lines = text.split(b"\n")
        if k == 0:
            out.extend(x for x in lines if x.startswith(b"#"))
        for x in lines:
            if x and not x.startswith(b"#"):
                f = x.split(b"\t")
                f[0] = c.encode()
                if first_pos:
                    f[1] = str(int(f[1]) + first_pos).encode()
                    f[7] = b";".join(b"END=%d" % (int(i[4:]) + first_pos) if i.startswith(b"END=") else i
                                     for i in f[7].split(b";"))
                out.append(b"\t".join(f))
    return b"\n".join(out) + b"\n"
