"""VCF text -> BCF 2.2 bytes (VCF v4.3 specification, section 6.3), pure python, following htslib's choices:

- IDX= on every FILTER / INFO / FORMAT / contig line of the header (``idx=False`` leaves them out);
- a PASS filter line when the text has none, and "Dummy" lines for contigs, filters, INFO and FORMAT keys the records
  use but the header does not declare;
- integers in the smallest type that holds them (htslib's ranges: int8 from -120, int16 from -32760), GT included
  (``gt_type`` forces int16 or int32);
- a vector's count is the largest count among the samples; shorter vectors are padded with the type's vector_end;
- rlen from the END rule of the text parse (header INFO/END of Type=Integer, the first END= key, digits only, when it
  lies past POS - 1), else the REF length.

``gt_pos`` moves GT to that FORMAT position.  The result is uncompressed; wrap it with ``synth.bgzf_compress`` or gzip.
"""
from __future__ import annotations

import re
import struct

INT8, INT16, INT32, FLOAT, CHAR = 1, 2, 3, 5, 7
_PACK = {INT8: "b", INT16: "h", INT32: "i"}
VECTOR_END = {INT8: -127, INT16: -32767, INT32: -2147483647}
MISSING = {INT8: -128, INT16: -32768, INT32: -2147483648}
FLOAT_MISSING, FLOAT_END = 0x7F800001, 0x7F800002
_STRUCT_LINES = ("##FILTER=<", "##INFO=<", "##FORMAT=<", "##contig=<")


def int_type(values) -> int:
    lo, hi = min(values, default=0), max(values, default=0)
    if lo >= -120 and hi <= 127:
        return INT8
    if lo >= -32760 and hi <= 32767:
        return INT16
    return INT32


def type_byte(count: int, ty: int) -> bytes:
    if count < 15:
        return bytes([count << 4 | ty])
    return bytes([0xF0 | ty]) + typed_int(count)


def typed_int(v: int) -> bytes:
    ty = int_type([v])
    return bytes([0x10 | ty]) + struct.pack("<" + _PACK[ty], v)


def typed_ints(values, ty=None) -> bytes:
    ty = ty or int_type(values)
    return type_byte(len(values), ty) + struct.pack("<%d%s" % (len(values), _PACK[ty]), *values)


def typed_str(s: bytes) -> bytes:
    return type_byte(len(s), CHAR) + s


def hrec_attr(line: str, key: str):
    m = re.search(r"[<,]%s=(\"(?:[^\"\\]|\\.)*\"|[^,>]*)" % re.escape(key), line)
    return None if m is None else m.group(1).strip('"')


def dictionaries(header_lines):
    """(string dictionary {ID: index}, contig names by index) as htslib builds them from a header: IDX= wins; without it
    PASS = 0, then FILTER / INFO / FORMAT IDs in order of first appearance (one index per ID), contigs in order."""
    strs, nxt, contigs = {"PASS": 0}, 1, {}
    for line in header_lines:
        if not line.startswith(_STRUCT_LINES):
            continue
        ident, idx = hrec_attr(line, "ID"), hrec_attr(line, "IDX")
        if line.startswith("##contig=<"):
            contigs[int(idx) if idx is not None else (max(contigs) + 1 if contigs else 0)] = ident
        elif idx is not None:
            strs[ident] = int(idx)
            nxt = max(nxt, int(idx) + 1)
        elif ident not in strs:
            strs[ident] = nxt
            nxt += 1
    names = [contigs.get(i, "") for i in range(max(contigs) + 1 if contigs else 0)]
    return strs, names


def _end_rlen(info: str, ref: str, pos0: int, end_is_int: bool) -> int:
    rlen = len(ref)
    if end_is_int and info != ".":
        for item in info.split(";"):
            if item.startswith("END="):
                v = item[4:]
                if v and all("0" <= c <= "9" for c in v) and int(v) > pos0:
                    rlen = int(v) - pos0
                break
    return rlen


def _gt_values(field: str):
    if field in (".", ""):
        return [0]
    parts = re.split(r"([|/])", field)
    vals = []
    for i in range(0, len(parts), 2):
        a = -1 if parts[i] == "." else int(parts[i])
        phased = 1 if i > 0 and parts[i - 1] == "|" else 0
        vals.append((a + 1) << 1 | phased)
    return vals


def _fmt_field(key, ftype, subs, gt_type):
    """FORMAT field `key`: typed key is added by the caller; returns the type byte + values of all samples."""
    if key == "GT":
        vecs = [_gt_values(s) for s in subs]
        ty = gt_type or int_type([v for vec in vecs for v in vec])
        n = max(len(v) for v in vecs)
        flat = [x for vec in vecs for x in vec + [VECTOR_END[ty]] * (n - len(vec))]
        return type_byte(n, ty) + struct.pack("<%d%s" % (len(flat), _PACK[ty]), *flat)
    if ftype == "Integer":
        vecs = [[MISSING[INT32] if x == "." else int(x) for x in s.split(",")] for s in subs]
        ty = int_type([x for vec in vecs for x in vec if x != MISSING[INT32]])
        n = max(len(v) for v in vecs)
        flat = []
        for vec in vecs:
            flat += [MISSING[ty] if x == MISSING[INT32] else x for x in vec] + [VECTOR_END[ty]] * (n - len(vec))
        return type_byte(n, ty) + struct.pack("<%d%s" % (len(flat), _PACK[ty]), *flat)
    if ftype == "Float":
        vecs = [[None if x == "." else float(x) for x in s.split(",")] for s in subs]
        n = max(len(v) for v in vecs)
        out = b""
        for vec in vecs:
            for x in vec:
                out += struct.pack("<I", FLOAT_MISSING) if x is None else struct.pack("<f", x)
            out += struct.pack("<I", FLOAT_END) * (n - len(vec))
        return type_byte(n, FLOAT) + out
    bs = [s.encode() for s in subs]
    n = max(len(b) for b in bs)
    return type_byte(n, CHAR) + b"".join(b + b"\0" * (n - len(b)) for b in bs)


def _info_value(ftype, value):
    if ftype == "Flag" or value is None:
        return b"\x00"
    if ftype == "Integer":
        return typed_ints([MISSING[INT32] if x == "." else int(x) for x in value.split(",")])
    if ftype == "Float":
        vals = value.split(",")
        return type_byte(len(vals), FLOAT) + b"".join(
            struct.pack("<I", FLOAT_MISSING) if x == "." else struct.pack("<f", float(x)) for x in vals)
    return typed_str(value.encode())


def vcf_to_bcf(text: bytes, idx: bool = True, gt_type: int | None = None, gt_pos: int | None = None) -> bytes:
    lines = text.decode().replace("\r\n", "\n").split("\n")
    if lines and lines[-1] == "":
        lines.pop()
    head = [ln for ln in lines if ln.startswith("##")]
    chrom_line = next(ln for ln in lines if ln.startswith("#CHROM"))
    recs = [ln.split("\t") for ln in lines if ln and not ln.startswith("#")]
    end_is_int = any(ln.startswith("##INFO=<ID=END,") and "Type=Integer" in ln for ln in head)

    # declarations the records need and the header lacks
    declared = {(ln.split("=<")[0], hrec_attr(ln, "ID")) for ln in head if ln.startswith(_STRUCT_LINES)}
    if ("##FILTER", "PASS") not in declared:
        at = 1 if head and head[0].startswith("##fileformat") else 0
        head.insert(at, '##FILTER=<ID=PASS,Description="All filters passed">')
        declared.add(("##FILTER", "PASS"))

    def need(kind, ident, line):
        if (kind, ident) not in declared:
            declared.add((kind, ident))
            head.append(line)

    for f in recs:
        need("##contig", f[0], "##contig=<ID=%s>" % f[0])
        if f[6] != ".":
            for x in f[6].split(";"):
                need("##FILTER", x, '##FILTER=<ID=%s,Description="Dummy">' % x)
        if f[7] != ".":
            for item in f[7].split(";"):
                k = item.split("=")[0]
                kind = '##INFO=<ID=%s,Number=1,Type=String,Description="Dummy">' if "=" in item else \
                    '##INFO=<ID=%s,Number=0,Type=Flag,Description="Dummy">'
                need("##INFO", k, kind % k)
        if len(f) > 8:
            for k in f[8].split(":"):
                need("##FORMAT", k, '##FORMAT=<ID=%s,Number=1,Type=String,Description="Dummy">' % k)

    strs, contigs = dictionaries(head)
    if idx:
        out_head = []
        for ln in head:
            if ln.startswith(_STRUCT_LINES):
                ident = hrec_attr(ln, "ID")
                i = contigs.index(ident) if ln.startswith("##contig=<") else strs[ident]
                ln = ln[:-1] + ",IDX=%d>" % i
            out_head.append(ln)
        head = out_head
    types = {}
    for ln in head:
        if ln.startswith(("##INFO=<", "##FORMAT=<")):
            types[(ln[2:ln.index("=")], hrec_attr(ln, "ID"))] = hrec_attr(ln, "Type")
    htext = ("\n".join(head + [chrom_line]) + "\n").encode() + b"\0"
    n_samples = max(0, len(chrom_line.split("\t")) - 9)

    body = []
    for f in recs:
        pos0 = int(f[1]) - 1
        alleles = [f[3]] + ([] if f[4] == "." else f[4].split(","))
        shared = struct.pack("<iii", contigs.index(f[0]), pos0, _end_rlen(f[7], f[3], pos0, end_is_int))
        shared += struct.pack("<I", FLOAT_MISSING) if f[5] == "." else struct.pack("<f", float(f[5]))
        infos = [] if f[7] == "." else f[7].split(";")
        keys = f[8].split(":") if len(f) > 8 else []
        shared += struct.pack("<II", len(alleles) << 16 | len(infos), len(keys) << 24 | n_samples)
        shared += typed_str(b"" if f[2] == "." else f[2].encode())
        shared += b"".join(typed_str(a.encode()) for a in alleles)
        shared += b"\x00" if f[6] == "." else typed_ints([strs[x] for x in f[6].split(";")])
        for item in infos:
            k, _, v = item.partition("=")
            shared += typed_int(strs[k]) + _info_value(types.get(("INFO", k)), v if "=" in item else None)
        indiv = b""
        if keys:
            subs = [s.split(":") for s in f[9:]]
            order = list(range(len(keys)))
            if gt_pos is not None and "GT" in keys:
                g = keys.index("GT")
                order.remove(g)
                order.insert(min(gt_pos, len(order)), g)
            for ki in order:
                k = keys[ki]
                col = [s[ki] if ki < len(s) else "." for s in subs]
                indiv += typed_int(strs[k]) + _fmt_field(k, types.get(("FORMAT", k)), col, gt_type)
        body.append(struct.pack("<II", len(shared), len(indiv)) + shared + indiv)
    return b"BCF\x02\x02" + struct.pack("<I", len(htext)) + htext + b"".join(body)


def bcf_from_columns(header: bytes, chrom: str, start, ref, alt, gt0, gt1) -> bytes:
    """A GT-only BCF of one-base REF / ALT records built with numpy from site columns and allele planes ([S, n] int8,
    -9 = missing): fixed-size records, ID ".", FILTER PASS, no INFO, rlen 1, GT "a0|a1" as int8.  For inputs of bench
    size, where vcf_to_bcf would take too long.  header: the VCF header text, #CHROM line included."""
    import numpy as np
    head = vcf_to_bcf(header)
    l_text = struct.unpack("<I", head[5:9])[0]
    strs, contigs = dictionaries(head[9:9 + l_text - 1].decode().split("\n"))
    S, n = gt0.shape
    hdr = np.zeros(n, dtype=[("ls", "<u4"), ("li", "<u4"), ("chrom", "<i4"), ("pos", "<i4"), ("rlen", "<i4"),
                             ("qual", "<u4"), ("na", "<u4"), ("ns", "<u4")])
    hdr["ls"], hdr["li"], hdr["chrom"], hdr["pos"], hdr["rlen"] = 31, 3 + 2 * S, contigs.index(chrom), start, 1
    hdr["qual"], hdr["na"], hdr["ns"] = FLOAT_MISSING, 2 << 16, 1 << 24 | S
    rec = np.zeros((n, 42 + 2 * S), np.uint8)
    rec[:, :32] = hdr.view(np.uint8).reshape(n, 32)
    rec[:, 32:42] = [0x07, 0x17, 0, 0x17, 0, 0x11, strs["PASS"], 0x11, strs["GT"], 0x21]
    rec[:, 34] = np.frombuffer(np.asarray(ref, "S1").tobytes(), np.uint8)
    rec[:, 36] = np.frombuffer(np.asarray(alt, "S1").tobytes(), np.uint8)
    v = rec[:, 42:].reshape(n, S, 2)
    for p, g in ((0, gt0), (1, gt1)):
        a = g.T.astype(np.int16)
        v[:, :, p] = np.where(a < 0, 0, (a + 1) << 1) | p
    return head + rec.tobytes()
