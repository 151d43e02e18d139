"""minih5 -- a minimal HDF5 (file format 1.x, "earliest" feature set) writer and reader.

Why it exists: the reference stores its output through h5py/libhdf5 (`vcf_to_h5.py:131-135`), and
neither is installed in this image (no network).  GPU-compressed chunks enter a stock HDF5 file
through the direct-chunk-write API when h5py is present (`container.py`); when it is not, this
module writes the same on-disk structures itself: superblock v0, v1 object headers, old-style
groups (v1 B-tree + local heap + symbol-table nodes), chunked datasets indexed by a v1 chunk
B-tree, filter pipeline message v1 -- exactly what h5py's default (libver="earliest") emits for
the reference's `/donor_{id}/chr_{N}/snp_data` layout.

STATUS: written from the published HDF5 File Format Specification v1.1 from memory; no libhdf5
is reachable here to confirm that a stock reader accepts these files.  The reader below parses the
same subset (and is what the dataset mirror uses in this image).  Scope: 1-D datasets of a
compound / fixed-string / integer type, chunked (+ optional filter) or contiguous.
"""
from __future__ import annotations

import struct
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

UNDEF = 0xFFFFFFFFFFFFFFFF
SIGNATURE = b"\x89HDF\r\n\x1a\n"
GROUP_LEAF_K = 4          # symbol-table node holds up to 2K entries
GROUP_INTERNAL_K = 16     # group B-tree node holds up to 2K children
CHUNK_K = 32              # chunk B-tree node holds up to 2K children (library default, not stored in superblock v0)
SUPERBLOCK_RESERVE = 2048


def _pad8(b: bytes) -> bytes:
    return b + b"\0" * (-len(b) % 8)


# ------------------------------------------------------------------------------------------------
# datatype messages
# ------------------------------------------------------------------------------------------------
def _dtype_message(dt: np.dtype) -> bytes:
    dt = np.dtype(dt)
    if dt.fields:
        members = b""
        for name in dt.names:
            fdt, off = dt.fields[name][0], dt.fields[name][1]
            members += _pad8(name.encode() + b"\0")
            members += struct.pack("<IB3xII4I", off, 0, 0, 0, 0, 0, 0, 0)
            members += _dtype_message(fdt)
        n = len(dt.names)
        return struct.pack("<BBBBI", 0x16, n & 0xFF, (n >> 8) & 0xFF, 0, dt.itemsize) + members
    if dt.kind == "S":
        return struct.pack("<BBBBI", 0x13, 0x01, 0, 0, dt.itemsize)            # fixed string, null-padded, ASCII
    if dt.kind in "iu":
        bits = 0x08 if dt.kind == "i" else 0x00                                 # little-endian, signed flag
        return struct.pack("<BBBBIHH", 0x10, bits, 0, 0, dt.itemsize, 0, 8 * dt.itemsize)
    raise TypeError(f"minih5: unsupported dtype {dt}")


def _parse_dtype(buf: bytes, pos: int = 0) -> Tuple[np.dtype, int]:
    cv, b0, b1, b2, size = struct.unpack_from("<BBBBI", buf, pos)
    cls, ver = cv & 0x0F, cv >> 4
    pos += 8
    if cls == 0:
        pos += 4
        return np.dtype(("<i" if b0 & 0x08 else "<u") + str(size)), pos
    if cls == 3:
        return np.dtype("S%d" % size), pos
    if cls == 6:
        n = b0 | (b1 << 8)
        names, fmts, offs = [], [], []
        for _ in range(n):
            e = buf.index(b"\0", pos)
            name = buf[pos:e].decode()
            if ver < 3:
                pos += (e - pos + 8) & ~7
            else:
                pos = e + 1
            if ver == 1:
                off = struct.unpack_from("<I", buf, pos)[0]
                pos += 4 + 28
            elif ver == 2:
                off = struct.unpack_from("<I", buf, pos)[0]
                pos += 4
            else:
                nb = max(1, (size.bit_length() + 7) // 8)
                off = int.from_bytes(buf[pos:pos + nb], "little")
                pos += nb
            fdt, pos = _parse_dtype(buf, pos)
            names.append(name); fmts.append(fdt); offs.append(off)
        return np.dtype({"names": names, "formats": fmts, "offsets": offs, "itemsize": size}), pos
    raise TypeError(f"minih5: unsupported datatype class {cls}")


# ------------------------------------------------------------------------------------------------
# writer
# ------------------------------------------------------------------------------------------------
class _Group:
    def __init__(self):
        self.children: Dict[str, object] = {}     # name -> _Group | int (object header address)


class H5Writer:
    """Append-only writer: dataset payloads are written as they arrive, all metadata at close()."""

    def __init__(self, path: str):
        self.f = open(path, "wb")
        self.f.write(b"\0" * SUPERBLOCK_RESERVE)
        self.pos = SUPERBLOCK_RESERVE
        self.root = _Group()
        self.closed = False

    # -- low level
    def _write(self, b: bytes, align: int = 8) -> int:
        pad = -self.pos % align
        if pad:
            self.f.write(b"\0" * pad)
            self.pos += pad
        addr = self.pos
        self.f.write(b)
        self.pos += len(b)
        return addr

    def _object_header(self, messages: Sequence[Tuple[int, bytes]]) -> int:
        body = b""
        for mtype, data in messages:
            data = _pad8(data)
            body += struct.pack("<HHB3x", mtype, len(data), 0) + data
        hdr = struct.pack("<BBHII4x", 1, 0, len(messages), 1, len(body))
        return self._write(hdr + body)

    def _link(self, path: str, addr: int):
        parts = [p for p in path.split("/") if p]
        g = self.root
        for p in parts[:-1]:
            nxt = g.children.get(p)
            if nxt is None:
                nxt = _Group()
                g.children[p] = nxt
            if not isinstance(nxt, _Group):
                raise ValueError(f"{p} is not a group")
            g = nxt
        if parts[-1] in g.children:
            raise ValueError(f"{path} already exists")
        g.children[parts[-1]] = addr

    # -- datasets
    def _common_messages(self, dtype: np.dtype, n: int) -> List[Tuple[int, bytes]]:
        dataspace = struct.pack("<BBB5xQQ", 1, 1, 1, n, n)
        fill = struct.pack("<BBBBi", 2, 3, 2, 1, 0)           # v2, alloc incremental, write if-set, default value
        return [(0x0001, dataspace), (0x0003, _dtype_message(dtype)), (0x0005, fill)]

    def create_dataset_contiguous(self, path: str, data: np.ndarray):
        data = np.ascontiguousarray(data)
        addr = self._write(data.tobytes()) if data.nbytes else UNDEF
        layout = struct.pack("<BBQQ", 3, 1, addr, data.nbytes)
        msgs = self._common_messages(data.dtype, data.shape[0])
        msgs[2] = (0x0005, struct.pack("<BBBBi", 2, 1, 2, 1, 0))   # contiguous: early allocation
        self._link(path, self._object_header(msgs + [(0x0008, layout)]))

    def create_dataset_chunked(self, path: str, dtype: np.dtype, n: int, chunk: int, chunks: Sequence[bytes],
                               filter_id: Optional[int] = None, cd_values: Sequence[int] = (), filter_name: str = "",
                               masks: Optional[Sequence[int]] = None):
        """chunks[k] = the bytes to store for chunk k (already filtered when filter_id is given).  masks[k] = chunk k's
        filter mask: bit i set = filter i of the pipeline was skipped, as HDF5 does when an optional filter fails."""
        dtype = np.dtype(dtype)
        entries = []
        for k, payload in enumerate(chunks):
            mask = int(masks[k]) if masks is not None else 0
            entries.append((len(payload), mask, k * chunk, self._write(bytes(payload), align=1)))
        btree = self._chunk_btree(entries, chunk, len(entries) * chunk) if entries else UNDEF
        layout = struct.pack("<BBBQII", 3, 2, 2, btree, chunk, dtype.itemsize)
        msgs = self._common_messages(dtype, n) + [(0x0008, layout)]
        if filter_id is not None:
            name = _pad8(filter_name.encode() + b"\0") if filter_name else b""
            cd = b"".join(struct.pack("<I", v & 0xFFFFFFFF) for v in cd_values)
            if len(cd_values) % 2:
                cd += b"\0\0\0\0"
            filt = struct.pack("<HHHH", filter_id, len(name), 1, len(cd_values)) + name + cd
            msgs.append((0x000B, struct.pack("<BB6x", 1, 1) + filt))
        self._link(path, self._object_header(msgs))

    def write_blob(self, data, align: int = 16) -> int:
        """Append raw bytes (anything with the buffer protocol) and return their address.  Used to put ALL stored
        chunks of many datasets into the file with one write; the datasets are then declared with
        create_dataset_chunked_at."""
        pad = -self.pos % align
        if pad:
            self.f.write(b"\0" * pad)
            self.pos += pad
        addr = self.pos
        mv = memoryview(data).cast("B")
        self.f.write(mv)
        self.pos += mv.nbytes
        return addr

    def create_dataset_chunked_at(self, path: str, dtype: np.dtype, n: int, chunk: int, addrs: np.ndarray,
                                  sizes: np.ndarray, filter_id: Optional[int] = None, cd_values: Sequence[int] = (),
                                  filter_name: str = ""):
        """Chunked dataset whose stored chunks already sit in the file: chunk k = sizes[k] bytes at addrs[k]."""
        dtype = np.dtype(dtype)
        addrs = np.asarray(addrs, np.uint64)
        sizes = np.asarray(sizes, np.uint32)
        btree = self._chunk_btree_np(sizes, addrs, chunk) if len(addrs) else UNDEF
        layout = struct.pack("<BBBQII", 3, 2, 2, btree, chunk, dtype.itemsize)
        msgs = self._common_messages(dtype, n) + [(0x0008, layout)]
        if filter_id is not None:
            name = _pad8(filter_name.encode() + b"\0") if filter_name else b""
            cd = b"".join(struct.pack("<I", v & 0xFFFFFFFF) for v in cd_values)
            if len(cd_values) % 2:
                cd += b"\0\0\0\0"
            filt = struct.pack("<HHHH", filter_id, len(name), 1, len(cd_values)) + name + cd
            msgs.append((0x000B, struct.pack("<BB6x", 1, 1) + filt))
        self._link(path, self._object_header(msgs))

    _KEY_DT = np.dtype([("size", "<u4"), ("mask", "<u4"), ("off", "<u8"), ("zero", "<u8"), ("child", "<u8")])

    def _chunk_btree_np(self, sizes: np.ndarray, addrs: np.ndarray, chunk: int) -> int:
        """_chunk_btree with the node bodies assembled by numpy (a node body is an array of key+child records)."""
        cap = 2 * CHUNK_K
        node_size = 24 + (cap + 1) * 24 + cap * 8
        n = len(sizes)
        rec = np.zeros(n, self._KEY_DT)
        rec["size"], rec["off"], rec["child"] = sizes, np.arange(n, dtype=np.uint64) * np.uint64(chunk), addrs
        last_key = struct.pack("<IIQQ", 0, 0, n * chunk, 0)
        level = 0
        while True:
            m = len(rec)
            ngroups = (m + cap - 1) // cap
            base = self._write(b"", align=8)
            node_addr = base + np.arange(ngroups, dtype=np.uint64) * np.uint64(node_size)
            raw = rec.tobytes()
            out = bytearray()
            for gi in range(ngroups):
                lo, hi = gi * cap, min(m, (gi + 1) * cap)
                body = raw[lo * 32:hi * 32]
                final = raw[hi * 32:hi * 32 + 24] if hi < m else last_key
                left = int(node_addr[gi - 1]) if gi > 0 else UNDEF
                right = int(node_addr[gi + 1]) if gi + 1 < ngroups else UNDEF
                node = b"TREE" + struct.pack("<BBHQQ", 1, level, hi - lo, left, right) + body + final
                out += node + b"\0" * (node_size - len(node))
            self._write(bytes(out))
            if ngroups == 1:
                return int(node_addr[0])
            nxt = np.zeros(ngroups, self._KEY_DT)
            first = rec[::cap]
            nxt["size"], nxt["mask"], nxt["off"], nxt["child"] = first["size"], first["mask"], first["off"], node_addr
            rec = nxt
            level += 1

    def _chunk_btree(self, entries, chunk: int, end_offset: int) -> int:
        """v1 B-tree, node type 1.  entries: (stored size, filter mask, element offset, address), offset-sorted."""
        def key(size, mask, off):
            return struct.pack("<IIQQ", size, mask, off, 0)
        cap = 2 * CHUNK_K
        level = 0
        nodes = [(key(s, m, o), a, None) for s, m, o, a in entries]   # (first key, child address, last key of subtree)
        last_key = key(0, 0, end_offset)
        while True:
            groups = [nodes[i:i + cap] for i in range(0, len(nodes), cap)]
            addrs = []
            node_size = 24 + (cap + 1) * 24 + cap * 8
            base = self._write(b"", align=8)
            for gi in range(len(groups)):
                addrs.append(base + gi * node_size)
            out = []
            for gi, g in enumerate(groups):
                body = b""
                for k, a, _ in g:
                    body += k + struct.pack("<Q", a)
                final = groups[gi + 1][0][0] if gi + 1 < len(groups) else last_key
                body += final
                body += b"\0" * (node_size - 24 - len(body))
                left = addrs[gi - 1] if gi > 0 else UNDEF
                right = addrs[gi + 1] if gi + 1 < len(groups) else UNDEF
                self._write(b"TREE" + struct.pack("<BBHQQ", 1, level, len(g), left, right) + body)
                out.append((g[0][0], addrs[gi], None))
            if len(out) == 1:
                return out[0][1]
            nodes = out
            level += 1

    # -- groups
    def _write_group(self, g: _Group) -> Tuple[int, int, int]:
        """Returns (object header address, btree address, heap address)."""
        items = []
        for name, child in g.children.items():
            if isinstance(child, _Group):
                child = self._write_group(child)[0]
            items.append((name.encode(), child))
        items.sort(key=lambda t: t[0])                     # strcmp order
        heap = bytearray(b"\0" * 8)                        # offset 0: the empty string
        offs = []
        for name, _ in items:
            offs.append(len(heap))
            heap += _pad8(name + b"\0")
        heap_data = self._write(bytes(heap))
        heap_addr = self._write(b"HEAP" + struct.pack("<B3xQQQ", 0, len(heap), 1, heap_data))
        # symbol-table nodes
        cap = 2 * GROUP_LEAF_K
        snods = []
        for i in range(0, max(1, len(items)), cap):
            part = list(zip(offs[i:i + cap], items[i:i + cap]))
            body = b""
            for off, (_, addr) in part:
                body += struct.pack("<QQII16x", off, addr, 0, 0)
            body += b"\0" * (40 * (cap - len(part)))
            a = self._write(b"SNOD" + struct.pack("<BBH", 1, 0, len(part)) + body)
            snods.append((a, part[-1][0] if part else 0))
        # group B-tree (node type 0): key[i+1] = heap offset of the largest name under child i
        capb = 2 * GROUP_INTERNAL_K
        level = 0
        nodes = snods
        while True:
            groups = [nodes[i:i + capb] for i in range(0, len(nodes), capb)]
            node_size = 24 + (capb + 1) * 8 + capb * 8
            base = self._write(b"", align=8)
            addrs = [base + gi * node_size for gi in range(len(groups))]
            out = []
            prev_last = 0
            for gi, grp in enumerate(groups):
                body = struct.pack("<Q", prev_last)
                for a, last in grp:
                    body += struct.pack("<QQ", a, last)
                body += b"\0" * (node_size - 24 - len(body))
                left = addrs[gi - 1] if gi > 0 else UNDEF
                right = addrs[gi + 1] if gi + 1 < len(groups) else UNDEF
                self._write(b"TREE" + struct.pack("<BBHQQ", 0, level, len(grp), left, right) + body)
                prev_last = grp[-1][1]
                out.append((addrs[gi], grp[-1][1]))
            if len(out) == 1:
                btree = out[0][0]
                break
            nodes = out
            level += 1
        ohdr = self._object_header([(0x0011, struct.pack("<QQ", btree, heap_addr))])
        return ohdr, btree, heap_addr

    def close(self):
        if self.closed:
            return
        ohdr, btree, heap = self._write_group(self.root)
        eof = self._write(b"", align=8)
        sb = SIGNATURE + struct.pack("<BBBBBBBBHHI", 0, 0, 0, 0, 0, 8, 8, 0, GROUP_LEAF_K, GROUP_INTERNAL_K, 0)
        sb += struct.pack("<QQQQ", 0, UNDEF, eof, UNDEF)
        sb += struct.pack("<QQII", 0, ohdr, 1, 0) + struct.pack("<QQ", btree, heap)
        self.f.seek(0)
        self.f.write(sb)
        self.f.close()
        self.closed = True

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


# ------------------------------------------------------------------------------------------------
# reader
# ------------------------------------------------------------------------------------------------
class DatasetInfo:
    def __init__(self):
        self.dtype = None
        self.shape = ()
        self.layout = None            # "contiguous" | "chunked"
        self.addr = UNDEF
        self.size = 0
        self.chunk = 0
        self.btree = UNDEF
        self.filters: List[Tuple[int, Tuple[int, ...]]] = []


class H5Reader:
    def __init__(self, path: str):
        self.f = open(path, "rb")
        head = self.f.read(96)
        if head[:8] != SIGNATURE:
            raise OSError(f"{path}: not an HDF5 file")
        if head[8] != 0 or head[13] != 8 or head[14] != 8:
            raise OSError("minih5 reads superblock version 0 with 8-byte offsets/lengths only")
        self.leaf_k, self.internal_k = struct.unpack_from("<HH", head, 16)
        root = head[56:96]
        self.root_ohdr = struct.unpack_from("<Q", root, 8)[0]
        self._groups: Dict[int, Dict[str, int]] = {}

    def _read(self, addr: int, n: int) -> bytes:
        self.f.seek(addr)
        return self.f.read(n)

    def _messages(self, addr: int) -> List[Tuple[int, bytes]]:
        ver, _, nmsg, _, hsize = struct.unpack("<BBHII", self._read(addr, 12))
        if ver != 1:
            raise OSError("minih5 reads version 1 object headers only")
        out = []
        blocks = [(addr + 16, hsize)]
        while blocks and len(out) < nmsg:
            baddr, bsize = blocks.pop(0)
            buf = self._read(baddr, bsize)
            p = 0
            while p + 8 <= len(buf) and len(out) < nmsg:
                mtype, msize, _ = struct.unpack_from("<HHB", buf, p)
                data = buf[p + 8:p + 8 + msize]
                p += 8 + msize
                if mtype == 0x0010:                       # continuation
                    blocks.append(struct.unpack("<QQ", data[:16]))
                out.append((mtype, data))
        return out

    def _group_entries(self, ohdr: int) -> Dict[str, int]:
        if ohdr in self._groups:
            return self._groups[ohdr]
        st = [d for t, d in self._messages(ohdr) if t == 0x0011]
        if not st:
            raise KeyError("not a group")
        btree, heap = struct.unpack("<QQ", st[0][:16])
        hv = self._read(heap, 32)
        seg_size, _, seg_addr = struct.unpack_from("<QQQ", hv, 8)
        names = self._read(seg_addr, seg_size)
        entries: Dict[str, int] = {}

        def walk(node):
            h = self._read(node, 24)
            if h[:4] == b"SNOD":
                nsym = struct.unpack_from("<H", h, 6)[0]
                body = self._read(node + 8, 40 * nsym)
                for i in range(nsym):
                    off, oa = struct.unpack_from("<QQ", body, 40 * i)
                    e = names.index(b"\0", off)
                    entries[names[off:e].decode()] = oa
                return
            if h[:4] != b"TREE":
                raise OSError("bad group node")
            used = struct.unpack_from("<H", h, 6)[0]
            body = self._read(node + 24, 8 + 16 * used)
            for i in range(used):
                walk(struct.unpack_from("<Q", body, 8 + 16 * i)[0])

        walk(btree)
        self._groups[ohdr] = entries
        return entries

    def _resolve(self, path: str) -> int:
        addr = self.root_ohdr
        for p in [x for x in path.split("/") if x]:
            ent = self._group_entries(addr)
            if p not in ent:
                raise KeyError(path)
            addr = ent[p]
        return addr

    def __contains__(self, path: str) -> bool:
        try:
            self._resolve(path)
            return True
        except KeyError:
            return False

    def keys(self, path: str = "/") -> List[str]:
        return sorted(self._group_entries(self._resolve(path)))

    def dataset_info(self, path: str) -> DatasetInfo:
        info = DatasetInfo()
        for t, d in self._messages(self._resolve(path)):
            if t == 0x0001:
                rank, flags = d[1], d[2]
                info.shape = struct.unpack_from("<%dQ" % rank, d, 8)
            elif t == 0x0003:
                info.dtype = _parse_dtype(d)[0]
            elif t == 0x0008:
                if d[0] != 3:
                    raise OSError("minih5 reads layout message version 3 only")
                if d[1] == 1:
                    info.layout = "contiguous"
                    info.addr, info.size = struct.unpack_from("<QQ", d, 2)
                elif d[1] == 2:
                    info.layout = "chunked"
                    nd = d[2]
                    info.btree = struct.unpack_from("<Q", d, 3)[0]
                    info.chunk = struct.unpack_from("<%dI" % nd, d, 11)[0]
                else:
                    raise OSError("minih5: compact layout not supported")
            elif t == 0x000B:
                nf = d[1]
                p = 8
                for _ in range(nf):
                    fid, nlen, _, ncd = struct.unpack_from("<HHHH", d, p)
                    p += 8 + nlen
                    cd = struct.unpack_from("<%dI" % ncd, d, p)
                    p += 4 * ncd + (4 if ncd % 2 else 0)
                    info.filters.append((fid, tuple(cd)))
        return info

    def chunks(self, info: DatasetInfo) -> List[Tuple[int, bytes]]:
        """[(element offset, stored bytes)] in offset order (the filter masks dropped: see chunks_with_masks)."""
        return [(off, b) for off, b, _ in self.chunks_with_masks(info)]

    def chunks_with_masks(self, info: DatasetInfo) -> List[Tuple[int, bytes, int]]:
        """[(element offset, stored bytes, filter mask)] in offset order.  Bit i of the mask set = filter i of the
        pipeline was not applied to this chunk (an optional filter that failed on it): those bytes are not filtered."""
        out = []

        def walk(node):
            h = self._read(node, 24)
            if h[:4] != b"TREE" or h[4] != 1:
                raise OSError("bad chunk B-tree node")
            level, used = h[5], struct.unpack_from("<H", h, 6)[0]
            body = self._read(node + 24, used * 32 + 24)
            for i in range(used):
                size, mask, off, _ = struct.unpack_from("<IIQQ", body, 32 * i)
                child = struct.unpack_from("<Q", body, 32 * i + 24)[0]
                if level:
                    walk(child)
                else:
                    out.append((off, self._read(child, size), mask))

        if info.btree != UNDEF:
            walk(info.btree)
        out.sort(key=lambda t: t[0])
        return out

    def read_contiguous(self, info: DatasetInfo) -> np.ndarray:
        n = info.shape[0]
        raw = self._read(info.addr, n * info.dtype.itemsize) if n else b""
        return np.frombuffer(raw, info.dtype).copy()

    def close(self):
        self.f.close()
