"""Kernel 0 (inflate_bgzf_kernel) on DEFLATE streams that Python's zlib never writes, but bgzip built with libdeflate
and other encoders do: code-length repeats across the literal/length -> distance boundary, codes of every length
1-15 on both sides of the primary-table widths, empty and one-bit distance codes, block types mixed inside one member,
every length / distance symbol at both ends of its extra bits, runs of every short period, and members at every payload
alignment.  The streams come from the small bit writer below, built from explicit code lengths and symbol lists.

The CPU tests check the writer itself against stock zlib: every valid stream inflates with zlib to the bytes a plain
Python LZ77 expansion of its tokens gives, and every invalid stream makes zlib raise.  The GPU tests then require the
kernel to give zlib's bytes for the valid streams and to refuse each invalid one."""
import gzip
import random
import struct
import zlib

import pytest

# ---------------------------------------------------------------------------------------------------------------------
# DEFLATE bit writer (RFC 1951)

CLORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
LBASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
DBASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
         6145, 8193, 12289, 16385, 24577]
DEXTRA = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]
FIXED_LIT = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
FIXED_DIST = [5] * 32


class BitWriter:
    def __init__(self):
        self.acc, self.n, self.out = 0, 0, bytearray()

    def put(self, v, k):                                   # k bits of v, least significant first
        self.acc |= (v & ((1 << k) - 1)) << self.n
        self.n += k
        while self.n >= 8:
            self.out.append(self.acc & 255)
            self.acc >>= 8
            self.n -= 8

    def put_code(self, code):                              # a Huffman code goes most significant bit first
        v, k = code
        self.put(int(format(v, "0%db" % k)[::-1], 2) if k else 0, k)

    def align(self):
        if self.n:
            self.put(0, 8 - self.n)

    def getvalue(self):
        self.align()
        return bytes(self.out)


def canonical(lens):
    """code lengths -> [(code, length) or None] (RFC 1951 3.2.2)"""
    mx = max(lens, default=0)
    bl = [0] * (mx + 2)
    for L in lens:
        if L:
            bl[L] += 1
    code, nxt = 0, [0] * (mx + 2)
    for b in range(1, mx + 1):
        code = (code + bl[b - 1]) << 1
        nxt[b] = code
    codes = []
    for L in lens:
        if L:
            codes.append((nxt[L], L))
            nxt[L] += 1
        else:
            codes.append(None)
    return codes


def complete_lengths(symbols, n):
    """A complete code over `symbols` (>= 2 of them) among n: lengths m-1 and m"""
    k = len(symbols)
    m = (k - 1).bit_length()
    short = (1 << m) - k
    lens = [0] * n
    for i, s in enumerate(sorted(symbols)):
        lens[s] = m - 1 if i < short else m
    return lens


def kraft(lens):
    return sum(2.0 ** -L for L in lens if L)


def rle_lengths(seq):
    """code lengths -> code-length symbols [(sym, extra)], repeats allowed across the literal/length -> distance
    boundary (libdeflate does this; zlib sends the two sets apart)"""
    out, i = [], 0
    while i < len(seq):
        v, j = seq[i], i
        while j < len(seq) and seq[j] == v:
            j += 1
        run = j - i
        if v == 0 and run >= 3:
            r = min(run, 138)
            out.append((18, r - 11) if r >= 11 else (17, r - 3))
            i += r
            continue
        out.append((v, 0))
        i += 1
        run -= 1
        while run >= 3:
            r = min(run, 6)
            out.append((16, r - 3))
            i += r
            run -= r
    return out


def expand_cl(cl_syms):
    seq = []
    for s, e in cl_syms:
        if s < 16:
            seq.append(s)
        elif s == 16:
            seq += [seq[-1]] * (3 + e)
        elif s == 17:
            seq += [0] * (3 + e)
        else:
            seq += [0] * (11 + e)
    return seq


CL_EXTRA = {16: 2, 17: 3, 18: 7}


def dynamic_header(w, litlens, distlens, cl_syms=None, cllens=None, hclen=None):
    """HLIT / HDIST / HCLEN, the code-length code and the code lengths.  Returns (literal codes, distance codes)."""
    if cl_syms is None:
        cl_syms = rle_lengths(litlens + distlens)
    if cllens is None:
        used = sorted({s for s, _ in cl_syms})
        if len(used) == 1:                                 # a complete code-length code needs two codes
            used.append(0 if used[0] else 1)
        cllens = complete_lengths(used, 19)
    if hclen is None:
        hclen = max(4, max(i + 1 for i, s in enumerate(CLORDER) if cllens[s]))
    w.put(len(litlens) - 257, 5)
    w.put(len(distlens) - 1, 5)
    w.put(hclen - 4, 4)
    for s in CLORDER[:hclen]:
        w.put(cllens[s], 3)
    cc = canonical(cllens)
    for s, e in cl_syms:
        w.put_code(cc[s])
        if s in CL_EXTRA:
            w.put(e, CL_EXTRA[s])
    return canonical(litlens), canonical(distlens)


def length_token(length):
    s = max(i for i in range(29) if LBASE[i] <= length and (i < 28 or length == 258))
    if length == 258:
        s = 28
    return 257 + s, length - LBASE[s]


def dist_token(d):
    s = max(i for i in range(30) if DBASE[i] <= d)
    return s, d - DBASE[s]


def match(length, d):
    """('m', length symbol, its extra, distance symbol, its extra)"""
    return ("m",) + length_token(length) + dist_token(d)


def put_symbols(w, lc, dc, toks):
    """toks: ints (literal bytes / 256 / any raw literal-length symbol) or match tuples; no end-of-block is added"""
    for t in toks:
        if isinstance(t, int):
            w.put_code(lc[t])
            continue
        _, ls, le, ds, de = t
        w.put_code(lc[ls])
        if 257 <= ls <= 284:
            w.put(le, LEXTRA[ls - 257])
        w.put_code(dc[ds])
        if ds < 30:
            w.put(de, DEXTRA[ds])


def expand(toks, out):
    """plain LZ77 expansion of tokens onto bytearray `out` (the reference the kernel is held to)"""
    for t in toks:
        if isinstance(t, int):
            assert t < 256
            out.append(t)
            continue
        _, ls, le, ds, de = t
        length, d = LBASE[ls - 257] + le, DBASE[ds] + de
        assert 3 <= length <= 258 and d <= len(out)
        for _ in range(length):
            out.append(out[-d])
    return out


class Stream:
    """Blocks appended one by one; .expected is the LZ77 expansion of every token written"""

    def __init__(self):
        self.w, self.expected = BitWriter(), bytearray()

    def dynamic(self, toks, litlens, distlens, last=False, **hdr):
        self.w.put(int(last), 1)
        self.w.put(2, 2)
        lc, dc = dynamic_header(self.w, litlens, distlens, **hdr)
        put_symbols(self.w, lc, dc, list(toks) + [256])
        expand(toks, self.expected)
        return self

    def fixed(self, toks, last=False):
        self.w.put(int(last), 1)
        self.w.put(1, 2)
        put_symbols(self.w, canonical(FIXED_LIT), canonical(FIXED_DIST), list(toks) + [256])
        expand(toks, self.expected)
        return self

    def stored(self, data, last=False, nlen=None):
        self.w.put(int(last), 1)
        self.w.put(0, 2)
        self.w.align()
        self.w.put(len(data), 16)
        self.w.put((~len(data) & 0xFFFF) if nlen is None else nlen, 16)
        self.w.out += data
        self.expected += data
        return self

    def getvalue(self):
        return self.w.getvalue()


def lit_lens_for(toks, extra=(), n=None):
    """a complete literal/length code over the symbols the tokens use (+ 256 + extra)"""
    syms = {256, *extra}
    for t in toks:
        syms.add(t if isinstance(t, int) else t[1])
    n = n or max(257, max(syms) + 1)
    return complete_lengths(sorted(syms), n)


def dist_lens_for(toks, n=None):
    syms = {t[3] for t in toks if not isinstance(t, int)}
    n = n or max(1, max(syms, default=0) + 1)
    if len(syms) < 2:
        syms |= {0, 1} if n > 1 else set()
    if not syms:
        return [0] * n
    return complete_lengths(sorted(syms), max(n, max(syms) + 1))


def dyn_stream(toks, last=True, litlens=None, distlens=None, **hdr):
    s = Stream()
    s.dynamic(toks, litlens or lit_lens_for(toks), distlens or dist_lens_for(toks), last=last, **hdr)
    return s


# ---------------------------------------------------------------------------------------------------------------------
# BGZF framing (SAM/BAM spec 4.1): gzip member with a 'BC' subfield holding BSIZE - 1

def bgzf_member(payload, text, extra_before=None, extra_after=None, isize=None, crc=None):
    """one member; extra_before / extra_after: data bytes of a foreign subfield ('XY') placed before / after BC"""
    sub = b""
    if extra_before is not None:
        sub += b"XY" + struct.pack("<H", len(extra_before)) + extra_before
    bc_at = len(sub)
    sub += b"BC\x02\x00\x00\x00"
    if extra_after is not None:
        sub += b"XY" + struct.pack("<H", len(extra_after)) + extra_after
    total = 12 + len(sub) + len(payload) + 8
    assert total <= 65536, total
    sub = bytearray(sub)
    sub[bc_at + 4:bc_at + 6] = struct.pack("<H", total - 1)
    head = struct.pack("<BBBBIBBH", 0x1f, 0x8b, 8, 4, 0, 0, 0xff, len(sub))
    tail = struct.pack("<II", zlib.crc32(text) if crc is None else crc, len(text) if isize is None else isize)
    return head + bytes(sub) + payload + tail


BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")

# XLEN 6 (BC only) and 10..13 (a subfield of 0-3 data bytes): DEFLATE payloads start at every address mod 4
FRAMINGS = [dict(), dict(extra_before=b""), dict(extra_after=b"\x01"), dict(extra_before=b"\x01\x02"),
            dict(extra_after=b"\x01\x02\x03")]


def framings_for(members):
    """the framings every member fits in (the largest stored block fits with XLEN 6 only)"""
    return [fr for fr in FRAMINGS
            if all(12 + 6 + sum(4 + len(v) for v in fr.values()) + len(p) + 8 <= 65536 for p, _ in members)]


def bgzf_file(members, **framing):
    """members: [(payload, text)] -> a BGZF file ending in the EOF member"""
    return b"".join(bgzf_member(p, t, **framing) for p, t in members) + BGZF_EOF


# ---------------------------------------------------------------------------------------------------------------------
# valid streams: name -> [(payload, expected text)], one per member

def _rand(n, seed):
    return bytes(random.Random(seed).getrandbits(8) for _ in range(n))


def _repeat_at(cl, sym, pos):
    """the code-length symbols of `cl` that are repeats `sym` starting at or before `pos` and ending after it"""
    i, hits = 0, []
    for s, e in cl:
        n = 1 if s < 16 else 3 + e if s < 18 else 11 + e
        if s == sym and i <= pos < i + n:
            hits.append(i)
        i += n
    return hits


def s_repeats_across_boundary():
    """16 / 17 / 18 spanning HLIT -> HDIST, and a 16 whose previous length is the last literal/length length"""
    out = []
    # a: literal/length 97:2 98:2 256:2 258:2 (HLIT 259), distance 0..3 all 2 bits: the 16 starts at the first
    #    distance length and repeats lit[258]
    lit = [0] * 259
    lit[97] = lit[98] = lit[256] = lit[258] = 2
    toks = [97, 98, 97, 98, match(4, 2), match(4, 4), match(4, 1), 98, match(4, 3)]
    out.append(("16_after_last_litlen", lit, [2, 2, 2, 2], toks, 16, 259, 259))
    # b: literal/length 97:1 256:2 257:3 258:3, eight 3-bit distance codes: a run of ten 3s from 257 on
    lit = [0] * 259
    lit[97], lit[256], lit[257], lit[258] = 1, 2, 3, 3
    toks = [97] * 8 + [match(3, d) for d in range(1, 9)] + [match(4, 8), 97]
    out.append(("16_spans_boundary", lit, [3] * 8, toks, 16, 259, None))
    # c: literal-only code, HLIT 270: 13 zero literal/length lengths and 20 zero distance lengths in one 18
    lit = [0] * 270
    lit[65], lit[66], lit[256] = 2, 2, 1
    out.append(("18_spans_boundary", lit, [0] * 20 + [1, 1], [65, 66, 65], 18, 270, None))
    # d: HLIT 263, five zero lengths 258..262 and two zero distance lengths in one 17
    lit = [0] * 263
    lit[65], lit[66], lit[256], lit[257] = 2, 2, 2, 2
    out.append(("17_spans_boundary", lit, [0, 0, 1, 1], [65, 66, 65, match(3, 3)], 17, 263, None))
    res = []
    for name, lit, dist, toks, sym, nlit, start in out:
        assert kraft(lit) == 1 and kraft(dist) in (0, 1)
        cl = rle_lengths(lit + dist)
        assert expand_cl(cl) == lit + dist
        hits = _repeat_at(cl, sym, nlit)
        assert hits and (hits[0] == start if start is not None else hits[0] < nlit), (name, cl)
        res.append((name, dyn_stream(toks, litlens=lit, distlens=dist)))
    return res


def s_code_lengths_1_to_15():
    """literal/length and distance codes of every length 1..15 (two of 15), each code used: the 10-bit and 8-bit
    codes sit exactly at the primary-table widths, longer ones take decode_slow"""
    rng = random.Random(7)
    lit_syms = [256, 257, 258, 265, 270, 280, 284, 285] + rng.sample(range(256), 8)
    rng.shuffle(lit_syms)
    lit = [0] * 286
    for L, s in zip(list(range(1, 16)) + [15], lit_syms):
        lit[s] = L
    dist_syms = list(range(30))
    rng.shuffle(dist_syms)
    dist = [0] * 30
    for L, s in zip(list(range(1, 16)) + [15], dist_syms[:16]):
        dist[s] = L
    assert kraft(lit) == 1 and kraft(dist) == 1
    lits = [s for s in lit_syms if s < 256]
    lens = [s for s in lit_syms if s > 256]
    dsyms = dist_syms[:16]
    toks = [lits[i % len(lits)] for i in range(40000)]     # history for every distance symbol used
    for i in range(max(len(lens), len(dsyms)) * 2):
        ls, ds = lens[i % len(lens)], dsyms[i % len(dsyms)]
        le = (i // len(lens)) % 2 * ((1 << LEXTRA[ls - 257]) - 1) if ls < 285 else 0
        de = (i // len(dsyms)) % 2 * ((1 << DEXTRA[ds]) - 1)
        toks.append(("m", ls, le, ds, de))
        toks.append(lits[i % len(lits)])
    return [("lit_and_dist_1_to_15", dyn_stream(toks, litlens=lit, distlens=dist))]


def s_hclen():
    toks = [1, 2, 3, 250, 251]
    # HCLEN 19: every code-length code length sent, the trailing ones zero
    a = dyn_stream(toks, hclen=19)
    # HCLEN 5 (16 17 18 0 8): 255 literals + 256 all 8 bits, no distance code
    lit = [8] * 256 + [8]
    lit[0] = 0
    b = dyn_stream(list(range(1, 256)), litlens=lit, distlens=[0])
    return [("hclen_19", a), ("hclen_5_all_8_bit", b)]


def s_small_codes():
    toks = [120, 121, 120]
    # HLIT 257, HDIST 1, distance length 0: a literal-only block
    a = dyn_stream(toks, litlens=lit_lens_for(toks, n=257), distlens=[0])
    # a single distance code of one bit, used
    toks2 = [120, 121, 122, match(3, 3), match(10, 3)]
    b = dyn_stream(toks2, distlens=[0, 0, 1])
    # a literal/length code with a single 1-bit code (the end of block): an empty block, then a final one
    lit = [0] * 257
    lit[256] = 1
    c = Stream().dynamic([], lit, [0]).fixed([65, 66], last=True)
    # HLIT 286 / HDIST 30: every literal/length and distance symbol has a code
    toks4 = list(range(256)) + [match(258, 256), match(3, 1), 7]
    d = dyn_stream(toks4, litlens=complete_lengths(list(range(286)), 286), distlens=complete_lengths(list(range(30)), 30))
    return [("hlit257_hdist1_len0", a), ("one_1bit_distance_code", b), ("single_1bit_litlen_code", c), ("hlit286_hdist30", d)]


def _mixed(bit_offset):
    """dynamic -> stored (its header at `bit_offset` in its byte) -> fixed -> empty stored -> dynamic final"""
    lit = [0] * 257
    lit[120], lit[256], lit[121] = 1, 2, 2
    for k in range(8):
        s = Stream()
        s.dynamic([121] + [120] * k, lit, [0])
        if s.w.n == bit_offset:
            break
    else:
        raise AssertionError("no padding gives bit offset %d" % bit_offset)
    s.stored(_rand(300 + bit_offset, bit_offset))
    s.fixed([65, 66, match(40, 302), match(258, 1), 0, 255, 143, 144])
    s.stored(b"")
    toks = [match(30, 150), 67, 68]
    s.dynamic(toks, lit_lens_for(toks), dist_lens_for(toks), last=True)
    return s


def s_mixed_blocks():
    return [("mixed_stored_at_bit_%d" % b, _mixed(b)) for b in range(8)]


def s_fixed_every_symbol():
    """after 32 KiB of stored history: every length symbol 257..285 and every distance symbol 0..29, each at its
    smallest and largest extra bits (284 + 31 = 258 included; 29 + 8191 = distance 32,768)"""
    hist = _rand(32768, 11)
    toks = []
    ls = [(s, e) for s in range(257, 286) for e in sorted({0, (1 << LEXTRA[s - 257]) - 1})]
    ds = [(s, e) for s in range(30) for e in sorted({0, (1 << DEXTRA[s]) - 1})]
    for i in range(max(len(ls), len(ds))):
        (l, le), (d, de) = ls[i % len(ls)], ds[i % len(ds)]
        toks.append(("m", l, le, d, de))
    assert ("m", 284, 31) == toks[ls.index((284, 31))][:3]
    s = Stream().stored(hist).fixed(toks, last=True)
    assert len(s.expected) <= 65536
    return [("fixed_every_symbol", s)]


RUN_LENGTHS = (3, 31, 32, 33, 64, 258)


def s_runs():
    """for every period d in 1..40: d distinct bytes, then runs of length 3, d, d+1, 31, 32, 33, 64 and 258 at
    distance d back to back; several members, of odd sizes"""
    members, cur, rng = [], None, random.Random(3)
    for d in range(1, 41):
        if cur is None or len(cur.expected) > 20000:
            if cur is not None:
                cur.fixed([], last=True)
                members.append(cur)
            cur = Stream()
        pattern = rng.sample(range(256), d)
        lengths = sorted({L for L in RUN_LENGTHS + (d, d + 1) if L >= 3})
        cur.fixed(pattern + [match(L, d) for L in lengths])
    cur.fixed([7], last=True)
    members.append(cur)
    return [("runs_of_period_1_to_40", *members)]


def s_largest_members():
    a = Stream().stored(_rand(65505, 5), last=True)           # 18 + 5 + 65,505 + 8 = 65,536 bytes: BSIZE's limit
    toks = list(_rand(300, 6)) + [match(258, 300)] * 252 + [match(220, 33)]
    b = dyn_stream(toks)
    assert len(b.expected) == 65536
    return [("largest_stored_block", a), ("isize_65536", b)]


def valid_streams():
    out = []
    for f in (s_repeats_across_boundary, s_code_lengths_1_to_15, s_hclen, s_small_codes, s_mixed_blocks,
              s_fixed_every_symbol, s_runs, s_largest_members):
        for name, *streams in f():
            out.append((name, [(s.getvalue(), bytes(s.expected)) for s in streams]))
    return out


VALID = valid_streams()

# ---------------------------------------------------------------------------------------------------------------------
# invalid streams: name -> (payload, text the member claims), each refused by zlib and by the kernel


def _block_header(w, kind, last=True):
    w.put(int(last), 1)
    w.put(kind, 2)


def i_dynamic(litlens, distlens, toks, **hdr):
    w = BitWriter()
    _block_header(w, 2)
    lc, dc = dynamic_header(w, litlens, distlens, **hdr)
    put_symbols(w, lc, dc, toks)
    return w.getvalue()


def invalid_streams():
    """name -> (payload, the text a decoder that skipped the broken check would give, zlib's message).  The member
    claims that text (CRC, ISIZE), so only the check under test can catch the stream."""
    toks = [65, 66, 67]
    good_lit = lit_lens_for(toks)                           # 65 66 67 256: four 2-bit codes
    fixed_lc, fixed_dc = canonical(FIXED_LIT), canonical(FIXED_DIST)
    out = {}
    over = list(good_lit)
    over[68] = 2                                            # a fifth 2-bit code
    out["oversubscribed_litlen"] = (i_dynamic(over, [0], toks + [256]), b"ABC", "invalid literal/lengths set")
    inc = list(good_lit)
    inc[256] = 3                                            # the end-of-block code one bit longer: a hole in the code
    out["incomplete_litlen"] = (i_dynamic(inc, [0], toks + [256]), b"ABC", "invalid literal/lengths set")
    dtoks = [65, 66, match(3, 2)]
    out["incomplete_dist"] = (i_dynamic(lit_lens_for(dtoks), [0, 2, 2, 2], dtoks + [256]), b"ABABA",
                              "invalid distances set")     # three 2-bit distance codes
    cl = rle_lengths(good_lit + [0])
    used = sorted({s for s, _ in cl})
    cll = complete_lengths(used, 19)
    cll[used[-1]] += 1                                      # the code-length code's last code one bit longer
    assert kraft(cll) < 1
    out["incomplete_code_length_code"] = (i_dynamic(good_lit, [0], toks + [256], cl_syms=cl, cllens=cll), b"ABC",
                                          "invalid code lengths set")
    cl1 = [0] * 19
    cl1[0] = 1                                              # a code-length code of one 1-bit code (never allowed)
    out["code_length_code_single_1bit"] = (i_dynamic([0] * 257, [0], [], cl_syms=[(0, 0)] * 258, cllens=cl1), b"",
                                           "invalid code lengths set")
    # HLIT 287 / HDIST 31: the 5-bit fields at their (invalid) maxima
    out["hlit_287"] = (i_dynamic(complete_lengths([65, 256], 288), [0], [65, 256]), b"A",
                       "too many length or distance symbols")
    out["hdist_31"] = (i_dynamic(good_lit, complete_lengths([0, 1], 32), toks + [256]), b"ABC",
                       "too many length or distance symbols")
    # 16 as the first code length; a repeat past HLIT + HDIST
    out["repeat_16_first"] = (i_dynamic(good_lit, [0], toks + [256], cl_syms=[(16, 0)] + rle_lengths(good_lit + [0])),
                              b"ABC", "invalid bit length repeat")
    out["repeat_past_end"] = (i_dynamic(good_lit, [0], toks + [256], cl_syms=rle_lengths(good_lit) + [(17, 5)]),
                              b"ABC", "invalid bit length repeat")
    # HCLEN 4: only 16 17 18 0 have code lengths, so no length can be non-zero and there is no end-of-block code
    out["hclen_4_no_end_of_block"] = (i_dynamic([0] * 257, [0], [], cl_syms=[(18, 127), (18, 108), (0, 0)], hclen=4),
                                      b"", "missing end-of-block")
    eob0 = complete_lengths([65, 66, 67, 257], 258)
    out["end_of_block_length_0"] = (i_dynamic(eob0, [0], toks), b"ABC", "missing end-of-block")
    # fixed blocks: literal/length symbols 286 / 287, distance symbols 30 / 31
    for bad in (286, 287):
        w = BitWriter()
        _block_header(w, 1)
        put_symbols(w, fixed_lc, fixed_dc, toks + [bad, 256])
        out["fixed_litlen_%d" % bad] = (w.getvalue(), b"ABC", "invalid literal/length code")
    for bad in (30, 31):
        w = BitWriter()
        _block_header(w, 1)
        put_symbols(w, fixed_lc, fixed_dc, toks + [("m", 257, 0, bad, 0), 256])
        out["fixed_dist_%d" % bad] = (w.getvalue(), b"ABCABC", "invalid distance code")
    # a distance one byte before the start of the member (the previous member's text is there in memory)
    w = BitWriter()
    _block_header(w, 1)
    put_symbols(w, fixed_lc, fixed_dc, toks + [match(3, 4), 256])
    out["distance_before_member"] = (w.getvalue(), b"ABC9AB", "invalid distance too far back")
    # stored: LEN / NLEN mismatch; more data announced than the payload holds
    out["stored_nlen_mismatch"] = (Stream().stored(b"abcdef", last=True, nlen=0x1234).getvalue(), b"abcdef",
                                   "invalid stored block lengths")
    data = _rand(100, 1)
    out["stored_past_payload"] = (Stream().stored(data, last=True).getvalue()[:60], data, "truncated")
    w = BitWriter()
    _block_header(w, 3)
    w.put(0, 16)
    out["block_type_3"] = (w.getvalue(), b"", "invalid block type")
    data = _rand(2000, 2)
    full = dyn_stream(list(data)).getvalue()
    out["truncated_mid_symbol"] = (full[:len(full) // 2], data, "truncated")
    return out


INVALID = invalid_streams()


def _valid_ids():
    return [n for n, _ in VALID]


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the writer against stock zlib


@pytest.mark.parametrize("name,members", VALID, ids=_valid_ids())
def test_writer_valid_stream_is_zlib_clean(name, members):
    for payload, text in members:
        d = zlib.decompressobj(-15)
        assert d.decompress(payload) + d.flush() == text
        assert d.eof and d.unused_data == b""
        assert len(text) <= 65536
    assert gzip.decompress(bgzf_file(members)) == b"".join(t for _, t in members)
    for fr in framings_for(members):
        f = bgzf_file(members, **fr)
        assert gzip.decompress(f) == b"".join(t for _, t in members)


@pytest.mark.parametrize("name", sorted(INVALID))
def test_writer_invalid_stream_is_refused_by_zlib(name):
    payload, _, reason = INVALID[name]
    with pytest.raises(zlib.error, match=reason):
        zlib.decompress(payload, -15)


def test_writer_size_limits():
    largest = dict(VALID)["largest_stored_block"]
    assert len(bgzf_file(largest)) - len(BGZF_EOF) == 65536
    assert len(dict(VALID)["isize_65536"][0][1]) == 65536


def test_writer_isize_mismatch_is_refused_by_gzip():
    payload, text = dict(VALID)["hclen_19"][0]
    for isize in (len(text) - 1, len(text) + 1):
        with pytest.raises(gzip.BadGzipFile):
            gzip.decompress(bgzf_member(payload, text, isize=isize) + BGZF_EOF)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: kernel 0 against zlib


@pytest.fixture(scope="module")
def capi(built):
    from haplohyped_varawareml_b200 import capi as c
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("name,members", VALID, ids=_valid_ids())
def test_kernel_inflates_stream(capi, name, members):
    want = b"".join(t for _, t in members)
    frs = framings_for(members)
    assert len(frs) == (1 if name == "largest_stored_block" else len(FRAMINGS))
    for fr in frs:
        assert capi.bgzf_inflate(bgzf_file(members, **fr)) == want, fr


@pytest.mark.gpu
def test_kernel_inflates_all_streams_in_one_file(capi):
    """every valid member in one file, behind a 1-byte-text member: members at many offsets of one launch"""
    members = [(zlib.compress(b"!", 9)[2:-4], b"!")] + [m for n, ms in VALID for m in ms if n != "largest_stored_block"]
    assert capi.bgzf_inflate(bgzf_file(members, extra_after=b"\x01")) == b"".join(t for _, t in members)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(INVALID))
def test_kernel_refuses_invalid_stream(capi, name):
    payload, claimed, _ = INVALID[name]
    lead = (zlib.compress(b"0123456789", 9)[2:-4], b"0123456789")    # text in memory just before the bad member
    if not claimed:
        claimed = b"?"                                                 # an ISIZE of 0 would make it an empty member
    with pytest.raises(capi.HaploError):
        capi.bgzf_inflate(bgzf_file([lead, (payload, claimed)]))


@pytest.mark.gpu
@pytest.mark.parametrize("delta", [-1, 1])
def test_kernel_refuses_isize_mismatch(capi, delta):
    payload, text = dict(VALID)["mixed_stored_at_bit_3"][0]
    with pytest.raises(capi.HaploError):
        capi.bgzf_inflate(bgzf_member(payload, text, isize=len(text) + delta) + BGZF_EOF)
