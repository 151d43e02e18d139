"""The pure-Python tabix / CSI restatement (tests/index_writer.py): the binning scheme against the specs' worked values,
writer -> reader round trips, and the region query against a brute-force overlap test."""
import random

import pytest

import bcf_writer
import index_writer as iw
import synth


def test_reg2bin_spec_values():
    # SAMv1 5.3: level 5 bins cover 16 kb and start at 4681, level 4 at 585, level 3 at 73, 2 at 9, 1 at 1, 0 is bin 0
    assert iw.reg2bin(0, 1) == 4681
    assert iw.reg2bin(0, 1 << 14) == 4681
    assert iw.reg2bin(1 << 14, (1 << 14) + 1) == 4682
    assert iw.reg2bin(0, (1 << 14) + 1) == 585
    assert iw.reg2bin((1 << 17) - 1, (1 << 17) + 1) == 73
    assert iw.reg2bin(0, 1 << 26) == 1
    assert iw.reg2bin(0, (1 << 26) + 1) == 0
    assert iw.reg2bin(0, 1 << 29) == 0
    # CSI with min_shift 14 and depth 6: one more level on top
    assert iw.reg2bin(0, 1, 14, 6) == iw.bin_first(6)
    assert iw.reg2bin((1 << 30) + 5, (1 << 30) + 6, 14, 6) == iw.bin_first(6) + (((1 << 30) + 5) >> 14)


def test_reg2bins_spec_values():
    assert iw.reg2bins(0, 1) == [0, 1, 9, 73, 585, 4681]
    assert iw.reg2bins(0, 1 << 29) [:3] == [0, 1, 2]
    assert len(iw.reg2bins(0, 1 << 29)) == sum(8 ** k for k in range(6))
    assert iw.reg2bins(5, 5) == []
    for _ in range(200):
        rng = random.Random(_)
        beg = rng.randrange(1 << 28)
        end = beg + rng.randrange(1, 1 << 20)
        bins = set(iw.reg2bins(beg, end))
        assert iw.reg2bin(beg, end) in bins
        for x in (beg, end - 1, (beg + end) // 2):
            assert iw.reg2bin(x, x + 1) in bins


def _vcf(block, fmt="GT", info_end=True, first_pos=0):
    text = iw.multi_contig_vcf(["chr1", "chr2", "chrX"], 700, 5, seed=3, fmt=fmt, info_end=info_end, first_pos=first_pos)
    return text, synth.bgzf_compress(text, block=block)


@pytest.mark.parametrize("fmt", ["tbi", "csi"])
@pytest.mark.parametrize("block", [300, 0xff00])
def test_round_trip(fmt, block):
    text, bgzf = _vcf(block)
    raw = iw.index_vcf(text, bgzf, fmt)
    idx = iw.read(iw.write(raw))
    assert idx["fmt"] == (b"TBI\1" if fmt == "tbi" else b"CSI\1")
    assert idx["names"] == ["chr1", "chr2", "chrX"]
    assert (idx["min_shift"], idx["depth"]) == ((14, 5) if fmt == "tbi" else (14, 6))
    assert iw.serialise(idx["refs"], fmt, idx["min_shift"], idx["depth"], idx["names"]) == raw
    meta = iw.bin_first(idx["depth"] + 1)
    assert [bins[meta][1][1][0] for bins, _ in idx["refs"]] == [700, 700, 700]      # n_mapped per sequence


def test_round_trip_bcf():
    text, _ = _vcf(0xff00, info_end=False)
    raw = bcf_writer.vcf_to_bcf(text)
    bgzf = synth.bgzf_compress(raw, block=500)
    idx = iw.read(iw.write(iw.index_bcf(raw, bgzf)))
    assert idx["fmt"] == b"CSI\1" and idx["names"] is None and idx["depth"] == 6
    assert sum(1 for bins, _ in idx["refs"] if bins) == 3


def _covered(chunks, u, v):
    return any(a <= u and v <= b for a, b in chunks)


@pytest.mark.parametrize("fmt", ["tbi", "csi"])
def test_query_against_brute_force(fmt):
    text, bgzf = _vcf(300)
    vo = iw.VirtualOffsets(iw.bgzf_members(bgzf))
    names, _, recs = iw.vcf_records(text, vo)
    idx = iw.read(iw.write(iw.index_vcf(text, bgzf, fmt)))
    rng = random.Random(11)
    lo, hi = min(r[1] for r in recs), max(r[2] for r in recs)
    for _ in range(300):
        tid = rng.randrange(len(names) + 1)
        beg = rng.randrange(lo - 1000, hi + 1000)
        end = beg + rng.choice([1, 10, 500, 20_000, 300_000])
        chunks = iw.query(idx, tid, beg, end)
        assert chunks == sorted(chunks)
        for t, b, e, u, v in recs:
            if t == tid and b < end and e > beg:
                assert _covered(chunks, u, v), (tid, beg, end, b, e)
    # a small region reads far less than the file
    ch = iw.query(idx, 1, recs[900][1], recs[900][1] + 1)
    assert ch and (ch[-1][1] >> 16) - (ch[0][0] >> 16) < len(bgzf) // 10


def test_high_positions_need_csi():
    text, bgzf = _vcf(0xff00, info_end=False, first_pos=1 << 29)
    with pytest.raises(ValueError):
        iw.index_vcf(text, bgzf, "tbi")
    idx = iw.read(iw.write(iw.index_vcf(text, bgzf, "csi")))
    vo = iw.VirtualOffsets(iw.bgzf_members(bgzf))
    _, _, recs = iw.vcf_records(text, vo)
    t, b, e, u, v = recs[1000]
    assert _covered(iw.query(idx, t, b, e), u, v)


def test_writer_refuses_what_tabix_refuses():
    text, bgzf = _vcf(0xff00, info_end=False)
    lines = text.split(b"\n")
    body = [x for x in lines if x and not x.startswith(b"#")]
    head = [x for x in lines if x.startswith(b"#")]
    swapped = b"\n".join(head + [body[5], body[4]] + body[6:]) + b"\n"
    with pytest.raises(ValueError, match="unsorted"):
        iw.index_vcf(swapped, synth.bgzf_compress(swapped), "tbi")
    split = b"\n".join(head + body[:10] + body[800:810] + body[10:20]) + b"\n"
    with pytest.raises(ValueError, match="not continuous"):
        iw.index_vcf(split, synth.bgzf_compress(split), "tbi")
