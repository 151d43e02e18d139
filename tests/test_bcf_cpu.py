"""The BCF writer the GPU tests use (tests/bcf_writer.py): byte for byte against a hand-assembled BCF 2.2 file, and the
header dictionary rules (VCF v4.3 specification, section 6.3)."""
import struct

import bcf_writer

HEADER = (
    "##fileformat=VCFv4.2\n"
    '##FILTER=<ID=PASS,Description="All filters passed">\n'
    "##contig=<ID=chr22>\n"
    '##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">\n'
    "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tA\tB\n"
)
TEXT = (HEADER +
        "chr22\t100\trs1\tA\tG\t50\tPASS\t.\tGT\t0|1\t1/1\n"
        "chr22\t200\t.\tC\tT\t.\tPASS\t.\tGT\t0\t./.\n"
        "chr22\t300\t.\tG\tA,C\t.\t.\t.\tGT\t1|2\t0|0\n").encode()


def _golden() -> bytes:
    # header text as htslib writes it into a BCF: IDX= on the dictionary lines, NUL-terminated
    text = (HEADER.replace("All filters passed\">", "All filters passed\",IDX=0>")
                  .replace("##contig=<ID=chr22>", "##contig=<ID=chr22,IDX=0>")
                  .replace("Description=\"Genotype\">", "Description=\"Genotype\",IDX=1>")).encode() + b"\0"
    out = b"BCF\x02\x02"                                  # magic: "BCF", major 2, minor 2
    out += struct.pack("<I", len(text)) + text              # uint32 l_text, header text
    recs = [
        # CHROM 0 (chr22), POS 99 (0-based), rlen 1, QUAL 50.0
        (struct.pack("<iiif", 0, 99, 1, 50.0)
         + struct.pack("<II", 2 << 16 | 0, 1 << 24 | 2)   # n_allele 2 << 16 | n_info 0, n_fmt 1 << 24 | n_sample 2
         + b"\x37rs1"                                      # ID: typed string, count 3, type 7 (char)
         + b"\x17A" + b"\x17G"                             # alleles: REF "A", ALT "G"
         + b"\x11\x00",                                    # FILTER: one int8, PASS = 0; no INFO pairs
         b"\x11\x01"                                       # FORMAT key: typed int8 1 (GT)
         + b"\x21"                                         # values: count 2, type 1 (int8)
         + bytes([2, 5, 4, 4])),                           # A 0|1 = (0+1)<<1, (1+1)<<1|1; B 1/1 = 4, 4
        (struct.pack("<iiiI", 0, 199, 1, 0x7F800001)       # QUAL "." = float missing 0x7F800001
         + struct.pack("<II", 2 << 16, 1 << 24 | 2)
         + b"\x07"                                         # ID ".": typed string of count 0
         + b"\x17C" + b"\x17T" + b"\x11\x00",
         b"\x11\x01\x21"
         + bytes([2, 0x81, 0, 0])),                        # A haploid 0, padded with int8 vector_end 0x81; B ./. = 0, 0
        (struct.pack("<iiiI", 0, 299, 1, 0x7F800001)
         + struct.pack("<II", 3 << 16, 1 << 24 | 2)        # three alleles
         + b"\x07" + b"\x17G" + b"\x17A" + b"\x17C"
         + b"\x00",                                        # FILTER ".": typed vector of count 0, type 0
         b"\x11\x01\x21"
         + bytes([4, 7, 2, 3])),                           # A 1|2 = 4, (2+1)<<1|1; B 0|0 = 2, 3
    ]
    for shared, indiv in recs:
        out += struct.pack("<II", len(shared), len(indiv)) + shared + indiv   # l_shared, l_indiv
    return out


def test_writer_reproduces_the_hand_assembled_file():
    assert bcf_writer.vcf_to_bcf(TEXT) == _golden()


def test_writer_types_and_padding():
    b16 = bcf_writer.vcf_to_bcf(TEXT, gt_type=bcf_writer.INT16)
    assert b"\x22" + struct.pack("<4h", 2, 5, 4, 4) in b16
    assert b"\x22" + struct.pack("<4h", 2, -32767, 0, 0) in b16      # int16 vector_end
    big = TEXT.replace(b"\t1|2\t", b"\t1|200\t")
    assert b"\x22" + struct.pack("<4h", 4, 403, 2, 3) in bcf_writer.vcf_to_bcf(big)   # 403 > 127: int16


def test_dictionaries_without_idx():
    lines = ['##FILTER=<ID=PASS,Description="x">', '##INFO=<ID=DP,Number=1,Type=Integer,Description="a, b">',
             '##contig=<ID=chr2>', '##FORMAT=<ID=GT,Number=1,Type=String,Description="g">',
             '##FORMAT=<ID=DP,Number=1,Type=Integer,Description="d">', '##FILTER=<ID=q10,Description="q">',
             '##contig=<ID=chr1>']
    strs, contigs = bcf_writer.dictionaries(lines)
    assert strs == {"PASS": 0, "DP": 1, "GT": 2, "q10": 3}           # a shared ID (INFO and FORMAT DP) has one index
    assert contigs == ["chr2", "chr1"]
    strs, _ = bcf_writer.dictionaries(lines[1:])                     # PASS is 0 whether declared or not
    assert strs["PASS"] == 0 and strs["GT"] == 2


def test_dictionaries_with_idx():
    lines = ['##INFO=<ID=DP,Number=1,Type=Integer,Description="d",IDX=7>',
             '##FORMAT=<ID=GT,Number=1,Type=String,Description="g",IDX=3>',
             '##contig=<ID=chrB,IDX=1>', '##contig=<ID=chrA,IDX=0>']
    strs, contigs = bcf_writer.dictionaries(lines)
    assert strs == {"PASS": 0, "DP": 7, "GT": 3}
    assert contigs == ["chrA", "chrB"]
    head = bcf_writer.vcf_to_bcf(TEXT, idx=False)
    assert b"IDX=" not in head and bcf_writer.vcf_to_bcf(TEXT).count(b"IDX=") == 3
