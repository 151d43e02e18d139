"""GPU parity tests: the CUDA path (through the C ABI / the pybind11 `parse_vcf` module) against
the CPU oracle on the same inputs.  Bit-exact: all arithmetic on this path is integer/byte."""
import json
import os
import sys
import tempfile

import numpy as np
import pytest

import oracle
import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def capi(built):
    from haplohyped_varawareml_b200 import capi as c
    return c


@pytest.fixture(scope="module")
def parse_vcf(built):
    sys.path.insert(0, os.path.join(ROOT, "haplohyped-varawareml_b200"))
    import parse_vcf as m
    return m


def _check_matrix(capi, text, n_samples, region, tokenizer=0, end_is_int=False):
    ora = oracle.parse_text(text, "*", region)
    p = capi.Parse.from_host(synth.body_of(text), n_samples, region=region, tokenizer=tokenizer, end_is_int=end_is_int)
    info = p.info
    assert info.n_records == ora["n"]
    start, stop, ref, alt = p.sites()
    assert np.array_equal(start, ora["start"]) and np.array_equal(stop, ora["stop"])
    assert np.array_equal(ref, ora["ref"]) and np.array_equal(alt, ora["alt"])
    assert p.chrom_column() == ora["chrom"]
    g0, g1 = p.matrix()
    assert np.array_equal(g0, ora["gt0"]), "phase1 plane differs"
    assert np.array_equal(g1, ora["gt1"]), "phase2 plane differs"
    for s in (0, n_samples // 2, n_samples - 1):
        a0, a1 = p.sample(s)
        assert np.array_equal(a0, ora["gt0"][s]) and np.array_equal(a1, ora["gt1"][s])
    pl, bg = p.sample_errors()
    assert pl.sum() == 0 and bg.sum() == 0
    return p, info


def test_fixture_through_pybind_module(parse_vcf, golden_dir):
    """config 1: the reference's own fixture, through the reference's own API names."""
    gold = json.load(open(os.path.join(golden_dir, "fixture_load_vcf.json")))
    vcf = os.path.join(golden_dir, "chr22.filtered.vcf.gz")
    loader = parse_vcf.VCFLoader()
    for s in gold["samples"]:
        exp = [tuple(r) for r in gold["load_vcf"][s]]
        assert loader.load_vcf(vcf, s, "chr22") == exp               # class method (parse_vcf.cpp:120)
        assert parse_vcf.load_vcf(vcf, s, "chr22") == exp            # module-level (vcf_to_h5.py:101)
        assert loader.load_vcf(in_vcf=vcf, sample=s, chrom="chr22") == oracle.load_vcf(vcf, s, "chr22")
    sites = loader.load_vcf_without_sample(vcf, "chr22")
    assert sites == [tuple(r[:5]) for r in gold["load_vcf"][gold["samples"][0]]]
    assert loader.load_vcf(vcf, gold["samples"][0], "chr1") == []
    assert len(loader.load_vcf(vcf, gold["samples"][0])) == 1000    # chrom defaults to ""
    cols = loader.load_vcf_columns(vcf, gold["samples"][1], "chr22")
    exp = gold["load_vcf"][gold["samples"][1]]
    assert list(cols["phase1"]) == [r[5] for r in exp] and list(cols["start"]) == [r[1] for r in exp]


def test_errors_match_reference_contract(parse_vcf, golden_dir):
    vcf = os.path.join(golden_dir, "chr22.filtered.vcf.gz")
    with pytest.raises(RuntimeError, match="Error parsing VCF file: the 1-th sample are not in the VCF"):
        parse_vcf.load_vcf(vcf, "nobody", "chr22")
    with pytest.raises(RuntimeError, match="Error parsing VCF file"):
        parse_vcf.load_vcf("/nonexistent/file.vcf.gz", "x", "chr22")
    S = ["a", "b"]
    bad = (synth.header(S) + "chr22\t100\t.\tA\tC\t.\t.\t.\tGT\t0\t0|1\n").encode()
    with tempfile.NamedTemporaryFile(suffix=".vcf", delete=False) as f:
        f.write(bad)
    try:
        with pytest.raises(RuntimeError, match="ploidy"):
            parse_vcf.load_vcf(f.name, "a", "chr22")                  # reference: assert -> SIGABRT
        assert parse_vcf.load_vcf(f.name, "b", "chr22") == [("chr22", 99, 100, "A", "C", 0, 1)]
    finally:
        os.unlink(f.name)


@pytest.mark.parametrize("tokenizer", [0, 1, 2, 3])
@pytest.mark.parametrize("fmt,kinds,multidigit", [("GT", "phased", False), ("GT", "mixed", False),
                                                   ("GT", "mixed", True), ("GT:GQ:DP", "mixed", True),
                                                   ("DP:GT", "mixed", False)])
def test_random_vcf_matrix_parity(capi, fmt, kinds, multidigit, tokenizer):
    text, samples = synth.random_vcf(700, 301, seed=5, fmt=fmt, kinds=kinds, multidigit=multidigit)
    _check_matrix(capi, text, len(samples), "chr22", tokenizer=tokenizer)
    _check_matrix(capi, text, len(samples), "", tokenizer=tokenizer)


@pytest.mark.parametrize("n_samples", [1, 3, 127, 128, 129, 1000])
def test_sample_count_edges(capi, n_samples):
    text, samples = synth.random_vcf(300, n_samples, seed=n_samples, fmt="GT", kinds="mixed")
    _check_matrix(capi, text, n_samples, "chr22")
    text, samples = synth.random_vcf(150, n_samples, seed=n_samples + 1, fmt="GT:GQ:DP", kinds="mixed")
    _check_matrix(capi, text, n_samples, "chr22")


def test_crlf_info_end_and_regions(capi):
    text, samples = synth.random_vcf(500, 40, seed=9, fmt="GT", kinds="mixed", crlf=True)
    _check_matrix(capi, text, len(samples), "chr22")
    text, samples = synth.random_vcf(500, 40, seed=10, fmt="GT", kinds="mixed", info_end=True)
    _check_matrix(capi, text, len(samples), "chr22", end_is_int=True)
    _check_matrix(capi, text, len(samples), "chr22:10020000-10060000", end_is_int=True)
    _check_matrix(capi, text, len(samples), "chr22_KI270731v1_random", end_is_int=True)
    p, info = _check_matrix(capi, text, len(samples), "chrNope", end_is_int=True)
    assert info.n_records == 0


def test_empty_and_tiny_inputs(capi):
    S = ["a", "b", "c"]
    one = (synth.header(S) + "chr22\t5\t.\tA\tC\t.\t.\t.\tGT\t0|1\t1|1\t./.\n").encode()
    _check_matrix(capi, one, 3, "chr22")
    p = capi.Parse.from_host(b"", 3, region="chr22")
    assert p.info.n_records == 0 and p.info.n_lines == 0
    # no trailing newline on the last record
    _check_matrix(capi, one[:-1], 3, "chr22")


def test_per_sample_errors(capi):
    S = ["a", "b", "c"]
    rows = ["chr22\t5\t.\tA\tC\t.\t.\t.\tGT\t0|1\t1\t0|1", "chr22\t6\t.\tA\tC\t.\t.\t.\tGT\t0|1\t0/1/1\tx|1",
            "chr22\t7\t.\tA\tC\t.\t.\t.\tGT\t1|1\t0|0\t0|1"]
    text = (synth.header(S) + "\n".join(rows) + "\n").encode()
    p = capi.Parse.from_host(synth.body_of(text), 3, region="chr22")
    pl, bg = p.sample_errors()
    assert list(pl) == [0, 2, 0] and list(bg) == [0, 0, 1]
    a0, a1 = p.sample(0)
    assert list(a0) == [0, 0, 1] and list(a1) == [1, 1, 1]
    ora = oracle.parse_text(text, "a", "chr22")
    assert np.array_equal(a0, ora["gt0"]) and np.array_equal(a1, ora["gt1"])
    with pytest.raises(RuntimeError):
        oracle.parse_text(text, "b", "chr22")


def test_synth_device_equals_host_and_parses(capi):
    import torch
    for mix in (0, 1):
        spec = capi.synth_spec(5000, 515, seed=42 + mix, mix=mix)
        host = capi.synth_host(spec)
        n = capi.lib().hb_synth_body_bytes(spec)
        assert n == len(host)
        buf = torch.zeros(n + 256, dtype=torch.uint8, device="cuda:0")
        capi.check(capi.lib().hb_synth_device(spec, buf.data_ptr(), n, 0, None))
        assert bytes(buf[:n].cpu().numpy().tobytes()) == host
        p = capi.Parse.from_device(buf.data_ptr(), n, spec.n_samples, region="chr22")
        ora = oracle.parse_text(capi.synth_header(spec) + host, "*", "chr22")
        g0, g1 = p.matrix()
        assert p.info.n_records == ora["n"] and p.info.n_nonuniform == 0
        assert np.array_equal(g0, ora["gt0"]) and np.array_equal(g1, ora["gt1"])
        p.rerun()                                   # steady-state path used by the bench
        h0, h1 = p.matrix()
        assert np.array_equal(h0, g0) and np.array_equal(h1, g1)


def test_many_tiles_lookback(capi):
    """> 2 x SM-count tokenizer tiles and > 1 site tile: exercises both decoupled look-backs."""
    spec = capi.synth_spec(40000, 257, seed=3)
    text = capi.synth_header(spec) + capi.synth_host(spec)
    assert len(text) > 40 * 1024 * 1024
    _check_matrix(capi, text, spec.n_samples, "chr22", tokenizer=1)
    _check_matrix(capi, text, spec.n_samples, "chr22", tokenizer=2)
    p, info = _check_matrix(capi, text, spec.n_samples, "chr22", tokenizer=0)       # auto -> head walker
    assert info.tokenizer_used == 3 and info.walker_fallbacks == 0 and info.n_lines == 40000


# ------------------------------------------------------------------------------------------------
# head walker (tokenizer 3): records located by jumping 4*S bytes from the 9th tab
# ------------------------------------------------------------------------------------------------
@pytest.fixture
def walker_lines(capi):
    """hb_set_walker_lines for one test (1-3 lines per walker put a walker boundary at every line)."""
    def set_lines(n):
        capi.lib().hb_set_walker_lines(int(n))
    yield set_lines
    capi.lib().hb_set_walker_lines(0)


@pytest.mark.parametrize("lines_per_walker", ["1", "3", "16", "20"])
@pytest.mark.parametrize("mix", [0, 1])
def test_walker_uniform_text(capi, walker_lines, lines_per_walker, mix):
    walker_lines(lines_per_walker)
    spec = capi.synth_spec(6000, 300, seed=17 + mix, mix=mix)
    text = capi.synth_header(spec) + capi.synth_host(spec)
    p, info = _check_matrix(capi, text, spec.n_samples, "chr22", tokenizer=0)
    assert info.tokenizer_used == 3 and info.walker_fallbacks == 0 and info.n_lines == 6000
    _check_matrix(capi, text, spec.n_samples, "chr22:10050000-10120000", tokenizer=3)
    p.rerun()
    assert p.info.tokenizer_used == 3 and p.info.n_records == info.n_records


def test_walker_odd_lines_stay_exact(capi, walker_lines):
    """Comment lines, empty lines, CRLF, wide records, other FORMATs and a missing final newline inside
    otherwise uniform text: the walker searches those newlines instead of jumping."""
    walker_lines(4)
    S = synth.sample_names(260)
    rng = np.random.default_rng(0)

    def rec(pos, gts=None, fmt="GT", ref="A", alt="C", eol="\n"):
        gts = gts if gts is not None else ["%d|%d" % (a, b) for a, b in rng.integers(0, 2, (260, 2))]
        return "\t".join(["chr22", str(pos), ".", ref, alt, ".", "PASS", ".", fmt] + gts) + eol

    lines = []
    for i in range(400):
        pos = 1000 + 10 * i
        if i == 5:
            lines.append("#late comment\twith\ttabs\n")
        if i == 9:
            lines.append("\n")
        if i % 37 == 3:
            lines.append(rec(pos, eol="\r\n"))
        elif i % 41 == 4:
            g = ["%d|%d" % (a, b) for a, b in rng.integers(0, 2, (260, 2))]
            g[17] = "10|1"
            lines.append(rec(pos, g))
        elif i % 43 == 5:
            lines.append(rec(pos, ["0|1:%d" % d for d in rng.integers(1, 99, 260)], fmt="GT:DP"))
        elif i % 47 == 6:
            lines.append(rec(pos, ref="AT"))                          # dropped: its span goes to the verify kernel
        else:
            lines.append(rec(pos))
    text = (synth.header(S) + "".join(lines)).encode()
    p, info = _check_matrix(capi, text, 260, "chr22", tokenizer=3)
    assert info.tokenizer_used == 3 and info.walker_fallbacks == 0
    assert info.n_lines == len(lines)
    _check_matrix(capi, text[:-1], 260, "chr22", tokenizer=3)        # no final newline


def test_walker_cannot_be_fooled_by_hidden_newlines(capi, walker_lines):
    """Two short records whose lengths add up so that (9th tab of the first) + 4*S lands exactly on the
    second one's newline: the jump is accepted by the walker and must be caught afterwards -- by the
    verify kernel when the merged record is dropped, by the GT decoder when it is kept."""
    walker_lines(2)
    n = 300
    S = synth.sample_names(n)
    rng = np.random.default_rng(1)

    def groups(k):
        return "".join("\t%d|%d" % (a, b) for a, b in rng.integers(0, 2, (k, 2)))

    def head(pos, ref, alt, rid="."):
        return "\t".join(["chr22", str(pos), rid, ref, alt, ".", "PASS", ".", "GT"])

    for ref, expect_error in (("AT", False), ("A", True)):
        lines = [head(100 + i, "A", "C") + groups(n) + "\n" for i in range(50)]
        h2 = head(7000, ref, "G")
        h2 = head(7000, ref, "G", "r" * (1 + (3 - len(h2)) % 4))       # make 4*n - 4*m - 1 - len(h2) a multiple of 4
        m = 100
        k2 = (4 * n - 4 * m - 1 - len(h2))
        assert k2 % 4 == 0 and k2 > 0, (k2, len(h2))
        pair = head(6000, ref, "G") + groups(m) + "\n" + h2 + groups(k2 // 4) + "\n"
        lines.insert(20, pair)
        lines += [head(9000 + i, "A", "C") + groups(n) + "\n" for i in range(50)]
        text = (synth.header(S) + "".join(lines)).encode()
        body = synth.body_of(text)
        if expect_error:
            for tok in (1, 3):
                with pytest.raises(capi.HaploError, match="Number of columns"):
                    capi.Parse.from_host(body, n, region="chr22", tokenizer=tok)
        else:
            p, info = _check_matrix(capi, text, n, "chr22", tokenizer=3)
            assert info.walker_fallbacks == 1 and info.tokenizer_used == 1 and info.n_lines == 102
            assert info.n_records == 100


@pytest.mark.parametrize("fmt,kinds,slab", [("GT", "phased", 3000), ("GT", "mixed", 20000), ("GT:GQ:DP", "mixed", 7000),
                                            ("GT", "mixed", 1 << 30)])
def test_stream_host_equals_oracle(capi, fmt, kinds, slab):
    """hb_parse_stream_host: slabs cut at line boundaries, two device slots, H2D / kernels / D2H overlapped --
    the concatenated result is the same matrix, whatever the slab size (here: many slabs, and one)."""
    text, samples = synth.random_vcf(1500, 41, seed=77, fmt=fmt, kinds=kinds)
    ora = oracle.parse_text(text, "*", "chr22")
    body = synth.body_of(text)
    r = capi.parse_stream_host(body, len(samples), capacity=1500, region="chr22", slab_bytes=slab)
    assert r["n"] == ora["n"] and r["n_slabs"] == (1 if slab >= len(body) else r["n_slabs"]) and r["n_slabs"] >= 1
    if slab < len(body):
        assert r["n_slabs"] >= len(body) // slab
    assert np.array_equal(r["gt0"], ora["gt0"]) and np.array_equal(r["gt1"], ora["gt1"])
    assert np.array_equal(r["start"], ora["start"]) and np.array_equal(r["stop"], ora["stop"])
    assert np.array_equal(r["ref"], ora["ref"]) and np.array_equal(r["alt"], ora["alt"])
    assert r["ploidy_err"].sum() == 0 and r["badgt_err"].sum() == 0
    with pytest.raises(capi.HaploError):                               # capacity is checked, not overrun
        capi.parse_stream_host(body, len(samples), capacity=ora["n"] - 1, region="chr22", slab_bytes=slab)


def test_stream_host_uniform_text_and_errors(capi):
    spec = capi.synth_spec(4000, 300, seed=3, mix=1)
    text = capi.synth_header(spec) + capi.synth_host(spec)
    ora = oracle.parse_text(text, "*", "chr22")
    body = synth.body_of(text)
    r = capi.parse_stream_host(body, 300, capacity=4000, region="chr22", slab_bytes=len(body) // 7)
    assert r["n"] == ora["n"] and r["n_slabs"] >= 7
    assert np.array_equal(r["gt0"], ora["gt0"]) and np.array_equal(r["gt1"], ora["gt1"]) and np.array_equal(r["start"], ora["start"])
    # a haploid call of one sample in a late slab is reported for that sample only
    S = ["a", "b", "c"]
    lines = [f"chr22\t{100 + i}\t.\tA\tC\t.\t.\t.\tGT\t0|1\t1|1\t0|0\n" for i in range(400)]
    lines[333] = "chr22\t433\t.\tA\tC\t.\t.\t.\tGT\t0|1\t1\t0|0\n"
    r = capi.parse_stream_host("".join(lines).encode(), 3, capacity=400, region="", slab_bytes=2000)
    assert r["n"] == 400 and list(r["ploidy_err"]) == [0, 1, 0] and r["n_slabs"] > 3
    # the same lines behind a header, in BGZF: streamed into host arrays, and into one resident parse
    gz = synth.bgzf_compress((synth.header(S) + "".join(lines)).encode(), block=1000)
    r = capi.parse_stream_bgzf_host(gz, capacity=400, region="", slab_bytes=2000)
    assert r["n"] == 400 and list(r["ploidy_err"]) == [0, 1, 0] and r["n_slabs"] > 3
    p, n_slabs = capi.Parse.from_vcf_bytes_streamed(gz, region="", slab_bytes=2000)
    assert p.info.n_records == 400 and n_slabs > 3
    pl, bg = p.sample_errors()
    assert list(pl) == [0, 1, 0] and list(bg) == [0, 0, 0]


def test_biobank_width_200k_samples(capi):
    """BASELINE configs[3] at reduced depth: 200,000 sample columns (a record is ~800 KB of text), multiallelic /
    indel sites dropped by the SNP filter, unphased and missing calls -- parse, then kernel 4 on a few samples."""
    S = 200_000
    spec = capi.synth_spec(48, S, seed=17, mix=1)
    text = capi.synth_header(spec) + capi.synth_host(spec)
    ora = oracle.parse_text(text, "*", "chr22")
    assert 0 < ora["n"] < 48
    for tok in (0, 1):                                   # head walker (auto) and plain newline tokenizer
        p = capi.Parse.from_host(synth.body_of(text), S, region="chr22", tokenizer=tok)
        assert p.info.n_records == ora["n"]
        g0, g1 = p.matrix()
        assert np.array_equal(g0, ora["gt0"]) and np.array_equal(g1, ora["gt1"])
        start, stop, ref, alt = p.sites()
        assert np.array_equal(start, ora["start"]) and np.array_equal(alt, ora["alt"])
    fr = p.compress(0)
    assert fr.info.n_samples == S and fr.info.n_chunks == 1
    cr = int(fr.info.chunk_records)
    for s in (0, 99_999, S - 1):
        rec = oracle.records_from_columns(ora["chrom"], ora["start"], ora["stop"], ora["ref"], ora["alt"], ora["gt0"][s], ora["gt1"][s])
        raw = rec.tobytes() + b"\0" * (cr * 35 - rec.nbytes)
        (f,) = fr.sample(s)
        assert oracle.blosc_chunk_decode(f, cr * 35).tobytes() == raw


def test_stream_slots_are_reused_and_safe_across_options_and_threads(capi):
    """The streaming entry points keep their device slots between calls (hb_api.cu, StreamSlots cache): same options ->
    reused; other options / other text shapes -> rebuilt; a concurrent call gets its own slots; hb_cache_clear frees them."""
    import threading
    t1, s1 = synth.random_vcf(900, 33, seed=5, fmt="GT", kinds="mixed")
    t2, s2 = synth.random_vcf(700, 57, seed=6, fmt="GT:GQ:DP", kinds="mixed")
    spec = capi.synth_spec(3000, 300, seed=8, mix=1)
    t3 = capi.synth_header(spec) + capi.synth_host(spec)
    cases = [(t1, len(s1)), (t2, len(s2)), (t3, 300), (t1, len(s1)), (t1, len(s1))]
    oras = {id(t): oracle.parse_text(t, "*", "chr22") for t, _ in cases}

    def check(text, ns, slab):
        ora = oras[id(text)]
        r = capi.parse_stream_host(synth.body_of(text), ns, capacity=ora["n"], region="chr22", slab_bytes=slab)
        assert r["n"] == ora["n"]
        assert np.array_equal(r["gt0"], ora["gt0"]) and np.array_equal(r["gt1"], ora["gt1"]) and np.array_equal(r["start"], ora["start"])

    for text, ns in cases:                       # same handle options twice in a row, then others, then back
        check(text, ns, 9000)
        check(text, ns, 50000)                   # larger slabs than the cached buffers were made for
    capi.lib().hb_cache_clear()
    errs = []

    def worker(text, ns):
        try:
            for _ in range(3):
                check(text, ns, 7000)
        except Exception as ex:                  # noqa: BLE001
            errs.append(ex)

    th = [threading.Thread(target=worker, args=c) for c in cases[:3] + cases[:1]]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errs, errs
    # the BGZF form, alternating inputs
    for text, ns in cases[:3] + cases[:1]:
        ora = oras[id(text)]
        for slab in (8000, 1 << 30):
            r = capi.parse_stream_bgzf_host(synth.bgzf_compress(text, block=2500), capacity=ora["n"], region="chr22", slab_bytes=slab)
            assert r["n"] == ora["n"] and np.array_equal(r["gt0"], ora["gt0"]) and np.array_equal(r["stop"], ora["stop"])
    capi.lib().hb_cache_clear()


def test_load_vcf_cache_follows_the_file_and_is_bounded(capi, parse_vcf, tmp_path):
    """The per-(file, region) cache behind load_vcf: a file rewritten at the same path is parsed again (size / mtime / inode
    are part of the key), hb_cache_set_limit bounds the HBM it pins (least recently used entries go), and an empty sample
    name is an error, not a crash."""
    import os, time
    S = synth.sample_names(4)
    def write(path, alt, n):
        body = "".join("chr22\t%d\t.\tA\t%s\t.\t.\t.\tGT\t0|1\t1|1\t0|0\t1|0\n" % (100 + 7 * i, alt) for i in range(n))
        with open(path, "w") as f:
            f.write(synth.header(S) + body)
    a = str(tmp_path / "a.vcf")
    write(a, "C", 50)
    first = parse_vcf.load_vcf(a, S[0], "chr22")
    assert len(first) == 50 and first[0][4] == "C"
    time.sleep(0.01)
    write(a, "G", 70)                                   # same path, new content
    again = parse_vcf.load_vcf(a, S[1], "chr22")
    assert len(again) == 70 and again[0][4] == "G" and again[0][5:] == (1, 1)
    # a limit of one byte: every finished entry but the newest is dropped; results stay correct
    capi.lib().hb_cache_set_limit(1)
    try:
        paths = []
        for k in range(4):
            pth = str(tmp_path / ("b%d.vcf" % k))
            write(pth, "ACGT"[k], 30 + k)
            paths.append(pth)
        for rnd in range(2):
            for k, pth in enumerate(paths):
                got = parse_vcf.load_vcf(pth, S[3], "chr22")
                assert len(got) == 30 + k and got[0][4] == "ACGT"[k] and got[0][5:] == (1, 0)
    finally:
        capi.lib().hb_cache_set_limit(0)
        capi.lib().hb_cache_clear()
    with pytest.raises(RuntimeError, match="Error parsing VCF file"):
        parse_vcf.load_vcf(a, "", "chr22")
    assert len(parse_vcf.load_vcf_without_sample(a, "chr22")) == 70


def test_two_devices_in_one_process(capi):
    """Kernels with > 48 KB of dynamic shared memory opt in per function AND per device: a process that parses on device 0
    and then on device 1 (vcf_to_h5 --devices, a notebook that switches GPUs) must be served on both."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    text, samples = synth.random_vcf(700, 150, seed=3, fmt="GT", kinds="mixed")
    ora = oracle.parse_text(text, "*", "chr22")
    for dev in (0, 1, 0):
        p = capi.Parse.from_host(synth.body_of(text), len(samples), region="chr22", device=dev)
        g0, g1 = p.matrix()
        assert np.array_equal(g0, ora["gt0"]) and np.array_equal(g1, ora["gt1"])
        fr = p.compress(64)
        rec = oracle.records_from_columns(ora["chrom"], ora["start"], ora["stop"], ora["ref"], ora["alt"], ora["gt0"][7], ora["gt1"][7])
        raw = rec.tobytes() + b"\0" * (int(fr.info.n_chunks) * 64 * 35 - rec.nbytes)
        for k, f in enumerate(fr.sample(7)):
            assert oracle.blosc_chunk_decode(f, 64 * 35).tobytes() == raw[k * 64 * 35:(k + 1) * 64 * 35]
        fr.close(); p.close()
