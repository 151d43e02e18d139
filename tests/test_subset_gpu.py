"""Sample-subset parses (kernels 3 and 3b, kSubset = true): for every selected sample a subset parse gives exactly what the
full parse of the same bytes gives -- rows, site columns, CHROM runs, planes, per-sample error counts, stored chunks -- on
every route a parse takes, and file-level errors stay file-level."""
import gzip
import os

import numpy as np
import pytest

import bcf_writer
import oracle
import synth

pytestmark = pytest.mark.gpu

S = 300
SUBSETS = {
    "one": [5],
    "first_last": [0, S - 1],
    "tile_seam": [127, 128, 129],
    "every_7th": list(range(0, S, 7)),
    "random_37": sorted(np.random.default_rng(37).choice(S, 37, replace=False).tolist()),
    "all_but_one": [c for c in range(S) if c != 200],
}


@pytest.fixture(scope="module")
def capi(built):
    from haplohyped_varawareml_b200 import capi as c
    return c


@pytest.fixture
def walker_lines(capi):
    def set_(n):
        capi.lib().hb_set_walker_lines(int(n))
    yield set_
    capi.lib().hb_set_walker_lines(0)


def _set_field(text: bytes, rec: int, col: int, value: str) -> bytes:
    """The text with sample column `col` of body record `rec` replaced by `value`."""
    head, body = text[:len(text) - len(synth.body_of(text))], synth.body_of(text).split(b"\n")
    f = body[rec].split(b"\t")
    f[9 + col] = value.encode()
    body[rec] = b"\t".join(f)
    return head + b"\n".join(body)


def _same(full, sub, cols, names=None, lines=True):
    """sub is the subset cols of full (lines=False: one of them read only the lines an index lists)."""
    fi, si = full.info, sub.info
    assert si.n_samples == len(cols) and si.n_records == fi.n_records and (not lines or si.n_lines == fi.n_lines)
    assert si.n_nogt == fi.n_nogt and si.n_bad_cols == fi.n_bad_cols
    for a, b in zip(full.sites(), sub.sites()):
        assert np.array_equal(a, b)
    assert sub.chrom_runs() == full.chrom_runs()
    g0, g1 = full.matrix()
    s0, s1 = sub.matrix()
    assert np.array_equal(s0, g0[cols]) and np.array_equal(s1, g1[cols])
    pl, bg = full.sample_errors()
    spl, sbg = sub.sample_errors()
    assert np.array_equal(spl, pl[cols]) and np.array_equal(sbg, bg[cols])
    assert si.n_bad_gt == int(bg[cols].sum())
    if names is not None:
        assert sub.sample_names() == [names[c] for c in cols]


def _oracle(text, region, sub, cols, names):
    """The oracle, donor by donor (it fails on a donor with a haploid call or an unreadable allele, as the reference does)."""
    s0, s1 = sub.matrix()
    pl, bg = sub.sample_errors()
    for j, c in enumerate(cols):
        if not pl[j] and not bg[j]:
            ora = oracle.parse_text(text, names[c], region)
            assert sub.info.n_records == ora["n"]
            assert np.array_equal(s0[j], ora["gt0"]) and np.array_equal(s1[j], ora["gt1"])


def _text(fmt, seed=1, n=700, site_mix=True):
    text, names = synth.random_vcf(n, S, seed=seed, fmt=fmt, kinds="mixed", multidigit=True, info_end=True, site_mix=site_mix)
    # haploid calls and unreadable alleles in a few columns, both selected and unselected ones
    for rec, col, v in ((3, 5, "1"), (10, 6, "A|0"), (40, 128, "0"), (41, 200, "x/1"), (90, 299, "1|B"), (91, 1, "0|1|1")):
        keys = fmt.split(":")
        sub = ["7"] * len(keys)
        sub[keys.index("GT")] = v
        text = _set_field(text, rec, col, ":".join(sub))
    return text, names


@pytest.mark.parametrize("fmt", ["GT", "GT:GQ:DP"])
@pytest.mark.parametrize("tokenizer", [0, 1, 2, 3])
def test_text_subsets(capi, fmt, tokenizer):
    text, names = _text(fmt)
    body = synth.body_of(text)
    for region in ("chr22", "chr22:10050000-10200000"):
        full = capi.Parse.from_host(body, S, region=region, tokenizer=tokenizer)
        for key, cols in SUBSETS.items():
            sub = capi.Parse.from_host(body, S, region=region, tokenizer=tokenizer, samples=cols)
            assert sub.info.tokenizer_used == full.info.tokenizer_used, key
            _same(full, sub, cols)
            if key in ("tile_seam", "random_37"):
                _oracle(text, region, sub, cols, names)
            sub.rerun()                                      # the subset is kept on the handle
            _same(full, sub, cols)


def test_device_text_subset(capi):
    import torch
    text, _ = _text("GT")
    body = synth.body_of(text)
    d = torch.zeros(len(body) + 256, dtype=torch.uint8, device="cuda")
    d[:len(body)] = torch.frombuffer(bytearray(body), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    full = capi.Parse.from_device(d.data_ptr(), len(body), S, region="chr22")
    cols = SUBSETS["random_37"]
    sub = capi.Parse.from_device(d.data_ptr(), len(body), S, region="chr22", samples=cols)
    _same(full, sub, cols)


@pytest.mark.parametrize("lines", [1, 2, 3])
def test_walker(capi, walker_lines, lines):
    walker_lines(lines)
    text, _ = synth.random_vcf(900, S, seed=lines, fmt="GT", kinds="phased", site_mix=True)
    body = synth.body_of(text)
    full = capi.Parse.from_host(body, S, region="chr22")
    assert full.info.tokenizer_used == 3 and full.info.walker_fallbacks == 0
    for key, cols in SUBSETS.items():
        sub = capi.Parse.from_host(body, S, region="chr22", samples=cols)
        assert sub.info.tokenizer_used == 3 and sub.info.walker_fallbacks == 0, key
        _same(full, sub, cols)


def _files(tmp_path, text):
    out = {}
    for name, data in (("x.vcf", text), ("x.vcf.gz", synth.bgzf_compress(text, block=4099)), ("x.gzip.vcf.gz", gzip.compress(text)),
                       ("x8.bcf", synth.bgzf_compress(bcf_writer.vcf_to_bcf(text))),
                       ("x16.bcf", synth.bgzf_compress(bcf_writer.vcf_to_bcf(text, gt_type=bcf_writer.INT16)))):
        (tmp_path / name).write_bytes(data)
        out[name] = str(tmp_path / name)
    return out


def test_file_inputs(capi, tmp_path):
    text, names = synth.random_vcf(400, S, seed=5, fmt="GT:GQ:DP", kinds="mixed", multidigit=True)
    text = _set_field(_set_field(text, 7, 9, "1:7:7"), 30, 130, "0:7:7")       # haploid calls
    files = _files(tmp_path, text)
    rng = np.random.default_rng(2)
    for name, path in files.items():
        full = capi.Parse.from_file(path, region="chr22")
        assert capi.file_sample_names(path) == names
        for key, cols in SUBSETS.items():
            scrambled = [names[c] for c in rng.permutation(cols)]
            sub = capi.Parse.from_file(path, region="chr22", samples=scrambled)
            if name.endswith(".bcf"):
                assert sub.info.tokenizer_used == 4
            _same(full, sub, cols, names)
            raw = np.fromfile(path, np.uint8)
            sb = capi.Parse.from_vcf_bytes(raw, region="chr22", samples=scrambled)
            _same(full, sb, cols, names)


def test_index_route(capi, tmp_path):
    text, names = _text("GT", seed=6, n=3000, site_mix=False)               # sorted, one contig: tabix indexes it
    path = tmp_path / "x.vcf.gz"
    data = synth.bgzf_compress(text, block=3001)
    path.write_bytes(data)
    ix = capi.build_index(data, "tbi")
    (tmp_path / "x.vcf.gz.tbi").write_bytes(ix)
    region = "chr22:10100000-10200000"
    cols = SUBSETS["every_7th"]
    picked = [names[c] for c in reversed(cols)]
    sub = capi.Parse.from_file(str(path), region=region, samples=picked)
    used, nread, _ = sub.index_info
    assert used and nread < len(data)
    with capi.use_index(False):
        scan = capi.Parse.from_file(str(path), region=region, samples=picked)
        full = capi.Parse.from_file(str(path), region=region)
    assert not scan.index_info[0]
    _same(full, sub, cols, names, lines=False)
    _same(scan, sub, list(range(len(cols))), lines=False)
    sb = capi.Parse.from_vcf_bytes(data, region=region, index=ix, samples=picked)
    assert sb.index_info[0]
    _same(full, sb, cols, names, lines=False)


def test_streamed_route(capi, tmp_path):
    text, names = _text("GT", seed=7, n=3000)
    data = synth.bgzf_compress(text, block=4099)
    path = tmp_path / "x.vcf.gz"
    path.write_bytes(data)
    cols = SUBSETS["random_37"]
    picked = [names[c] for c in cols]
    whole = capi.Parse.from_file(str(path), region="chr22", samples=picked)
    full = capi.Parse.from_file(str(path), region="chr22")
    limit = len(text) // 3                                   # two slabs of limit / 2 are resident: >= 6 slabs
    capi.lib().hb_parse_set_text_limit(limit)
    try:
        streamed = capi.Parse.from_file(str(path), region="chr22", samples=picked)
        streamed_b = capi.Parse.from_vcf_bytes(data, region="chr22", samples=picked)
    finally:
        capi.lib().hb_parse_set_text_limit(0)
    assert len(text) // (limit // 2) >= 5
    with pytest.raises(capi.HaploError):
        streamed.rerun()                                     # the streamed handle has no text: proof it took that route
    for p in (whole, streamed, streamed_b):
        _same(full, p, cols, names)


@pytest.mark.parametrize("chunk", [1075, 4883])
def test_frames(capi, chunk):
    text, _ = _text("GT", seed=8, n=11000)
    body = synth.body_of(text)
    cols = SUBSETS["tile_seam"] + [250]
    full = capi.Parse.from_host(body, S, region="chr22")
    sub = capi.Parse.from_host(body, S, region="chr22", samples=cols)
    ff = full.compress(chunk)
    sf = sub.compress(chunk)
    assert sf.info.n_samples == len(cols)
    want = [ff.sample(c) for c in cols]
    assert [sf.sample(j) for j in range(len(cols))] == want
    win = sub.compress(chunk, 1, 2)                          # sample ranges are relative to the subset
    assert [win.sample(0), win.sample(1)] == want[1:3]
    sub.attach(sf)
    sub.rerun()
    sf.rerun(sub)
    assert [sf.sample(j) for j in range(len(cols))] == want
    sub.attach(None)


def test_column_count_errors_stay_file_level(capi):
    text, _ = synth.random_vcf(300, S, seed=9, fmt="GT", kinds="mixed", site_mix=False)
    body = synth.body_of(text).split(b"\n")
    f = body[100].split(b"\t")
    extra = b"\t".join(f + [b"0|1"])
    missing = b"\t".join(f[:200] + f[201:])
    for bad in (extra, missing):
        t = b"\n".join(body[:100] + [bad] + body[101:])
        for tok in (0, 1, 2, 3):
            for cols in (None, [3], [0, 299], SUBSETS["every_7th"]):
                with pytest.raises(capi.HaploError) as e:
                    capi.Parse.from_host(t, S, region="chr22", tokenizer=tok, samples=cols)
                assert e.value.code == capi.HB_ERR_FORMAT


def test_gt_errors_of_unselected_samples_do_not_count(capi):
    text, _ = _text("GT", seed=10, n=300)
    body = synth.body_of(text)
    full = capi.Parse.from_host(body, S, region="chr22")
    pl, bg = full.sample_errors()
    assert pl.sum() and bg.sum() and full.info.n_bad_gt
    clean = [c for c in range(S) if not pl[c] and not bg[c]]
    for tok in (0, 1, 2):
        sub = capi.Parse.from_host(body, S, region="chr22", tokenizer=tok, samples=clean)
        spl, sbg = sub.sample_errors()
        assert not spl.any() and not sbg.any() and sub.info.n_bad_gt == 0
        _same(full, sub, clean)


def test_hidden_newline_in_unselected_span_falls_back(capi, walker_lines):
    """A record the walker jumps over that holds a newline: the decoder still reads the unselected columns, sees it, and
    the parse falls back to the tokenizer as the full parse does (test_parse_gpu's construction)."""
    walker_lines(2)
    n = S
    rng = np.random.default_rng(1)

    def groups(k):
        return "".join("\t%d|%d" % (a, b) for a, b in rng.integers(0, 2, (k, 2)))

    def head(pos, ref, alt, rid="."):
        return "\t".join(["chr22", str(pos), rid, ref, alt, ".", "PASS", ".", "GT"])

    lines = [head(100 + i, "A", "C") + groups(n) + "\n" for i in range(50)]
    h2 = head(7000, "AT", "G")
    h2 = head(7000, "AT", "G", "r" * (1 + (3 - len(h2)) % 4))
    m = 100
    k2 = 4 * n - 4 * m - 1 - len(h2)
    pair = head(6000, "AT", "G") + groups(m) + "\n" + h2 + groups(k2 // 4) + "\n"
    lines.insert(20, pair)
    lines += [head(9000 + i, "A", "C") + groups(n) + "\n" for i in range(50)]
    body = synth.body_of((synth.header(synth.sample_names(n)) + "".join(lines)).encode())
    full = capi.Parse.from_host(body, n, region="chr22", tokenizer=3)
    assert full.info.walker_fallbacks == 1 and full.info.tokenizer_used == 1
    for cols in ([0], [5, 250], [299]):
        sub = capi.Parse.from_host(body, n, region="chr22", tokenizer=3, samples=cols)
        assert sub.info.walker_fallbacks == 1 and sub.info.tokenizer_used == 1
        _same(full, sub, cols)


def test_argument_errors(capi, tmp_path):
    text, names = synth.random_vcf(50, 20, seed=11)
    body = synth.body_of(text)
    for cols, code in (([], capi.HB_ERR_ARG), ([20], capi.HB_ERR_ARG), ([3, 2], capi.HB_ERR_ARG), ([1, 1], capi.HB_ERR_ARG),
                       ([-1], capi.HB_ERR_ARG)):
        with pytest.raises(capi.HaploError) as e:
            capi.Parse.from_host(body, 20, samples=cols)
        assert e.value.code == code, cols
    path = tmp_path / "x.vcf.gz"
    path.write_bytes(synth.bgzf_compress(text))
    for sel, code in (([], capi.HB_ERR_ARG), ([names[2], names[2]], capi.HB_ERR_ARG), (["nobody"], capi.HB_ERR_SAMPLE),
                      ([names[0], "nobody"], capi.HB_ERR_SAMPLE)):
        for parse in (lambda: capi.Parse.from_file(str(path), samples=sel),
                      lambda: capi.Parse.from_vcf_bytes(path.read_bytes(), samples=sel)):
            with pytest.raises(capi.HaploError) as e:
                parse()
            assert e.value.code == code, sel
            if code == capi.HB_ERR_SAMPLE:
                assert "nobody" in str(e.value)
    # every sample: the ordinary parse
    full = capi.Parse.from_file(str(path))
    every = capi.Parse.from_file(str(path), samples=list(reversed(names)))
    _same(full, every, list(range(20)), names)


def test_converter_parses_only_the_listed_donors(capi, tmp_path, built):
    from haplohyped_varawareml_b200 import h5_reader, vcf_to_h5
    text, names = _text("GT", seed=12, n=2500)
    vdir = tmp_path / "vcf"
    vdir.mkdir()
    (vdir / "chr22.filtered.vcf.gz").write_bytes(synth.bgzf_compress(text))
    pl, bg = capi.Parse.from_host(synth.body_of(text), S, region="chr22").sample_errors()
    bad = [names[c] for c in range(S) if pl[c] or bg[c]]
    few = [names[250], names[3], names[128], names[127], "not_in_the_file"] + bad[:2]
    (tmp_path / "few.txt").write_text("\n".join(few))
    (tmp_path / "all.txt").write_text("\n".join(names + ["not_in_the_file"]))
    got = {}
    for key in ("few", "all"):
        conv = vcf_to_h5.VCFtoHDF5Converter("c", str(vdir), str(tmp_path / key), str(tmp_path / f"{key}.txt"), 2, 4,
                                            chromosomes=[22])
        if key == "few":
            cp = vcf_to_h5._ChromParse(str(vdir / "chr22.filtered.vcf.gz"), 22, 0, None, few)
            assert cp.samples == [n for n in names if n in few]              # the subset parse, header order
            cp.close()
        conv.run()
        rd = h5_reader.VCFH5Reader(str(tmp_path / key / "c.h5"))
        got[key] = (conv.stats, {d: (rd.stored_chunks(d, 22), rd.fetch_genotypes(d, 22).tobytes())
                                 for d in few if d in names and d not in bad})
        rd.close()
    stats_few, data_few = got["few"]
    stats_all, data_all = got["all"]
    assert data_few and data_few == {d: data_all[d] for d in data_few}
    assert stats_few["datasets"] == len(data_few) and stats_few["skipped_donors"] == len([d for d in few if d not in data_few])
    assert stats_few["records"] == stats_all["records"] // stats_all["datasets"] * len(data_few)
    assert stats_few["stored_bytes"] == sum(len(c) for d in data_few for c in data_all[d][0][3])
