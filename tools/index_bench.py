"""Tabix indexes on the GPU and region queries through them.

(a) Building the .tbi of the config-2 shape (--variants x --samples, one contig, bgzipped at level 6 by
    hb_bgzf_compress_host): the split HB_TRACE reports (parse = file bytes to H2D + inflate + newline tokenizer, kernel 7a,
    kernel 7b, host assembly) and the wall time of hb_index_bgzf, median of --reps.
(b) hb_parse_file wall time with the index and with hb_set_use_index(0), medians of --reps alternating:
    - a 1 Mb region and the whole contig of that file;
    - one chromosome of a 22-contig file (--g-variants split over 22 contigs in proportion to GRCh38 lengths,
      --g-samples samples).
Prints the card and its power limit, then one JSON line, also written to --out/index_bench_1gpu.json.

  python tools/index_bench.py [--variants 1100000] [--samples 2504] [--g-variants 3000000] [--g-samples 256] [--reps 3]
"""
from __future__ import annotations

import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

GRCH38 = [248956422, 242193529, 198295559, 190214555, 181538259, 170805979, 159345973, 145138636, 138394717, 133797422,
          135086622, 133275309, 114364328, 107043718, 101991189, 90338345, 83257441, 80373285, 58617616, 64444167,
          46709983, 50818468]


def gpu_label():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def traced(fn):
    """fn() with HB_TRACE on and the library's stderr lines captured."""
    os.environ["HB_TRACE"] = "1"
    with tempfile.TemporaryFile() as f:
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["HB_TRACE"]
        f.seek(0)
        return f.read().decode(errors="replace")


def query_times(capi, path, region, reps):
    on, off = [], []
    for _ in range(reps):
        for use, acc in ((True, on), (False, off)):
            with capi.use_index(use):
                t = time.perf_counter()
                p = capi.Parse.from_file(path, region)
                acc.append(1e3 * (time.perf_counter() - t))
                if use:
                    info = p.index_info
                p.close()
    return {"region": region, "ms_with_index": statistics.median(on), "ms_full_scan": statistics.median(off),
            "compressed_bytes_read": info[1], "file_bytes": os.path.getsize(path)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--variants", type=int, default=1_100_000)
    ap.add_argument("--samples", type=int, default=2504)
    ap.add_argument("--g-variants", type=int, default=3_000_000)
    ap.add_argument("--g-samples", type=int, default=256)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    a = ap.parse_args()
    from haplohyped_varawareml_b200 import capi
    card = gpu_label()
    print(card, flush=True)
    res = {"gpu": card}
    with tempfile.TemporaryDirectory() as d:
        # (a) + (b) on the config-2 shape
        spec = capi.synth_spec(a.variants, a.samples, seed=42)
        text = capi.synth_header(spec) + capi.synth_host(spec)
        data = capi.bgzf_compress_host(text, 6).tobytes()
        del text
        path = os.path.join(d, "c2.vcf.gz")
        open(path, "wb").write(data)
        walls, lines = [], []
        capi.build_index(data, "tbi")                       # warm-up
        for _ in range(a.reps):
            t = time.perf_counter()
            lines.append(traced(lambda: capi.build_index(data, "tbi")))
            walls.append(1e3 * (time.perf_counter() - t))
        parts = {}
        for ln in lines:
            m = re.search(r"parse \(H2D \+ inflate \+ locate\) ([\d.]+) ms, kernel 7a ([\d.]+) ms, 7b ([\d.]+) ms, host assembly "
                          r"([\d.]+) ms, total ([\d.]+) ms", ln)
            if m:
                for k, v in zip(("parse_ms", "kernel_7a_ms", "kernel_7b_ms", "host_assembly_ms", "total_ms"), m.groups()):
                    parts.setdefault(k, []).append(float(v))
        res["build_tbi"] = {"shape": "%d variants x %d samples, one contig" % (a.variants, a.samples),
                            "bgzf_bytes": len(data), "wall_ms": statistics.median(walls),
                            **{k: statistics.median(v) for k, v in parts.items()},
                            "note": "parse_ms covers reading the bytes from host memory, H2D, kernel 0 and the tokenizer"}
        capi.index_file(path)
        first = 10_000_000 + 35 * (a.variants // 2)
        res["query_config2"] = [query_times(capi, path, "chr22:%d-%d" % (first, first + 1_000_000), a.reps),
                                query_times(capi, path, "chr22", a.reps)]
        del data
        # (b) one chromosome of a 22-contig file
        tot = sum(GRCH38)
        parts_txt = []
        for i, ln in enumerate(GRCH38):
            n = max(1, a.g_variants * ln // tot)
            s = capi.synth_spec(n, a.g_samples, seed=100 + i, chrom="chr%d" % (i + 1))
            parts_txt.append((capi.synth_header(s) if i == 0 else b"") + capi.synth_host(s))
        gdata = capi.bgzf_compress_host(b"".join(parts_txt), 6).tobytes()
        del parts_txt
        gpath = os.path.join(d, "genome.vcf.gz")
        open(gpath, "wb").write(gdata)
        capi.index_file(gpath)
        res["query_genome"] = {"shape": "%d variants x %d samples in 22 contigs" % (a.g_variants, a.g_samples),
                               "bgzf_bytes": len(gdata), "chr20": query_times(capi, gpath, "chr20", a.reps)}
    line = json.dumps(res)
    print(line)
    os.makedirs(a.out, exist_ok=True)
    open(os.path.join(a.out, "index_bench_1gpu.json"), "w").write(line + "\n")


if __name__ == "__main__":
    main()
