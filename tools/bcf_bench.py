"""BCF input at the bench shape: 1.1 M variants x 2,504 samples, u^8 cohort (the bench's headline workload).

The VCF text is the bench's synthetic text.  The BCF of the same records is built with numpy from the VCF parse's site
columns and planes (tests/bcf_writer.bcf_from_columns: fixed-size record heads, ID "."), and both files are BGZF-
compressed with hb_bgzf_compress_host.  One run prints the card and its power limit, then:
  1. the device step on the decompressed BCF in HBM (hb_parse_rerun): kernel times of locate (kernel 1b chain + proof),
     sites and GT decode (kernel 3b), medians over --reps; achieved bytes = BCF body read + 2 V' S + 33 V' written, over
     the time of the three, and that rate as a share of 6,540 GB/s;
  2. the file parse from pinned host BGZF bytes (hb_parse_vcf_bytes), BCF against the .vcf.gz of the same records: wall
     time (median over --reps after one warm-up), ms_inflate, compressed bytes;
  3. the check: planes, sites, and every frame of donors 0, S/2 and S - 1 identical to the VCF parse's.

  python tools/bcf_bench.py [--variants 1100000] [--samples 2504] [--reps 5] [--out DIR]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

AF_SKEW_HEADLINE = 1 << 8          # the bench's headline cohort (u^8 ALT frequencies)
HBM_GBS = 6540.0


def gpu_label():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def pinned(a: np.ndarray):
    import torch
    t = torch.empty(a.size, dtype=torch.uint8, pin_memory=True)
    t.numpy()[:] = a
    return t


def timed_parse(capi, t, reps):
    walls, p = [], None
    for i in range(reps + 1):
        if p is not None:
            p.close()
        t0 = time.perf_counter()
        p = capi.Parse.from_vcf_bytes(t.data_ptr(), nbytes=t.numel())
        if i:
            walls.append((time.perf_counter() - t0) * 1e3)
    return p, float(np.median(walls))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--variants", type=int, default=1_100_000)
    ap.add_argument("--samples", type=int, default=2504)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import __graft_entry__ as g
    g.build()
    from haplohyped_varawareml_b200 import capi
    import bcf_writer

    V, S = args.variants, args.samples
    res = {"gpu": gpu_label(), "variants": V, "samples": S}
    spec = capi.synth_spec(V, S, seed=7, chrom="chr22", mix=AF_SKEW_HEADLINE)
    header = capi.synth_header(spec)
    text = np.frombuffer(header + capi.synth_host(spec), np.uint8)
    vgz = capi.bgzf_compress_host(text, 1)
    del text
    tv = pinned(vgz)
    del vgz
    pv, res["vcf_parse_ms"] = timed_parse(capi, tv, args.reps)
    iv = pv.info
    res["vcf_ms_inflate"], res["vcf_compressed_bytes"] = round(iv.ms_inflate, 3), int(iv.compressed_bytes)
    start, stop, ref, alt = pv.sites()
    g0, g1 = pv.matrix()
    bcf = np.frombuffer(bcf_writer.bcf_from_columns(header, "chr22", start, ref, alt, g0, g1), np.uint8)
    l_text = int(bcf[5:9].view("<u4")[0])
    body = bcf.size - 9 - l_text
    bgz = capi.bgzf_compress_host(bcf, 1)
    del bcf
    tb = pinned(bgz)
    del bgz
    pb, res["bcf_parse_ms"] = timed_parse(capi, tb, args.reps)
    ib = pb.info
    res["bcf_ms_inflate"], res["bcf_compressed_bytes"] = round(ib.ms_inflate, 3), int(ib.compressed_bytes)
    res["tokenizer_used"] = ib.tokenizer_used

    loc, sit, dec = [], [], []
    pb.rerun()
    for _ in range(args.reps):
        pb.rerun()
        i = pb.info
        loc.append(i.ms_tokenize); sit.append(i.ms_sites); dec.append(i.ms_decode)
    ms = [float(np.median(x)) for x in (loc, sit, dec)]
    Vk = int(ib.n_records)
    moved = body + 2 * Vk * S + 33 * Vk
    res.update({"ms_locate": round(ms[0], 3), "ms_sites": round(ms[1], 3), "ms_decode": round(ms[2], 3),
                "ms_device_step": round(sum(ms), 3), "bcf_body_bytes": int(body), "algorithmic_bytes": int(moved),
                "achieved_GBs": round(moved / sum(ms) / 1e6, 1),
                "share_of_6540_GBs": round(moved / sum(ms) / 1e6 / HBM_GBS, 3)})

    b0, b1 = pb.matrix()
    same = bool(np.array_equal(b0, g0) and np.array_equal(b1, g1))
    del b0, b1
    same = same and all(np.array_equal(a, b) for a, b in zip(pb.sites(), (start, stop, ref, alt)))
    fb, fv = pb.compress(0), pv.compress(0)
    for s in (0, S // 2, S - 1):
        same = same and all(np.array_equal(a, b) for a, b in zip(fb.sample(s), fv.sample(s)))
    res["identical_to_vcf"] = same
    print(json.dumps(res))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bcf_bench.json"), "w") as f:
            json.dump(res, f, indent=1)
    return 0 if same else 1


if __name__ == "__main__":
    sys.exit(main())
