"""Cost of the BGZF CRC32 check (hb_set_bgzf_crc_check) at the bench shape: 1.1 M variants x 2,504 samples, u^8 cohort.

The text is the bench's synthetic text (seed 42), BGZF-compressed with hb_bgzf_compress_host at level 6 as bench.py does
(~169 K members).  One run prints the card and its power limit, then one JSON line with, for the check off and on:
  1. kernel 0 alone (hb_bgzf_inflate): kernel time from CUDA events, median over --reps calls taken off / on alternately
     after one warm-up of each, and GB/s of text;
  2. the file parse from pinned host BGZF bytes (hb_parse_vcf_bytes): wall time and ms_inflate, medians the same way;
  3. the check: the text inflated with the check on is byte-identical to the text inflated with it off.

  python tools/crc_bench.py [--variants 1100000] [--samples 2504] [--reps 5] [--out DIR]
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

AF_SKEW_HEADLINE = 1 << 8          # the bench's headline cohort (u^8 ALT frequencies)


def gpu_label():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--variants", type=int, default=1_100_000)
    ap.add_argument("--samples", type=int, default=2504)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    from haplohyped_varawareml_b200 import capi
    if not torch.cuda.is_available():
        raise SystemExit("crc_bench needs a CUDA device")
    label = gpu_label()
    print("# GPU:", label, flush=True)
    spec = capi.synth_spec(args.variants, args.samples, seed=42, mix=AF_SKEW_HEADLINE)
    text = capi.synth_header(spec) + capi.synth_host(spec)
    bg = capi.bgzf_compress_host(text, 6)
    n_members = 0
    p = 0
    raw = bg.tobytes()
    while p < len(raw):                                    # members with text (the EOF marker has none)
        bsize = int.from_bytes(raw[p + 16:p + 18], "little") + 1
        n_members += int.from_bytes(raw[p + bsize - 4:p + bsize], "little") > 0
        p += bsize
    pin = torch.empty(bg.size, dtype=torch.uint8, pin_memory=True)
    pin.numpy()[:] = bg

    kern = {False: [], True: [], "digest": {}}
    for i in range(args.reps + 1):
        for on in (False, True):
            capi.set_bgzf_crc_check(on)
            got, ms = capi.bgzf_inflate(raw, with_ms=True)
            if i:
                kern[on].append(ms)
            else:
                kern["digest"][on] = hashlib.sha256(got).hexdigest() if len(got) == len(text) else "wrong length"
            del got
    capi.set_bgzf_crc_check(False)
    identical = kern["digest"][False] == kern["digest"][True] == hashlib.sha256(text).hexdigest()

    e2e = {False: [], True: []}
    inf = {False: [], True: []}
    for i in range(args.reps + 1):
        for on in (False, True):
            capi.set_bgzf_crc_check(on)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            h = capi.Parse.from_vcf_bytes(pin.data_ptr(), nbytes=pin.numel())
            wall = (time.perf_counter() - t0) * 1e3
            ms_inf = float(h.info.ms_inflate)
            h.close()
            if i:
                e2e[on].append(wall)
                inf[on].append(ms_inf)
    capi.set_bgzf_crc_check(False)

    med = lambda v: float(np.median(v))
    k_off, k_on = med(kern[False]), med(kern[True])
    res = {
        "tool": "crc_bench", "gpu": label, "variants": args.variants, "samples": args.samples,
        "text_bytes": len(text), "bgzf_bytes": int(bg.size), "members": n_members, "reps": args.reps,
        "kernel0_ms_off": k_off, "kernel0_ms_on": k_on,
        "kernel0_text_gbs_off": len(text) / k_off / 1e6, "kernel0_text_gbs_on": len(text) / k_on / 1e6,
        "kernel0_cost_pct": 100.0 * (k_on / k_off - 1.0),
        "kernel0_ms_all": {"off": kern[False], "on": kern[True]},
        "e2e_parse_ms_off": med(e2e[False]), "e2e_parse_ms_on": med(e2e[True]),
        "e2e_ms_inflate_off": med(inf[False]), "e2e_ms_inflate_on": med(inf[True]),
        "e2e_parse_ms_all": {"off": e2e[False], "on": e2e[True]},
        "text_identical": bool(identical),
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "crc_bench.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
