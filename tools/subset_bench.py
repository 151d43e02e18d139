"""Sample-subset parses against the full parse (kernel 3 <kSubset = true> against <false>).

One run prints the card and its power limit, then, for each shape, the full parse and subset parses of k samples of the
same text in HBM, re-run in alternation (full, k1, k2, ... then again) so that drift on a shared machine hits every
configuration alike.  Per configuration: medians over --reps of the stage times (ms_tokenize = locate, ms_sites,
ms_decode: CUDA events inside the parse), of the parse's wall time (host clock around hb_parse_rerun, which ends in a
device synchronise), and the genotype-plane bytes the handle holds (byte planes 2 x gt_stride x k + bit planes
gt_stride / 2 x k).  The text is ~11 GB (config 2) and ~10 GB (wide shape), far above the 126 MB of L2.

  config 2: 1.1 M variants x 2,504 samples, GT-only u^8 text (what bench.py makes), k = 1, 32, 256, 1,252, 2,503
  wide:     25,000 variants x 100,000 samples, GT-only, k = 1,000

Each subset is checked against the full parse (planes of a few of its samples).

  python tools/subset_bench.py [--reps 7] [--out DIR]   (writes DIR/subset_bench_1gpu.json)
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

AF_SKEW_HEADLINE = 1 << 8          # bench.py's headline cohort (u^8 ALT frequencies)


def gpu_label():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def shape(capi, torch, V, S, ks, reps, seed):
    spec = capi.synth_spec(V, S, seed=seed, chrom="chr22", mix=AF_SKEW_HEADLINE)
    T = int(capi.lib().hb_synth_body_bytes(spec))
    text = torch.empty(T + 256, dtype=torch.uint8, device="cuda")
    text[T:].zero_()
    capi.check(capi.lib().hb_synth_device(spec, text.data_ptr(), T, 0, None))
    torch.cuda.synchronize()
    rng = np.random.default_rng(seed)
    cols = {None: None}
    for k in ks:
        cols[k] = np.sort(rng.choice(S, k, replace=False)).tolist()
    handles = {k: capi.Parse.from_device(text.data_ptr(), T, S, region="chr22", samples=c) for k, c in cols.items()}
    times = {k: {"tok": [], "sites": [], "decode": [], "wall": []} for k in cols}
    for k, h in handles.items():                         # warm-up of every configuration
        h.rerun()
    for _ in range(reps):
        for k, h in handles.items():
            t0 = time.perf_counter()
            h.rerun()
            wall = (time.perf_counter() - t0) * 1e3
            i = h.info
            times[k]["tok"].append(i.ms_tokenize); times[k]["sites"].append(i.ms_sites)
            times[k]["decode"].append(i.ms_decode); times[k]["wall"].append(wall)
    full = handles[None]
    rows = []
    for k, h in handles.items():
        i = h.info
        n = int(i.n_samples)
        same = True
        if k is not None:
            assert n == k and i.n_records == full.info.n_records
            for j in sorted({0, k // 2, k - 1}):
                a, b = h.sample(j), full.sample(cols[k][j])
                same = same and all(np.array_equal(x, y) for x, y in zip(a, b))
        med = {m: round(float(np.median(v)), 3) for m, v in times[k].items()}
        rows.append({"k": S if k is None else k, "full": k is None, "ms_tokenize": med["tok"], "ms_sites": med["sites"],
                     "ms_decode": med["decode"], "ms_parse_wall": med["wall"], "tokenizer_used": int(i.tokenizer_used),
                     "plane_bytes": int(2.5 * i.gt_stride * n), "identical_to_full": same})
    res = {"variants": V, "samples": S, "text_bytes": T, "n_records": int(full.info.n_records), "reps": reps, "rows": rows}
    for h in handles.values():
        h.close()
    del text
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    import __graft_entry__ as g
    g.build()
    from haplohyped_varawareml_b200 import capi

    res = {"gpu": gpu_label()}
    res["config2"] = shape(capi, torch, 1_100_000, 2504, [1, 32, 256, 1252, 2503], args.reps, 7)
    res["wide"] = shape(capi, torch, 25_000, 100_000, [1000], args.reps, 9)
    print(json.dumps(res))
    ok = all(r["identical_to_full"] for s in ("config2", "wide") for r in res[s]["rows"])
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "subset_bench_1gpu.json"), "w") as f:
            json.dump(res, f, indent=1)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
