"""Kernels 4a / 4b and kernel 6 at explicit HDF5 chunk sizes, small (kernels 4a / 4b / 6) and large (4a-L / 4b-L / 6-L).

For every chunk size the bench's device step runs on the bench's workload (device-synthesised text, 1.1 M variants x
2,504 samples, u^8 cohort, site templates made while the GT decoder runs) and reports:
  step_ms          the whole step (parse + frames), CUDA events on the launching stream, median over --steps
  ms_site          kernel 4a or 4a-L (hb_frames_info.ms_site), median
  ms_frames        kernel 4b or 4b-L (hb_frames_info.ms_frames), median
  bytes_per_record stored chunk bytes per (record, sample): C_out / (V' * S)
  slot_bytes_per_raw  device frame-buffer bytes (padded slots) per raw record byte: what vcf_to_h5._ChromParse's
                   sample-window estimate (0.25) must bound
  k6_us_B32 / k6_us_B1024  hb_decode_columns_device_large (kernel 6, or 6-L above a warp's shared memory) on B
                   chunks of random (sample, chunk) pairs that stay resident in HBM (one chunk per window of a batch),
                   CUDA events over 20 launches after 3 warm-up launches
then checks the two expectations: the 4,883 step within 1.25x of the 1,075 step, and bytes per record no worse.

  python tools/large_chunk_bench.py [--variants 1100000] [--samples 2504] [--crs 1075,2730,4883,7489] [--steps 5]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

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


def kernel6_us(capi, torch, fr, cr, B, rng, reps=20):
    """hb_decode_columns_device_large on B resident chunks (random sample, random chunk) of fr, microseconds per launch"""
    import numpy as np
    info = fr.info
    offs, sizes = fr.layout()
    S, nc = offs.shape
    s = rng.integers(0, S, B)
    c = rng.integers(0, nc, B)
    dev = torch.device("cuda:0")
    addr = torch.from_numpy((np.uint64(info.d_frames) + offs[s, c].astype(np.uint64)).view(np.int64)).to(dev)
    lens = torch.from_numpy(sizes[s, c].astype(np.uint32).view(np.int32)).to(dev)
    rows = torch.from_numpy((np.arange(B, dtype=np.int64) * cr)).to(dev)
    start = torch.empty(B * cr, dtype=torch.int32, device=dev)
    ref = torch.empty(B * cr, dtype=torch.uint8, device=dev)
    alt = torch.empty_like(ref)
    p1 = torch.empty(B * cr, dtype=torch.int8, device=dev)
    p2 = torch.empty_like(p1)
    status = torch.empty(B, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream

    def launch():
        capi.check(capi.lib().hb_decode_columns_device_large(None, addr.data_ptr(), lens.data_ptr(), rows.data_ptr(), B, cr,
                                                             start.data_ptr(), None, ref.data_ptr(), alt.data_ptr(), p1.data_ptr(),
                                                             p2.data_ptr(), status.data_ptr(), stream))
    for _ in range(3):
        launch()
    torch.cuda.synchronize()
    assert not bool(status.any().item()), "a resident chunk did not decode"
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        launch()
    e1.record()
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--variants", type=int, default=1_100_000)
    ap.add_argument("--samples", type=int, default=2504)
    ap.add_argument("--crs", default="1075,2730,4883,7489")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--json", default="", help="also write the result here")
    args = ap.parse_args()
    crs = [int(x) for x in args.crs.split(",")]

    import numpy as np
    import torch
    from haplohyped_varawareml_b200 import capi
    if not torch.cuda.is_available():
        raise SystemExit("large_chunk_bench: no CUDA device (the kernels have no CPU fallback)")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    V, S = args.variants, args.samples
    spec = capi.synth_spec(V, S, seed=args.seed, chrom="chr22", mix=AF_SKEW_HEADLINE)
    T = int(capi.lib().hb_synth_body_bytes(spec))
    text = torch.empty(T + 256, dtype=torch.uint8, device=dev)
    text[T:].zero_()
    capi.check(capi.lib().hb_synth_device(spec, text.data_ptr(), T, 0, None))
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream().cuda_stream
    p = capi.Parse.from_device(text.data_ptr(), T, S, region="chr22", device=0, stream=stream)
    Vk = int(p.info.n_records)
    rows = []
    for cr in crs:
        fr = p.compress(cr)
        p.attach(fr)
        for _ in range(args.warmup):
            p.rerun()
            fr.rerun(p)
        torch.cuda.synchronize()
        step, ks, kf = [], [], []
        for _ in range(args.steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            p.rerun()
            fr.rerun(p)
            e1.record()
            torch.cuda.synchronize()
            step.append(e0.elapsed_time(e1))
            fi = fr.info
            ks.append(fi.ms_site)
            kf.append(fi.ms_frames)
        fi = fr.info
        rng = np.random.default_rng(cr)
        row = {"cr": cr, "n_chunks": int(fi.n_chunks), "step_ms": float(np.median(step)), "ms_site": float(np.median(ks)),
               "ms_frames": float(np.median(kf)), "bytes_per_record": fi.total_bytes / (Vk * S),
               "slot_bytes_per_raw": fi.padded_bytes / (35.0 * Vk * S), "site_lz4_bytes_per_record": fi.site_lz4_bytes / Vk,
               "k6_us_B32": kernel6_us(capi, torch, fr, cr, 32, rng), "k6_us_B1024": kernel6_us(capi, torch, fr, cr, 1024, rng)}
        rows.append(row)
        print(json.dumps(row), flush=True)
        p.attach(None)
        fr.close()
    p.close()
    by = {r["cr"]: r for r in rows}
    checks = {}
    if 1075 in by and 4883 in by:
        checks["step_4883_over_1075"] = by[4883]["step_ms"] / by[1075]["step_ms"]
        checks["step_within_1.25x"] = checks["step_4883_over_1075"] <= 1.25
        checks["bytes_per_record_no_worse"] = by[4883]["bytes_per_record"] <= by[1075]["bytes_per_record"]
    out = {"gpu": gpu_label(), "variants": V, "kept_records": Vk, "samples": S, "rows": rows, "checks": checks}
    print(json.dumps(out), flush=True)
    if args.json:
        with open(args.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
