#!/usr/bin/env python
"""bench.py -- genotype calls/sec of the VCF -> tensor hot path on B200.

A "step" = one pass of the whole device-resident path over one synthetic VCF body resident in HBM:
record location (head walker / tokenizer) -> site extraction -> GT decode (kernels 1-3, output in the
byte-shuffled planar layout + allele bit planes) -> kernel 4 (site templates, allele-plane LZ4, frame
assembly): decompressed text in, stored HDF5 chunks (bare Blosc chunks, filter 32001) of every (donor,
chunk) out -- SURVEY.md 8(d)'s timing span.  `--parse-only` times kernels 1-3 alone.

N=1 workload: BASELINE.json configs[1] (synthetic chr22-like, 1.1M biallelic variants x 2504 phased
samples, ~11.1 GB of text) with the ALT-frequency spectrum SURVEY 8(d) names (u^8, mean 0.11, about
Beta(0.2, 2)); the denser u^4 cohort of round 1 is timed beside it (`stress_u4`).  N>1: every rank runs
that step on its own chromosome-sized shard (weak scaling; the path shards by chromosome / BGZF range with
no collective on the data path; a 6-int64 all_gather of per-shard index metadata is the only exchange).

Further legs in the same JSON line:
  e2e          BGZF bytes of the .vcf.gz in pinned host memory -> GPU inflate -> parse -> frames -> the packed
               frame image + chunk index + site columns in pinned host memory (what the converter writes to the
               HDF5 file), on EVERY rank, through the C ABI; sub-legs: BGZF streamed -> genotype matrix (every
               rank), host text -> matrix and whole-file BGZF -> matrix (rank 0).
  config3      BASELINE.json configs[2]: 3M variants x 2504 samples in 22 chromosomes, sharded by chromosome
               (LPT) over the N ranks, STRONG scaling: text generated and handles allocated outside the timed
               region; at N > 1 rank 0 also times the whole genome alone, so speedup_vs_n1 is from one job.
  general_text FORMAT=GT:GQ:DP text (the shape of the reference's own fixture): tokenizer + general decode.
  dataset      kernel 5 at BASELINE.json configs[4] shapes.

Contract: python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]; rank 0 prints ONE JSON
line.  --dump-outputs writes a fixed sample of what rank 0's last timed step computed as DIR/<name>.npy (see dump_outputs).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NOMINAL_HBM_GBS = 7700.0
FALLBACK_HBM_GBS = 6650.0
GRCH38_MB = [248.96, 242.19, 198.30, 190.21, 181.54, 170.81, 159.35, 145.14, 138.39, 133.80, 135.09, 133.28, 114.36,
             107.04, 101.99, 90.34, 83.26, 80.37, 58.62, 64.44, 46.71, 50.82]
AF_SKEW_HEADLINE = 1 << 8          # hb_synth_spec.mix bits 8-15 = 1: site ALT frequency u^8 (SURVEY 8d config 2)


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.proc = None
        self.lines = []
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def numa_local_affinity(local: int):
    """Pin this process to the CPUs next to its GPU before any pinned buffer is allocated (first touch decides the
    NUMA node of the pages): with 8 ranks streaming GBs in and out of host memory the copies otherwise cross sockets."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1]
        allowed = set(os.sched_getaffinity(0))
        cpus = [c for c in cpus if c in allowed]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return "cpus %d-%d (%d) next to GPU %d" % (min(cpus), max(cpus), len(cpus), local)
    except Exception as ex:
        return "not set (%s)" % type(ex).__name__
    return "not set"


def cpu_baseline(text_with_header: bytes, sample_names, n_variants_sample: int, threads: int, passes_per_thread: int = 1):
    """The reference's driving pattern (vcf_to_h5.py:150-152,191-192): one whole-text load_vcf pass per
    donor, `threads` donors in parallel.  Runs the CPU oracle: oracle/_ref (the reference's own parse_vcf.cpp compiled
    over the htslib shim, kind "reference") when it was built, else the C port (kind "port").
    Returns (genotype calls/s = donor passes * variants / wall, seconds, donors, kind)."""
    import oracle
    oracle.lib()
    ref = getattr(oracle, "reference_parse_text", None) if getattr(oracle, "have_reference", lambda: False)() else None
    donors = [sample_names[(k * 7919) % len(sample_names)] for k in range(threads * passes_per_thread)]
    done = []

    def work(k):
        for j in range(passes_per_thread):
            d = donors[k * passes_per_thread + j]
            r = ref(text_with_header, d, "") if ref else oracle.parse_text(text_with_header, d, "")
            done.append(r["n"])

    t0 = time.perf_counter()
    th = [threading.Thread(target=work, args=(k,)) for k in range(threads)]
    [t.start() for t in th]
    [t.join() for t in th]
    dt = time.perf_counter() - t0
    calls = sum(done)
    return calls / dt, dt, len(donors), ("reference" if ref else "port")


def run_reference(args):
    """--impl reference: the reference path's CPU implementation on the host cores, on a bounded sample of the same
    workload.  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from haplohyped_varawareml_b200 import capi
    cores = os.cpu_count() or 1
    nv = args.cpu_sample_variants
    spec = capi.synth_spec(nv, args.samples, seed=args.seed, mix=AF_SKEW_HEADLINE)
    text = capi.synth_header(spec) + capi.synth_host(spec)
    names = capi.synth_sample_names(spec)
    kind = "port"
    per = max(1, args.cpu_passes // 4)            # a step = cores * per donor passes over the sample (a few seconds)
    for _ in range(args.warmup):
        cpu_baseline(text, names, nv, cores)
    t_tot, calls_tot = 0.0, 0.0
    for _ in range(args.steps):
        v, dt, nd, kind = cpu_baseline(text, names, nv, cores, passes_per_thread=per)
        t_tot += dt
        calls_tot += v * dt
    value = calls_tot / t_tot
    sample = (f"first {nv} variants x {args.samples} samples of the workload text ({len(text) / 1e6:.0f} MB); per step "
              f"{cores} host threads x {per} donors each, one whole-text load_vcf pass per donor (reference driving pattern)")
    line = {"impl": "reference", "metric": "genotype calls/sec", "value": value, "unit": "calls/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(args),
            "cpu_baseline": {"value": value, "unit": "calls/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "calls/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": ("the reference's own cpp/parse_vcf.cpp + cpp/vcfpp.h compiled unmodified over oracle/hts_shim (a minimal "
                     "restatement of the htslib calls they make; htslib itself is absent)" if kind == "reference" else
                     "oracle C port of parse_vcf.cpp:30-71 semantics; the reference binary needs htslib (absent)")}
    print(json.dumps(line), flush=True)


def workload_config(args):
    return {"workload": f"synthetic chr22-like VCF body: {args.variants} biallelic SNPs x {args.samples} phased samples, "
                        f"FORMAT=GT, site ALT frequency u^8 (mean 0.11, SURVEY 8d), seed {args.seed} (BASELINE.json configs[1])",
            "variants": args.variants, "samples": args.samples,
            "l2": "inputs (GBs of text) are far larger than the 126 MB L2; no flush needed",
            "per_rank": "each rank parses its own shard of this shape (seed + rank)"}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, p, frames, seed):
    """--dump-outputs: what the timed step hands its caller, as float32 / float64 .npy files, so that two builds can be
    compared output for output.  The genotype matrix, the site columns and the stored chunks are GBs at the bench shape,
    so a fixed sample drawn with `seed` is written (under 64 MB in all):
      index_donors [D], index_records [R]   the sampled donors (rows of the matrix) and records (columns)
      gt0, gt1 [D, R]                       allele calls of those donors at those records (-9 = missing)
      start, stop [R]; ref, alt [R]         site columns at those records (REF / ALT as byte values)
      chunk_sizes [D, n_chunks]             size in bytes of every stored chunk (Blosc frame) of the sampled donors
      index_chunks [P, 2]                   P of those chunks: (row of index_donors, chunk)
      chunk_bytes [sum of their sizes]      their stored bytes, back to back in index_chunks order"""
    import numpy as np
    rng = np.random.default_rng(seed)
    info = p.info
    V, S = int(info.n_records), int(info.n_samples)
    donors = np.sort(rng.choice(S, min(S, 32), replace=False))
    records = np.sort(rng.choice(V, min(V, 1 << 16), replace=False))
    out = {"index_donors": donors.astype(np.float64), "index_records": records.astype(np.float64)}
    rows = [p.sample(int(s)) for s in donors]
    out["gt0"] = np.stack([g0[records] for g0, _ in rows]).astype(np.float32)
    out["gt1"] = np.stack([g1[records] for _, g1 in rows]).astype(np.float32)
    start, stop, ref, alt = p.sites()
    out["start"], out["stop"] = start[records].astype(np.float64), stop[records].astype(np.float64)
    out["ref"], out["alt"] = ref[records].view(np.uint8).astype(np.float32), alt[records].view(np.uint8).astype(np.float32)
    if frames is not None:
        fi = frames.info
        nc, cr = int(fi.n_chunks), int(fi.chunk_records)
        stored = [frames.sample(int(s)) for s in donors]
        out["chunk_sizes"] = np.array([[len(f) for f in row] for row in stored], np.float32).reshape(len(donors), nc)
        # a stored chunk holds at most its cr 35-byte records plus the Blosc header: at most 16 MB of chunk_bytes
        n_pairs = min(len(donors) * nc, 64, max(1, (4 << 20) // (35 * cr + 1024)))
        pairs = np.sort(rng.choice(len(donors) * nc, n_pairs, replace=False))
        out["index_chunks"] = np.stack([pairs // nc, pairs % nc], axis=1).astype(np.float64)
        blob = b"".join(stored[int(k) // nc][int(k) % nc] for k in pairs)
        out["chunk_bytes"] = np.frombuffer(blob, np.uint8).astype(np.float32)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# =====================================================================================================================
def leg_general_text(capi, torch, dev, local, peak, blocks=96, block_variants=160, S=2504):
    """FORMAT=GT:GQ:DP text: the tokenizer (kernel 1b, column checkpoints) + the general decode path of kernel 3."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np
    import synth
    text, samples = synth.random_vcf(block_variants, S, seed=5, fmt="GT:GQ:DP", kinds="mixed", site_mix=False)
    body = np.frombuffer(synth.body_of(text), np.uint8)
    blk = torch.from_numpy(body.copy()).to(dev)
    T = blk.numel() * blocks
    buf = torch.empty(T + 256, dtype=torch.uint8, device=dev)
    buf[:T].view(blocks, -1).copy_(blk.unsqueeze(0).expand(blocks, -1))       # the block repeated (POS repeat: the parser does not care)
    buf[T:].zero_()
    torch.cuda.synchronize()
    p = capi.Parse.from_device(buf.data_ptr(), T, S, region="chr22", device=local)
    for _ in range(3):
        p.rerun()
    t1, t2, t3 = [], [], []
    for _ in range(5):
        p.rerun()
        i = p.info
        t1.append(i.ms_tokenize); t2.append(i.ms_sites); t3.append(i.ms_decode)
    med = lambda a: float(sorted(a)[len(a) // 2])
    i = p.info
    V = block_variants * blocks
    ms = med(t1) + med(t2) + med(t3)
    out = {"format": "GT:GQ:DP", "variants": V, "samples": S, "records_kept": int(i.n_records), "text_bytes": T,
           "bytes_per_call": T / (V * S), "tokenizer_used": int(i.tokenizer_used),
           "tokenize": {"ms": med(t1), "gbs": T / med(t1) / 1e6, "frac": T / med(t1) / 1e6 / peak, "bytes": T},
           "sites_ms": med(t2),
           "decode_gt": {"ms": med(t3), "gbs": (T + 2.0 * i.n_records * S) / med(t3) / 1e6,
                         "frac": (T + 2.0 * i.n_records * S) / med(t3) / 1e6 / peak, "bytes": T + 2.0 * i.n_records * S},
           "text_gbs": T / ms / 1e6, "calls_per_s": float(V) * S / ms * 1e3,
           "note": "one 160-variant block of tests/synth.random_vcf text repeated %d times in HBM" % blocks}
    p.close()
    del buf, blk
    return out


def leg_dataset(capi, torch, dev, peak):
    """Kernel 5 (RandomHaplotypeDataset batch encode) at BASELINE.json configs[4] shapes, C = 5: windows and record columns
    resident, hap1 / hap2 float32 one-hot out.  Algorithmic bytes = B*L + 2*B*L*C*4."""
    import numpy as np
    from haplohyped_varawareml_b200 import haplotype_dataset as hd
    from haplohyped_varawareml_b200.common_utils import parse_encode_dict
    rng = np.random.default_rng(1)
    chrom_len = 64_000_000
    seq = torch.from_numpy(rng.choice(np.frombuffer(b"ACGT", np.uint8), size=chrom_len)).to(dev)
    n_rec = chrom_len // 1000
    start = torch.from_numpy(np.sort(rng.integers(0, chrom_len, n_rec)).astype(np.uint32).view(np.int32)).to(dev)
    ref = torch.from_numpy(rng.choice(np.frombuffer(b"ACGT", np.uint8), n_rec)).to(dev)
    alt = torch.from_numpy(rng.choice(np.frombuffer(b"ACGT", np.uint8), n_rec)).to(dev)
    p1 = torch.from_numpy(rng.integers(0, 2, n_rec).astype(np.int8)).to(dev)
    p2 = torch.from_numpy(rng.integers(0, 2, n_rec).astype(np.int8)).to(dev)
    lut = hd.build_lut(parse_encode_dict(None), True)
    lut_t = torch.from_numpy(lut.copy()).to(dev)
    out = []
    for B, L in ((32, 1000), (1024, 1000), (32, 131072), (1024, 131072)):
        ws = rng.integers(0, chrom_len - L, B)
        meta = np.zeros((9, B), dtype=np.uint64)
        meta[0] = [seq.data_ptr() + int(w) for w in ws]
        meta[3], meta[4], meta[5], meta[6], meta[7], meta[8] = start.data_ptr(), ref.data_ptr(), alt.data_ptr(), p1.data_ptr(), p2.data_ptr(), n_rec
        m = torch.from_numpy(meta.view(np.int64)).to(dev)
        lens32 = torch.full((B,), L, dtype=torch.int32, device=dev)
        ws32 = torch.from_numpy(ws.astype(np.uint32).view(np.int32)).to(dev)
        hap1 = torch.empty((B, L, 5), dtype=torch.float32, device=dev)
        hap2 = torch.empty((B, L, 5), dtype=torch.float32, device=dev)
        hb = capi.HapBatch()
        hb.B, hb.L, hb.C = B, L, 5
        hb.item_seq, hb.item_len, hb.item_win_start = m[0].data_ptr(), lens32.data_ptr(), ws32.data_ptr()
        hb.item_start, hb.item_ref, hb.item_alt = m[3].data_ptr(), m[4].data_ptr(), m[5].data_ptr()
        hb.item_p1, hb.item_p2, hb.item_nrec = m[6].data_ptr(), m[7].data_ptr(), m[8].data_ptr()
        hb.lut, hb.hap1, hb.hap2 = lut_t.data_ptr(), hap1.data_ptr(), hap2.data_ptr()
        hb.stream = torch.cuda.current_stream(dev).cuda_stream
        for _ in range(3):
            capi.check(capi.lib().hb_encode_haplotypes(C.byref(hb)))
        torch.cuda.synchronize()
        t = []
        for _ in range(5 if B * L > 1e8 else 30):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            capi.check(capi.lib().hb_encode_haplotypes(C.byref(hb)))
            e1.record()
            torch.cuda.synchronize()
            t.append(e0.elapsed_time(e1))
        ms = sorted(t)[len(t) // 2]
        alg = B * L + 2.0 * B * L * 5 * 4
        out.append({"B": B, "L": L, "C": 5, "ms": ms, "gbs": alg / ms / 1e6, "frac": alg / ms / 1e6 / peak,
                    "bases_per_s": B * L / ms * 1e3})
        del hap1, hap2
    return out


def leg_dataset_store(capi, torch, dev, local, peak, V=400_000, S=64):
    """Row f4 end to end: a cohort's stored chunks resident in HBM (converter output, compressed) -> per batch the device decodes
    only the chunks its windows touch (hb_decode_columns_device) -> kernel 5.  Times one whole batch, host work included."""
    import numpy as np
    from haplohyped_varawareml_b200 import haplotype_dataset as hd
    spec = capi.synth_spec(V, S, seed=7, chrom="chr22", mix=AF_SKEW_HEADLINE)
    T = int(capi.lib().hb_synth_body_bytes(spec))
    text = torch.empty(T + 256, dtype=torch.uint8, device=dev)
    text[T:].zero_()
    capi.check(capi.lib().hb_synth_device(spec, text.data_ptr(), T, local, None))
    torch.cuda.synchronize()
    p = capi.Parse.from_device(text.data_ptr(), T, S, region="chr22", device=local)
    fr = p.compress(0)
    names = capi.synth_sample_names(spec)
    store = hd.GenotypeStore(dev)
    for c in range(1, 23):
        store.add_frames(c, fr, names)
    start = p.sites()[0]
    lo, hi = int(start.min()), int(start.max())
    rng = np.random.default_rng(3)
    seq = torch.from_numpy(rng.choice(np.frombuffer(b"ACGT", np.uint8), size=hi + 200_000)).to(dev)
    rg = hd.ReferenceGenome(sequences={}, device=dev)
    for c in range(1, 23):
        rg._dev[f"chr{c}"] = seq
    import tempfile
    tmp = tempfile.mkdtemp()
    with open(os.path.join(tmp, "s.txt"), "w") as f:
        f.write("\n".join(names))
    with open(os.path.join(tmp, "r.bed"), "w") as f:
        f.write("".join("chr22\t%d\t%d\n" % (a, a + 1000) for a in rng.integers(lo, hi, 4096)))
    out = []
    for B, L in ((32, 1000), (1024, 1000), (32, 131072), (1024, 131072)):
        ds = hd.RandomHaplotypeDataset(os.path.join(tmp, "r.bed"), None, None, os.path.join(tmp, "s.txt"), batch_size=B, seq_length=L,
                                       device=dev, genotype_store=store, reference_genome=rg)
        for _ in range(2):
            h = ds[0]
        torch.cuda.synchronize()
        del h
        t, nchunks = [], 0
        for _ in range(3 if B * L > 1e8 else 10):
            t0 = time.perf_counter()
            h1, h2 = ds[0]
            torch.cuda.synchronize()
            t.append(1e3 * (time.perf_counter() - t0))
            del h1, h2
        items = ds.draw()
        cols, keep = store.window_columns([(d, c, a, e) for c, d, a, e in items])
        nchunks = sum(k[5].numel() for k in keep) if keep else 0
        torch.cuda.synchronize()
        ms = sorted(t)[len(t) // 2]
        alg = B * L + 2.0 * B * L * 5 * 4
        out.append({"B": B, "L": L, "ms_per_batch": ms, "item_us": 1e3 * ms / B, "chunks_decoded_per_batch": int(nchunks),
                    "chunks_per_dataset": int(fr.info.n_chunks), "gbs": alg / ms / 1e6, "frac": alg / ms / 1e6 / peak})
    crec = int(fr.info.chunk_records)
    store.close()
    fr.close(); p.close()
    return {"what": "RandomHaplotypeDataset.__getitem__ on a compressed-resident cohort (%d variants x %d donors, chunk %d records): draw + chunk "
                    "selection (host) + hb_decode_columns_device + hb_encode_haplotypes, wall clock per batch; the reference decodes the whole "
                    "(donor, chromosome) dataset per item" % (V, S, crec), "rows": out}


def leg_config3(args, capi, torch, dist, dev, local, rank, world, shard):
    """configs[2]: the whole genome, sharded by chromosome (LPT), strong scaling; kernels only (text resident, handles
    allocated and warmed outside the timed region)."""
    V_TOTAL, S = args.config3_variants, args.samples
    tot = sum(GRCH38_MB)
    nv = [int(round(V_TOTAL * m / tot)) for m in GRCH38_MB]
    nv[0] += V_TOTAL - sum(nv)
    plan = shard.plan_shards(nv, world)
    stream = torch.cuda.current_stream().cuda_stream

    class Chrom:
        def __init__(self, c):
            self.spec = capi.synth_spec(nv[c], S, seed=args.seed + 100 + c, chrom="chr%d" % (c + 1), mix=AF_SKEW_HEADLINE)
            self.T = int(capi.lib().hb_synth_body_bytes(self.spec))
            self.text = torch.empty(self.T + 256, dtype=torch.uint8, device=dev)
            self.text[self.T:].zero_()
            capi.check(capi.lib().hb_synth_device(self.spec, self.text.data_ptr(), self.T, local, None))
            torch.cuda.synchronize()
            self.p = capi.Parse.from_device(self.text.data_ptr(), self.T, S, region="", device=local, stream=stream)
            self.f = self.p.compress(0)
            self.p.attach(self.f)

        def step(self):
            self.p.rerun()
            self.f.rerun(self.p)

        def close(self):
            self.p.attach(None); self.f.close(); self.p.close()

    def timed(chroms, steps, sync_all):
        def bar():
            if sync_all and world > 1:
                dist.barrier()
            torch.cuda.synchronize()
        for _ in range(2):
            [c.step() for c in chroms]
        bar()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            [c.step() for c in chroms]
        e1.record()
        bar()
        t = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=dev)
        if sync_all and world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    chroms = {c: Chrom(c) for c in plan[rank]}
    ms_n = timed([chroms[c] for c in sorted(chroms, key=lambda c: -nv[c])], args.steps, True)
    meta = {"n_records": sum(int(ch.p.info.n_records) for ch in chroms.values()),
            "n_lines": sum(int(ch.p.info.n_lines) for ch in chroms.values()),
            "text_bytes": sum(ch.T for ch in chroms.values()),
            "out_bytes": sum(int(ch.f.info.total_bytes) for ch in chroms.values())}
    gathered = shard.gather_metadata(meta, device=dev)
    ms_1, err_1 = (ms_n if world == 1 else None), None
    if world > 1:                          # the same genome on rank 0 alone: the N = 1 time of this very job
        if rank == 0:
            try:
                for c in range(len(nv)):
                    if c not in chroms:
                        chroms[c] = Chrom(c)
                ms_1 = timed([chroms[c] for c in sorted(chroms, key=lambda c: -nv[c])], max(2, args.steps // 2), False)
            except Exception as ex:
                err_1 = "%s: %s" % (type(ex).__name__, ex)
        dist.barrier()
    for ch in chroms.values():
        ch.close()
    chroms.clear()
    capi.lib().hb_cache_clear()
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    recs = sum(g["n_records"] for g in gathered)
    out = {"workload": "synthetic whole genome: %d variants x %d samples in 22 chromosomes (variant counts proportional to GRCh38 "
                       "lengths), sharded by chromosome over %d rank(s) with LPT bin packing (BASELINE.json configs[2])" % (V_TOTAL, S, world),
           "scaling": "strong", "n_gpus": world, "records": recs, "text_bytes": sum(g["text_bytes"] for g in gathered),
           "c_out_bytes": sum(g["out_bytes"] for g in gathered), "seconds": ms_n / 1e3, "calls_per_s": float(V_TOTAL) * S / (ms_n / 1e3),
           "variants_per_s": V_TOTAL / (ms_n / 1e3), "largest_bin_share": max(sum(nv[c] for c in b) for b in plan) / V_TOTAL,
           "lpt_speedup_cap": V_TOTAL / max(sum(nv[c] for c in b) for b in plan),
           "seconds_n1_same_job": None if ms_1 is None else ms_1 / 1e3,
           "speedup_vs_n1": None if ms_1 is None else ms_1 / ms_n,
           "timing": "kernels 1-4 of every chromosome of the rank, CUDA events, max over ranks; text in HBM and handles allocated "
                     "before the timed region; the N = 1 time is rank 0 running all 22 chromosomes alone in this job"}
    if err_1:
        out["n1_error"] = err_1
    return out


# =====================================================================================================================
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--variants", type=int, default=1_100_000)
    ap.add_argument("--samples", type=int, default=2504)
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--cpu-sample-variants", type=int, default=60000)
    ap.add_argument("--cpu-passes", type=int, default=24, help="donor passes per host thread of the CPU arm (about 10-20 s of CPU work)")
    ap.add_argument("--config3-variants", type=int, default=3_000_000)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the general-text, dataset and config-3 legs")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--slab-bytes", type=int, default=1 << 30, help="slab size of the streamed e2e paths")
    ap.add_argument("--parse-only", action="store_true", help="step = kernels 1-3 only (no frames)")
    ap.add_argument("--site-matcher", choices=["fast", "deep"], default="fast",
                    help="deep: 4-way hash buckets in the site-plane encoder (hb_set_site_matcher): smaller chunks, slower kernel 4a")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a fixed sample of what rank 0's last step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; --impl reference has none")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup

    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from haplohyped_varawareml_b200 import capi, shard

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback")
    affinity = numa_local_affinity(local)
    # host threads of the library (frame assembly in hb_frames_fetch_packed): this rank's share of the CPUs it may run on
    host_threads = max(1, min(16, len(os.sched_getaffinity(0)) // max(1, world)))
    capi.lib().hb_set_host_threads(host_threads)
    capi.lib().hb_set_site_matcher(1 if args.site_matcher == "deep" else 0)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # rank 0 prints ONE line on stdout: whatever libraries print there meanwhile (NCCL's version banner, when NCCL_DEBUG
    # is set in the environment) goes to stderr -- file descriptor 1 is pointed at stderr until the JSON line is written
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    V, S = args.variants, args.samples
    spec = capi.synth_spec(V, S, seed=args.seed + rank, chrom="chr22", mix=AF_SKEW_HEADLINE)
    T = int(capi.lib().hb_synth_body_bytes(spec))
    text = torch.empty(T + 256, dtype=torch.uint8, device=dev)
    text[T:].zero_()
    capi.check(capi.lib().hb_synth_device(spec, text.data_ptr(), T, local, None))
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream().cuda_stream

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    meta = torch.zeros(6, dtype=torch.int64, device=dev)
    gathered = [torch.zeros(6, dtype=torch.int64, device=dev) for _ in range(world)]
    frames = [None]

    def step(p):
        p.rerun()
        if not args.parse_only:
            frames[0].rerun(p)
        if world > 1:            # the path's only exchange: per-shard index metadata
            i = p.info
            meta[0], meta[1], meta[2] = int(i.n_records), int(i.n_lines), int(i.text_bytes)
            dist.all_gather(gathered, meta)

    def timed_steps(p, steps):
        tok, sit, dec, ks, kf = [], [], [], [], []
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            step(p)
            i = p.info
            tok.append(i.ms_tokenize); sit.append(i.ms_sites); dec.append(i.ms_decode)
            if frames[0] is not None:
                fi = frames[0].info
                ks.append(fi.ms_site); kf.append(fi.ms_frames)
        ev1.record()
        barrier()
        return ev0.elapsed_time(ev1), tok, sit, dec, ks, kf

    # first parse allocates; it is warm-up step 1
    p = capi.Parse.from_device(text.data_ptr(), T, S, region="chr22", device=local, stream=stream)
    if not args.parse_only:
        frames[0] = p.compress(0)
        p.attach(frames[0])                         # site templates are made while the GT decoder runs
    for _ in range(args.warmup - 1):
        step(p)
    info = p.info
    Vk = int(info.n_records)

    barrier()
    launches0 = capi.kernel_launches()
    clocks = ClockSampler(local) if rank == 0 else None
    ms, tok, sit, dec, k4s, k4f = timed_steps(p, args.steps)
    clk = clocks.stop() if clocks else None
    launches = capi.kernel_launches() - launches0
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    calls_total = float(V) * S * world
    value = calls_total / (ms / 1e3 / args.steps)
    fi_head = frames[0].info if frames[0] is not None else None
    c_out_head = float(fi_head.total_bytes) if fi_head is not None else 0.0
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, p, frames[0], args.seed)

    # ---- parity of what was just measured (oracle as the checker): whole HDF5 chunks of three donors -- every record
    # of the chunk, site columns and both alleles, through the stored chunk bytes -- plus the genotype matrix rows
    parity = None
    if rank == 0:
        import oracle
        ok = True
        cr = int(fi_head.chunk_records) if fi_head is not None else 1075
        n_chunks = (Vk + cr - 1) // cr
        donors = (0, S // 2, S - 1)
        stored = {s: frames[0].sample(s) for s in donors} if frames[0] is not None else {}
        checked = 0
        for c in sorted({0, n_chunks // 2, n_chunks - 1}):
            first = c * cr
            cnt = min(cr, V - first)
            part = capi.synth_header(spec) + capi.synth_host(spec, first, cnt)
            ora = oracle.parse_text(part, "*", "chr22")
            ok = ok and ora["n"] == cnt                       # (all synthetic records are kept: chunk c = lines [c*cr, ...))
            for s in donors:
                g0, g1 = p.sample(s)
                ok = ok and np.array_equal(g0[first:first + cnt], ora["gt0"][s]) and np.array_equal(g1[first:first + cnt], ora["gt1"][s])
                if stored:
                    rec = oracle.records_from_columns(ora["chrom"], ora["start"], ora["stop"], ora["ref"], ora["alt"],
                                                      ora["gt0"][s], ora["gt1"][s])
                    raw = rec.tobytes() + b"\0" * (cr * 35 - rec.nbytes)
                    ok = ok and oracle.blosc_chunk_decode(stored[s][c], cr * 35).tobytes() == raw
                    checked += 1
        parity = {"ok": bool(ok), "chunks_decoded": checked, "records_per_chunk": cr,
                  "what": "whole HDF5 chunks (first, middle, last) of donors 0, S/2, S-1: stored chunk -> oracle Blosc decode == "
                          "oracle parse of the same text lines, + the genotype matrix rows of those records"}
        del stored

    # ---- the denser cohort of round 1 (site ALT frequency u^4, mean 0.2) through the same handles
    stress = None
    if not args.parse_only:
        spec4 = capi.synth_spec(V, S, seed=args.seed + rank, chrom="chr22", mix=0)
        T4 = int(capi.lib().hb_synth_body_bytes(spec4))
        if T4 == T:
            capi.check(capi.lib().hb_synth_device(spec4, text.data_ptr(), T, local, None))
            torch.cuda.synchronize()
            for _ in range(2):
                step(p)
            barrier()
            ms4, _, _, dec4, _, kf4 = timed_steps(p, 3)
            t4 = torch.tensor([ms4], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t4, op=dist.ReduceOp.MAX)
            med_ = lambda a: float(sorted(a)[len(a) // 2])
            stress = {"af": "u^4 (mean 0.20)", "ms_per_step": float(t4.item()) / 3, "value": calls_total / (float(t4.item()) / 3e3),
                      "donor_frames_ms": med_(kf4), "decode_gt_ms": med_(dec4), "c_out_bytes": int(frames[0].info.total_bytes)}
            capi.check(capi.lib().hb_synth_device(spec, text.data_ptr(), T, local, None))      # back to the headline cohort
            torch.cuda.synchronize()
            step(p)

    # ---- e2e through the C ABI with HOST buffers
    e2e = None
    bg_path = "/dev/shm/hb_bench_%s.vcf.gz" % os.environ.get("MASTER_PORT", str(os.getpid()))
    try:
      if not args.no_e2e and not args.parse_only:
          # the .vcf.gz: rank 0 compresses ITS text once (stock zlib, all cores: what `bgzip -@` does), every rank converts
          # those bytes (same content on every rank: the leg measures transfer + kernels, not content)
          t_comp = None
          if rank == 0:
              hdr = capi.synth_header(spec)
              full = np.empty(len(hdr) + T, np.uint8)
              full[:len(hdr)] = np.frombuffer(hdr, np.uint8)
              full[len(hdr):] = text[:T].cpu().numpy()
              t0 = time.perf_counter()
              bg = capi.bgzf_compress_host(full, 6)
              t_comp = time.perf_counter() - t0
              del full
              bg.tofile(bg_path)
              del bg
          barrier()
          nb = os.path.getsize(bg_path)
          bgp = torch.empty(nb, dtype=torch.uint8).pin_memory()
          with open(bg_path, "rb") as fh:
              fh.readinto(memoryview(bgp.numpy()))
          barrier()
          if rank == 0:
              os.unlink(bg_path)
          # free the device-resident leg's big buffers: the e2e calls allocate their own
          p.attach(None)
          ref_rows = p.sample(S // 3) if rank == 0 else None
          ref_frames = frames[0].sample(S // 3) if rank == 0 else None
          frames[0].close(); frames[0] = None
          p.close(); p = None
          cap = int(c_out_head * 1.02) + 64 * 1024 * 1024
          alloc_err = None
          try:
              pin = torch.empty(cap, dtype=torch.uint8).pin_memory()
              sites = [torch.empty(Vk, dtype=torch.int32).pin_memory(), torch.empty(Vk, dtype=torch.int32).pin_memory(),
                       torch.empty(Vk, dtype=torch.uint8).pin_memory(), torch.empty(Vk, dtype=torch.uint8).pin_memory()]
          except Exception as ex:
              alloc_err = "%s: %s" % (type(ex).__name__, ex)
          okf = torch.tensor([0 if alloc_err else 1], dtype=torch.int32, device=dev)
          if world > 1:
              dist.all_reduce(okf, op=dist.ReduceOp.MIN)
          if int(okf.item()) == 0:
              raise RuntimeError("pinned host buffers for the e2e leg could not be allocated on every rank (%s)" % (alloc_err or "another rank"))
          last = {}

          def convert_step():
              q = capi.Parse.from_vcf_bytes(bgp.data_ptr(), region="chr22", device=local, nbytes=nb)
              fr = q.compress(0)
              tot, offs, sizes = fr.fetch_packed(out=(pin.data_ptr(), cap))
              capi.check(capi.lib().hb_parse_fetch_sites(q._h, *[a.data_ptr() for a in sites]))
              last.update(tot=int(tot), offs=offs, sizes=sizes, n=int(q.info.n_records), ms_inflate=float(q.info.ms_inflate),
                          ms_frames=float(fr.info.ms_frames))
              fr.close(); q.close()

          convert_step()
          barrier()
          t0 = time.perf_counter()
          for _ in range(args.e2e_steps):
              convert_step()
          barrier()
          dt = time.perf_counter() - t0
          tt = torch.tensor([dt], dtype=torch.float64, device=dev)
          if world > 1:
              dist.all_reduce(tt, op=dist.ReduceOp.MAX)
          dt_serial = float(tt.item())

          # the converter's driving pattern (vcf_to_h5.VCFtoHDF5Converter._run_files): a second host thread parses and
          # compresses file k + 1 (H2D + GPU inflate + kernels 1-4) while the frames of file k leave the GPU; every byte of
          # every file still crosses PCIe inside the timed region, pipeline fill included
          from concurrent.futures import ThreadPoolExecutor

          def parse_step():
              q = capi.Parse.from_vcf_bytes(bgp.data_ptr(), region="chr22", device=local, nbytes=nb)
              return q, q.compress(0)

          def fetch_step(q, fr):
              tot, offs, sizes = fr.fetch_packed(out=(pin.data_ptr(), cap))
              capi.check(capi.lib().hb_parse_fetch_sites(q._h, *[a.data_ptr() for a in sites]))
              last.update(tot=int(tot), offs=offs, sizes=sizes, n=int(q.info.n_records), ms_inflate=float(q.info.ms_inflate),
                          ms_frames=float(fr.info.ms_frames), d2h=int(capi.lib().hb_frames_last_d2h_bytes(fr._h)))
              fr.close(); q.close()

          K = max(2, args.e2e_steps + 1)
          with ThreadPoolExecutor(max_workers=1) as ex:
              def files(n):
                  nxt = ex.submit(parse_step)
                  for i in range(n):
                      q, fr = nxt.result()
                      nxt = ex.submit(parse_step) if i + 1 < n else None
                      fetch_step(q, fr)
              files(3)                                 # warm-up: two files' device buffers exist at once from here on
              barrier()
              t0 = time.perf_counter()
              files(K)
              barrier()
              dt = time.perf_counter() - t0
          tt = torch.tensor([dt], dtype=torch.float64, device=dev)
          if world > 1:
              dist.all_reduce(tt, op=dist.ReduceOp.MAX)
          dt = float(tt.item())
          Vb = float(last["n"])                    # (every rank converts rank 0's file)
          e2e = {"value": Vb * S * world / (dt / K), "unit": "calls/s", "h2d_bytes_per_step": nb * world,
                 "d2h_bytes_per_step": (last["d2h"] + 10 * last["n"]) * world, "steps": K,
                 "ms_per_step": 1e3 * dt / K, "ranks": world, "host_affinity": affinity,
                 "api": "per file and rank: hb_parse_vcf_bytes (BGZF of the .vcf.gz in pinned host memory -> H2D compressed -> GPU "
                        "inflate -> GPU parse) + hb_compress_records (kernel 4) + hb_frames_fetch_packed (the packed image of every "
                        "donor's stored chunks in pinned host memory + the chunk index: the chunk templates cross PCIe once, per donor "
                        "only 32 header bytes and the own tail, %d host threads put the frames together with streaming stores) + "
                        "hb_parse_fetch_sites = what vcf_to_h5 writes to the HDF5 file with one write; %d files back to back driven as the converter drives them (the next file is parsed by a second "
                        "host thread while this file's frames cross PCIe), pipeline fill inside the timed region" % (host_threads, K),
                 "one_call_at_a_time": {"value": Vb * S * world / (dt_serial / args.e2e_steps), "ms_per_step": 1e3 * dt_serial / args.e2e_steps,
                                        "steps": args.e2e_steps, "what": "the same calls strictly one after the other (no second thread)"},
                 "inflate_kernel_ms": last["ms_inflate"], "donor_frames_ms": last["ms_frames"], "text_over_bgzf": T / float(nb),
                 "packed_bytes": last["tot"], "bgzip_equivalent_host_s": t_comp}
          if rank == 0:
              o, z = last["offs"][S // 3], last["sizes"][S // 3]
              e2e["matches_device_path"] = bool(all(pin.numpy()[int(o[k]):int(o[k]) + int(z[k])].tobytes() == ref_frames[k]
                                                    for k in range(len(ref_frames))))
          del pin
          # ---- sub-leg, every rank: the same bytes streamed (slabs of BGZF members) -> genotype matrix + site columns
          out0 = torch.empty((S, Vk), dtype=torch.int8).pin_memory()
          out1 = torch.empty((S, Vk), dtype=torch.int8).pin_memory()
          nrec = C.c_uint64()

          def bgzf_stream_step():
              capi.check(capi.lib().hb_parse_stream_bgzf_host(bgp.data_ptr(), nb, b"chr22", 1, local, args.slab_bytes,
                                                              out0.data_ptr(), out1.data_ptr(), Vk, sites[0].data_ptr(),
                                                              sites[1].data_ptr(), sites[2].data_ptr(), sites[3].data_ptr(),
                                                              None, None, C.byref(nrec), None))

          bgzf_stream_step()
          ok_stream = bool(rank != 0 or (np.array_equal(out0[S // 3].numpy(), ref_rows[0]) and np.array_equal(out1[S // 3].numpy(), ref_rows[1])))
          barrier()
          t0 = time.perf_counter()
          for _ in range(args.e2e_steps):
              bgzf_stream_step()
          barrier()
          tt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
          if world > 1:
              dist.all_reduce(tt, op=dist.ReduceOp.MAX)
          dts = float(tt.item())
          e2e["bgzf_to_matrix_streamed"] = {"value": Vb * S * world / (dts / args.e2e_steps), "unit": "calls/s", "h2d_bytes_per_step": nb * world,
                                            "d2h_bytes_per_step": (2 * S * Vk + 10 * Vk) * world, "steps": args.e2e_steps, "ranks": world,
                                            "matches_device_path": ok_stream,
                                            "api": "hb_parse_stream_bgzf_host: slabs of %d MiB of text: H2D compressed + GPU inflate / GPU parse / "
                                                   "D2H of the matrix overlapped" % (args.slab_bytes >> 20)}
          if rank == 0:
              # ---- sub-legs, rank 0: whole-file BGZF -> matrix; pinned host TEXT -> matrix (round 1's e2e)
              def bgzf_whole_step():
                  q = capi.Parse.from_vcf_bytes(bgp.data_ptr(), region="chr22", device=local, nbytes=nb)
                  capi.check(capi.lib().hb_parse_fetch_matrix(q._h, out0.data_ptr(), out1.data_ptr()))
                  capi.check(capi.lib().hb_parse_fetch_sites(q._h, *[a.data_ptr() for a in sites]))
                  q.close()

              bgzf_whole_step()
              torch.cuda.synchronize()
              tw = []
              for _ in range(args.e2e_steps):
                  t0 = time.perf_counter()
                  bgzf_whole_step()
                  tw.append(time.perf_counter() - t0)
              e2e["bgzf_to_matrix_whole_file"] = {"value": Vb * S / (sum(tw) / len(tw)), "unit": "calls/s", "h2d_bytes_per_step": nb,
                                                  "d2h_bytes_per_step": 2 * S * Vk + 10 * Vk, "steps": args.e2e_steps,
                                                  "step_seconds": tw, "api": "hb_parse_vcf_bytes + hb_parse_fetch_matrix + hb_parse_fetch_sites; rank 0 only"}
              host = torch.empty(T, dtype=torch.uint8).pin_memory()
              host.copy_(text[:T])
              opts = capi.Parse._opts(S, "chr22", False, True, local, 0, None)

              def text_step():
                  capi.check(capi.lib().hb_parse_stream_host(host.data_ptr(), T, C.byref(opts), args.slab_bytes, out0.data_ptr(),
                                                             out1.data_ptr(), Vk, sites[0].data_ptr(), sites[1].data_ptr(),
                                                             sites[2].data_ptr(), sites[3].data_ptr(), None, None, C.byref(nrec), None))

              text_step()
              t0 = time.perf_counter()
              for _ in range(args.e2e_steps):
                  text_step()
              dtt = time.perf_counter() - t0
              e2e["text_to_matrix_streamed"] = {"value": float(V) * S / (dtt / args.e2e_steps), "unit": "calls/s", "h2d_bytes_per_step": T,
                                                "d2h_bytes_per_step": 2 * S * Vk + 10 * Vk, "steps": args.e2e_steps,
                                                "api": "hb_parse_stream_host: pinned host text -> matrix + site columns; rank 0 only"}
              del host
          del out0, out1, bgp
    except Exception as ex:          # e.g. not enough pinnable host memory on a crowded box: the device-resident numbers stand
        e2e = {"value": None, "unit": "calls/s", "error": "%s: %s" % (type(ex).__name__, ex)}
        try:
            if os.path.exists(bg_path) and rank == 0:
                os.unlink(bg_path)
        except OSError:
            pass

    # ---- release the headline leg's buffers before the extra legs
    if frames[0] is not None:
        p.attach(None)
        frames[0].close(); frames[0] = None
    if p is not None:
        p.close(); p = None
    del text
    capi.lib().hb_cache_clear()
    torch.cuda.empty_cache()

    peak, peak_src = measured_peak()
    extra = {}
    if not args.no_extra and not args.parse_only:
        for name, fn in (("config3", lambda: leg_config3(args, capi, torch, dist, dev, local, rank, world, shard)),
                         ("general_text", lambda: leg_general_text(capi, torch, dev, local, peak, S=S) if rank == 0 else None),
                         ("dataset", lambda: leg_dataset(capi, torch, dev, peak) if rank == 0 else None),
                         ("dataset_store", lambda: leg_dataset_store(capi, torch, dev, local, peak) if rank == 0 else None)):
            try:
                extra[name] = fn()
            except Exception as ex:
                extra[name] = {"error": "%s: %s" % (type(ex).__name__, ex)}
            if world > 1:
                dist.barrier()
            torch.cuda.empty_cache()

    if rank == 0:
        med = lambda a: float(sorted(a)[len(a) // 2])
        alg_dec = 4.0 * Vk * S + 2.0 * Vk * S
        alg_parse = T + 2.0 * Vk * S + 33.0 * Vk
        step_s = ms / 1e3 / args.steps
        walker = int(info.tokenizer_used) == 3
        loc_bytes = 64.0 * int(info.n_lines) if walker else float(T)
        stages = {"locate_records": {"ms": med(tok), "bytes": loc_bytes, "gbs": loc_bytes / (med(tok) / 1e3) / 1e9,
                                     "note": ("head walker: reads the head of every record (two 32-byte sectors per record counted) and "
                                              "chains 9th-TAB + 4*S jumps; the decoder proves every jump" if walker else
                                              "tokenizer: reads all of the text")},
                  "sites": {"ms": med(sit)},
                  "decode_gt": {"ms": med(dec), "gbs": alg_dec / (med(dec) / 1e3) / 1e9, "bytes": alg_dec,
                                "frac": alg_dec / (med(dec) / 1e3) / 1e9 / peak}}
        alg_all = alg_parse
        store = None
        if fi_head is not None:
            c_out = c_out_head
            alg_store = 2.0 * Vk * S + 33.0 * Vk + c_out
            alg_all = alg_parse + alg_store
            stages["site_templates"] = {"ms": med(k4s), "note": "runs on a side stream while decode_gt runs"}
            alg_df = 2.0 * Vk * S + c_out           # SURVEY 8d: allele planes read once, every frame written once
            stages["donor_frames"] = {"ms": med(k4f), "bytes": alg_df, "gbs": alg_df / (med(k4f) / 1e3) / 1e9,
                                      "frac": alg_df / (med(k4f) / 1e3) / 1e9 / peak,
                                      "note": "fused: allele-plane LZ4 (from the decoder's bit planes) + frame assembly into closed-form slots, "
                                              "template and tail leave by TMA bulk stores"}
            store = {"c_out_bytes": int(c_out), "frames": int(fi_head.n_chunks) * S, "chunk_records": int(fi_head.chunk_records),
                     "compression_ratio": float(fi_head.raw_bytes) / max(1.0, c_out), "raw_bytes_logical": int(fi_head.raw_bytes),
                     "format": "bare Blosc1 chunk per HDF5 chunk (filter 32001 = hdf5-blosc): 16-byte header, bstarts, one LZ4 block"}
        # the dominant kernel = the stage with the largest measured time that has algorithmic bytes
        dom = max((k for k in stages if "frac" in stages[k]), key=lambda k: stages[k]["ms"])
        traffic, traffic_note = None, None
        try:        # DRAM bytes per launch from the ncu --set full capture of this kernel at this shape (profiles/)
            if V == 1_100_000 and S == 2504 and args.site_matcher == "fast":      # (the capture is of this workload only)
                tr = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))[dom]
                traffic = tr["dram_bytes_per_launch"]
                traffic_note = tr["note"]
        except Exception:
            pass
        roof = {"bound": "hbm", "kernel": dom, "achieved": stages[dom]["gbs"], "peak": peak, "unit": "GB/s",
                "frac": stages[dom]["gbs"] / peak, "traffic": traffic, "traffic_note": traffic_note,
                "peak_source": peak_src, "nominal_peak": NOMINAL_HBM_GBS,
                "algorithmic_bytes_per_launch": stages[dom]["bytes"], "ms_per_launch": stages[dom]["ms"],
                "path": {"algorithmic_bytes": alg_all, "gbs": alg_all / step_s / 1e9, "frac": alg_all / step_s / 1e9 / peak,
                         "definition": ("T + 2*(2*V'*S + 33*V') + C_out per step (SURVEY.md 8d 'fused total'), whole step incl. host syncs"
                                        if fi_head is not None else
                                        "T + 2*V'*S + 33*V' per step (SURVEY.md 8d parse+decode), whole step incl. host syncs")},
                "stages": stages, "store": store}
        cpu = None
        if not args.no_cpu:
            nv = args.cpu_sample_variants
            cs = capi.synth_spec(nv, S, seed=args.seed, mix=AF_SKEW_HEADLINE)
            ctext = capi.synth_header(cs) + capi.synth_host(cs)
            cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
            try:
                os.sched_setaffinity(0, range(os.cpu_count()))          # the CPU arm may use every core of the box
                cores = os.cpu_count() or cores
            except Exception:
                pass
            v, dt, nd, kind = cpu_baseline(ctext, capi.synth_sample_names(cs), nv, cores, passes_per_thread=args.cpu_passes)
            cpu = {"value": v, "unit": "calls/s", "cores": cores, "kind": kind,
                   "sample": f"first {nv} variants x {S} samples ({len(ctext) / 1e6:.0f} MB); {nd} donors in parallel, one "
                             f"whole-text load_vcf pass per donor (reference driving pattern); {dt:.1f} s"}
        line = {"metric": "genotype calls/sec", "value": value, "unit": "calls/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": workload_config(args),
                "variants_per_s": float(V) * world / step_s, "records_kept": Vk, "text_bytes_per_rank": T,
                "step": "parse only (kernels 1-3)" if args.parse_only else "text -> stored HDF5 chunks (kernels 1-4)",
                "tokenizer": int(info.tokenizer_used), "parity_spot_check": parity, "stress_u4": stress,
                "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clk}
        line.update(extra)
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
