"""Host-side mirror of the reference's conversion driver and CLI (src/haplohyped/vcf_to_h5.py).

Same class, constructor arguments, method names, click options, input naming
(`{vcf}/chr{N}.filtered.vcf.gz`, N = 1..22, :51,:151), output path (`{outdir}/{cohort}.h5`, :161),
group / dataset names (`donor_{id}/chr_{N}/snp_data`, :132-134), record dtype (:119-127) and filter
(32001 with opts (2,2,0,0,5,1,2), :135).

What changes is the shape of the work.  The reference calls `parse_vcf.load_vcf` once per (donor,
chromosome) -- S whole-file scans per chromosome -- then builds records in two per-record Python
loops, lets h5py/hdf5plugin compress them on the CPU into one temporary file each and copies every
temporary file into the final one (:98-135,:154-180).  Here one chromosome file is parsed ONCE on the
GPU for all donors (`hb_parse_file`), kernel 4 emits the Blosc2 frames of every donor's chunks
(`hb_compress_records`), and the frames are stored as-is (HDF5 direct chunk write) straight into the
final file; the 35-byte records are never materialised on the host.

Documented deviations (each replaces a crash or a silent loss in the reference, SURVEY.md D11-D13):
a chromosome file that does not exist is skipped with a warning (the reference dereferences NULL);
a donor that is not in the VCF header is reported and skipped (the reference's worker exception
vanishes inside `executor.map`); `tmp_files/` is still created and removed but never used.

`verify_crc=True` (CLI `--verify-crc`) checks the CRC32 of every BGZF member, as htslib's reader does
(`capi.crc_check`); a file that fails it is skipped, counted and logged like any other unreadable file.
"""
from __future__ import annotations

import contextlib
import logging
import os
import shutil
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from typing import Dict, List, Optional

import numpy as np

from . import capi
from .container import open_h5
from .h5_reader import RECORD_DTYPE

logger = logging.getLogger(__name__)


def _configure_logging():
    """The reference configures this at import (vcf_to_h5.py:17-25); here only the CLI does."""
    logging.basicConfig(level=logging.INFO, format="%(asctime)s - %(name)s - %(levelname)s - %(message)s",
                        handlers=[logging.FileHandler("haplohyped.log"), logging.StreamHandler()])


class _ChromParse:
    """One chromosome file: device-resident parse + Blosc2 frames of the donors' chunks.

    When the donors of the sample list that the file has are fewer than its samples, only theirs are decoded (a sample
    subset, in header order): 1,000 donors of a 200,000-sample cohort keep 1/200 of the genotype planes.  The datasets are
    those an all-sample parse gives.

    The frames of ALL donors of a big chromosome may not fit in HBM next to the genotype planes (1000G chr1: 64 GB of
    text, 32 GB of planes, ~100 GB of frames), so the text is given back right after the parse and the frames are made
    for a WINDOW of samples at a time; the window is as large as free HBM allows -- all samples for anything chr22-sized."""

    def __init__(self, data_path: str, chromosome: int, device: int, window: Optional[int] = None,
                 donors: Optional[List[str]] = None):
        subset = None
        if donors is not None:
            wanted = set(donors)
            header = capi.file_sample_names(data_path)
            subset = list(dict.fromkeys(s for s in header if s in wanted))
            if not subset or len(subset) == len(header):
                subset = None                           # nothing to leave out (or no donor here: the file is still checked)
        self.parse = capi.Parse.from_file(data_path, region=f"chr{chromosome}", want_gt=True, device=device, samples=subset)
        self.samples = self.parse.sample_names()
        self.index = {s: i for i, s in enumerate(self.samples)}
        info = self.parse.info
        self.n_records = int(info.n_records)
        self.ploidy_err, self.badgt_err = self.parse.sample_errors()
        self.parse.release_text()
        self.frames = None
        self.win0 = self.win_n = 0
        self.chunk_records = int(capi.lib().hb_guess_chunk_records(max(1, self.n_records))) if self.n_records else 0
        n = len(self.samples)
        if window is None and self.n_records and n:
            import torch
            free, _ = torch.cuda.mem_get_info(device)
            est_row = int(0.25 * 35 * self.n_records) + (1 << 16)         # slots are ~0.2 x the raw record bytes per sample
            window = max(1, min(n, int(0.8 * free / est_row)))
        self.window = max(1, min(n, window or n)) if n else 0

    def windows(self):
        """(s0, ns) of every sample window."""
        return [(s0, min(self.window, len(self.samples) - s0)) for s0 in range(0, len(self.samples), max(1, self.window))]

    def frames_for(self, s0: int, ns: int):
        """Frames handle positioned on samples [s0, s0 + ns): made on first use, re-run when the window moves."""
        if not self.n_records:
            return None
        if self.frames is None:
            self.frames = self.parse.compress(0, 0, self.window)           # window 0; also fixes the allocation
            self.win0, self.win_n = 0, self.window
        if (s0, ns) != (self.win0, self.win_n):
            self.frames.set_window(s0, ns)
            self.frames.rerun(self.parse)
            self.win0, self.win_n = s0, ns
        return self.frames

    def donor_frames(self, donor_id: str):
        if donor_id not in self.index:
            raise RuntimeError("Error parsing VCF file: the 1-th sample are not in the VCF.\nparameter samples:" + donor_id)
        s = self.index[donor_id]
        if self.badgt_err[s]:
            raise RuntimeError("Error parsing VCF file: Couldn't read GT data: value not a number or '.'")
        if self.ploidy_err[s]:
            raise RuntimeError("Error parsing VCF file: ploidy != 2 (reference: assert(var.ploidy() == 2), parse_vcf.cpp:46)")
        if not self.n_records:
            return []
        s0 = s - s % self.window
        fr = self.frames_for(s0, min(self.window, len(self.samples) - s0))
        return fr.sample(s - s0)

    def close(self):
        if self.frames:
            self.frames.close()
        self.parse.close()


class VCFtoHDF5Converter:
    def __init__(self, cohort_name: str, vcf_dir: str, out_dir: str, sample_list_path: str, cores: int,
                 cxx_threads: int, device: int = 0, chromosomes=None, backend: Optional[str] = None,
                 sample_window: Optional[int] = None, devices: Optional[List[int]] = None, verify_crc: bool = False):
        self.cohort_name = cohort_name
        self.vcf_dir = vcf_dir
        self.out_dir = out_dir
        self.sample_list_path = sample_list_path
        self.cores = cores
        self.cxx_threads = cxx_threads            # kept for interface parity; a no-op in the reference too (SURVEY 2.2)
        self.device = device
        # several GPUs of one box: the chromosome files are bin-packed onto them by size (shard.plan_shards, the reference's
        # fan-out is executor.map over donors, :191-192); every GPU parses and compresses its own files, the datasets go into
        # the one output file under a lock -- no genotype byte ever moves between GPUs
        self.devices = [int(d) for d in devices] if devices else [device]
        self._wlock = threading.RLock()
        self.backend = backend
        self.sample_window = sample_window        # None: as many samples per frames pass as free HBM allows
        self.verify_crc = verify_crc              # BGZF CRC32 check (process-wide while this converter parses)
        self.donor_ids = self.read_sample_list(sample_list_path)
        self.chromosomes = range(1, 23) if chromosomes is None else chromosomes
        self.tmp_dir = os.path.join(out_dir, "tmp_files")
        os.makedirs(self.tmp_dir, exist_ok=True)
        self._out = None
        self._chrom: Dict[int, _ChromParse] = {}
        self.stats = {"datasets": 0, "records": 0, "stored_bytes": 0, "skipped_files": 0, "skipped_donors": 0}

    def read_sample_list(self, sample_list_path: str) -> List[str]:
        try:
            with open(sample_list_path, "r") as f:
                return [line.strip() for line in f]
        except FileNotFoundError as e:
            logger.error(f"Sample list file not found: {e}")
            raise
        except Exception as e:
            logger.error(f"An error occurred while reading the sample list: {e}")
            raise

    # -- output file, opened lazily so that single-call use of genotype_vcf_to_hdf5 works too
    def _final(self):
        with self._wlock:
            if self._out is None:
                os.makedirs(self.out_dir, exist_ok=True)
                self._out = open_h5(os.path.join(self.out_dir, f"{self.cohort_name}.h5"), "w", backend=self.backend)
            return self._out

    def _count(self, **kw):
        with self._wlock:
            for k, v in kw.items():
                self.stats[k] += v

    def _crc_scope(self):
        return capi.crc_check(True) if self.verify_crc else contextlib.nullcontext()

    def _chrom_parse(self, data_path: str, chromosome: int, device: Optional[int] = None) -> _ChromParse:
        with self._wlock:
            cp = self._chrom.get(chromosome)
        if cp is None:
            with self._crc_scope():
                cp = _ChromParse(data_path, chromosome, self.device if device is None else device, self.sample_window,
                                 self.donor_ids)
            with self._wlock:
                self._chrom[chromosome] = cp
        return cp

    def genotype_vcf_to_hdf5(self, data_path: str, donor_id: str, chromosome: int) -> None:
        """One (donor, chromosome) dataset -- the reference's unit of work (:79-140)."""
        logger.info(f"Processing VCF file {data_path} for chromosome {chromosome} and donor {donor_id}")
        try:
            if donor_id:
                cp = self._chrom_parse(data_path, chromosome)
                frames = cp.donor_frames(donor_id)
                chunk = cp.chunk_records or int(capi.lib().hb_guess_chunk_records(max(1, cp.n_records)))
                with self._wlock:
                    self._final().write_chunked(f"donor_{donor_id}/chr_{chromosome}/snp_data", RECORD_DTYPE, cp.n_records,
                                                chunk, frames)
                self._count(datasets=1, records=cp.n_records, stored_bytes=sum(len(f) for f in frames))
                logger.info(f"Finished processing VCF file for donor {donor_id} and chromosome {chromosome}")
        except Exception as e:
            logger.error(f"An error occurred while processing VCF file: {e}")
            raise

    def process_chromosome(self, chromosome: int, device: Optional[int] = None) -> None:
        """All donors of one chromosome file: one GPU parse + one compression pass."""
        vcf_file = os.path.join(self.vcf_dir, f"chr{chromosome}.filtered.vcf.gz")
        if not os.path.exists(vcf_file):
            logger.warning(f"{vcf_file} does not exist; chromosome {chromosome} skipped")
            self._count(skipped_files=1)
            return
        cp = self._chrom_parse(vcf_file, chromosome, device)
        good = [d for d in self.donor_ids if d in cp.index and not cp.badgt_err[cp.index[d]] and not cp.ploidy_err[cp.index[d]]]
        bulk = cp.n_records > 0 and len(good) * 4 >= len(cp.samples) and hasattr(self._final(), "write_frames_bulk")
        if bulk:
            # window by window: the frames of all its donors leave the GPU in one copy and enter the file with one write;
            # each dataset's chunk index then points into that block (no per-chunk work on the host)
            for s0, ns in cp.windows():
                mine = [d for d in good if s0 <= cp.index[d] < s0 + ns]
                if not mine:
                    continue
                fr = cp.frames_for(s0, ns)
                buf, offs, sizes = fr.fetch_packed()            # gathered on the device: no slot padding crosses PCIe or reaches the file
                rows = [cp.index[d] - s0 for d in mine]
                with self._wlock:
                    self._final().write_frames_bulk([f"donor_{d}/chr_{chromosome}/snp_data" for d in mine], RECORD_DTYPE,
                                                    cp.n_records, cp.chunk_records, buf, offs[rows], sizes[rows])
                self._count(datasets=len(mine), records=cp.n_records * len(mine), stored_bytes=int(sizes[rows].sum()))
                del buf
        done = set(good) if bulk else set()
        for donor_id in self.donor_ids:
            if donor_id in done:
                continue
            try:
                self.genotype_vcf_to_hdf5(vcf_file, donor_id, chromosome)
            except capi.HaploError:
                raise                                   # the file itself is unreadable / malformed
            except RuntimeError:
                self._count(skipped_donors=1)           # this donor only (unknown, haploid, bad GT)
        with self._wlock:
            cp = self._chrom.pop(chromosome, None)
        if cp is not None:
            cp.close()

    def process_donor(self, donor_id: str) -> None:
        """The reference's per-donor loop (:142-152), kept for callers that drive it directly."""
        logger.info(f"Processing donor {donor_id}")
        for chromosome in self.chromosomes:
            vcf_file = os.path.join(self.vcf_dir, f"chr{chromosome}.filtered.vcf.gz")
            if not os.path.exists(vcf_file):
                logger.warning(f"{vcf_file} does not exist; chromosome {chromosome} skipped")
                continue
            self.genotype_vcf_to_hdf5(vcf_file, donor_id, chromosome)

    def merge_h5_files(self) -> None:
        """Nothing to merge: datasets were written into the final file directly.  Closes it."""
        final_h5_file = os.path.join(self.out_dir, f"{self.cohort_name}.h5")
        self._final().close()
        self._out = None
        logger.info(f"Finished writing {final_h5_file}")

    def run(self):
        start_time = time.time()
        try:
            with self._crc_scope():
                # chromosome-major: one device-resident parse is shared by every donor.  `cores` host
                # threads overlap the BGZF inflate of the next files with the GPU work of the current one.
                present = [c for c in self.chromosomes
                           if os.path.exists(os.path.join(self.vcf_dir, f"chr{c}.filtered.vcf.gz"))]
                self.stats["skipped_files"] += len(list(self.chromosomes)) - len(present)
                for c in self.chromosomes:
                    if c not in present:
                        logger.warning(f"chr{c}.filtered.vcf.gz does not exist in {self.vcf_dir}; skipped")
                if len(self.devices) > 1 and len(present) > 1:
                    self._run_devices(present)
                else:
                    self._run_files(present, self.devices[0])
                merge_start_time = time.time()
                self.merge_h5_files()
                end_time = time.time()
                logger.info(f"Time taken to merge HDF5 files: {end_time - merge_start_time:.2f} seconds")
                logger.info(f"Total time taken: {end_time - start_time:.2f} seconds")
        except Exception as e:
            logger.error(f"An error occurred: {e}")
            raise
        finally:
            for cp in self._chrom.values():
                cp.close()
            self._chrom.clear()
            if self._out is not None:
                self._out.close()
                self._out = None
            shutil.rmtree(self.tmp_dir, ignore_errors=True)

    def _run_files(self, files: List[int], device: int) -> None:
        """The chromosome files of one GPU, in order.  One chromosome ahead, no more: the parse of the next file (file read +
        H2D + GPU inflate + kernels) overlaps the frames / D2H / file write of the current one, and at most two chromosomes'
        genotype planes are in HBM."""
        with ThreadPoolExecutor(max_workers=1) as executor:
            nxt = executor.submit(self._safe_parse, files[0], device) if files else None
            for k, c in enumerate(files):
                cp = nxt.result()
                nxt = executor.submit(self._safe_parse, files[k + 1], device) if k + 1 < len(files) else None
                if cp is None:
                    continue
                with self._wlock:
                    self._chrom[c] = cp
                self.process_chromosome(c, device)

    def plan_devices(self, files: List[int]) -> List[List[int]]:
        """Which chromosome files each GPU converts: longest-processing-time bin packing by file size, largest first."""
        from .shard import plan_shards
        sizes = [os.path.getsize(os.path.join(self.vcf_dir, f"chr{c}.filtered.vcf.gz")) for c in files]
        bins = plan_shards(sizes, len(self.devices))
        return [sorted((files[i] for i in b), key=lambda c: -sizes[files.index(c)]) for b in bins]

    def _run_devices(self, present: List[int]) -> None:
        plan = self.plan_devices(present)
        for d, b in zip(self.devices, plan):
            logger.info(f"GPU {d}: chromosomes {b}")
        errors: List[BaseException] = []

        def work(device, files):
            try:
                self._run_files(files, device)
            except BaseException as e:           # noqa: BLE001 -- re-raised in the caller's thread
                errors.append(e)

        threads = [threading.Thread(target=work, args=(d, b), name=f"gpu{d}") for d, b in zip(self.devices, plan) if b]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errors:
            raise errors[0]

    def _safe_parse(self, chromosome: int, device: Optional[int] = None):
        vcf_file = os.path.join(self.vcf_dir, f"chr{chromosome}.filtered.vcf.gz")
        try:
            return _ChromParse(vcf_file, chromosome, self.device if device is None else device, self.sample_window,
                               self.donor_ids)
        except capi.HaploError as e:
            logger.error(f"An error occurred while processing VCF file: Error parsing VCF file: {e}")
            if e.code in (capi.HB_ERR_MEM, capi.HB_ERR_CUDA):
                raise                                   # out of device memory / a device fault: not this file's problem
            self._count(skipped_files=1)                # an unreadable or malformed file: the others still convert
            return None


def main(argv=None):
    import click

    @click.command()
    @click.option("--cohort_name", required=True, type=str, help="Cohort specific name")
    @click.option("--vcf", required=True, type=str, help="Path to VCF files directory")
    @click.option("--outdir", required=True, type=str, help="Path to results save folder")
    @click.option("--sample_list", required=True, type=str, help="Path to sample list file")
    @click.option("--cores", default=os.cpu_count(), type=int, help="Number of CPU cores to use")
    @click.option("--cxx_threads", default=4, type=int, help="Number of threads to use in the C++ code")
    @click.option("--device", default=0, type=int, help="CUDA device ordinal")
    @click.option("--devices", default=None, type=str,
                  help="CUDA device ordinals, comma-separated (e.g. 0,1,2,3,4,5,6,7) or 'all': chromosome files are spread over them")
    @click.option("--verify-crc", "verify_crc", is_flag=True, default=False,
                  help="Check the CRC32 of every BGZF member, as htslib does; a file that fails is skipped and logged")
    def _main(cohort_name, vcf, outdir, sample_list, cores, cxx_threads, device, devices, verify_crc):
        _configure_logging()
        devs = None
        if devices:
            if devices.strip().lower() == "all":
                import torch
                devs = list(range(torch.cuda.device_count()))
            else:
                devs = [int(x) for x in devices.split(",") if x.strip() != ""]
        VCFtoHDF5Converter(cohort_name=cohort_name, vcf_dir=vcf, out_dir=outdir, sample_list_path=sample_list,
                           cores=cores, cxx_threads=cxx_threads, device=device, devices=devs, verify_crc=verify_crc).run()

    return _main(args=argv, standalone_mode=argv is None)


if __name__ == "__main__":
    main()
