"""ctypes binding of libhaplo_b200.so (include/haplo_b200.h).

This is plumbing: the work happens in the CUDA kernels behind the C ABI.  There is no Python or
CPU fallback -- if the library is missing or no sm_100 device is present, calls raise.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhaplo_b200.so")
_lib = None


HB_ERR_IO, HB_ERR_HEADER, HB_ERR_SAMPLE, HB_ERR_PLOIDY, HB_ERR_GT, HB_ERR_FORMAT, HB_ERR_NOGT, HB_ERR_MEM, HB_ERR_CUDA, HB_ERR_ARG = range(1, 11)


class HaploError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(msg)
        self.code = code


class ParseOpts(C.Structure):
    _fields_ = [("n_samples", C.c_uint32), ("region", C.c_char_p), ("end_is_int", C.c_int),
                ("want_gt", C.c_int), ("device", C.c_int), ("tokenizer", C.c_int), ("stream", C.c_void_p)]


class ParseInfo(C.Structure):
    _fields_ = [("text_bytes", C.c_uint64), ("n_lines", C.c_uint64), ("n_records", C.c_uint64),
                ("n_samples", C.c_uint32), ("gt_stride", C.c_uint64), ("d_gt", C.c_void_p * 2),
                ("d_start", C.c_void_p), ("d_stop", C.c_void_p), ("d_ref", C.c_void_p), ("d_alt", C.c_void_p),
                ("n_nonuniform", C.c_uint64), ("n_bad_gt", C.c_uint64), ("n_bad_cols", C.c_uint64),
                ("n_nogt", C.c_uint64), ("tokenizer_used", C.c_int),
                ("ms_tokenize", C.c_float), ("ms_sites", C.c_float), ("ms_decode", C.c_float),
                ("walker_fallbacks", C.c_int), ("ms_inflate", C.c_float), ("compressed_bytes", C.c_uint64)]


class Records(C.Structure):
    _fields_ = [("n", C.c_uint64), ("n_samples", C.c_uint32),
                ("start", C.POINTER(C.c_uint32)), ("stop", C.POINTER(C.c_uint32)),
                ("ref", C.POINTER(C.c_char)), ("alt", C.POINTER(C.c_char)),
                ("chrom_off", C.POINTER(C.c_uint32)), ("chrom_pool", C.POINTER(C.c_char)),
                ("chrom_pool_len", C.c_uint64),
                ("gt0", C.POINTER(C.c_int8)), ("gt1", C.POINTER(C.c_int8)), ("owner_", C.c_void_p)]


class FramesInfo(C.Structure):
    _fields_ = [("n_records", C.c_uint64), ("n_chunks", C.c_uint64), ("chunk_records", C.c_uint64),
                ("n_samples", C.c_uint32), ("total_bytes", C.c_uint64), ("raw_bytes", C.c_uint64),
                ("ms_site", C.c_float), ("ms_frames", C.c_float), ("padded_bytes", C.c_uint64), ("d_frames", C.c_void_p),
                ("site_lz4_bytes", C.c_uint64)]


class HapBatch(C.Structure):
    _fields_ = [("B", C.c_uint32), ("L", C.c_uint32), ("C", C.c_uint32),
                ("item_seq", C.c_void_p), ("item_len", C.c_void_p), ("item_win_start", C.c_void_p),
                ("item_start", C.c_void_p), ("item_ref", C.c_void_p), ("item_alt", C.c_void_p),
                ("item_p1", C.c_void_p), ("item_p2", C.c_void_p), ("item_nrec", C.c_void_p),
                ("lut", C.c_void_p), ("hap1", C.c_void_p), ("hap2", C.c_void_p), ("stream", C.c_void_p)]


class SynthSpec(C.Structure):
    _fields_ = [("n_variants", C.c_uint64), ("n_samples", C.c_uint32), ("seed", C.c_uint64),
                ("first_pos", C.c_uint32), ("pos_step", C.c_uint32), ("mix", C.c_uint32), ("chrom", C.c_char * 16)]


EXPORTS = [
    "hb_last_error", "hb_version", "hb_kernel_launches",
    "hb_load_vcf", "hb_load_vcf_without_sample", "hb_records_free", "hb_cache_clear", "hb_cache_set_limit",
    "hb_parse_host_text", "hb_parse_stream_host", "hb_parse_stream_bgzf_host", "hb_parse_stream_bgzf_resident", "hb_parse_set_text_limit", "hb_set_walker_lines", "hb_set_bcf_segment_bytes", "hb_bgzf_vcf_info", "hb_parse_device_text", "hb_parse_file", "hb_parse_vcf_bytes", "hb_parse_samples", "hb_parse_rerun", "hb_parse_rerun_bytes", "hb_parse_get_info",
    "hb_parse_fetch_sites", "hb_parse_fetch_sample", "hb_parse_fetch_matrix", "hb_parse_fetch_sample_errors",
    "hb_parse_chrom_runs", "hb_parse_free",
    "hb_bgzf_inflate", "hb_bgzf_compress_host",
    "hb_compress_records", "hb_compress_sample_range", "hb_frames_set_window", "hb_parse_release_text", "hb_parse_attach_frames", "hb_frames_rerun", "hb_frames_get_info", "hb_frames_layout", "hb_frames_fetch_all", "hb_frames_fetch_packed", "hb_set_fetch_mode", "hb_set_bgzf_crc_check", "hb_get_bgzf_crc_check", "hb_set_use_index", "hb_get_use_index", "hb_parse_vcf_bytes_indexed", "hb_parse_index_info",
    "hb_parse_host_text_subset", "hb_parse_device_text_subset", "hb_parse_file_subset", "hb_parse_vcf_bytes_subset", "hb_file_samples", "hb_index_bgzf", "hb_index_file", "hb_set_host_threads", "hb_frames_last_d2h_bytes",
    "hb_frames_fetch_sample", "hb_frames_free",
    "hb_guess_chunk_records", "hb_set_site_matcher", "hb_decode_frames", "hb_decode_columns_device", "hb_decode_columns_device_large",
    "hb_encode_haplotypes",
    "hb_synth_body_bytes", "hb_synth_header", "hb_synth_device", "hb_synth_host",
]


def lib():
    """Load libhaplo_b200.so; raise (never fall back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise HaploError(9, f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`; "
                                "there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        L.hb_last_error.restype = C.c_char_p
        L.hb_version.restype = C.c_char_p
        L.hb_kernel_launches.restype = C.c_uint64
        L.hb_load_vcf.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(Records)]
        L.hb_load_vcf_without_sample.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(Records)]
        L.hb_records_free.argtypes = [C.POINTER(Records)]
        L.hb_cache_set_limit.argtypes = [C.c_uint64]
        L.hb_cache_set_limit.restype = None
        L.hb_set_walker_lines.argtypes = [C.c_uint32]
        L.hb_set_walker_lines.restype = None
        L.hb_set_bcf_segment_bytes.argtypes = [C.c_uint64]
        L.hb_set_bcf_segment_bytes.restype = None
        L.hb_set_fetch_mode.argtypes = [C.c_int]
        L.hb_set_fetch_mode.restype = None
        L.hb_set_bgzf_crc_check.argtypes = [C.c_int]
        L.hb_set_bgzf_crc_check.restype = None
        L.hb_get_bgzf_crc_check.restype = C.c_int
        L.hb_set_use_index.argtypes = [C.c_int]
        L.hb_set_use_index.restype = None
        L.hb_get_use_index.restype = C.c_int
        L.hb_parse_vcf_bytes_indexed.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_char_p, C.c_int, C.c_int,
                                                 C.POINTER(C.c_void_p)]
        L.hb_parse_host_text_subset.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(ParseOpts), C.c_void_p, C.c_uint32,
                                                C.POINTER(C.c_void_p)]
        L.hb_parse_device_text_subset.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(ParseOpts), C.c_void_p, C.c_uint32,
                                                  C.POINTER(C.c_void_p)]
        L.hb_parse_file_subset.argtypes = [C.c_char_p, C.c_char_p, C.c_void_p, C.c_uint32, C.c_int, C.POINTER(C.c_void_p)]
        L.hb_parse_vcf_bytes_subset.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_char_p, C.c_void_p, C.c_uint32,
                                                C.c_int, C.POINTER(C.c_void_p)]
        L.hb_file_samples.argtypes = [C.c_char_p, C.POINTER(C.c_uint32), C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.hb_parse_index_info.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.hb_index_bgzf.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.hb_index_file.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_char_p]
        L.hb_set_host_threads.argtypes = [C.c_int]
        L.hb_set_host_threads.restype = None
        L.hb_frames_last_d2h_bytes.argtypes = [C.c_void_p]
        L.hb_frames_last_d2h_bytes.restype = C.c_uint64
        L.hb_parse_set_text_limit.argtypes = [C.c_uint64]
        L.hb_parse_set_text_limit.restype = None
        L.hb_parse_host_text.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(ParseOpts), C.POINTER(C.c_void_p)]
        L.hb_parse_stream_host.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(ParseOpts), C.c_uint64, C.c_void_p, C.c_void_p,
                                           C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]
        L.hb_bgzf_vcf_info.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.hb_parse_stream_bgzf_host.argtypes = [C.c_void_p, C.c_uint64, C.c_char_p, C.c_int, C.c_int, C.c_uint64, C.c_void_p, C.c_void_p,
                                                C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]
        L.hb_parse_stream_bgzf_resident.argtypes = [C.c_void_p, C.c_uint64, C.c_char_p, C.c_int, C.c_int, C.c_uint64, C.POINTER(C.c_void_p),
                                                    C.POINTER(C.c_uint32)]
        L.hb_parse_device_text.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(ParseOpts), C.POINTER(C.c_void_p)]
        L.hb_parse_file.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.hb_parse_vcf_bytes.argtypes = [C.c_void_p, C.c_uint64, C.c_char_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.hb_parse_samples.argtypes = [C.c_void_p, C.POINTER(C.c_uint32), C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.hb_parse_rerun.argtypes = [C.c_void_p]
        L.hb_parse_rerun_bytes.argtypes = [C.c_void_p, C.c_uint64]
        L.hb_parse_get_info.argtypes = [C.c_void_p, C.POINTER(ParseInfo)]
        L.hb_parse_fetch_sites.argtypes = [C.c_void_p] + [C.c_void_p] * 4
        L.hb_parse_fetch_sample.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
        L.hb_parse_fetch_matrix.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.hb_parse_fetch_sample_errors.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.hb_parse_chrom_runs.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p, C.c_uint64, C.c_void_p,
                                          C.c_uint64, C.POINTER(C.c_uint64)]
        L.hb_parse_free.argtypes = [C.c_void_p]
        L.hb_bgzf_compress_host.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.hb_bgzf_inflate.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.c_int,
                                      C.POINTER(C.c_float)]
        if hasattr(L, "hb_compress_records"):
            L.hb_compress_records.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]
            L.hb_frames_get_info.argtypes = [C.c_void_p, C.POINTER(FramesInfo)]
            L.hb_frames_rerun.argtypes = [C.c_void_p, C.c_void_p]
            L.hb_compress_sample_range.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]
            L.hb_frames_set_window.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
            L.hb_parse_release_text.argtypes = [C.c_void_p]
            L.hb_parse_attach_frames.argtypes = [C.c_void_p, C.c_void_p]
            L.hb_frames_layout.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
            L.hb_frames_fetch_all.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
            L.hb_frames_fetch_packed.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]
            L.hb_frames_fetch_sample.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64,
                                                 C.POINTER(C.c_uint64)]
            L.hb_frames_free.argtypes = [C.c_void_p]
            L.hb_guess_chunk_records.argtypes = [C.c_uint64]
            L.hb_guess_chunk_records.restype = C.c_uint64
            L.hb_set_site_matcher.argtypes = [C.c_int]
            L.hb_set_site_matcher.restype = None
            L.hb_decode_frames.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_int, C.c_int]
            L.hb_decode_columns_device.argtypes = [C.c_void_p] * 4 + [C.c_uint64, C.c_uint32] + [C.c_void_p] * 8
            L.hb_decode_columns_device_large.argtypes = [C.c_void_p] * 4 + [C.c_uint64, C.c_uint32] + [C.c_void_p] * 8
        L.hb_encode_haplotypes.argtypes = [C.POINTER(HapBatch)]
        L.hb_synth_body_bytes.argtypes = [C.POINTER(SynthSpec)]
        L.hb_synth_body_bytes.restype = C.c_uint64
        L.hb_synth_header.argtypes = [C.POINTER(SynthSpec), C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.hb_synth_device.argtypes = [C.POINTER(SynthSpec), C.c_void_p, C.c_uint64, C.c_int, C.c_void_p]
        L.hb_synth_host.argtypes = [C.POINTER(SynthSpec), C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint64,
                                    C.POINTER(C.c_uint64)]
        _lib = L
    return _lib


def check(rc: int):
    if rc != 0:
        raise HaploError(rc, lib().hb_last_error().decode(errors="replace"))


def kernel_launches() -> int:
    return int(lib().hb_kernel_launches())


def _columns(samples) -> np.ndarray:
    """Column indices of a text-level sample subset as the C ABI takes them (the library checks them)."""
    return np.ascontiguousarray(np.asarray(list(samples), dtype=np.int64).astype(np.uint32))


def _names(samples):
    """(encoded names, const char *[] over them) of a file-level sample subset."""
    names = [s.encode() if isinstance(s, str) else bytes(s) for s in samples]
    return names, (C.c_char_p * max(1, len(names)))(*names)


def file_sample_names(path: str):
    """The header's sample names of a .vcf / .vcf.gz / .bcf, read from its leading bytes only (hb_file_samples; host only)."""
    n, ln = C.c_uint32(), C.c_uint64()
    check(lib().hb_file_samples(path.encode(), C.byref(n), None, 0, C.byref(ln)))
    buf = C.create_string_buffer(max(1, ln.value))
    check(lib().hb_file_samples(path.encode(), C.byref(n), buf, ln.value, C.byref(ln)))
    return [x.decode() for x in buf.raw[:ln.value].split(b"\0")[:n.value]]


# ------------------------------------------------------------------------------------------------
class Parse:
    """Device-resident parse of decompressed VCF body text (section B of the C ABI)."""

    def __init__(self, handle):
        self._h = handle

    @classmethod
    def _opts(cls, n_samples, region, end_is_int, want_gt, device, tokenizer, stream):
        o = ParseOpts()
        o.n_samples = n_samples
        o.region = (region or "").encode()
        o.end_is_int = int(end_is_int)
        o.want_gt = int(want_gt)
        o.device = device
        o.tokenizer = tokenizer
        o.stream = stream
        return o

    @classmethod
    def from_host(cls, text, n_samples, region="", end_is_int=False, want_gt=True, device=0, tokenizer=0,
                  stream=None, nbytes=None, samples=None):
        """text: bytes / numpy uint8 array / raw host address (with nbytes).  samples: column indices of a sample subset
        (ascending, distinct; hb_parse_host_text_subset), None = every sample."""
        if isinstance(text, (bytes, bytearray)):
            keep = np.frombuffer(text, np.uint8)
            addr, n = keep.ctypes.data, keep.size
        elif isinstance(text, np.ndarray):
            addr, n, keep = text.ctypes.data, text.size, text
        else:
            addr, n, keep = int(text), int(nbytes), None
        h = C.c_void_p()
        o = cls._opts(n_samples, region, end_is_int, want_gt, device, tokenizer, stream)
        if samples is None:
            check(lib().hb_parse_host_text(addr, n, C.byref(o), C.byref(h)))
        else:
            cols = _columns(samples)
            check(lib().hb_parse_host_text_subset(addr, n, C.byref(o), cols.ctypes.data, cols.size, C.byref(h)))
        del keep
        return cls(h)

    @classmethod
    def from_device(cls, d_ptr: int, nbytes: int, n_samples, region="", end_is_int=False, want_gt=True, device=0,
                    tokenizer=0, stream=None, samples=None):
        """samples: column indices of a sample subset (hb_parse_device_text_subset), None = every sample."""
        h = C.c_void_p()
        o = cls._opts(n_samples, region, end_is_int, want_gt, device, tokenizer, stream)
        if samples is None:
            check(lib().hb_parse_device_text(d_ptr, nbytes, C.byref(o), C.byref(h)))
        else:
            cols = _columns(samples)
            check(lib().hb_parse_device_text_subset(d_ptr, nbytes, C.byref(o), cols.ctypes.data, cols.size, C.byref(h)))
        return cls(h)

    @classmethod
    def from_file(cls, path: str, region="", want_gt=True, device=0, samples=None):
        """samples: names of a sample subset, in any order (hb_parse_file_subset; the planes come in header order), None =
        every sample."""
        h = C.c_void_p()
        if samples is None:
            check(lib().hb_parse_file(path.encode(), (region or "").encode(), int(want_gt), device, C.byref(h)))
        else:
            names, arr = _names(samples)
            check(lib().hb_parse_file_subset(path.encode(), (region or "").encode(), arr, len(names), device, C.byref(h)))
        return cls(h)

    @classmethod
    def from_vcf_bytes(cls, data, region="", want_gt=True, device=0, nbytes=None, index=None, samples=None):
        """The bytes of a .vcf / .vcf.gz / .bcf in host memory (bytes, uint8 array, or address + nbytes).  index: the bytes
        of its .tbi / .csi; a region query then inflates only the BGZF members the index lists for the region.  samples:
        names of a sample subset, as for from_file."""
        if isinstance(data, (bytes, bytearray)):
            keep = np.frombuffer(data, np.uint8); addr, n = keep.ctypes.data, keep.size
        elif isinstance(data, np.ndarray):
            keep = data; addr, n = data.ctypes.data, data.size
        else:
            keep = None; addr, n = int(data), int(nbytes)
        h = C.c_void_p()
        ix = None if index is None else np.frombuffer(bytes(index), np.uint8)
        if samples is not None:
            names, arr = _names(samples)
            check(lib().hb_parse_vcf_bytes_subset(addr, n, None if ix is None else ix.ctypes.data, 0 if ix is None else ix.size,
                                                  (region or "").encode(), arr, len(names), device, C.byref(h)))
        elif ix is None:
            check(lib().hb_parse_vcf_bytes(addr, n, (region or "").encode(), int(want_gt), device, C.byref(h)))
        else:
            check(lib().hb_parse_vcf_bytes_indexed(addr, n, ix.ctypes.data, ix.size, (region or "").encode(), int(want_gt),
                                                   device, C.byref(h)))
        del keep
        return cls(h)

    @classmethod
    def from_vcf_bytes_streamed(cls, data, region="", want_gt=True, device=0, slab_bytes=0, nbytes=None):
        """BGZF bytes of a .vcf.gz -> the same resident parse as from_vcf_bytes, but the text passes through HBM slab by slab
        (hb_parse_stream_bgzf_resident).  Returns (Parse, n_slabs)."""
        if isinstance(data, (bytes, bytearray)):
            keep = np.frombuffer(data, np.uint8); addr, n = keep.ctypes.data, keep.size
        elif isinstance(data, np.ndarray):
            keep = data; addr, n = data.ctypes.data, data.size
        else:
            keep = None; addr, n = int(data), int(nbytes)
        h, ns = C.c_void_p(), C.c_uint32()
        check(lib().hb_parse_stream_bgzf_resident(addr, n, (region or "").encode(), int(want_gt), device, slab_bytes, C.byref(h), C.byref(ns)))
        del keep
        return cls(h), int(ns.value)

    def sample_names(self):
        n, ln = C.c_uint32(), C.c_uint64()
        check(lib().hb_parse_samples(self._h, C.byref(n), None, 0, C.byref(ln)))
        buf = C.create_string_buffer(max(1, ln.value))
        check(lib().hb_parse_samples(self._h, C.byref(n), buf, ln.value, C.byref(ln)))
        return [x.decode() for x in buf.raw[:ln.value].split(b"\0")[:n.value]]

    def rerun(self):
        check(lib().hb_parse_rerun(self._h))

    @property
    def info(self) -> ParseInfo:
        i = ParseInfo()
        check(lib().hb_parse_get_info(self._h, C.byref(i)))
        return i

    @property
    def index_info(self):
        """(used, compressed_bytes_read, n_chunks) of a region query through an index (hb_parse_index_info)."""
        used, nread, nch = C.c_int(), C.c_uint64(), C.c_uint64()
        check(lib().hb_parse_index_info(self._h, C.byref(used), C.byref(nread), C.byref(nch)))
        return bool(used.value), int(nread.value), int(nch.value)

    def sites(self):
        n = self.info.n_records
        start, stop = np.empty(n, np.uint32), np.empty(n, np.uint32)
        ref, alt = np.empty(n, "S1"), np.empty(n, "S1")
        check(lib().hb_parse_fetch_sites(self._h, start.ctypes.data, stop.ctypes.data, ref.ctypes.data, alt.ctypes.data))
        return start, stop, ref, alt

    def sample(self, s: int):
        n = self.info.n_records
        g0, g1 = np.empty(n, np.int8), np.empty(n, np.int8)
        check(lib().hb_parse_fetch_sample(self._h, s, g0.ctypes.data, g1.ctypes.data))
        return g0, g1

    def matrix(self):
        i = self.info
        g0 = np.empty((i.n_samples, i.n_records), np.int8)
        g1 = np.empty((i.n_samples, i.n_records), np.int8)
        check(lib().hb_parse_fetch_matrix(self._h, g0.ctypes.data, g1.ctypes.data))
        return g0, g1

    def sample_errors(self):
        ns = self.info.n_samples
        pl, bg = np.zeros(ns, np.uint32), np.zeros(ns, np.uint32)
        check(lib().hb_parse_fetch_sample_errors(self._h, pl.ctypes.data, bg.ctypes.data))
        return pl, bg

    def chrom_runs(self):
        n = C.c_uint64()
        ln = C.c_uint64()
        check(lib().hb_parse_chrom_runs(self._h, C.byref(n), None, 0, None, 0, C.byref(ln)))
        rows = np.zeros(max(1, n.value), np.uint64)
        names = C.create_string_buffer(max(1, ln.value))
        check(lib().hb_parse_chrom_runs(self._h, C.byref(n), rows.ctypes.data, n.value, names, ln.value, C.byref(ln)))
        nm = names.raw[:ln.value].split(b"\0")[:n.value]
        return [int(r) for r in rows[:n.value]], [x.decode() for x in nm]

    def chrom_column(self):
        rows, names = self.chrom_runs()
        n = self.info.n_records
        out = []
        for k, r in enumerate(rows):
            e = rows[k + 1] if k + 1 < len(rows) else n
            out.extend([names[k]] * (e - r))
        return out

    def attach(self, frames: "Frames | None"):
        """Overlap the frames' site-template kernel with the GT decoder on every rerun (hb_parse_attach_frames)."""
        check(lib().hb_parse_attach_frames(self._h, frames._h if frames is not None else None))

    def compress(self, chunk_records: int = 0, s0: int = 0, ns: int | None = None) -> "Frames":
        """Blosc frames of samples [s0, s0 + ns) (default: all)."""
        h = C.c_void_p()
        if ns is None and s0 == 0:
            check(lib().hb_compress_records(self._h, chunk_records, C.byref(h)))
        else:
            check(lib().hb_compress_sample_range(self._h, chunk_records, s0, self.info.n_samples - s0 if ns is None else ns, C.byref(h)))
        return Frames(h)

    def release_text(self):
        check(lib().hb_parse_release_text(self._h))

    def close(self):
        if self._h:
            lib().hb_parse_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Frames:
    """Stored HDF5 chunks = bare Blosc chunks (one per sample per HDF5 chunk), device resident (section C)."""

    def __init__(self, handle):
        self._h = handle

    @property
    def info(self) -> FramesInfo:
        i = FramesInfo()
        check(lib().hb_frames_get_info(self._h, C.byref(i)))
        return i

    def rerun(self, parse: "Parse"):
        check(lib().hb_frames_rerun(self._h, parse._h))

    def set_window(self, s0: int, ns: int):
        """Move the sample window (ns <= the window the frames were made for); then rerun(parse)."""
        check(lib().hb_frames_set_window(self._h, s0, ns))

    def layout(self):
        """(offsets uint64 [n_samples, n_chunks] into the frame buffer, sizes uint32 [n_samples, n_chunks])"""
        i = self.info
        offs = np.zeros((i.n_samples, i.n_chunks), np.uint64)
        sizes = np.zeros((i.n_samples, i.n_chunks), np.uint32)
        check(lib().hb_frames_layout(self._h, offs.ctypes.data, sizes.ctypes.data))
        return offs, sizes

    def fetch_all(self) -> np.ndarray:
        """The whole device frame buffer (frames 16-byte aligned, [sample][chunk] order) in one D2H copy."""
        buf = np.empty(max(1, self.info.padded_bytes), np.uint8)
        check(lib().hb_frames_fetch_all(self._h, buf.ctypes.data, buf.size))
        return buf[:self.info.padded_bytes]

    def fetch_packed(self, out=None):
        """All frames back to back (16-byte aligned), [sample][chunk] order: (buf uint8, offsets uint64 [n_samples, n_chunks]
        into buf, sizes uint32 [n_samples, n_chunks]).  out: a pre-allocated uint8 array / (address, capacity) to fill (e.g.
        pinned memory), else a new numpy array."""
        i = self.info
        offs = np.empty((i.n_samples, i.n_chunks), np.uint64)
        sizes = np.empty((i.n_samples, i.n_chunks), np.uint32)
        tot = C.c_uint64()
        if out is None:                                   # how many bytes?  then one more call for the data
            check(lib().hb_frames_fetch_packed(self._h, None, 0, None, None, C.byref(tot)))
            out = np.empty(max(1, tot.value), np.uint8)
        addr, cap = (out.ctypes.data, out.size) if isinstance(out, np.ndarray) else (int(out[0]), int(out[1]))
        check(lib().hb_frames_fetch_packed(self._h, addr, cap, offs.ctypes.data, sizes.ctypes.data, C.byref(tot)))
        return (out[:tot.value] if isinstance(out, np.ndarray) else tot.value), offs, sizes

    def sample(self, s: int):
        i = self.info
        sizes = np.zeros(max(1, i.n_chunks), np.uint64)
        tot = C.c_uint64()
        check(lib().hb_frames_fetch_sample(self._h, s, sizes.ctypes.data, None, 0, C.byref(tot)))
        buf = np.empty(max(1, tot.value), np.uint8)
        check(lib().hb_frames_fetch_sample(self._h, s, sizes.ctypes.data, buf.ctypes.data, buf.size, C.byref(tot)))
        out, o = [], 0
        for k in range(i.n_chunks):
            out.append(buf[o:o + int(sizes[k])].tobytes())
            o += int(sizes[k])
        return out

    def close(self):
        if self._h:
            lib().hb_frames_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ------------------------------------------------------------------------------------------------
def parse_stream_host(text, n_samples, capacity, region="", end_is_int=False, want_gt=True, device=0, tokenizer=0,
                      slab_bytes=0):
    """hb_parse_stream_host on a bytes / uint8 array: returns a dict of numpy arrays trimmed to n_records."""
    keep = np.frombuffer(text, np.uint8) if isinstance(text, (bytes, bytearray)) else text
    o = Parse._opts(n_samples, region, end_is_int, want_gt, device, tokenizer, None)
    g0 = np.empty((n_samples, capacity), np.int8)
    g1 = np.empty((n_samples, capacity), np.int8)
    start, stop = np.empty(capacity, np.uint32), np.empty(capacity, np.uint32)
    ref, alt = np.empty(capacity, "S1"), np.empty(capacity, "S1")
    pl, bg = np.zeros(max(1, n_samples), np.uint32), np.zeros(max(1, n_samples), np.uint32)
    n, ns = C.c_uint64(), C.c_uint32()
    check(lib().hb_parse_stream_host(keep.ctypes.data, keep.size, C.byref(o), slab_bytes, g0.ctypes.data, g1.ctypes.data,
                                     capacity, start.ctypes.data, stop.ctypes.data, ref.ctypes.data, alt.ctypes.data,
                                     pl.ctypes.data, bg.ctypes.data, C.byref(n), C.byref(ns)))
    k = int(n.value)
    return {"n": k, "n_slabs": int(ns.value), "gt0": g0[:, :k], "gt1": g1[:, :k], "start": start[:k], "stop": stop[:k],
            "ref": ref[:k], "alt": alt[:k], "ploidy_err": pl[:n_samples], "badgt_err": bg[:n_samples]}


def bgzf_vcf_info(data):
    """(n_samples, decompressed bytes, offset of the first record) of the BGZF bytes of a .vcf.gz"""
    keep = np.frombuffer(data, np.uint8) if isinstance(data, (bytes, bytearray)) else data
    ns, tb, bo = C.c_uint32(), C.c_uint64(), C.c_uint64()
    check(lib().hb_bgzf_vcf_info(keep.ctypes.data, keep.size, C.byref(ns), C.byref(tb), C.byref(bo)))
    return int(ns.value), int(tb.value), int(bo.value)


def parse_stream_bgzf_host(data, capacity, region="", want_gt=True, device=0, slab_bytes=0, out=None):
    """hb_parse_stream_bgzf_host on the BGZF bytes of a .vcf.gz (bytes / uint8 array, ideally pinned): a dict of numpy
    arrays trimmed to n_records.  out: pre-allocated (gt0, gt1, start, stop, ref, alt) to write into (e.g. pinned)."""
    keep = np.frombuffer(data, np.uint8) if isinstance(data, (bytes, bytearray)) else data
    n_samples, _, _ = bgzf_vcf_info(keep)
    if out is None:
        g0 = np.empty((n_samples, capacity), np.int8)
        g1 = np.empty((n_samples, capacity), np.int8)
        start, stop = np.empty(capacity, np.uint32), np.empty(capacity, np.uint32)
        ref, alt = np.empty(capacity, "S1"), np.empty(capacity, "S1")
    else:
        g0, g1, start, stop, ref, alt = out
    pl, bg = np.zeros(max(1, n_samples), np.uint32), np.zeros(max(1, n_samples), np.uint32)
    n, ns = C.c_uint64(), C.c_uint32()
    check(lib().hb_parse_stream_bgzf_host(keep.ctypes.data, keep.size, (region or "").encode(), int(want_gt), device, slab_bytes,
                                          g0.ctypes.data, g1.ctypes.data, capacity, start.ctypes.data, stop.ctypes.data,
                                          ref.ctypes.data, alt.ctypes.data, pl.ctypes.data, bg.ctypes.data, C.byref(n), C.byref(ns)))
    k = int(n.value)
    return {"n": k, "n_samples": n_samples, "n_slabs": int(ns.value), "gt0": g0[:, :k], "gt1": g1[:, :k], "start": start[:k],
            "stop": stop[:k], "ref": ref[:k], "alt": alt[:k], "ploidy_err": pl[:n_samples], "badgt_err": bg[:n_samples]}


def load_vcf_columns(path: str, sample: str, chrom: str = ""):
    """hb_load_vcf / hb_load_vcf_without_sample through ctypes, columnar."""
    r = Records()
    if sample:
        check(lib().hb_load_vcf(path.encode(), sample.encode(), (chrom or "").encode(), C.byref(r)))
    else:
        check(lib().hb_load_vcf_without_sample(path.encode(), (chrom or "").encode(), C.byref(r)))
    try:
        n = int(r.n)
        pool = C.string_at(r.chrom_pool, int(r.chrom_pool_len)) if r.chrom_pool_len else b""
        offs = np.ctypeslib.as_array(r.chrom_off, (n,)).copy() if n else np.zeros(0, np.uint32)
        names = {int(o): pool[int(o):pool.index(b"\0", int(o))].decode() for o in np.unique(offs)}
        d = {
            "n": n, "n_samples": int(r.n_samples),
            "chrom": [names[int(o)] for o in offs],
            "start": np.ctypeslib.as_array(r.start, (n,)).copy() if n else np.zeros(0, np.uint32),
            "stop": np.ctypeslib.as_array(r.stop, (n,)).copy() if n else np.zeros(0, np.uint32),
            "ref": np.frombuffer(C.string_at(r.ref, n), "S1").copy() if n else np.zeros(0, "S1"),
            "alt": np.frombuffer(C.string_at(r.alt, n), "S1").copy() if n else np.zeros(0, "S1"),
        }
        if sample:
            d["gt0"] = np.ctypeslib.as_array(r.gt0, (n,)).copy() if n else np.zeros(0, np.int8)
            d["gt1"] = np.ctypeslib.as_array(r.gt1, (n,)).copy() if n else np.zeros(0, np.int8)
        return d
    finally:
        lib().hb_records_free(C.byref(r))


def bgzf_compress_host(text, level: int = 6) -> np.ndarray:
    """text (bytes / uint8 array) -> BGZF bytes (uint8 array), stock zlib on all host threads (test / bench utility)."""
    src = np.frombuffer(text, np.uint8) if isinstance(text, (bytes, bytearray)) else text
    L = lib()
    n = C.c_uint64()
    check(L.hb_bgzf_compress_host(src.ctypes.data, src.size, level, None, 0, C.byref(n)))
    out = np.empty(n.value, np.uint8)
    check(L.hb_bgzf_compress_host(src.ctypes.data, src.size, level, out.ctypes.data, out.size, C.byref(n)))
    return out[:n.value]


def set_bgzf_crc_check(on: bool) -> None:
    """Check every BGZF member's CRC32 against its trailer, as htslib does (hb_set_bgzf_crc_check; process-wide, off by default)."""
    lib().hb_set_bgzf_crc_check(1 if on else 0)


def get_bgzf_crc_check() -> bool:
    return bool(lib().hb_get_bgzf_crc_check())


@contextlib.contextmanager
def crc_check(on: bool = True):
    """`with crc_check(): ...` runs the block with the BGZF CRC32 check set to `on` and restores the setting after it."""
    was = get_bgzf_crc_check()
    set_bgzf_crc_check(on)
    try:
        yield
    finally:
        set_bgzf_crc_check(was)


def set_use_index(on: bool) -> None:
    """Answer region queries through <file>.tbi / <file>.csi when one is there (hb_set_use_index; process-wide, on by default)."""
    lib().hb_set_use_index(1 if on else 0)


def get_use_index() -> bool:
    return bool(lib().hb_get_use_index())


@contextlib.contextmanager
def use_index(on: bool = True):
    """`with use_index(False): ...` runs the block with region queries through an index set to `on` and restores the setting."""
    was = get_use_index()
    set_use_index(on)
    try:
        yield
    finally:
        set_use_index(was)


INDEX_FORMATS = {"tbi": 0, "csi": 1}


def build_index(data, fmt: str = "tbi", min_shift: int = 14, device: int = 0) -> bytes:
    """The .tbi / .csi of BGZF bytes (a .vcf.gz, or a .bcf with fmt="csi"), built on the GPU (hb_index_bgzf): the bytes of
    the index file, BGZF-compressed."""
    src = np.frombuffer(bytes(data), np.uint8) if isinstance(data, (bytes, bytearray, memoryview)) else data
    n = C.c_uint64()
    cap = max(1 << 20, src.size // 8)
    out = np.empty(cap, np.uint8)
    rc = lib().hb_index_bgzf(src.ctypes.data, src.size, INDEX_FORMATS[fmt], min_shift, device, out.ctypes.data, cap, C.byref(n))
    if rc == 10 and n.value > cap:
        out = np.empty(n.value, np.uint8)
        rc = lib().hb_index_bgzf(src.ctypes.data, src.size, INDEX_FORMATS[fmt], min_shift, device, out.ctypes.data, out.size,
                                 C.byref(n))
    check(rc)
    return out[:n.value].tobytes()


def index_file(path: str, fmt: str = "tbi", min_shift: int = 14, device: int = 0, out_path: str | None = None) -> str:
    """Write the index of `path` (hb_index_file) to out_path, by default <path>.tbi / <path>.csi; returns where."""
    check(lib().hb_index_file(path.encode(), INDEX_FORMATS[fmt], min_shift, device, out_path.encode() if out_path else None))
    return out_path or path + "." + fmt


def bgzf_inflate(data: bytes, device: int = 0, with_ms: bool = False):
    """BGZF bytes -> text, inflated on the GPU (hb_bgzf_inflate)."""
    src = np.frombuffer(data, np.uint8)
    n = C.c_uint64()
    check(lib().hb_bgzf_inflate(src.ctypes.data, src.size, None, 0, C.byref(n), device, None))
    out = np.empty(max(1, n.value), np.uint8)
    ms = C.c_float()
    check(lib().hb_bgzf_inflate(src.ctypes.data, src.size, out.ctypes.data, out.size, C.byref(n), device, C.byref(ms)))
    text = out[:n.value].tobytes()
    return (text, float(ms.value)) if with_ms else text


def decode_frames(frames, chunk_nbytes: int, planar: bool = False, device: int = 0) -> np.ndarray:
    """Stored HDF5 chunks (bare Blosc chunks, filter 32001) -> uint8 [n_frames, chunk_nbytes], decoded on the GPU."""
    n = len(frames)
    out = np.empty((n, chunk_nbytes), np.uint8)
    if n == 0:
        return out
    offs = np.zeros(n + 1, np.uint64)
    offs[1:] = np.cumsum([len(f) for f in frames])
    blob = np.frombuffer(b"".join(bytes(f) for f in frames), np.uint8)
    check(lib().hb_decode_frames(blob.ctypes.data, offs.ctypes.data, n, chunk_nbytes, out.ctypes.data, int(planar), device))
    return out


def synth_spec(n_variants, n_samples, seed=42, chrom="chr22", first_pos=10_000_000, pos_step=35, mix=0) -> SynthSpec:
    s = SynthSpec()
    s.n_variants, s.n_samples, s.seed = n_variants, n_samples, seed
    s.first_pos, s.pos_step, s.mix = first_pos, pos_step, mix
    s.chrom = chrom.encode()
    return s


def synth_header(spec: SynthSpec) -> bytes:
    ln = C.c_uint64()
    check(lib().hb_synth_header(C.byref(spec), None, 0, C.byref(ln)))
    buf = C.create_string_buffer(ln.value)
    check(lib().hb_synth_header(C.byref(spec), buf, ln.value, C.byref(ln)))
    return buf.raw[:ln.value]


def synth_host(spec: SynthSpec, first=0, n=None) -> bytes:
    n = spec.n_variants - first if n is None else n
    ln = C.c_uint64()
    check(lib().hb_synth_host(C.byref(spec), first, n, None, 0, C.byref(ln)))
    buf = np.empty(max(1, ln.value), np.uint8)
    check(lib().hb_synth_host(C.byref(spec), first, n, buf.ctypes.data, buf.size, C.byref(ln)))
    return buf[:ln.value].tobytes()


def synth_sample_names(spec: SynthSpec):
    return ["S%06d" % k for k in range(spec.n_samples)]
