"""HDF5 container access for the reference's on-disk layout (vcf_to_h5.py:131-135, h5_reader.py:37-41).

    {cohort}.h5 / donor_{id} / chr_{N} / snp_data     1-D, 35-byte compound, chunked, filter 32001

Two backends behind one small interface (`open_h5`):

  * h5py + hdf5plugin when both import: GPU-compressed Blosc chunks enter the file through HDF5's
    direct-chunk-write call (`dset.id.write_direct_chunk`), which stores pre-filtered bytes without
    running the filter; reads pull the stored chunks with `read_direct_chunk`.  (Neither package is
    in this image, so this branch has not been run here -- see DESIGN.md.)
  * otherwise `minih5`, this repo's own writer/reader of the same HDF5 structures.

Either way the chunk payloads are bare Blosc1 chunks (what hdf5-blosc, filter 32001, stores), produced by kernel 4 (`hb_compress_records`) on the
way in and decoded by `hb_decode_frames` on the way out: no CPU codec is involved in the product path.
"""
from __future__ import annotations

import numpy as np

from . import minih5

FILTER_BLOSC = 32001
# what the reference passes (vcf_to_h5.py:135); the filter's set_local overwrites slots 0-3 with
# (filter revision, Blosc format version, typesize, chunk bytes) before they reach the file
BLOSC_OPTS = (2, 2, 0, 0, 5, 1, 2)


def _cd_values(itemsize: int, chunk_nbytes: int):
    return (BLOSC_OPTS[0], BLOSC_OPTS[1], itemsize, chunk_nbytes) + BLOSC_OPTS[4:]


def have_h5py() -> bool:
    try:
        import h5py  # noqa: F401
        import hdf5plugin  # noqa: F401
        return True
    except Exception:
        return False


def _decode(frames, dtype: np.dtype, n: int, chunk: int) -> np.ndarray:
    from . import capi
    raw = capi.decode_frames(frames, chunk * dtype.itemsize)
    return raw.reshape(-1).view(dtype)[:n].copy()


def _decode_masked(chunks, dtype: np.dtype, n: int, chunk: int) -> np.ndarray:
    """chunks: [(stored bytes, filter mask)] of a dataset behind the Blosc filter alone.  A chunk with mask bit 0 set was
    stored unfiltered (hdf5-blosc gives c-blosc an output buffer of the chunk's size, so a chunk Blosc cannot shrink,
    e.g. one of 1-3 records, fails the optional filter): its bytes are the records.  The others decode on the GPU."""
    from . import capi
    nbytes = chunk * dtype.itemsize
    if not any(m & 1 for _, m in chunks):
        return _decode([b for b, _ in chunks], dtype, n, chunk)
    out = np.zeros((len(chunks), nbytes), np.uint8)
    blosc = [k for k, (_, m) in enumerate(chunks) if not m & 1]
    if blosc:
        out[blosc] = capi.decode_frames([chunks[k][0] for k in blosc], nbytes)
    for k, (b, m) in enumerate(chunks):
        if m & 1:
            if len(b) != nbytes:
                raise OSError(f"unfiltered chunk {k} holds {len(b)} bytes, not {nbytes}")
            out[k] = np.frombuffer(b, np.uint8)
    return out.reshape(-1).view(dtype)[:n].copy()


class _MiniFile:
    backend = "minih5"

    def __init__(self, path: str, mode: str):
        self.mode = mode
        self._w = minih5.H5Writer(path) if mode == "w" else None
        self._r = minih5.H5Reader(path) if mode == "r" else None

    # ---- write
    def write_chunked(self, path: str, dtype, n: int, chunk: int, frames):
        dtype = np.dtype(dtype)
        self._w.create_dataset_chunked(path, dtype, n, chunk, frames, filter_id=FILTER_BLOSC,
                                       cd_values=_cd_values(dtype.itemsize, chunk * dtype.itemsize), filter_name="blosc")

    def write_frames_bulk(self, paths, dtype, n: int, chunk: int, buf: np.ndarray, offsets: np.ndarray, sizes: np.ndarray):
        """Many datasets at once: `buf` (all their stored chunks, e.g. hb_frames_fetch_all) goes into the file with ONE
        write; dataset i = chunks sizes[i, k] bytes at buf offset offsets[i, k].  No per-chunk Python work."""
        dtype = np.dtype(dtype)
        base = self._w.write_blob(buf)
        cd = _cd_values(dtype.itemsize, chunk * dtype.itemsize)
        for i, path in enumerate(paths):
            self._w.create_dataset_chunked_at(path, dtype, n, chunk, np.uint64(base) + offsets[i].astype(np.uint64), sizes[i],
                                              filter_id=FILTER_BLOSC, cd_values=cd, filter_name="blosc")

    def write_array(self, path: str, data: np.ndarray):
        self._w.create_dataset_contiguous(path, np.asarray(data))

    # ---- read
    def __contains__(self, path: str) -> bool:
        return path in self._r

    def keys(self, path: str = "/"):
        return self._r.keys(path)

    def read_dataset(self, path: str) -> np.ndarray:
        info = self._r.dataset_info(path)
        if info.layout == "contiguous":
            return self._r.read_contiguous(info)
        n = int(info.shape[0])
        stored = self._r.chunks_with_masks(info)
        if not info.filters:
            raw = b"".join(b for _, b, _ in stored)
            return np.frombuffer(raw, info.dtype)[:n].copy()
        if [f for f, _ in info.filters] != [FILTER_BLOSC]:
            raise OSError(f"{path}: unsupported filter pipeline {info.filters}")
        return _decode_masked([(b, m) for _, b, m in stored], info.dtype, n, info.chunk)

    def stored_chunks(self, path: str):
        """The dataset as it is stored: (n_records, chunk_records, dtype, [stored chunk bytes in order]) -- no decoding.
        None for a dataset that is not a 1-D chunked array behind filter 32001 alone, or that holds a chunk HDF5 stored
        unfiltered (filter mask bit 0: the optional Blosc filter failed on it); read_dataset reads those."""
        info = self._r.dataset_info(path)
        if info.layout == "contiguous" or [f for f, _ in info.filters] != [FILTER_BLOSC]:
            return None
        stored = self._r.chunks_with_masks(info)
        if any(m & 1 for _, _, m in stored):
            return None
        return int(info.shape[0]), int(info.chunk), info.dtype, [b for _, b, _ in stored]

    def close(self):
        if self._w is not None:
            self._w.close()
        if self._r is not None:
            self._r.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


class _H5pyFile:
    backend = "h5py"

    def __init__(self, path: str, mode: str):
        import h5py
        import hdf5plugin  # noqa: F401  (registers filter 32001)
        self._f = h5py.File(path, mode)

    def write_chunked(self, path: str, dtype, n: int, chunk: int, frames):
        dtype = np.dtype(dtype)
        d = self._f.create_dataset(path, shape=(n,), dtype=dtype, chunks=(chunk,), compression=FILTER_BLOSC,
                                   compression_opts=BLOSC_OPTS)
        for k, payload in enumerate(frames):
            d.id.write_direct_chunk((k * chunk,), bytes(payload))

    def write_frames_bulk(self, paths, dtype, n: int, chunk: int, buf: np.ndarray, offsets: np.ndarray, sizes: np.ndarray):
        for i, path in enumerate(paths):
            self.write_chunked(path, dtype, n, chunk,
                               [buf[int(o):int(o) + int(z)].tobytes() for o, z in zip(offsets[i], sizes[i])])

    def write_array(self, path: str, data: np.ndarray):
        self._f.create_dataset(path, data=np.asarray(data))

    def __contains__(self, path: str) -> bool:
        return path in self._f

    def keys(self, path: str = "/"):
        return sorted(self._f[path].keys())

    def read_dataset(self, path: str) -> np.ndarray:
        d = self._f[path]
        if d.chunks is None or d.compression is None and not d.id.get_create_plist().get_nfilters():
            return d[()]
        chunk, n = d.chunks[0], d.shape[0]
        frames = [d.id.read_direct_chunk((off,)) for off in range(0, n, chunk)]       # (filter mask, stored bytes)
        return _decode_masked([(b, m) for m, b in frames], d.dtype, n, chunk)

    def stored_chunks(self, path: str):
        d = self._f[path]
        pl = d.id.get_create_plist()
        if d.chunks is None or d.ndim != 1 or pl.get_nfilters() != 1 or pl.get_filter(0)[0] != FILTER_BLOSC:
            return None
        chunk, n = d.chunks[0], d.shape[0]
        frames = [d.id.read_direct_chunk((off,)) for off in range(0, n, chunk)]
        if any(m & 1 for m, _ in frames):
            return None
        return int(n), int(chunk), d.dtype, [b for _, b in frames]

    def close(self):
        self._f.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def open_h5(path: str, mode: str = "r", backend: str | None = None):
    """mode 'r' or 'w'.  backend: None (h5py when importable, else minih5), 'h5py' or 'minih5'."""
    if mode not in ("r", "w"):
        raise ValueError("mode must be 'r' or 'w'")
    if backend is None:
        backend = "h5py" if have_h5py() else "minih5"
    if backend == "h5py":
        return _H5pyFile(path, mode)
    if backend == "minih5":
        return _MiniFile(path, mode)
    raise ValueError(f"unknown backend {backend}")
