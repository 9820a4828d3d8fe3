"""ctypes binding of the C ABI in include/cbcg.h (cbc_b200/_build/libcbcg.so).

Python mirror of the reference's seams for the aligned-read coding path (SURVEY.md 8b):
``Codec.compress`` / ``Codec.decompress`` stand where ``compress()`` / ``decompress()``
(src/compression.c:112-216) stand in the reference, over SoA batches instead of SAM text.
There is no CPU path: a missing library or GPU raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Tuple

import numpy as np

from .batch import Batch, CBatch, Genome

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CBCG_LIB") or os.path.join(_HERE, "_build", "libcbcg.so")   # CBCG_LIB: tuning builds only

REC_DTYPE = np.dtype([("pos", "<u4"), ("flag", "<u2"), ("len", "<u2"), ("edit_off", "<u4"),
                      ("match", "u1"), ("n_snps", "u1"), ("n_dels", "u1"), ("n_ins", "u1")])
SYM_DTYPE = np.dtype([("key", "<u4"), ("value", "<u4")])

class CBatchCompact(C.Structure):
    """Mirror of ``cbcg_batch_compact`` (include/cbcg.h): the form of a batch that crosses the host-device link."""
    _fields_ = [("n_reads", C.c_uint64), ("pos", C.c_void_p), ("flag", C.c_void_p), ("seq_len", C.c_void_p),
                ("cigar_len", C.c_void_p), ("md_len", C.c_void_p), ("n_runs", C.c_uint32), ("pad", C.c_uint32),
                ("run_first", C.c_void_p), ("run_chr", C.c_void_p), ("seq2", C.c_void_p), ("n_exc", C.c_uint64),
                ("exc_read", C.c_void_p), ("exc_base", C.c_void_p), ("exc_char", C.c_void_p), ("cigar", C.c_void_p),
                ("md", C.c_void_p), ("tile_base", C.c_void_p), ("max_len", C.c_uint32), ("min_len", C.c_uint32)]


class _CbchCompact(C.Structure):
    """Mirror of ``cbch_compact`` (csrc/host/sam_ingest.h)."""
    _fields_ = [("v", CBatchCompact), ("alloc", C.c_void_p), ("release", C.c_void_p), ("bytes", C.c_uint64)]


EXPORTS = ["cbcg_create", "cbcg_destroy", "cbcg_strerror", "cbcg_last_error", "cbcg_abi_version", "cbcg_get_stats",
           "cbcg_host_alloc", "cbcg_host_free", "cbcg_set_reference", "cbcg_extract", "cbcg_extract_symbols",
           "cbcg_encode", "cbcg_encode_bound", "cbcg_decode", "cbcg_decoded_size", "cbcg_decode_edits",
           "cbcg_reconstruct", "cbcg_batch_upload", "cbcg_encode_resident", "cbcg_decode_resident",
           "cbcg_fetch_container", "cbcg_fetch_decoded", "cbcg_fetch_index", "cbcg_mark", "cbcg_elapsed_ms",
           "cbcg_encode_compact", "cbcg_batch_upload_compact", "cbcg_cigar_bound", "cbcg_cigar_pack", "cbcg_cigar_unpack",
           "cbcg_region_plan", "cbcg_decode_region", "cbcg_sam_header", "cbcg_decode_sam", "cbcg_derive_md",
           "cbcg_pileup", "cbcg_bam_header", "cbcg_decode_bam", "cbcg_bgzf_inflate", "cbcg_bam_open", "cbcg_batch_upload_bam",
           "cbcg_cigar_pack_resident"]


UINT64_MAX = (1 << 64) - 1
PILEUP_COLUMNS = ("A", "C", "G", "T", "N", "DEL", "INS", "REF")      # CBCG_PU_A .. CBCG_PU_REF
PILEUP_FLAG_EXCLUDE = 0x704                                          # UNMAP | SECONDARY | QCFAIL | DUP
BAM_HEADER, BAM_EOF = 1, 2                                           # CBCG_BAM_HEADER, CBCG_BAM_EOF
BAM_DERIVE_MD, BAM_LAST = 1, 2                                       # CBCG_BAM_DERIVE_MD, CBCG_BAM_LAST
BLOCK_AUTO = 0xFFFFFFFF                                              # CBCG_BLOCK_AUTO


class BamInfo(C.Structure):
    """Mirror of ``cbcg_bam_info`` (include/cbcg.h)."""
    _fields_ = [("n_records", C.c_uint64), ("n_unmapped", C.c_uint64), ("n_reads", C.c_uint64), ("len_first", C.c_uint32),
                ("len_second", C.c_uint32), ("max_len", C.c_uint32), ("min_len", C.c_uint32), ("inflated_bytes", C.c_uint64),
                ("tail_len", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class Region(C.Structure):
    """Mirror of ``cbcg_region`` (include/cbcg.h): 1-based, both ends inclusive; end UINT64_MAX = to the end of the record."""
    _fields_ = [("name", C.c_char_p), ("start", C.c_uint64), ("end", C.c_uint64)]


def _region_array(regions):
    """(name,), (name, start) or (name, start, end) tuples -> a ctypes array of Region (the names stay referenced by it)."""
    regions = list(regions)
    arr = (Region * max(len(regions), 1))()
    for k, r in enumerate(regions):
        name = r[0].encode() if isinstance(r[0], str) else bytes(r[0])
        start = int(r[1]) if len(r) > 1 else 1
        end = int(r[2]) if len(r) > 2 else UINT64_MAX
        arr[k] = Region(name, start, end)
    return arr, len(regions)


def region_plan(data: bytes, regions, legacy: bool = False) -> dict:
    """What ``Codec.decompress_region`` would decode, from the container's header and block index alone (no device):
    n_blocks, n_reads (decoded, not returned), payload_bytes read and max_seq_bytes (a bound on the text returned).
    A legacy stream does not store its read count: n_reads and max_seq_bytes are UINT64_MAX there."""
    lib = load_library()
    src = np.frombuffer(data, np.uint8)
    arr, n = _region_array(regions)
    out = [C.c_uint64(0) for _ in range(4)]
    rc = lib.cbcg_region_plan(src.ctypes.data, src.nbytes, int(legacy), arr, n, *[C.byref(v) for v in out])
    if rc:
        raise CbcgError(rc, lib.cbcg_strerror(rc).decode())
    return dict(zip(("n_blocks", "n_reads", "payload_bytes", "max_seq_bytes"), (v.value for v in out)))


def sam_header(data: bytes) -> bytes:
    """@HD and one @SQ line per chromosome of a blocked container's table, from its header alone (no device). The
    container does not store record lengths, so the @SQ lines carry no LN (``Codec.decompress_sam`` adds it from the
    loaded reference)."""
    lib = load_library()
    src = np.frombuffer(data, np.uint8)
    n = C.c_uint64(0)
    rc = lib.cbcg_sam_header(src.ctypes.data, src.nbytes, None, 0, C.byref(n))
    out = np.empty(max(n.value, 1), np.uint8)
    if rc == -5:
        rc = lib.cbcg_sam_header(src.ctypes.data, src.nbytes, out.ctypes.data, out.nbytes, C.byref(n))
    if rc:
        raise CbcgError(rc, lib.cbcg_strerror(rc).decode())
    return out[:n.value].tobytes()


class EncodeOpts(C.Structure):
    _fields_ = [("read_len_header", C.c_uint32), ("block_reads", C.c_uint32), ("gen_mode", C.c_uint32),
                ("substreams", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [("ms_h2d", C.c_float), ("ms_extract", C.c_float), ("ms_plan", C.c_float), ("ms_code", C.c_float),
                ("ms_gather", C.c_float), ("ms_reconstruct", C.c_float), ("ms_d2h", C.c_float), ("ms_total", C.c_float),
                ("ms_k1", C.c_float), ("ms_k3", C.c_float),
                ("n_reads", C.c_uint64), ("n_blocks", C.c_uint64), ("n_symbols", C.c_uint64), ("n_edits", C.c_uint64),
                ("payload_bytes", C.c_uint64), ("container_bytes", C.c_uint64),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("kernel_launches", C.c_uint32), ("retried", C.c_uint32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class CbcgError(RuntimeError):
    def __init__(self, status: int, text: str):
        super().__init__(f"cbcg status {status}: {text}")
        self.status = status


_LIB = None


def load_library():
    """Loads libcbcg.so; raises (never falls back) when it has not been built."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: build it with `make cuda` or __graft_entry__.build(); "
                               "there is no CPU implementation of this path")
        lib = C.CDLL(LIB_PATH)
        vp, u64, u32 = C.c_void_p, C.c_uint64, C.c_uint32
        P = C.POINTER
        lib.cbcg_create.argtypes = [C.c_int, P(vp)]
        lib.cbcg_destroy.argtypes = [vp]; lib.cbcg_destroy.restype = None
        lib.cbcg_strerror.argtypes = [C.c_int]; lib.cbcg_strerror.restype = C.c_char_p
        lib.cbcg_last_error.argtypes = [vp]; lib.cbcg_last_error.restype = C.c_char_p
        lib.cbcg_get_stats.argtypes = [vp, P(Stats)]
        lib.cbcg_host_alloc.argtypes = [C.c_size_t]; lib.cbcg_host_alloc.restype = vp
        lib.cbcg_host_free.argtypes = [vp]; lib.cbcg_host_free.restype = None
        lib.cbcg_set_reference.argtypes = [vp, u32, vp, vp, vp]
        lib.cbcg_extract.argtypes = [vp, P(CBatch), vp, vp, u64, P(u64)]
        lib.cbcg_extract_symbols.argtypes = [vp, P(CBatch), P(EncodeOpts), vp, u64, P(u64), vp, u64, P(u64)]
        lib.cbcg_encode.argtypes = [vp, P(CBatch), P(EncodeOpts), vp, u64, P(u64)]
        lib.cbcg_encode_bound.argtypes = [P(CBatch), P(EncodeOpts)]; lib.cbcg_encode_bound.restype = u64
        lib.cbcg_decode.argtypes = [vp, vp, u64, C.c_int, vp, u64, P(u64), P(u64)]
        lib.cbcg_decoded_size.argtypes = [vp, u64, P(u64), P(u64)]
        lib.cbcg_decode_edits.argtypes = [vp, vp, u64, C.c_int, vp, u64, vp, vp, u64, P(u64), P(u64)]
        lib.cbcg_reconstruct.argtypes = [vp, u64, vp, vp, vp, u64, vp, u64, P(u64)]
        lib.cbcg_batch_upload.argtypes = [vp, P(CBatch)]
        lib.cbcg_batch_upload_compact.argtypes = [vp, P(CBatchCompact)]
        lib.cbcg_encode_compact.argtypes = [vp, P(CBatchCompact), P(EncodeOpts), vp, u64, P(u64)]
        lib.cbcg_encode_resident.argtypes = [vp, P(EncodeOpts)]
        lib.cbcg_decode_resident.argtypes = [vp]
        lib.cbcg_fetch_container.argtypes = [vp, vp, u64, P(u64)]
        lib.cbcg_fetch_decoded.argtypes = [vp, vp, u64, P(u64)]
        lib.cbcg_fetch_index.argtypes = [vp, vp, u64, P(u64), P(u64)]
        lib.cbcg_cigar_bound.argtypes = [P(CBatch)]; lib.cbcg_cigar_bound.restype = u64
        lib.cbcg_cigar_pack.argtypes = [vp, P(CBatch), vp, u64, P(u64)]
        lib.cbcg_cigar_unpack.argtypes = [vp, vp, u64, C.c_int, vp, u64, vp, u64, P(u64), P(u64)]
        lib.cbcg_region_plan.argtypes = [vp, u64, C.c_int, P(Region), u32, P(u64), P(u64), P(u64), P(u64)]
        lib.cbcg_decode_region.argtypes = [vp, vp, u64, C.c_int, P(Region), u32, vp, u64, P(u64), vp, u64, P(u64)]
        lib.cbcg_sam_header.argtypes = [vp, u64, vp, u64, P(u64)]
        lib.cbcg_decode_sam.argtypes = [vp, vp, u64, C.c_int, vp, u64, P(Region), u32, u32, vp, u64, P(u64), vp, u64, P(u64)]
        lib.cbcg_derive_md.argtypes = [vp, P(CBatch), vp, u64, P(u64)]
        lib.cbcg_pileup.argtypes = [vp, vp, u64, C.c_int, vp, u64, P(Region), u32, u32, vp, u64, P(u64), vp, P(u64)]
        lib.cbcg_bam_header.argtypes = [vp, vp, u64, C.c_int, vp, u64, P(u64)]
        lib.cbcg_decode_bam.argtypes = [vp, vp, u64, C.c_int, vp, u64, P(Region), u32, u32, vp, u64, P(u64), vp, u64, P(u64)]
        lib.cbcg_bgzf_inflate.argtypes = [vp, vp, u64, vp, u64, P(u64)]
        lib.cbcg_bam_open.argtypes = [vp, vp, u64, P(u64), vp, u64, P(u64)]
        lib.cbcg_batch_upload_bam.argtypes = [vp, vp, u64, vp, u64, u32, P(BamInfo), vp, u64]
        lib.cbcg_cigar_pack_resident.argtypes = [vp, vp, u64, P(u64)]
        lib.cbcg_mark.argtypes = [vp, C.c_int]
        lib.cbcg_elapsed_ms.argtypes = [vp, C.c_int, C.c_int, P(C.c_float)]
        _LIB = lib
    return _LIB


def pinned_empty(n: int, dtype) -> np.ndarray:
    """numpy array over page-locked memory from cbcg_host_alloc (kept alive by the array's base)."""
    lib = load_library()
    dt = np.dtype(dtype)
    nbytes = max(int(n) * dt.itemsize, 1)
    p = lib.cbcg_host_alloc(nbytes)
    if not p:
        raise MemoryError("cbcg_host_alloc")

    class _Owner:
        def __init__(self, ptr): self.ptr = ptr
        def __del__(self):
            try: lib.cbcg_host_free(self.ptr)
            except Exception: pass
    buf = (C.c_uint8 * nbytes).from_address(p)
    buf._owner = _Owner(p)
    return np.frombuffer(buf, dtype=dt, count=int(n))


def pin_batch(b: Batch) -> Batch:
    """Copy of a batch in page-locked memory (what a production ingest thread would fill directly)."""
    def pin(a):
        if a is None:
            return None
        out = pinned_empty(a.shape[0], a.dtype)
        out[:] = a
        return out
    return Batch(pin(b.pos), pin(b.flag), pin(b.seq_len), pin(b.chr), pin(b.seq_off), pin(b.seq),
                 pin(b.cigar_off), pin(b.cigar), pin(b.md_off), pin(b.md))


_HOSTLIB = None


def _hostlib():
    global _HOSTLIB
    if _HOSTLIB is None:
        path = os.path.join(_HERE, "_build", "libcbchost.so")
        if not os.path.exists(path):
            raise RuntimeError(f"{path} is missing: run `make host`")
        _HOSTLIB = C.CDLL(path)
        _HOSTLIB.cbch_pack_batch.argtypes = [C.POINTER(CBatch), C.c_int, C.c_void_p, C.c_void_p, C.POINTER(_CbchCompact)]
        _HOSTLIB.cbch_free_compact.argtypes = [C.POINTER(_CbchCompact)]
        _HOSTLIB.cbch_free_compact.restype = None
    return _HOSTLIB


class CompactBatch:
    """A batch packed for the link by the host C code (cbch_pack_batch): 2 bits per base, text lengths, chromosome runs.
    pinned: its arrays live in page-locked memory from cbcg_host_alloc."""

    def __init__(self, batch: Batch, pinned: bool = True, threads: int = 0):
        self.c = _CbchCompact()
        self.n_reads = batch.n_reads
        cb = batch.c_struct()
        alloc = release = None
        if pinned:
            lib = load_library()
            alloc = C.cast(lib.cbcg_host_alloc, C.c_void_p)
            release = C.cast(lib.cbcg_host_free, C.c_void_p)
        rc = _hostlib().cbch_pack_batch(C.byref(cb), threads, alloc, release, C.byref(self.c))
        if rc:
            raise MemoryError(f"cbch_pack_batch: {rc}")

    @property
    def link_bytes(self) -> int:
        return int(self.c.bytes)

    def close(self):
        if self.c is not None:
            _hostlib().cbch_free_compact(C.byref(self.c))
            self.c = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Codec:
    """One context per GPU; one host thread per context."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.cbcg_create(device, C.byref(h))
        if rc:
            raise CbcgError(rc, self.lib.cbcg_strerror(rc).decode())
        self.h = h
        self._genome_keep = None
        self.last_pileup_reads = 0                   # reads the last ``pileup`` counted

    def close(self):
        if getattr(self, "h", None):
            self.lib.cbcg_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc:
            raise CbcgError(rc, self.lib.cbcg_last_error(self.h).decode() or self.lib.cbcg_strerror(rc).decode())

    def stats(self) -> dict:
        s = Stats()
        self._check(self.lib.cbcg_get_stats(self.h, C.byref(s)))
        return s.as_dict()

    # ---- reference genome (store_reference_in_memory, src/read_decompression.c:17-53)
    def set_reference(self, genome: Genome):
        ptrs, lens, names = genome.c_arrays()
        self._genome_keep = (genome, ptrs, lens, names)
        self._check(self.lib.cbcg_set_reference(self.h, genome.n_chr, C.cast(names, C.c_void_p),
                                                C.cast(ptrs, C.c_void_p), C.cast(lens, C.c_void_p)))

    # ---- K1
    def extract(self, batch: Batch) -> Tuple[np.ndarray, np.ndarray]:
        cb = batch.c_struct()
        recs = np.zeros(max(batch.n_reads, 1), REC_DTYPE)
        cap = batch.total_bases() // 8 + 4096
        while True:
            edits = np.zeros(cap, np.uint16)
            n = C.c_uint64(0)
            rc = self.lib.cbcg_extract(self.h, C.byref(cb), recs.ctypes.data, edits.ctypes.data, cap, C.byref(n))
            if rc == -5 and n.value > cap:
                cap = n.value + 16
                continue
            self._check(rc)
            return recs[:batch.n_reads], edits[:n.value].copy()

    def symbols(self, batch: Batch, read_len_header: int, block_reads: int = 0, gen_mode: int = 0):
        cb = batch.c_struct()
        opts = EncodeOpts(read_len_header, block_reads, gen_mode, 0)
        cap = 16 * batch.n_reads + batch.total_bases() // 4 + 8192
        nb_cap = (batch.n_reads // block_reads + 4200) if block_reads else 1
        while True:
            syms = np.zeros(cap, SYM_DTYPE)
            counts = np.zeros(nb_cap, np.uint64)
            n, nb = C.c_uint64(0), C.c_uint64(0)
            rc = self.lib.cbcg_extract_symbols(self.h, C.byref(cb), C.byref(opts), syms.ctypes.data, cap, C.byref(n),
                                               counts.ctypes.data, nb_cap, C.byref(nb))
            if rc == -5 and (n.value > cap or nb.value > nb_cap):
                cap, nb_cap = max(cap, n.value + 16), max(nb_cap, nb.value + 1)
                continue
            self._check(rc)
            return syms[:n.value].copy(), counts[:nb.value].copy()

    # ---- compress() / decompress() (src/compression.c:112-216) over host buffers
    def compress(self, batch: Batch, read_len_header: int, block_reads: int = 0, gen_mode: int = 0,
                 out: Optional[np.ndarray] = None, substreams: int = 1) -> bytes:
        """block_reads == 0: the reference's own single stream (byte-identical to `program -c 1`, -DDEBUG).
        gen_mode 1: generation-primed blocks (DESIGN.md). substreams 4: four arithmetic-coded substreams per block."""
        cb = batch.c_struct()
        opts = EncodeOpts(read_len_header, block_reads, gen_mode, substreams)
        cap = int(self.lib.cbcg_encode_bound(C.byref(cb), C.byref(opts)))
        buf = out if out is not None and out.nbytes >= cap else np.empty(cap, np.uint8)
        n = C.c_uint64(0)
        rc = self.lib.cbcg_encode(self.h, C.byref(cb), C.byref(opts), buf.ctypes.data, buf.nbytes, C.byref(n))
        if rc == -5 and n.value > buf.nbytes:
            buf = np.empty(n.value, np.uint8)
            rc = self.lib.cbcg_fetch_container(self.h, buf.ctypes.data, buf.nbytes, C.byref(n))
        self._check(rc)
        return buf[:n.value].tobytes()

    def decompress(self, data: bytes, legacy: bool = False) -> Tuple[bytes, int]:
        """Returns (SEQ + '\\n' per read, read count): what `program -x` writes (print_line, src/compression.c:16-40)."""
        src = np.frombuffer(data, np.uint8)
        n_reads, cap = C.c_uint64(0), C.c_uint64(0)
        if not legacy:
            rc = self.lib.cbcg_decoded_size(src.ctypes.data, src.nbytes, C.byref(n_reads), C.byref(cap))
            if rc:
                raise CbcgError(rc, self.lib.cbcg_strerror(rc).decode())
            size = cap.value
        else:
            size = 1 << 20
        while True:
            out = np.empty(max(size, 1), np.uint8)
            n, nr = C.c_uint64(0), C.c_uint64(0)
            rc = self.lib.cbcg_decode(self.h, src.ctypes.data, src.nbytes, int(legacy), out.ctypes.data, out.nbytes,
                                      C.byref(n), C.byref(nr))
            if rc == -5 and n.value > out.nbytes:
                out = np.empty(n.value, np.uint8)
                rc = self.lib.cbcg_fetch_decoded(self.h, out.ctypes.data, out.nbytes, C.byref(n))
            self._check(rc)
            return out[:n.value].tobytes(), nr.value

    def decompress_region(self, data: bytes, regions, legacy: bool = False) -> Tuple[bytes, np.ndarray]:
        """The reads that overlap at least one region, each once, in container order: (SEQ + '\\n' per read, their
        ordinals in the container as uint64). regions: (name,), (name, start) or (name, start, end), 1-based, inclusive."""
        src = np.frombuffer(data, np.uint8)
        arr, n_regions = _region_array(regions)
        if legacy:
            size, n_ids = 1 << 20, 1 << 16
        else:
            p = region_plan(data, regions)
            size, n_ids = p["max_seq_bytes"], p["n_reads"]
        while True:
            out = np.empty(max(size, 1), np.uint8)
            ids = np.empty(max(n_ids, 1), np.uint64)
            n, nr = C.c_uint64(0), C.c_uint64(0)
            rc = self.lib.cbcg_decode_region(self.h, src.ctypes.data, src.nbytes, int(legacy), arr, n_regions,
                                             out.ctypes.data, out.nbytes, C.byref(n), ids.ctypes.data, ids.size, C.byref(nr))
            if rc == -5 and (n.value > out.nbytes or nr.value > ids.size):
                size, n_ids = max(size, n.value), max(n_ids, nr.value)
                continue
            self._check(rc)
            return out[:n.value].tobytes(), ids[:nr.value].copy()

    def decompress_sam(self, data: bytes, cigar_section: Optional[bytes] = None, regions=None, header: bool = True,
                       legacy: bool = False) -> Tuple[bytes, np.ndarray]:
        """SAM text of a container (include/cbcg.h, cbcg_decode_sam): the header (header=True), then one alignment record per
        read in container order, or per read that overlaps one of the regions (as ``decompress_region``); and each line's read
        ordinal in the container as uint64. cigar_section: the CIGAR side section (``cigar_pack``); None: implied CIGARs."""
        src = np.frombuffer(data, np.uint8)
        sec = np.frombuffer(cigar_section, np.uint8) if cigar_section is not None else None
        if regions is not None:
            arr, n_regions = _region_array(regions)                          # an empty list is CBCG_ERR_ARG
        else:
            arr, n_regions = None, 0
        n_ids = 1 << 16
        size = max(len(data) * 8, 1 << 20)
        if not legacy:
            n_reads, cap = C.c_uint64(0), C.c_uint64(0)
            if self.lib.cbcg_decoded_size(src.ctypes.data, src.nbytes, C.byref(n_reads), C.byref(cap)) == 0:
                size, n_ids = max(size, 2 * cap.value + 1024), max(n_reads.value, 1)
        while True:
            out = np.empty(size, np.uint8)
            ids = np.empty(n_ids, np.uint64)
            n, nr = C.c_uint64(0), C.c_uint64(0)
            rc = self.lib.cbcg_decode_sam(self.h, src.ctypes.data, src.nbytes, int(legacy),
                                          sec.ctypes.data if sec is not None else None, sec.nbytes if sec is not None else 0,
                                          arr, n_regions, 1 if header else 0, out.ctypes.data, out.nbytes, C.byref(n),
                                          ids.ctypes.data, ids.size, C.byref(nr))
            if rc == -5 and (n.value > out.nbytes or nr.value > ids.size):
                size, n_ids = max(size, n.value), max(n_ids, nr.value)
                continue
            self._check(rc)
            return out[:n.value].tobytes(), ids[:nr.value].copy()

    def decompress_bam(self, data: bytes, cigar_section: Optional[bytes] = None, regions=None, header: bool = True,
                       eof: bool = True, legacy: bool = False) -> Tuple[bytes, np.ndarray]:
        """BAM of a container (include/cbcg.h, cbcg_decode_bam): ``decompress_sam``'s reads as BAM records in BGZF blocks,
        after the header blocks (header=True) and before the end-of-file block (eof=True); and each record's read ordinal in
        the container as uint64. cigar_section and regions: as ``decompress_sam``. The output of several calls without
        header and EOF concatenates into one file between ``bam_header`` and the EOF block."""
        src = np.frombuffer(data, np.uint8)
        sec = np.frombuffer(cigar_section, np.uint8) if cigar_section is not None else None
        if regions is not None:
            arr, n_regions = _region_array(regions)                          # an empty list is CBCG_ERR_ARG
        else:
            arr, n_regions = None, 0
        flags = (BAM_HEADER if header else 0) | (BAM_EOF if eof else 0)
        n_ids = 1 << 16
        size = max(len(data) * 8, 1 << 20)
        if not legacy:
            n_reads, cap = C.c_uint64(0), C.c_uint64(0)
            if self.lib.cbcg_decoded_size(src.ctypes.data, src.nbytes, C.byref(n_reads), C.byref(cap)) == 0:
                size, n_ids = max(size, 2 * cap.value + 1024), max(n_reads.value, 1)
        while True:
            out = np.empty(size, np.uint8)
            ids = np.empty(n_ids, np.uint64)
            n, nr = C.c_uint64(0), C.c_uint64(0)
            rc = self.lib.cbcg_decode_bam(self.h, src.ctypes.data, src.nbytes, int(legacy),
                                          sec.ctypes.data if sec is not None else None, sec.nbytes if sec is not None else 0,
                                          arr, n_regions, flags, out.ctypes.data, out.nbytes, C.byref(n),
                                          ids.ctypes.data, ids.size, C.byref(nr))
            if rc == -5 and (n.value > out.nbytes or nr.value > ids.size):
                size, n_ids = max(size, n.value), max(n_ids, nr.value)
                continue
            self._check(rc)
            return out[:n.value].tobytes(), ids[:nr.value].copy()

    def bam_header(self, data: bytes, legacy: bool = False) -> bytes:
        """The BAM header of a container in BGZF blocks (include/cbcg.h, cbcg_bam_header): its table's names with the loaded
        reference's lengths (legacy: the loaded reference's names). Host only; needs ``set_reference``."""
        src = np.frombuffer(data, np.uint8)
        n = C.c_uint64(0)
        rc = self.lib.cbcg_bam_header(self.h, src.ctypes.data, src.nbytes, int(legacy), None, 0, C.byref(n))
        if rc != -5:
            self._check(rc)
        out = np.empty(max(n.value, 1), np.uint8)
        self._check(self.lib.cbcg_bam_header(self.h, src.ctypes.data, src.nbytes, int(legacy), out.ctypes.data, out.nbytes, C.byref(n)))
        return out[:n.value].tobytes()

    def pileup(self, data: bytes, regions, cigar_section: Optional[bytes] = None, flag_exclude: int = PILEUP_FLAG_EXCLUDE,
               legacy: bool = False) -> List[np.ndarray]:
        """Per-position counts over regions (include/cbcg.h, cbcg_pileup): one [rows, 8] uint32 array per region, in the
        order given, columns A C G T N DEL INS REF (PILEUP_COLUMNS), one row per position start .. min(end, LN). The reads
        are ``decompress_sam``'s for the same regions without those whose FLAG & flag_exclude; cigar_section: as there.
        The arrays are views into one buffer, sized by the library's capacity answer before anything is decoded."""
        src = np.frombuffer(data, np.uint8)
        sec = np.frombuffer(cigar_section, np.uint8) if cigar_section is not None else None
        arr, n_regions = _region_array(regions)                              # an empty list is CBCG_ERR_ARG
        per = np.zeros(max(n_regions, 1), np.uint64)
        n, nr = C.c_uint64(0), C.c_uint64(0)
        args = (self.h, src.ctypes.data, src.nbytes, int(legacy), sec.ctypes.data if sec is not None else None,
                sec.nbytes if sec is not None else 0, arr, n_regions, int(flag_exclude))
        rc = self.lib.cbcg_pileup(*args, None, 0, C.byref(n), per.ctypes.data, None)
        if rc != -5:
            self._check(rc)
        rows = np.empty((max(n.value, 1), len(PILEUP_COLUMNS)), np.uint32)
        self._check(self.lib.cbcg_pileup(*args, rows.ctypes.data, n.value, C.byref(n), per.ctypes.data, C.byref(nr)))
        self.last_pileup_reads = nr.value
        ends = np.cumsum(per[:n_regions].astype(np.int64))
        return [rows[e - int(k):e] for e, k in zip(ends.tolist(), per[:n_regions].tolist())]

    def cigar_pack(self, batch: Batch) -> bytes:
        """The CIGAR side section of a batch (SURVEY.md 8f row 4, cbcg.h): reads whose CIGAR is not the one their indels
        imply, as a class (end operations are soft clips) or verbatim."""
        cb = batch.c_struct()
        cap = int(self.lib.cbcg_cigar_bound(C.byref(cb)))
        out = np.empty(max(cap, 24), np.uint8)
        n = C.c_uint64(0)
        self._check(self.lib.cbcg_cigar_pack(self.h, C.byref(cb), out.ctypes.data, out.nbytes, C.byref(n)))
        return out[:n.value].tobytes()

    def cigar_pack_resident(self) -> bytes:
        """``cigar_pack`` of the resident batch, without an upload (the batch of ``upload_bam`` exists only on the device)."""
        n = C.c_uint64(0)
        rc = self.lib.cbcg_cigar_pack_resident(self.h, None, 0, C.byref(n))
        if rc != -5:
            self._check(rc)
        out = np.empty(max(n.value, 24), np.uint8)
        self._check(self.lib.cbcg_cigar_pack_resident(self.h, out.ctypes.data, out.nbytes, C.byref(n)))
        return out[:n.value].tobytes()

    # ---- BAM input (include/cbcg.h, DESIGN.md 5g)
    def bgzf_inflate(self, data: bytes) -> bytes:
        """Whole BGZF members -> their inflated concatenation, inflated on the GPU."""
        src = np.frombuffer(data, np.uint8)
        n = C.c_uint64(0)
        rc = self.lib.cbcg_bgzf_inflate(self.h, src.ctypes.data, src.nbytes, None, 0, C.byref(n))
        if rc != -5:
            self._check(rc)
        out = np.empty(max(n.value, 1), np.uint8)
        self._check(self.lib.cbcg_bgzf_inflate(self.h, src.ctypes.data, src.nbytes, out.ctypes.data, out.nbytes, C.byref(n)))
        return out[:n.value].tobytes()

    def bam_open(self, data: bytes) -> Tuple[int, bytes]:
        """Reads the BAM header from the start of ``data`` (the whole file will do): (bytes of the members it consumed, the
        record bytes after the header in the last of them). Needs ``set_reference``."""
        src = np.frombuffer(data, np.uint8)
        used, n = C.c_uint64(0), C.c_uint64(0)
        tail = np.empty(1 << 17, np.uint8)
        self._check(self.lib.cbcg_bam_open(self.h, src.ctypes.data, src.nbytes, C.byref(used), tail.ctypes.data, tail.nbytes, C.byref(n)))
        return used.value, tail[:n.value].tobytes()

    def upload_bam(self, data: bytes, carry: bytes = b"", derive_md: bool = False, last: bool = True) -> Tuple[dict, bytes]:
        """Whole BGZF members after ``carry`` -> the resident batch: (cbcg_bam_info as a dict, the bytes after the last whole
        record, the next call's carry)."""
        src = np.frombuffer(data, np.uint8)
        car = np.frombuffer(carry, np.uint8)
        info = BamInfo()
        flags = (BAM_DERIVE_MD if derive_md else 0) | (BAM_LAST if last else 0)
        cap = 1 << 17
        while True:
            tail = np.empty(cap, np.uint8)
            rc = self.lib.cbcg_batch_upload_bam(self.h, car.ctypes.data if car.size else None, car.size,
                                                src.ctypes.data if src.size else None, src.size, flags, C.byref(info),
                                                tail.ctypes.data, tail.nbytes)
            if rc == -5 and info.tail_len > cap:
                cap = int(info.tail_len)
                continue
            self._check(rc)
            return info.as_dict(), tail[:info.tail_len].tobytes()

    def compress_bam(self, data: bytes, read_len_header: Optional[int] = None, block_reads: int = BLOCK_AUTO, gen_mode: int = 1,
                     substreams: int = 1, derive_md: bool = False, var_length: bool = False) -> Tuple[bytes, dict]:
        """A whole BAM file -> (container, cbcg_bam_info dict): ``bam_open``, one ``upload_bam``, ``encode_resident``,
        ``fetch_container``. read_len_header None: get_read_length's answer, the second record's l_seq (var_length: the
        longest read)."""
        used, tail = self.bam_open(data)
        info, _ = self.upload_bam(data[used:], carry=tail, derive_md=derive_md, last=True)
        if read_len_header is None:
            read_len_header = info["max_len"] if var_length else (info["len_second"] if info["n_records"] >= 2 else info["len_first"])
        self.encode_resident(read_len_header, block_reads, gen_mode, substreams)
        return self.fetch_container().tobytes(), info

    def cigar_unpack(self, data: bytes, section: Optional[bytes], legacy: bool = False) -> Tuple[bytes, int]:
        """(CIGAR + '\\n' per read in read order, read count) of a container and its side section (None: the implied CIGARs)."""
        src = np.frombuffer(data, np.uint8)
        sec = np.frombuffer(section, np.uint8) if section is not None else None
        size = max(len(data) * 4, 1 << 16)
        while True:
            out = np.empty(size, np.uint8)
            n, nr = C.c_uint64(0), C.c_uint64(0)
            rc = self.lib.cbcg_cigar_unpack(self.h, src.ctypes.data, src.nbytes, int(legacy),
                                            sec.ctypes.data if sec is not None else None, sec.nbytes if sec is not None else 0,
                                            out.ctypes.data, out.nbytes, C.byref(n), C.byref(nr))
            if rc == -5 and n.value > out.nbytes:
                size = int(n.value)
                continue
            self._check(rc)
            return out[:n.value].tobytes(), nr.value

    def compress_into(self, batch: Batch, read_len_header: int, block_reads: int, out: np.ndarray, gen_mode: int = 0,
                      substreams: int = 1) -> int:
        """cbcg_encode into a caller-owned (ideally pinned) buffer; returns the container size."""
        cb = batch.c_struct()
        opts = EncodeOpts(read_len_header, block_reads, gen_mode, substreams)
        n = C.c_uint64(0)
        self._check(self.lib.cbcg_encode(self.h, C.byref(cb), C.byref(opts), out.ctypes.data, out.nbytes, C.byref(n)))
        return n.value

    def compress_compact_into(self, compact: "CompactBatch", read_len_header: int, block_reads: int, out: np.ndarray,
                              gen_mode: int = 0, substreams: int = 1) -> int:
        """cbcg_encode_compact: the same container from a third of the bytes on the link."""
        opts = EncodeOpts(read_len_header, block_reads, gen_mode, substreams)
        n = C.c_uint64(0)
        self._check(self.lib.cbcg_encode_compact(self.h, C.byref(compact.c.v), C.byref(opts), out.ctypes.data, out.nbytes, C.byref(n)))
        return n.value

    def upload_compact(self, compact: "CompactBatch"):
        self._check(self.lib.cbcg_batch_upload_compact(self.h, C.byref(compact.c.v)))

    def decompress_into(self, data: np.ndarray, out: np.ndarray, legacy: bool = False) -> Tuple[int, int]:
        """cbcg_decode from / into caller-owned buffers; returns (text bytes, reads)."""
        n, nr = C.c_uint64(0), C.c_uint64(0)
        self._check(self.lib.cbcg_decode(self.h, data.ctypes.data, data.nbytes, int(legacy), out.ctypes.data, out.nbytes,
                                         C.byref(n), C.byref(nr)))
        return n.value, nr.value

    def decode_edits(self, data: bytes, legacy: bool = False):
        src = np.frombuffer(data, np.uint8)
        rcap, ecap = 1 << 16, 1 << 18
        while True:
            recs = np.zeros(rcap, REC_DTYPE); chr_ = np.zeros(rcap, np.uint32); edits = np.zeros(ecap, np.uint16)
            nr, ne = C.c_uint64(0), C.c_uint64(0)
            rc = self.lib.cbcg_decode_edits(self.h, src.ctypes.data, src.nbytes, int(legacy), recs.ctypes.data, rcap,
                                            chr_.ctypes.data, edits.ctypes.data, ecap, C.byref(nr), C.byref(ne))
            if rc == -5 and (nr.value > rcap or ne.value > ecap):
                rcap, ecap = max(rcap, nr.value), max(ecap, ne.value)
                continue
            self._check(rc)
            return recs[:nr.value].copy(), chr_[:nr.value].copy(), edits[:ne.value].copy()

    def derive_md(self, batch: Batch) -> bytes:
        """Each read's MD as a batch without MD gets it on the GPU (include/cbcg.h, cbcg_derive_md): MD + '\\n' per read, in
        read order. Any MD the batch carries is ignored. The batch becomes the resident batch, with the derived MD."""
        cb = batch.c_struct()
        cap = batch.total_bases() // 4 + 16 * batch.n_reads + 4096
        while True:
            out = np.empty(max(cap, 1), np.uint8)
            n = C.c_uint64(0)
            rc = self.lib.cbcg_derive_md(self.h, C.byref(cb), out.ctypes.data, out.nbytes, C.byref(n))
            if rc == -5 and n.value > out.nbytes:
                cap = n.value
                continue
            self._check(rc)
            return out[:n.value].tobytes()

    # ---- K3
    def reconstruct(self, recs: np.ndarray, chr_: np.ndarray, edits: np.ndarray) -> bytes:
        recs = np.ascontiguousarray(recs); chr_ = np.ascontiguousarray(chr_, np.uint32)
        edits = np.ascontiguousarray(edits, np.uint16)
        cap = int(recs["len"].astype(np.int64).sum()) + len(recs) + 64
        out = np.empty(cap, np.uint8)
        n = C.c_uint64(0)
        self._check(self.lib.cbcg_reconstruct(self.h, len(recs), recs.ctypes.data, chr_.ctypes.data,
                                              edits.ctypes.data if edits.size else None, edits.size,
                                              out.ctypes.data, cap, C.byref(n)))
        return out[:n.value].tobytes()

    # ---- device-resident variants
    def upload(self, batch: Batch):
        cb = batch.c_struct()
        self._check(self.lib.cbcg_batch_upload(self.h, C.byref(cb)))

    def encode_resident(self, read_len_header: int, block_reads: int, gen_mode: int = 0, substreams: int = 1):
        opts = EncodeOpts(read_len_header, block_reads, gen_mode, substreams)
        self._check(self.lib.cbcg_encode_resident(self.h, C.byref(opts)))

    def decode_resident(self):
        self._check(self.lib.cbcg_decode_resident(self.h))

    def fetch_container(self, out: Optional[np.ndarray] = None) -> np.ndarray:
        n = C.c_uint64(0)
        rc = self.lib.cbcg_fetch_container(self.h, out.ctypes.data if out is not None else None,
                                           out.nbytes if out is not None else 0, C.byref(n))
        if rc == -5:
            out = np.empty(n.value, np.uint8)
            rc = self.lib.cbcg_fetch_container(self.h, out.ctypes.data, out.nbytes, C.byref(n))
        self._check(rc)
        return out[:n.value]

    def fetch_decoded(self, out: Optional[np.ndarray] = None) -> np.ndarray:
        n = C.c_uint64(0)
        rc = self.lib.cbcg_fetch_decoded(self.h, out.ctypes.data if out is not None else None,
                                         out.nbytes if out is not None else 0, C.byref(n))
        if rc == -5:
            out = np.empty(n.value, np.uint8)
            rc = self.lib.cbcg_fetch_decoded(self.h, out.ctypes.data, out.nbytes, C.byref(n))
        self._check(rc)
        return out[:n.value]

    def fetch_index(self) -> Tuple[bytes, int]:
        """(container header + per-block index, payload byte count) of the last encode."""
        n, pb = C.c_uint64(0), C.c_uint64(0)
        self.lib.cbcg_fetch_index(self.h, None, 0, C.byref(n), C.byref(pb))
        out = np.empty(max(n.value, 1), np.uint8)
        self._check(self.lib.cbcg_fetch_index(self.h, out.ctypes.data, out.nbytes, C.byref(n), C.byref(pb)))
        return out[:n.value].tobytes(), pb.value

    def mark(self, slot: int):
        self._check(self.lib.cbcg_mark(self.h, slot))

    def elapsed_ms(self, a: int, b: int) -> float:
        ms = C.c_float(0)
        self._check(self.lib.cbcg_elapsed_ms(self.h, a, b, C.byref(ms)))
        return ms.value
