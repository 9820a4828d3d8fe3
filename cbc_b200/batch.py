"""SoA read batch and genome containers shared by the host-side Python code.

A ``Batch`` is what the reference's ``load_sam_line`` (src/sam_file_allocation.c:437-529)
yields per SAM record, laid out structure-of-arrays: POS, FLAG, SEQ length, chromosome
ordinal and three byte pools (SEQ, CIGAR text, MD:Z payload) with n+1 offsets each.
A batch without MD (``md_off`` and ``md`` None) has its MD derived on the GPU (include/cbcg.h).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np


class CBatch(C.Structure):
    """Mirror of ``cbcg_batch`` (include/cbcg.h)."""
    _fields_ = [
        ("n_reads", C.c_uint64),
        ("pos", C.c_void_p), ("flag", C.c_void_p), ("seq_len", C.c_void_p), ("chr", C.c_void_p),
        ("seq_off", C.c_void_p), ("seq", C.c_void_p),
        ("cigar_off", C.c_void_p), ("cigar", C.c_void_p),
        ("md_off", C.c_void_p), ("md", C.c_void_p),
    ]


@dataclass
class Batch:
    pos: np.ndarray        # uint32 [n]
    flag: np.ndarray       # uint16 [n]
    seq_len: np.ndarray    # uint16 [n]
    chr: np.ndarray        # uint32 [n]
    seq_off: np.ndarray    # uint64 [n+1]
    seq: np.ndarray        # uint8
    cigar_off: np.ndarray  # uint64 [n+1]
    cigar: np.ndarray      # uint8
    md_off: Optional[np.ndarray]   # uint64 [n+1]; None with md: no MD, the library derives it
    md: Optional[np.ndarray]       # uint8

    @property
    def n_reads(self) -> int:
        return int(self.pos.shape[0])

    def c_struct(self) -> CBatch:
        for name, dt in (("pos", np.uint32), ("flag", np.uint16), ("seq_len", np.uint16), ("chr", np.uint32),
                         ("seq_off", np.uint64), ("seq", np.uint8), ("cigar_off", np.uint64),
                         ("cigar", np.uint8), ("md_off", np.uint64), ("md", np.uint8)):
            a = getattr(self, name)
            assert (a is None and name in ("md_off", "md")) or (a.dtype == dt and a.flags["C_CONTIGUOUS"]), name
        s = CBatch()
        s.n_reads = self.n_reads
        for name in ("pos", "flag", "seq_len", "chr", "seq_off", "seq", "cigar_off", "cigar", "md_off", "md"):
            a = getattr(self, name)
            setattr(s, name, a.ctypes.data if a is not None else None)
        return s

    def without_md(self) -> "Batch":
        """The same reads without MD (the arrays are shared): the library derives each read's MD on the GPU."""
        return Batch(self.pos, self.flag, self.seq_len, self.chr, self.seq_off, self.seq, self.cigar_off, self.cigar, None, None)

    def slice(self, r0: int, r1: int) -> "Batch":
        """Reads [r0, r1) as an independent batch (pools re-based)."""
        def pool(off, data):
            lo, hi = int(off[r0]), int(off[r1])
            return (off[r0:r1 + 1] - off[r0]).astype(np.uint64), np.ascontiguousarray(data[lo:hi])
        so, s = pool(self.seq_off, self.seq)
        co, c = pool(self.cigar_off, self.cigar)
        mo, m = pool(self.md_off, self.md) if self.md_off is not None else (None, None)
        return Batch(self.pos[r0:r1].copy(), self.flag[r0:r1].copy(), self.seq_len[r0:r1].copy(),
                     self.chr[r0:r1].copy(), so, s, co, c, mo, m)

    def seq_lines(self) -> bytes:
        """SEQ column, one read per line: what the decoder must reproduce."""
        n = self.n_reads
        if n == 0:
            return b""
        lo, hi = int(self.seq_off[0]), int(self.seq_off[n])
        out = np.full(hi - lo + n, 10, dtype=np.uint8)            # '\n' everywhere, then the bases around them
        keep = np.ones(hi - lo + n, dtype=bool)
        keep[(self.seq_off[1:] - np.uint64(lo)).astype(np.int64) + np.arange(n, dtype=np.int64)] = False
        out[keep] = self.seq[lo:hi]
        return out.tobytes()

    def total_bases(self) -> int:
        return int(self.seq_len.astype(np.uint64).sum())


@dataclass
class Genome:
    names: List[str]
    bases: List[np.ndarray] = field(default_factory=list)   # uint8, upper-case

    @property
    def n_chr(self) -> int:
        return len(self.names)

    def c_arrays(self):
        n = self.n_chr
        ptrs = (C.c_void_p * n)(*[b.ctypes.data for b in self.bases])
        lens = (C.c_uint64 * n)(*[int(b.shape[0]) for b in self.bases])
        names = (C.c_char_p * n)(*[s.encode() for s in self.names])
        return ptrs, lens, names
