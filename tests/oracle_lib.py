"""ctypes wrapper of the CPU oracle (oracle/cbc_oracle.c) and of the prebuilt reference
binaries in oracle/_ref/. TEST INFRASTRUCTURE: only tests/, smoke() and bench.py's CPU
baseline may import this; nothing under cbc_b200/ does."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from cbc_b200.batch import Batch, CBatch, Genome

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_BIN = os.path.join(ORACLE_DIR, "_ref", "cbc_ref")
TRACE_BIN = os.path.join(ORACLE_DIR, "_ref", "cbc_trace")

REC_DTYPE = np.dtype([("pos", "<u4"), ("flag", "<u2"), ("len", "<u2"), ("edit_off", "<u4"),
                      ("match", "u1"), ("n_snps", "u1"), ("n_dels", "u1"), ("n_ins", "u1")])
SYM_DTYPE = np.dtype([("key", "<u4"), ("value", "<u4")])

STREAMS = ["codebook", "same_ref", "rname", "rlength", "pos", "pos_alpha", "flag", "match", "snps",
           "indels", "var", "chars", "pos_x"]


class _Genome(C.Structure):
    _fields_ = [("n_chr", C.c_uint32), ("bases", C.c_void_p), ("len", C.c_void_p), ("name", C.c_void_p)]


class _Buf(C.Structure):
    _fields_ = [("data", C.c_void_p), ("size", C.c_uint64), ("cap", C.c_uint64)]


_LIB = None


def build():
    subprocess.run(["make", "-C", ORACLE_DIR, "port"], check=True, capture_output=True)


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(ORACLE_DIR, "_build", "libcbc_oracle.so")
        if not os.path.exists(path):
            build()
        _LIB = C.CDLL(path)
        _LIB.cbco_extract.restype = C.c_int64
        _LIB.cbco_reconstruct.restype = C.c_int64
    return _LIB


class _G:
    """Keeps the ctypes arrays of a Genome alive."""
    def __init__(self, genome: Genome):
        self.ptrs, self.lens, self.names = genome.c_arrays()
        self.s = _Genome(genome.n_chr, C.cast(self.ptrs, C.c_void_p), C.cast(self.lens, C.c_void_p),
                         C.cast(self.names, C.c_void_p))


def _take(buf: _Buf) -> bytes:
    out = C.string_at(buf.data, buf.size) if buf.size else b""
    lib().cbco_buf_free(C.byref(buf))
    return out


def extract(batch: Batch, genome: Genome):
    g = _G(genome)
    cb = batch.c_struct()
    recs = np.zeros(batch.n_reads, REC_DTYPE)
    cap = int(batch.seq_len.astype(np.int64).sum()) + (255 + 8) * batch.n_reads + 64    # CBCO_EDITS_PER_READ
    edits = np.zeros(cap, np.uint16)
    n = lib().cbco_extract(C.byref(cb), C.byref(g.s), recs.ctypes.data_as(C.c_void_p),
                           edits.ctypes.data_as(C.c_void_p), C.c_uint64(cap))
    if n < 0:
        raise RuntimeError(f"cbco_extract: {n}")
    return recs, edits[:n].copy()


def reconstruct(recs, edits, chr_, genome: Genome) -> bytes:
    g = _G(genome)
    cap = int(recs["len"].astype(np.int64).sum()) + len(recs) + 16
    out = np.zeros(cap, np.uint8)
    edits = np.ascontiguousarray(edits, np.uint16)
    if edits.size == 0:
        edits = np.zeros(1, np.uint16)
    chr_ = np.ascontiguousarray(chr_, np.uint32)
    n = lib().cbco_reconstruct(C.c_uint64(len(recs)), recs.ctypes.data_as(C.c_void_p),
                               edits.ctypes.data_as(C.c_void_p), chr_.ctypes.data_as(C.c_void_p),
                               C.byref(g.s), out.ctypes.data_as(C.c_void_p), C.c_uint64(cap))
    if n < 0:
        raise RuntimeError(f"cbco_reconstruct: {n}")
    return out[:n].tobytes()


def encode_legacy(batch: Batch, genome: Genome, read_len_header: int, want_trace: bool = False):
    g = _G(genome)
    cb = batch.c_struct()
    out, tr = _Buf(), _Buf()
    rc = lib().cbco_encode_legacy(C.byref(cb), C.byref(g.s), C.c_uint32(read_len_header), C.byref(out),
                                  C.byref(tr) if want_trace else None)
    if rc:
        raise RuntimeError(f"cbco_encode_legacy: {rc}")
    stream = _take(out)
    trace = np.frombuffer(_take(tr), SYM_DTYPE) if want_trace else None
    return stream, trace


def decode_legacy(stream: bytes, genome: Genome):
    g = _G(genome)
    out = _Buf()
    n = C.c_uint64(0)
    rc = lib().cbco_decode_legacy(stream, C.c_uint64(len(stream)), C.byref(g.s), C.byref(out), C.byref(n))
    data = _take(out)
    if rc:
        raise RuntimeError(f"cbco_decode_legacy: {rc}")
    return data, n.value


def symbols(batch: Batch, genome: Genome, recs, edits, r0: int, r1: int, read_len_header: int, legacy: bool):
    g = _G(genome)
    cb = batch.c_struct()
    out = _Buf()
    edits = np.ascontiguousarray(edits, np.uint16)
    if edits.size == 0:
        edits = np.zeros(1, np.uint16)
    rc = lib().cbco_symbols(C.byref(cb), C.byref(g.s), recs.ctypes.data_as(C.c_void_p),
                            edits.ctypes.data_as(C.c_void_p), C.c_uint64(r0), C.c_uint64(r1),
                            C.c_uint32(read_len_header), C.c_int(int(legacy)), C.byref(out))
    if rc:
        raise RuntimeError(f"cbco_symbols: {rc}")
    return np.frombuffer(_take(out), SYM_DTYPE)


def encode_blocked(batch: Batch, genome: Genome, read_len_header: int, block_reads: int, gen_mode: int = 0) -> bytes:
    g = _G(genome)
    cb = batch.c_struct()
    out = _Buf()
    rc = lib().cbco_encode_blocked(C.byref(cb), C.byref(g.s), C.c_uint32(read_len_header),
                                   C.c_uint32(block_reads), C.c_uint32(gen_mode), C.byref(out))
    if rc:
        raise RuntimeError(f"cbco_encode_blocked: {rc}")
    return _take(out)


def encode_like(container: bytes, batch: Batch, genome: Genome) -> bytes:
    """The batch coded by the CPU restatement with the block cut recorded in `container`'s index."""
    g = _G(genome)
    cb = batch.c_struct()
    out = _Buf()
    rc = lib().cbco_encode_like(container, C.c_uint64(len(container)), C.byref(cb), C.byref(g.s), C.byref(out))
    if rc:
        raise RuntimeError(f"cbco_encode_like: {rc}")
    return _take(out)


def decode_blocked(container: bytes, genome: Genome):
    g = _G(genome)
    out = _Buf()
    n = C.c_uint64(0)
    rc = lib().cbco_decode_blocked(container, C.c_uint64(len(container)), C.byref(g.s), C.byref(out), C.byref(n))
    data = _take(out)
    if rc:
        raise RuntimeError(f"cbco_decode_blocked: {rc}")
    return data, n.value


# ---------------------------------------------------------------- the real reference (prebuilt)

def have_reference() -> bool:
    return os.access(REF_BIN, os.X_OK) and os.access(TRACE_BIN, os.X_OK)


def run_reference(sam_path: str, fasta_path: str, workdir: str, trace: bool = False, var_length: bool = False):
    """`program -c 1 sam out ref` (+ optional symbol trace). Returns (stream bytes, trace array|None, seconds)."""
    import re
    out = os.path.join(workdir, "ref.cbc")
    env = dict(os.environ)
    tr_path = os.path.join(workdir, "trace.bin")
    if trace:
        env["CBC_TRACE_OUT"] = tr_path
    cmd = [TRACE_BIN if trace else REF_BIN, "-c", "1"] + (["-l"] if var_length else []) + [sam_path, out, fasta_path]
    p = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=workdir)
    if not os.path.exists(out):
        raise RuntimeError(f"reference encoder failed rc={p.returncode}: {p.stdout[-300:]} {p.stderr[-300:]}")
    m = re.search(r"Compression took ([0-9.]+)", p.stdout)
    secs = float(m.group(1)) if m else float("nan")
    if "Compression took" not in p.stdout:
        raise RuntimeError(f"reference encoder died rc={p.returncode}: {p.stderr[-300:]}")
    with open(out, "rb") as f:
        stream = f.read()
    tr = np.fromfile(tr_path, SYM_DTYPE) if trace else None
    return stream, tr, secs


def run_reference_decode(stream_path: str, fasta_path: str, workdir: str):
    import re
    out = os.path.join(workdir, "ref.out.txt")
    p = subprocess.run([REF_BIN, "-x", stream_path, out, fasta_path], capture_output=True, text=True, cwd=workdir)
    m = re.search(r"Decompression took ([0-9.]+)", p.stdout)
    if not m:
        raise RuntimeError(f"reference decoder died rc={p.returncode}: {p.stderr[-300:]}")
    with open(out, "rb") as f:
        return f.read(), float(m.group(1))


def expand_pos(raw: np.ndarray) -> np.ndarray:
    """Turn a raw symbol list (POS as pos_x) into the tracer's sequence by replaying the dynamic
    pos alphabet (compress_pos, src/read_compression.c:113-159)."""
    keys, vals = [], []
    amap = {}
    card = 1
    POSX, POS, PA = 12 << 24, 4 << 24, 5 << 24
    for k, v in zip(raw["key"].tolist(), raw["value"].tolist()):
        if k != POSX:
            keys.append(k); vals.append(v)
            continue
        if v in amap:
            keys.append(POS); vals.append(amap[v])
        else:
            keys.append(POS); vals.append(0)
            for b in range(4):
                keys.append(PA | b); vals.append((v >> (24 - 8 * b)) & 0xff)
            amap[v] = card
            card += 1
    out = np.zeros(len(keys), SYM_DTYPE)
    out["key"] = keys
    out["value"] = vals
    return out
