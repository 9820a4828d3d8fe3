"""A Python restatement of the SAM line that cbcg_decode_sam writes (include/cbcg.h, k6_sam.cu), for the tests:

    *  FLAG  RNAME  POS  255  CIGAR  *  0  0  SEQ  *  NM:i:<n>  MD:Z:<md>

MD and NM are computed from the line's CIGAR, its SEQ and the upper-cased reference: M, = and X consume read and
reference, I and S the read, D the reference, H and P neither. An aligned base is a mismatch when it differs from the
reference base, so N against N is not one (samtools calmd counts it). MD: a number before every event and at the end,
0 included; letters are reference bases. NM = mismatches + I bases + D bases.

TEST INFRASTRUCTURE: imported by tests/test_gpu_sam.py and tests/test_sam_header.py."""
from __future__ import annotations

import re
from typing import List, Optional

import numpy as np

CIGAR_OP = re.compile(rb"(\d+)([MIDNSHP=X])")

# SAM spec v1 field regexes of the mandatory fields, and the two tags
FIELD_RE = [rb"\*|[!-?A-~][!-~]{0,253}", rb"[0-9]+", rb"\*|[0-9A-Za-z!#$%&+./:;?@^_|~-][0-9A-Za-z!#$%&*+./:;=?@^_|~-]*",
            rb"[0-9]+", rb"[0-9]+", rb"\*|([0-9]+[MIDNSHPX=])+", rb"\*|=|[0-9A-Za-z!#$%&+./:;?@^_|~-][0-9A-Za-z!#$%&*+./:;=?@^_|~-]*",
            rb"[0-9]+", rb"-?[0-9]+", rb"\*|[A-Za-z=.]+", rb"[!-~]+"]
NM_RE = re.compile(rb"NM:i:[0-9]+")
MD_RE = re.compile(rb"MD:Z:[0-9]+(([A-Z]|\^[A-Z]+)[0-9]+)*")


def upper(genome):
    """The genome's records upper-cased, as the library uploads them."""
    return [np.where((g >= ord("a")) & (g <= ord("z")), g - 32, g).astype(np.uint8) for g in genome.bases]


def md_nm(cigar: bytes, seq: bytes, ref: np.ndarray, pos: int):
    """(MD text, NM) of an aligned read; ref: its chromosome, upper-cased; pos: 1-based."""
    md, run, nm, ri, rp = [], 0, 0, 0, pos - 1
    for n, op in CIGAR_OP.findall(cigar):
        n = int(n)
        if op in b"M=X":
            for _ in range(n):
                rb = int(ref[rp])
                if seq[ri] != rb:
                    md.append(f"{run}{chr(rb)}"); run = 0; nm += 1
                else:
                    run += 1
                ri += 1; rp += 1
        elif op == b"I":
            ri += n; nm += n
        elif op == b"S":
            ri += n
        elif op == b"D":
            md.append(f"{run}^{bytes(ref[rp:rp + n]).decode()}"); run = 0; rp += n; nm += n
        elif op == b"N":
            rp += n
    md.append(str(run))
    return "".join(md).encode(), nm


def line(flag: int, rname: bytes, pos: int, cigar: bytes, seq: bytes, ref: np.ndarray) -> bytes:
    md, nm = md_nm(cigar, seq, ref, pos)
    return b"\t".join([b"*", b"%d" % flag, rname, b"%d" % pos, b"255", cigar, b"*", b"0", b"0", seq, b"*",
                       b"NM:i:%d" % nm, b"MD:Z:" + md]) + b"\n"


def batch_cigars(b) -> List[bytes]:
    c = b.cigar.tobytes()
    return [c[int(b.cigar_off[i]):int(b.cigar_off[i + 1])] for i in range(b.n_reads)]


def batch_seqs(b) -> List[bytes]:
    s = b.seq.tobytes()
    return [s[int(b.seq_off[i]):int(b.seq_off[i + 1])] for i in range(b.n_reads)]


def batch_mds(b) -> List[bytes]:
    m = b.md.tobytes()
    return [m[int(b.md_off[i]):int(b.md_off[i + 1])] for i in range(b.n_reads)]


def implied_cigar(rec, edits, clip_first: bool = False, clip_last: bool = False) -> bytes:
    """The CIGAR a record's deletions and insertions imply (k4_cigar.cu, cig_implied), the end I operations as S on request."""
    if rec["match"]:
        return b"%dM" % int(rec["len"])
    nd, ns, ni = int(rec["n_dels"]), int(rec["n_snps"]), int(rec["n_ins"])
    e = edits[int(rec["edit_off"]):int(rec["edit_off"]) + nd + ns + ni].astype(np.int64) & 0xff
    dels = np.cumsum(e[:nd]).tolist(); ins = np.cumsum(e[nd + ns:]).tolist()
    ops, cur, kd, ki = [], 0, 0, 0
    while kd < nd or ki < ni:
        at = min(dels[kd] if kd < nd else 1 << 30, ins[ki] if ki < ni else 1 << 30)
        if at > cur:
            ops.append([at - cur, "M"]); cur = at
        if ki < ni and ins[ki] == at:
            k = 0
            while ki < ni and ins[ki] == at:
                ki += 1; k += 1
            ops.append([k, "I"])
        if kd < nd and dels[kd] == at:
            k = 0
            while kd < nd and dels[kd] == at:
                kd += 1; k += 1
            ops.append([k, "D"])
    total_m = int(rec["len"]) - ni
    if total_m > cur:
        ops.append([total_m - cur, "M"])
    if ops and clip_first and ops[0][1] == "I":
        ops[0][1] = "S"
    if len(ops) > 1 and clip_last and ops[-1][1] == "I":
        ops[-1][1] = "S"
    return "".join(f"{n}{op}" for n, op in ops).encode()


def cigar_class(rec, edits, cigar: bytes) -> int:
    """The side section's class of a read: 0 implied, 1 / 2 / 3 end I as S, 4 verbatim."""
    for c in range(4):
        if implied_cigar(rec, edits, bool(c & 1), bool(c & 2)) == cigar:
            return c
    return 4


def sam_lines(b, genome_upper, names, cigars: Optional[List[bytes]] = None) -> List[bytes]:
    """The lines of batch b (its FLAG, chromosome, POS and SEQ); cigars: per read (default: the batch's own)."""
    cigars = cigars if cigars is not None else batch_cigars(b)
    seqs = batch_seqs(b)
    return [line(int(b.flag[i]), names[int(b.chr[i])].encode(), int(b.pos[i]), cigars[i], seqs[i], genome_upper[int(b.chr[i])])
            for i in range(b.n_reads)]


def header(names, lengths=None) -> bytes:
    out = [b"@HD\tVN:1.6\tSO:coordinate\n"]
    for k, n in enumerate(names):
        out.append(b"@SQ\tSN:" + n.encode() + (b"\tLN:%d" % lengths[k] if lengths is not None else b"") + b"\n")
    return b"".join(out)


def check_fields(text: bytes):
    """Every record line of a SAM text matches the spec's field regexes."""
    for ln in text.split(b"\n")[:-1]:
        if ln.startswith(b"@"):
            continue
        f = ln.split(b"\t")
        assert len(f) == 13, ln
        for v, rx in zip(f[:11], FIELD_RE):
            assert re.fullmatch(rx, v), (v, ln)
        assert NM_RE.fullmatch(f[11]) and MD_RE.fullmatch(f[12]), ln
