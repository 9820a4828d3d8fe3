"""A Python restatement of the pileup that cbcg_pileup returns (include/cbcg.h, k8_pileup.cu), for the tests.

Reads are (flag, chromosome ordinal, POS, CIGAR, SEQ); each CIGAR is walked base by base (K8 instead adds difference
arrays over aligned runs and reads no base of a read whose CIGAR the edit list implies):

    M = X   a base aligned to the position: counted under A, C, G, T, or N for any other character
    D       the position is deleted: DEL
    I       inserted bases after the last reference position consumed (M, =, X, D): INS, once per read and position,
            only when an M / = / X of at least one base comes before and after the I
    S H P   nothing; N skips reference

A row is u32[8] = A C G T N DEL INS REF, REF the upper-cased reference byte. A region (name,), (name, start) or
(name, start, end) gives the rows start .. min(end, LN); a name the genome does not hold raises KeyError.

TEST INFRASTRUCTURE: imported by tests/test_pileup_restate.py and tests/test_gpu_pileup.py."""
from __future__ import annotations

from typing import List, Sequence, Tuple

import numpy as np

from sam_restate import CIGAR_OP

UINT64_MAX = (1 << 64) - 1
FLAG_EXCLUDE = 0x704
CODE = np.full(256, 4, np.int64)
for _k, _c in enumerate(b"ACGT"):
    CODE[_c] = _k


def read_events(cigar: bytes, seq: bytes, pos: int):
    """(positions of aligned bases, their base codes, deleted positions, insertion positions) of one read."""
    ops = [(int(n), op) for n, op in CIGAR_OP.findall(cigar)]
    aligned = [i for i, (n, op) in enumerate(ops) if op in (b"M", b"=", b"X") and n > 0]
    bp, bc, dp, ip = [], [], [], []
    rp, ri = pos, 0
    for i, (n, op) in enumerate(ops):
        if op in (b"M", b"=", b"X"):
            for j in range(n):
                bp.append(rp); bc.append(int(CODE[seq[ri]]))
                rp += 1; ri += 1
        elif op == b"I":
            if n and aligned and aligned[0] < i < aligned[-1] and (not ip or ip[-1] != rp - 1):
                ip.append(rp - 1)
            ri += n
        elif op == b"S":
            ri += n
        elif op == b"D":
            for j in range(n):
                dp.append(rp); rp += 1
        elif op == b"N":
            rp += n
    return bp, bc, dp, ip


def resolve(regions, names: Sequence[str], genome_upper) -> List[Tuple[int, int, int]]:
    """(chromosome, start, last row position) per region; last < start: no rows."""
    idx = {n: k for k, n in enumerate(names)}
    out = []
    for r in regions:
        g = idx[r[0]]
        s = int(r[1]) if len(r) > 1 else 1
        e = int(r[2]) if len(r) > 2 else UINT64_MAX
        out.append((g, s, min(e, len(genome_upper[g]))))
    return out


def pileup(reads, genome_upper, names: Sequence[str], regions, flag_exclude: int = FLAG_EXCLUDE) -> List[np.ndarray]:
    """One [rows, 8] uint32 array per region."""
    regs = resolve(regions, names, genome_upper)
    events = {g: ([], [], [], []) for g, s, e in regs}       # chromosome -> positions of bases, codes, deletions, insertions
    for flag, chr_, pos, cigar, seq in reads:
        if int(flag) & flag_exclude or int(chr_) not in events:
            continue
        for into, got in zip(events[int(chr_)], read_events(cigar, seq, int(pos))):
            into.extend(got)
    events = {g: [np.asarray(x, np.int64) for x in ev] for g, ev in events.items()}
    out = []
    for g, s, e in regs:
        n = e - s + 1 if s <= e else 0
        rows = np.zeros((n, 8), np.uint32)
        if n:
            bp, bc, dp, ip = events[g]
            a = np.zeros((n, 7), np.int64)
            keep = (bp >= s) & (bp <= e)
            np.add.at(a, (bp[keep] - s, bc[keep]), 1)
            for col, p in ((5, dp), (6, ip)):
                np.add.at(a[:, col], p[(p >= s) & (p <= e)] - s, 1)
            rows[:, :7] = a
            rows[:, 7] = genome_upper[g][s - 1:e]
        out.append(rows)
    return out


def batch_reads(b, cigars=None):
    """(flag, chr, pos, cigar, seq) per read of a batch; cigars: per read (default: the batch's own)."""
    c = b.cigar.tobytes()
    s = b.seq.tobytes()
    return [(int(b.flag[i]), int(b.chr[i]), int(b.pos[i]),
             cigars[i] if cigars is not None else c[int(b.cigar_off[i]):int(b.cigar_off[i + 1])],
             s[int(b.seq_off[i]):int(b.seq_off[i + 1])]) for i in range(b.n_reads)]


def sam_reads(text: bytes, names: Sequence[str]):
    """(flag, chr, pos, cigar, seq) per record line of a SAM text."""
    idx = {n.encode(): k for k, n in enumerate(names)}
    out = []
    for ln in text.split(b"\n"):
        if not ln or ln.startswith(b"@"):
            continue
        f = ln.split(b"\t")
        out.append((int(f[1]), idx[f[2]], int(f[3]), f[5], f[9]))
    return out
