"""A catalogue of reads at the limits of the format, built by hand rather than by the synthetic generator: lengths 1 to
252, edit counts at every boundary the kernels branch on, reads at chromosome ends and POS steps around the single
stream's limit, lowercase and N reference bases, N in SEQ. Each case is a Batch, the outcome the CPU oracle gives it
(coded or refused, in the single stream and in blocked containers), and a check of the property the case exists for,
run on the oracle's records so that a change to the builder cannot quietly drop the coverage.

TEST INFRASTRUCTURE: imported by tests/test_oracle_edges.py (CPU) and tests/test_gpu_format_edges.py (GPU)."""
from __future__ import annotations

import re
from dataclasses import dataclass
from typing import Callable, List, Optional

import numpy as np

from cbc_b200.batch import Batch, Genome

MAX_POS_X = 5_000_000          # CBCG_MAX_POS_X: the largest POS step x = pos - prev_pos + 1 of the single stream
K3_EDITS_SMALL = 64            # k3_reconstruct.cu: more edits of one kind than this take the full-size scratch
K1_ECACHE = 4                  # k1_extract.cu: edits per read kept from the count pass
TILE = 128                     # reads per K1 / K3 tile
REF_WINDOW = 8192              # K1_REF_CAP: bytes of reference staged per tile
L_MAX = 252                    # CBCG_MAX_READ_LEN
LENGTHS = [1, 2, 3, 4, 5, 15, 16, 17, 31, 32, 33, 251, 252]

# chromosome lengths 3, 1 and 15 mod 16 (REF_PAD and window arithmetic); e1 carries a lowercase stretch and an N run
CHR_NAMES = ["e0", "e1", "e2"]
CHR_LENS = [5_011, 70_001, 12_000_015]
LOWER = (1_000, 1_400)         # e1[LOWER[0]:LOWER[1]] is lowercase in the genome the GPU is given
NRUN = (2_000, 2_100)          # e1[NRUN[0]:NRUN[1]] is N


def make_genomes(seed: int = 11):
    """(genome for the GPU, the same genome upper-cased for the oracle). The GPU upper-cases on upload."""
    rng = np.random.default_rng(seed)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    bases = [acgt[rng.integers(0, 4, n)].copy() for n in CHR_LENS]
    bases[1][NRUN[0]:NRUN[1]] = ord("N")
    upper = Genome(list(CHR_NAMES), [b.copy() for b in bases])
    lower = [b.copy() for b in bases]
    lower[1][LOWER[0]:LOWER[1]] += 32
    return Genome(list(CHR_NAMES), lower), upper


# ------------------------------------------------------------------ building reads

def _other(b: int, k: int = 1) -> int:
    """A base that differs from reference base b (any base when b is N)."""
    order = b"ACGT"
    if b not in order:
        return order[k % 4]
    return order[(order.index(b) + k) % 4]


class Read:
    """One aligned read, built from the reference by a list of operations, with its CIGAR and standard MD:Z
    ([0-9]+(([A-Z]|^[A-Z]+)[0-9]+)*: a 0 between adjacent mismatches and between a deletion and a mismatch).
    Operations: ("M", n) matches, ("X", n) mismatches, ("D", n) deletion, ("I", n) insertion, ("S", n) soft clip,
    ("N", n) read base N over the reference."""

    def __init__(self, genome: Genome, chr_: int, pos: int, ops, flag: int = 0, seed: int = 0):
        ref = genome.bases[chr_]
        rng = np.random.default_rng(seed + 7919 * pos + 104729 * chr_)
        seq, cig, md = bytearray(), [], []
        run = 0
        p = pos - 1

        def cigar(op, n):
            if cig and cig[-1][0] == op:
                cig[-1][1] += n
            else:
                cig.append([op, n])

        for op, n in ops:
            if op == "M":
                seq += bytes(ref[p:p + n]); run += n; p += n; cigar("M", n)
            elif op in "XN":
                for k in range(n):
                    b = int(ref[p])
                    seq.append(ord("N") if op == "N" else _other(b, 1 + int(rng.integers(0, 3))))
                    md.append(f"{run}{chr(b)}"); run = 0; p += 1
                cigar("M", n)
            elif op == "D":
                md.append(f"{run}^{bytes(ref[p:p + n]).decode()}"); run = 0; p += n; cigar("D", n)
            elif op in "IS":
                seq += bytes(np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)]); cigar(op, n)
            else:
                raise ValueError(op)
        md.append(str(run))
        self.chr, self.pos, self.flag = chr_, pos, flag
        self.seq = bytes(seq)
        self.cigar = "".join(f"{n}{op}" for op, n in cig).encode()
        self.md = "".join(md).encode()
        self.span = p - (pos - 1)                              # reference bases covered


def read_at(genome, chr_, pos, ops, **kw) -> Read:
    return Read(genome, chr_, pos, ops, **kw)


def ending_at(genome, chr_, ops, **kw) -> Read:
    """A read whose reference span ends at the chromosome's last base."""
    span = sum(n for op, n in ops if op in "MXND")
    return Read(genome, chr_, len(genome.bases[chr_]) - span + 1, ops, **kw)


def make_batch(genome: Genome, reads: List[Read]) -> Batch:
    """Position-sorted batch. A single stream names chromosomes in FASTA order, one after the other, so every chromosome
    before the last one used gets a 20-base read at POS 1 when the case has none on it."""
    used = {r.chr for r in reads}
    top = max(used) if used else 0
    reads = list(reads) + [read_at(genome, c, 1, [("M", 20)]) for c in range(top) if c not in used]
    reads.sort(key=lambda r: (r.chr, r.pos))

    def pool(items):
        off = np.zeros(len(items) + 1, np.uint64)
        off[1:] = np.cumsum([len(x) for x in items])
        data = np.frombuffer(b"".join(items), np.uint8).copy() if sum(map(len, items)) else np.zeros(1, np.uint8)
        return off, data
    so, s = pool([r.seq for r in reads])
    co, c = pool([r.cigar for r in reads])
    mo, m = pool([r.md for r in reads])
    return Batch(np.array([r.pos for r in reads], np.uint32), np.array([r.flag for r in reads], np.uint16),
                 np.array([len(r.seq) for r in reads], np.uint16), np.array([r.chr for r in reads], np.uint32),
                 so, s, co, c, mo, m)


# ------------------------------------------------------------------ cases

@dataclass
class Case:
    name: str
    batch: Batch
    L: int                                   # read length in the header: the snps / indels / var alphabets
    extract_ok: bool = True                  # K1 (and the oracle's extraction) accepts every read
    legacy_ok: bool = True                   # the single stream codes it
    blocked_ok: bool = True                  # blocked containers code it
    check: Optional[Callable] = None         # check(batch, recs, edits): the property the case exists for
    regions: Optional[list] = None           # region queries for the region decode (name, start, end)


def _tiles_with_short_line(b):
    return [t for t in range(0, b.n_reads, TILE) if int(b.seq_len[t:t + TILE].min()) + 1 < 17]


def _need(cond, what):
    assert cond, f"precondition lost: {what}"


def cases(genome: Genome) -> List[Case]:
    """genome: the upper-cased genome (the oracle's). The GPU gets make_genomes()[0], which differs only in case."""
    g = genome
    out: List[Case] = []
    clen = [len(b) for b in g.bases]

    # ---- lengths: perfect, all-SNP, one SNP at the first and at the last base
    for n in LENGTHS:
        # n SNPs need an snps alphabet of more than n symbols: at 252 bases the last one matches (snps_L_refused)
        allsnp = [("X", n)] if n < L_MAX else [("X", n - 1), ("M", 1)]
        reads = [read_at(g, 0, 101, [("M", n)]), read_at(g, 0, 401, allsnp)]
        if n >= 2:
            reads += [read_at(g, 0, 701, [("X", 1), ("M", n - 1)]), read_at(g, 0, 1001, [("M", n - 1), ("X", 1)])]

        def chk(b, recs, edits, n=n):
            _need(recs["len"].max() == n and recs["match"][0] == 1, f"a perfect {n}-base read")
            _need(recs["n_snps"].max() == min(n, L_MAX - 1), f"an all-SNP {n}-base read")
        out.append(Case(f"len_{n}", make_batch(g, reads), L_MAX, check=chk, regions=[("e0", 101, 101), ("e0", 1001 + n - 1, 1001 + n - 1)]))

    # a tile of 1..16-base reads only, and a tile of 127 150-base reads and one 1-base read
    reads = []
    for i in range(300):
        n = 1 + i % 16
        ops = [("M", n)] if i % 3 == 0 else ([("X", 1), ("M", n - 1)] if i % 3 == 1 else [("M", n - 1), ("X", 1)])
        if n == 1 and i % 3:
            ops = [("X", 1)]
        reads.append(read_at(g, 0, 50 + 13 * i, ops))
    out.append(Case("short_tile", make_batch(g, reads), 16,
                    check=lambda b, recs, e: _need(int(b.seq_len[:TILE].max()) <= 16 and b.n_reads >= TILE,
                                                   "a whole tile of reads of 16 bases or fewer")))
    reads = [read_at(g, 0, 10 + 20 * i, [("M", 70), ("X", 1), ("M", 79)] if i % 4 else [("M", 150)]) for i in range(127)]
    reads.insert(64, read_at(g, 0, 10 + 20 * 63 + 5, [("X", 1)]))
    reads += [read_at(g, 0, 3_000 + 7 * i, [("M", 150)]) for i in range(40)]
    out.append(Case("tile_127x150_plus_1", make_batch(g, reads), 150,
                    check=lambda b, recs, e: _need(_tiles_with_short_line(b) == [0] and int(b.seq_len[:TILE].max()) == 150,
                                                   "one tile mixing 150-base lines and a 2-byte line")))

    # ---- edit counts
    for k in (4, 5, 63, 64, 65):
        reads = [read_at(g, 1, 3_001 + 11 * i, [("M", 2), ("X", 1)] * k + [("M", 150 - 3 * k)] if 3 * k < 150
                         else [("X", 1), ("M", 1)] * k + [("M", 150 - 2 * k)]) for i in range(3)]
        out.append(Case(f"snps_{k}", make_batch(g, reads), 252,
                        check=lambda b, recs, e, k=k: _need(int(recs["n_snps"].max()) == k, f"{k} SNPs in a read")))
    # K1's edit cache: 4 and 5 edits of mixed kinds
    for k in (K1_ECACHE, K1_ECACHE + 1):
        ops = [("M", 10), ("D", 1), ("M", 10), ("I", 1), ("M", 10), ("X", 1), ("M", 10), ("D", 1), ("M", 10)]
        if k == 5:
            ops += [("I", 1), ("M", 10)]
        reads = [read_at(g, 1, 6_001 + 9 * i, ops) for i in range(40)]
        out.append(Case(f"mixed_edits_{k}", make_batch(g, reads), 100,
                        check=lambda b, recs, e, k=k: _need(
                            int((recs["n_snps"] + recs["n_dels"] + recs["n_ins"]).max()) == k, f"{k} edits of mixed kinds")))
    reads = [read_at(g, 1, 9_001, [("X", 251), ("M", 1)]), read_at(g, 1, 9_301, [("M", 1), ("X", 251)])]
    out.append(Case("snps_L_minus_1", make_batch(g, reads), 252,
                    check=lambda b, recs, e: _need(int(recs["n_snps"].max()) == 251, "251 SNPs at L = 252")))
    out.append(Case("snps_L_refused", make_batch(g, [read_at(g, 1, 9_001, [("X", 252)])]), 252,
                    legacy_ok=False, blocked_ok=False,
                    check=lambda b, recs, e: _need(int(recs["n_snps"].max()) == 252, "252 SNPs at L = 252")))
    for k in (63, 64, 65, 125, 251):
        tail = min(20, L_MAX - k)
        reads = [read_at(g, 1, 12_001 + 600 * i, [("M", 1), ("D", 1)] * k + [("M", tail)], flag=16 * i) for i in range(2)]
        out.append(Case(f"dels_{k}", make_batch(g, reads), 252,
                        check=lambda b, recs, e, k=k: _need(int(recs["n_dels"].max()) == k, f"{k} single-base deletions")))
    out.append(Case("del_run_200", make_batch(g, [read_at(g, 1, 15_001, [("M", 50), ("D", 200), ("M", 50)])]), 252,
                    check=lambda b, recs, e: _need(int(recs["n_dels"].max()) == 200, "a 200-base deletion")))
    out.append(Case("del_run_255_refused", make_batch(g, [read_at(g, 1, 15_001, [("M", 10), ("D", 255), ("M", 10)])]), 252,
                    legacy_ok=False, blocked_ok=False,
                    check=lambda b, recs, e: _need(int(recs["n_dels"].max()) == 255, "255 deletions at L = 252")))
    out.append(Case("del_run_256_refused", make_batch(g, [read_at(g, 1, 15_001, [("M", 10), ("D", 256), ("M", 10)])]), 252,
                    extract_ok=False, legacy_ok=False, blocked_ok=False))
    for k in (64, 65, 200):
        reads = [read_at(g, 1, 16_001 + 50 * i, [("S", k), ("M", 30)] if i % 2 == 0 else [("M", 30), ("S", k)], flag=16 * (i // 2))
                 for i in range(4)]
        out.append(Case(f"clips_{k}", make_batch(g, reads), 252,
                        check=lambda b, recs, e, k=k: _need(int(recs["n_ins"].max()) == k, f"{k}-base soft clips")))
    # several reads of one tile, in different warps, that need K3's full-size scratch; some over the limit in two kinds
    reads = []
    for i in range(TILE):
        p = 20_001 + 40 * i
        if i in (3, 37):
            ops = [("X", 1), ("D", 1)] * 70 + [("M", 60)]         # 70 SNPs and 70 deletions
        elif i in (70, 71):
            ops = [("X", 1), ("I", 1)] * 70 + [("M", 60)]         # 70 SNPs and 70 insertions
        elif i == 101:
            ops = [("M", 1), ("X", 1)] * 100 + [("M", 50)]        # 100 SNPs
        elif i == 127:
            ops = [("M", 1), ("D", 1)] * 66 + [("S", 66), ("M", 20)]   # 66 deletions, 66 insertions
        else:
            ops = [("M", 60), ("X", 1), ("M", 89)]
        reads.append(read_at(g, 1, p, ops, flag=16 * (i % 2)))

    def chk_big(b, recs, e):
        k = np.stack([recs["n_snps"], recs["n_dels"], recs["n_ins"]])[:, :TILE].astype(int)
        big = np.nonzero((k > K3_EDITS_SMALL).any(axis=0))[0]
        _need(len({int(i) // 32 for i in big}) == 4, "reads of one tile in four warps that need the full-size scratch")
        _need(int(((k > K3_EDITS_SMALL).sum(axis=0) >= 2).sum()) >= 4, "reads over the limit in two kinds at once")
    out.append(Case("k3_big_scratch", make_batch(g, reads), 252, check=chk_big))

    # ---- positions
    reads = [read_at(g, c, 1, ops) for c in range(3) for ops in ([("M", 50)], [("X", 1), ("M", 49)])]
    out.append(Case("pos_1", make_batch(g, reads), 100,
                    check=lambda b, recs, e: _need(int((recs["pos"] == 1).sum()) == 6, "reads at POS 1"),
                    regions=[("e0", 1, 1), ("e2", 40, 60)]))
    for c in range(3):
        reads = []
        for n in LENGTHS:
            reads.append(ending_at(g, c, [("M", n)]))
            reads.append(ending_at(g, c, [("M", n - 1), ("X", 1)] if n > 1 else [("X", 1)]))
        reads.append(ending_at(g, c, [("M", 10), ("D", 5), ("M", 10)]))
        # insertions and a trailing clip carry SEQ past the end; the reference span they align to still ends at it
        reads.append(ending_at(g, c, [("M", 10), ("I", 3), ("M", 10)]))
        reads.append(ending_at(g, c, [("M", 20), ("S", 5)]))
        # steps up to e2's end that the single stream can take
        reads += [read_at(g, c, p, [("M", 30)]) for p in range(1, clen[c] - 300, MAX_POS_X - 100)]

        def chk_end(b, recs, e, c=c):
            on = b.chr == c
            ends = b.pos[on].astype(int) + np.array([r for r in _spans(b)])[on] - 1
            _need(int((ends == clen[c]).sum()) == 2 * len(LENGTHS) + 3, f"reads ending at the last base of {CHR_NAMES[c]}")
            _need(int((b.pos[on].astype(int) - 1 + b.seq_len[on] > clen[c]).sum()) == 2, "SEQ past the end, span inside")
        out.append(Case(f"chr_end_{CHR_NAMES[c]}", make_batch(g, reads), 252, check=chk_end,
                        regions=[(CHR_NAMES[c], clen[c], clen[c]), (CHR_NAMES[c], clen[c] - 40, clen[c] - 20)]))
    # reference spans one base past the end: the decoder could not rebuild these, so they are refused
    past = read_at(g, 0, 1, [("M", 20)])
    past.pos = clen[0] - 18                                   # 20 bases, the last one past the end
    past.seq = bytes(g.bases[0][clen[0] - 19:]) + b"A"
    past.cigar, past.md = b"20M", b"20"
    out.append(Case("one_past_chr_end_refused", make_batch(g, [read_at(g, 0, 4_000, [("M", 30)]), past]), 100,
                    extract_ok=False, legacy_ok=False, blocked_ok=False))
    del_past = ending_at(g, 0, [("M", 10), ("D", 5), ("M", 10)])
    del_past.pos += 1                                         # SEQ inside, the deletion pushes the span past the end
    out.append(Case("deletion_past_chr_end_refused", make_batch(g, [read_at(g, 0, 4_000, [("M", 30)]), del_past]), 100,
                    extract_ok=False, legacy_ok=False, blocked_ok=False))
    reads = [read_at(g, 1, 30_001, [("M", 100)] if i % 3 else [("M", 40), ("X", 1), ("M", 59)], flag=i % 7)
             for i in range(300)]
    reads += [read_at(g, 1, 30_002, [("M", 100)]) for _ in range(3)]
    out.append(Case("same_pos_300", make_batch(g, reads), 100,
                    check=lambda b, recs, e: _need(int((recs["pos"] == 30_001).sum()) == 300, "300 reads at one POS"),
                    regions=[("e1", 30_100, 30_100), ("e1", 30_101, 30_101)]))
    reads = [read_at(g, 1, 40_001 + 97 * i, [("M", 80)] if i % 2 else [("M", 30), ("X", 2), ("M", 48)]) for i in range(2 * TILE)]
    out.append(Case("tile_wider_than_window", make_batch(g, reads), 80,
                    check=lambda b, recs, e: _need(int(b.pos[TILE - 1]) - int(b.pos[0]) > REF_WINDOW,
                                                   "a tile whose reads span more than the 8 KiB window")))
    # POS steps x = pos - prev_pos + 1 around the single stream's limit, inside a chromosome
    for x in (MAX_POS_X - 1, MAX_POS_X, MAX_POS_X + 1, 6_000_000, 11_000_000):
        p0 = 501
        reads = [read_at(g, 2, p0 + 30 * i, [("M", 100)] if i % 2 else [("M", 50), ("X", 1), ("M", 49)]) for i in range(20)]
        last = p0 + 30 * 19
        reads += [read_at(g, 2, last + x - 1 + 30 * i, [("M", 100)] if i % 2 else [("M", 20), ("X", 1), ("M", 79)])
                  for i in range(20)]

        def chk_gap(b, recs, e, x=x):
            _need(int(np.diff(b.pos[b.chr == 2].astype(np.int64)).max()) + 1 == x, f"a POS step of {x}")
        out.append(Case(f"pos_step_{x}", make_batch(g, reads), 100, legacy_ok=x <= MAX_POS_X, check=chk_gap,
                        regions=[("e2", last + x - 1 - 10, last + x - 1 + 10), ("e2", last, last + x - 200)]))
    reads = [read_at(g, 2, 101 + 40 * i, [("M", 90), ("X", 1), ("M", 9)]) for i in range(6)]
    reads += [read_at(g, 2, 5_000_301 + 40 * i, [("M", 100)]) for i in range(6)]
    reads += [read_at(g, 2, 11_000_501 + 40 * i, [("M", 40), ("X", 1), ("M", 59)]) for i in range(6)]

    def chk_gaps(b, recs, e):
        steps = np.diff(b.pos[b.chr == 2].astype(np.int64))[:15] + 1
        _need(int((steps > MAX_POS_X).sum()) == 2, "two steps over 5 M among the first 16 reads of a chromosome")
    out.append(Case("pos_steps_in_one_block", make_batch(g, reads), 100, legacy_ok=False, check=chk_gaps,
                    regions=[("e2", 5_000_000, 5_000_400), ("e2", 11_000_000, 12_000_015)]))

    # ---- reference bases
    reads = [read_at(g, 1, LOWER[0] - 50 + 25 * i, [("M", 100)] if i % 2 else [("M", 45), ("X", 2), ("M", 53)]) for i in range(18)]
    out.append(Case("lowercase_reference", make_batch(g, reads), 100,
                    check=lambda b, recs, e: _need(int(b.pos[0]) < LOWER[0] < int(b.pos[-1]) < LOWER[1], "reads over the lowercase stretch")))
    reads = [read_at(g, 1, NRUN[0] - 60 + 20 * i, [("M", 100)] if i % 2 else [("M", 50), ("X", 1), ("M", 49)]) for i in range(10)]

    def chk_refn(b, recs, e):
        _need((g.bases[1][NRUN[0]:NRUN[1]] == ord("N")).all(), "an N run")
        snp_refn = ((e >> 11) & 7) == 4                          # CBCG_EDIT(delta, target, refb): refb in bits 11..13
        _need(bool(snp_refn.any()), "a SNP with N on the reference side")
        _need(int(recs["match"].sum()) >= 3, "perfect matches over the N run")
    out.append(Case("reference_n_run", make_batch(g, reads), 100, check=chk_refn))
    reads = [read_at(g, 0, 2_001 + 30 * i, [("M", 10), ("N", 1 + i % 3), ("M", 30), ("N", 1), ("M", 20)]) for i in range(40)]
    reads += [read_at(g, 0, 3_300, [("N", 60)])]
    out.append(Case("n_in_seq", make_batch(g, reads), 100,
                    check=lambda b, recs, e: _need(int((b.seq == ord("N")).sum()) > 100, "N bases in SEQ")))

    # ---- MD spellings: a 0 between adjacent mismatches, multi-digit runs, a ^ run next to a mismatch on either side
    reads = [read_at(g, 0, 4_201, [("M", 12), ("X", 3), ("M", 123), ("D", 2), ("X", 1), ("M", 10), ("X", 1), ("D", 3), ("M", 20)]),
             read_at(g, 0, 4_501, [("X", 1), ("D", 1), ("X", 1), ("M", 100), ("I", 2), ("X", 1), ("M", 9)])]

    def chk_md(b, recs, e):
        md = b.md.tobytes()
        for pat in (rb"[ACGTN]0[ACGTN]", rb"[0-9]{3}", rb"\^[ACGTN]+0[ACGTN]", rb"[ACGTN]0\^"):
            _need(re.search(pat, md), f"an MD spelling matching {pat!r}")
    out.append(Case("md_spellings", make_batch(g, reads), 252, check=chk_md))
    return out


def _spans(b):
    text = b.cigar.tobytes()
    return [sum(int(n) for n, op in re.findall(rb"(\d+)([MIDSHP=X])", text[b.cigar_off[i]:b.cigar_off[i + 1]])
                if op in b"MD=X") for i in range(b.n_reads)]
