"""The pileup restatement (tests/pileup_restate.py) on hand-built reads, and the command line's -P argument checks. CPU
only: the GPU side is tests/test_gpu_pileup.py, which compares cbcg_pileup with this restatement."""
import os
import subprocess

import numpy as np
import pytest

import pileup_restate as P
from sam_restate import CIGAR_OP

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "cbc_b200", "_build", "cbc")
NAMES = ["c1", "c2"]
GENOME = [np.frombuffer(b"ACGTACGTNNACGTACGTAC", np.uint8).copy(), np.frombuffer(b"TTTTGGGGCCCCAAAA", np.uint8).copy()]
A, C, G, T, N, DEL, INS, REF = range(8)


def _rows(reads, regions, **kw):
    return P.pileup(reads, GENOME, NAMES, regions, **kw)


def _col(rows, c):
    return rows[:, c].tolist()


def test_leading_and_trailing_insertions_and_clips_never_count():
    # 2S 5M 1I 3M 2I at POS 3: aligned 3..7, an interior insertion after 7, aligned 8..10, a trailing insertion
    seq = b"TT" + bytes(GENOME[0][2:7]) + b"A" + bytes(GENOME[0][7:10]) + b"GG"
    for cig in (b"2S5M1I3M2I", b"2I5M1I3M2S", b"2I5M1I3M2I"):
        (r,) = _rows([(0, 0, 3, cig, seq)], [("c1", 1, 12)])
        assert _col(r, INS) == [0] * 6 + [1] + [0] * 5, cig
        depth = r[:, :5].sum(axis=1).tolist()
        assert depth == [0, 0] + [1] * 8 + [0, 0]
        assert (r[:, REF] == GENOME[0][:12]).all()


def test_insertion_next_to_a_deletion_counts_after_the_last_reference_base():
    seq = b"ACGTTACG"
    (r,) = _rows([(0, 0, 1, b"3M2I2D3M", seq)], [("c1", 1, 10)])
    assert _col(r, INS) == [0, 0, 1] + [0] * 7                # after POS 3, before the deletion
    assert _col(r, DEL) == [0, 0, 0, 1, 1, 0, 0, 0, 0, 0]
    (r,) = _rows([(0, 0, 1, b"3M2D2I3M", seq)], [("c1", 1, 10)])
    assert _col(r, INS) == [0, 0, 0, 0, 1] + [0] * 5          # after the deleted POS 5
    assert _col(r, DEL) == [0, 0, 0, 1, 1, 0, 0, 0, 0, 0]
    (r,) = _rows([(0, 0, 1, b"3M2I1P1I3M", b"ACGTTCACG")], [("c1", 1, 10)])
    assert _col(r, INS) == [0, 0, 1] + [0] * 7                # two I operations at one position count once


def test_eq_x_hard_clips_and_padding():
    # 2H 3= 1X 2P 1I 2M at POS 11 (ACGTACGTAC from 11): aligned 11..16, an insertion after 14
    seq = b"ACG" + b"A" + b"C" + b"AC"
    (r,) = _rows([(0, 0, 11, b"2H3=1X2P1I2M", seq)], [("c1", 11, 16)])
    assert _col(r, A) == [1, 0, 0, 1, 1, 0]
    assert _col(r, C) == [0, 1, 0, 0, 0, 1]
    assert _col(r, G) == [0, 0, 1, 0, 0, 0]
    assert _col(r, T) == [0] * 6
    assert _col(r, INS) == [0, 0, 0, 1, 0, 0]
    assert _col(r, REF) == list(b"ACGTAC")


def test_n_in_the_read_and_in_the_reference():
    # POS 7: reference GTNNAC; the read has N over G and A, C over the reference's N
    (r,) = _rows([(0, 0, 7, b"6M", b"NTNCNC")], [("c1", 7, 12)])
    assert _col(r, N) == [1, 0, 1, 0, 1, 0]
    assert _col(r, C) == [0, 0, 0, 1, 0, 1]
    assert _col(r, T) == [0, 1, 0, 0, 0, 0]
    assert _col(r, REF) == list(b"GTNNAC")
    # a base that is neither A, C, G nor T counts as N
    (r,) = _rows([(0, 1, 1, b"2M", b"RY")], [("c2", 1, 2)])
    assert _col(r, N) == [1, 1]


def test_runs_at_region_ends_and_reads_that_start_before_a_region():
    seq = bytes(GENOME[0][:10])
    reads = [(0, 0, 1, b"10M", seq), (0, 0, 3, b"4M2D2M", bytes(GENOME[0][2:6]) + bytes(GENOME[0][8:10]))]
    (r,) = _rows(reads, [("c1", 5, 8)])
    assert r[:, :5].sum(axis=1).tolist() == [2, 2, 1, 1]      # the second read: 3..6, deleted 7..8, 9..10
    assert _col(r, DEL) == [0, 0, 1, 1]
    (r,) = _rows(reads, [("c1", 10, 10)])
    assert r[:, :5].sum(axis=1).tolist() == [2]


def test_overlapping_repeated_and_past_the_end_regions():
    rng = np.random.default_rng(1)
    reads = []
    for p in sorted(rng.integers(1, 15, size=20).tolist()):
        reads.append((0, 0, p, b"6M", bytes(rng.choice(list(b"ACGTN"), 6).astype(np.uint8))))
    full, a, b, again, past, whole = _rows(reads, [("c1", 1, 20), ("c1", 1, 5), ("c1", 3, 9), ("c1", 3, 9), ("c1", 25, 30), ("c1",)])
    assert np.array_equal(a, full[0:5]) and np.array_equal(b, full[2:9]) and np.array_equal(again, b)
    assert past.shape == (0, 8) and np.array_equal(whole, full)
    (end,) = _rows(reads, [("c1", 18, 1 << 40)])
    assert np.array_equal(end, full[17:20])
    with pytest.raises(KeyError):
        _rows(reads, [("chrNone", 1, 5)])


def test_flags_are_excluded_by_the_mask():
    seq = bytes(GENOME[1][:4])
    reads = [(f, 1, 1, b"4M", seq) for f in (0, 16, 0x4, 0x100, 0x200, 0x400, 0x800)]
    (r,) = _rows(reads, [("c2", 1, 4)])
    assert _col(r, T) == [3] * 4                               # 0, 16 and the supplementary 0x800
    (r,) = _rows(reads, [("c2", 1, 4)], flag_exclude=0)
    assert _col(r, T) == [7] * 4


def test_depth_equals_the_coverage_of_the_reference_spans():
    """A+C+G+T+N is the number of reads whose M / = / X operations cover a position, computed from the spans."""
    rng = np.random.default_rng(7)
    g = [rng.choice(list(b"ACGTN"), 3000).astype(np.uint8)]
    reads, cover = [], np.zeros(3002, np.int64)
    for _ in range(300):
        p = int(rng.integers(1, 2700))
        ops, n_read = [], 0
        for _ in range(int(rng.integers(1, 6))):
            op = rng.choice([b"M", b"=", b"X", b"I", b"D", b"S", b"H", b"P"])
            ops.append((int(rng.integers(1, 12)), op))
        cig = b"".join(b"%d%s" % (n, op) for n, op in ops)
        n_read = sum(n for n, op in ops if op in (b"M", b"=", b"X", b"I", b"S"))
        reads.append((0, 0, p, cig, bytes(rng.choice(list(b"ACGTN"), n_read).astype(np.uint8))))
        rp = p
        for n, op in CIGAR_OP.findall(cig):
            n = int(n)
            if op in (b"M", b"=", b"X"):
                cover[rp:rp + n] += 1
            if op in (b"M", b"=", b"X", b"D", b"N"):
                rp += n
    (r,) = P.pileup(reads, g, ["x"], [("x",)])
    assert r[:, :5].sum(axis=1).tolist() == cover[1:3001].tolist()


def _cli(*args):
    return subprocess.run([CLI, *args], capture_output=True, text=True, timeout=60)


@pytest.mark.skipif(not os.path.exists(CLI), reason="cbc is not built")
def test_cli_pileup_argument_errors():
    for args, msg in ((["-d", "-P", "a", "b", "c"], "-r"), (["-d", "-P", "-S", "-r", "x", "a", "b", "c"], "-S"),
                      (["-c", "-P", "a", "b", "c"], "-d"), (["-d", "-F", "4", "-r", "x", "a", "b", "c"], "-P"),
                      (["-d", "-P", "-F", "0xz", "-r", "x", "a", "b", "c"], "mask")):
        p = _cli(*args)
        assert p.returncode == 2 and msg in p.stderr, (args, p.stderr)
