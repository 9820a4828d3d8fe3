"""The BAM restatement (tests/bam_restate.py) against an independent reader and zlib / gzip, and the command line's -Z
argument checks. CPU only: the GPU side is tests/test_gpu_bam.py, which compares cbcg_decode_bam with this restatement
byte for byte."""
import gzip
import os
import random
import struct
import subprocess
import zlib

import pytest

import bam_restate as B
import edge_reads as E
import sam_restate as R
from cbc_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "cbc_b200", "_build", "cbc")

SHAPES = {   # test_gpu_sam.py's shapes
    "config1": dict(seed=71, genome_len=2_000_000, n_chr=2, n_reads=30_000, len_min=100, len_max=100, p_sub=0.005,
                    p_indel=0.002, p_clip=0.05),
    "config5": dict(seed=72, genome_len=2_000_000, n_chr=2, n_reads=20_000, len_min=50, len_max=250, p_sub=0.005,
                    p_indel=0.02, p_clip=0.3),
}


def _shape(name):
    cfg = synth.SynthConfig(**SHAPES[name])
    g = synth.make_genome(cfg)
    b = synth.make_reads(cfg, g)
    return g, R.sam_lines(b, R.upper(g), g.names)


def _seq_coded(line: bytes) -> bytes:
    """A SAM line with its SEQ through the 4-bit code, as a BAM reader gives it back."""
    f = line.split(b"\t")
    f[9] = bytes(B.NT16[B._code(c)] for c in f[9])
    return b"\t".join(f)


def _check(lines, names, lengths):
    data = B.bam(lines, names, lengths)
    got_names, got_len, text, got = B.read_bam(data)
    assert got_names == list(names) and got_len == list(lengths)
    assert text == R.header(names, lengths)
    assert got == [_seq_coded(x) for x in lines]
    # gzip reads the concatenated members as one stream: the header, then every record
    idx = {n.encode(): k for k, n in enumerate(names)}
    stream = gzip.decompress(data)
    assert stream.endswith(b"".join(B.record(x, idx)[0] for x in lines))
    for _, total, raw in B.members(data):
        assert total <= 65536 and len(raw) <= 65280
    return data


@pytest.mark.parametrize("shape", list(SHAPES))
def test_shapes_read_back_as_the_sam_lines(shape):
    g, lines = _shape(shape)
    lengths = [x.size for x in g.bases]
    data = _check(lines, g.names, lengths)
    ms = B.members(data)
    assert len(ms) > 3                                   # several record blocks
    # every record member but the last holds >= the cut's worth of records, the call's last one the rest
    recs = [m for m in ms[1:-1]]
    assert all(len(m[2]) < B.CUT + B.MAX_RECORD for m in recs)
    assert sum(len(m[2]) for m in recs[:-1]) // B.CUT == len(recs) - 1


def test_edge_catalogue_reads_back():
    gpu_genome, genome = E.make_genomes()
    up = R.upper(gpu_genome)
    lines = []
    for c in E.cases(genome):
        if c.blocked_ok:
            lines += R.sam_lines(c.batch, up, E.CHR_NAMES)
    lengths = [x.size for x in gpu_genome.bases]
    _check(lines, E.CHR_NAMES, lengths)


def test_cut_rule():
    assert B.cut([]) == []
    assert B.cut([100] * 3) == [(0, 3)]
    # record 491 starts at 49 100 (block 0), record 492 at 49 200: floor changes -> a new block there
    sizes = [100] * 1000
    assert B.cut(sizes) == [(0, 492), (492, 984), (984, 1000)]
    sizes = [8000] * 20
    blocks = B.cut(sizes)
    assert all(sum(sizes[a:b]) < B.CUT + B.MAX_RECORD for a, b in blocks)


def _long_line(rng, pos):
    """A 252-base read with a long verbatim CIGAR: one-base operations, hard clips and padding between them."""
    ops, q = [], 0
    while q < 252:
        k = rng.choice("MIS=XHP")
        if k in "MIS=X":
            ops.append(b"1" + k.encode()); q += 1
        else:
            ops.append(b"%d%c" % (rng.randrange(1, 10**6), ord(k)))
    seq = bytes(rng.choice(b"ACGTN") for _ in range(252))
    md = b"0" + b"".join(b"A0" for _ in range(100))
    return b"\t".join([b"*", b"0", b"c1", b"%d" % pos, b"255", b"".join(ops), b"*", b"0", b"0", seq, b"*", b"NM:i:300",
                       b"MD:Z:" + md]) + b"\n"


def test_maximum_length_reads_with_long_verbatim_cigars_keep_the_block_limits():
    rng = random.Random(5)
    lines = [_long_line(rng, 1000 + i) for i in range(120)]
    idx = {b"c1": 0}
    sizes = [len(B.record(x, idx)[0]) for x in lines]
    assert max(sizes) > 2000 and max(sizes) <= B.MAX_RECORD
    data = _check(lines, ["c1"], [1 << 20])
    for _, total, raw in B.members(data)[1:-1]:
        assert len(raw) < B.CUT + B.MAX_RECORD and total <= 65536
    # NM above 255 is typed S
    rec = B.record(lines[0], idx)[0]
    assert b"NMS" + struct.pack("<H", 300) in rec


def test_worst_case_block_fits_the_bgzf_limit():
    """57 343 bytes of nine-bit literals: the largest block the cut allows."""
    bw = B.BitWriter()
    bw.bits(1, 1); bw.bits(1, 2)
    raw = bytes([200]) * (B.CUT + B.MAX_RECORD - 1)
    for b in raw:
        bw.lit(b)
    bw.lit(256)
    block = B.gzip_member(bw.flush(), raw)
    assert len(block) == 64539 and zlib.decompress(block[18:-8], -15) == raw


def test_header_of_thousands_of_long_names_spans_several_blocks():
    names = [f"contig_{k:05d}_" + "x" * 180 for k in range(3000)]
    lengths = [1000 + k for k in range(3000)]
    h = B.header(names, lengths)
    ms = B.members(h + B.EOF_BLOCK)
    assert len(ms) >= 10 and all(len(m[2]) == B.STORED for m in ms[:-2])
    got_names, got_len, text, lines = B.read_bam(h + B.EOF_BLOCK)
    assert got_names == names and got_len == lengths and lines == []
    assert text == R.header(names, lengths)


def test_eof_block_is_an_empty_member():
    assert gzip.decompress(B.EOF_BLOCK) == b""
    assert B.members(B.EOF_BLOCK)[0][1:] == (28, b"")


def _cli(*args):
    return subprocess.run([CLI, *args], capture_output=True, text=True, timeout=60)


@pytest.mark.skipif(not os.path.exists(CLI), reason="cbc is not built")
def test_cli_bam_argument_errors(tmp_path):
    src, out, fa = (str(tmp_path / x) for x in ("in.cbc", "out.bam", "r.fa"))
    for flags in (["-Z", "-S"], ["-Z", "-P", "-r", "c1"], ["-c", "-Z"]):
        p = _cli(*flags, src, out, fa) if "-c" in flags else _cli("-d", *flags, src, out, fa)
        assert p.returncode == 2 and "-Z" in p.stderr, (flags, p.stderr)
