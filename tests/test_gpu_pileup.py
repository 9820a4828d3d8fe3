"""Pileup on the GPU (cbcg_pileup, Codec.pileup, `cbc -d -P`): every row against the restatement in tests/pileup_restate.py,
over the input batch's CIGARs (with the CIGAR side section), over the implied CIGARs of the oracle's records (without it)
and over the lines cbcg_decode_sam returns for the same regions. Every decode runs with CBCG_POISON_DECODE=1."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import edge_reads as E
import oracle_lib as O
import pileup_restate as P
import sam_restate as R
from cbc_b200 import synth
from cbc_b200.batch import Batch, Genome
from cbc_b200.codec import CbcgError, Codec
from test_region_plan import model_plan, parse_container

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "cbc_b200", "_build", "cbc")
AUTO = 0xFFFFFFFF
ERR_ARG, ERR_CAPACITY, ERR_NO_REFERENCE, ERR_FORMAT = -1, -5, -7, -8

SHAPES = {   # two chromosomes, sparse coverage, variable length, indels and clips: as the region tests
    "config1": (dict(seed=71, genome_len=2_000_000, n_chr=2, n_reads=30_000, len_min=100, len_max=100, p_sub=0.005,
                     p_indel=0.002, p_clip=0.05), 100),
    "config5": (dict(seed=72, genome_len=2_000_000, n_chr=2, n_reads=20_000, len_min=50, len_max=250, p_sub=0.005,
                     p_indel=0.02, p_clip=0.3), 250),
}
SETTINGS = [  # (gen_mode, block_reads, substreams)
    (1, AUTO, 0), (1, AUTO, 1), (1, AUTO, 4), (0, 1024, 1), (1, 400, 1),
]


@pytest.fixture(autouse=True)
def _poison(monkeypatch):
    monkeypatch.setenv("CBCG_POISON_DECODE", "1")


@pytest.fixture(scope="module")
def codec():
    c = Codec(0)
    yield c
    c.close()


_CACHE = {}


def _shape(name):
    """genome, batch, L, upper-cased genome, reads by the input CIGARs, reads by the implied CIGARs"""
    if name not in _CACHE:
        kw, L = SHAPES[name]
        cfg = synth.SynthConfig(**kw)
        g = synth.make_genome(cfg)
        b = synth.make_reads(cfg, g)
        recs, edits = O.extract(b, g)
        implied = [R.implied_cigar(recs[i], edits) for i in range(b.n_reads)]
        _CACHE[name] = (g, b, L, R.upper(g), P.batch_reads(b), P.batch_reads(b, implied))
    return _CACHE[name]


def _regions(g, b):
    n0, n1 = g.bases[0].size, g.bases[1].size
    p = int(b.pos[b.n_reads // 3])
    return [
        (g.names[0], 1, 300),                                # the early generations
        (g.names[1], int(n1 * 0.5), int(n1 * 0.5) + 2_000),   # the middle
        (g.names[0], n0 - 700, n0 + 1_000),                  # across the record's end
        (g.names[1],),                                       # a whole record
        (g.names[0], p, p + 500), (g.names[0], p + 200, p + 900), (g.names[0], p, p + 500),   # overlapping, repeated
        (g.names[0], 40_000, 40_100),                        # unsorted
        (g.names[0], n0 + 10, n0 + 20),                      # past the end: no rows
    ]


_WANT = {}


def _want(shape, which, regs):
    """the restatement of a shape's regions over its input ("input") or implied ("implied") CIGARs, computed once"""
    if (shape, which) not in _WANT:
        g, b, L, up, reads, implied = _shape(shape)
        _WANT[(shape, which)] = P.pileup(reads if which == "input" else implied, up, g.names, regs)
    return _WANT[(shape, which)]


def _same(got, want, regions):
    assert len(got) == len(want) == len(regions)
    for g_, w, r in zip(got, want, regions):
        assert g_.shape == w.shape, r
        if not np.array_equal(g_, w):
            bad = np.nonzero((g_ != w).any(axis=1))[0]
            raise AssertionError(f"{r}: {len(bad)} rows differ, first at {bad[0]}: {g_[bad[0]].tolist()} != {w[bad[0]].tolist()}")


@pytest.mark.parametrize("setting", SETTINGS, ids=[f"g{s[0]}_b{'auto' if s[1] == AUTO else s[1]}_s{s[2]}" for s in SETTINGS])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_pileup_matches_the_input(codec, shape, setting):
    g, b, L, up, reads, implied = _shape(shape)
    gen_mode, block_reads, sub = setting
    codec.set_reference(g)
    cont = codec.compress(b, L, block_reads=block_reads, gen_mode=gen_mode, substreams=sub)
    sec = codec.cigar_pack(b)
    regs = _regions(g, b)
    got = codec.pileup(cont, regs, sec)
    _same(got, _want(shape, "input", regs), regs)
    assert got[-1].shape == (0, 8) and int(got[3][:, :5].sum()) > 0
    _same(codec.pileup(cont, regs), _want(shape, "implied", regs), regs)
    if setting == SETTINGS[0]:
        # the lines decode_sam returns for the same regions
        for s in (sec, None):
            text, _ = codec.decompress_sam(cont, s, regions=regs, header=False)
            lines = P.sam_reads(text, g.names)
            _same(codec.pileup(cont, regs, s), P.pileup(lines, up, g.names, regs), regs)
            assert codec.last_pileup_reads == len(lines)


def test_flag_exclude(codec):
    g, b0, L, up, _, _ = _shape("config1")
    rng = np.random.default_rng(4)
    values = np.array([0, 16, 0x4, 0x100, 0x200, 0x400, 0x800, 0x10 | 0x400, 1 | 2 | 64], np.uint16)
    flag = np.ascontiguousarray(values[rng.integers(0, values.size, size=b0.n_reads)])
    b = Batch(b0.pos, flag, b0.seq_len, b0.chr, b0.seq_off, b0.seq, b0.cigar_off, b0.cigar, b0.md_off, b0.md)
    codec.set_reference(g)
    cont = codec.compress(b, L, block_reads=AUTO, gen_mode=1)
    sec = codec.cigar_pack(b)
    reads = P.batch_reads(b)
    regs = [(g.names[0], 1, 60_000), (g.names[1], 100_000, 140_000)]
    for mask in (0x704, 0, 0x10, 0xffff):
        got = codec.pileup(cont, regs, sec, flag_exclude=mask)
        _same(got, P.pileup(reads, up, g.names, regs, flag_exclude=mask), regs)


GPU_GENOME, GENOME = E.make_genomes()
EDGE = [c for c in E.cases(GENOME) if c.blocked_ok]
EDGE_UP = R.upper(GPU_GENOME)


def _edge_regions(b):
    """a region around each cluster of reads (POS steps of millions of bases are not one region)"""
    regs = []
    for c in sorted(set(b.chr.tolist())):
        p = np.sort(b.pos[b.chr == c].astype(np.int64))
        cut = np.nonzero(np.diff(p) > 2_000)[0]
        for lo, hi in zip(np.r_[0, cut + 1], np.r_[cut, p.size - 1]):
            regs.append((E.CHR_NAMES[c], max(1, int(p[lo]) - 5), int(p[hi]) + 600))
    return regs


@pytest.mark.parametrize("case", EDGE + ["general"], ids=[c.name for c in EDGE] + ["general_path_cigars"])
def test_edge_catalogue(codec, case):
    if case == "general":
        from test_gpu_sam import _general_batch
        b, L = _general_batch(), 100
    else:
        b, L = case.batch, case.L
    codec.set_reference(GPU_GENOME)
    cont = codec.compress(b, L, block_reads=16, gen_mode=1)
    sec = codec.cigar_pack(b)
    regs = _edge_regions(b)
    _same(codec.pileup(cont, regs, sec), P.pileup(P.batch_reads(b), EDGE_UP, E.CHR_NAMES, regs), regs)
    recs, edits = O.extract(b, GENOME)
    implied = P.batch_reads(b, [R.implied_cigar(recs[i], edits) for i in range(b.n_reads)])
    _same(codec.pileup(cont, regs), P.pileup(implied, EDGE_UP, E.CHR_NAMES, regs), regs)


def test_legacy_stream_and_a_batch_without_md(codec):
    g, b, L, up, reads, implied = _shape("config5")
    codec.set_reference(g)
    sec = codec.cigar_pack(b)
    regs = [(g.names[1], 5_000, 9_000), (g.names[0], 1, 100), (g.names[0], 300_000, 330_000)]
    stream = codec.compress(b, L, block_reads=0)
    _same(codec.pileup(stream, regs, sec, legacy=True), P.pileup(reads, up, g.names, regs), regs)
    _same(codec.pileup(stream, regs, legacy=True), P.pileup(implied, up, g.names, regs), regs)
    assert codec.stats()["n_blocks"] == 1
    cont = codec.compress(b.without_md(), L, block_reads=AUTO, gen_mode=1)     # MD derived by K7
    _same(codec.pileup(cont, regs, sec), P.pileup(reads, up, g.names, regs), regs)


def test_names_in_the_reference_and_not_in_the_container(codec):
    g, b, L, up, reads, _ = _shape("config1")
    codec.set_reference(g)
    cont = codec.compress(b, L, block_reads=AUTO, gen_mode=1)
    extra = np.frombuffer(b"acgtNNNNACGT" * 50, np.uint8).copy()
    codec.set_reference(Genome(list(g.names) + ["chrExtra"], list(g.bases) + [extra]))
    regs = [("chrExtra", 5, 100), (g.names[0], 1_000, 3_000), ("chrExtra",)]
    got = codec.pileup(cont, regs)
    assert got[0].shape == (96, 8) and not got[0][:, :7].any()
    assert got[0][:, 7].astype(np.uint8).tobytes() == bytes(R.upper(Genome(["x"], [extra]))[0][4:100])
    assert got[2].shape == (extra.size, 8) and not got[2][:, :7].any()
    _same(got[1:2], P.pileup(reads, up, g.names, regs[1:2], ), regs[1:2])
    with pytest.raises(CbcgError) as e:
        codec.pileup(cont, [(g.names[0], 1, 10), ("chrNone", 1, 10)])
    assert e.value.status == ERR_NO_REFERENCE
    codec.set_reference(g)


def test_capacity_is_answered_before_any_decode_and_errors(codec):
    g, b, L, up, reads, _ = _shape("config5")
    codec.set_reference(g)
    cont = codec.compress(b, L, block_reads=AUTO, gen_mode=1, substreams=0)
    sec = codec.cigar_pack(b)
    n1 = g.bases[1].size
    regs = [(g.names[1], int(n1 * 0.6), int(n1 * 0.6) + 2_000), (g.names[0], 10, 19), (g.names[1], n1 - 5, n1 + 50)]
    want = P.pileup(reads, up, g.names, regs)
    # every payload byte overwritten: the capacity answer needs none of them
    h = parse_container(cont)
    bad = bytearray(cont)
    bad[h["payload_off"]:] = b"\xff" * (len(cont) - h["payload_off"])
    from cbc_b200 import codec as cm
    arr, nr = cm._region_array(regs)
    src = np.frombuffer(bytes(bad), np.uint8)
    per = np.zeros(3, np.uint64)
    n = C.c_uint64(0)
    rows = np.zeros((4, 8), np.uint32)
    for ptr, cap in ((None, 0), (rows.ctypes.data, 4)):
        rc = codec.lib.cbcg_pileup(codec.h, src.ctypes.data, src.nbytes, 0, None, 0, arr, nr, 0x704, ptr, cap, C.byref(n),
                                   per.ctypes.data, None)
        assert rc == ERR_CAPACITY and n.value == sum(w.shape[0] for w in want)
        assert per.tolist() == [2_001, 10, 6]
    # untouched payload overwritten: the same rows
    sel = set(model_plan(cont, regs[:1])[4])
    bad = bytearray(cont)
    for k, blk in enumerate(h["blocks"]):
        if k not in sel and blk["pay"]:
            at = h["payload_off"] + blk["pay_off"]
            bad[at:at + blk["pay"]] = b"\xff" * blk["pay"]
    _same(codec.pileup(bytes(bad), regs[:1], sec), want[:1], regs[:1])
    # errors
    for regs_bad in ([], [(g.names[0], 0, 10)], [(g.names[0], 20, 10)]):
        with pytest.raises(CbcgError) as e:
            codec.pileup(cont, regs_bad, sec)
        assert e.value.status == ERR_ARG
    other = codec.cigar_pack(b.slice(0, b.n_reads - 1))
    with pytest.raises(CbcgError) as e:
        codec.pileup(cont, regs, other)
    assert e.value.status == ERR_FORMAT


def _run(*args, ok=True):
    p = subprocess.run([CLI, *args], capture_output=True, text=True, timeout=300)
    if ok:
        assert p.returncode == 0, p.stdout + p.stderr
    return p


def _tsv(rows, names, regions, genome_upper):
    out = [b"#chrom\tpos\tref\tA\tC\tG\tT\tN\tdel\tins\n"]
    for (g, s, e), r in zip(P.resolve(regions, names, genome_upper), rows):
        for k in range(r.shape[0]):
            x = r[k]
            out.append(b"%s\t%d\t%c\t%d\t%d\t%d\t%d\t%d\t%d\t%d\n" % (names[g].encode(), s + k, int(x[7]), *[int(v) for v in x[:7]]))
    return b"".join(out)


def test_cli_pileup_of_a_multi_batch_file():
    from cbc_b200 import shard
    cfg = synth.SynthConfig(seed=73, genome_len=1_200_000, n_chr=2, n_reads=40_000, len_min=100, len_max=100, p_sub=0.005,
                            p_indel=0.002, p_clip=0.05)
    g = synth.make_genome(cfg); b = synth.make_reads(cfg, g)
    up = R.upper(g)
    recs, edits = O.extract(b, g)
    implied = P.batch_reads(b, [R.implied_cigar(recs[i], edits) for i in range(b.n_reads)])
    with tempfile.TemporaryDirectory() as d:
        fa, sam, cbcs, out = (os.path.join(d, x) for x in ("r.fa", "r.sam", "a.cbcs", "o.tsv"))
        synth.write_fasta(fa, g); synth.write_sam(sam, b, g)
        _run("-c", "-C", "-B", "1", sam, cbcs, fa)
        with open(cbcs, "rb") as f:
            shards = shard.read_shards(f.read())
        assert len(shards) >= 3
        ends = np.cumsum([int.from_bytes(s[16:24], "little") for s in shards])
        r = int(ends[1])                                                 # the first read of batch 2
        assert b.chr[r - 1] == b.chr[r]
        name = g.names[int(b.chr[r])]
        regs = [(name, int(b.pos[r - 1]) - 300, int(b.pos[r]) + 300), (g.names[1], 1, 400)]
        args = [a for x in regs for a in ("-r", f"{x[0]}:{x[1]}-{x[2]}")]
        for flags, rd in ((["-C"], P.batch_reads(b)), ([], implied)):
            _run("-d", "-P", *flags, *args, cbcs, out, fa)
            with open(out, "rb") as f:
                assert f.read() == _tsv(P.pileup(rd, up, g.names, regs), g.names, regs, up), flags
        _run("-d", "-P", "-F", "0", "-r", f"{g.names[0]}:5-9", cbcs, out, fa)
        p = _run("-d", "-P", "-r", "chrNone:1-10", cbcs, out, fa, ok=False)
        assert p.returncode != 0
