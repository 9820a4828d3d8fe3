"""SAM output on the GPU (cbcg_decode_sam, Codec.decompress_sam, `cbc -d -S`): every line against the restatement in
tests/sam_restate.py, computed from the input batch (FLAG, chromosome, POS, CIGAR, SEQ) and the upper-cased genome; MD
against the input's MD where the generator wrote it canonically. Whole containers and regions, with and without the
CIGAR side section, the edge-read catalogue, errors and the command line, including a SAM -> container -> SAM -> container
round trip. Every decode runs with CBCG_POISON_DECODE=1."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import edge_reads as E
import oracle_lib as O
import sam_restate as R
from cbc_b200 import synth
from cbc_b200.codec import CbcgError, Codec, sam_header
from test_region_plan import model_plan, overlapping, parse_container

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "cbc_b200", "_build", "cbc")
AUTO = 0xFFFFFFFF
ERR_ARG, ERR_CAPACITY, ERR_FORMAT = -1, -5, -8

SHAPES = {   # two chromosomes, sparse coverage, as the region tests
    "config1": (dict(seed=71, genome_len=2_000_000, n_chr=2, n_reads=30_000, len_min=100, len_max=100, p_sub=0.005,
                     p_indel=0.002, p_clip=0.05), 100),
    "config5": (dict(seed=72, genome_len=2_000_000, n_chr=2, n_reads=20_000, len_min=50, len_max=250, p_sub=0.005,
                     p_indel=0.02, p_clip=0.3), 250),
}
SETTINGS = [  # (gen_mode, block_reads, substreams); block_reads 0: the single-block (legacy) stream
    (1, AUTO, 0), (1, AUTO, 1), (1, AUTO, 4), (0, 1024, 1), (1, 400, 1), (0, 0, 1),
]
SETTING_IDS = [f"g{s[0]}_b{'auto' if s[1] == AUTO else s[1]}_s{s[2]}" for s in SETTINGS]


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
    if name not in _CACHE:
        kw, L = SHAPES[name]
        cfg = synth.SynthConfig(**kw)
        g = synth.make_genome(cfg)
        b = synth.make_reads(cfg, g)
        up = R.upper(g)
        _CACHE[name] = (g, b, L, up, R.sam_lines(b, up, g.names))
    return _CACHE[name]


def _split(text):
    """(header lines, record lines)"""
    lines = text.split(b"\n")[:-1]
    k = 0
    while k < len(lines) and lines[k].startswith(b"@"):
        k += 1
    return [x + b"\n" for x in lines[:k]], [x + b"\n" for x in lines[k:]]


def _implied(b, genome_upper_g):
    recs, edits = O.extract(b, genome_upper_g)
    return [R.implied_cigar(recs[i], edits) for i in range(b.n_reads)], recs, edits


@pytest.mark.parametrize("setting", SETTINGS, ids=SETTING_IDS)
@pytest.mark.parametrize("shape", list(SHAPES))
def test_sam_matches_the_input(codec, shape, setting):
    g, b, L, up, want = _shape(shape)
    gen_mode, block_reads, sub = setting
    legacy = block_reads == 0
    codec.set_reference(g)
    cont = codec.compress(b, L, block_reads=block_reads, gen_mode=gen_mode, substreams=sub)
    sec = codec.cigar_pack(b)
    text, ids = codec.decompress_sam(cont, sec, legacy=legacy)
    head, recs = _split(text)
    lengths = [x.size for x in g.bases]
    assert b"".join(head) == R.header(g.names, lengths)
    if not legacy:
        assert sam_header(cont) == R.header(g.names)
    assert recs == want
    assert np.array_equal(ids, np.arange(b.n_reads, dtype=np.uint64))
    R.check_fields(text)
    # field by field: the input's FLAG, RNAME, POS, CIGAR, SEQ and (canonical generator) MD
    f = [x.split(b"\t") for x in recs]
    assert [int(x[1]) for x in f] == b.flag.tolist() and [int(x[3]) for x in f] == b.pos.tolist()
    assert [x[2] for x in f] == [g.names[c].encode() for c in b.chr]
    assert [x[5] for x in f] == R.batch_cigars(b) and [x[9] for x in f] == R.batch_seqs(b)
    assert [x[12][5:].rstrip(b"\n") for x in f] == R.batch_mds(b)
    # without the section: the implied CIGARs
    cig, orecs, oedits = _implied(b, g)
    text0, _ = codec.decompress_sam(cont, legacy=legacy, header=False)
    assert text0 == b"".join(R.sam_lines(b, up, g.names, cig))
    if shape == "config5":          # reads on the general path: verbatim CIGARs, among them match records with a clip
        cls = [R.cigar_class(orecs[i], oedits, c) for i, c in enumerate(R.batch_cigars(b))]
        assert cls.count(4) > 0
        assert any(orecs[i]["match"] and cls[i] == 4 for i in range(b.n_reads))


GPU_GENOME, GENOME = E.make_genomes()
EDGE = [c for c in E.cases(GENOME) if c.blocked_ok]
EDGE_UP = R.upper(GPU_GENOME)


def _general_batch():
    """CIGARs spelled with =, X, a leading H and P, and one-base trailing clips over matching reference bases: section class 4."""
    g = GENOME
    reads, cigars = [], []
    for i in range(40):
        p = 5_001 + 300 * i
        reads.append(E.read_at(g, 1, p, [("M", 10), ("X", 1), ("M", 20), ("D", 2), ("M", 19)])); cigars.append(b"10=1X20=2D19=")
        reads.append(E.read_at(g, 1, p + 100, [("M", 30), ("X", 1), ("M", 19)])); cigars.append(b"5H30M1X19M")
        reads.append(E.read_at(g, 1, p + 200, [("M", 12), ("I", 2), ("M", 36)])); cigars.append(b"12M2P2I36M")
        reads.append(E.read_at(g, 1, p + 250, [("M", 50)])); cigars.append(b"49M1S")
    b = E.make_batch(g, reads)
    order = {(r.chr, r.pos): c for r, c in zip(reads, cigars)}
    own = R.batch_cigars(b)                              # make_batch's filler read on e0 keeps its CIGAR
    texts = [order.get((int(b.chr[i]), int(b.pos[i])), own[i]) for i in range(b.n_reads)]
    off = np.zeros(b.n_reads + 1, np.uint64); off[1:] = np.cumsum([len(t) for t in texts])
    from cbc_b200.batch import Batch
    return Batch(b.pos, b.flag, b.seq_len, b.chr, b.seq_off, b.seq, off, np.frombuffer(b"".join(texts), np.uint8).copy(), b.md_off, b.md)


@pytest.mark.parametrize("case", EDGE + ["general"], ids=[c.name for c in EDGE] + ["general_path_cigars"])
def test_edge_catalogue(codec, case):
    b, L = (_general_batch(), 100) if case == "general" else (case.batch, case.L)
    codec.set_reference(GPU_GENOME)
    cont = codec.compress(b, L, block_reads=16, gen_mode=1)
    sec = codec.cigar_pack(b)
    text, _ = codec.decompress_sam(cont, sec, header=False)
    assert text == b"".join(R.sam_lines(b, EDGE_UP, E.CHR_NAMES))
    R.check_fields(text)
    cig, orecs, oedits = _implied(b, GENOME)
    text0, _ = codec.decompress_sam(cont, header=False)
    assert text0 == b"".join(R.sam_lines(b, EDGE_UP, E.CHR_NAMES, cig))
    if case == "general":
        assert all(R.cigar_class(orecs[i], oedits, c) == 4 for i, c in enumerate(R.batch_cigars(b)) if b.chr[i] == 1)


@pytest.mark.parametrize("with_section", [True, False], ids=["section", "implied"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_regions(codec, shape, with_section):
    g, b, L, up, want = _shape(shape)
    codec.set_reference(g)
    cont = codec.compress(b, L, block_reads=AUTO, gen_mode=1, substreams=0)
    sec = codec.cigar_pack(b) if with_section else None
    _, full = _split(codec.decompress_sam(cont, sec)[0])
    n1 = g.bases[1].size
    rng = np.random.default_rng(3)
    many = [(g.names[int(b.chr[i])], max(1, int(b.pos[i]) - 150), int(b.pos[i]) + 150) for i in rng.choice(b.n_reads, 40, replace=False)]
    for regs in ([(g.names[0], 1, 300)], [(g.names[1], int(n1 * 0.9), int(n1 * 0.9) + 400)], [(g.names[1],)], many,
                 [("chrNone", 1, 10)]):
        text, ids = codec.decompress_sam(cont, sec, regions=regs, header=False)
        _, rids = codec.decompress_region(cont, regs)
        assert np.array_equal(ids, rids), regs
        assert np.array_equal(ids, overlapping(b, g.names, regs).astype(np.uint64)), regs
        assert text == b"".join(full[i] for i in ids), regs
        # untouched payload overwritten with 0xff gives the same answer
        h = parse_container(cont)
        sel = set(model_plan(cont, regs)[4])
        bad = bytearray(cont)
        for k, blk in enumerate(h["blocks"]):
            if k not in sel and blk["pay"]:
                at = h["payload_off"] + blk["pay_off"]
                bad[at:at + blk["pay"]] = b"\xff" * blk["pay"]
        text2, ids2 = codec.decompress_sam(bytes(bad), sec, regions=regs, header=False)
        assert text2 == text and np.array_equal(ids2, ids)
    # the single-block stream: decoded whole, then filtered
    stream = codec.compress(b, L, block_reads=0)
    regs = [(g.names[1], 5_000, 9_000), (g.names[0], 1, 100)]
    text, ids = codec.decompress_sam(stream, sec, regions=regs, header=False, legacy=True)
    assert np.array_equal(ids, overlapping(b, g.names, regs).astype(np.uint64))
    assert text == b"".join(full[i] for i in ids)


def test_errors(codec):
    g, b, L, up, want = _shape("config1")
    codec.set_reference(g)
    cont = codec.compress(b, L, block_reads=AUTO, gen_mode=1)
    sec = codec.cigar_pack(b)
    full, _ = codec.decompress_sam(cont, sec)
    src = np.frombuffer(cont, np.uint8)
    s = np.frombuffer(sec, np.uint8)
    out = np.empty(100, np.uint8); ids = np.empty(4, np.uint64)
    n, k = C.c_uint64(0), C.c_uint64(0)
    rc = codec.lib.cbcg_decode_sam(codec.h, src.ctypes.data, src.nbytes, 0, s.ctypes.data, s.nbytes, None, 0, 1, out.ctypes.data,
                                   out.nbytes, C.byref(n), ids.ctypes.data, ids.size, C.byref(k))
    assert rc == ERR_CAPACITY and n.value == len(full) and k.value == b.n_reads
    assert codec.fetch_decoded().tobytes() == full
    # a section of another batch: its read count does not match
    other = codec.cigar_pack(b.slice(0, b.n_reads - 1))
    with pytest.raises(CbcgError) as e:
        codec.decompress_sam(cont, other)
    assert e.value.status == ERR_FORMAT
    # regions: none, start 0, start > end
    for regs in ([], [(g.names[0], 0, 10)], [(g.names[0], 20, 10)]):
        with pytest.raises(CbcgError) as e:
            codec.decompress_sam(cont, sec, regions=regs)
        assert e.value.status == ERR_ARG
    with pytest.raises(CbcgError) as e:
        sam_header(cont[:30])
    assert e.value.status == ERR_FORMAT


def _run(*args, ok=True):
    p = subprocess.run([CLI, *args], capture_output=True, text=True, timeout=300)
    if ok:
        assert p.returncode == 0, p.stdout + p.stderr
    return p


def _read(path):
    with open(path, "rb") as f:
        return f.read()


def test_cli_multi_batch_file():
    from cbc_b200 import shard
    cfg = synth.SynthConfig(seed=73, genome_len=1_200_000, n_chr=2, n_reads=40_000, len_min=100, len_max=100, p_sub=0.005,
                            p_indel=0.002, p_clip=0.05)
    g = synth.make_genome(cfg); b = synth.make_reads(cfg, g)
    want = R.sam_lines(b, R.upper(g), g.names)
    head = R.header(g.names, [x.size for x in g.bases])
    with tempfile.TemporaryDirectory() as d:
        fa, sam, cbcs, out = (os.path.join(d, x) for x in ("r.fa", "r.sam", "a.cbcs", "o.sam"))
        synth.write_fasta(fa, g); synth.write_sam(sam, b, g)
        _run("-c", "-C", "-B", "1", sam, cbcs, fa)
        assert len(shard.read_shards(_read(cbcs))) >= 4
        _run("-d", "-S", "-C", cbcs, out, fa)
        assert _read(out) == head + b"".join(want)
        p0 = int(b.pos[b.n_reads // 3])
        for flags in (["-S"], ["-S", "-C"]):
            _run("-d", *flags, "-r", f"{g.names[0]}:{p0}-{p0 + 300}", "-r", g.names[1], cbcs, out, fa)
            sel = overlapping(b, g.names, [(g.names[0], p0, p0 + 300), (g.names[1],)])
            text = _read(out)
            assert text.startswith(head)
            recs = text[len(head):].splitlines(keepends=True)
            if "-C" in flags:
                assert recs == [want[i] for i in sel]
            else:
                assert [x.split(b"\t")[9] for x in recs] == [want[i].split(b"\t")[9] for i in sel]
        p = _run("-d", "-C", "-r", g.names[0], cbcs, out, fa, ok=False)          # -C -r without -S is still refused
        assert p.returncode != 0 and "-C" in p.stderr


@pytest.mark.parametrize("shape", list(SHAPES))
def test_cli_round_trip(shape):
    """SAM -> container -> SAM -> container: the same container byte for byte, and the same side section."""
    g, b, L, up, want = _shape(shape)
    flags = ["-l"] if shape == "config5" else []
    with tempfile.TemporaryDirectory() as d:
        fa, sam, c1, s1, c2 = (os.path.join(d, x) for x in ("r.fa", "r.sam", "a.cbc", "a.sam", "b.cbc"))
        synth.write_fasta(fa, g); synth.write_sam(sam, b, g)
        _run("-c", "-C", *flags, sam, c1, fa)
        _run("-d", "-S", "-C", c1, s1, fa)
        assert _read(s1).split(b"\n", len(g.names) + 1)[-1] == b"".join(want)
        _run("-c", "-C", *flags, s1, c2, fa)
        assert _read(c1) == _read(c2)
        assert _read(c1 + ".cig") == _read(c2 + ".cig")
