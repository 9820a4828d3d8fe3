"""BAM output on the GPU (cbcg_decode_bam, Codec.decompress_bam, `cbc -d -Z`): byte for byte against the restatement in
tests/bam_restate.py, built from the SAM lines of tests/sam_restate.py; read back by the restatement's independent reader
as cbcg_decode_sam's text (SEQ through the 4-bit code). Whole containers and regions, with and without the CIGAR side
section, blocked and legacy containers, the edge-read catalogue and the general path, errors and the command line, with
test_gpu_sam.py's shapes and settings. Every decode runs with CBCG_POISON_DECODE=1."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import bam_restate as B
import edge_reads as E
import sam_restate as R
from cbc_b200 import synth
from cbc_b200.batch import Genome
from cbc_b200.codec import CbcgError, Codec
from test_gpu_sam import EDGE, EDGE_UP, GENOME, GPU_GENOME, SETTING_IDS, SETTINGS, SHAPES, _general_batch, _implied, _shape, _split
from test_region_plan import model_plan, overlapping, parse_container

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "cbc_b200", "_build", "cbc")
AUTO = 0xFFFFFFFF
ERR_ARG, ERR_CAPACITY, ERR_NO_REFERENCE, ERR_FORMAT = -1, -5, -7, -8


@pytest.fixture(autouse=True)
def _poison(monkeypatch):
    monkeypatch.setenv("CBCG_POISON_DECODE", "1")


@pytest.fixture(scope="module")
def codec():
    c = Codec(0)
    yield c
    c.close()


def _table(cont, legacy, genome_names):
    return list(genome_names) if legacy else parse_container(cont)["names"]


def _lengths(table, g):
    by = {n: x.size for n, x in zip(g.names, g.bases)}
    return [by[n] for n in table]


def _coded(lines):
    out = []
    for x in lines:
        f = x.split(b"\t")
        f[9] = bytes(B.NT16[B._code(c)] for c in f[9])
        out.append(b"\t".join(f))
    return out


@pytest.mark.parametrize("setting", SETTINGS, ids=SETTING_IDS)
@pytest.mark.parametrize("shape", list(SHAPES))
def test_bam_matches_the_restatement(codec, shape, setting):
    g, b, L, up, want = _shape(shape)
    gen_mode, block_reads, sub = setting
    legacy = block_reads == 0
    codec.set_reference(g)
    cont = codec.compress(b, L, block_reads=block_reads, gen_mode=gen_mode, substreams=sub)
    sec = codec.cigar_pack(b)
    table = _table(cont, legacy, g.names)
    lengths = _lengths(table, g)
    data, ids = codec.decompress_bam(cont, sec, legacy=legacy)
    assert data == B.bam(want, table, lengths)
    assert np.array_equal(ids, np.arange(b.n_reads, dtype=np.uint64))
    assert codec.bam_header(cont, legacy=legacy) == B.header(table, lengths)
    # read back: decompress_sam's text, up to the SEQ code
    names, got_len, text, lines = B.read_bam(data)
    sam, _ = codec.decompress_sam(cont, sec, legacy=legacy)
    head, recs = _split(sam)
    assert names == table and got_len == lengths and text == b"".join(head)
    assert lines == _coded(recs)
    # without the section: the implied CIGARs
    cig, _, _ = _implied(b, g)
    data0, _ = codec.decompress_bam(cont, legacy=legacy, header=False, eof=False)
    assert data0 == B.record_blocks(R.sam_lines(b, up, g.names, cig), table)


@pytest.mark.parametrize("case", EDGE + ["general"], ids=[c.name for c in EDGE] + ["general_path_cigars"])
def test_edge_catalogue(codec, case):
    b, L = (_general_batch(), 100) if case == "general" else (case.batch, case.L)
    codec.set_reference(GPU_GENOME)
    cont = codec.compress(b, L, block_reads=16, gen_mode=1)
    sec = codec.cigar_pack(b)
    table = _table(cont, False, E.CHR_NAMES)
    data, _ = codec.decompress_bam(cont, sec, header=False, eof=False)
    assert data == B.record_blocks(R.sam_lines(b, EDGE_UP, E.CHR_NAMES), table)
    cig, _, _ = _implied(b, GENOME)
    data0, _ = codec.decompress_bam(cont)
    assert data0 == B.bam(R.sam_lines(b, EDGE_UP, E.CHR_NAMES, cig), table, _lengths(table, GPU_GENOME))
    sam, _ = codec.decompress_sam(cont)
    assert B.read_bam(data0)[3] == _coded(_split(sam)[1])


@pytest.mark.parametrize("with_section", [True, False], ids=["section", "implied"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_regions(codec, shape, with_section):
    g, b, L, up, want = _shape(shape)
    codec.set_reference(g)
    cont = codec.compress(b, L, block_reads=AUTO, gen_mode=1, substreams=0)
    sec = codec.cigar_pack(b) if with_section else None
    table = _table(cont, False, g.names)
    _, full = _split(codec.decompress_sam(cont, sec)[0])
    n1 = g.bases[1].size
    rng = np.random.default_rng(3)
    many = [(g.names[int(b.chr[i])], max(1, int(b.pos[i]) - 150), int(b.pos[i]) + 150) for i in rng.choice(b.n_reads, 40, replace=False)]
    for regs in ([(g.names[0], 1, 300)], [(g.names[1], int(n1 * 0.9), int(n1 * 0.9) + 400)], [(g.names[1],)], many,
                 [("chrNone", 1, 10)]):
        data, ids = codec.decompress_bam(cont, sec, regions=regs, header=False, eof=False)
        _, sids = codec.decompress_sam(cont, sec, regions=regs, header=False)
        assert np.array_equal(ids, sids), regs
        assert data == B.record_blocks([full[i] for i in ids], table), regs
        h = parse_container(cont)
        sel = set(model_plan(cont, regs)[4])
        bad = bytearray(cont)
        for k, blk in enumerate(h["blocks"]):
            if k not in sel and blk["pay"]:
                at = h["payload_off"] + blk["pay_off"]
                bad[at:at + blk["pay"]] = b"\xff" * blk["pay"]
        data2, ids2 = codec.decompress_bam(bytes(bad), sec, regions=regs, header=False, eof=False)
        assert data2 == data and np.array_equal(ids2, ids)
    stream = codec.compress(b, L, block_reads=0)
    regs = [(g.names[1], 5_000, 9_000), (g.names[0], 1, 100)]
    data, ids = codec.decompress_bam(stream, sec, regions=regs, legacy=True)
    assert np.array_equal(ids, overlapping(b, g.names, regs).astype(np.uint64))
    assert data == B.bam([full[i] for i in ids], list(g.names), [x.size for x in g.bases])


def test_errors(codec):
    g, b, L, up, want = _shape("config1")
    codec.set_reference(g)
    cont = codec.compress(b, L, block_reads=AUTO, gen_mode=1)
    sec = codec.cigar_pack(b)
    full, _ = codec.decompress_bam(cont, sec)
    src = np.frombuffer(cont, np.uint8)
    s = np.frombuffer(sec, np.uint8)
    out = np.empty(100, np.uint8); ids = np.empty(4, np.uint64)
    n, k = C.c_uint64(0), C.c_uint64(0)
    rc = codec.lib.cbcg_decode_bam(codec.h, src.ctypes.data, src.nbytes, 0, s.ctypes.data, s.nbytes, None, 0, 3, out.ctypes.data,
                                   out.nbytes, C.byref(n), ids.ctypes.data, ids.size, C.byref(k))
    assert rc == ERR_CAPACITY and n.value == len(full) and k.value == b.n_reads
    assert codec.fetch_decoded().tobytes() == full
    other = codec.cigar_pack(b.slice(0, b.n_reads - 1))
    with pytest.raises(CbcgError) as e:
        codec.decompress_bam(cont, other)
    assert e.value.status == ERR_FORMAT
    for regs in ([], [(g.names[0], 0, 10)], [(g.names[0], 20, 10)]):
        with pytest.raises(CbcgError) as e:
            codec.decompress_bam(cont, sec, regions=regs)
        assert e.value.status == ERR_ARG
    rc = codec.lib.cbcg_decode_bam(codec.h, src.ctypes.data, src.nbytes, 0, None, 0, None, 0, 4, out.ctypes.data, out.nbytes, C.byref(n),
                                   None, 0, None)
    assert rc == ERR_ARG                                  # an unknown flag
    # a table name the loaded reference lacks: the header needs its length
    renamed = Genome([g.names[0], "elsewhere"], g.bases)
    codec.set_reference(renamed)
    for call in (lambda: codec.decompress_bam(cont, sec), lambda: codec.bam_header(cont)):
        with pytest.raises(CbcgError) as e:
            call()
        assert e.value.status == ERR_NO_REFERENCE


def _run(*args, ok=True):
    p = subprocess.run([CLI, *args], capture_output=True, text=True, timeout=300)
    if ok:
        assert p.returncode == 0, p.stdout + p.stderr
    return p


def _read(path):
    with open(path, "rb") as f:
        return f.read()


def test_cli_one_batch_and_multi_batch_files():
    from cbc_b200 import shard
    cfg = synth.SynthConfig(seed=73, genome_len=1_200_000, n_chr=2, n_reads=40_000, len_min=100, len_max=100, p_sub=0.005,
                            p_indel=0.002, p_clip=0.05)
    g = synth.make_genome(cfg); b = synth.make_reads(cfg, g)
    want = R.sam_lines(b, R.upper(g), g.names)
    lengths = [x.size for x in g.bases]
    head = B.header(g.names, lengths)
    p0 = int(b.pos[b.n_reads // 3])
    regs = [(g.names[0], p0, p0 + 300), (g.names[1],)]
    sel = set(overlapping(b, g.names, regs).tolist())
    with tempfile.TemporaryDirectory() as d:
        fa, sam, one, cbcs, out = (os.path.join(d, x) for x in ("r.fa", "r.sam", "a.cbc", "a.cbcs", "o.bam"))
        synth.write_fasta(fa, g); synth.write_sam(sam, b, g)
        _run("-c", "-C", sam, one, fa)
        _run("-d", "-Z", "-C", one, out, fa)
        assert _read(out) == head + B.record_blocks(want, g.names) + B.EOF_BLOCK
        _run("-c", "-C", "-B", "1", sam, cbcs, fa)
        shards = shard.read_shards(_read(cbcs))
        assert len(shards) >= 4
        counts = [sum(blk["n"] for blk in parse_container(x)["blocks"]) for x in shards]
        starts = np.concatenate([[0], np.cumsum(counts)]).tolist()
        _run("-d", "-Z", "-C", cbcs, out, fa)
        assert _read(out) == head + b"".join(B.record_blocks(want[a:e], g.names) for a, e in zip(starts, starts[1:])) + B.EOF_BLOCK
        _run("-d", "-Z", "-C", "-r", f"{g.names[0]}:{p0}-{p0 + 300}", "-r", g.names[1], cbcs, out, fa)
        per = [B.record_blocks([want[i] for i in range(a, e) if i in sel], g.names) for a, e in zip(starts, starts[1:])]
        assert _read(out) == head + b"".join(per) + B.EOF_BLOCK
        assert B.read_bam(_read(out))[3] == _coded([want[i] for i in sorted(sel)])
