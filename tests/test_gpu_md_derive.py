"""Batches without MD (include/cbcg.h; K7, k7_md.cu): each read's MD derived on the GPU while the batch is made resident.

The property everything here checks: a batch B without MD codes to the same bytes as B*, the same batch carrying
md_nm(CIGAR, SEQ, upper(reference), POS) as its MD (tests/sam_restate.py, the rule K6 prints), in every container setting,
plain and compact, in the one-stream, overlapped and pipelined orders; the same goes for extraction, CIGAR sections and
refusals, plus one refusal of its own (a CIGAR whose query length is not the SEQ length). The generator writes canonical
MD (tests/test_sam_header.py::test_md_rule_reproduces_the_generator), so for its batches B* is B."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

import edge_reads as E
import oracle_lib as O
import sam_restate as R
from cbc_b200 import synth
from cbc_b200.batch import Batch
from cbc_b200.codec import CbcgError, Codec, CompactBatch
from test_gpu_sam import SETTINGS, SETTING_IDS, SHAPES, _general_batch, _shape

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "cbc_b200", "_build", "cbc")
AUTO = 0xFFFFFFFF
ERR_ARG, ERR_CAPACITY, ERR_INPUT, ERR_NO_REFERENCE = -1, -5, -6, -7

GPU_GENOME, GENOME = E.make_genomes()
EDGE_UP = R.upper(GPU_GENOME)
CASES = E.cases(GENOME)


@pytest.fixture(scope="module")
def codec():
    c = Codec(0)
    yield c
    c.close()


def _with_md(b: Batch, mds) -> Batch:
    off = np.zeros(b.n_reads + 1, np.uint64)
    off[1:] = np.cumsum([len(m) for m in mds])
    data = np.frombuffer(b"".join(mds), np.uint8).copy() if off[-1] else np.zeros(1, np.uint8)
    return Batch(b.pos, b.flag, b.seq_len, b.chr, b.seq_off, b.seq, b.cigar_off, b.cigar, off, data)


def _mds(b: Batch, up):
    """md_nm of every read: the MD the batch without MD gets. A read whose span runs past its chromosome keeps its own MD
    (both refuse it: K1 checks the span whatever the MD says)."""
    out, own = [], R.batch_mds(b)
    for i, (c, s) in enumerate(zip(R.batch_cigars(b), R.batch_seqs(b))):
        try:
            out.append(R.md_nm(c, s, up[int(b.chr[i])], int(b.pos[i]))[0])
        except IndexError:
            out.append(own[i])
    return out


def _star(b: Batch, up) -> Batch:
    return _with_md(b, _mds(b, up))


def _compact_bytes(codec, batch, L, block_reads, gen_mode=1, substreams=1):
    cb = CompactBatch(batch)
    out = np.empty(batch.total_bases() + 16 * batch.n_reads + (1 << 20), np.uint8)
    n = codec.compress_compact_into(cb, L, block_reads, out, gen_mode=gen_mode, substreams=substreams)
    cb.close()
    return out[:n].tobytes()


def _outcome(fn):
    try:
        return fn()
    except CbcgError as e:
        return e.status


# ------------------------------------------------------------------ 1. MD text

@pytest.mark.parametrize("shape", list(SHAPES))
def test_derived_md_equals_the_rule_on_the_generator_shapes(codec, shape):
    g, b, L, up, want = _shape(shape)
    codec.set_reference(g)
    mds = [x.split(b"\t")[12][5:].rstrip(b"\n") for x in want]      # md_nm of every read (sam_restate.sam_lines)
    assert mds == R.batch_mds(b)                                     # the generator's MD is canonical: B* is B
    assert codec.derive_md(b) == b"".join(m + b"\n" for m in mds)
    assert codec.derive_md(b.without_md()) == b"".join(m + b"\n" for m in mds)


@pytest.mark.parametrize("case", [c for c in CASES if c.extract_ok] + ["general"],
                         ids=[c.name for c in CASES if c.extract_ok] + ["general_path_cigars"])
def test_derived_md_equals_the_rule_on_the_edge_catalogue(codec, case):
    b = _general_batch() if case == "general" else case.batch
    codec.set_reference(GPU_GENOME)
    assert codec.derive_md(b) == b"".join(m + b"\n" for m in _mds(b, EDGE_UP))


# ------------------------------------------------------------------ 2. containers

@pytest.mark.parametrize("setting", SETTINGS, ids=SETTING_IDS)
@pytest.mark.parametrize("shape", list(SHAPES))
def test_container_without_md_equals_the_container_of_b_star(codec, shape, setting):
    g, b, L, up, want = _shape(shape)
    gen_mode, block_reads, sub = setting
    codec.set_reference(g)
    bare = b.without_md()
    want_c = codec.compress(b, L, block_reads=block_reads, gen_mode=gen_mode, substreams=sub)
    assert codec.compress(bare, L, block_reads=block_reads, gen_mode=gen_mode, substreams=sub) == want_c
    if block_reads == 0:
        assert want_c == O.encode_legacy(b, g, L)[0]
    else:
        assert _compact_bytes(codec, bare, L, block_reads, gen_mode, sub) == want_c
    codec.upload(bare)
    codec.encode_resident(L, block_reads, gen_mode, substreams=sub)
    assert codec.fetch_container().tobytes() == want_c


@pytest.mark.parametrize("case", [c for c in CASES if c.blocked_ok] + ["general"],
                         ids=[c.name for c in CASES if c.blocked_ok] + ["general_path_cigars"])
def test_edge_catalogue_containers_and_outputs(codec, case):
    b, L = (_general_batch(), 100) if case == "general" else (case.batch, case.L)
    codec.set_reference(GPU_GENOME)
    star, bare = _star(b, EDGE_UP), b.without_md()
    want = codec.compress(star, L, block_reads=16, gen_mode=1)
    assert codec.compress(bare, L, block_reads=16, gen_mode=1) == want
    assert _compact_bytes(codec, bare, L, 16) == want
    if case != "general" and case.legacy_ok:
        assert codec.compress(bare, L, block_reads=0) == codec.compress(star, L, block_reads=0)
    recs, edits = codec.extract(bare)
    srecs, sedits = codec.extract(star)
    assert np.array_equal(recs, srecs) and np.array_equal(edits, sedits)
    assert codec.cigar_pack(bare) == codec.cigar_pack(star)
    s1, c1 = codec.symbols(bare, L, block_reads=16, gen_mode=1)
    s2, c2 = codec.symbols(star, L, block_reads=16, gen_mode=1)
    assert np.array_equal(s1, s2) and np.array_equal(c1, c2)
    text, n = codec.decompress(want)
    assert n == b.n_reads and text == b.seq_lines()


@pytest.fixture(scope="module")
def large():
    cfg = synth.SynthConfig.named("config2", scale=0.1)                  # ~300 k reads: the pipelined and overlapped orders
    g = synth.make_genome(cfg)
    return g, synth.make_reads(cfg, g)


def test_pipelined_and_resident_orders(codec, large, monkeypatch):
    g, b = large
    codec.set_reference(g)
    bare = b.without_md()
    monkeypatch.setenv("CBCG_PIPE_MIN_READS", "200000")
    want = codec.compress(b, 150, block_reads=AUTO, gen_mode=1)        # pipelined, with MD
    assert codec.compress(bare, 150, block_reads=AUTO, gen_mode=1) == want
    assert _compact_bytes(codec, bare, 150, AUTO) == _compact_bytes(codec, b, 150, AUTO)
    codec.upload(b)
    codec.encode_resident(150, AUTO, 1)
    resident = codec.fetch_container().tobytes()
    for no_overlap in (False, True):
        if no_overlap:
            monkeypatch.setenv("CBCG_NO_OVERLAP", "1")
        codec.upload(bare)
        codec.encode_resident(150, AUTO, 1)
        assert codec.fetch_container().tobytes() == resident
    monkeypatch.delenv("CBCG_NO_OVERLAP")
    text, n = codec.decompress(want)
    assert n == b.n_reads and text == b.seq_lines()


# ------------------------------------------------------------------ 3. other outputs

def test_seq_round_trips_even_when_the_md_tags_were_wrong(codec):
    """A batch whose MD tags belong to other reads (each read carries the next read's): coded with them, the container is
    not the batch's; with the tags dropped it is, and SEQ comes back exactly."""
    g, b, L, up, want = _shape("config1")
    codec.set_reference(g)
    mds = R.batch_mds(b)
    stale = _with_md(b, mds[1:] + mds[:1])
    want_c = codec.compress(b, L, block_reads=AUTO, gen_mode=1)
    assert _outcome(lambda: codec.compress(stale, L, block_reads=AUTO, gen_mode=1)) != want_c
    cont = codec.compress(stale.without_md(), L, block_reads=AUTO, gen_mode=1)
    assert cont == want_c
    text, n = codec.decompress(cont)
    assert n == b.n_reads and text == b.seq_lines()
    assert codec.derive_md(stale) == b"".join(x + b"\n" for x in R.batch_mds(b))


# ------------------------------------------------------------------ 4. refusals

@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_refusals_follow_b_star(codec, case):
    codec.set_reference(GPU_GENOME)
    star = _star(case.batch, EDGE_UP)
    for block_reads, gen_mode in ((16, 1), (0, 0)):
        a = _outcome(lambda: codec.compress(star, case.L, block_reads=block_reads, gen_mode=gen_mode))
        bb = _outcome(lambda: codec.compress(case.batch.without_md(), case.L, block_reads=block_reads, gen_mode=gen_mode))
        assert a == bb, (block_reads, a, bb)
        assert a == ERR_INPUT or isinstance(a, bytes)
        assert isinstance(a, bytes) == (case.blocked_ok if block_reads else case.legacy_ok)
    ok = CASES[0]
    assert codec.compress(ok.batch.without_md(), ok.L, block_reads=16, gen_mode=1) == codec.compress(ok.batch, ok.L, block_reads=16, gen_mode=1)


def _one(cigar: bytes, seq: bytes, md: bytes, pos: int, chr_: int = 1) -> Batch:
    """A read in front of a filler read on e0, with the given CIGAR, SEQ and MD."""
    filler = E.read_at(GENOME, 0, 1, [("M", 20)])
    reads = [(0, 1, b"20M", filler.seq, filler.md), (chr_, pos, cigar, seq, md)]
    off = lambda xs: np.concatenate([[0], np.cumsum([len(x) for x in xs])]).astype(np.uint64)
    pool = lambda xs: np.frombuffer(b"".join(xs), np.uint8).copy()
    return Batch(np.array([r[1] for r in reads], np.uint32), np.zeros(2, np.uint16), np.array([len(r[3]) for r in reads], np.uint16),
                 np.array([r[0] for r in reads], np.uint32), off([r[3] for r in reads]), pool([r[3] for r in reads]),
                 off([r[2] for r in reads]), pool([r[2] for r in reads]), off([r[4] for r in reads]), pool([r[4] for r in reads]))


def test_refusals_of_single_reads(codec):
    codec.set_reference(GPU_GENOME)
    ref = bytes(GENOME.bases[1][5_000:5_100])
    # the CIGAR's query length is not the SEQ length: coded with MD as before, refused without
    b = _one(b"50M", ref[:51], b"50", 5_001)
    assert isinstance(codec.compress(b, 100, block_reads=16, gen_mode=1), bytes)
    for fn in (lambda: codec.compress(b.without_md(), 100, block_reads=16, gen_mode=1), lambda: codec.derive_md(b)):
        with pytest.raises(CbcgError) as e:
            fn()
        assert e.value.status == ERR_INPUT
    # refused with MD and without: '*', an N operation, more than 255 deletions, a span past the chromosome's end. Each
    # read has a mismatch in its first base: K1 codes a read whose SEQ equals the reference as a perfect match without
    # walking its CIGAR, while K7 checks every CIGAR before it derives an MD
    e0_end = len(GENOME.bases[0])
    bad = bytes([E._other(ref[0])]) + ref[1:]
    for cig, seq, md, pos, c in ((b"*", bad[:50], b"0" + ref[:1] + b"49", 5_001, 1), (b"20M10N30M", bad[:50], b"0" + ref[:1] + b"49", 5_001, 1),
                                 (b"10M256D10M", bad[:20], b"0" + ref[:1] + b"9^" + bytes(GENOME.bases[1][5_010:5_266]) + b"10", 5_001, 1),
                                 (b"20M", bytes(GENOME.bases[0][e0_end - 19:]) + b"A", b"20", e0_end - 18, 0)):
        b = _one(cig, seq, md, pos, c)
        for batch in (b, b.without_md()):
            with pytest.raises(CbcgError) as e:
                codec.compress(batch, 100, block_reads=16, gen_mode=1)
            assert e.value.status == ERR_INPUT, cig
        good = CASES[0]
        assert codec.compress(good.batch.without_md(), good.L, block_reads=16, gen_mode=1) == \
            codec.compress(good.batch, good.L, block_reads=16, gen_mode=1)


# ------------------------------------------------------------------ 5. capacity

def _snp_heavy(g, n, seed=5):
    """n reads of 150 bases, 100 SNPs each (bases 3k and 3k + 1 differ from the reference), with their canonical MD:
    about 200 bytes per read, eight times what the MD pool is first sized for."""
    rng = np.random.default_rng(seed)
    ref = R.upper(g)[0]
    pos = np.sort(rng.integers(1, ref.size - 200, n)).astype(np.uint32)
    idx = (pos.astype(np.int64) - 1)[:, None] + np.arange(150)
    r = ref[idx]
    lut = np.full(256, ord("A"), np.uint8)                   # a base that differs from the reference base (N too)
    lut[np.frombuffer(b"ACGT", np.uint8)] = np.frombuffer(b"CGTA", np.uint8)
    other = lut[r]
    snp = (np.arange(150) % 3) != 2
    seq = np.where(snp, other, r).astype(np.uint8)
    md_rows = []
    for k in range(50):                                   # "0X0X" then "1X0X" ..., a final "1"
        md_rows += [np.full((n, 1), ord("0" if k == 0 else "1"), np.uint8), r[:, 3 * k:3 * k + 1], np.full((n, 1), ord("0"), np.uint8),
                    r[:, 3 * k + 1:3 * k + 2]]
    md = np.concatenate(md_rows + [np.full((n, 1), ord("1"), np.uint8)], axis=1)
    w = md.shape[1]
    return Batch(pos, np.zeros(n, np.uint16), np.full(n, 150, np.uint16), np.zeros(n, np.uint32),
                 (np.arange(n + 1, dtype=np.uint64) * 150), seq.reshape(-1).copy(),
                 (np.arange(n + 1, dtype=np.uint64) * 4), np.frombuffer(b"150M" * n, np.uint8).copy(),
                 (np.arange(n + 1, dtype=np.uint64) * w), md.reshape(-1).copy())


def test_md_larger_than_the_first_guess(codec, large, monkeypatch):
    g, _ = large
    codec.set_reference(g)
    b = _snp_heavy(g, 2000)
    up = R.upper(g)
    assert _mds(b.slice(0, 50), up) == R.batch_mds(b.slice(0, 50))          # the builder's MD is the rule's
    want = codec.compress(b, 150, block_reads=1024, gen_mode=0)
    assert codec.compress(b.without_md(), 150, block_reads=1024, gen_mode=0) == want          # one-stream: retried
    text, _ = codec.decompress(want)
    assert text == b.seq_lines()
    # derive_md's capacity error reports the size it needs
    cb = b.c_struct()
    out = np.empty(1000, np.uint8)
    n = C.c_uint64(0)
    assert codec.lib.cbcg_derive_md(codec.h, C.byref(cb), out.ctypes.data, out.nbytes, C.byref(n)) == ERR_CAPACITY
    assert n.value == int(b.md_off[-1]) + b.n_reads
    # the pipelined order: the MD overflows the pool, the call falls back and derives the batch again. Whether a pipelined
    # call falls back depends on the buffers its context kept from earlier calls (the fallback cuts blocks without the
    # ramp), so every call here gets a fresh context: with MD the edit array overflows, without MD the MD pool does too
    monkeypatch.setenv("CBCG_PIPE_MIN_READS", "200000")
    big = _snp_heavy(g, 250_000, seed=6)

    def fresh(fn):
        c = Codec(0)
        try:
            c.set_reference(g)
            return fn(c)
        finally:
            c.close()
    want = fresh(lambda c: c.compress(big, 150, block_reads=AUTO, gen_mode=1))
    assert fresh(lambda c: c.compress(big.without_md(), 150, block_reads=AUTO, gen_mode=1)) == want
    assert fresh(lambda c: _compact_bytes(c, big.without_md(), 150, AUTO)) == fresh(lambda c: _compact_bytes(c, big, 150, AUTO))
    text, n2 = codec.decompress(want)
    assert n2 == big.n_reads and text == big.seq_lines()


# ------------------------------------------------------------------ 6. errors

def test_argument_and_state_errors(codec):
    g, b, L, up, want = _shape("config1")
    small = b.slice(0, 500)
    fresh = Codec(0)
    try:                                                  # no reference: an upload without MD cannot derive it
        for fn in (lambda: fresh.upload(small.without_md()), lambda: fresh.derive_md(small),
                   lambda: fresh.upload_compact(CompactBatch(small.without_md()))):
            with pytest.raises(CbcgError) as e:
                fn()
            assert e.value.status == ERR_NO_REFERENCE
    finally:
        fresh.close()
    codec.set_reference(g)
    for keep in ("md_off", "md"):                                             # one of the pair: a bad argument
        cb = small.c_struct()
        setattr(cb, "md" if keep == "md_off" else "md_off", None)
        assert codec.lib.cbcg_batch_upload(codec.h, C.byref(cb)) == ERR_ARG
    cc = CompactBatch(small)                                                  # a compact batch with MD, its MD pointers dropped
    v = cc.c.v
    saved = (v.md_len, v.md)
    v.md_len, v.md = None, None
    assert codec.lib.cbcg_batch_upload_compact(codec.h, C.byref(v)) == ERR_INPUT            # its MD column is not zero
    v.md_len = saved[0]
    assert codec.lib.cbcg_batch_upload_compact(codec.h, C.byref(v)) == ERR_ARG
    v.md = saved[1]
    cc.close()
    assert codec.compress(small.without_md(), L, block_reads=AUTO, gen_mode=1) == codec.compress(small, L, block_reads=AUTO, gen_mode=1)


# ------------------------------------------------------------------ 7. command line

def _run(*args, ok=True):
    p = subprocess.run([CLI, *args], capture_output=True, text=True, timeout=300)
    if ok:
        assert p.returncode == 0, p.stdout + p.stderr
    return p


def _read(path):
    with open(path, "rb") as f:
        return f.read()


def test_cli_derive_md():
    cfg = synth.SynthConfig(seed=74, genome_len=1_200_000, n_chr=2, n_reads=40_000, len_min=100, len_max=100, p_sub=0.005,
                            p_indel=0.002, p_clip=0.05)
    g = synth.make_genome(cfg); b = synth.make_reads(cfg, g)
    want = R.sam_lines(b, R.upper(g), g.names)
    with tempfile.TemporaryDirectory() as d:
        fa, sam, bare, a, m, out = (os.path.join(d, x) for x in ("r.fa", "r.sam", "bare.sam", "a.cbc", "m.cbc", "o.sam"))
        synth.write_fasta(fa, g); synth.write_sam(sam, b, g)
        # the MD tags renamed to a tag of the same length: no MD, and -B cuts the file at the same records as the original
        with open(sam, "rb") as f, open(bare, "wb") as o:
            o.write(f.read().replace(b"\tMD:Z:", b"\tXM:Z:"))
        for flags in ([], ["-1"], ["-C"], ["-C", "-1"]):
            batch = [] if "-1" in flags else ["-B", "1"]
            _run("-c", *flags, *batch, sam, a, fa)
            _run("-c", "-M", *flags, *batch, bare, m, fa)
            assert _read(a) == _read(m), flags
            if "-C" in flags:
                assert _read(a + ".cig") == _read(m + ".cig")
        stripped = os.path.join(d, "stripped.sam")                         # the tags removed outright: one batch, same container
        with open(sam, "rb") as f, open(stripped, "wb") as o:
            o.write(re.sub(rb"\tMD:Z:[^\t\n]*", b"", f.read()))
        _run("-c", "-1", sam, a, fa)
        _run("-c", "-M", "-1", stripped, m, fa)
        assert _read(a) == _read(m)
        p = _run("-c", "-B", "1", bare, m, fa, ok=False)
        assert p.returncode != 0
        _run("-c", "-M", "-C", "-B", "1", bare, m, fa)                   # with the input's CIGARs (-C): MD is md_nm of those
        _run("-d", "-S", "-C", m, out, fa)
        recs = [x + b"\n" for x in _read(out).split(b"\n")[:-1] if not x.startswith(b"@")]
        assert recs == want
