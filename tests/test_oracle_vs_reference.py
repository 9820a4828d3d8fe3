"""Pins the CPU oracle (oracle/cbc_oracle.c) to the unmodified reference.

* golden: tests/golden/*.cbc are byte streams written by the reference encoder built from
  /root/reference (tests/golden/make_golden.py); the oracle must reproduce them byte for byte,
  produce the same symbol trace (digest) and decode them to the reference decoder's output.
* known-answer: the traced example of SURVEY.md appendix A.
"""
import glob
import hashlib
import json
import os

import numpy as np
import pytest

import oracle_lib as O
from cbc_b200 import synth
from cbc_b200.batch import Batch, Genome

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.json")))


def _load(meta_path):
    with open(meta_path) as f:
        meta = json.load(f)
    cfg = synth.SynthConfig(**meta["synth"])
    g = synth.make_genome(cfg)
    b = synth.make_reads(cfg, g)
    with open(meta_path[:-5] + ".cbc", "rb") as f:
        stream = f.read()
    return meta, g, b, stream


@pytest.mark.parametrize("meta_path", GOLDEN, ids=[os.path.basename(p)[:-5] for p in GOLDEN])
def test_golden_stream_trace_and_decode(meta_path):
    meta, g, b, ref_stream = _load(meta_path)
    assert hashlib.sha256(ref_stream).hexdigest() == meta["stream_sha256"]
    stream, trace = O.encode_legacy(b, g, meta["read_len_header"], want_trace=True)
    assert stream == ref_stream                                   # byte-identical bitstream
    assert len(trace) == meta["trace_symbols"]
    assert hashlib.sha256(trace.tobytes()).hexdigest() == meta["trace_sha256"]   # identical symbol streams
    decoded, n = O.decode_legacy(ref_stream, g)
    assert n == meta["n_reads"]
    assert hashlib.sha256(decoded).hexdigest() == meta["decoded_sha256"]
    assert decoded == b.seq_lines()


def test_golden_present():
    assert len(GOLDEN) >= 10


@pytest.mark.parametrize("meta_path", GOLDEN[:4], ids=[os.path.basename(p)[:-5] for p in GOLDEN[:4]])
def test_raw_symbols_expand_to_trace(meta_path):
    """cbco_symbols (raw POS values) + the dynamic pos alphabet replay == the tracer sequence."""
    meta, g, b, _ = _load(meta_path)
    recs, edits = O.extract(b, g)
    raw = O.symbols(b, g, recs, edits, 0, b.n_reads, meta["read_len_header"], legacy=True)
    exp = O.expand_pos(raw)
    assert hashlib.sha256(exp.tobytes()).hexdigest() == meta["trace_sha256"]


@pytest.mark.parametrize("meta_path", GOLDEN, ids=[os.path.basename(p)[:-5] for p in GOLDEN])
def test_extract_reconstruct_roundtrip(meta_path):
    _, g, b, _ = _load(meta_path)
    recs, edits = O.extract(b, g)
    assert O.reconstruct(recs, edits, b.chr, g) == b.seq_lines()


@pytest.mark.parametrize("block_reads", [1, 7, 256, 100000])
def test_blocked_container_roundtrip(block_reads):
    meta, g, b, ref_stream = _load(GOLDEN[2])
    c = O.encode_blocked(b, g, meta["read_len_header"], block_reads)
    decoded, n = O.decode_blocked(c, g)
    assert n == b.n_reads and decoded == b.seq_lines()


def test_container_v4_fixed_length_flag_and_recoding_with_a_given_cut():
    """Equal-length input sets CBCG_MODE_FIXED_LEN (no length symbol), variable-length input does not; the restatement
    re-encodes a batch with the cut of an existing container (what the GPU's self-chosen cuts are checked with)."""
    import struct
    for lens, L, fixed in (((100, 100), 100, True), ((50, 250), 250, False)):
        cfg = synth.SynthConfig(seed=91, genome_len=120_000, n_chr=2, n_reads=6000, len_min=lens[0], len_max=lens[1], p_sub=0.01, p_indel=0.004, p_clip=0.1)
        g = synth.make_genome(cfg); b = synth.make_reads(cfg, g)
        for gen_mode in (0, 1):
            c = O.encode_blocked(b, g, L, 384, gen_mode)
            version, mode = struct.unpack_from("<I", c, 4)[0], struct.unpack_from("<I", c, 36)[0]
            assert version == 4 and (mode & 0xff) == gen_mode and bool(mode & 0x100) == fixed
            text, n = O.decode_blocked(c, g)
            assert n == b.n_reads and text == b.seq_lines()
            assert O.encode_like(c, b, g) == c


def _one_read_batch(pos, flag, seq, cigar, md):
    def pool(items):
        off = np.zeros(len(items) + 1, np.uint64)
        off[1:] = np.cumsum([len(x) for x in items])
        return off, np.frombuffer(b"".join(items), np.uint8).copy()
    so, s = pool(seq); co, c = pool(cigar); mo, m = pool(md)
    n = len(seq)
    return Batch(np.array(pos, np.uint32), np.array(flag, np.uint16), np.array([len(x) for x in seq], np.uint16),
                 np.zeros(n, np.uint32), so, s, co, c, mo, m)


def test_known_answer_survey_appendix_a():
    """SURVEY.md appendix A: FLAG=16 POS=4 CIGAR=17M2D32M1I41M1I1M3D7M MD:Z:17^TG74^AGC7."""
    rng = np.random.default_rng(3)
    ref = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 400)].copy()
    # force the deleted reference bases named by the MD string
    p0 = 3                                                   # 0-based start
    ref[p0 + 17:p0 + 19] = np.frombuffer(b"TG", np.uint8)
    ref[p0 + 19 + 74:p0 + 19 + 77] = np.frombuffer(b"AGC", np.uint8)
    r = ref.tobytes()
    seq = (r[p0:p0 + 17] + r[p0 + 19:p0 + 19 + 32] + b"A" + r[p0 + 51:p0 + 51 + 41] + b"C" + r[p0 + 92:p0 + 93]
           + r[p0 + 96:p0 + 103])
    assert len(seq) == 100
    second = r[10:110]
    b = _one_read_batch([4, 11], [16, 0], [seq, second], [b"17M2D32M1I41M1I1M3D7M", b"100M"], [b"17^TG74^AGC7", b"100"])
    g = Genome(["chrI"], [ref])
    _, trace = O.encode_legacy(b, g, 100, want_trace=True)
    keys = (trace["key"] >> 24).tolist()
    vals = trace["value"].tolist()
    ctxs = (trace["key"] & 0xffffff).tolist()
    # header: read_length, 32 x 0x55555555, LOSSLESS
    assert vals[:4] == [0, 0, 0, 100] and vals[4:8] == [85] * 4 and vals[132:136] == [0, 0, 0, 8]
    body = list(zip(keys[136:], ctxs[136:], vals[136:]))
    S = {n: i for i, n in enumerate(O.STREAMS)}
    expect = [(S["same_ref"], 0, 1), (S["rname"], 0, 99), (S["rname"], 99, 104), (S["rname"], 104, 114),
              (S["rname"], 114, 73), (S["rname"], 73, 0),
              (S["rlength"], 0, 100), (S["rlength"], 1, 0), (S["rlength"], 2, 0), (S["rlength"], 3, 0),
              (S["pos"], 0, 0), (S["pos_alpha"], 0, 0), (S["pos_alpha"], 1, 0), (S["pos_alpha"], 2, 0), (S["pos_alpha"], 3, 5),
              (S["flag"], 0, 16), (S["match"], 0, 0),
              (S["snps"], 0, 0), (S["indels"], 0, 0), (S["indels"], 0, 5), (S["indels"], 0, 2),
              (S["var"], 1, 17), (S["var"], 35, 0), (S["var"], 35, 74), (S["var"], 183, 0), (S["var"], 183, 0),
              (S["var"], 1, 49), (S["chars"], 5, 0), (S["var"], 99, 41), (S["chars"], 5, 1)]
    assert body[:len(expect)] == expect


def _rewrite_cigars(b: Batch, fn) -> Batch:
    """The batch with every read's CIGAR text replaced by fn(read ordinal, cigar bytes, md bytes)."""
    cig = [fn(r, b.cigar[int(b.cigar_off[r]):int(b.cigar_off[r + 1])].tobytes(), b.md[int(b.md_off[r]):int(b.md_off[r + 1])].tobytes())
           for r in range(b.n_reads)]
    off = np.zeros(b.n_reads + 1, np.uint64)
    off[1:] = np.cumsum([len(x) for x in cig])
    return Batch(b.pos, b.flag, b.seq_len, b.chr, b.seq_off, b.seq, off, np.frombuffer(b"".join(cig), np.uint8).copy(), b.md_off, b.md)


def _eqx_from_md(length: int, md: bytes) -> bytes:
    """'100M' with MD '60A39' -> '60=1X39=' (substitution-only reads)."""
    import re
    out, run = [], 0
    for tok in re.findall(rb"\d+|[A-Z]", md):
        if tok.isdigit():
            if int(tok):
                out.append(b"%d=" % int(tok))
        else:
            out.append(b"1X")
    return b"".join(out) or b"%d=" % length


def test_trailing_hard_clips_and_eq_x_cigars_are_read_as_written():
    """A CIGAR that ENDS in an operation the reference does not know ("100M7H", "60=1X39=") sends its parser past the end
    of the string (`while (*cigar != 0)` with a pointer that no longer advances: src/read_compression.c:308, :543):
    undefined behaviour, typically the `pos == chrPos` assertion of :41. Here they are read as written -- H and P
    skipped, = and X counted as M -- and give the stream of the plain spelling."""
    cfg = synth.SynthConfig(seed=131, genome_len=200_000, n_reads=3_000, len_min=100, len_max=100, p_sub=0.01)
    g = synth.make_genome(cfg)
    plain = synth.make_reads(cfg, g)

    def respell(r, cigar, md):
        return cigar + b"7H" if r % 3 == 0 else _eqx_from_md(100, md) if r % 3 == 1 else b"3H" + cigar + b"2P"
    b = _rewrite_cigars(plain, respell)
    stream, _ = O.encode_legacy(b, g, 100)
    assert stream == O.encode_legacy(plain, g, 100)[0]
    decoded, _ = O.decode_legacy(stream, g)
    assert decoded == b.seq_lines()


@pytest.mark.parametrize("seed,n_reads,p_indel,every_read", [(131, 6_000, 0.0, False), (132, 2_000, 0.01, True)])
def test_leading_hard_clips_are_skipped_in_front_of_indels_too(seed, n_reads, p_indel, every_read):
    """"5H" in front of the CIGAR of every other read, or of every read including more than 100 with an insertion.
    The reference's parser leaves the hard clip's count in front of the next operation (src/read_compression.c:543-547),
    which puts an insertion behind it at the wrong place (DESIGN.md section 2). The restatement skips H: the stream
    of the unclipped reads, decoded back to the input."""
    cfg = synth.SynthConfig(seed=seed, genome_len=200_000 if seed == 131 else 100_000, n_reads=n_reads, len_min=100,
                            len_max=100, p_sub=0.01 if seed == 131 else 0.005, p_indel=p_indel)
    g = synth.make_genome(cfg)
    plain = synth.make_reads(cfg, g)
    b = _rewrite_cigars(plain, lambda r, cigar, md: (b"5H" + cigar) if every_read or r % 2 == 0 else cigar)
    if every_read:
        assert sum(1 for r in range(b.n_reads) if b"I" in b.cigar[int(b.cigar_off[r]):int(b.cigar_off[r + 1])].tobytes()) > 100
    stream, _ = O.encode_legacy(b, g, 100)
    assert stream == O.encode_legacy(plain, g, 100)[0]
    decoded, _ = O.decode_legacy(stream, g)
    assert decoded == b.seq_lines()


@pytest.mark.parametrize("kw", [
    dict(seed=101, genome_len=300_000, n_reads=30_000, len_min=100, len_max=100, p_sub=0.005, p_indel=0.001),
    dict(seed=102, genome_len=100_000, n_reads=20_000, len_min=150, len_max=150, p_sub=0.005),
    dict(seed=103, genome_len=200_000, n_reads=10_000, len_min=200, len_max=200, p_sub=0.01, p_indel=0.02, p_clip=0.3),
    dict(seed=104, genome_len=1_500_000, n_reads=300_000, len_min=150, len_max=150, p_sub=0.005),
    dict(seed=105, genome_len=4_500_000, n_reads=300_000, len_min=100, len_max=100, p_sub=0.005, p_indel=0.001),
    dict(seed=141, genome_len=400_000, n_reads=8_000, len_min=50, len_max=250, p_sub=0.005, p_indel=0.02, p_clip=0.3),
    dict(seed=142, genome_len=300_000, n_reads=10_000, len_min=80, len_max=120, p_sub=0.01, p_indel=0.002),
], ids=lambda kw: f"seed{kw['seed']}")
def test_single_stream_round_trip(kw):
    """The restatement's single stream (header read length = the longest read, as `-l` writes it) decodes back to the
    input: fresh shapes beside the golden ones, two of 300 k reads where the FLAG, POS and SNP-count models pass the
    rescale threshold (2^20, src/stream_model.c:38-49) more than once, and variable-length reads."""
    cfg = synth.SynthConfig(**kw)
    g = synth.make_genome(cfg)
    b = synth.make_reads(cfg, g)
    stream, _ = O.encode_legacy(b, g, int(b.seq_len.max()))
    decoded, n = O.decode_legacy(stream, g)
    assert n == b.n_reads and decoded == b.seq_lines()


def test_hundreds_of_distinct_flag_values_in_the_single_stream():
    """The reference's FLAG model has all 65 536 symbols (src/sam_models.c:96-130): 700 distinct values in one stream
    round-trip through the restatement."""
    cfg = synth.SynthConfig(seed=106, genome_len=200_000, n_reads=20_000, len_min=100, len_max=100, p_sub=0.005)
    g = synth.make_genome(cfg)
    b0 = synth.make_reads(cfg, g)
    rng = np.random.default_rng(5)
    mapped = np.array([v for v in range(4096) if not v & 4], dtype=np.uint16)       # 0x4 = unmapped: not on this path
    values = rng.choice(mapped, size=700, replace=False)
    flag = np.ascontiguousarray(values[rng.integers(0, 700, size=b0.n_reads)])
    b = Batch(b0.pos, flag, b0.seq_len, b0.chr, b0.seq_off, b0.seq, b0.cigar_off, b0.cigar, b0.md_off, b0.md)
    assert len(np.unique(b.flag)) == 700
    stream, _ = O.encode_legacy(b, g, 100)
    decoded, n = O.decode_legacy(stream, g)
    assert n == b.n_reads and decoded == b.seq_lines()


def test_spliced_alignment_is_refused():
    """'N' (a skipped region): the reference ignores it and reconstructs the rest of the read against the wrong reference
    bases; here it is an input error (CBCG_ERR_INPUT on the GPU, < 0 from the restatement)."""
    cfg = synth.SynthConfig(seed=133, genome_len=50_000, n_reads=200, len_min=100, len_max=100, p_sub=0.01)
    g = synth.make_genome(cfg)
    plain = synth.make_reads(cfg, g)
    b = _rewrite_cigars(plain, lambda r, cigar, md: b"50M100N50M" if r == 17 else cigar)
    with pytest.raises(RuntimeError):
        O.encode_legacy(b, g, 100)
