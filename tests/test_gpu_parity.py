"""GPU parity tests proper: the CUDA path, called through the C ABI (cbc_b200/codec.py ->
libcbcg.so), against the CPU oracle on the same seeded inputs and against the committed golden
fixtures written by the unmodified reference (tests/golden/). Bit-exact everywhere: this path is
integer and byte work only.

Three parity definitions (BASELINE.json north_star):
  1. extracted symbol streams are bit-exact to the reference's;
  2. single-block mode emits a byte-identical bitstream;
  3. decoded reads are bit-exact to the input SEQ and to the reference decoder's output.
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

pytestmark = pytest.mark.gpu

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.json")))
IDS = [os.path.basename(p)[:-5] for p in GOLDEN]


@pytest.fixture(scope="module")
def codec():
    from cbc_b200.codec import Codec
    c = Codec(0)
    yield c
    c.close()


def _load(meta_path):
    with open(meta_path) as f:
        meta = json.load(f)
    cfg = synth.SynthConfig(**meta["synth"])
    g = synth.make_genome(cfg)
    b = synth.make_reads(cfg, g)
    with open(meta_path[:-5] + ".cbc", "rb") as f:
        stream = f.read()
    return meta, g, b, stream


def _synth(**kw):
    cfg = synth.SynthConfig(**kw)
    g = synth.make_genome(cfg)
    return g, synth.make_reads(cfg, g)


# ------------------------------------------------------------------ K1: edit extraction

@pytest.mark.parametrize("meta_path", GOLDEN, ids=IDS)
def test_extract_matches_oracle(codec, meta_path):
    _, g, b, _ = _load(meta_path)
    codec.set_reference(g)
    recs, edits = codec.extract(b)
    orecs, oedits = O.extract(b, g)
    assert np.array_equal(recs, orecs)
    assert np.array_equal(edits, oedits)


# ------------------------------------------------------------------ parity 1: symbol streams

@pytest.mark.parametrize("meta_path", GOLDEN, ids=IDS)
def test_symbol_stream_equals_reference_trace(codec, meta_path):
    """Whole-stream symbol sequence == the reference tracer's (digest pinned in the fixture)."""
    meta, g, b, _ = _load(meta_path)
    codec.set_reference(g)
    raw, counts = codec.symbols(b, meta["read_len_header"], 0)
    assert len(counts) == 1 and counts[0] == len(raw)
    exp = O.expand_pos(raw)
    assert len(exp) == meta["trace_symbols"]
    assert hashlib.sha256(exp.tobytes()).hexdigest() == meta["trace_sha256"]


@pytest.mark.parametrize("block_reads", [1, 97, 1000])
def test_block_symbol_lists_match_oracle(codec, block_reads):
    meta, g, b, _ = _load(GOLDEN[IDS.index("two_chr")])
    codec.set_reference(g)
    raw, counts = codec.symbols(b, meta["read_len_header"], block_reads)
    recs, edits = O.extract(b, g)
    # oracle block cuts: block_reads reads, never across a chromosome change
    cuts, r = [], 0
    while r < b.n_reads:
        e = r + 1
        while e < b.n_reads and e - r < block_reads and b.chr[e] == b.chr[r]:
            e += 1
        cuts.append((r, e)); r = e
    assert len(counts) == len(cuts)
    o = 0
    for (r0, r1), n in zip(cuts, counts.tolist()):
        exp = O.symbols(b, g, recs, edits, r0, r1, meta["read_len_header"], legacy=False)
        assert n == len(exp)
        assert np.array_equal(raw[o:o + n], exp), (r0, r1)
        o += n


# ------------------------------------------------------------------ parity 2: byte-identical single stream

@pytest.mark.parametrize("meta_path", GOLDEN, ids=IDS)
def test_single_block_stream_is_byte_identical_to_reference(codec, meta_path):
    meta, g, b, ref_stream = _load(meta_path)
    codec.set_reference(g)
    stream = codec.compress(b, meta["read_len_header"], block_reads=0)
    assert hashlib.sha256(stream).hexdigest() == meta["stream_sha256"]
    assert stream == ref_stream


def test_single_block_stream_past_the_rescale_thresholds(codec):
    """300 k reads in the one warp of the single-block mode: FLAG, POS and SNP-count models pass rescale = 2^20 several
    times. The CPU restatement wrote the reference encoder's bytes for this very input when it was checked against the
    reference binary (DESIGN.md section 2); the GPU must write them too, and read them back."""
    cfg = synth.SynthConfig(seed=104, genome_len=1_500_000, n_reads=300_000, len_min=150, len_max=150, p_sub=0.005)
    g = synth.make_genome(cfg)
    b = synth.make_reads(cfg, g)
    codec.set_reference(g)
    stream = codec.compress(b, 150, block_reads=0)
    want, _ = O.encode_legacy(b, g, 150)
    assert stream == want
    text, n = codec.decompress(stream, legacy=True)
    assert n == b.n_reads and text == b.seq_lines()


# ------------------------------------------------------------------ parity 3: decoded reads

@pytest.mark.parametrize("meta_path", GOLDEN, ids=IDS)
def test_decode_reference_stream(codec, meta_path):
    """The GPU decoder reads streams written by the unmodified reference encoder."""
    meta, g, b, ref_stream = _load(meta_path)
    codec.set_reference(g)
    text, n = codec.decompress(ref_stream, legacy=True)
    assert n == meta["n_reads"]
    assert hashlib.sha256(text).hexdigest() == meta["decoded_sha256"]     # == reference decoder's output
    assert text == b.seq_lines()                                         # == input SEQ


@pytest.mark.parametrize("meta_path", GOLDEN, ids=IDS)
def test_decode_edits_match_extraction(codec, meta_path):
    meta, g, b, ref_stream = _load(meta_path)
    codec.set_reference(g)
    recs, chr_, edits = codec.decode_edits(ref_stream, legacy=True)
    orecs, oedits = O.extract(b, g)
    assert np.array_equal(recs, orecs) and np.array_equal(edits, oedits) and np.array_equal(chr_, b.chr)


@pytest.mark.parametrize("meta_path", GOLDEN, ids=IDS)
def test_reconstruct_matches_oracle(codec, meta_path):
    _, g, b, _ = _load(meta_path)
    codec.set_reference(g)
    recs, edits = O.extract(b, g)
    assert codec.reconstruct(recs, b.chr, edits) == O.reconstruct(recs, edits, b.chr, g) == b.seq_lines()


# ------------------------------------------------------------------ blocked container

@pytest.mark.parametrize("substreams", [1, 4, 0])
@pytest.mark.parametrize("gen_mode", [0, 1])
@pytest.mark.parametrize("name,block_reads", [("subs_150", 256), ("indels_100", 1), ("clips_100", 97),
                                              ("two_chr", 1000), ("indels_250", 64), ("paired_flags_n", 100000),
                                              ("sparse_cov", 33)])
def test_blocked_container_equals_oracle_and_roundtrips(codec, name, block_reads, gen_mode, substreams):
    """One stream per block (every symbol of a read in the reference's order) and four substreams per block
    (CBCG_MODE_SPLIT4): the same models and symbols, both byte-identical to the CPU restatement's container."""
    meta, g, b, _ = _load(GOLDEN[IDS.index(name)])
    codec.set_reference(g)
    c = codec.compress(b, meta["read_len_header"], block_reads=block_reads, gen_mode=gen_mode, substreams=substreams)
    flags = gen_mode | (0x200 if substreams == 4 else 0x400 if substreams == 0 else 0)   # 0x400: the default cut's own layout
    assert c == O.encode_blocked(b, g, meta["read_len_header"], block_reads, flags)
    text, n = codec.decompress(c)
    assert n == b.n_reads and text == b.seq_lines()
    otext, on = O.decode_blocked(c, g)
    assert otext == text and on == n


def test_variable_length_reads_roundtrip(codec):
    """Config-5 shape: the reference decoder cannot decode these (SURVEY.md 8c-B1); the contract is
    symbol streams == the restated encoder's and own decode == input SEQ."""
    g, b = _synth(seed=80, genome_len=300_000, n_reads=20_000, len_min=50, len_max=250, p_sub=0.005,
                  p_indel=0.02, p_clip=0.3)
    codec.set_reference(g)
    recs, edits = codec.extract(b)
    orecs, oedits = O.extract(b, g)
    assert np.array_equal(recs, orecs) and np.array_equal(edits, oedits)
    for gen_mode in (0, 1):
        c = codec.compress(b, 250, block_reads=512, gen_mode=gen_mode)
        assert c == O.encode_blocked(b, g, 250, 512, gen_mode)
        text, n = codec.decompress(c)
        assert n == b.n_reads and text == b.seq_lines()


def test_large_block_uses_direct_var_rows(codec):
    """> 32768 edits in one block switches the var-row store from the hash to direct indexing."""
    g, b = _synth(seed=9, genome_len=2_000_000, n_reads=60_000, len_min=100, len_max=100, p_sub=0.01, p_indel=0.002)
    codec.set_reference(g)
    c = codec.compress(b, 100, block_reads=60_000)
    assert c == O.encode_blocked(b, g, 100, 60_000)
    text, n = codec.decompress(c)
    assert n == b.n_reads and text == b.seq_lines()
    legacy = codec.compress(b, 100, block_reads=0)
    ostream, _ = O.encode_legacy(b, g, 100)
    assert legacy == ostream


# ------------------------------------------------------------------ edges

def _batch(pos, flag, seq, cigar, md, chr_=None):
    def pool(items):
        off = np.zeros(len(items) + 1, np.uint64)
        off[1:] = np.cumsum([len(x) for x in items])
        data = np.frombuffer(b"".join(items), np.uint8).copy() if items and sum(map(len, items)) else np.zeros(1, np.uint8)
        return off, data
    so, s = pool(seq); co, c = pool(cigar); mo, m = pool(md)
    n = len(seq)
    return Batch(np.array(pos, np.uint32), np.array(flag, np.uint16), np.array([len(x) for x in seq], np.uint16),
                 np.zeros(n, np.uint32) if chr_ is None else np.array(chr_, np.uint32), so, s, co, c, mo, m)


def test_empty_batch(codec):
    g, _ = _synth(seed=1, genome_len=10_000, n_reads=10)
    codec.set_reference(g)
    b = _batch([], [], [], [], [])
    c = codec.compress(b, 100, block_reads=128)
    text, n = codec.decompress(c)
    assert n == 0 and text == b""


def test_known_answer_survey_appendix_a(codec):
    """SURVEY.md appendix A, through the GPU symbol path."""
    rng = np.random.default_rng(3)
    ref = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 400)].copy()
    p0 = 3
    ref[p0 + 17:p0 + 19] = np.frombuffer(b"TG", np.uint8)
    ref[p0 + 19 + 74:p0 + 19 + 77] = np.frombuffer(b"AGC", np.uint8)
    r = ref.tobytes()
    seq = (r[p0:p0 + 17] + r[p0 + 19:p0 + 19 + 32] + b"A" + r[p0 + 51:p0 + 51 + 41] + b"C" + r[p0 + 92:p0 + 93]
           + r[p0 + 96:p0 + 103])
    b = _batch([4, 11], [16, 0], [seq, r[10:110]], [b"17M2D32M1I41M1I1M3D7M", b"100M"], [b"17^TG74^AGC7", b"100"])
    g = Genome(["chrI"], [ref])
    codec.set_reference(g)
    raw, _ = codec.symbols(b, 100, 0)
    exp = O.expand_pos(raw)
    _, trace = O.encode_legacy(b, g, 100, want_trace=True)
    assert np.array_equal(exp, trace)
    body = [(int(k) >> 24, int(k) & 0xffffff, int(v)) for k, v in zip(exp["key"][136:], exp["value"][136:])]
    S = {n: i for i, n in enumerate(O.STREAMS)}
    assert body[16:30] == [(S["match"], 0, 0), (S["snps"], 0, 0), (S["indels"], 0, 0), (S["indels"], 0, 5),
                           (S["indels"], 0, 2), (S["var"], 1, 17), (S["var"], 35, 0), (S["var"], 35, 74),
                           (S["var"], 183, 0), (S["var"], 183, 0), (S["var"], 1, 49), (S["chars"], 5, 0),
                           (S["var"], 99, 41), (S["chars"], 5, 1)]
    stream = codec.compress(b, 100, 0)
    ostream, _ = O.encode_legacy(b, g, 100)
    assert stream == ostream
    text, n = codec.decompress(stream, legacy=True)
    assert n == 2 and text == b.seq_lines()


def test_bad_inputs_are_reported_not_asserted(codec):
    from cbc_b200.codec import CbcgError
    g, b = _synth(seed=1, genome_len=10_000, n_reads=50)
    codec.set_reference(g)
    seq = g.bases[0][:100].tobytes()
    for bad in (_batch([0], [0], [seq], [b"100M"], [b"100"]),                   # POS 0
                _batch([1], [0], [seq[:60] + b"ACGT" * 10], [b"*"], [b"100"]),   # CIGAR '*' on a non-matching read
                _batch([5], [0], [seq], [b"100M"], [b"100"], chr_=[7])):         # chromosome out of range
        with pytest.raises(CbcgError) as e:
            codec.compress(bad, 100, block_reads=16)
        assert e.value.status in (-6, -7)
    with pytest.raises(CbcgError):
        codec.decompress(b"not a container at all, just some bytes to be rejected........")
    # unsorted positions inside a block
    ub = _batch([500, 100], [0, 0], [g.bases[0][499:599].tobytes(), g.bases[0][99:199].tobytes()], [b"100M"] * 2, [b"100"] * 2)
    with pytest.raises(CbcgError):
        codec.compress(ub, 100, block_reads=16)


def test_corrupt_payload_does_not_hang(codec):
    meta, g, b, _ = _load(GOLDEN[IDS.index("indels_100")])
    codec.set_reference(g)
    c = bytearray(codec.compress(b, 100, block_reads=200))
    rng = np.random.default_rng(5)
    for i in rng.integers(len(c) // 2, len(c), 64):
        c[i] ^= 0xff
    from cbc_b200.codec import CbcgError
    try:
        text, n = codec.decompress(bytes(c))
        assert n == b.n_reads            # structure survives; content differs
    except CbcgError as e:
        assert e.status in (-9, -5, -6, -11)


# ------------------------------------------------------------------ size-independent properties at larger size

def test_config2_slice_roundtrip_and_resident_path(codec):
    """~200 k reads of the config-2 shape: encode -> decode round trip on the device-resident path, container
    equality with the host-buffer path, and bits/base sanity."""
    cfg = synth.SynthConfig.named("config2", scale=1 / 15)
    g = synth.make_genome(cfg)
    b = synth.make_reads(cfg, g)
    codec.set_reference(g)
    sizes = {}
    for gen_mode in (0, 1):
        codec.upload(b)
        codec.encode_resident(150, 1024, gen_mode)
        st = codec.stats()
        assert st["n_reads"] == b.n_reads
        if gen_mode == 0:
            assert st["n_blocks"] == (b.n_reads + 1023) // 1024
        cont = codec.fetch_container().tobytes()
        codec.decode_resident()
        text = codec.fetch_decoded().tobytes()
        assert text == b.seq_lines()
        assert cont == codec.compress(b, 150, block_reads=1024, gen_mode=gen_mode)
        assert cont == O.encode_blocked(b, g, 150, 1024, gen_mode)
        text2, n2 = codec.decompress(cont)
        assert n2 == b.n_reads and text2 == text
        bits_per_base = 8.0 * len(cont) / b.total_bases()
        assert 0.02 < bits_per_base < 0.5
        sizes[gen_mode] = len(cont)
        # idempotence: a second encode of the resident batch gives the same bytes
        codec.upload(b)
        codec.encode_resident(150, 1024, gen_mode)
        assert codec.fetch_container().tobytes() == cont
    assert sizes[1] < 0.8 * sizes[0]              # primed blocks recover most of the cold-start loss


def test_cigar_operations_beyond_midS_on_the_gpu(codec):
    """K1 reads a CIGAR as written -- H and P skipped, = and X counted as M -- like the restatement (which was checked against the
    reference binary where the reference's own parser survives them: DESIGN.md section 2); a skipped region (N) is an
    input error."""
    from test_oracle_vs_reference import _rewrite_cigars, _eqx_from_md
    from cbc_b200.codec import CbcgError
    g, plain = _synth(seed=131, genome_len=200_000, n_reads=6_000, len_min=100, len_max=100, p_sub=0.01, p_indel=0.004)

    def respell(r, cigar, md):
        if b"I" in cigar or b"D" in cigar:
            return b"4H" + cigar + b"6H"
        return cigar + b"7H" if r % 3 == 0 else _eqx_from_md(100, md) if r % 3 == 1 else b"3H" + cigar + b"2P"
    b = _rewrite_cigars(plain, respell)
    codec.set_reference(g)
    recs, edits = codec.extract(b)
    orecs, oedits = O.extract(plain, g)
    assert np.array_equal(recs, orecs) and np.array_equal(edits, oedits)
    stream = codec.compress(b, 100, block_reads=0)
    assert stream == O.encode_legacy(plain, g, 100)[0]
    text, n = codec.decompress(stream, legacy=True)
    assert n == b.n_reads and text == b.seq_lines()
    victim = int(np.flatnonzero(orecs["match"] == 0)[5])         # a perfectly matching read never has its CIGAR looked at (:291-296)
    bad = _rewrite_cigars(plain, lambda r, cigar, md: b"50M100N50M" if r == victim else cigar)
    with pytest.raises(CbcgError) as e:
        codec.extract(bad)
    assert e.value.status == -6


def _with_flags(b, n_distinct, seed, random_head=False):
    """The batch with its FLAG column replaced by n_distinct values (strand bit included), position order untouched.
    random_head: values drawn at random from the first read on; otherwise the first n_distinct reads carry one each."""
    rng = np.random.default_rng(seed)
    values = rng.choice(4096, size=n_distinct, replace=False).astype(np.uint16)
    flag = values[rng.integers(0, n_distinct, size=b.n_reads)]
    if not random_head:
        flag[:n_distinct] = values                               # every value occurs
    return Batch(b.pos, np.ascontiguousarray(flag), b.seq_len, b.chr, b.seq_off, b.seq, b.cigar_off, b.cigar, b.md_off, b.md)


@pytest.mark.gpu
def test_two_hundred_distinct_flags(codec):
    """The sparse FLAG table holds 256 touched values per block and per snapshot (the reference's model has all 65 536:
    src/sam_models.c:96-130). 200 distinct values in one block and in the merged snapshots: single-block stream, cold and
    generation-primed containers equal the restatement's, and decode back; the warp-per-chain encoder's table leaves its
    registers for shared memory at the 33rd value."""
    g, b0 = _synth(seed=31, genome_len=200_000, n_reads=30_000, len_min=100, len_max=100, p_sub=0.01, p_indel=0.0)
    b = _with_flags(b0, 200, 7)
    codec.set_reference(g)
    stream = codec.compress(b, 100, block_reads=0)
    ostream, _ = O.encode_legacy(b, g, 100)
    assert stream == ostream
    for gen_mode, block_reads in ((0, 30_000), (1, 4_000), (1, 512)):
        c = codec.compress(b, 100, block_reads=block_reads, gen_mode=gen_mode, substreams=1)
        assert c == O.encode_blocked(b, g, 100, block_reads, gen_mode)
        text, n = codec.decompress(c)
        assert n == b.n_reads and text == b.seq_lines()


@pytest.mark.gpu
@pytest.mark.parametrize("n_distinct,random_head", [(300, False), (1500, True), (400, True)])
def test_more_distinct_flags_than_a_block_adapts(codec, n_distinct, random_head):
    """Blocked containers bound the FLAG model by design (cbcg_format.h, rules F1 / F2): a block adapts 256 distinct values
    and codes further new ones at their initial count of 1, a merged snapshot keeps the 256 largest counts. 300 ... 1 500
    distinct values -- more than a block and more than any snapshot holds; with random_head the blocks of one generation
    adapt different values, so that their merge has to drop some (F2) -- in cold, generation-primed, one-stream,
    four-substream and default-layout containers: the restatement's bytes, and the input back. The single-block mode is
    the reference's own stream, whose model adapts every value (the restatement was checked against the
    reference binary on 700 values: DESIGN.md section 2): byte-identical there too."""
    g, b0 = _synth(seed=32, genome_len=150_000, n_reads=24_000, len_min=100, len_max=100, p_sub=0.01, p_indel=0.0)
    b = _with_flags(b0, n_distinct, 8, random_head)
    codec.set_reference(g)
    for gen_mode, block_reads, sub in ((0, 24_000, 1), (0, 3_000, 1), (1, 2_000, 1), (1, 512, 1), (1, 2_000, 4), (1, 0xffffffff, 0)):
        c = codec.compress(b, 100, block_reads=block_reads, gen_mode=gen_mode, substreams=sub)
        if sub == 1:
            assert c == O.encode_blocked(b, g, 100, block_reads, gen_mode), (gen_mode, block_reads)
        else:
            assert c == O.encode_like(c, b, g), (gen_mode, block_reads, sub)
        text, n = codec.decompress(c)
        assert n == b.n_reads and text == b.seq_lines(), (gen_mode, block_reads, sub)
        otext, on = O.decode_blocked(c, g)
        assert on == b.n_reads and otext == b.seq_lines()
    # the single-block mode is the reference's own stream: every value adapts (the table continues in the workspace)
    stream = codec.compress(b, 100, block_reads=0)
    ostream, _ = O.encode_legacy(b, g, 100)
    assert stream == ostream
    text, n = codec.decompress(stream, legacy=True)
    assert n == b.n_reads and text == b.seq_lines()


@pytest.mark.gpu
@pytest.mark.parametrize("block_reads", [1500, 6000])
def test_var_contexts_shared_by_many_symbols_of_a_block(codec, block_reads):
    """Sparse coverage: no earlier SNP site lies under any read, so the first SNP of every read has the same var context
    (sentinel delta, strand). The model kernel's context-grouped walk over the edit positions (last generation) meets
    contexts with hundreds of symbols per block (block_reads 1500: inside its limit) and with thousands (6000: the block
    falls back to the serial walk after the grouping pass); both must write the restatement's container."""
    g, b = _synth(seed=41, genome_len=2_000_000, n_reads=6_000, len_min=100, len_max=100, p_sub=0.02, p_indel=0.0)
    codec.set_reference(g)
    for gen_mode in (0, 1):
        c = codec.compress(b, 100, block_reads=block_reads, gen_mode=gen_mode, substreams=1)
        assert c == O.encode_blocked(b, g, 100, block_reads, gen_mode)
        text, n = codec.decompress(c)
        assert n == b.n_reads and text == b.seq_lines()
