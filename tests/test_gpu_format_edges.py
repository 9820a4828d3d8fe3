"""The edge-read catalogue (tests/edge_reads.py) through the CUDA path, against the CPU oracle, bit for bit: K1 extraction,
K3 reconstruction, K2 in the single stream and in blocked containers of every layout, K0's compact upload and K5's region
decode. Where the oracle refuses a batch, the GPU must refuse it with CBCG_ERR_INPUT and then code a valid batch in the
same context. Every decode runs with CBCG_POISON_DECODE=1, so that what an encode left in the decoder's buffers cannot
make a case pass."""
import numpy as np
import pytest

import edge_reads as E
import oracle_lib as O
from cbc_b200.codec import CbcgError, CompactBatch
from test_region_plan import overlapping

pytestmark = pytest.mark.gpu
AUTO = 0xFFFFFFFF
ERR_INPUT = -6

GPU_GENOME, GENOME = E.make_genomes()
CASES = E.cases(GENOME)
IDS = [c.name for c in CASES]
SETTINGS = [(0, 0, 1), (1, 0, 1), (16, 0, 1), (16, 1, 1), (16, 1, 4), (AUTO, 1, 0)]   # (block_reads, gen_mode, substreams)
SETTING_IDS = [f"b{'auto' if s[0] == AUTO else s[0]}_g{s[1]}_s{s[2]}" for s in SETTINGS]


@pytest.fixture(autouse=True)
def _poison(monkeypatch):
    monkeypatch.setenv("CBCG_POISON_DECODE", "1")


@pytest.fixture(scope="module")
def codec():
    from cbc_b200.codec import Codec
    c = Codec(0)
    c.set_reference(GPU_GENOME)
    yield c
    c.close()


_VALID = E.make_batch(GENOME, [E.read_at(GENOME, 1, 5_001 + 40 * i, [("M", 60), ("X", 1), ("M", 39)]) for i in range(50)])


def _still_codes(codec):
    """After a refusal the context codes a valid batch."""
    cont = codec.compress(_VALID, 100, block_reads=16)
    assert cont == O.encode_blocked(_VALID, GENOME, 100, 16)
    assert codec.decompress(cont) == (_VALID.seq_lines(), _VALID.n_reads)


def _refused(fn):
    with pytest.raises(CbcgError) as ei:
        fn()
    assert ei.value.status == ERR_INPUT


def _oracle_extract(case):
    recs, edits = O.extract(case.batch, GENOME)
    if case.check:
        case.check(case.batch, recs, edits)
    return recs, edits


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_k1_extract(codec, case):
    b = case.batch
    if not case.extract_ok:
        _refused(lambda: codec.extract(b))
        _still_codes(codec)
        return
    recs, edits = codec.extract(b)
    orecs, oedits = _oracle_extract(case)
    assert np.array_equal(recs, orecs)
    assert np.array_equal(edits, oedits)


@pytest.mark.parametrize("case", [c for c in CASES if c.extract_ok], ids=[c.name for c in CASES if c.extract_ok])
def test_k3_reconstruct(codec, case):
    b = case.batch
    orecs, oedits = _oracle_extract(case)
    want = b.seq_lines()
    assert O.reconstruct(orecs, oedits, b.chr, GENOME) == want
    assert codec.reconstruct(orecs, b.chr, oedits) == want


@pytest.mark.parametrize("setting", SETTINGS, ids=SETTING_IDS)
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_k2_container(codec, case, setting):
    b = case.batch
    block_reads, gen_mode, sub = setting
    legacy = block_reads == 0
    enc = lambda: codec.compress(b, case.L, block_reads=block_reads, gen_mode=gen_mode, substreams=sub)
    if not (case.legacy_ok if legacy else case.blocked_ok):
        _refused(enc)
        _still_codes(codec)
        return
    cont = enc()
    if legacy:
        want, _ = O.encode_legacy(b, GENOME, case.L)
        assert cont == want
        assert O.decode_legacy(cont, GENOME) == (b.seq_lines(), b.n_reads)
    else:
        want = O.encode_blocked(b, GENOME, case.L, block_reads, gen_mode) if sub == 1 else O.encode_like(cont, b, GENOME)
        assert cont == want
        assert O.decode_blocked(cont, GENOME) == (b.seq_lines(), b.n_reads)
    assert codec.decompress(cont, legacy=legacy) == (b.seq_lines(), b.n_reads)
    recs, chr_, edits = codec.decode_edits(cont, legacy=legacy)
    orecs, oedits = _oracle_extract(case)
    assert np.array_equal(recs, orecs) and np.array_equal(edits, oedits) and np.array_equal(chr_, b.chr)


@pytest.mark.parametrize("case", [c for c in CASES if c.blocked_ok], ids=[c.name for c in CASES if c.blocked_ok])
def test_k0_compact_upload(codec, case):
    b = case.batch
    want = codec.compress(b, case.L, block_reads=16, gen_mode=1)
    out = np.empty(len(want) + 4096, np.uint8)
    n = codec.compress_compact_into(CompactBatch(b), case.L, 16, out, gen_mode=1)
    assert out[:n].tobytes() == want


REGION_CASES = [c for c in CASES if c.regions and c.blocked_ok]      # across the POS steps, over 1..252-base reads


@pytest.mark.parametrize("block_reads", [16, AUTO], ids=["b16", "bauto"])
@pytest.mark.parametrize("case", REGION_CASES, ids=[c.name for c in REGION_CASES])
def test_k5_region(codec, case, block_reads):
    b = case.batch
    cont = codec.compress(b, case.L, block_reads=block_reads, gen_mode=1)
    lines = b.seq_lines().split(b"\n")[:-1]
    assert len(overlapping(b, E.CHR_NAMES, case.regions)) > 0
    for regs in [[r] for r in case.regions] + [case.regions]:
        want = overlapping(b, E.CHR_NAMES, regs)
        text, ids = codec.decompress_region(cont, regs)
        assert np.array_equal(ids, want.astype(np.uint64)), regs
        assert text == b"".join(lines[i] + b"\n" for i in want), regs
