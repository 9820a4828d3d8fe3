"""Region decode on the GPU (cbcg_decode_region, Codec.decompress_region, `cbc -d -r`): the reads that overlap the regions,
each once, in container order, against the answer taken from the input batch (chromosome, POS and the reference span of
its CIGAR, M + D + = + X). Every decode here runs with CBCG_POISON_DECODE=1, so that records and edits an encode left in
the decoder's buffers cannot make a case pass."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from cbc_b200 import synth
from cbc_b200.batch import Batch
from cbc_b200.codec import Codec, CompactBatch, region_plan
from test_region_plan import model_plan, overlapping, parse_container, ref_spans

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "cbc_b200", "_build", "cbc")
AUTO = 0xFFFFFFFF

SHAPES = {   # two chromosomes, sparse coverage (about 1.5x and 1.9x)
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
    if name not in _CACHE:
        kw, L = SHAPES[name]
        cfg = synth.SynthConfig(**kw)
        g = synth.make_genome(cfg)
        _CACHE[name] = (g, synth.make_reads(cfg, g), L)
    return _CACHE[name]


def _lines(b):
    seq = b.seq.tobytes()
    return [seq[b.seq_off[i]:b.seq_off[i + 1]] + b"\n" for i in range(b.n_reads)]


_SPANS = {}


def _want(b, names, regions):
    if id(b) not in _SPANS:
        _SPANS[id(b)] = (b, ref_spans(b))
    return overlapping(b, names, regions, _SPANS[id(b)][1])


def _check(codec, cont, b, lines, names, regions, legacy=False):
    text, ids = codec.decompress_region(cont, regions, legacy=legacy)
    want = _want(b, names, regions)
    assert np.array_equal(ids, want.astype(np.uint64)), regions
    assert text == b"".join(lines[i] for i in want), regions
    return ids


def _many_regions(g, b, seed):
    """unsorted, overlapping regions on both chromosomes around reads far apart"""
    rng = np.random.default_rng(seed)
    regs = []
    for i in rng.choice(b.n_reads, size=48, replace=False):
        p = int(b.pos[i])
        regs.append((g.names[int(b.chr[i])], max(1, p - 150), p + 150))
    regs += [(r[0], r[1] + 100, r[2] + 400) for r in regs[:8]]          # overlapping the first few
    regs += [regs[3], ("not_in_this_container", 1, 10_000)]
    rng.shuffle(regs)
    return regs


@pytest.mark.parametrize("setting", SETTINGS, ids=[f"g{s[0]}_b{'auto' if s[1] == AUTO else s[1]}_s{s[2]}" for s in SETTINGS])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_region_decode_matches_the_input(codec, shape, setting):
    g, b, L = _shape(shape)
    gen_mode, block_reads, sub = setting
    codec.set_reference(g)
    cont = codec.compress(b, L, block_reads=block_reads, gen_mode=gen_mode, substreams=sub)
    lines = _lines(b)
    full, n = codec.decompress(cont)
    assert n == b.n_reads and full == b"".join(lines)
    blocks = parse_container(cont)["blocks"]
    names = g.names
    # the very start of the genome: early generations only, a reduced table without the container's longest block
    _check(codec, cont, b, lines, names, [(names[0], 1, 300)])
    # the last generation: fewer blocks than the container has, as many as the plan says
    n1 = g.bases[1].size
    regs = [(names[1], int(n1 * 0.9), int(n1 * 0.9) + 400)]
    ids = _check(codec, cont, b, lines, names, regs)
    assert len(ids) > 0
    st = codec.stats()
    plan = region_plan(cont, regs)
    assert st["n_blocks"] == plan["n_blocks"] == model_plan(cont, regs)[0] < len(blocks)
    assert st["n_reads"] == plan["n_reads"] >= len(ids)
    # a whole chromosome: the matching slice of the full decode
    text, ids = codec.decompress_region(cont, [(names[1],)])
    assert np.array_equal(ids, np.nonzero(b.chr == 1)[0].astype(np.uint64))
    assert text == b"".join(lines[i] for i in ids)
    # many regions at once: one K3 tile crosses regions and chromosomes, every read comes once
    ids = _check(codec, cont, b, lines, names, _many_regions(g, b, 5 + gen_mode))
    assert len(ids) >= 128 and len(set(ids.tolist())) == len(ids)
    assert len(set(b.chr[ids].tolist())) == 2
    # nothing: past the end of a record, and a name the container does not hold
    for regs in ([(names[0], g.bases[0].size + 10_000, g.bases[0].size + 20_000)], [("chrNone",)]):
        text, ids = codec.decompress_region(cont, regs)
        assert text == b"" and len(ids) == 0


def test_untouched_payload_is_never_read(codec):
    g, b, L = _shape("config5")
    codec.set_reference(g)
    cont = codec.compress(b, L, block_reads=AUTO, gen_mode=1, substreams=0)
    lines = _lines(b)
    h = parse_container(cont)
    n1 = g.bases[1].size
    for regs in ([(g.names[0], 1, 500)], [(g.names[1], int(n1 * 0.6), int(n1 * 0.6) + 2_000)],
                 [(g.names[0], 200_000, 200_300), (g.names[1], n1 - 3_000, n1)]):
        sel = set(model_plan(cont, regs)[4])
        bad = bytearray(cont)
        n_bad = 0
        for k, blk in enumerate(h["blocks"]):
            if k not in sel and blk["pay"]:
                at = h["payload_off"] + blk["pay_off"]
                bad[at:at + blk["pay"]] = b"\xff" * blk["pay"]
                n_bad += 1
        assert n_bad > 0
        _check(codec, bytes(bad), b, lines, g.names, regs)


def test_more_flag_values_than_a_block_adapts(codec):
    g, b0, L = _shape("config1")
    rng = np.random.default_rng(9)
    values = rng.choice(4096, size=320, replace=False).astype(np.uint16)
    flag = values[rng.integers(0, 320, size=b0.n_reads)]
    b = Batch(b0.pos, np.ascontiguousarray(flag), b0.seq_len, b0.chr, b0.seq_off, b0.seq, b0.cigar_off, b0.cigar, b0.md_off, b0.md)
    codec.set_reference(g)
    lines = _lines(b)
    n1 = g.bases[1].size
    for gen_mode, block_reads, sub in ((1, AUTO, 0), (1, 400, 1)):
        cont = codec.compress(b, L, block_reads=block_reads, gen_mode=gen_mode, substreams=sub)
        for regs in ([(g.names[0], 1, 400)], [(g.names[0], 600_000, 601_000)], [(g.names[1], n1 - 5_000, n1)]):
            _check(codec, cont, b, lines, g.names, regs)


def test_legacy_stream(codec):
    g, b, L = _shape("config1")
    codec.set_reference(g)
    stream = codec.compress(b, L, block_reads=0)
    lines = _lines(b)
    _check(codec, stream, b, lines, g.names, [(g.names[1], 5_000, 9_000), (g.names[0], 1, 100)], legacy=True)
    assert codec.stats()["n_blocks"] == 1
    text, ids = codec.decompress_region(stream, [("chrNone", 1, 10)], legacy=True)
    assert text == b"" and len(ids) == 0


def test_host_buffer_encoder_with_blocks_of_several_sizes(codec, monkeypatch):
    monkeypatch.setenv("CBCG_PIPE_MIN_READS", "200000")
    cfg = synth.SynthConfig.named("config2", scale=0.2)                 # ~600 k reads: the chunked, overlapped encode
    g = synth.make_genome(cfg)
    b = synth.make_reads(cfg, g)
    codec.set_reference(g)
    cb = CompactBatch(b)
    out = np.empty(b.n_reads * 64 + (1 << 20), np.uint8)
    cont = out[:codec.compress_compact_into(cb, 150, AUTO, out, 1)].tobytes()
    cb.close()
    blocks = parse_container(cont)["blocks"]
    last = [x["n"] for x in blocks if x["gen"] == blocks[-1]["gen"]]
    assert len(set(last)) >= 3                                           # the ramp left blocks of several sizes
    lines = _lines(b)
    n = g.bases[0].size
    for regs in ([(g.names[0], 1, 1_000)], [(g.names[0], int(n * 0.5), int(n * 0.5) + 10_000)],
                 [(g.names[0], n - 20_000, n)], _many_regions(g, b, 11)):
        _check(codec, cont, b, lines, g.names, regs)
    full, _ = codec.decompress(cont)
    assert full == b"".join(lines)


def test_capacity_errors_report_the_sizes(codec):
    from cbc_b200 import codec as cm
    g, b, L = _shape("config1")
    codec.set_reference(g)
    cont = codec.compress(b, L, block_reads=AUTO, gen_mode=1)
    regs = [(g.names[0], 50_000, 60_000)]
    want_text, want_ids = codec.decompress_region(cont, regs)
    assert len(want_ids) > 10
    arr, nr = cm._region_array(regs)
    src = np.frombuffer(cont, np.uint8)
    out = np.empty(16, np.uint8); ids = np.empty(4, np.uint64)
    n, k = C.c_uint64(0), C.c_uint64(0)
    rc = codec.lib.cbcg_decode_region(codec.h, src.ctypes.data, src.nbytes, 0, arr, nr, out.ctypes.data, out.nbytes, C.byref(n),
                                      ids.ctypes.data, ids.size, C.byref(k))
    assert rc == -5 and n.value == len(want_text) and k.value == len(want_ids)
    assert codec.fetch_decoded().tobytes() == want_text
    big = np.empty(len(want_text), np.uint8)                             # text fits, ids do not
    rc = codec.lib.cbcg_decode_region(codec.h, src.ctypes.data, src.nbytes, 0, arr, nr, big.ctypes.data, big.nbytes, C.byref(n),
                                      ids.ctypes.data, ids.size, C.byref(k))
    assert rc == -5 and k.value == len(want_ids)
    rc = codec.lib.cbcg_decode_region(codec.h, src.ctypes.data, src.nbytes, 0, arr, nr, big.ctypes.data, big.nbytes, C.byref(n),
                                      None, 0, C.byref(k))                # no ids wanted
    assert rc == 0 and big.tobytes() == want_text


def test_only_the_decoded_blocks_need_the_reference(codec):
    """A reference that lacks the second record: a query at the start of the first decodes only blocks of the first."""
    g, b, L = _shape("config1")
    codec.set_reference(g)
    cont = codec.compress(b, L, block_reads=AUTO, gen_mode=1)
    lines = _lines(b)
    from cbc_b200.batch import Genome
    codec.set_reference(Genome([g.names[0]], [g.bases[0]]))
    _check(codec, cont, b, lines, g.names, [(g.names[0], 1, 2_000)])
    with pytest.raises(Exception) as e:
        codec.decompress_region(cont, [(g.names[1], 1, 2_000)])
    assert getattr(e.value, "status", None) == -7
    codec.set_reference(g)


def _run(*args, ok=True):
    p = subprocess.run([CLI, *args], capture_output=True, text=True, timeout=300)
    if ok:
        assert p.returncode == 0, p.stdout + p.stderr
    return p


def test_cli_region_decode_of_a_multi_batch_file():
    from cbc_b200 import shard
    cfg = synth.SynthConfig(seed=73, genome_len=1_200_000, n_chr=2, n_reads=40_000, len_min=100, len_max=100, p_sub=0.005, p_indel=0.002)
    g = synth.make_genome(cfg); b = synth.make_reads(cfg, g)
    lines = _lines(b)
    with tempfile.TemporaryDirectory() as d:
        fa, sam, cbcs = os.path.join(d, "r.fa"), os.path.join(d, "r.sam"), os.path.join(d, "a.cbcs")
        synth.write_fasta(fa, g); synth.write_sam(sam, b, g)
        _run("-c", "-B", "1", sam, cbcs, fa)
        with open(cbcs, "rb") as f:
            shards = shard.read_shards(f.read())
        assert len(shards) >= 4
        ends = np.cumsum([int.from_bytes(s[16:24], "little") for s in shards])
        r = int(ends[1])                                                 # the first read of batch 2
        assert b.chr[r - 1] == b.chr[r]

        def region(*regs):
            out = os.path.join(d, "r.txt")
            args = ["-d"]
            for x in regs:
                args += ["-r", x]
            p = _run(*args, cbcs, out, fa)
            assert "Decompression took" in p.stdout
            with open(out, "rb") as f:
                return f.read()

        def want(*regs):
            return b"".join(lines[i] for i in _want(b, g.names, regs))

        p0 = int(b.pos[int(ends[0]) // 2])                               # inside the first batch
        assert region(f"{g.names[0]}:{p0}-{p0 + 200}") == want((g.names[0], p0, p0 + 200))
        pa, pb = int(b.pos[r - 1]), int(b.pos[r])                        # across the boundary of batches 1 and 2
        name = g.names[int(b.chr[r])]
        assert region(f"{name}:{pa}-{pb + 50}") == want((name, pa, pb + 50))
        full = os.path.join(d, "all.txt")
        _run("-d", cbcs, full, fa)
        with open(full, "rb") as f:
            all_lines = f.read().splitlines(keepends=True)
        whole = region(g.names[1])                                       # a whole record: `cbc -d` restricted to it
        assert whole == b"".join(all_lines[i] for i in np.nonzero(b.chr == 1)[0])
        assert region(f"{g.names[1]}:{pb}") == want((g.names[1], pb))   # START alone: to the end of the record
        assert region("chrNone:1-100") == b""
        assert region(f"{g.names[0]}:1-100", f"{g.names[0]}:50-300") == want((g.names[0], 1, 300))
        p = _run("-d", "-C", "-r", g.names[0], cbcs, os.path.join(d, "x.txt"), fa, ok=False)
        assert p.returncode != 0 and "-C" in p.stderr
        # a single-block stream (-1) is decoded whole, then filtered
        stream = os.path.join(d, "s.cbc")
        _run("-c", "-1", sam, stream, fa)
        out = os.path.join(d, "s.txt")
        _run("-d", "-r", f"{g.names[0]}:{p0}-{p0 + 500}", stream, out, fa)
        with open(out, "rb") as f:
            assert f.read() == want((g.names[0], p0, p0 + 500))
