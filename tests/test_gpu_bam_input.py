"""BAM input on the GPU (cbcg_bgzf_inflate, cbcg_bam_open, cbcg_batch_upload_bam, cbcg_cigar_pack_resident; Codec.bgzf_inflate,
bam_open, upload_bam, compress_bam; `cbc -c x.bam`). The inflater against zlib over every deflate setting and the format's
corners; corrupt input against its status code; containers of BAM uploads against the same batch's upload, byte for byte;
record boundaries cut everywhere, members without a record start and a decoy chain; files fed in several calls; a BAM ->
container -> BAM -> container round trip; errors; and the command line against the SAM path."""
import ctypes as C
import os
import random
import struct
import subprocess
import tempfile
import zlib

import numpy as np
import pytest

import bam_input as BI
import edge_reads as E
import sam_restate as R
from cbc_b200 import synth
from cbc_b200.batch import Batch, Genome
from cbc_b200.codec import BamInfo, CbcgError, Codec
from test_gpu_sam import SETTINGS, SETTING_IDS, SHAPES, _shape

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "cbc_b200", "_build", "cbc")
AUTO = 0xFFFFFFFF
ERR_ARG, ERR_CAPACITY, ERR_INPUT, ERR_NO_REF, ERR_FORMAT, ERR_CORRUPT = -1, -5, -6, -7, -8, -9


@pytest.fixture(scope="module")
def codec():
    c = Codec(0)
    yield c
    c.close()


def _status(fn, *a, **k):
    with pytest.raises(CbcgError) as e:
        fn(*a, **k)
    return e.value.status


def _nt16_batch(b):
    """the batch a BAM reader's SAM text gives: SEQ through the 4-bit code"""
    seq = np.frombuffer(BI.nt16(b.seq.tobytes()), np.uint8).copy()
    return Batch(b.pos, b.flag, b.seq_len, b.chr, b.seq_off, seq, b.cigar_off, b.cigar, b.md_off, b.md)


def _mapped(b):
    """the reads of a batch without FLAG & 4: what a SAM or BAM ingest keeps"""
    keep = [i for i in range(b.n_reads) if not int(b.flag[i]) & 4]
    if len(keep) == b.n_reads:
        return b
    def pool(off, data):
        parts = [data[int(off[i]):int(off[i + 1])] for i in keep]
        o = np.zeros(len(keep) + 1, np.uint64); o[1:] = np.cumsum([len(x) for x in parts])
        return o, np.concatenate(parts).astype(np.uint8)
    k = np.array(keep)
    so, sq = pool(b.seq_off, b.seq); co, cg = pool(b.cigar_off, b.cigar)
    mo, md = pool(b.md_off, b.md) if b.md_off is not None else (None, None)
    return Batch(b.pos[k].copy(), b.flag[k].copy(), b.seq_len[k].copy(), b.chr[k].copy(), so, sq, co, cg, mo, md)


def _container(codec, L, setting):
    g, br, s = setting
    codec.encode_resident(L, br, g, s)
    return codec.fetch_container().tobytes()


# ---------------------------------------------------------------- inflate
def _inflate_cases():
    rng = random.Random(5)
    text = b"".join(b"read%d\tACGT%s\n" % (i, bytes(rng.choice(b"ACGT") for _ in range(rng.randint(0, 40)))) for i in range(3000))
    cases = [("setting_%d" % k, text[k * 2000:k * 2000 + 60000], st) for k, st in enumerate(BI.SETTINGS)]
    cases.append(("empty", b"", (6, 0, 8)))
    cases.append(("isize_65536_zeros", bytes(65536), (6, 0, 8)))
    cases.append(("isize_65536_fixed", b"AC" * 32768, (9, zlib.Z_FIXED, 8)))
    for d in (1, 2, 3, 7, 31, 32, 33, 258, 1000, 4097, 16385, 32767, 32768):     # matches at distance d, overlapping where d < len
        unit = bytes(rng.randrange(256) for _ in range(d))
        raw = (unit * (60000 // d + 2))[:60000] if d < 30000 else unit + unit[:65000 - d]
        cases.append(("dist_%d" % d, raw, (9, 0, 8)))
    fib = [1, 1]
    while len(fib) < 23:
        fib.append(fib[-1] + fib[-2])
    skew = bytearray()
    for sym, f in enumerate(fib):
        skew += bytes([sym * 11 % 256]) * f
    rng.shuffle(skew)
    cases.append(("fibonacci_15_bit_codes", bytes(skew[:65000]), (6, zlib.Z_HUFFMAN_ONLY, 9)))
    cases.append(("random", bytes(rng.randrange(256) for _ in range(65000)), (6, 0, 8)))
    cases.append(("random_short", bytes(rng.randrange(256) for _ in range(77)), (1, 0, 8)))
    return cases


INFLATE = _inflate_cases()


def _max_code_length(cdata):
    """the longest literal/length code of the first dynamic block (BTYPE 2) of a raw deflate stream"""
    bits = int.from_bytes(cdata[:400], "little")
    take = lambda n, at: ((bits >> at) & ((1 << n) - 1), at + n)
    _, at = take(1, 0); bt, at = take(2, at)
    assert bt == 2
    hlit, at = take(5, at); hdist, at = take(5, at); hclen, at = take(4, at)
    order = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
    cl = [0] * 19
    for k in range(hclen + 4):
        cl[order[k]], at = take(3, at)
    return max(l for l in range(16) if cl[l])                          # the longest code length the block's lengths use


def test_fibonacci_case_reaches_15_bits():
    raw, st = next((r, s) for n, r, s in INFLATE if n.startswith("fibonacci"))
    assert _max_code_length(BI.deflate_raw(raw, st)) == 15


@pytest.mark.parametrize("name,raw,setting", INFLATE, ids=[c[0] for c in INFLATE])
def test_inflate_equals_zlib(codec, name, raw, setting):
    data = BI.member(raw, setting=setting)
    assert codec.bgzf_inflate(data) == raw


def test_inflate_many_members_and_eof(codec):
    rng = random.Random(9)
    text = bytes(rng.choice(b"ACGTACGTNNxy\n\t") for _ in range(400_000))
    data = BI.bgzf(text, seed=3) + BI.member(b"") + BI.EOF_BLOCK
    assert codec.bgzf_inflate(data) == text
    assert codec.bgzf_inflate(BI.EOF_BLOCK) == b""


def _bits(fields):
    """raw deflate bits from (value, n_bits) pairs, LSB first; Huffman codes as (code, n, 'h') are written MSB first"""
    acc, n = 0, 0
    for f in fields:
        v, k = f[0], f[1]
        if len(f) == 3:
            v = int(format(v, "0%db" % k)[::-1], 2)
        acc |= v << n; n += k
    return acc.to_bytes((n + 7) // 8, "little")


def test_corrupt_input(codec):
    raw = b"ACGT" * 1000
    good = BI.member(raw)
    cases = {
        "crc": (BI.member(raw, crc=zlib.crc32(raw) ^ 1), ERR_CORRUPT),
        "isize": (BI.member(raw, isize=len(raw) + 1), ERR_CORRUPT),
        "btype_3": (BI.member(b"x", cdata=bytes([0x07, 0, 0, 0])), ERR_CORRUPT),
        # fixed block: length 3 (code 257) at distance 1 with nothing before it
        "distance_before_start": (BI.member(b"abc", cdata=_bits([(1, 1), (1, 2), (1, 7, "h"), (0, 5, "h"), (0, 7, "h")])), ERR_CORRUPT),
        "truncated": (BI.member(raw, cdata=BI.deflate_raw(raw, (6, zlib.Z_HUFFMAN_ONLY, 8))[:200]), ERR_CORRUPT),
        "bsize_past_end": (good[:-5], ERR_FORMAT),
        "gzip_without_bc": (__import__("gzip").compress(raw), ERR_FORMAT),
    }
    for name, (data, want) in cases.items():
        assert _status(codec.bgzf_inflate, data) == want, name
    assert codec.bgzf_inflate(good) == raw                  # the context still works


# ---------------------------------------------------------------- containers
_BAMS = {}


def _bam(shape, with_md=True):
    key = (shape, with_md)
    if key not in _BAMS:
        g, b, L, up, want = _shape(shape)
        _BAMS[key] = BI.write_bam(b, g.names, BI.genome_lengths(g), seed=11, with_md=with_md)
    return _BAMS[key]


@pytest.mark.parametrize("setting", SETTINGS, ids=SETTING_IDS)
@pytest.mark.parametrize("shape", list(SHAPES))
def test_containers_equal_the_batch_upload(codec, shape, setting):
    g, b, L, up, want = _shape(shape)
    b = _nt16_batch(b)
    codec.set_reference(g)
    codec.upload(b)
    want_cont = _container(codec, L, setting)
    want_sec = codec.cigar_pack(b)
    codec.upload(b.without_md())
    want_derived = _container(codec, L, setting)
    data = _bam(shape)
    used, tail = codec.bam_open(data)
    info, rest = codec.upload_bam(data[used:], carry=tail)
    assert rest == b"" and info["n_reads"] == b.n_reads and info["n_unmapped"] > 0
    assert info["n_records"] == b.n_reads + info["n_unmapped"] and info["inflated_bytes"] == len(tail) + len(codec.bgzf_inflate(data[used:]))
    assert (info["min_len"], info["max_len"]) == (int(b.seq_len.min()), int(b.seq_len.max()))
    assert _container(codec, L, setting) == want_cont
    assert codec.cigar_pack_resident() == want_sec
    codec.upload_bam(data[used:], carry=tail, derive_md=True)
    assert _container(codec, L, setting) == want_derived
    nomd = _bam(shape, with_md=False)
    used, tail = codec.bam_open(nomd)
    codec.upload_bam(nomd[used:], carry=tail, derive_md=True)
    assert _container(codec, L, setting) == want_derived
    assert _status(codec.upload_bam, nomd[used:], carry=tail) == ERR_INPUT    # no MD:Z without the flag


@pytest.mark.parametrize("shape", list(SHAPES))
def test_compress_bam_read_length_header(codec, shape):
    g, b, L, up, want = _shape(shape)
    b = _nt16_batch(b)
    codec.set_reference(g)
    data = _bam(shape)
    # get_read_length: the file's second record, mapped or not (reads of config 5 longer than it are refused, as for SAM)
    _, lens = BI.stream(b, 2, seed=11)
    if shape == "config1":
        cont, info = codec.compress_bam(data, block_reads=AUTO, gen_mode=1)
        assert info["len_first"] == lens[0] and info["len_second"] == lens[1]
        assert cont == codec.compress(b, lens[1], block_reads=AUTO, gen_mode=1)
    cont, info = codec.compress_bam(data, block_reads=AUTO, gen_mode=1, var_length=True)
    assert cont == codec.compress(b, int(b.seq_len.max()), block_reads=AUTO, gen_mode=1)


# ---------------------------------------------------------------- record boundaries
def _small():
    cfg = synth.SynthConfig(seed=41, genome_len=400_000, n_chr=2, n_reads=3_000, len_min=60, len_max=200, p_sub=0.005,
                            p_indel=0.02, p_clip=0.2)
    g = synth.make_genome(cfg)
    return g, _nt16_batch(synth.make_reads(cfg, g))


def _upload_cont(codec, data, L=200):
    used, tail = codec.bam_open(data)
    info, _ = codec.upload_bam(data[used:], carry=tail)
    codec.encode_resident(L, 256, 1, 1)
    return codec.fetch_container().tobytes(), info


def test_members_cut_inside_every_field(codec):
    g, b = _small()
    codec.set_reference(g)
    want = codec.compress(b, 200, block_reads=256, gen_mode=1)
    h = BI.header(g.names, BI.genome_lengths(g))
    recs, lens = BI.stream(b, 2, seed=4)
    # offsets of the fields of records along the stream: cut inside block_size, the fixed fields, the name, CIGAR, SEQ, QUAL, aux
    starts, o = [], 0
    while o < len(recs):
        starts.append(o); o += 4 + struct.unpack_from("<I", recs, o)[0]
    cuts = []
    for k, s in enumerate(starts[5:-5:7]):
        lrn, n_cig, l_seq = recs[s + 12], struct.unpack_from("<H", recs, s + 16)[0], struct.unpack_from("<I", recs, s + 20)[0]
        name, cig = s + 36, s + 36 + lrn
        seq = cig + 4 * n_cig; qual = seq + (l_seq + 1) // 2; aux = qual + l_seq
        cuts.append([s + 2, s + 4 + 10, name + lrn // 2, cig + 2 * n_cig, seq + l_seq // 4, qual + l_seq // 2, aux + 3][k % 7])
    cuts = sorted(set(len(h) + c for c in cuts))
    data = BI.bgzf(h + recs, cuts=cuts, seed=2)
    cont, info = _upload_cont(codec, data)
    assert cont == want and info["n_reads"] == b.n_reads


def test_members_without_a_record_start(codec):
    """records with a 150 KB B array: members cut inside them hold no record start"""
    g, b = _small()
    codec.set_reference(g)
    rng = random.Random(3)
    h = BI.header(g.names, BI.genome_lengths(g))
    recs = []
    for i in range(b.n_reads):
        flag, chr_, pos, cigar, seq, md = BI.batch_records(b, i)
        recs.append(BI.record(chr_, pos - 1, flag, cigar, seq, md, rng, b"q%d" % i, big_b=150_000 if i in (100, 2000) else 0))
    big_at = [len(h) + sum(len(x) for x in recs[:i]) for i in (100, 2000)]
    stream = h + b"".join(recs)
    cuts = [p + d for p in big_at for d in (1000, 60_000, 120_000)]
    cuts += [c for c in range(0, len(stream), 50_000) if all(abs(c - x) > 1000 for x in cuts)]
    data = BI.bgzf(stream, cuts=sorted(cuts), seed=5, settings=[(1, 0, 8)])
    cont, info = _upload_cont(codec, data)
    assert info["n_reads"] == b.n_reads
    assert cont == codec.compress(b, 200, block_reads=256, gen_mode=1)


def test_decoy_chain_is_repaired(codec):
    """a B array whose bytes are a chain of plausible records, with a member starting at its first byte"""
    g, b = _small()
    codec.set_reference(g)
    rng = random.Random(8)
    h = BI.header(g.names, BI.genome_lengths(g))
    fake = b"".join(BI.record(0, 100 + k, 0, b"20M", b"C" * 20, b"20", random.Random(k), b"fake%d" % k) for k in range(30))
    recs, cut = [], None
    for i in range(b.n_reads):
        flag, chr_, pos, cigar, seq, md = BI.batch_records(b, i)
        r = BI.record(chr_, pos - 1, flag, cigar, seq, md, rng, b"q%d" % i)
        if i == 700:
            body = r[4:] + b"ZZBC" + struct.pack("<I", len(fake)) + fake
            r = struct.pack("<I", len(body)) + body
            cut = len(h) + sum(len(x) for x in recs) + len(r) - len(fake)
        recs.append(r)
    stream = h + b"".join(recs)
    cuts = [cut, cut + 3000] + [c for c in range(0, len(stream), 50_000) if abs(c - cut) > 4000]
    data = BI.bgzf(stream, cuts=sorted(cuts), seed=6, settings=[(6, 0, 8)])
    cont, info = _upload_cont(codec, data)
    assert info["n_reads"] == b.n_reads
    assert cont == codec.compress(b, 200, block_reads=256, gen_mode=1)


def test_one_record_and_header_only_files(codec):
    g, b = _small()
    codec.set_reference(g)
    one = b.slice(0, 1)
    data = BI.write_bam(one, g.names, BI.genome_lengths(g), seed=1, unmapped=False)
    cont, info = _upload_cont(codec, data)
    assert info["n_records"] == 1 and info["len_second"] == 0
    assert cont == codec.compress(one, 200, block_reads=256, gen_mode=1)
    h = BI.bgzf(BI.header(g.names, BI.genome_lengths(g)), seed=2)
    used, tail = codec.bam_open(h)
    info, rest = codec.upload_bam(h[used:], carry=tail)
    assert info["n_records"] == 0 and info["n_reads"] == 0 and rest == b""


def test_block_size_below_32_is_a_format_error(codec):
    """a record area that is not records: a chain of block_size < 32 must stop with CBCG_ERR_FORMAT, not run on"""
    g, b = _small()
    codec.set_reference(g)
    h = BI.header(g.names, BI.genome_lengths(g))
    good = b""
    for i in range(50):
        flag, chr_, pos, cigar, seq, md = BI.batch_records(b, i)
        good += BI.record(chr_, pos - 1, flag, cigar, seq, md, random.Random(i), b"g%d" % i)
    bad = struct.pack("<I", 20) + bytes(20)                 # block_size 20: below the 32 bytes of fixed fields
    cases = {"zeroed_record_area": h + bytes(65000), "short_record_after_good_ones": h + good + bad + good,
             "zeroed_record_area_in_a_later_member": h + good + bytes(120000)}
    for name, stream in cases.items():
        data = BI.bgzf(stream, cuts=list(range(len(h) + 7, len(stream), 30000)), settings=[(6, 0, 8)])
        used, tail = codec.bam_open(data)
        assert _status(codec.upload_bam, data[used:], carry=tail) == ERR_FORMAT, name
    data = BI.bgzf(h, settings=[(6, 0, 8)])                # a caller's carry of zeros
    used, tail = codec.bam_open(data)
    assert _status(codec.upload_bam, data[used:], carry=tail + bytes(4000)) == ERR_FORMAT
    ok = BI.write_bam(b, g.names, BI.genome_lengths(g), seed=2)
    used, tail = codec.bam_open(ok)                          # the context still works
    assert codec.upload_bam(ok[used:], carry=tail)[0]["n_reads"] == b.n_reads


# ---------------------------------------------------------------- batches
def test_file_fed_in_several_calls(codec):
    g, b, L, up, want = _shape("config1")
    b = _nt16_batch(b)
    codec.set_reference(g)
    data = _bam("config1")
    used, carry = codec.bam_open(data)
    ends, o = [], used
    while o < len(data):
        o += struct.unpack_from("<H", data, o + 16)[0] + 1
        ends.append(o)
    rng = random.Random(2)
    picks = sorted(rng.sample(ends[:-1], 4)) + [len(data)]
    done, a = 0, used
    for k, e in enumerate(picks):
        info, carry = codec.upload_bam(data[a:e], carry=carry, last=(e == len(data)))
        n = info["n_reads"]
        codec.encode_resident(L, 512, 1, 1)
        got = codec.fetch_container().tobytes()
        if n:
            assert got == codec.compress(b.slice(done, done + n), L, block_reads=512, gen_mode=1)
        done += n; a = e
    assert done == b.n_reads and carry == b""
    # a partial record under CBCG_BAM_LAST
    used, carry = codec.bam_open(data)
    assert _status(codec.upload_bam, data[used:picks[0]], carry=carry, last=True) == ERR_FORMAT


# ---------------------------------------------------------------- round trip
@pytest.mark.parametrize("shape", list(SHAPES))
def test_round_trip(codec, shape):
    g, b, L, up, want = _shape(shape)
    codec.set_reference(g)
    cont = codec.compress(b, L, block_reads=AUTO, gen_mode=1)
    sec = codec.cigar_pack(b)
    bam, _ = codec.decompress_bam(cont, sec)
    cont2, info = codec.compress_bam(bam, L, block_reads=AUTO, gen_mode=1)
    sec2 = codec.cigar_pack_resident()
    assert codec.decompress_sam(cont2, sec2)[0] == codec.decompress_sam(cont, sec)[0]


# ---------------------------------------------------------------- errors
def test_abi_errors(codec):
    g, b = _small()
    fresh = Codec(0)
    try:
        data = BI.write_bam(b, g.names, BI.genome_lengths(g), seed=1)
        assert _status(fresh.bam_open, data) == ERR_NO_REF
        fresh.set_reference(g)
        assert _status(fresh.upload_bam, data) == ERR_ARG             # no cbcg_bam_open on this context
        used, tail = fresh.bam_open(data)
        fresh.set_reference(g)                                         # forgets the header
        assert _status(fresh.upload_bam, data[used:], carry=tail) == ERR_ARG
        used, tail = fresh.bam_open(data)
        ends, o = [], used                                             # members up to one that ends inside a record
        while o < len(data):
            o += struct.unpack_from("<H", data, o + 16)[0] + 1
            ends.append(o)
        end = ends[len(ends) // 2]
        stream = tail + b"".join(
            zlib.decompress(data[x + 18:y - 8], -15) for x, y in zip([used] + ends[:-1], ends) if y <= end)
        at = 0
        while at + 4 <= len(stream) and at + 4 + struct.unpack_from("<I", stream, at)[0] <= len(stream):
            at += 4 + struct.unpack_from("<I", stream, at)[0]
        assert at < len(stream)
        info = BamInfo()
        src = np.frombuffer(data[used:end], np.uint8)
        car = np.frombuffer(tail, np.uint8)
        rc = fresh.lib.cbcg_batch_upload_bam(fresh.h, car.ctypes.data if car.size else None, car.size, src.ctypes.data, src.nbytes, 0,
                                             C.byref(info), None, 0)
        assert rc == ERR_CAPACITY and info.tail_len == len(stream) - at and info.inflated_bytes == len(stream)
        info2, rest = fresh.upload_bam(data[used:end], carry=tail, last=False)
        assert rest == stream[at:]
        assert _status(fresh.upload_bam, data[used:end], carry=tail, last=True) == ERR_FORMAT
        # a reference without the second chromosome: the mapped reads on it are refused
        fresh.set_reference(Genome(names=[g.names[0]], bases=[g.bases[0]]))
        used, tail = fresh.bam_open(data)
        assert _status(fresh.upload_bam, data[used:], carry=tail) == ERR_NO_REF
        # not BAM inside BGZF
        fresh.set_reference(g)
        assert _status(fresh.bam_open, BI.bgzf(b"SAM\1" + bytes(100))) == ERR_FORMAT
        assert _status(fresh.bam_open, BI.bgzf(BI.header(g.names, BI.genome_lengths(g))[:-3], eof=False)) == ERR_FORMAT
        # l_seq 0 in a mapped record
        h = BI.header(g.names, BI.genome_lengths(g))
        rec = BI.record(0, 10, 0, b"*", b"", b"0", random.Random(1), b"empty")
        data = BI.bgzf(h + rec)
        used, tail = fresh.bam_open(data)
        assert _status(fresh.upload_bam, data[used:], carry=tail) == ERR_INPUT
    finally:
        fresh.close()


EDGE_GPU_GENOME, EDGE_GENOME = E.make_genomes()


@pytest.mark.parametrize("case", E.cases(EDGE_GENOME), ids=lambda c: c.name)
def test_edge_catalogue_refusals_equal_the_batch(codec, case):
    b = _nt16_batch(case.batch)
    codec.set_reference(EDGE_GPU_GENOME)
    lengths = [int(x.shape[0]) for x in EDGE_GPU_GENOME.bases]
    data = BI.write_bam(b, EDGE_GPU_GENOME.names, lengths, seed=3)

    def run(upload):
        try:
            upload()
            codec.encode_resident(case.L, 16, 1, 1)
            return codec.fetch_container().tobytes()
        except CbcgError as e:
            return e.status

    def bam_upload():
        used, tail = codec.bam_open(data)
        codec.upload_bam(data[used:], carry=tail)

    assert run(bam_upload) == run(lambda: codec.upload(_mapped(b)))


# ---------------------------------------------------------------- command line
def _run(*args, ok=True):
    p = subprocess.run([CLI, *map(str, args)], capture_output=True)
    assert (p.returncode == 0) == ok, p.stderr.decode()
    return p


def _read(path):
    with open(path, "rb") as f:
        return f.read()


def _sam_text(b, names, with_md=True):
    lines = [b"@HD\tVN:1.6\tSO:coordinate\n"]
    for i in range(b.n_reads):
        flag, chr_, pos, cigar, seq, md = BI.batch_records(b, i)
        tags = [b"MD:Z:" + md] if with_md else []
        lines.append(b"\t".join([b"r%d" % i, b"%d" % flag, names[chr_].encode(), b"%d" % pos, b"60", cigar, b"*", b"0", b"0",
                                 BI.nt16(seq), b"*"] + tags) + b"\n")
    return b"".join(lines)


def _with_extra_subfield(data):
    """every member re-framed with an 'XY' subfield of 4 bytes before BC (XLEN 14)"""
    out, o = [], 0
    while o < len(data):
        total = struct.unpack_from("<H", data, o + 16)[0] + 1
        body = data[o + 18:o + total]
        out.append(data[o:o + 10] + struct.pack("<H", 14) + b"XY" + struct.pack("<H", 4) + b"abcd" + b"BC" + struct.pack("<HH", 2, total + 8 - 1) + body)
        o += total
    return b"".join(out)


def test_members_with_other_extra_subfields(codec):
    g, b = _small()
    codec.set_reference(g)
    data = BI.write_bam(b, g.names, BI.genome_lengths(g), seed=4)
    assert codec.bgzf_inflate(_with_extra_subfield(data)) == codec.bgzf_inflate(data)


def test_cli_bam_equals_sam():
    g, b, L, up, want = _shape("config1")
    b = _nt16_batch(b)
    with tempfile.TemporaryDirectory() as d:
        fa = os.path.join(d, "g.fa")
        with open(fa, "wb") as f:
            for n, x in zip(g.names, g.bases):
                f.write(b">" + n.encode() + b"\n" + x.tobytes() + b"\n")
        sam, bam = os.path.join(d, "x.sam"), os.path.join(d, "x.bam")
        with open(sam, "wb") as f:
            f.write(_sam_text(b, g.names))
        with open(bam, "wb") as f:
            f.write(BI.write_bam(b, g.names, BI.genome_lengths(g), seed=7, unmapped=False))
        for opts in ([], ["-1"], ["-l"], ["-C"], ["-M"]):
            a, z = os.path.join(d, "a.cbc"), os.path.join(d, "z.cbc")
            _run("-c", *opts, sam, a, fa)
            _run("-c", *opts, bam, z, fa)
            assert _read(a) == _read(z), opts
            if "-C" in opts:
                assert _read(a + ".cig") == _read(z + ".cig")
        # members whose extra field holds another subfield before BC: read all the same, whole members per batch
        with open(bam, "wb") as f:
            f.write(_with_extra_subfield(BI.write_bam(b, g.names, BI.genome_lengths(g), seed=7, unmapped=False)))
        a, z = os.path.join(d, "a.cbc"), os.path.join(d, "z.cbc")
        _run("-c", sam, a, fa)
        _run("-c", bam, z, fa)
        assert _read(a) == _read(z)
        # several batches: decodes agree
        a, z = os.path.join(d, "a.cbc"), os.path.join(d, "z.cbc")
        _run("-c", "-B", "1", "-g", "0,0", sam, a, fa)
        _run("-c", "-B", "1", "-g", "0,0", bam, z, fa)
        for extra in ([], ["-S"]):
            da, dz = os.path.join(d, "a.out"), os.path.join(d, "z.out")
            _run("-d", *extra, a, da, fa)
            _run("-d", *extra, z, dz, fa)
            assert _read(da) == _read(dz), extra
