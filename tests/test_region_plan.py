"""cbcg_region_plan on the CPU: which blocks, reads and payload bytes a region decode takes, against an independent Python
model that parses the container's varint index itself (include/cbcg_format.h, cbc_b200/csrc/container.h) and applies the
generation-prefix rule (DESIGN.md, "Region decode"). The containers come from the CPU restatement (tests/oracle_lib.py)."""
import ctypes as C
import os
import re
import struct
import subprocess

import numpy as np
import pytest

import oracle_lib as O
from cbc_b200 import codec, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UINT64_MAX = (1 << 64) - 1
ERR_ARG, ERR_FORMAT = -1, -8


# ---------------------------------------------------------------- the model

def _varints(buf):
    o = 0
    while o < len(buf):
        v, sh = 0, 0
        while True:
            c = buf[o]; o += 1
            v |= (c & 0x7f) << sh; sh += 7
            if not c & 0x80:
                break
        yield v


def _unzz(v):
    return (v >> 1) ^ -(v & 1)


def parse_container(cont: bytes):
    """Header, names and per-block (n_reads, chr, gen, base_pos, payload bytes) of a "CBCB" v4 container."""
    magic, version, max_len, L = struct.unpack_from("<4I", cont, 0)
    assert magic == 0x42434243 and version == 4
    n_reads, = struct.unpack_from("<Q", cont, 16)
    n_blocks, n_chr, block_reads, mode = struct.unpack_from("<4I", cont, 24)
    o, names = 40, []
    for _ in range(n_chr):
        nl, = struct.unpack_from("<I", cont, o); o += 4
        names.append(cont[o:o + nl].decode()); o += (nl + 3) & ~3
    ix_len, = struct.unpack_from("<I", cont, o); o += 4
    it = _varints(cont[o:o + ix_len])
    n, chr_, gen, base, d1, sub, blocks = block_reads, 0, 0, 0, 0, [0, 0, 0, 0], []
    for _ in range(n_blocks):
        v = next(it)
        n += _unzz(v >> 2)
        if v & 2:
            chr_ = next(it); base = 0; d1 = 0
        if v & 1:
            gen += next(it) + 1
        d1 += _unzz(next(it)); base += d1
        next(it)                                                       # edit count
        n_sub = 4 if (mode & 0x200) or gen < ((mode >> 16) & 0xff) else 1
        for q in range(n_sub):
            sub[q] += _unzz(next(it))
        blocks.append(dict(n=n, chr=chr_, gen=gen, base=base, pay=sum(sub[:n_sub])))
    first = pay = 0
    for b in blocks:
        b["first"], b["pay_off"] = first, pay
        first += b["n"]; pay += b["pay"]
    assert first == n_reads
    return dict(max_len=max_len, names=names, blocks=blocks, payload_off=o + ix_len)


def model_plan(cont: bytes, regions):
    """(n_blocks, n_reads, payload_bytes, max_seq_bytes, selected block indices, touched block indices)."""
    h = parse_container(cont)
    blocks, names, reach = h["blocks"], h["names"], h["max_len"] + 255
    touched = []
    for k, b in enumerate(blocks):
        hi = blocks[k + 1]["base"] if k + 1 < len(blocks) and blocks[k + 1]["chr"] == b["chr"] else float("inf")
        for r in regions:
            s = r[1] if len(r) > 1 else 1
            e = r[2] if len(r) > 2 else UINT64_MAX
            # a read of this block starts in [base, hi] and covers at most `reach` reference bases
            if names[b["chr"]] == r[0] and b["base"] <= e and hi + reach - 1 >= s:
                touched.append(k)
                break
    if not touched:
        return 0, 0, 0, 0, [], []
    g_star = max(blocks[k]["gen"] for k in touched)
    sel = [k for k, b in enumerate(blocks) if b["gen"] < g_star or (b["gen"] == g_star and k in touched)]
    return (len(sel), sum(blocks[k]["n"] for k in sel), sum(blocks[k]["pay"] for k in sel),
            sum(blocks[k]["n"] for k in touched) * (h["max_len"] + 1), sel, touched)


def ref_spans(b):
    """Reference bases each read covers: M + D + = + X of its input CIGAR."""
    out = np.empty(b.n_reads, np.int64)
    text = b.cigar.tobytes()
    for i in range(b.n_reads):
        cig = text[b.cigar_off[i]:b.cigar_off[i + 1]].decode()
        out[i] = sum(int(n) for n, op in re.findall(r"(\d+)([MIDNSHP=X])", cig) if op in "MD=X")
    return out


def overlapping(b, names, regions, span=None):
    """Ordinals of the input reads that overlap at least one region (the expected answer of a region decode).
    span: ref_spans(b), when the caller has it."""
    span = ref_spans(b) if span is None else span
    pos = b.pos.astype(np.int64)
    keep = np.zeros(b.n_reads, bool)
    for r in regions:
        if r[0] not in names:
            continue
        s = r[1] if len(r) > 1 else 1
        e = r[2] if len(r) > 2 else UINT64_MAX
        keep |= (b.chr == names.index(r[0])) & (pos <= e) & (pos + span - 1 >= s)
    return np.nonzero(keep)[0]


# ---------------------------------------------------------------- inputs

def _synth(**kw):
    cfg = synth.SynthConfig(**kw)
    g = synth.make_genome(cfg)
    return cfg, g, synth.make_reads(cfg, g)


@pytest.fixture(scope="module")
def one_chr():
    """variable length, indels and soft clips; generation-primed with several generations, and cold"""
    cfg, g, b = _synth(seed=61, genome_len=400_000, n_reads=20_000, len_min=60, len_max=200, p_sub=0.005, p_indel=0.01, p_clip=0.2)
    return g, b, {1: O.encode_blocked(b, g, 200, 700, 1), 0: O.encode_blocked(b, g, 200, 700, 0)}


@pytest.fixture(scope="module")
def two_chr():
    cfg, g, b = _synth(seed=62, genome_len=600_000, n_chr=2, n_reads=16_000, len_min=150, len_max=150, p_sub=0.005, p_indel=0.002)
    return g, b, O.encode_blocked(b, g, 150, 600, 1)


def _plan(cont, regions, legacy=False):
    p = codec.region_plan(cont, regions, legacy)
    return p["n_blocks"], p["n_reads"], p["payload_bytes"], p["max_seq_bytes"]


def _check(cont, b, names, regions):
    want = model_plan(cont, regions)
    assert _plan(cont, regions) == want[:4], regions
    # the model is generous, never short: every read that overlaps lies in a touched block
    blocks = parse_container(cont)["blocks"]
    firsts = np.array([x["first"] for x in blocks])
    owners = set(np.searchsorted(firsts, overlapping(b, names, regions), side="right") - 1)
    assert owners <= set(want[5]), regions
    return want


# ---------------------------------------------------------------- tests

def test_the_container_has_several_generations(one_chr):
    g, b, conts = one_chr
    gens = {x["gen"] for x in parse_container(conts[1])["blocks"]}
    assert len(gens) >= 3
    assert {x["gen"] for x in parse_container(conts[0])["blocks"]} == {0}


@pytest.mark.parametrize("where", ["start", "middle", "end"])
@pytest.mark.parametrize("gen_mode", [1, 0])
def test_plan_matches_the_model_along_the_chromosome(one_chr, where, gen_mode):
    g, b, conts = one_chr
    cont, name, n = conts[gen_mode], g.names[0], g.bases[0].size
    at = {"start": 1, "middle": n // 2, "end": n - 2_000}[where]
    want = _check(cont, b, g.names, [(name, at, at + 1_000)])
    assert 0 < want[0] <= len(parse_container(cont)["blocks"])
    if gen_mode == 0:                                                   # cold blocks: only the touched ones
        assert want[4] == want[5]


def test_region_at_the_start_takes_only_early_generations(one_chr):
    g, b, conts = one_chr
    blocks = parse_container(conts[1])["blocks"]
    want = _check(conts[1], b, g.names, [(g.names[0], 1, 50)])
    last_gen = blocks[-1]["gen"]
    assert all(blocks[k]["gen"] < last_gen for k in want[4])
    assert max(blocks[k]["n"] for k in want[4]) < max(x["n"] for x in blocks)   # the reduced table lacks the longest block


def test_region_in_the_last_generation_skips_most_blocks(one_chr):
    g, b, conts = one_chr
    blocks = parse_container(conts[1])["blocks"]
    n = g.bases[0].size
    want = _check(conts[1], b, g.names, [(g.names[0], int(n * 0.9), int(n * 0.9) + 300)])
    assert blocks[want[4][-1]]["gen"] == blocks[-1]["gen"]
    assert want[0] < len(blocks)


def test_region_across_a_block_boundary(one_chr):
    g, b, conts = one_chr
    blocks = parse_container(conts[1])["blocks"]
    k = len(blocks) - 5
    assert blocks[k]["chr"] == blocks[k - 1]["chr"]
    at = blocks[k]["base"]
    want = _check(conts[1], b, g.names, [(g.names[0], at - 3, at + 3)])
    assert {k - 1, k} <= set(want[5])


def test_whole_chromosome_and_absent_name(one_chr):
    g, b, conts = one_chr
    blocks = parse_container(conts[1])["blocks"]
    want = _check(conts[1], b, g.names, [(g.names[0],)])
    assert want[0] == len(blocks) and want[1] == b.n_reads
    assert _plan(conts[1], [("no_such_record", 1, 100)]) == (0, 0, 0, 0)
    assert _plan(conts[1], [("no_such_record",), (g.names[0], 1, 10)]) == model_plan(conts[1], [(g.names[0], 1, 10)])[:4]


def test_two_chromosomes(two_chr):
    g, b, cont = two_chr
    n1 = g.bases[1].size
    _check(cont, b, g.names, [(g.names[1], n1 // 2, n1 // 2 + 5_000)])
    _check(cont, b, g.names, [(g.names[1], 1, 100), (g.names[0], 1_000, 1_200), (g.names[0], 1_100, 9_000)])
    _check(cont, b, g.names, [(g.names[0], g.bases[0].size - 500, UINT64_MAX)])
    want = _check(cont, b, g.names, [(g.names[1],)])
    blocks = parse_container(cont)["blocks"]
    assert {k for k, x in enumerate(blocks) if x["chr"] == 1} == set(want[5])
    assert want[1] >= int((b.chr == 1).sum())


def test_legacy_stream_is_one_block():
    cfg, g, b = _synth(seed=63, genome_len=100_000, n_reads=3_000, len_min=100, len_max=100, p_sub=0.005)
    stream, _ = O.encode_legacy(b, g, 100)
    assert _plan(stream, [(g.names[0], 10, 20)], legacy=True) == (1, UINT64_MAX, len(stream), UINT64_MAX)


def test_bad_arguments_and_a_truncated_index(two_chr):
    g, b, cont = two_chr
    lib = codec.load_library()
    src = np.frombuffer(cont, np.uint8)

    def rc(regs, n=None, data=src, legacy=0):
        arr = (codec.Region * max(len(regs), 1))(*regs)
        out = [C.c_uint64(7) for _ in range(4)]
        return lib.cbcg_region_plan(data.ctypes.data, data.nbytes, legacy, arr, len(regs) if n is None else n,
                                    *[C.byref(v) for v in out]), [v.value for v in out]

    name = g.names[0].encode()
    assert rc([codec.Region(name, 0, 10)])[0] == ERR_ARG                # start 0
    assert rc([codec.Region(name, 11, 10)])[0] == ERR_ARG               # start > end
    assert rc([codec.Region(None, 1, 10)])[0] == ERR_ARG                # no name
    assert rc([codec.Region(name, 1, 10)], n=0)[0] == ERR_ARG           # no regions
    assert rc([codec.Region(name, 1, 10)], legacy=1)[0] == 0
    assert rc([codec.Region(name, 0, 10)], legacy=1)[0] == ERR_ARG
    h = parse_container(cont)
    ix_end = h["payload_off"]
    cut = np.frombuffer(cont[:ix_end - 3], np.uint8)                     # the index runs past the end
    got, out = rc([codec.Region(name, 1, 10)], data=cut)
    assert got == ERR_FORMAT and out == [0, 0, 0, 0]
    short = np.frombuffer(cont[:ix_end + 10], np.uint8)                  # the payload is cut short
    assert rc([codec.Region(name, 1, 10)], data=short)[0] == ERR_FORMAT
    assert rc([codec.Region(name, 1, 10)], data=np.frombuffer(b"CBCB" + bytes(60), np.uint8))[0] == ERR_FORMAT
    with pytest.raises(codec.CbcgError):
        codec.region_plan(cont, [(g.names[0], 5, 4)])


def test_region_mirror_matches_the_header_layout(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "cbcg.h"\nint main(void) {\n'
                   '    printf("%zu %zu %zu %zu\\n", sizeof(cbcg_region), offsetof(cbcg_region, name), '
                   'offsetof(cbcg_region, start), offsetof(cbcg_region, end));\n    return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    R = codec.Region
    assert got == [C.sizeof(R), R.name.offset, R.start.offset, R.end.offset]
