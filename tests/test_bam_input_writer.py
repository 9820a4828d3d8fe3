"""The BAM writer of the BAM input tests (tests/bam_input.py), checked without a GPU: Python's gzip inflates its files,
every member's BSIZE, CRC32 and ISIZE are valid, and an independent struct reader gives back the reads' SAM fields."""
import gzip
import struct
import zlib

import pytest

import bam_input as BI
from cbc_b200 import synth


def _batch():
    cfg = synth.SynthConfig(seed=31, genome_len=300_000, n_chr=2, n_reads=2_000, len_min=50, len_max=250, p_sub=0.005,
                            p_indel=0.02, p_clip=0.3)
    g = synth.make_genome(cfg)
    return g, synth.make_reads(cfg, g)


def _members(data):
    """(BSIZE + 1, CRC32, ISIZE, raw) per member, framing read with struct"""
    out, o = [], 0
    while o < len(data):
        id1, id2, cm, flg, xlen = struct.unpack_from("<BBBB6xH", data, o)
        assert (id1, id2, cm, flg) == (0x1f, 0x8b, 8, 4)
        si1, si2, slen, bsize = struct.unpack_from("<BBHH", data, o + 12)
        assert (si1, si2, slen, xlen) == (ord("B"), ord("C"), 2, 6)
        total = bsize + 1
        crc, isize = struct.unpack_from("<II", data, o + total - 8)
        raw = zlib.decompress(data[o + 18:o + total - 8], -15)
        out.append((total, crc, isize, raw))
        o += total
    assert o == len(data)
    return out


def _records(s, o):
    """SAM fields of the records of stream s from offset o"""
    out = []
    while o < len(s):
        size, ref, pos, l_name, _, _, n_ops, flag, l_seq = struct.unpack_from("<IiiBBHHHI", s, o)
        q = o + 36
        q += l_name
        ops = struct.unpack_from(f"<{n_ops}I", s, q); q += 4 * n_ops
        cigar = b"".join(b"%d%c" % (v >> 4, b"MIDNSHP=X"[v & 15]) for v in ops) or b"*"
        seq = bytes(b"=ACMGRSVTWYHKDBN"[(s[q + (j >> 1)] >> (4 * (1 - (j & 1)))) & 15] for j in range(l_seq))
        q += (l_seq + 1) // 2 + l_seq
        md, end = None, o + 4 + size
        while q < end:
            tag, typ = s[q:q + 2], chr(s[q + 2]); q += 3
            if typ in "AcC":
                q += 1
            elif typ in "sS":
                q += 2
            elif typ in "iIf":
                q += 4
            elif typ in "ZH":
                e = s.index(b"\0", q)
                if tag == b"MD" and typ == "Z" and md is None:
                    md = s[q:e]
                q = e + 1
            else:
                assert typ == "B"
                sub, n = chr(s[q]), struct.unpack_from("<I", s, q + 1)[0]
                q += 5 + n * {"c": 1, "C": 1, "s": 2, "S": 2, "i": 4, "I": 4, "f": 4}[sub]
        assert q == end
        out.append((flag, ref, pos + 1, cigar, seq, md))
        o = end
    return out


@pytest.mark.parametrize("with_md", [True, False])
def test_writer_round_trip(with_md):
    g, b = _batch()
    data = BI.write_bam(b, g.names, BI.genome_lengths(g), seed=3, with_md=with_md)
    ms = _members(data)
    assert data.endswith(BI.EOF_BLOCK) and ms[-1][3] == b""
    for total, crc, isize, raw in ms:
        assert total <= 65536 and isize == len(raw) <= 65536 and crc == zlib.crc32(raw)
    s = gzip.decompress(data)
    assert s == b"".join(m[3] for m in ms)
    assert s[:4] == b"BAM\1"
    l_text, = struct.unpack_from("<i", s, 4)
    o = 8 + l_text
    n_ref, = struct.unpack_from("<i", s, o); o += 4
    names = []
    for _ in range(n_ref):
        ln, = struct.unpack_from("<i", s, o)
        names.append(s[o + 4:o + 3 + ln].decode()); o += 8 + ln
    assert names == g.names
    recs = _records(s, o)
    mapped = [r for r in recs if not r[0] & 4]
    assert len(mapped) == b.n_reads and len(recs) > b.n_reads              # unmapped records are among them
    assert any(r[1] == -1 for r in recs) and any(r[0] & 4 and r[1] >= 0 for r in recs)
    for i, r in enumerate(mapped):
        flag, chr_, pos, cigar, seq, md = BI.batch_records(b, i)
        assert r == (flag, chr_, pos, cigar, BI.nt16(seq), md if with_md else None)


def test_every_setting_inflates():
    data = bytes(range(256)) * 100 + b"ACGT" * 5000
    for k, st in enumerate(BI.SETTINGS):
        raw = data[k * 100:k * 100 + 40000]
        m = BI.member(raw, setting=st)
        assert gzip.decompress(m) == raw, st
    mixed = BI.deflate_raw(data[:60000], "mixed")
    assert zlib.decompress(mixed, -15) == data[:60000]
