"""A Python restatement of the BAM that cbcg_decode_bam writes (include/cbcg.h, k9_bam.cu, DESIGN.md 5f), for the tests.

The records are SAM lines (sam_restate.sam_lines) encoded as BAM (SAMv1 4.2): refID the RNAME's index in the header's
name list, pos POS - 1, read name "*", MAPQ 255, bin reg2bin(pos, pos + the CIGAR's M D N = X span, or pos + 1), the CIGAR
as u32 len << 4 | op, SEQ in the 4-bit code =ACMGRSVTWYHKDBN, QUAL 0xff per base, no mate, then NM (C, S above 255) and MD
(Z). Blocks hold whole records: record i > 0 opens a block when floor(U_i / 49152) != floor(U_{i-1} / 49152), U_i the
record bytes before it. Each BGZF block is one final fixed-Huffman deflate block: every byte a literal except QUAL, which
is one literal 0xff, then one match <l_seq - 1, distance 1> when l_seq - 1 >= 3. The header is "BAM\\1", l_text, the SAM
header text, n_ref and (l_name, name\\0, l_ref) per name, in stored deflate blocks of 65 280 bytes.

`read_bam` is an independent reader (struct + zlib) that turns BGZF BAM back into SAM lines.

TEST INFRASTRUCTURE: imported by tests/test_bam_restate.py and tests/test_gpu_bam.py."""
from __future__ import annotations

import re
import struct
import zlib
from typing import Dict, List, Sequence, Tuple

import sam_restate as R

CUT = 49152
MAX_RECORD = 8192
STORED = 65280
CIGAR_OPS = b"MIDNSHP=X"
NT16 = b"=ACMGRSVTWYHKDBN"
EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
_CIG = re.compile(rb"(\d+)([MIDNSHP=X])")

LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]


def _code(c: int) -> int:
    u = c - 32 if ord("a") <= c <= ord("z") else c
    k = NT16.find(bytes([u]))
    return 15 if k < 0 else k


def reg2bin(beg: int, end: int) -> int:
    end -= 1
    for shift, off in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        if beg >> shift == end >> shift:
            return off + (beg >> shift)
    return 0


def record(line: bytes, ref_index: Dict[bytes, int]) -> Tuple[bytes, int]:
    """(record bytes, l_seq) of one SAM line of cbcg_decode_sam."""
    f = line.rstrip(b"\n").split(b"\t")
    flag, rname, pos, cigar, seq = int(f[1]), f[2], int(f[3]), f[5], f[9]
    nm, md = int(f[11][5:]), f[12][5:]
    ops = [(int(n), CIGAR_OPS.index(op)) for n, op in _CIG.findall(cigar)] if cigar != b"*" else []
    span = sum(n for n, op in ops if op in (0, 2, 3, 7, 8))
    beg = pos - 1
    l_seq = len(seq)
    packed = bytes((_code(seq[j]) << 4) | (_code(seq[j + 1]) if j + 1 < l_seq else 0) for j in range(0, l_seq, 2))
    tags = (b"NMC" + struct.pack("<B", nm) if nm <= 255 else b"NMS" + struct.pack("<H", nm)) + b"MDZ" + md + b"\0"
    body = struct.pack("<iiBBHHHIiii", ref_index[rname] if rname != b"*" else -1, beg, 2, 255,
                       reg2bin(beg, beg + (span or 1)), len(ops), flag, l_seq, -1, -1, 0)
    body += b"*\0" + b"".join(struct.pack("<I", n << 4 | op) for n, op in ops) + packed + b"\xff" * l_seq + tags
    rec = struct.pack("<I", len(body)) + body
    assert len(rec) <= MAX_RECORD, "a record above 8 192 bytes is CBCG_ERR_FORMAT"
    return rec, l_seq


def cut(sizes: Sequence[int]) -> List[Tuple[int, int]]:
    """[first, end) record ranges of the blocks of one call's record stream."""
    out, u, first = [], 0, 0
    for i, n in enumerate(sizes):
        if i > 0 and u // CUT != (u - sizes[i - 1]) // CUT:
            out.append((first, i)); first = i
        u += n
    if sizes:
        out.append((first, len(sizes)))
    return out


class BitWriter:
    """Deflate's LSB-first bit order; Huffman codes go most significant bit first."""

    def __init__(self):
        self.acc, self.n, self.out = 0, 0, bytearray()

    def bits(self, v: int, n: int):
        self.acc |= v << self.n; self.n += n
        while self.n >= 8:
            self.out.append(self.acc & 255); self.acc >>= 8; self.n -= 8

    def huff(self, code: int, n: int):
        self.bits(int(format(code, f"0{n}b")[::-1], 2), n)

    def lit(self, v: int):
        if v < 144:
            self.huff(0x30 + v, 8)
        elif v < 256:
            self.huff(0x190 + v - 144, 9)
        elif v < 280:
            self.huff(v - 256, 7)
        else:
            self.huff(0xC0 + v - 280, 8)

    def match(self, length: int):
        k = max(i for i in range(29) if LEN_BASE[i] <= length) if length < 258 else 28
        self.lit(257 + k)
        self.bits(length - LEN_BASE[k], LEN_EXTRA[k])
        self.huff(0, 5)                                   # distance 1

    def flush(self) -> bytes:
        if self.n:
            self.out.append(self.acc & 255)
        return bytes(self.out)


def gzip_member(cdata: bytes, raw: bytes) -> bytes:
    head = b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", len(cdata) + 25)
    return head + cdata + struct.pack("<II", zlib.crc32(raw), len(raw))


def data_block(recs: Sequence[Tuple[bytes, int]]) -> bytes:
    bw = BitWriter()
    bw.bits(1, 1); bw.bits(1, 2)                          # BFINAL 1, BTYPE 01
    for rec, l_seq in recs:
        qa = _qual_at(rec)
        for b in rec[:qa]:
            bw.lit(b)
        if l_seq:
            bw.lit(0xFF)
            if l_seq - 1 >= 3:
                bw.match(l_seq - 1)
            else:
                for _ in range(l_seq - 1):
                    bw.lit(0xFF)
        for b in rec[qa + l_seq:]:
            bw.lit(b)
    bw.lit(256)
    return gzip_member(bw.flush(), b"".join(r for r, _ in recs))


def _qual_at(rec: bytes) -> int:
    n_ops, = struct.unpack_from("<H", rec, 16)
    l_seq, = struct.unpack_from("<I", rec, 20)
    return 36 + 2 + 4 * n_ops + (l_seq + 1) // 2


def record_blocks(lines: Sequence[bytes], names: Sequence[str]) -> bytes:
    """The BGZF blocks of one call's records."""
    idx = {}
    for k, n in enumerate(names):
        idx.setdefault(n.encode(), k)
    recs = [record(x, idx) for x in lines]
    return b"".join(data_block(recs[a:b]) for a, b in cut([len(r) for r, _ in recs]))


def header(names: Sequence[str], lengths: Sequence[int]) -> bytes:
    """The header's BGZF blocks: stored deflate blocks of 65 280 bytes."""
    text = R.header(names, lengths)
    raw = b"BAM\1" + struct.pack("<I", len(text)) + text + struct.pack("<I", len(names))
    for n, ln in zip(names, lengths):
        raw += struct.pack("<I", len(n) + 1) + n.encode() + b"\0" + struct.pack("<I", ln)
    out = []
    for a in range(0, len(raw), STORED):
        piece = raw[a:a + STORED]
        out.append(gzip_member(b"\x01" + struct.pack("<HH", len(piece), len(piece) ^ 0xFFFF) + piece, piece))
    return b"".join(out)


def bam(lines: Sequence[bytes], names: Sequence[str], lengths: Sequence[int], with_header=True, with_eof=True) -> bytes:
    return (header(names, lengths) if with_header else b"") + record_blocks(lines, names) + (EOF_BLOCK if with_eof else b"")


# ---------------------------------------------------------------- an independent reader
def members(data: bytes) -> List[Tuple[int, int, bytes]]:
    """(offset, BSIZE + 1, inflated payload) of every BGZF member; checks the framing, CRC32 and ISIZE."""
    out, o = [], 0
    while o < len(data):
        id1, id2, cm, flg, _, _, _, xlen = struct.unpack_from("<BBBBIBBH", data, o)
        assert (id1, id2, cm, flg, xlen) == (31, 139, 8, 4, 6), o
        si1, si2, slen, bsize = struct.unpack_from("<BBHH", data, o + 12)
        assert (si1, si2, slen) == (66, 67, 2), o
        total = bsize + 1
        cdata = data[o + 18:o + total - 8]
        crc, isize = struct.unpack_from("<II", data, o + total - 8)
        raw = zlib.decompress(cdata, -15)
        assert len(raw) == isize and zlib.crc32(raw) == crc, o
        out.append((o, total, raw))
        o += total
    assert o == len(data)
    return out


def read_bam(data: bytes, check_blocks: bool = True):
    """(names, lengths, SAM text of the header, SAM record lines) of a BGZF BAM file; check_blocks: no record spans two
    members, and the file ends with the EOF block."""
    ms = members(data)
    assert data.endswith(EOF_BLOCK)
    stream = b"".join(m[2] for m in ms)
    assert stream[:4] == b"BAM\1"
    l_text, = struct.unpack_from("<I", stream, 4)
    text = stream[8:8 + l_text]
    o = 8 + l_text
    n_ref, = struct.unpack_from("<I", stream, o); o += 4
    names, lengths = [], []
    for _ in range(n_ref):
        ln, = struct.unpack_from("<I", stream, o); o += 4
        names.append(stream[o:o + ln - 1].decode()); o += ln
        lengths.append(struct.unpack_from("<I", stream, o)[0]); o += 4
    head_end = o
    bounds, at = set(), 0
    for m in ms:
        at += len(m[2]); bounds.add(at)
    assert head_end in bounds, "the header ends a member"
    lines = []
    while o < len(stream):
        size, = struct.unpack_from("<I", stream, o)
        rec = stream[o + 4:o + 4 + size]
        if check_blocks:
            assert not any(o < b < o + 4 + size for b in bounds), "a record spans two members"
        ref_id, pos, l_name, mapq, bin_, n_ops, flag, l_seq, nref, npos, tlen = struct.unpack_from("<iiBBHHHIiii", rec, 0)
        q = 32
        qname = rec[q:q + l_name - 1]; q += l_name
        ops = struct.unpack_from(f"<{n_ops}I", rec, q); q += 4 * n_ops
        cigar = b"".join(b"%d%c" % (v >> 4, CIGAR_OPS[v & 15]) for v in ops) or b"*"
        packed = rec[q:q + (l_seq + 1) // 2]; q += (l_seq + 1) // 2
        seq = bytes(NT16[(packed[j >> 1] >> (4 * (1 - (j & 1)))) & 15] for j in range(l_seq))
        qual = rec[q:q + l_seq]; q += l_seq
        assert qual == b"\xff" * l_seq
        span = sum(v >> 4 for v in ops if (v & 15) in (0, 2, 3, 7, 8))
        assert bin_ == reg2bin(pos, pos + (span or 1))
        assert (mapq, nref, npos, tlen) == (255, -1, -1, 0)
        tags = []
        while q < len(rec):
            tag, typ = rec[q:q + 2], rec[q + 2:q + 3]; q += 3
            if typ == b"C":
                v = b"%d" % rec[q]; q += 1; typ = b"i"
            elif typ == b"S":
                v = b"%d" % struct.unpack_from("<H", rec, q)[0]; q += 2; typ = b"i"
            elif typ == b"Z":
                e = rec.index(b"\0", q); v = rec[q:e]; q = e + 1
            else:
                raise AssertionError(typ)
            tags.append(tag + b":" + typ + b":" + v)
        rname = names[ref_id].encode() if ref_id >= 0 else b"*"
        lines.append(b"\t".join([qname, b"%d" % flag, rname, b"%d" % (pos + 1), b"%d" % mapq, cigar, b"*", b"0", b"0", seq, b"*"] + tags) + b"\n")
        o += 4 + size
    return names, lengths, text, lines
