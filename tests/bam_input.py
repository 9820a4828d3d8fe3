"""BAM files for the BAM input tests (cbcg_bgzf_inflate, cbcg_bam_open, cbcg_batch_upload_bam): a Batch and its genome
written as a realistic coordinate-sorted BAM (SAMv1 4.2) in BGZF members (SAMv1 4.1).

Records carry what aligners write and the library drops: QNAMEs and QUALs from a seed, MAPQ and mate fields, aux tags of
every type before and after MD:Z (A, c, C, s, S, i, I, f, Z, H and B arrays of every subtype), and unmapped records, placed
ones between the mapped records and unplaced ones at the end. The record stream is cut into members at arbitrary offsets,
not at record boundaries, and every member is deflated by Python's zlib with its own settings: levels 0-9, the default,
filtered, Huffman-only, RLE and fixed strategies, memLevel 1 (many deflate blocks per member), and raw streams
concatenated after Z_SYNC_FLUSH, so that one member mixes stored, fixed and dynamic blocks."""
import random
import re
import struct
import zlib
from typing import List, Optional, Sequence, Tuple

from bam_restate import CIGAR_OPS, EOF_BLOCK, NT16, reg2bin

_CIG = re.compile(rb"(\d+)([MIDNSHP=X])")
MAX_ISIZE = 65280                    # what htslib puts in a member: its stored-block worst case fits BSIZE

# (level, strategy, memLevel), or "mixed": stored | fixed | dynamic raw streams after Z_SYNC_FLUSH
SETTINGS = [(lv, zlib.Z_DEFAULT_STRATEGY, 8) for lv in range(10)] + [
    (6, zlib.Z_FILTERED, 8), (6, zlib.Z_HUFFMAN_ONLY, 8), (6, zlib.Z_RLE, 8), (6, zlib.Z_FIXED, 8), (9, zlib.Z_FIXED, 8),
    (6, zlib.Z_DEFAULT_STRATEGY, 1), (1, zlib.Z_HUFFMAN_ONLY, 1), "mixed"]


def deflate_raw(data: bytes, setting=(6, zlib.Z_DEFAULT_STRATEGY, 8)) -> bytes:
    if setting == "mixed":
        a, b = len(data) // 3, 2 * len(data) // 3
        out = b""
        for part, (lv, st), fin in ((data[:a], (0, zlib.Z_DEFAULT_STRATEGY), zlib.Z_SYNC_FLUSH),
                                    (data[a:b], (6, zlib.Z_FIXED), zlib.Z_SYNC_FLUSH),
                                    (data[b:], (6, zlib.Z_DEFAULT_STRATEGY), zlib.Z_FINISH)):
            o = zlib.compressobj(lv, zlib.DEFLATED, -15, 8, st)
            out += o.compress(part) + o.flush(fin)
        return out
    lv, st, mem = setting
    o = zlib.compressobj(lv, zlib.DEFLATED, -15, mem, st)
    return o.compress(data) + o.flush()


def member(raw: bytes, cdata: Optional[bytes] = None, setting=(6, zlib.Z_DEFAULT_STRATEGY, 8), crc: Optional[int] = None,
           isize: Optional[int] = None) -> bytes:
    """One BGZF member holding raw (cdata: its deflate stream, else deflate_raw(raw, setting))."""
    if cdata is None:
        cdata = deflate_raw(raw, setting)
    total = 18 + len(cdata) + 8
    assert total <= 65536 and len(raw) <= 65536, (total, len(raw))
    head = struct.pack("<BBBBIBBHBBHH", 31, 139, 8, 4, 0, 0, 255, 6, 66, 67, 2, total - 1)
    return head + cdata + struct.pack("<II", zlib.crc32(raw) if crc is None else crc, len(raw) if isize is None else isize)


def bgzf(stream: bytes, cuts: Optional[Sequence[int]] = None, seed: int = 0, settings=None, eof: bool = True) -> bytes:
    """stream in members: cut at the given offsets (else at random sizes of 1 .. MAX_ISIZE bytes), each deflated with a
    setting drawn from `settings` (default: every one of SETTINGS in turn)."""
    rng = random.Random(seed)
    settings = settings or SETTINGS
    if cuts is None:
        cuts, at = [], 0
        while at < len(stream):
            at += rng.choice([rng.randint(1, 400), rng.randint(1, MAX_ISIZE), MAX_ISIZE, rng.randint(20000, MAX_ISIZE)])
            if at < len(stream):
                cuts.append(at)
    bounds = [0] + [c for c in cuts if 0 < c < len(stream)] + [len(stream)]
    out = [member(stream[a:b], setting=settings[k % len(settings)]) for k, (a, b) in enumerate(zip(bounds, bounds[1:])) if b > a]
    return b"".join(out) + (EOF_BLOCK if eof else b"")


def header(names: Sequence[str], lengths: Sequence[int], seed: int = 0) -> bytes:
    """magic, the SAM header text (@HD, @SQ, @RG, @PG), n_ref and the references"""
    text = "@HD\tVN:1.6\tSO:coordinate\n" + "".join(f"@SQ\tSN:{n}\tLN:{l}\n" for n, l in zip(names, lengths))
    text += f"@RG\tID:grp{seed}\tSM:sample\n@PG\tID:bwa\tPN:bwa\tCL:bwa mem ref.fa r1.fq r2.fq\n"
    t = text.encode()
    out = b"BAM\1" + struct.pack("<i", len(t)) + t + struct.pack("<i", len(names))
    for n, l in zip(names, lengths):
        out += struct.pack("<i", len(n) + 1) + n.encode() + b"\0" + struct.pack("<i", l)
    return out


def _aux(rng: random.Random, md: Optional[bytes], big_b: int = 0) -> bytes:
    """aux fields of every type, MD:Z among them (md None: no MD)"""
    before = [b"XAA" + bytes([rng.choice(b"ACGT")]), b"XCc" + struct.pack("<b", rng.randint(-128, 127)),
              b"NMC" + bytes([rng.randint(0, 9)]), b"XSs" + struct.pack("<h", rng.randint(-30000, 30000)),
              b"XFf" + struct.pack("<f", rng.random()), b"RGZgrp0\0",
              b"XBBc" + struct.pack("<I", 3) + bytes([1, 255, 7]),
              b"XHH" + b"1AE301\0"]
    after = [b"ASi" + struct.pack("<i", rng.randint(-2**31, 2**31 - 1)), b"XTS" + struct.pack("<H", rng.randint(0, 65535)),
             b"XII" + struct.pack("<I", rng.randint(0, 2**32 - 1)),
             b"ZBBs" + struct.pack("<I", 2) + struct.pack("<hh", -5, 5), b"ZIBI" + struct.pack("<I", 1) + struct.pack("<I", 9),
             b"ZFBf" + struct.pack("<I", 2) + struct.pack("<ff", 0.5, 1.5), b"ZSBS" + struct.pack("<I", 1) + struct.pack("<H", 3),
             b"ZiBi" + struct.pack("<I", 1) + struct.pack("<i", -3), b"ZCBC" + struct.pack("<I", 2) + bytes([0, 200])]
    rng.shuffle(before); rng.shuffle(after)
    k = rng.randint(0, len(before)); j = rng.randint(0, len(after))
    out = b"".join(before[:k]) + (b"MDZ" + md + b"\0" if md is not None else b"") + b"".join(after[:j])
    if big_b:
        out += b"ZZBC" + struct.pack("<I", big_b) + bytes(rng.randrange(256) for _ in range(min(big_b, 64))) + bytes(max(0, big_b - 64))
    return out


def record(ref: int, pos0: int, flag: int, cigar: bytes, seq: bytes, md: Optional[bytes], rng: random.Random, qname: bytes,
           big_b: int = 0) -> bytes:
    """one BAM record, block_size first. cigar: SAM text ('*' for none); seq: SAM text; pos0: 0-based (-1 for none)."""
    ops = [(int(n), CIGAR_OPS.index(o)) for n, o in _CIG.findall(cigar)] if cigar != b"*" else []
    span = sum(n for n, o in ops if o in (0, 2, 3, 7, 8))
    l_seq = len(seq)
    codes = [NT16.find(bytes([c])) if NT16.find(bytes([c])) >= 0 else 15 for c in seq.upper()]
    packed = bytes((codes[j] << 4) | (codes[j + 1] if j + 1 < l_seq else 0) for j in range(0, l_seq, 2))
    qual = bytes(rng.choice((2, 12, 23, 37)) for _ in range(l_seq))
    mate_ref = ref if rng.random() < 0.8 else -1
    body = struct.pack("<iiBBHHHIiii", ref, pos0, len(qname) + 1, rng.choice((0, 3, 60, 255)),
                       reg2bin(max(pos0, 0), max(pos0, 0) + (span or 1)), len(ops), flag, l_seq, mate_ref,
                       pos0 + rng.randint(-500, 500) if mate_ref >= 0 else -1, rng.randint(-600, 600))
    body += qname + b"\0" + b"".join(struct.pack("<I", n << 4 | o) for n, o in ops) + packed + qual + _aux(rng, md, big_b)
    return struct.pack("<I", len(body)) + body


def batch_records(b, i: int):
    """(flag, chr, POS, CIGAR, SEQ, MD or None) of read i of a Batch"""
    s, e = int(b.seq_off[i]), int(b.seq_off[i + 1])
    c0, c1 = int(b.cigar_off[i]), int(b.cigar_off[i + 1])
    md = None
    if b.md_off is not None:
        md = b.md[int(b.md_off[i]):int(b.md_off[i + 1])].tobytes()
    return int(b.flag[i]), int(b.chr[i]), int(b.pos[i]), b.cigar[c0:c1].tobytes(), b.seq[s:e].tobytes(), md


def stream(b, n_chr: int, seed: int = 0, unmapped: bool = True, with_md: bool = True) -> Tuple[bytes, List[int]]:
    """(record stream, l_seq of every record in order) of a Batch's reads, with unmapped records among them"""
    rng = random.Random(seed)
    out, lens = [], []
    for i in range(b.n_reads):
        flag, chr_, pos, cigar, seq, md = batch_records(b, i)
        if unmapped and rng.random() < 0.02:            # a placed unmapped record (the mate's position) before this read
            useq = bytes(rng.choice(b"ACGTN") for _ in range(rng.randint(0, 151)))
            out.append(record(chr_, pos - 1, 4 | 1 | 8, b"*", useq, None, rng, b"u%d" % i)); lens.append(len(useq))
        out.append(record(chr_, pos - 1, flag, cigar, seq, md if with_md else None, rng, b"r%d:%d" % (seed, i))); lens.append(len(seq))
    if unmapped:
        for k in range(rng.randint(1, 20)):             # unplaced unmapped records at the end
            useq = bytes(rng.choice(b"ACGT") for _ in range(rng.randint(0, 151)))
            out.append(record(-1, -1, 4, b"*", useq, None, rng, b"z%d" % k)); lens.append(len(useq))
    return b"".join(out), lens


def write_bam(b, names: Sequence[str], lengths: Sequence[int], seed: int = 0, unmapped: bool = True, with_md: bool = True,
              cuts=None, settings=None) -> bytes:
    """the header and the record stream as one stream cut anywhere (cuts: offsets into it), then the EOF block"""
    recs, _ = stream(b, len(names), seed, unmapped, with_md)
    return bgzf(header(names, lengths, seed) + recs, cuts=cuts, seed=seed + 1, settings=settings)


def genome_lengths(g) -> List[int]:
    return [int(x.shape[0]) for x in g.bases]


def nt16(seq: bytes) -> bytes:
    """SEQ as a BAM reader prints it"""
    return bytes(NT16[NT16.find(bytes([c])) if NT16.find(bytes([c])) >= 0 else 15] for c in seq.upper())

