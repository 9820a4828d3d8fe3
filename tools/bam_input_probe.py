"""BAM input against SAM input of the same reads (DESIGN.md 5g, "BAM input").

One batch of bench config 2 (or 5 with --config 5). The BAM is the container's own BAM output (cbcg_decode_bam) with QUAL
replaced by seeded qualities binned to four levels, as modern Illumina output, inflated and deflated again by zlib at level 6
(htslib's default) in members of 65 280 bytes; the SAM is cbcg_decode_sam's text of the same reads. Measured, medians after a
warm-up call:
  - cbcg_bgzf_inflate of the record members, in GB/s of inflated output (device time, stats ms_total: copies included);
  - cbcg_batch_upload_bam (ms_h2d), and a torch.profiler run of one call split into copy (host to device), inflate,
    boundaries (guess, chain, record starts), parse (count, write) and K7 (with derive_md);
  - cbcg_batch_upload of the same batch without MD (ms_h2d: its K7 included), and the CLI's host SAM ingest (`cbc -c`
    prints it);
  - single-threaded host zlib inflate of the same members, for scale;
  - `cbc -c x.bam` against `cbc -c x.sam` (config 5: with -l), wall clock. The SAM path of a batch this large runs the
    pipelined encode, the BAM path the resident one, so the two files need not be equal byte for byte (cli_same_file).
Before anything is timed, the upload's container is compared with the batch's (reported, not asserted).

The card's name and power limit are read in the same run (nvidia-smi, read-only query).

    python tools/bam_input_probe.py [--config 2|5] [--reps 5] [--out bam_input_probe.json]
"""
import argparse
import json
import os
import re
import statistics
import struct
import subprocess
import sys
import tempfile
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from cbc_b200 import synth                                        # noqa: E402
from cbc_b200.batch import Batch                                  # noqa: E402
from cbc_b200.codec import Codec                                  # noqa: E402
import bam_input as BI                                            # noqa: E402

AUTO = 0xFFFFFFFF
CLI = os.path.join(ROOT, "cbc_b200", "_build", "cbc")


def card():
    p = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return p.stdout.strip().splitlines()[0] if p.returncode == 0 and p.stdout.strip() else "unknown"


def med(v):
    return round(statistics.median(v[1:]), 3)                     # the first call is a warm-up


def realistic_bam(bam, seed):
    """the records of a K9 BAM with binned qualities, re-deflated at level 6 in 65 280-byte members; (file, stream)"""
    stream = bytearray(b"".join(zlib.decompress(bam[o + 18:o + struct.unpack_from("<H", bam, o + 16)[0] + 1 - 8], -15)
                                for o in _member_offsets(bam)))
    l_text, = struct.unpack_from("<i", stream, 4)
    o = 8 + l_text
    n_ref, = struct.unpack_from("<i", stream, o); o += 4
    for _ in range(n_ref):
        o += 8 + struct.unpack_from("<i", stream, o)[0]
    qa, ql = [], []
    while o < len(stream):
        size, = struct.unpack_from("<I", stream, o)
        lrn, n_cig, l_seq = stream[o + 12], struct.unpack_from("<H", stream, o + 16)[0], struct.unpack_from("<I", stream, o + 20)[0]
        qa.append(o + 36 + lrn + 4 * n_cig + (l_seq + 1) // 2); ql.append(l_seq)
        o += 4 + size
    qa, ql = np.array(qa, np.int64), np.array(ql, np.int64)
    idx = np.repeat(qa - np.concatenate(([0], np.cumsum(ql)[:-1])), ql) + np.arange(int(ql.sum()))
    rng = np.random.default_rng(seed)
    buf = np.frombuffer(stream, np.uint8).copy()
    buf[idx] = rng.choice(np.array([2, 12, 23, 37], np.uint8), size=idx.size, p=[0.02, 0.05, 0.13, 0.8])
    s = buf.tobytes()
    cuts = list(range(BI.MAX_ISIZE, len(s), BI.MAX_ISIZE))
    return BI.bgzf(s, cuts=cuts, settings=[(6, zlib.Z_DEFAULT_STRATEGY, 8)]), s


def _member_offsets(data):
    o = 0
    while o < len(data):
        yield o
        o += struct.unpack_from("<H", data, o + 16)[0] + 1


def profile_upload(c, data, used, tail, derive):
    """kernel and copy times of one cbcg_batch_upload_bam, by torch.profiler (CUDA activities)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        c.upload_bam(data[used:], carry=tail, derive_md=derive)
        torch.cuda.synchronize()
    parts = dict(copy=0.0, inflate=0.0, boundaries=0.0, parse=0.0, k7=0.0, other=0.0)
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        n, ms = e.name, e.device_time_total / 1e3 if hasattr(e, "device_time_total") else e.cuda_time_total / 1e3
        key = ("copy" if "HtoD" in n else "inflate" if "k10_inflate" in n else
               "boundaries" if re.search(r"k10_(guess|chain|rec_start)", n) else "parse" if re.search(r"k10_(count|write)", n) else
               "k7" if "k7_" in n else "other")
        parts[key] += ms
    return {k: round(v, 3) for k, v in parts.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=2, choices=(2, 5))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="bam_input_probe.json")
    a = ap.parse_args()
    cfg = synth.SynthConfig.named(f"config{a.config}")
    g = synth.make_genome(cfg)
    b = synth.make_reads(cfg, g)
    L = int(b.seq_len.max())
    c = Codec(0)
    c.set_reference(g)
    cont = c.compress(b, L, block_reads=AUTO, gen_mode=1, substreams=0)
    sec = c.cigar_pack(b)
    k9, _ = c.decompress_bam(cont, sec)
    sam, _ = c.decompress_sam(cont, sec)
    data, stream = realistic_bam(k9, 7)
    # the reads as the SAM text gives them (SEQ through the 4-bit code)
    b = Batch(b.pos, b.flag, b.seq_len, b.chr, b.seq_off, np.frombuffer(BI.nt16(b.seq.tobytes()), np.uint8).copy(), b.cigar_off,
              b.cigar, b.md_off, b.md)
    # the BAM's MD is K6's (md_rule.cuh), the rule K7 derives by: its upload codes as the batch without MD does
    used, tail = c.bam_open(data)
    info, _ = c.upload_bam(data[used:], carry=tail)
    c.encode_resident(L, AUTO, 1, 0)
    got = c.fetch_container().tobytes()
    c.upload(b.without_md())
    c.encode_resident(L, AUTO, 1, 0)
    same_container = got == c.fetch_container().tobytes()
    rows = dict(inflate_ms=[], upload_bam_ms=[], upload_bam_derive_ms=[], upload_ms=[], zlib_host_ms=[])
    recs = data[used:]
    for _ in range(a.reps + 1):
        c.bgzf_inflate(recs); rows["inflate_ms"].append(c.stats()["ms_total"])
        c.upload_bam(recs, carry=tail); rows["upload_bam_ms"].append(c.stats()["ms_h2d"])
        c.upload_bam(recs, carry=tail, derive_md=True); rows["upload_bam_derive_ms"].append(c.stats()["ms_h2d"])
        c.upload(b.without_md()); rows["upload_ms"].append(c.stats()["ms_h2d"])
        t = time.perf_counter()
        for o in _member_offsets(recs):
            zlib.decompress(recs[o + 18:o + struct.unpack_from("<H", recs, o + 16)[0] + 1 - 8], -15)
        rows["zlib_host_ms"].append(1e3 * (time.perf_counter() - t))
    m = {k: med(v) for k, v in rows.items()}
    inflated = info["inflated_bytes"] - len(tail)
    res = dict(card=card(), config=a.config, n_reads=b.n_reads, bam_bytes=len(data), inflated_bytes=len(stream),
               sam_bytes=len(sam), reps=a.reps, same_container_as_the_batch=same_container, medians=m,
               inflate_gb_s=round(inflated / (m["inflate_ms"] * 1e6), 2), zlib_host_gb_s=round(inflated / (m["zlib_host_ms"] * 1e6), 3),
               upload_bam_split=profile_upload(c, data, used, tail, False),
               upload_bam_derive_split=profile_upload(c, data, used, tail, True))
    c.close()
    with tempfile.TemporaryDirectory() as d:
        fa, xs, xb = os.path.join(d, "g.fa"), os.path.join(d, "x.sam"), os.path.join(d, "x.bam")
        with open(fa, "wb") as f:
            for n, x in zip(g.names, g.bases):
                f.write(b">" + n.encode() + b"\n" + x.tobytes() + b"\n")
        with open(xs, "wb") as f:
            f.write(sam)
        with open(xb, "wb") as f:
            f.write(data)
        cli = dict(sam=[], bam=[])
        for _ in range(3):
            for kind, path in (("sam", xs), ("bam", xb)):
                t = time.perf_counter()
                var = ["-l"] if a.config == 5 else []         # reads of 50..250 bases: the header length is the longest
                p = subprocess.run([CLI, "-c", *var, path, os.path.join(d, kind + ".cbc"), fa], capture_output=True, text=True)
                cli[kind].append(1e3 * (time.perf_counter() - t))
                assert p.returncode == 0, p.stderr
                res.setdefault("cli_" + kind + "_report", p.stdout.strip().splitlines()[-2])
        res["cli_wall_ms"] = {k: round(statistics.median(v[1:]), 1) for k, v in cli.items()}
        with open(os.path.join(d, "sam.cbc"), "rb") as x, open(os.path.join(d, "bam.cbc"), "rb") as y:
            res["cli_same_file"] = x.read() == y.read()
    print(json.dumps(res), flush=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
