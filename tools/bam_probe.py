"""BAM output against SAM output of the same container (DESIGN.md 5f, "BAM output").

One batch of bench config 2 (or 5 with --config 5) coded with the default settings. cbcg_decode_bam and cbcg_decode_sam
(with the header, without a CIGAR section) are alternated --reps times; per call the device time (stats ms_total),
ms_reconstruct (K3 + K9 for cbcg_decode_bam, K3 + K6 for cbcg_decode_sam), ms_k3 and ms_d2h (CUDA events), and a wall
clock around the call. Medians after the first (warm-up) call are reported, with the bytes per read of each output. Before
anything is timed the BAM is checked: its header against the restatement (tests/bam_restate.py), every BGZF member's
framing, CRC32 and ISIZE, and the records of its first members against the restatement of the SAM lines.

The card's name and power limit are read in the same run (nvidia-smi, read-only query).

    python tools/bam_probe.py [--config 2|5] [--reps 5] [--out bam_probe.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from cbc_b200 import synth                                        # noqa: E402
from cbc_b200.codec import Codec                                  # noqa: E402
import bam_restate as B                                           # noqa: E402
import sam_restate as R                                           # noqa: E402

AUTO = 0xFFFFFFFF


def card():
    p = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return p.stdout.strip().splitlines()[0] if p.returncode == 0 and p.stdout.strip() else "unknown"


def timed(fn):
    t = time.perf_counter()
    out = fn()
    return out, 1e3 * (time.perf_counter() - t)


def med(v):
    return round(statistics.median(v[1:]), 3)                     # the first call is a warm-up


def check(data, sam, names, lengths, n_reads):
    """Header blocks, every member's framing / CRC / ISIZE, and the first members' records against the restatement."""
    head = B.header(names, lengths)
    assert data.startswith(head) and data.endswith(B.EOF_BLOCK)
    ms = B.members(data[len(head):])
    lines = [x + b"\n" for x in sam.split(b"\n")[:-1] if not x.startswith(b"@")]
    assert len(lines) == n_reads
    idx = {n.encode(): k for k, n in enumerate(names)}
    stream = b"".join(m[2] for m in ms[:8])
    want, k = bytearray(), 0
    while len(want) < len(stream):
        want += B.record(lines[k], idx)[0]; k += 1
    assert bytes(want) == stream, "BAM records differ from the restatement"
    return len(ms) - 1, k


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=2, choices=(2, 5))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="bam_probe.json")
    a = ap.parse_args()
    cfg = synth.SynthConfig.named(f"config{a.config}")
    g = synth.make_genome(cfg)
    b = synth.make_reads(cfg, g)
    L = int(b.seq_len.max())
    c = Codec(0)
    c.set_reference(g)
    cont = c.compress(b, L, block_reads=AUTO, gen_mode=1, substreams=0)
    bam, ids = c.decompress_bam(cont)
    sam, _ = c.decompress_sam(cont)
    n_blocks, checked = check(bam, sam, list(g.names), [x.size for x in g.bases], b.n_reads)
    print(json.dumps(dict(checked_records=checked, record_blocks=n_blocks)), flush=True)
    keys = ("ms_total", "ms_code", "ms_reconstruct", "ms_k3", "ms_d2h")
    bam_rows = {x: [] for x in keys + ("wall",)}
    sam_rows = {x: [] for x in keys + ("wall",)}
    for _ in range(a.reps + 1):
        (bam, _), w = timed(lambda: c.decompress_bam(cont))
        st = c.stats()
        for x in keys:
            bam_rows[x].append(st[x])
        bam_rows["wall"].append(w)
        (sam, _), w = timed(lambda: c.decompress_sam(cont))
        st = c.stats()
        for x in keys:
            sam_rows[x].append(st[x])
        sam_rows["wall"].append(w)
    c.close()
    one = dict(bam={x: med(v) for x, v in bam_rows.items()}, sam={x: med(v) for x, v in sam_rows.items()},
               bam_bytes=len(bam), sam_bytes=len(sam), bam_bytes_per_read=round(len(bam) / b.n_reads, 2),
               sam_bytes_per_read=round(len(sam) / b.n_reads, 2), record_blocks=n_blocks)
    one["k9_ms_estimate"] = round(one["bam"]["ms_reconstruct"] - one["bam"]["ms_k3"], 3)
    one["k6_ms_estimate"] = round(one["sam"]["ms_reconstruct"] - one["sam"]["ms_k3"], 3)
    print(json.dumps(one), flush=True)
    res = dict(card=card(), config=a.config, n_reads=b.n_reads, container_bytes=len(cont), reps=a.reps, one_batch=one)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(f"card: {res['card']}")


if __name__ == "__main__":
    main()
