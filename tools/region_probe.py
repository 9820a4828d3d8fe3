"""Region decode against a full decode of the same container (DESIGN.md, "Region decode").

One batch: bench config 2 (or 3 with --config 3) coded with the default settings (generation-primed, automatic block
size, default layout). Per region (1 kb, 100 kb and 1 Mb, placed inside the early generations and at 50 % and 95 % of the
record): the cbcg_region_plan figures, then cbcg_decode_region and a full cbcg_decode alternated --reps times, each with
its device time (stats ms_total, CUDA events) and a wall clock around the call (both calls end in a device synchronise).
Medians are reported.

Several batches: the same input as SAM through `cbc -c -B MB` (at least 8 batches in a "CBCS" file), then `cbc -d` against
`cbc -d -r` for a 100 kb region, alternated, wall clock of the whole process and the device time the CLI reports.

The card's name and power limit are read in the same run (nvidia-smi, read-only query).

    python tools/region_probe.py [--config 2|3] [--reps 5] [--out region_probe.json]
"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from cbc_b200 import synth                                        # noqa: E402
from cbc_b200.codec import Codec, region_plan                     # noqa: E402

AUTO = 0xFFFFFFFF
CLI = os.path.join(ROOT, "cbc_b200", "_build", "cbc")


def card():
    p = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return p.stdout.strip().splitlines()[0] if p.returncode == 0 and p.stdout.strip() else "unknown"


def timed(fn):
    t = time.perf_counter()
    out = fn()
    return out, 1e3 * (time.perf_counter() - t)


def one_batch(c, cont, g, b, reps):
    name, n = g.names[0], g.bases[0].size
    early_pos = int(b.pos[20_000])                                 # inside the early generations (the first ~225 k reads)
    rows = []
    for size in (1_000, 100_000, 1_000_000):
        for where, at in (("early", early_pos), ("50%", n // 2), ("95%", int(n * 0.95))):
            regs = [(name, at, min(at + size - 1, n))]
            plan = region_plan(cont, regs)
            reg_dev, reg_wall, full_dev, full_wall = [], [], [], []
            reg_st = None
            for _ in range(reps + 1):                              # the first pair is a warm-up
                (text, ids), w = timed(lambda: c.decompress_region(cont, regs))
                reg_st = c.stats()
                reg_dev.append(reg_st["ms_total"]); reg_wall.append(w)
                (_, nr), w = timed(lambda: c.decompress(cont))
                full_dev.append(c.stats()["ms_total"]); full_wall.append(w)
            med = lambda v: round(statistics.median(v[1:]), 3)    # noqa: E731
            rows.append(dict(region_bases=size, where=where, start=regs[0][1], end=regs[0][2], plan=plan,
                             reads_returned=int(len(ids)), text_bytes=len(text), k2_blocks=reg_st["n_blocks"],
                             k2_reads=reg_st["n_reads"], region_ms_device=med(reg_dev), region_ms_wall=med(reg_wall),
                             region_ms_k2=round(reg_st["ms_code"], 3), region_ms_k3=round(reg_st["ms_k3"], 3),
                             region_ms_d2h=round(reg_st["ms_d2h"], 3),
                             full_ms_device=med(full_dev), full_ms_wall=med(full_wall), full_reads=int(nr)))
            print(json.dumps(rows[-1]), flush=True)
    return rows


def multi_batch(g, b, reps, batch_mb):
    with tempfile.TemporaryDirectory() as d:
        fa, sam, cbcs = os.path.join(d, "r.fa"), os.path.join(d, "r.sam"), os.path.join(d, "a.cbcs")
        synth.write_fasta(fa, g)
        synth.write_sam(sam, b, g)
        subprocess.run([CLI, "-c", "-B", str(batch_mb), sam, cbcs, fa], check=True, capture_output=True)
        with open(cbcs, "rb") as f:
            head = f.read(16)
        n_batches = int.from_bytes(head[8:12], "little") if head[:4] == b"CBCS" else 1
        n = g.bases[0].size
        region = f"{g.names[0]}:{n // 2}-{n // 2 + 99_999}"

        def run(*extra):
            out = os.path.join(d, "o.txt")
            p, w = timed(lambda: subprocess.run([CLI, "-d", *extra, cbcs, out, fa], check=True, capture_output=True, text=True))
            dev = float(re.search(r"device ([0-9.]+) ms", p.stdout).group(1))
            return w, dev, os.path.getsize(out)

        full, reg = [], []
        for _ in range(reps + 1):
            full.append(run())
            reg.append(run("-r", region))
        med = lambda v, k: round(statistics.median(x[k] for x in v[1:]), 3)   # noqa: E731
        row = dict(batches=n_batches, sam_bytes=os.path.getsize(sam), region=region,
                   full_wall_ms=med(full, 0), full_device_ms=med(full, 1), full_text_bytes=full[-1][2],
                   region_wall_ms=med(reg, 0), region_device_ms=med(reg, 1), region_text_bytes=reg[-1][2])
        print(json.dumps(row), flush=True)
        return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=2, choices=(2, 3))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--batch-mb", type=int, default=0, help="SAM MB per CLI batch (default: 1/8 of the SAM, rounded down)")
    ap.add_argument("--out", default="region_probe.json")
    a = ap.parse_args()
    cfg = synth.SynthConfig.named(f"config{a.config}")
    g = synth.make_genome(cfg)
    b = synth.make_reads(cfg, g)
    c = Codec(0)
    c.set_reference(g)
    cont = c.compress(b, 150, block_reads=AUTO, gen_mode=1, substreams=0)
    text, nr = c.decompress(cont)
    assert nr == b.n_reads and text == b.seq_lines()
    res = dict(card=card(), config=a.config, n_reads=b.n_reads, container_bytes=len(cont), reps=a.reps,
               one_batch=one_batch(c, cont, g, b, a.reps))
    c.close()
    sam_mb = b.n_reads * 330 >> 20                                 # about 330 bytes per 150-base SAM line
    res["multi_batch"] = multi_batch(g, b, max(1, a.reps // 2), a.batch_mb or max(1, sam_mb // 9))
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(f"card: {res['card']}")


if __name__ == "__main__":
    main()
