"""Pileup against SAM output of the same regions (DESIGN.md, "Pileup").

One batch of bench config 2 (or 5 with --config 5) coded with the default settings (generation-primed, automatic block
size, default layout), with its CIGAR side section. Per region (1 kb, 100 kb and 1 Mb inside the early generations and at
50 % and 95 % of the record, and the whole record): cbcg_pileup and cbcg_decode_sam alternated --reps times after a
warm-up pair, medians of the device time (stats ms_total, CUDA events) and of a wall clock around the call (both calls end
in a device synchronise); the device time split into K2 (ms_code), K3 (ms_k3, when it ran) and the rest of ms_reconstruct
(the pileup kernels, or K6); and the bytes each returns. The first pass checks the rows against the restatement in
tests/pileup_restate.py over the SAM lines of the 1 kb regions.

The card's name and power limit are read in the same run (nvidia-smi, read-only query).

    python tools/pileup_probe.py [--config 2|5] [--reps 3] [--out pileup_probe.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from cbc_b200 import synth                                        # noqa: E402
from cbc_b200.codec import Codec                                  # noqa: E402
import pileup_restate as P                                        # noqa: E402
import sam_restate as R                                           # noqa: E402

AUTO = 0xFFFFFFFF


def card():
    p = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return p.stdout.strip().splitlines()[0] if p.returncode == 0 and p.stdout.strip() else "unknown"


def timed(fn):
    t = time.perf_counter()
    out = fn()
    return out, 1e3 * (time.perf_counter() - t)


def split(st):
    k3 = st["ms_k3"]
    return dict(k2=round(st["ms_code"], 3), k3=round(k3, 3), after_k2=round(st["ms_reconstruct"], 3),
                d2h=round(st["ms_d2h"], 3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=2, choices=(2, 5))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="pileup_probe.json")
    a = ap.parse_args()
    cfg = synth.SynthConfig.named(f"config{a.config}")
    g = synth.make_genome(cfg)
    b = synth.make_reads(cfg, g)
    L = int(b.seq_len.max())
    c = Codec(0)
    c.set_reference(g)
    cont = c.compress(b, L, block_reads=AUTO, gen_mode=1, substreams=0)
    sec = c.cigar_pack(b)
    up = R.upper(g)
    name, n = g.names[0], g.bases[0].size
    early = int(b.pos[20_000])                                     # inside the early generations
    cases = [(size, where, at) for size in (1_000, 100_000, 1_000_000)
             for where, at in (("early", early), ("50%", n // 2), ("95%", int(n * 0.95)))] + [(n, "record", 1)]
    rows = []
    for size, where, at in cases:
        regs = [(name, at, min(at + size - 1, n))]
        pu_dev, pu_wall, sam_dev, sam_wall = [], [], [], []
        for k in range(a.reps + 1):                                # the first pair is a warm-up
            got, w = timed(lambda: c.pileup(cont, regs, sec))
            pu_st = c.stats(); pu_dev.append(pu_st["ms_total"]); pu_wall.append(w)
            reads = c.last_pileup_reads
            (text, _), w = timed(lambda: c.decompress_sam(cont, sec, regions=regs, header=False))
            sam_st = c.stats(); sam_dev.append(sam_st["ms_total"]); sam_wall.append(w)
            if k == 0 and size == 1_000:
                want = P.pileup(P.sam_reads(text, g.names), up, g.names, regs)
                assert np.array_equal(got[0], want[0]), "pileup != restatement over the SAM lines"
        med = lambda v: round(statistics.median(v[1:]), 3)        # noqa: E731
        rows.append(dict(region_bases=size, where=where, start=regs[0][1], end=regs[0][2], reads_counted=reads,
                         k2_blocks=pu_st["n_blocks"], k2_reads=pu_st["n_reads"],
                         pileup_ms_device=med(pu_dev), pileup_ms_wall=med(pu_wall), pileup_split_ms=split(pu_st),
                         pileup_bytes=int(got[0].nbytes),
                         sam_ms_device=med(sam_dev), sam_ms_wall=med(sam_wall), sam_split_ms=split(sam_st), sam_bytes=len(text)))
        print(json.dumps(rows[-1]), flush=True)
    res = dict(card=card(), config=a.config, n_reads=b.n_reads, container_bytes=len(cont), section_bytes=len(sec), reps=a.reps,
               note="after_k2: ms_reconstruct (K3 when it ran, then K8 or K6, and the host round trip that reads the totals)",
               cases=rows)
    c.close()
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(f"card: {res['card']}")


if __name__ == "__main__":
    main()
