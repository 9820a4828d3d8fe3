"""SAM output against SEQ output of the same container (DESIGN.md, "SAM output").

One batch of bench config 2 (or 5 with --config 5) coded with the default settings. cbcg_decode and cbcg_decode_sam
(with the header, without a CIGAR section) are alternated --reps times; per call the device time (stats ms_total),
ms_reconstruct (K3 alone for cbcg_decode; K3 + K6 for cbcg_decode_sam), ms_k3 and ms_d2h (CUDA events), and a wall clock
around the call. Medians are reported, with the SAM bytes per read. Then the same input as a SAM file through the command
line: `cbc -d` against `cbc -d -S`, alternated, wall clock of the whole process. The SAM output is checked against the
restatement (tests/sam_restate.py) on the first 20 000 reads before anything is timed.

The card's name and power limit are read in the same run (nvidia-smi, read-only query).

    python tools/sam_probe.py [--config 2|5] [--reps 5] [--out sam_probe.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from cbc_b200 import synth                                        # noqa: E402
from cbc_b200.codec import Codec                                  # noqa: E402
import sam_restate as R                                           # noqa: E402

AUTO = 0xFFFFFFFF
CLI = os.path.join(ROOT, "cbc_b200", "_build", "cbc")


def card():
    p = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return p.stdout.strip().splitlines()[0] if p.returncode == 0 and p.stdout.strip() else "unknown"


def timed(fn):
    t = time.perf_counter()
    out = fn()
    return out, 1e3 * (time.perf_counter() - t)


def med(v):
    return round(statistics.median(v[1:]), 3)                     # the first call is a warm-up


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=2, choices=(2, 5))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="sam_probe.json")
    a = ap.parse_args()
    cfg = synth.SynthConfig.named(f"config{a.config}")
    g = synth.make_genome(cfg)
    b = synth.make_reads(cfg, g)
    L = int(b.seq_len.max())
    c = Codec(0)
    c.set_reference(g)
    cont = c.compress(b, L, block_reads=AUTO, gen_mode=1, substreams=0)
    sam, _ = c.decompress_sam(cont, header=False)
    k = 20_000
    head = sam.split(b"\n", k)[:k]
    if a.config == 2:                                              # config 2 has no indels or clips: implied == input CIGAR
        assert [x + b"\n" for x in head] == R.sam_lines(b.slice(0, k), R.upper(g), g.names)
    keys = ("ms_total", "ms_code", "ms_reconstruct", "ms_k3", "ms_d2h")
    seq_rows = {x: [] for x in keys + ("wall",)}
    sam_rows = {x: [] for x in keys + ("wall",)}
    for _ in range(a.reps + 1):
        (text, nr), w = timed(lambda: c.decompress(cont))
        st = c.stats()
        for x in keys:
            seq_rows[x].append(st[x])
        seq_rows["wall"].append(w)
        (sam, ids), w = timed(lambda: c.decompress_sam(cont))
        st = c.stats()
        for x in keys:
            sam_rows[x].append(st[x])
        sam_rows["wall"].append(w)
    c.close()
    one = dict(seq={x: med(v) for x, v in seq_rows.items()}, sam={x: med(v) for x, v in sam_rows.items()},
               seq_bytes=len(text), sam_bytes=len(sam), sam_bytes_per_read=round(len(sam) / b.n_reads, 2))
    one["k6_ms_estimate"] = round(one["sam"]["ms_reconstruct"] - one["sam"]["ms_k3"], 3)
    one["ms_reconstruct_difference"] = round(one["sam"]["ms_reconstruct"] - one["seq"]["ms_reconstruct"], 3)
    print(json.dumps(one), flush=True)
    with tempfile.TemporaryDirectory() as d:
        fa, sam_in, cbc, out = (os.path.join(d, x) for x in ("r.fa", "r.sam", "a.cbc", "o.txt"))
        synth.write_fasta(fa, g)
        synth.write_sam(sam_in, b, g)
        subprocess.run([CLI, "-c", *(["-l"] if a.config == 5 else []), sam_in, cbc, fa], check=True, capture_output=True)
        plain, withs = [], []
        for _ in range(max(2, a.reps // 2) + 1):
            plain.append(timed(lambda: subprocess.run([CLI, "-d", cbc, out, fa], check=True, capture_output=True))[1])
            withs.append(timed(lambda: subprocess.run([CLI, "-d", "-S", cbc, out, fa], check=True, capture_output=True))[1])
        cli = dict(decode_wall_ms=med(plain), decode_sam_wall_ms=med(withs), sam_file_bytes=os.path.getsize(out))
    print(json.dumps(cli), flush=True)
    res = dict(card=card(), config=a.config, n_reads=b.n_reads, container_bytes=len(cont), reps=a.reps, one_batch=one, cli=cli)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(f"card: {res['card']}")


if __name__ == "__main__":
    main()
