"""Encoding without MD against encoding with it (DESIGN.md 5d, "Encoding without MD").

One batch of bench config 2 (or 5 with --config 5). First the check: the container of the batch without MD is the
container of the batch with its MD (the generator writes canonical MD, so the batch is its own B*). Then, alternated
--reps times:
  - cbcg_encode (host buffers: the pipelined path) with and without MD, plain and compact: stats ms_total and a wall clock
    around the call;
  - cbcg_batch_upload with and without MD: ms_h2d (K7's time is part of it) and the wall clock.
Medians are reported. K7's kernel time comes from torch.profiler with CUDA activities, in a run of its own (an upload
without MD, then a resident encode for K1's time beside it). Last, the same batch as a SAM file with its MD tags stripped
through the command line: `cbc -c` of the original file against `cbc -c -M` of the stripped one, alternated, wall clock of
the whole process, and the two outputs compared.

The card's name and power limit are read in the same run (nvidia-smi, read-only query).

    python tools/md_probe.py [--config 2|5] [--reps 5] [--out md_probe.json]
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
from cbc_b200.codec import Codec, CompactBatch                    # noqa: E402

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


def kernel_ms(c, bare, L):
    """K7 and K1 device times from torch.profiler (CUDA activities), one upload without MD and one resident encode."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    c.upload(bare)                                                 # warm-up outside the trace
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        c.upload(bare)
        c.encode_resident(L, AUTO, 1, substreams=0)
    torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        for key, name in (("k7_ms", "k7_md_kernel"), ("k1_ms", "k1_extract_kernel")):
            if name in ev.key:
                t = getattr(ev, "device_time_total", None)
                out[key] = out.get(key, 0.0) + (t if t is not None else ev.cuda_time_total) / 1e3
    return {k: round(v, 3) for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=2, choices=(2, 5))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="md_probe.json")
    a = ap.parse_args()
    cfg = synth.SynthConfig.named(f"config{a.config}")
    g = synth.make_genome(cfg)
    b = synth.make_reads(cfg, g)
    bare = b.without_md()
    L = int(b.seq_len.max())
    c = Codec(0)
    c.set_reference(g)
    cont = c.compress(b, L, block_reads=AUTO, gen_mode=1, substreams=0)
    assert c.compress(bare, L, block_reads=AUTO, gen_mode=1, substreams=0) == cont, "container without MD != container with MD"
    cb, cb_bare = CompactBatch(b), CompactBatch(bare)
    out = np.empty(len(cont) + (1 << 24), np.uint8)

    def compact(x):
        return c.compress_compact_into(x, L, AUTO, out, gen_mode=1, substreams=0)
    cont_compact = out[:compact(cb)].tobytes()                    # the pipelined compact path cuts blocks by a ramp of its own
    assert out[:compact(cb_bare)].tobytes() == cont_compact, "compact container without MD != container with MD"
    rows = {k: {"ms_total": [], "ms_h2d": [], "wall": []} for k in ("plain_md", "plain_derived", "compact_md", "compact_derived",
                                                                     "upload_md", "upload_derived")}

    def run(key, fn):
        _, w = timed(fn)
        st = c.stats()
        rows[key]["ms_total"].append(st["ms_total"]); rows[key]["ms_h2d"].append(st["ms_h2d"]); rows[key]["wall"].append(w)
    for _ in range(a.reps + 1):
        run("plain_md", lambda: c.compress(b, L, block_reads=AUTO, gen_mode=1, substreams=0))
        run("plain_derived", lambda: c.compress(bare, L, block_reads=AUTO, gen_mode=1, substreams=0))
        run("compact_md", lambda: compact(cb))
        run("compact_derived", lambda: compact(cb_bare))
        run("upload_md", lambda: c.upload(b))
        run("upload_derived", lambda: c.upload(bare))
    cb.close(); cb_bare.close()
    one = {k: {x: med(v) for x, v in r.items()} for k, r in rows.items()}
    one["md_bytes"] = int(b.md_off[-1])
    print(json.dumps(one), flush=True)
    kern = kernel_ms(c, bare, L)
    print(json.dumps(kern), flush=True)
    c.close()
    with tempfile.TemporaryDirectory() as d:
        fa, sam_in, bare_in, x, y = (os.path.join(d, n) for n in ("r.fa", "r.sam", "bare.sam", "a.cbc", "m.cbc"))
        synth.write_fasta(fa, g)
        synth.write_sam(sam_in, b, g)
        with open(sam_in, "rb") as f, open(bare_in, "wb") as o:
            for chunk in iter(lambda: f.readlines(1 << 26), []):
                o.write(re.sub(rb"\tMD:Z:[^\t\n]*", b"", b"".join(chunk)))
        flags = ["-l"] if a.config == 5 else []
        plain, derived = [], []
        for _ in range(max(2, a.reps // 2) + 1):
            plain.append(timed(lambda: subprocess.run([CLI, "-c", *flags, sam_in, x, fa], check=True, capture_output=True))[1])
            derived.append(timed(lambda: subprocess.run([CLI, "-c", "-M", *flags, bare_in, y, fa], check=True, capture_output=True))[1])
        with open(x, "rb") as f1, open(y, "rb") as f2:
            same = f1.read() == f2.read()
        cli = dict(encode_wall_ms=med(plain), encode_derive_md_wall_ms=med(derived), same_output=same,
                   sam_bytes=os.path.getsize(sam_in), stripped_sam_bytes=os.path.getsize(bare_in))
    print(json.dumps(cli), flush=True)
    res = dict(card=card(), config=a.config, n_reads=b.n_reads, bases=b.total_bases(), container_bytes=len(cont), reps=a.reps,
               one_batch=one, kernels=kern, cli=cli)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(f"card: {res['card']}")


if __name__ == "__main__":
    main()
