"""Wall-clock of the host-buffer calls (cbcg_encode / cbcg_decode, pinned buffers) with the pipelined path on and off,
on one GPU. usage: e2e_probe.py [scale] [mode ...]   mode = on | off"""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cbc_b200 import synth                      # noqa: E402
from cbc_b200.codec import Codec, pin_batch, pinned_empty     # noqa: E402

scale = float(sys.argv[1]) if len(sys.argv) > 1 else 1.0
modes = sys.argv[2:] or ["off", "on"]
cfg = synth.SynthConfig.named("config2", scale=scale)
g = synth.make_genome(cfg)
b = synth.make_reads(cfg, g)
c = Codec(0)
c.set_reference(g)
pb = pin_batch(b)
out_c = pinned_empty(max(16 << 20, b.n_reads * 4), np.uint8)
out_t = pinned_empty(b.total_bases() + b.n_reads + 64, np.uint8)
ref = b.seq_lines()
AUTO = 0xffffffff
for mode in modes:
    os.environ["CBCG_PIPE_MIN_READS"] = "1000000000000" if mode == "off" else "100000"
    te, td = [], []
    for it in range(5):
        t0 = time.perf_counter()
        nc = c.compress_into(pb, 150, AUTO, out_c, 1)
        t1 = time.perf_counter()
        nt, nr = c.decompress_into(out_c[:nc], out_t)
        t2 = time.perf_counter()
        te.append((t1 - t0) * 1e3); td.append((t2 - t1) * 1e3)
    ok = out_t[:nt].tobytes() == ref
    print(json.dumps({"pipelined": mode, "ok": ok, "container": int(nc), "enc_ms": [round(x, 2) for x in te], "dec_ms": [round(x, 2) for x in td],
                      "enc_med": round(float(np.median(te[1:])), 2), "dec_med": round(float(np.median(td[1:])), 2)}), flush=True)
