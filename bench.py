#!/usr/bin/env python
"""bench.py -- compress + decompress throughput of the aligned-read coding path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 1..5] [--impl b200|reference] [--replicas]
                    [--dump-outputs DIR]

A step is one pass of the hot path over one batch of synthetic reads: compress the batch (K1 edit
extraction -> K2 block coder -> container index), then decompress it (K2 block decoder -> K3 read
reconstruction). `value` times the step with the batch already resident in HBM (CUDA events on the
library's own stream); `e2e` times the same step through the host-buffer C-ABI calls (cbcg_encode /
cbcg_decode) with pinned host buffers, host<->device copies inside the timed region.

Workloads are the five named shapes of BASELINE.json (`--config`, SURVEY.md 8d):
  N = 1 defaults to config 2 (150 bp reads at 30x over a 15.07 Mbp chromosome, 0.5 % substitutions);
  N = 2, 4 default to config 3 (64 Mbp, 12.8 M reads) and N = 8 to a config-4-shaped input (24 records, scaled
  to what one box generates in a minute: `--scale`, stated in config.workload). For N > 1 (torchrun) the
  ONE position-sorted input is cut into N contiguous region shards (cbc_b200.shard.shard_ranges), every rank
  generates and codes only its shard (no collective on the coding path), the ranks all-gather their block
  tables over NCCL for the container index, write one "CBCS" file with a pwrite each, and every rank decodes
  its neighbour's shard from that file (outside the timed region): the concatenation of the shards is the input.
  `--replicas` keeps round 1's N > 1 workload (one config-2-sized region per rank).

--impl reference: the UNMODIFIED reference encoder/decoder (oracle/_ref/cbc_ref, built from
/root/reference by oracle/Makefile) on the host CPU, one thread (it has no threading), on the same
configuration (all of configs 1, 2, 5; the first 3 M reads of configs 3 and 4), start-up reported apart.
"""
import argparse
import hashlib
import json
import os
import re
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

from cbc_b200 import synth                                    # noqa: E402

METRIC = "compress+decompress round-trip reads/s"
UNIT = "reads/s"
REF_SAMPLE_READS = 3_100_000          # the reference arm's step on configs 3 / 4: a config-2-sized prefix
CFG_TEXT = {
    1: "config1: 1 M x 100 bp reads over 15.07 Mbp, 0.5 % substitutions, 0.1 % indels",
    2: "config2: 150 bp reads at 30x over 15.07 Mbp, 0.5 % substitutions",
    3: "config3: 64 Mbp reference, 150 bp reads at 30x (12.8 M reads), 0.5 % substitutions",
    4: "config4: GRCh38-shaped reference in 24 records, 150 bp reads (~600 M at scale 1), 0.5 % substitutions",
    5: "config5: 50-250 bp reads at 30x over 15.07 Mbp, 2 % indels, soft clips, 0.5 % substitutions",
}
DEFAULT_SCALE = {1: 1.0, 2: 1.0, 3: 1.0, 4: 0.1, 5: 1.0}
# --dump-outputs: elements kept per array (float32, 4 bytes each: 56 MB for both at most). Config 2's container
# (5 054 923 bytes) is written whole; its decoded text (3 014 484 lines of 150 bases + newline, 455 MB) is sampled.
DUMP_CAP = {"container": 6_000_000, "decoded": 8_000_000}
DUMP_SEED = 20240601


def dump_outputs(outdir: str, outputs: dict):
    """Writes each uint8 array of `outputs` as <outdir>/<name>.npy in float32 (every byte value is exact there): whole when
    it has at most DUMP_CAP[name] elements, else the elements at DUMP_CAP[name] distinct positions drawn with DUMP_SEED, in
    ascending order, the same positions for the same length in every run. <outdir>/lengths.npy holds the full lengths, in
    the order of `outputs`."""
    os.makedirs(outdir, exist_ok=True)
    for name, arr in outputs.items():
        if arr.size > DUMP_CAP[name]:
            arr = arr[np.sort(np.random.default_rng(DUMP_SEED).choice(arr.size, DUMP_CAP[name], replace=False))]
        np.save(os.path.join(outdir, name + ".npy"), arr.astype(np.float32))
    np.save(os.path.join(outdir, "lengths.npy"), np.array([a.size for a in outputs.values()], np.float64))


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def pick_config(args, world: int) -> int:
    if args.config:
        return args.config
    if args.replicas or world == 1:
        return 2
    return 4 if world >= 8 else 3


def read_len_header(cfg) -> int:
    """What get_read_length returns: the common length, or the longest read with -l (src/sam_file_allocation.c:26-79)."""
    return cfg.len_max


def workload(args, rank: int, world: int):
    """(cfg, genome, this rank's shard, (r0, r1), text)."""
    from cbc_b200 import shard
    c = pick_config(args, world)
    scale = args.scale if args.scale else DEFAULT_SCALE[c]
    cfg = synth.SynthConfig.named(f"config{c}", scale=scale)
    if args.replicas and world > 1:
        cfg.seed += 1000 * rank                               # round 1: every rank its own region of a larger genome
        g = synth.make_genome(cfg)
        return c, cfg, g, synth.make_reads(cfg, g), (0, cfg.n_reads), CFG_TEXT[c] + f" (scale {scale:g}), one such region per GPU (replicas)"
    g = synth.make_genome(cfg)
    r0, r1 = shard.shard_ranges(cfg.n_reads, world)[rank]
    b = synth.make_reads(cfg, g, r0, r1)
    text = CFG_TEXT[c] + f" (scale {scale:g}: {cfg.n_reads} reads, {cfg.genome_len} bp)"
    if world > 1:
        text += f", ONE position-sorted input cut into {world} region shards"
    return c, cfg, g, b, (r0, r1), text


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,"
         "utilization.gpu")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, busy, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
                busy.append(float(f[9]) if len(f) > 9 else 100.0)
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        loaded = [c for c, u in zip(sm, busy) if u >= 10.0] or sm       # samples taken while the GPU was working
        return {"sm_mhz": float(np.median(loaded)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm),
                "samples_under_load": len(loaded) if len(loaded) != len(sm) or busy and min(busy) >= 10.0 else 0}


# ---------------------------------------------------------------------------------------------- CPU reference

def cpu_reference_once(sample, genome, workdir, write_inputs=True, var_length=False):
    """One encode + decode of `sample` by oracle/_ref/cbc_ref. Returns (enc_s, dec_s, stream bytes, stream, wall_s)."""
    import oracle_lib as O
    fa, sam = os.path.join(workdir, "r.fa"), os.path.join(workdir, "r.sam")
    if write_inputs:
        synth.write_fasta(fa, genome)
        synth.write_sam(sam, sample, genome)
    t0 = time.perf_counter()
    stream, _, enc_s = O.run_reference(sam, fa, workdir, var_length=var_length)
    decoded, dec_s = O.run_reference_decode(os.path.join(workdir, "ref.cbc"), fa, workdir)
    wall = time.perf_counter() - t0
    if decoded != sample.seq_lines():
        raise RuntimeError("reference decoder output != input SEQ")
    return enc_s, dec_s, len(stream), stream, wall


def cpu_port_once(sample, genome, L):
    """Fallback when oracle/_ref is absent: the plain-C restatement (single stream)."""
    import oracle_lib as O
    t0 = time.perf_counter()
    stream, _ = O.encode_legacy(sample, genome, L)
    t1 = time.perf_counter()
    decoded, _ = O.decode_legacy(stream, genome)
    t2 = time.perf_counter()
    if decoded != sample.seq_lines():
        raise RuntimeError("oracle decode != input SEQ")
    return t1 - t0, t2 - t1, len(stream), stream, t2 - t0


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def reference_workload(args, world):
    """The reference arm's input: the B200 arm's configuration, whole where a step stays around ten seconds
    (configs 1, 2), else its first REF_SAMPLE_READS reads. Config 5: the reference's decoder cannot decode
    variable-length reads at all (SURVEY.md 8c B1), so its arm runs the equal-length variant (150 bp, same indel and
    clip rates), as SURVEY.md 8d prescribes."""
    c = pick_config(args, world)
    scale = args.scale if args.scale else DEFAULT_SCALE[c]
    cfg = synth.SynthConfig.named(f"config{c}", scale=scale)
    note = ""
    if c == 5:
        cfg.len_min = cfg.len_max = 150
        note = "; equal-length variant (150 bp): the reference decoder cannot decode variable-length reads"
    g = synth.make_genome(cfg)
    n = cfg.n_reads if c in (1, 2) else min(cfg.n_reads, REF_SAMPLE_READS)
    b = synth.make_reads(cfg, g, 0, n)
    whole = n == cfg.n_reads
    text = CFG_TEXT[c] + f" (scale {scale:g})" + note
    sample = ("all %d reads" % n) if whole else ("first %d of %d reads" % (n, cfg.n_reads))
    return c, cfg, g, b, text, sample, whole


def reference_startup(genome, cfg, workdir):
    """The reference's fixed cost per run (model allocation, FASTA load: BASELINE.md), measured on a 1 000-read input."""
    d = os.path.join(workdir, "startup")
    os.makedirs(d, exist_ok=True)
    tiny = synth.make_reads(cfg, genome, 0, 1000)
    e, dd, _, _, _ = cpu_reference_once(tiny, genome, d)
    return e, dd


def run_reference_arm(args):
    import oracle_lib as O
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    c, cfg, g, b, text, sample_text, whole = reference_workload(args, world)
    n = b.n_reads
    L = read_len_header(cfg)
    kind = "reference" if O.have_reference() else "port"
    times = []
    startup = None
    with tempfile.TemporaryDirectory() as d:
        first = True
        for _ in range(args.warmup + args.steps):
            if kind == "reference":
                e, dd, sz, _, _ = cpu_reference_once(b, g, d, write_inputs=first)
            else:
                e, dd, sz, _, _ = cpu_port_once(b, g, L)
            first = False
            times.append((e, dd))
        if kind == "reference":
            startup = reference_startup(g, cfg, d)
    timed = times[args.warmup:] or times
    enc_s = float(np.mean([e for e, _ in timed])); dec_s = float(np.mean([dd for _, dd in timed]))
    step_s = enc_s + dec_s
    value = n / step_s
    desc = (f"{sample_text} of the workload through oracle/_ref/cbc_ref -c 1 / -x (program's own clock() lines: SAM parsing, FASTA "
            f"loading and coding)" if kind == "reference" else f"{sample_text} through the C restatement oracle/cbc_oracle.c")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": text, "n_reads_per_step": n, "read_len": L, "whole_workload": whole},
        "compress_reads_per_s": n / enc_s, "decompress_reads_per_s": n / dec_s,
        "bits_per_base": 8.0 * sz / b.total_bases(),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": kind, "sample": desc, "cpu": cpu_model(),
                         "host_cores": os.cpu_count()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if startup:
        se, sd = startup
        line["startup_s"] = {"compress": se, "decompress": sd,
                             "note": "the same binary on a 1 000-read input: model allocation and FASTA load, inside the program's clock() window"}
        me, md = max(enc_s - se, 1e-9), max(dec_s - sd, 1e-9)
        line["marginal"] = {"compress_reads_per_s": n / me, "decompress_reads_per_s": n / md, "round_trip_reads_per_s": n / (me + md)}
    emit(json.dumps(line))


# ---------------------------------------------------------------------------------------------- CLI leg

def cli_leg(sample, genome, L, var_length, workdir):
    """File to file: `cbc -c/-d` (this repo's C host + GPU) beside `cbc_ref -c 1/-x` on the same SAM / FASTA files."""
    import oracle_lib as O
    cbc = os.path.join(ROOT, "cbc_b200", "_build", "cbc")
    if not os.access(cbc, os.X_OK):
        return {"unavailable": "cbc_b200/_build/cbc not built"}
    fa, sam = os.path.join(workdir, "cli.fa"), os.path.join(workdir, "cli.sam")
    synth.write_fasta(fa, genome)
    synth.write_sam(sam, sample, genome)
    sam_bytes = os.path.getsize(sam)
    out, txt = os.path.join(workdir, "cli.cbcb"), os.path.join(workdir, "cli.txt")
    res = {"sam_bytes": sam_bytes, "reads": sample.n_reads}

    def run(cmd):
        t0 = time.perf_counter()
        p = subprocess.run(cmd, capture_output=True, text=True, cwd=workdir)
        return time.perf_counter() - t0, p

    best_c, best_d, own_c, own_d, ingest = None, None, None, None, None
    for _ in range(3):                                        # first run pays the page cache and CUDA context
        wc, p = run([cbc, "-c"] + (["-l"] if var_length else []) + [sam, out, fa])
        if p.returncode:
            return {"error": f"cbc -c failed: {p.stderr[-300:]}"}
        m = re.search(r"Compression took ([0-9.]+)", p.stdout); mi = re.search(r"ingest ([0-9.]+) s", p.stdout)
        wd, q = run([cbc, "-d", out, txt, fa])
        if q.returncode:
            return {"error": f"cbc -d failed: {q.stderr[-300:]}"}
        md = re.search(r"Decompression took ([0-9.]+)", q.stdout)
        if best_c is None or wc < best_c:
            best_c, own_c, ingest = wc, float(m.group(1)) if m else None, float(mi.group(1)) if mi else None
        if best_d is None or wd < best_d:
            best_d, own_d = wd, float(md.group(1)) if md else None
    with open(txt, "rb") as f:
        if f.read() != sample.seq_lines():
            return {"error": "cbc -d output != input SEQ"}
    res.update({"compress_s": best_c, "decompress_s": best_d, "compress_own_line_s": own_c, "decompress_own_line_s": own_d,
                "container_bytes": os.path.getsize(out), "ingest_s": ingest,
                "ingest_gbs": (sam_bytes / ingest / 1e9) if ingest else None,
                "compress_reads_per_s": sample.n_reads / best_c, "decompress_reads_per_s": sample.n_reads / best_d,
                "note": "wall time of the whole process (CUDA context creation, FASTA + SAM ingest, coding, file write), best of 3"})
    if O.have_reference() and not var_length:               # the reference cannot decode variable-length reads (SURVEY.md 8c B1)
        t0 = time.perf_counter()
        _, _, enc_s = O.run_reference(sam, fa, workdir, var_length=var_length)
        t1 = time.perf_counter()
        dec, dec_s = O.run_reference_decode(os.path.join(workdir, "ref.cbc"), fa, workdir)
        t2 = time.perf_counter()
        res["reference"] = {"compress_s": t1 - t0, "decompress_s": t2 - t1, "compress_own_line_s": enc_s, "decompress_own_line_s": dec_s,
                            "decoded_ok": bool(dec == sample.seq_lines())}
        res["speedup_wall"] = {"compress": (t1 - t0) / best_c, "decompress": (t2 - t1) / best_d}
    return res


# ---------------------------------------------------------------------------------------------- B200 arm

def auto_in_flight(n_reads: int) -> int:
    """Batches kept in flight per GPU when the command line does not say: two, and more for batches that fill only part
    of the device (config 1's 1 M reads occupy a third of the resident warp slots: 19.9 / 13.0 / 8.5 ms per batch at
    1 / 2 / 4 in flight, tools/inflight_probe.py; config 2: 12.1 / 11.0 / 10.5)."""
    return 2 if n_reads >= 2_000_000 else 3 if n_reads >= 1_200_000 else 4


def k2_issue_profile():
    """Per-launch figures of the block coder from the committed ncu capture (profiles/k2_issue.json, written by
    tools/ncu_summary.py from the `--set full` report of this command)."""
    path = os.path.join(ROOT, "profiles", "k2_issue.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return None


def run_b200_arm(args):
    import torch
    from cbc_b200.codec import Codec, CompactBatch, pin_batch, pinned_empty
    from cbc_b200 import shard

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # NCCL's version banner goes to stdout otherwise: stdout is the JSON line
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: there is no CPU implementation of this path")
    dev = torch.device("cuda", local)

    cnum, cfg, g, b, (r0, r1), wl_text = workload(args, rank, world)
    L = read_len_header(cfg)
    R = args.block_reads
    G = args.gen_mode
    codec = Codec(local)
    codec.set_reference(g)
    pb = pin_batch(b)
    n = b.n_reads
    bases = b.total_bases()
    input_text = b.seq_lines()

    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def max_over_ranks(x: float) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: float) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---------------- device-resident step (value)
    codec.upload(pb)
    stage = {k: [] for k in ("k1", "plan", "k2e", "gather", "k2d", "k3", "enc_total", "dec_total")}
    launches = 0
    index_bytes = 0
    block_reads_used = R
    layout = None

    def resident_step(record: bool, c=None, gather: bool = True):
        nonlocal launches, index_bytes, block_reads_used, layout
        c = c or codec
        c.encode_resident(L, R, G, args.substreams)
        se = c.stats()
        head, payload = c.fetch_index()
        if dist is not None and gather:                       # container index: all-gather of per-shard block tables
            layout = shard.gather_index(head, payload, dist, dev)
        c.decode_resident()
        sd = c.stats()
        if record:
            stage["k1"].append(se["ms_k1"]); stage["plan"].append(se["ms_plan"]); stage["k2e"].append(se["ms_code"])
            stage["gather"].append(se["ms_gather"]); stage["enc_total"].append(se["ms_total"])
            stage["k2d"].append(sd["ms_code"]); stage["k3"].append(sd["ms_k3"]); stage["dec_total"].append(sd["ms_total"])
        if c is codec:
            index_bytes = len(head)
            block_reads_used = int.from_bytes(head[32:36], "little")
        return se, sd

    # nvidia-smi needs ~0.1 s to come up and the timed region of the resident leg is ~0.1 s long: the sampler starts
    # before the warm-up steps (the same work) and runs until the end of the e2e leg, 20 ms apart
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(args.warmup):
        resident_step(False)
    barrier()
    # (1) ONE batch at a time: the library's own stage times (stage_ms, the roofline entries) and the round trip of a batch
    # that has the device to itself
    codec.mark(0)
    for _ in range(args.steps):
        se, sd = resident_step(True)
    codec.mark(1)
    single_ms = max_over_ranks(codec.elapsed_ms(0, 1)) / args.steps
    barrier()
    total_reads = sum_over_ranks(float(n))
    # (2) `--batches-in-flight` batches at once (the line's `value`): a context, a host thread and a set of streams per
    # batch, every context holding its own copy of the batch in HBM. The narrow early generations and the snapshot merges
    # of one batch (4 ... 700 of 2 960 resident warps) run in the slots the other batch's work leaves free. A step is one
    # round trip of EVERY batch in flight; timed with CUDA events recorded on an idle device at both ends.
    import threading
    KB = args.batches_in_flight if args.batches_in_flight > 0 else auto_in_flight(n)
    res_codecs = [codec]
    for _ in range(KB - 1):
        c2 = Codec(local)
        c2.set_reference(g)
        c2.upload(pb)
        res_codecs.append(c2)
    flight_stats = [None] * KB

    def flight(k, steps):
        for _ in range(steps):
            flight_stats[k] = resident_step(False, res_codecs[k], gather=(k == 0))

    def in_flight(steps):
        th = [threading.Thread(target=flight, args=(k, steps)) for k in range(1, KB)]
        for t in th:
            t.start()
        flight(0, steps)                                      # the main thread carries batch 0 (and the index all-gather at N > 1)
        for t in th:
            t.join()

    in_flight(max(1, min(args.warmup, 3)))
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    t0 = time.perf_counter()
    in_flight(args.steps)
    torch.cuda.synchronize(dev)
    ev1.record()
    torch.cuda.synchronize(dev)
    dev_ms = ev0.elapsed_time(ev1)
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    if args.dump_outputs and rank == 0:                       # batch 0's last timed round trip, before anything below codes it again
        dump_outputs(args.dump_outputs, {"container": codec.fetch_container(), "decoded": codec.fetch_decoded()})
    step_ms = max_over_ranks(dev_ms) / args.steps
    value = KB * total_reads / (step_ms * 1e-3)
    for k in range(KB):
        launches += args.steps * (flight_stats[k][0]["kernel_launches"] + flight_stats[k][1]["kernel_launches"])
    if any(fs[0]["container_bytes"] != se["container_bytes"] for fs in flight_stats):
        raise RuntimeError("contexts in flight produced different containers for the same batch")
    for c2 in res_codecs[1:]:
        if c2.fetch_decoded().tobytes() != input_text:
            raise RuntimeError("round trip mismatch in a second in-flight context")
        c2.close()
    container_bytes = se["container_bytes"]
    n_edits = se["n_edits"]

    # correctness of what was timed (every rank, outside the timed region): one more step with the decoder's output
    # buffers poisoned first -- they are the buffers K1 filled during the encode, so an idle decoder would otherwise
    # still hand K3 the right records -- then decoded text == input SEQ
    os.environ["CBCG_POISON_DECODE"] = "1"
    resident_step(False)
    del os.environ["CBCG_POISON_DECODE"]
    text = codec.fetch_decoded()
    if text.tobytes() != input_text:
        raise RuntimeError("round trip mismatch: decoded reads != input SEQ")
    if codec.stats()["n_reads"] != n:
        raise RuntimeError("decoder returned a different read count")

    # one sharded file for the whole job, every rank decodes its neighbour's shard from it
    sharded = None
    if dist is not None:
        cont = codec.fetch_container().tobytes()
        path = os.path.join(tempfile.gettempdir(), f"cbc_bench_{os.environ.get('MASTER_PORT', '0')}.cbcs")
        if rank == 0 and os.path.exists(path):
            os.unlink(path)
        barrier()
        shard.write_shard(path, rank, layout, cont)
        digest = torch.tensor(list(hashlib.sha256(input_text).digest()), dtype=torch.uint8, device=dev)
        digests = torch.empty(32 * world, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(digests, digest)
        barrier()
        with open(path, "rb") as f:
            data = f.read()
        shards = shard.read_shards(data)
        nb_rank = (rank + 1) % world
        txt, nr = codec.decompress(shards[nb_rank])
        want = bytes(digests.view(world, 32)[nb_rank].cpu().tolist())
        ok = hashlib.sha256(txt).digest() == want
        ok_all = sum_over_ranks(1.0 if ok else 0.0) == world
        if not ok_all:
            raise RuntimeError("sharded file: a shard does not decode to its region of the input")
        sharded = {"file_bytes": len(data), "shards": world, "every_shard_decoded_by_its_neighbour": True,
                   "layout": "CBCS: super-header + one self-contained CBCB container per region, written with one pwrite per rank"}
        barrier()
        if rank == 0:
            os.unlink(path)
        codec.upload(pb)                                      # the decode above replaced the resident state
        codec.encode_resident(L, R, G, args.substreams)

    # K1 alone, for its roofline entry: in the timed steps above the tail of K1 runs on a side stream beside the early
    # generations of the block coder (api.cu, encode_resident_overlapped), which stretches its own launch time;
    # CBCG_NO_OVERLAP=1 is the one-stream order (same container). Outside the timed region.
    os.environ["CBCG_NO_OVERLAP"] = "1"
    k1_alone = []
    for _ in range(3):
        codec.encode_resident(L, R, G, args.substreams)
        k1_alone.append(codec.stats()["ms_k1"])
    del os.environ["CBCG_NO_OVERLAP"]
    if codec.stats()["container_bytes"] != container_bytes:
        raise RuntimeError("one-stream and overlapped resident encodes disagree")

    # ---------------- end-to-end step through the host-buffer C ABI (e2e): pinned host buffers in, pinned host buffers
    # out, every copy inside the timed region. `--inflight` batches go through at once, a context, a host thread and a
    # set of CUDA streams each (the ABI's threading model): the text of batch k is on the PCIe link while batch k+1 is
    # being decoded, which is how a streaming caller keeps both busy. Every context codes the WHOLE batch from the same
    # pinned input into its own pinned output buffers; a step is one round trip of every batch in flight.
    K = args.inflight if args.inflight > 0 else auto_in_flight(n)
    codecs = [codec] + [Codec(local) for _ in range(K - 1)]
    for c2 in codecs[1:]:
        c2.set_reference(g)
    subs = [pb for _ in range(K)]
    # what crosses the link: the compact form of the batch (2 bits per base, text lengths, chromosome runs: cbcg_batch_compact),
    # packed by the host C code (cbch_pack_batch, what the SAM ingest hands over) into pinned memory before the timed region
    compact0 = CompactBatch(pb) if args.e2e_input == "compact" else None
    compacts = [compact0] * K if compact0 is not None else None
    outs_c = [pinned_empty(int(container_bytes * 1.5) + 65536, np.uint8) for _ in range(K)]
    outs_t = [pinned_empty(pb.total_bases() + pb.n_reads + 64, np.uint8) for _ in range(K)]

    def e2e_one(k):
        c2 = codecs[k]
        t_a = time.perf_counter()
        nc = (c2.compress_compact_into(compacts[k], L, R, outs_c[k], G, args.substreams) if compacts
              else c2.compress_into(subs[k], L, R, outs_c[k], G, args.substreams))
        t_b = time.perf_counter()
        s1 = c2.stats()
        head, payload = c2.fetch_index()
        t_c = time.perf_counter()
        nt, nr = c2.decompress_into(outs_c[k][:nc], outs_t[k])
        t_d = time.perf_counter()
        s2 = c2.stats()
        s1["wall_ms"] = (t_b - t_a) * 1e3; s2["wall_ms"] = (t_d - t_c) * 1e3
        return nc, nt, s1, s2, head, payload

    e2e_res = [None] * K

    def e2e_loop(k, steps):                                   # free-running: the batches drift apart, so that one's copies meet the other's kernels
        for _ in range(steps):
            r_ = e2e_one(k)
            if k == 0 and dist is not None:                   # container index across ranks
                shard.gather_index(r_[4], r_[5], dist, dev)
            e2e_res[k] = r_

    def e2e_run(steps):
        th = [threading.Thread(target=e2e_loop, args=(k, steps)) for k in range(1, K)]
        for t in th:
            t.start()
        e2e_loop(0, steps)
        for t in th:
            t.join()
        return list(e2e_res)

    e2e_run(max(1, min(args.warmup, 2)))
    barrier()
    t0 = time.perf_counter()
    res = e2e_run(args.steps)
    barrier()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / args.steps
    clocks = sampler.stop()
    for k in range(K):
        if outs_t[k][:res[k][1]].tobytes() != input_text:
            raise RuntimeError("e2e round trip mismatch")
    e2e_container = res[0][0]
    e2e = {"value": K * total_reads / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms, "batches_in_flight": K,
           "ms_per_batch": e2e_ms / K,
           "h2d_bytes_per_step": int(sum(r_[2]["h2d_bytes"] + r_[3]["h2d_bytes"] for r_ in res)),
           "d2h_bytes_per_step": int(sum(r_[2]["d2h_bytes"] + r_[3]["d2h_bytes"] for r_ in res)),
           "contexts_in_flight": K, "container_bytes": int(e2e_container), "input_form": args.e2e_input,
           "bits_per_base": 8.0 * e2e_container / bases,
           "note": "bytes per step are summed over the batches in flight; compress_ms / decompress_ms are per call, stretched by the overlap when more than one batch is in flight",
           "compress_ms": float(np.mean([r_[2]["ms_total"] for r_ in res])), "decompress_ms": float(np.mean([r_[3]["ms_total"] for r_ in res])),
           "compress_call_wall_ms": float(np.mean([r_[2]["wall_ms"] for r_ in res])), "decompress_call_wall_ms": float(np.mean([r_[3]["wall_ms"] for r_ in res]))}
    s1 = {"h2d_bytes": res[0][2]["h2d_bytes"]}
    for c2 in codecs[1:]:
        c2.close()

    # ---------------- roofline (SURVEY.md 8d figures, DESIGN.md "Measurement")
    peak, peak_src = peaks()
    cov = cfg.n_reads * (bases / max(n, 1)) / max(cfg.genome_len, 1)
    Lm = bases / max(n, 1)
    C_ = float(b.cigar_off[-1]) / n
    D_ = float(b.md_off[-1]) / n
    E_ = n_edits / n
    k1_bytes = (Lm + C_ + D_ + 24 + Lm / cov + 12 + 4 * E_) * n
    k3_bytes = (12 + 4 * E_ + Lm / cov + (Lm + 1)) * n
    syms = se["n_symbols"]
    k2_bytes = 4.0 * syms + se["payload_bytes"]
    med = {k: float(np.median(v)) for k, v in stage.items()}
    med["k1_alone"] = float(np.median(k1_alone))

    tr = {}
    tr_path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tr_path):
        with open(tr_path) as f:
            tr = json.load(f)
    tr_reads = float(tr.get("_reads_per_launch", 3014484))

    def traffic(name):
        if name not in tr:
            return None
        return float(tr[name]) * n / tr_reads                 # captured per launch on config 2 (one GPU), scaled by reads

    def roof(name, alg_bytes, ms):
        a = alg_bytes / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
        return {"kernel": name, "bound": "hbm", "achieved": a, "peak": peak, "unit": "GB/s", "frac": a / peak,
                "traffic": traffic(name), "ms": ms, "algorithmic_bytes": alg_bytes}

    sm_mhz = clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965.0
    issue_peak = 148 * 4 * sm_mhz * 1e6 / 1e9                 # warp instructions per second the 592 schedulers can issue (G/s)
    kp = k2_issue_profile() or {}

    def issue(name, key, ms):
        e = kp.get(key)
        ent = {"kernel": name, "bound": "issue", "unit": "G warp-instructions/s", "peak": issue_peak, "ms": ms,
               "symbols_per_s": syms / (ms * 1e-3) if ms > 0 else None, "traffic": traffic(name), "algorithmic_bytes": k2_bytes,
               "note": "serial integer work per block: bounded by instruction issue and dependent latency, not by HBM"}
        if e:                                                 # per-symbol figures of the committed ncu capture, applied to this run's symbol count and time
            inst = float(e["warp_inst_per_symbol"]) * syms
            ent.update({"achieved": inst / (ms * 1e-3) / 1e9 if ms > 0 else 0.0, "warp_inst_per_symbol": e["warp_inst_per_symbol"],
                        "issue_slot_util_ncu_pct": e.get("issue_active_pct"), "source": e.get("source")})
            ent["frac"] = ent["achieved"] / issue_peak
        else:
            ent.update({"achieved": None, "frac": None})
        return ent

    kernels = [roof("k1_extract_kernel", k1_bytes, med["k1_alone"]), issue("k2 block coder (encode)", "encode", med["k2e"]),
               issue("k2 block coder (decode)", "decode", med["k2d"]), roof("k3_reconstruct_kernel", k3_bytes, med["k3"])]
    dominant = max(kernels, key=lambda k: k["ms"])
    hbm_dom = max((k for k in kernels if k["bound"] == "hbm"), key=lambda k: k["ms"])
    roofline = {k: hbm_dom[k] for k in ("bound", "achieved", "peak", "unit", "frac", "traffic")}
    roofline.update({"kernel": hbm_dom["kernel"], "peak_source": peak_src, "longest_kernel": dominant["kernel"],
                     "note": "the HBM-bound kernels are K1 / K3 (this entry: the longer of the two); the block coder is serial integer work "
                             "per block, reported on its own bound (instruction issue) in roofline_kernels"})

    # ---------------- CPU baseline, blocking overhead, CLI leg (rank 0; bounded)
    cpu_baseline, overhead, cli = None, None, None
    if rank == 0 and not args.no_cpu:
        import oracle_lib as O
        var_length = cfg.len_min != cfg.len_max
        if world == 1:
            ns = min(500_000, n)
            sample = b.slice(0, ns)
            with tempfile.TemporaryDirectory() as d:
                if O.have_reference() and not var_length:
                    enc_s, dec_s, sz, ref_stream, _ = cpu_reference_once(sample, g, d)
                    kind = "reference"
                    desc = f"first {ns} reads of the workload through oracle/_ref/cbc_ref -c 1 / -x, program's own clock() lines"
                else:
                    enc_s, dec_s, sz, ref_stream, _ = cpu_port_once(sample, g, L)
                    kind = "port"
                    desc = f"first {ns} reads of the workload through oracle/cbc_oracle.c" + (" (the reference cannot decode variable-length reads)" if var_length else "")
            cpu_baseline = {"value": ns / (enc_s + dec_s), "unit": UNIT, "cores": 1, "kind": kind, "sample": desc,
                            "compress_reads_per_s": ns / enc_s, "decompress_reads_per_s": ns / dec_s,
                            "bits_per_base": 8.0 * sz / sample.total_bases(), "cpu": cpu_model(), "host_cores": os.cpu_count()}
            # single-block mode on the sample must be the reference's bytes (parity definition 2, at scale)
            single = codec.compress(sample, L, 0)
            identical = bool(single == ref_stream)
        else:
            ns, single, identical = 0, b"", None
        # blocking overhead of THIS configuration: this rank's blocked container against the reference's single stream over
        # the same reads, whose size comes from the CPU restatement (pinned byte for byte to cbc_ref; outside any timed region)
        full_single, _ = O.encode_legacy(b, g, L)
        overhead = {"single_stream_bytes": len(full_single), "blocked_bytes": int(container_bytes),
                    "single_bits_per_base": 8.0 * len(full_single) / bases,
                    "blocked_bits_per_base": 8.0 * container_bytes / bases,
                    "overhead_pct": 100.0 * (container_bytes - len(full_single)) / len(full_single),
                    "within_1pct_budget": bool(container_bytes <= 1.01 * len(full_single)),
                    "scope": "the whole workload" if world == 1 else f"rank 0's region shard ({n} reads)",
                    "sample_reads": ns, "sample_single_stream_bytes": len(single),
                    "single_stream_byte_identical_to_reference": identical}
        if world == 1 and not args.no_cli:
            with tempfile.TemporaryDirectory() as d:
                cli = cli_leg(b, g, L, var_length, d)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": wl_text, "named_config": cnum, "n_reads_per_gpu": n, "n_reads_total": int(total_reads), "read_len": L,
                   "block_reads": block_reads_used, "block_reads_auto": R == 0xffffffff, "gen_mode": G, "substreams_per_block": args.substreams, "blocks_per_gpu": int(se["n_blocks"]),
                   "l2": "inputs larger than L2 (batch %.0f MB, decoded text %.0f MB per GPU)" % (s1["h2d_bytes"] / 1e6, (bases + n) / 1e6),
                   "parallelism": (f"{world} region shard(s) of one position-sorted input" if not args.replicas else f"{world} replicas") + ", no collective on the coding path",
                   "batches_in_flight": KB, "n_reads_per_step": int(KB * total_reads),
                   "step": f"one resident round trip (compress + decompress) of each of the {KB} batches in flight per GPU"},
        "single_batch": {"ms_per_step": single_ms, "value": total_reads / (single_ms * 1e-3), "unit": UNIT,
                         "note": "one batch at a time with the device to itself (the stage_ms below are from these steps)"},
        "compress_reads_per_s": total_reads / (max_over_ranks(med["enc_total"]) * 1e-3),
        "decompress_reads_per_s": total_reads / (max_over_ranks(med["dec_total"]) * 1e-3),
        "bits_per_base": 8.0 * container_bytes / bases,
        "blocking": overhead, "sharded_file": sharded,
        "stage_ms": med, "wall_ms_per_step": wall_ms / args.steps,
        "roofline": roofline, "roofline_kernels": kernels,
        "cpu_baseline": cpu_baseline, "e2e": e2e, "cli": cli,
        "gpu_launches": int(launches), "clocks": clocks,
        "symbols_per_s_encode": syms / (med["k2e"] * 1e-3) if med["k2e"] > 0 else None,
        "symbols_per_s_decode": syms / (med["k2d"] * 1e-3) if med["k2d"] > 0 else None,
        "index_bytes_per_gpu": index_bytes,
        "decoder_output_poisoned_before_check": True,
    }
    if rank == 0:
        emit(json.dumps(line))
    codec.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


_JSON_OUT = None


def guard_stdout():
    """stdout carries exactly one JSON line. Libraries write there behind Python's back (NCCL's version banner did, under
    torchrun, NCCL_DEBUG_FILE notwithstanding): file descriptor 1 is pointed at stderr for the rest of the process and
    the JSON line goes to a private duplicate of the original stdout."""
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line: str):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(line + "\n")
    out.flush()


def main():
    guard_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=0, choices=[0, 1, 2, 3, 4, 5],
                    help="named shape of BASELINE.json; default: 2 on one GPU, 3 on 2 / 4 GPUs, 4 (scaled) on 8")
    ap.add_argument("--replicas", action="store_true", help="N > 1: one config-2-sized region per rank (round 1's workload) instead of region shards of one input")
    ap.add_argument("--block-reads", type=int, default=0xffffffff, help="reads per block; default: CBCG_BLOCK_AUTO")
    ap.add_argument("--batches-in-flight", type=int, default=0,
                    help="resident leg: batches coded at once per GPU, a context and a host thread each (value = their joint throughput); "
                         "default: 2, more for batches that fill only part of the device (auto_in_flight)")
    ap.add_argument("--inflight", type=int, default=0, help="e2e leg: batches in flight per GPU through the host-buffer calls, a context and a host thread each (default: as --batches-in-flight)")
    ap.add_argument("--gen-mode", type=int, default=1, help="1: generation-primed blocks (default), 0: cold blocks")
    ap.add_argument("--substreams", type=int, default=0, choices=[0, 1, 4],
                    help="arithmetic-coded streams per block: 0 = the library's default (four in the narrow early generations, one in the wide ones), 1, or 4 everywhere")
    ap.add_argument("--e2e-input", default="compact", choices=["compact", "soa"],
                    help="host buffers of the e2e leg: cbcg_batch_compact (2 bits per base; default) or the plain SoA cbcg_batch")
    ap.add_argument("--scale", type=float, default=0.0, help="shrink the workload; default 1.0 (config 4: 0.1, stated in config.workload)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline / blocking-overhead / CLI legs")
    ap.add_argument("--no-cli", action="store_true", help="skip the file-to-file CLI leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the container and decoded text of the last one as DIR/<name>.npy "
                         "(float32; a seeded sample where an array is larger than DUMP_CAP; rank 0's shard when N > 1)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the B200 arm computed: it needs --impl b200")
    args.warmup = max(args.warmup, 0)
    subprocess.run(["make", "-s", "-C", ROOT, "host"], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
