#!/usr/bin/env python3
"""Benchmark of the alignment hot path (BASELINE.json metric: GCUPS and reads/s, device-timed).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--reads B] [--config 2] [--impl reference] [--dump-outputs DIR]

Workload (N = 1): BASELINE config 2 — 10 kb synthetic chimeric ONT-like reads vs 20 plasmid-like
contigs of 7-9 kb, `--double-strand --circular`, local mode, default CLI scoring.  A step is one
pass of the hot path over one batch of B reads per GPU.  `value` is measured with the reads already
resident in HBM (stitch_custom_batch_device); `e2e` goes through the reference-facing call
(stitch_align_batch = Aligners::align, host buffers in, chains out, origin re-alignment included).
A cell update = one (contig-strand position, read base) pair; every DP fill is counted.

For N > 1 (torchrun, one rank per GPU) every rank aligns its own B reads (weak scaling, no
collective: reads are independent); the timed region is bracketed by barriers and the max over
ranks is taken.

--dump-outputs DIR writes the chains the last timed step of each pass returned (rank 0) as .npy files (see dump_results),
so that two builds can be compared output for output on the same seeded inputs.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from (which may be read-only)

ALG_OPS_PER_CELL = 32            # SURVEY.md section 8d: INT32 ops per cell update
ALG_BYTES_PER_CELL = 0.5         # SURVEY.md section 8d: the traceback stream, <= 0.5 B per cell update
# what the fill kernel really moves (DESIGN.md section 4, ncu profiles/): the rolling column state, one S key and one D key
# per cell, read and written once per column by every tile that is not skipped as quiet, plus checkpoints and jump records
STATE_BYTES_PER_CELL = 16.0


def read_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_baseline(kw, named, reads, truth, budget_s=30.0, max_threads=None):
    """Times the restated reference (oracle/, 16-byte cells in the reference's own matrix layout, one aligner per thread,
    as fg-stitch-cli/src/commands/align.rs:345-390 runs them) on host cores, on FULL-LENGTH reads of the workload.

    What bounds the sample is the contig axis, not the read: every thread aligns one whole read against `s` contig-strands
    (the ones it was drawn from first), s sized from a short calibration run so that the sample takes about `budget_s`
    seconds (a single strand truncated to fewer rows only when even one whole strand exceeds the budget).  The reference
    walks its (m+1) x (n+1) traceback matrix with a stride of 16 (n+1) bytes, so its cost per cell update depends on the
    read length and the host's memory system, hardly on the number of contig rows (profiles/r02_cpu_port_vs_n.json)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    from stitch_b200._abi import make_opts
    T = min(host_threads(), max_threads or 64, len(reads))
    n = max(len(r) for r in reads[:T])
    ns = len(named) * (2 if kw.get("double_strand") else 1)
    m_mean = sum(len(s) for _, s in named) / len(named)
    m_full = max(len(s) for _, s in named)
    oracle_lib.set_checker_layout(False)   # the reference's layout: this is the baseline, not a parity check
    # calibration: every thread, its read against the first 256 rows of one strand
    cal = oracle_lib.OracleAligners(make_opts(**kw), [(nm, s[:256]) for nm, s in named])
    _, ci = cal.batch(reads[:T], subsets=[[truth[r][0]] for r in range(T)], raw=False, threads=T)
    rate = max(1e5, ci["cells"] / max(ci["seconds"], 1e-3) / T)        # cell updates / s / thread
    rows = budget_s * rate / n
    try:   # 16 B x (n+1) x rows of traceback per thread (the reference's allocation)
        avail = int(next(l for l in open("/proc/meminfo") if l.startswith("MemAvailable")).split()[1]) * 1024
        rows = min(rows, avail * 0.5 / T / (16 * (n + 1)))
    except Exception:
        pass
    if rows >= m_mean:
        s_per = int(max(1, min(ns, rows // m_mean)))
        use, what = named, f"{s_per} whole contig-strand(s)"
    else:
        s_per = 1
        use, what = [(nm, s[:max(256, int(rows))]) for nm, s in named], f"the first {max(256, int(rows))} rows of one contig-strand"
    subsets = []
    for r in range(T):
        mine = list(truth[r])[:s_per]
        mine += [c for c in range(ns) if c not in mine][:s_per - len(mine)]
        subsets.append(sorted(mine))
    o = oracle_lib.OracleAligners(make_opts(**kw), use)
    _, info = o.batch(reads[:T], subsets=subsets, raw=False, threads=T)
    gcups = info["cells"] / info["seconds"] / 1e9
    return {"value": gcups, "unit": "GCUPS", "cores": T, "kind": "port",
            "sample": f"{T} full-length reads ({n} b) of the workload, one per thread, each against {what} (the ones it was drawn from first; "
                      f"same options; origin re-alignment fills included): {info['fills']} fills, {info['cells']} cells in {info['seconds']:.1f} s; "
                      f"one restated-reference aligner per thread, the reference's traceback layout (calibrated at {rate / 1e6:.1f} M cell "
                      f"updates/s/thread); the Rust reference itself cannot be built here (no cargo)",
            "seconds": info["seconds"], "cells": info["cells"]}


def cpu_sweep(kw, named, reads, truth, lengths=(300, 1000, 3000, 10000)):
    """CUPS of the restated reference against the read length (reads truncated to n, one contig-strand each)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    from stitch_b200._abi import make_opts
    out = []
    for threads in (1, min(host_threads(), 16)):
        for n in lengths:
            T = min(threads, len(reads))
            o = oracle_lib.OracleAligners(make_opts(**kw), named)
            _, info = o.batch([r[:n] for r in reads[:T]], subsets=[[truth[r][0]] for r in range(T)], raw=False, threads=T)
            out.append({"read_len": n, "threads": T, "cells": info["cells"], "seconds": info["seconds"],
                        "mcups_per_thread": info["cells"] / info["seconds"] / 1e6 / T})
    return out


def parity_check(al, kw, named, reads, truth, e2e_chains, n_check=4, pool=32):
    """After the timed region: `n_check` reads of the batch the e2e step just aligned, aligned again on the GPU restricted
    (subset_words) to the contig-strands they use plus two decoys, bit for bit against the oracle on the same subsets
    (all 40 strands would cost the oracle 51 GB per read); the subset score must equal the score of the timed e2e result."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import random
    import oracle_lib
    from stitch_b200._abi import make_opts
    ns = len(named) * (2 if kw.get("double_strand") else 1)
    rng = random.Random(1)
    pool = min(pool, len(reads))
    subsets = []
    for r in range(pool):
        a = e2e_chains[r][0]
        mine = set(truth[r]) | {a.start_contig_idx, a.end_contig_idx} | {x for k, x, _ in a.ops if k == 6}
        subsets.append(sorted(mine | set(rng.sample([c for c in range(ns) if c not in mine], 2))))
    check = sorted(range(pool), key=lambda r: (len(subsets[r]), r))[:n_check]
    got = al.align_batch([reads[r] for r in check], [subsets[r] for r in check])
    oracle_lib.set_checker_layout(True)
    try:
        exp, info = oracle_lib.OracleAligners(make_opts(**kw), named).batch([reads[r] for r in check], subsets=[subsets[r] for r in check],
                                                                            raw=False, threads=min(n_check, host_threads()))
    finally:
        oracle_lib.set_checker_layout(False)
    ok = all(len(g) == len(e) and all(x.key() == y.key() for x, y in zip(g, e)) for g, e in zip(got, exp))
    same_score = all(got[k][0].score == e2e_chains[r][0].score for k, r in enumerate(check))
    return {"reads": len(check), "ok": bool(ok and same_score), "bit_exact_vs_oracle": bool(ok), "score_equals_timed_e2e_result": bool(same_score),
            "read_indices": check, "subset_sizes": [len(subsets[r]) for r in check], "oracle_seconds": info["seconds"],
            "how": "GPU align_batch with per-read subset_words vs oracle/ on the same subsets, every field and operation of every chain"}


DUMP_BYTES = 64 << 20   # --dump-outputs: the size of all files together stays below this
CHAIN_FIELDS = ("score", "xstart", "xend", "ystart", "yend", "xlen", "ylen", "start_contig_idx", "end_contig_idx", "length")


def dump_results(lib, prefix_map, handle, out_dir, name, budget):
    """Writes the chains of a results handle (what the results accessors of `prefix_map` hand a caller, as in
    stitch_b200._lib.read_results) as float64 arrays, exact for the 32-bit fields:

        <name>_reads.npy   (r, 2)  read index, number of chains
        <name>_chains.npy  (c, 11) read index, then CHAIN_FIELDS
        <name>_ops.npy     (o, 4)  row of the chain in <name>_chains.npy, kind, a, b

    A full batch of long reads has more operations than `budget` bytes hold, so the files cover a fixed sample of the reads:
    the reads in a fixed random order (seed 0) as long as their rows fit the budget, written in read order.  Two builds that
    compute the same chains write the same files."""
    import numpy as np
    from stitch_b200._abi import StitchChain, StitchOp
    fn = {k: getattr(lib, v) for k, v in prefix_map.items()}
    n_reads = fn["n_reads"](handle)
    n_ch, n_op = C.c_uint64(), C.c_uint64()
    ch_ptr = fn["chains"](handle, C.byref(n_ch))
    op_ptr = fn["ops"](handle, C.byref(n_op))
    chains = np.ctypeslib.as_array(ch_ptr, (n_ch.value,)) if n_ch.value else np.zeros(0, np.dtype(StitchChain))
    ops = np.ctypeslib.as_array(op_ptr, (n_op.value,)) if n_op.value else np.zeros(0, np.dtype(StitchOp))
    first, count = C.c_uint64(), C.c_uint32()
    spans = []
    for r in range(n_reads):
        fn["read"](handle, r, C.byref(first), C.byref(count))
        spans.append((first.value, count.value))
    pick, used = [], 0
    for r in np.random.default_rng(0).permutation(n_reads):
        f, c = spans[r]
        cost = 8 * (2 + 11 * c + 4 * int(chains["n_ops"][f:f + c].sum()))
        if used + cost > budget:
            break
        pick.append(int(r))
        used += cost
    pick.sort()
    none = np.zeros(0, np.int64)
    rows = np.concatenate([np.arange(spans[r][0], spans[r][0] + spans[r][1]) for r in pick] + [none])
    sel = chains[rows]
    op_rows = np.concatenate([np.arange(o, o + n, dtype=np.int64) for o, n in zip(sel["ops_offset"], sel["n_ops"])] + [none])
    sel_ops = ops[op_rows]
    out = {
        "reads": np.array([(r, spans[r][1]) for r in pick], dtype=np.float64).reshape(-1, 2),
        "chains": np.column_stack([np.repeat(pick, [spans[r][1] for r in pick])] + [sel[f] for f in CHAIN_FIELDS]).astype(np.float64).reshape(-1, 11),
        "ops": np.column_stack([np.repeat(np.arange(len(sel)), sel["n_ops"]), sel_ops["kind"], sel_ops["a"], sel_ops["b"]]).astype(np.float64).reshape(-1, 4),
    }
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, f"{name}_{k}.npy"), a)
    return {"reads": len(pick), "of_reads": n_reads, "chains": len(sel), "ops": len(sel_ops)}


def via_cli(args):
    """The product's own multi-GPU path: ONE `stitch-b200 align --gpus N` process (a reader thread, one worker thread and one
    device context per GPU pulling batches from a bounded queue, formatter threads, an ordered BAM writer), timed by wall
    clock from process start to exit (context creation and file parsing included) on a synthetic FASTQ of the workload."""
    import tempfile
    from stitch_b200 import synth
    kw, named, pool = synth.config(args.config, min(args.reads, args.cli_pool), args.read_len)
    reads = [pool[k % len(pool)] for k in range(args.reads)]   # (the CLI only merges CONSECUTIVE identical reads, align.rs:364-375)
    cli = os.path.join(ROOT, "stitch_b200", "stitch-b200")
    with tempfile.TemporaryDirectory() as d:
        ref, fq, out = os.path.join(d, "ref.fa"), os.path.join(d, "reads.fq"), (os.path.join(d, "out.bam") if args.cli_out == "tmp" else args.cli_out)
        with open(ref, "wb") as f:
            for n, sq in named:
                f.write(b">" + n.encode() + b"\n" + sq + b"\n")
        with open(fq, "wb") as f:
            for k, r in enumerate(reads):
                f.write(b"@r%d\n" % k + r + b"\n+\n" + b"I" * len(r) + b"\n")
        cmd = [cli, "align", "-f", fq, "-r", ref, "--gpus", str(args.gpus), "--batch", str(args.cli_batch)]
        if kw.get("double_strand"):
            cmd.append("-d")
        if kw.get("circular"):
            cmd.append("-C")
        walls = []
        for _ in range(max(1, args.steps)):
            t0 = time.perf_counter()
            with open(out, "wb") as fo:
                p = subprocess.run(cmd, stdout=fo, stderr=subprocess.PIPE, env=dict(os.environ, STITCH_CLI_TIMING="1"))
            walls.append(time.perf_counter() - t0)
            if p.returncode != 0:
                print(json.dumps({"error": p.stderr.decode()[-500:]}))
                return 1
        size = os.path.getsize(out) if os.path.isfile(out) else None
    cells = sum(len(s) for _, s in named) * (2 if kw.get("double_strand") else 1) * sum(len(r) for r in reads)
    wall = min(walls)
    stages = None   # the CLI's own account of its last run: start-up, the span in which the devices aligned, busy time per stage
    for line in p.stderr.decode().splitlines():
        if line.startswith("stitch-b200 timing: "):
            stages = json.loads(line[len("stitch-b200 timing: "):])
    print(json.dumps({"metric": "reads/s through `stitch-b200 align` (wall clock of the whole process)", "value": len(reads) / wall, "unit": "reads/s",
                      "stages": stages,
                      "n_gpus": args.gpus, "reads": len(reads), "wall_s": wall, "walls_s": walls, "gcups_first_fills_only": cells / wall / 1e9,
                      "bam_bytes": size, "batch": args.cli_batch, "config": {"workload": f"config {args.config}", "read_len": len(reads[0])},
                      "stderr_tail": p.stderr.decode()[-200:]}))
    return 0


def workload_config(args, kw, named, world, read_len):
    """The `config` object of the JSON line: identical for both arms (the arms describe their own samples elsewhere)."""
    workload = {1: "config1: 10 kb chimeric reads vs 20 plasmids (7-9 kb), single strand, local",
                2: "config2: 10 kb chimeric reads vs 20 plasmids (7-9 kb), --double-strand --circular, local",
                3: "config3 slice: 5-20 kb reads vs 128 contigs x 2 strands (reference limit of 256 contig-strands)",
                4: "config4: 50-100 kb reads vs 50 x 20 kb contigs, --double-strand",
                6: "config2 reads vs a shared-backbone panel (every contig = 60 % common backbone + 40 % unique insert), -d -C"}[args.config]
    return {"workload": workload, "reads_per_gpu_per_step": args.reads, "read_len": read_len,
            "contig_strands": len(named) * (2 if kw.get("double_strand") else 1),
            "l2": "inputs larger than L2: the rolling state of the reads in flight (148 x 2.6 MB) is streamed by every computed "
                  "tile-column and a step touches > 100 GB of checkpoints; no flush needed",
            "parallelism": f"reads sharded over {world} GPU(s), no collective"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reads", type=int, default=1000, help="reads per GPU per step (config 1/2: 1k reads)")
    ap.add_argument("--config", type=int, default=2)
    ap.add_argument("--read-len", type=int, default=None)
    ap.add_argument("--impl", default="stitch_b200", choices=["stitch_b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity-check", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="diagnostic runs only: skip the end-to-end pass (the line is then not a bench line)")
    ap.add_argument("--cpu-budget-s", type=float, default=30.0, help="CPU seconds the cpu_baseline sample is sized for")
    ap.add_argument("--cpu-sweep", action="store_true", help="print the CPU port's CUPS against the read length and exit")
    ap.add_argument("--via-cli", action="store_true", help="time the product's own command line (stitch-b200 align --gpus N) on a FASTQ of "
                                                           "--reads reads: reader thread, one worker per GPU, ordered BAM writer")
    ap.add_argument("--cli-batch", type=int, default=256)
    ap.add_argument("--cli-pool", type=int, default=1000, help="--via-cli: distinct synthetic reads (cycled to --reads records)")
    ap.add_argument("--cli-out", default="/dev/null", help="--via-cli: where the BAM stream goes (default /dev/null: 650 KB per 10 kb read)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the chains the last timed step of each pass returned to DIR/*.npy "
                                                          f"(at most {DUMP_BYTES >> 20} MB in all, a seeded sample of the reads)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.via_cli or args.cpu_sweep or args.impl != "stitch_b200"):
        ap.error("--dump-outputs writes what the GPU passes compute: not with --via-cli, --cpu-sweep or --impl reference")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    from stitch_b200 import synth

    if args.via_cli:
        return via_cli(args)

    if args.cpu_sweep:
        truth = []
        kw, named, reads = synth.config(args.config, max(host_threads(), 1), args.read_len, truth=truth)
        print(json.dumps({"cpu_port_vs_read_len": cpu_sweep(kw, named, reads, truth), "host_threads": host_threads(),
                          "note": "restated reference (oracle/), one read per thread against one contig-strand; reads truncated to read_len"}))
        return 0

    if args.impl == "reference":
        if rank != 0:
            return 0
        truth = []
        kw, named, reads = synth.config(args.config, max(host_threads(), 1), args.read_len, truth=truth)
        n_steps = args.warmup + args.steps
        budget = max(2.0, min(30.0, 200.0 / max(1, n_steps)))   # the whole run ends within a few minutes
        vals = []
        for step in range(n_steps):
            base = cpu_baseline(kw, named, reads, truth, budget)
            if step >= args.warmup:
                vals.append(base)
        cells = sum(v["cells"] for v in vals)
        secs = sum(v["seconds"] for v in vals)
        g = cells / secs / 1e9
        base = dict(vals[-1]); base["value"] = g
        cells_per_read = sum(len(s) for _, s in named) * (2 if kw.get("double_strand") else 1) * len(reads[0])
        line = {"impl": "reference", "metric": "GCUPS", "value": g, "unit": "GCUPS", "n_gpus": args.gpus,
                "steps": len(vals), "warmup": args.warmup, "ms_per_step": secs / len(vals) * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
                "config": workload_config(args, kw, named, max(1, args.gpus), len(reads[0])),
                "note": "restated reference on host cores (the Rust reference cannot be built: no cargo/rustc); each step is a bounded "
                        "sample of the workload (see cpu_baseline.sample)",
                "reads_per_s_extrapolated": g * 1e9 / cells_per_read,
                "cpu_baseline": base,
                "e2e": {"value": g, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: stitch_b200 has no CPU path"}))
        return 1
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import stitch_b200
    from stitch_b200 import _abi, _lib
    lib = _lib.load()
    from stitch_b200 import sharding
    all_truth = []
    kw, named, all_reads = synth.config(args.config, args.reads * world, args.read_len, truth=all_truth)
    lo, hi = sharding.block_range(len(all_reads), rank, world)   # contiguous block per rank; no data-path collective
    reads, truth = all_reads[lo:hi], all_truth[lo:hi]
    targets = [stitch_b200.TargetSeq(n, s) for n, s in named]
    al = stitch_b200.Builder(**kw).build_aligners(targets, device=local_rank)

    # reads resident in HBM for the kernel-side number
    blob = b"".join(reads)
    d_reads = torch.frombuffer(bytearray(blob), dtype=torch.uint8).cuda()
    offs = (C.c_uint64 * (len(reads) + 1))()
    acc = 0
    for k, r in enumerate(reads):
        offs[k] = acc
        acc += len(r)
    offs[len(reads)] = acc

    kept = {"device": None, "e2e": None}   # the results of the last step of each pass (read back after the timed region)

    def step_device(last=False):
        res = C.c_void_p()
        rc = lib.stitch_custom_batch_device(al._h, C.c_void_p(d_reads.data_ptr()), offs, len(reads), C.byref(res))
        if rc != 0:
            raise RuntimeError(al.last_error())
        if last:   # (kept only then: held across steps, results slowed this pass by 0.7 % on a B200 at 1000 W)
            kept["device"] = res
        else:
            lib.stitch_free_results(res)
        return al.stats()

    host_buf, host_offs = _abi.pack_reads(reads)   # e2e: host buffers in, chains out

    def step_e2e(last=False):   # (every step's results live until the next step frees them)
        res = C.c_void_p()
        rc = lib.stitch_align_batch(al._h, host_buf, host_offs, len(reads), None, 0, C.byref(res))
        if rc != 0:
            raise RuntimeError(al.last_error())
        if kept["e2e"] is not None:
            lib.stitch_free_results(kept["e2e"])
        kept["e2e"] = res
        return al.stats()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        agg = {"cells": 0, "fill_ms": 0.0, "tb_ms": 0.0, "launches": 0, "h2d": 0, "d2h": 0, "fills": 0, "tb_bytes": 0,
               "packed_ms": 0.0, "wide_ms": 0.0, "redo_ms": 0.0, "packed_cells": 0, "redo_fills": 0, "tail_ms": 0.0, "packed_launches": 0,
               "tile_columns": 0, "quiet_tile_columns": 0}
        barrier()
        t0 = time.perf_counter()
        for k in range(steps):
            s = fn(last=k == steps - 1)
            agg["cells"] += s.cells; agg["fill_ms"] += s.fill_ms; agg["tb_ms"] += s.traceback_ms
            agg["launches"] += s.kernel_launches; agg["h2d"] += s.h2d_bytes; agg["d2h"] += s.d2h_bytes
            agg["fills"] += s.fills; agg["tb_bytes"] += s.traceback_bytes
            agg["packed_ms"] += s.packed_fill_ms; agg["wide_ms"] += s.wide_fill_ms; agg["redo_ms"] += s.redo_fill_ms
            agg["tile_columns"] += s.tile_columns; agg["quiet_tile_columns"] += s.quiet_tile_columns
            agg["packed_cells"] += s.packed_cells; agg["redo_fills"] += s.redo_fills; agg["tail_ms"] += s.tail_fill_ms; agg["packed_launches"] += s.packed_launches
        barrier()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
            c = torch.tensor([agg["cells"], agg["launches"]], dtype=torch.float64, device="cuda")
            dist.all_reduce(c, op=dist.ReduceOp.SUM)
            agg["cells_all"] = float(c[0].item()); agg["launches_all"] = int(c[1].item())
        else:
            agg["cells_all"] = float(agg["cells"]); agg["launches_all"] = agg["launches"]
        return dt, agg

    for _ in range(args.warmup):
        step_device()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    try:
        dt, agg = timed(step_device, args.steps)
    finally:   # (no nvidia-smi process outlives a failed step)
        clocks = sampler.stop() if rank == 0 else None
    # e2e: one warm-up, then the same number of steps
    if args.no_e2e:
        dt_e, agg_e = dt, dict(agg)
        args.no_parity_check = True
    else:
        step_e2e()
        dt_e, agg_e = timed(step_e2e, args.steps)

    if rank == 0:
        peaks, peak_src = read_peaks()
        gcups = agg["cells_all"] / dt / 1e9
        gcups_e = agg_e["cells_all"] / dt_e / 1e9
        fill_s = agg["packed_ms"] * 1e-3
        fill_gcups = agg["packed_cells"] / fill_s / 1e9 if fill_s > 0 else 0.0
        launches_fill = max(1, agg["packed_launches"])   # fill_packed_kernel launches in the timed region (one per chunk of reads)
        ach = agg["packed_cells"] * ALG_BYTES_PER_CELL / fill_s / 1e9 if fill_s > 0 else 0.0
        skipped_frac = agg["quiet_tile_columns"] / agg["tile_columns"] if agg["tile_columns"] else 0.0
        # HBM traffic of the fill kernel per launch, from the counters of the run itself: every computed tile-column reads and
        # writes its 2 KB of rolling state (a materialised tile only writes; counted as read + write: an upper bound), plus the
        # checkpoints and jump records (traceback_bytes), the tail columns and unit re-fills of the walk not included
        state_bytes = (agg["tile_columns"] - agg["quiet_tile_columns"]) * 2.0 * 2048.0
        traffic_est = (state_bytes + agg["tb_bytes"]) / launches_fill
        gops = C.c_double(0)
        lib.stitch_measure_int32_peak(local_rank, C.byref(gops))
        cfg = workload_config(args, kw, named, world, len(reads[0]))
        cfg["cells_per_step"] = agg["cells_all"] / args.steps
        line = {
            "metric": "GCUPS", "value": gcups, "unit": "GCUPS", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32", "data": "synthetic",
            "config": cfg,
            "reads_per_s": len(reads) * world * args.steps / dt,
            "clocks": clocks,
            "e2e": {"value": gcups_e, "unit": "GCUPS", "reads_per_s": len(reads) * world * args.steps / dt_e,
                    "h2d_bytes_per_step": agg_e["h2d"] / args.steps, "d2h_bytes_per_step": agg_e["d2h"] / args.steps,
                    "fills_per_step": agg_e["fills"] / args.steps, "ms_per_step": dt_e / args.steps * 1e3},
            "gpu_launches": agg["launches_all"],
            "quiet_tiles": {"tile_columns": agg["tile_columns"], "skipped": agg["quiet_tile_columns"],
                            "frac_skipped": skipped_frac,
                            "note": "bulk pass of fill_packed_kernel on this rank: (256-row tile, column) pairs proven to be in the closed form "
                                    "jump + substitution score and therefore neither loaded, computed nor stored (dp_packed.h, PkQuiet); "
                                    "GCUPS counts every cell of every fill, as the metric defines it"},
            "phases_ms_per_step": {"packed_fill": agg["packed_ms"] / args.steps, "packed_tail": agg["tail_ms"] / args.steps, "wide_fill": agg["wide_ms"] / args.steps,
                                   "window_reruns": agg["redo_ms"] / args.steps, "fixup_walk": agg["tb_ms"] / args.steps,
                                   "window_rerun_reads": agg["redo_fills"] / args.steps,
                                   "packed_kernel_gcups": (agg["packed_cells"] / (agg["packed_ms"] * 1e-3) / 1e9) if agg["packed_ms"] else None},
            "roofline": {"bound": "hbm", "kernel": "fill_packed_kernel", "achieved": ach, "peak": peaks.get("hbm_gbs"),
                         "unit": "GB/s", "frac": ach / peaks.get("hbm_gbs") if peaks.get("hbm_gbs") else None,
                         "traffic": traffic_est,
                         "traffic_source": "derived in this run from the kernel's own counters: computed tile-columns x 4 KB (2 KB of rolling "
                                           "state read + written) + checkpoint and jump-record bytes; the ncu capture of the same kernel is "
                                           "under profiles/ (dram__bytes_read + dram__bytes_write per launch)",
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_cell": ALG_BYTES_PER_CELL,
                         "avg_launch_ms": agg["packed_ms"] / launches_fill if launches_fill else None, "kernel_gcups": fill_gcups,
                         "state_stream_gbs": fill_gcups * STATE_BYTES_PER_CELL * (1.0 - skipped_frac),
                         "state_stream_frac_of_peak": fill_gcups * STATE_BYTES_PER_CELL * (1.0 - skipped_frac) / peaks.get("hbm_gbs") if peaks.get("hbm_gbs") else None,
                         "note": "achieved = 0.5 B x cell updates / CUDA-event time of fill_packed_kernel (one launch per step; its time "
                                 "includes the tail columns and the in-kernel fix-up/walk phase). The rolling column state (16 B per cell "
                                 "update of a computed tile) is streamed through HBM because a read's state (2.6 MB) does not fit one SM; "
                                 "quiet tiles are neither loaded nor stored. With them the kernel is not HBM-bound: see int_roofline and "
                                 "DESIGN.md section 4"},
            "int_roofline": {"bound": "int32", "achieved": fill_gcups * ALG_OPS_PER_CELL, "peak": gops.value,
                             "unit": "Gop/s", "frac": fill_gcups * ALG_OPS_PER_CELL / gops.value if gops.value else None,
                             "ops_per_cell": ALG_OPS_PER_CELL,
                             "peak_source": "stitch_measure_int32_peak (add+max issue-rate microbenchmark, measured in this run)"},
        }
        if args.dump_outputs:
            passes = [p for p in ("device", "e2e") if kept[p] is not None]
            line["dump_outputs"] = {p: dump_results(lib, _lib.PRODUCT_RESULTS, kept[p], args.dump_outputs, p, (DUMP_BYTES - 4096) // len(passes))
                                    for p in passes}
        if not args.no_parity_check:
            try:
                e2e_chains = _lib.read_results(lib, _lib.PRODUCT_RESULTS, kept["e2e"])
                line["parity_check"] = parity_check(al, kw, named, reads, truth, e2e_chains)
            except Exception as e:
                line["parity_check"] = {"reads": 0, "ok": False, "error": str(e)}
        if not args.no_cpu_baseline and world >= 1:
            try:
                line["cpu_baseline"] = cpu_baseline(kw, named, all_reads, all_truth, args.cpu_budget_s)
            except Exception as e:   # the baseline is reported, never required for the GPU number
                line["cpu_baseline"] = {"value": None, "unit": "GCUPS", "cores": 0, "kind": "port", "sample": f"failed: {e}"}
        print(json.dumps(line))
    for res in kept.values():
        if res is not None:
            lib.stitch_free_results(res)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
