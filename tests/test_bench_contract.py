"""bench.py: the reference arm (the restated reference timed on host cores) prints one JSON line with the keys a reader
of the benchmark expects; the GPU arm refuses to run without a device (there is no CPU path); `--dump-outputs` writes the
chains the timed passes computed (the writer on the CPU emulator, the whole option in the gpu tier)."""
import ctypes as C
import json
import os
import random
import subprocess
import sys

import numpy as np
import pytest

import gen
from stitch_b200 import _abi, _lib
from stitch_b200._abi import make_opts
from test_emul_parity import emul_lib  # noqa: F401

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load_dump(d, name):
    """{read index: [(chain fields, ops)]} of the files bench.dump_results wrote."""
    reads, chains, ops = (np.load(os.path.join(d, f"{name}_{k}.npy")) for k in ("reads", "chains", "ops"))
    assert reads.dtype == chains.dtype == ops.dtype == np.float64
    out = {int(r): [] for r, _ in reads}
    for row, c in enumerate(chains.astype(np.int64)):
        out[int(c[0])].append((tuple(c[1:]), [tuple(o) for o in ops[ops[:, 0] == row][:, 1:].astype(np.int64)]))
    assert [len(out[int(r)]) for r, _ in reads] == [int(n) for _, n in reads]
    return out


def as_dumped(a):
    return ((a.score, a.xstart, a.xend, a.ystart, a.yend, a.xlen, a.ylen, a.start_contig_idx, a.end_contig_idx, a.length), list(a.ops))


def test_dump_results_round_trip(emul_lib, tmp_path):
    """bench.dump_results writes every field and operation of the chains a results handle holds; a budget too small for
    all reads keeps a seeded sample of whole reads within it."""
    import bench
    rng = random.Random(3)
    contigs = [gen.rand_seq(rng, rng.randint(200, 400)) for _ in range(4)]
    reads = [gen.chimeric_read(rng, contigs, 200, 3, strands=True, wrap=True) for _ in range(30)]
    e = emul_lib.EmulAligners(make_opts(double_strand=True, circular=True, suboptimal=True, suboptimal_pct=90.0),
                              [(f"c{k}", s) for k, s in enumerate(contigs)])
    buf, offs = _abi.pack_reads(reads)
    res = C.c_void_p()
    assert e.e.emul_align_batch(e._h, buf, offs, len(reads), None, 0, C.byref(res)) == 0
    try:
        exp = _lib.read_results(e.e, emul_lib.EMUL_RESULTS, res)
        samples = []
        for budget in (1 << 30, 20000):
            d = str(tmp_path / str(budget))
            info = bench.dump_results(e.e, emul_lib.EMUL_RESULTS, res, d, "e2e", budget)
            got = load_dump(d, "e2e")
            assert info["reads"] == len(got) and info["of_reads"] == len(reads)
            assert got == {r: [as_dumped(a) for a in exp[r]] for r in got}
            assert sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)) <= budget + 3 * 128   # + the .npy headers
            samples.append(sorted(got))
        assert samples[0] == list(range(len(reads))) and 0 < len(samples[1]) < len(reads)
    finally:
        e.e.emul_free_results(res)
        e.close()


@pytest.mark.gpu
def test_dump_outputs_on_gpu(tmp_path):
    """`--dump-outputs DIR`: the chains of the last timed step of both passes, equal to what the library returns for the
    same seeded reads; `--steps K` timed steps of the full batch each."""
    import stitch_b200
    from stitch_b200 import synth
    d = str(tmp_path / "out")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "1", "--reads", "4", "--read-len", "300", "--steps", "2",
                        "--warmup", "1", "--no-cpu-baseline", "--no-parity-check", "--dump-outputs", d],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    line = json.loads(p.stdout.decode().strip().splitlines()[-1])
    kw, named, reads = synth.config(1, 4, 300)
    assert line["steps"] == 2 and line["config"]["cells_per_step"] == sum(len(s) for _, s in named) * sum(len(r) for r in reads)
    assert sorted(os.listdir(d)) == sorted(f"{x}_{k}.npy" for x in ("device", "e2e") for k in ("reads", "chains", "ops"))
    al = stitch_b200.Builder(**kw).build_aligners([stitch_b200.TargetSeq(n, s) for n, s in named], device=0)
    try:
        for name, exp in (("device", al.custom_batch(reads)), ("e2e", al.align_batch(reads))):
            assert load_dump(d, name) == {r: [as_dumped(a) for a in exp[r]] for r in range(len(reads))}, name
    finally:
        al.close()


def test_reference_arm_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--read-len", "300"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    line = json.loads(p.stdout.decode().strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "GCUPS" and line["unit"] == "GCUPS" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["n_gpus"] == 1 and "workload" in line["config"]
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "full-length reads (300 b)" in cb["sample"]
    e2e = line["e2e"]
    assert e2e["value"] == line["value"] and e2e["unit"] == "GCUPS" and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_gpu_arm_needs_a_device():
    import torch
    if torch.cuda.is_available():
        return
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, timeout=600)
    assert p.returncode != 0
    assert "no CUDA device" in p.stdout.decode()
