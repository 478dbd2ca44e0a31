"""GPU tier: the chains must not depend on the checkpoint spacing K the backend picks for a batch, nor on how often a chunk is
re-run because an operation buffer overflowed.  K decides where the packed fill stores checkpoints (regular every K columns,
late ones at n - 32 k), where its tail and the wide path's window re-runs restart, how long the walk's re-filled units are
(cone re-fills of more than 384 columns build their constants per column), and how much shared memory the walk needs
(whether it runs inside the packed kernel, whether it stages the contig's bases).  tests/ckplan.py restates those decisions;
every case here is checked against the oracle and against the kernel launches the restatement predicts."""
import os

import pytest

import ckplan
import gen
import keyedge
from stitch_b200._abi import make_opts
from test_gpu_parity import compare

pytestmark = pytest.mark.gpu

KNOBS = ("STITCH_CK_EVERY", "STITCH_TRACK_WINDOW", "STITCH_CLUSTER", "STITCH_CLUSTER_MIN_TILES", "STITCH_CLUSTER_SMEM",
         "STITCH_PACKED", "STITCH_QUIET", "STITCH_WALK_IN_KERNEL", "STITCH_CONE")
TUNINGS = {
    "default": {},
    "walk kernel": {"STITCH_WALK_IN_KERNEL": "0"},
    "no cone": {"STITCH_CONE": "0"},
    "cluster 4": {"STITCH_CLUSTER": "4", "STITCH_CLUSTER_MIN_TILES": "1", "STITCH_CLUSTER_SMEM": "0"},
    "wide": {"STITCH_PACKED": "0", "STITCH_TRACK_WINDOW": "3"},
}


@pytest.fixture
def aligners():
    """Builds CUDA aligners with the given STITCH_* knobs (read when a context is created) and clears every knob again."""
    import stitch_b200
    made = []

    def build(kw, contigs, knobs):
        for k in KNOBS:
            os.environ.pop(k, None)
        os.environ.update(knobs)
        try:
            al = stitch_b200.Builder(**kw).build_aligners([stitch_b200.TargetSeq(f"c{k}", s) for k, s in enumerate(contigs)], device=0)
        finally:
            for k in KNOBS:
                os.environ.pop(k, None)
        made.append(al)
        return al
    yield build
    for al in made:
        al.close()
    for k in KNOBS:
        os.environ.pop(k, None)


def num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def predicted_launches(kw, contigs, reads, K, knobs, sms):
    """Kernel launches of a single-chunk batch (one run() of the backend) before window re-runs and retries."""
    L = ckplan.layout([len(c) for c in contigs], kw.get("double_strand", False))
    m_max = max(len(c) for c in contigs)
    jobs = [(L, p if isinstance(p, int) else 0) for p in (keyedge.plan(kw, len(r), m_max, 8) for r in reads)]
    return ckplan.plan_chunk(jobs, K, sms, walk_in_kernel=knobs.get("STITCH_WALK_IN_KERNEL", "1") != "0",
                             cluster_pref=int(knobs.get("STITCH_CLUSTER", "0")),
                             cluster_min_tiles=int(knobs.get("STITCH_CLUSTER_MIN_TILES", ckplan.CLUSTER_MIN_TILES)),
                             packed=knobs.get("STITCH_PACKED", "1") != "0")


def packed_cells(kw, contigs, reads, knobs):
    if knobs.get("STITCH_PACKED") == "0":
        return 0
    rows = sum(len(c) for c in contigs) * (2 if kw.get("double_strand") else 1)
    m_max = max(len(c) for c in contigs)
    return sum(rows * len(r) for r in reads if isinstance(keyedge.plan(kw, len(r), m_max, 8), int))


# spacings at which every tuning runs (the others: default and separate walk kernels): both sides of 32 and of the
# 384-column cone-constant limit, regular columns at the edge read's best end (32, 384), K > n and the largest K
FULL_K = (7, 32, 33, 224, 384, 385, 1024, 8192)

MODES = {   # mode, options; local and query-local modes track y-suffix clips (packed tail, wide window re-runs)
    0: dict(mode=0, double_strand=True, circular=True),
    1: dict(mode=1, double_strand=True),
    2: dict(mode=2, circular=True),
    3: dict(mode=3, double_strand=True, circular=True),
}


@pytest.mark.parametrize("mode", sorted(MODES))
def test_k_sweep_against_oracle(oracle, aligners, mode):
    """Every swept K against the oracle (every tuning at FULL_K), through align_batch (with and without --suboptimal) and
    custom_batch.  Single chunk batches: custom_batch and non-circular align_batch make exactly the launches ckplan predicts
    (plus 2 per batch with window re-runs); every packed read counts its cells as packed; the same chains at every K."""
    kw = MODES[mode]
    contigs, reads = ckplan.spacing_case(mode)
    named = [(f"c{k}", s) for k, s in enumerate(contigs)]
    sub_kw = dict(kw, suboptimal=True, suboptimal_pct=0.0)
    exp_align, _ = oracle.OracleAligners(make_opts(**kw), named).batch(reads, raw=False)
    exp_custom, _ = oracle.OracleAligners(make_opts(**kw), named).batch(reads, raw=True)
    sub_reads = reads[::3]
    exp_sub, _ = oracle.OracleAligners(make_opts(**sub_kw), named).batch(sub_reads, raw=False)
    sms = num_sms()
    tracked = mode in (0, 1)
    seen_in_kernel = set()
    for K in ckplan.SWEEP_K:
        for name, tuning in TUNINGS.items():
            if K not in FULL_K and name not in ("default", "walk kernel"):
                continue
            knobs = dict(tuning, STITCH_CK_EVERY=str(K))
            ctx = f"mode {mode} K {K} {name}"
            al = aligners(kw, contigs, knobs)
            got = al.custom_batch(reads)
            st = al.stats()
            compare(got, exp_custom, ctx + " custom")
            plan = predicted_launches(kw, contigs, reads, K, knobs, sms)
            seen_in_kernel.add(plan["in_kernel"])
            assert st.kernel_launches == plan["launches"] + (2 if st.redo_fills else 0), (ctx, plan, st.kernel_launches, st.redo_fills)
            assert st.packed_cells == packed_cells(kw, contigs, reads, knobs), ctx
            if name == "wide" and tracked:   # a 3-column window: every read whose chain ends earlier is filled again
                assert st.redo_fills > 0, ctx
            if K == 8192 and name == "default":
                assert not plan["in_kernel"], "at K = 8192 the walk's staging does not fit beside the packed fill"
            compare(al.align_batch(reads), exp_align, ctx + " align")
            if name == "default" and K in FULL_K:
                al2 = aligners(sub_kw, contigs, knobs)
                got = al2.align_batch(sub_reads)
                compare(got, exp_sub, ctx + " suboptimal")
                if not kw.get("circular"):
                    st = al2.stats()
                    plan = predicted_launches(sub_kw, contigs, sub_reads, K, knobs, sms)
                    assert st.kernel_launches == plan["launches"] + (2 if st.redo_fills else 0), (ctx, plan, st.kernel_launches)
    assert seen_in_kernel == {True, False}


def test_base_staging_flips_with_k(oracle, aligners):
    """A contig of ~120 kb: the packed walk phase stages its bases at K <= 1024 and reads them from global memory at K = 2048;
    at K = 8192 the walk leaves the packed kernel and the walk kernel cannot stage them either (ckplan), and the chains stay
    the oracle's.  One CTA per read so that the walk may run inside the packed kernel."""
    import random
    rng = random.Random(611)
    contigs = [gen.rand_seq(rng, 120000), gen.rand_seq(rng, 900), gen.rand_seq(rng, 600)]
    reads = []
    for _ in range(4):
        s = rng.randrange(0, 120000 - 400)
        reads.append(gen.noisy(rng, contigs[0][s:s + 300]) + gen.revcomp(contigs[1][100:250]))
    kw = dict(double_strand=True)
    named = [(f"c{k}", s) for k, s in enumerate(contigs)]
    exp, _ = oracle.OracleAligners(make_opts(**kw), named).batch(reads, raw=True)
    sms = num_sms()
    decisions = {}
    for K in (96, 1024, 2048, 8192):
        for tuning in ({"STITCH_CLUSTER": "1"}, {"STITCH_CLUSTER": "1", "STITCH_WALK_IN_KERNEL": "0"}):
            knobs = dict(tuning, STITCH_CK_EVERY=str(K))
            al = aligners(kw, contigs, knobs)
            got = al.custom_batch(reads)
            st = al.stats()
            compare(got, exp, f"K {K} {tuning}")
            plan = predicted_launches(kw, contigs, reads, K, knobs, sms)
            assert st.kernel_launches == plan["launches"], (K, tuning, plan)
            decisions[(K, "STITCH_WALK_IN_KERNEL" in tuning)] = (plan["in_kernel"], plan["pstage_bases"], plan["wstage_bases"])
    assert decisions[(1024, False)] == (True, True, None)
    assert decisions[(2048, False)] == (True, False, None)
    assert decisions[(8192, False)] == (False, None, False)
    assert decisions[(2048, True)] == (False, None, True) and decisions[(8192, True)] == (False, None, False)


# ---- operation-buffer retries --------------------------------------------------------------------------------------------

RETRY_CASES = [   # (n, C, k, suboptimal): ckplan.retries of the read = 0, 1, 2, 3 and the case the old x64 ceiling refused
    (300, 1, 8, False),
    (1000, 8, 1, True),
    (1000, 32, 1, True),
    (1000, 128, 1, True),
    (3000, 256, 1, True),
]


def skip_batch(aligners, n, C, k, sub, knobs=None):
    contigs, read, blocks = ckplan.skip_case(n, C, k)
    kw = dict(ckplan.SKIP_SCORING, suboptimal=sub, suboptimal_pct=0.0)
    need = C * 2 * blocks if sub else 2 * blocks   # (each chain: its ops + the x-suffix clip that align_batch removes)
    return kw, contigs, read, blocks, need, aligners(kw, contigs, dict(knobs or {}))


@pytest.mark.parametrize("case", range(len(RETRY_CASES)))
def test_operation_buffer_retries(oracle, aligners, case):
    """Reads whose chains are k '=' and one 'I' in turn (ckplan.skip_case) against C copies of a contig: the suboptimal batch
    returns C chains of 2n run-length ops in one buffer.  The chunk is re-run with x4 buffers until they fit: at least as many
    re-runs as the restated buffer sizes force (each re-run repeats every launch of the chunk), at most as many as it takes to
    reach the bound no chain exceeds.  256 chains of a 3 kb read need more than the former fixed x64 ceiling allowed."""
    n, C, k, sub = RETRY_CASES[case]
    kw, contigs, read, blocks, need, al = skip_batch(aligners, n, C, k, sub)
    got = al.align_batch([read])[0]
    st = al.stats()
    single = predicted_launches(kw, contigs, [read], 256, {}, num_sms())["launches"]
    assert st.kernel_launches % single == 0, (st.kernel_launches, single)
    r = st.kernel_launches // single - 1
    expect = ckplan.retries(n, C, sub, need)
    assert expect == case if case < 4 else expect == 4
    assert expect <= r <= ckplan.retries(n, C, sub, ckplan.ops_cap(n, C, sub, 99)), (r, expect)
    assert st.packed_cells == (r + 1) * C * len(contigs[0]) * n
    assert len(got) == (C if sub else 1)
    for c, a in enumerate(got):
        assert ckplan.skip_chain_ok(a, n, k, blocks, c), (case, c, a.score, len(a.ops))
    if C <= 8:
        exp, _ = oracle.OracleAligners(make_opts(**kw), [(f"c{i}", s) for i, s in enumerate(contigs)]).batch([read], raw=False)
        compare([got], exp, f"retry case {case}")


def test_retried_read_in_a_mixed_batch(oracle, aligners):
    """A read that overflows its buffer next to ordinary noisy reads, two reads in flight per chunk, on the packed path, on the
    wide path (STITCH_PACKED=0, which also re-runs tracking windows) and at another K: the same chains as the oracle."""
    import random
    contigs, read, _ = ckplan.skip_case(700, 4, 1, seed=3)
    rng = random.Random(12)
    others = [gen.rand_seq(rng, 1500), gen.rand_seq(rng, 1200)]
    allc = contigs + others
    reads = [gen.chimeric_read(rng, others, rng.randint(300, 700), 2, strands=False) for _ in range(5)]
    reads.insert(2, read)
    kw = dict(ckplan.SKIP_SCORING, suboptimal=True, suboptimal_pct=0.0)
    named = [(f"c{k}", s) for k, s in enumerate(allc)]
    exp, _ = oracle.OracleAligners(make_opts(**kw), named).batch(reads, raw=False)
    for knobs in ({}, {"STITCH_PACKED": "0"}, {"STITCH_CK_EVERY": "160"}):
        al = aligners(kw, allc, knobs)
        al.set_max_inflight(2)
        got = al.align_batch(reads)
        compare(got, exp, f"mixed {knobs}")
