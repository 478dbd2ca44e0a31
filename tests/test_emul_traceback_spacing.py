"""CPU tier twin of test_gpu_traceback_spacing.py: the restated checkpoint plan (tests/ckplan.py) and, on the emulator, the
same kind of reads at the swept checkpoint spacings against the oracle.  The emulator shares dp_packed.h's cone re-fill with
the CUDA path, so walk units longer than PK_CONE_MAX_COLS columns (K > 384) run here too, with and without cones, for strips
of 1, 2 and 8 rows."""
import os

import pytest

import ckplan
import emul_lib
import keyedge
from stitch_b200._abi import make_opts
from test_emul_parity import compare

EMUL_KNOBS = ("EMUL_K", "EMUL_CONE", "EMUL_WINDOW", "EMUL_PACKED")


@pytest.fixture
def emul():
    """Builds emulator aligners with the given EMUL_* knobs (read when a context is created) and clears every knob again."""
    made = []

    def build(kw, contigs, knobs, strip):
        for k in EMUL_KNOBS:
            os.environ.pop(k, None)
        os.environ.update(knobs)
        try:
            e = emul_lib.EmulAligners(make_opts(**kw), [(f"c{k}", s) for k, s in enumerate(contigs)], strip=strip)
        finally:
            for k in EMUL_KNOBS:
                os.environ.pop(k, None)
        made.append(e)
        return e
    yield build
    for e in made:
        e.close()


def test_struct_sizes_match_the_headers():
    """The shared-memory restatement in ckplan uses the sizes the product's headers give these structs."""
    assert emul_lib.struct_sizes(8) == ckplan.SIZES
def test_tail_restart_plan():
    """The inputs of the sweep sit on both sides of every restart branch: the edge reads' first candidate column is a late
    checkpoint column for some K and a regular one for others, and the n - 80 read restarts from the late checkpoint n - 96."""
    branches = set()
    for K in ckplan.SWEEP_K:
        j0 = ckplan.tail_start(1536, 1600, K)
        branches.add("late" if j0 == 1504 and 1536 % K else ("regular" if 1536 % K == 0 else "other"))
        assert j0 < 1536
        j0 = ckplan.tail_start(1520, 1600, K)
        if (1519 // K) * K < 1504 and 1504 % K:
            assert j0 == 1504 and ckplan.ck_index(j0, 1600, K) == ckplan.regular_cks(1600, K) + 2
        assert ckplan.redo_start(1536, K) < 1536
    assert {"late", "regular"} <= branches
    cols = ckplan.ck_columns(1600, 2048)
    assert cols == {1504: 2, 1536: 1, 1568: 0}
    assert ckplan.ck_columns(1600, 32)[1568] == 48 and 1504 not in {j for j in ckplan.ck_columns(1600, 32) if j % 32}
    assert ckplan.k_candidates() == [128, 160, 192, 224, 256, 384, 512, 768, 1024, 1536, 2048, 3072, 4096, 6144, 8192]
    assert ckplan.k_candidates(auto=False)[0] == 256
    # units longer than the precomputed cone constants exist only for K > 384
    assert max(ckplan.cone_unit_cols(j, 384) for j in range(1, 4000)) == 384 < max(ckplan.cone_unit_cols(j, 385) for j in range(1, 4000))




EMUL_MODES = {8: 0, 2: 1, 1: 3}   # local (margin-0 tracking: the edge reads' best end is the first candidate column), query-local, global


@pytest.mark.parametrize("strip", [8, 2, 1])
def test_k_sweep_on_emulator(oracle, emul, strip):
    """Reads of the GPU sweep (lengths around multiples of K, edge reads ending at n - 64 and n - 80) at every K above the
    cone-constant limit and a share of the smaller ones, cone re-fills on and off, against the oracle; packed fills only (the
    strip's in-regime scoring), so that every walk unit is a packed re-fill."""
    contigs, reads = ckplan.spacing_case(strip)
    reads = [r for r in reads if len(r) in (385, 1024, 1600)]
    kw = dict(keyedge.LENGTH_SCORINGS[strip], mode=EMUL_MODES[strip], circular=strip == 2)
    m_max = max(len(c) for c in contigs)
    assert all(isinstance(keyedge.plan(kw, len(r), m_max, strip), int) for r in reads)
    named = [(f"c{k}", s) for k, s in enumerate(contigs)]
    exp, _ = oracle.OracleAligners(make_opts(**kw), named).batch(reads, raw=True)
    ks = [K for i, K in enumerate(ckplan.SWEEP_K) if K > ckplan.PK_CONE_MAX_COLS or i % 3 == (1, 2, 8).index(strip)]
    results = []
    for i, K in enumerate(ks):
        for cone in ("1", "0") if K in (385, 1024) else (str((i + strip) % 2),):
            before = emul_lib.path_counters(strip)["packed"]
            e = emul(kw, contigs, {"EMUL_K": str(K), "EMUL_CONE": cone, "EMUL_WINDOW": "3"}, strip)
            got = e.batch(reads, raw=True)
            compare(got, exp, f"strip {strip} K {K} cone {cone}")
            assert emul_lib.path_counters(strip)["packed"] - before == len(reads)
            results.append([[a.key() for a in l] for l in got])
    assert all(r == results[0] for r in results)
