"""CPU tier: the packed fill at the edges of its 32-bit key (stitch_b200/csrc/dp_packed.h), run through the CPU emulator
against the oracle: relative scores with the least headroom pk_plan accepts, alignment lengths filling the length field, and
jobs run with more length bits than their own plan (a CUDA launch gives every packed job the largest LB of the launch).
Every case asserts which path ran, so a plan that silently sends everything to the wide kernels fails here."""
import os
import random

import pytest

import emul_lib as emul_lib_mod
import keyedge
from test_emul_parity import compare, emul_lib, run_both  # noqa: F401


def _counted(strip, fn):
    before = emul_lib_mod.path_counters(strip)
    out = fn()
    after = emul_lib_mod.path_counters(strip)
    lb = {k: after["lb"].get(k, 0) - before["lb"].get(k, 0) for k in after["lb"]}
    return out, dict(packed=after["packed"] - before["packed"], wide=after["wide"] - before["wide"], lb={k: v for k, v in lb.items() if v})


@pytest.mark.parametrize("strip", [1, 2, 8])
@pytest.mark.parametrize("seed", range(8))
def test_score_headroom_edge(oracle, emul_lib, strip, seed):
    """Base scorings scaled to the largest k at which their reads stay packed: reads at max_n and max_n - 1 run packed with
    the score field nearly full (lim up to 99.9 % of 2^(SB-1)), a read at max_n + 1 runs wide; both call paths."""
    mode = seed % 4
    kw, contigs, edge, past, N = keyedge.headroom_case(seed, strip, mode)
    m_max = max(len(c) for c in contigs)
    LB = keyedge.plan(kw, N, m_max, strip)
    assert isinstance(LB, int) and not keyedge.accepted(kw, N + 1, m_max, strip)
    assert keyedge.headroom(kw, N, m_max, strip) > 0.5
    for raw in (True, False):
        (got, exp), c = _counted(strip, lambda: run_both(oracle, emul_lib, kw, contigs, edge, strip, raw=raw))
        compare(got, exp, f"edge seed {seed} strip {strip} raw {raw} N {N} {kw}")
        assert c["wide"] == 0 and c["packed"] >= 2, c
        if raw:   # one fill per read, each with the plan's LB
            assert c["lb"] == {LB: 2}, (c, LB)
    (got, exp), c = _counted(strip, lambda: run_both(oracle, emul_lib, kw, contigs, [past], strip, raw=True))
    compare(got, exp, f"past the edge seed {seed} strip {strip} {kw}")
    assert c["packed"] == 0 and c["wide"] >= 1, c   # (a wide fill may run twice: the full-tracking re-run)


@pytest.mark.parametrize("strip", [1, 2, 8])
@pytest.mark.parametrize("mode", range(4))
def test_length_field_edge(oracle, emul_lib, strip, mode):
    """Reads at the largest length whose plan takes 11 length bits, built so that the best path carries many contig-side
    insertions (strip 8: alignment lengths up to ~1.4 x the read length); chain lengths as the oracle's."""
    kw, contigs, reads, n = keyedge.length_case(mode, strip, mode)
    best = 0.0
    for raw in (True, False):
        (got, exp), c = _counted(strip, lambda: run_both(oracle, emul_lib, kw, contigs, reads, strip, raw=raw))
        compare(got, exp, f"length strip {strip} mode {mode} raw {raw} n {n} {kw}")
        assert c["wide"] == 0 and c["packed"] >= len(reads), c
        if raw:
            assert c["lb"] == {11: len(reads)}, c
        best = max([best] + [a.length / n for chains in got for a in chains])
    if strip == 8 and mode == 0:
        assert best > 1.25, best   # the insertion-heavy reads really lengthen the alignment


@pytest.mark.parametrize("strip", [1, 2, 8])
@pytest.mark.parametrize("seed", range(3))
def test_widened_length_bits(oracle, emul_lib, strip, seed):
    """A job run with more length bits than its own plan (EMUL_LB_MIN reproduces the CUDA launch's widening to the largest LB
    of the launch): every LB from the reads' own up to the largest one whose score field still holds the scoring's range."""
    kw, contigs, edge, _, _ = keyedge.headroom_case(seed + 20, strip, (seed + strip) % 4, n_edge=20000)
    m_max = max(len(c) for c in contigs)
    rng = random.Random(seed)
    short = [keyedge.exact_len(rng, edge[0][rng.randrange(0, 20):], rng.randint(8, 40)) for _ in range(3)]
    own = max(keyedge.plan(kw, len(r), m_max, strip) for r in short)
    top = keyedge.max_lb(kw, strip)
    assert isinstance(own, int) and top > own, (own, top)
    for raw in (True, False):
        exp = None
        for LB in range(own, top + 1):
            os.environ["EMUL_LB_MIN"] = str(LB)
            try:
                (got, e), c = _counted(strip, lambda: run_both(oracle, emul_lib, kw, contigs, short, strip, raw=raw))
            finally:
                os.environ.pop("EMUL_LB_MIN", None)
            exp = exp or e
            compare(got, exp, f"LB {LB} (own {own}) strip {strip} raw {raw} {kw}")
            assert c["wide"] == 0 and set(c["lb"]) == {LB}, (LB, c)
