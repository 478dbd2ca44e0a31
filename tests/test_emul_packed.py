"""CPU tier: the packed-key arithmetic of the fast fill (stitch_b200/csrc/dp_packed.h), run through the
CPU emulator with the kernel's structure (warp chunks, halo strips, special first/last tiles, hand-over
to the wide tail, wide re-fill for the traceback), must reproduce the oracle bit for bit."""
import itertools
import random

import pytest

import emul_lib as emul_lib_mod
import gen
import keyedge
from stitch_b200._abi import make_opts
from test_emul_parity import compare, emul_lib, run_both  # noqa: F401


@pytest.mark.parametrize("strip", [1, 2, 8])
@pytest.mark.parametrize("block", range(6))
def test_fuzz_packed_small(oracle, emul_lib, strip, block):
    for seed in range(block * 50, block * 50 + 50):
        alphabet = [b"ACGT", b"AC", b"A", b"ACGTN"][seed % 4]
        contigs, reads = gen.fuzz_case(seed + 7000, max_contigs=5, max_len=90, max_read=70, alphabet=alphabet)
        kw = gen.fuzz_opts_packed(seed, strip)
        got, exp = run_both(oracle, emul_lib, kw, contigs, reads, strip, raw=(seed % 3 != 0))
        compare(got, exp, f"seed {seed} strip {strip} {kw}")


@pytest.mark.parametrize("strip", [1, 2, 8])
@pytest.mark.parametrize("block", range(4))
def test_fuzz_packed_multi_tile(oracle, emul_lib, strip, block):
    """Contigs spanning several warp tiles and warp chunks (halo strips), reads long enough for several
    checkpoint blocks and for the column base to drift."""
    tile = 32 * strip
    for seed in range(block * 8, block * 8 + 8):
        rng = random.Random(9000 + seed * 31 + strip)
        alphabet = [b"ACGT", b"AC", b"ACG"][seed % 3]
        lens = [rng.randint(1, 5 * tile) for _ in range(rng.randint(1, 5))] + [tile + 1, tile, tile - 1][: seed % 4]
        contigs = [gen.rand_seq(rng, l, alphabet) for l in lens]
        reads = [gen.chimeric_read(rng, contigs, rng.randint(20, 260), rng.randint(1, 4), strands=True,
                                   wrap=rng.random() < 0.5, noise=rng.random() < 0.8, alphabet=alphabet) for _ in range(3)]
        reads = [r if r else b"A" for r in reads]
        kw = gen.fuzz_opts_packed(seed + 100 * block, strip)
        got, exp = run_both(oracle, emul_lib, kw, contigs, reads, strip, raw=(seed % 2 == 0))
        compare(got, exp, f"seed {seed} strip {strip} {kw}")


def _check_plan(kw, n, m_max, strip, ctx=""):
    """The restatement (tests/keyedge.py) and pk_plan (dp_packed.h, through the emulator library) agree; returns the plan."""
    p = keyedge.plan(kw, n, m_max, strip)
    got = emul_lib_mod.pk_plan(make_opts(**kw), n, m_max, strip)
    assert got == (p if isinstance(p, int) else 0), f"{ctx} {kw} n {n} m_max {m_max} strip {strip}: pk_plan {got}, restated {p}"
    return p


def _random_scoring(rng, strip=8):
    """Valid options, scores up to a few thousand; the gap extension inside the strip's insertion-chain reach 2 times in 3."""
    mult = int(2 ** rng.uniform(0, 11))
    kw = dict(mode=rng.randint(0, 3), match_score=rng.randint(0, 3) * mult,
              mismatch_score=(-rng.randint(0, 5) if rng.random() < 0.9 else rng.randint(0, 2)) * mult,
              gap_open=-rng.randint(0, 8) * mult, gap_extend=-rng.randint(0, 3) * mult)
    kw.update({k: -rng.randint(0, 12) * mult for k in keyedge.SCORE_KEYS[4:]})
    if rng.random() < 0.67:
        band = keyedge.terms(keyedge.scoring(kw))[3]
        kw["gap_extend"] = -(band // strip + 1 + rng.randint(0, 2))
    return kw


def _plan_regime(strip):
    rng = random.Random(61 + strip)
    reasons = {}
    for _ in range(3000):
        kw = _random_scoring(rng, strip)
        p = _check_plan(kw, int(2 ** rng.uniform(0, 25)), int(2 ** rng.uniform(0, 24)), strip, "random")
        reasons[p if isinstance(p, str) else "packed"] = reasons.get(p if isinstance(p, str) else "packed", 0) + 1
    for r in ("packed", "e >= 0", "insertion-chain reach", "length bits", "score range"):
        assert reasons.get(r, 0) >= 10, reasons
    # the largest accepted read length and score scale, and one step on either side
    for seed in range(40):
        base = gen.fuzz_opts_packed(seed, strip)
        m_max = int(2 ** rng.uniform(0, 14))
        N = keyedge.max_n(base, m_max, strip)
        assert N > 0
        for n in (N - 1, N, N + 1):
            _check_plan(base, max(n, 1), m_max, strip, "max_n")
        assert keyedge.accepted(base, N, m_max, strip) and not keyedge.accepted(base, N + 1, m_max, strip)
        n = rng.randint(1, N)
        k = keyedge.edge_scale(base, n, m_max, strip)
        assert k >= 1
        for kk in (k - 1, k, k + 1):
            if kk >= 1:
                _check_plan(keyedge.scale(base, kk), n, m_max, strip, "edge_scale")
        assert not keyedge.accepted(keyedge.scale(base, k + 1), n, m_max, strip)
    # insertion-chain reach band // |e| + 1 exactly STRIP (accepted) and STRIP + 1 (refused), band at both ends of its range
    for ae in range(1, 6):
        for reach in (strip, strip + 1):
            for band in ((reach - 1) * ae, (reach - 1) * ae + ae - 1):
                for mode in range(4):   # match = mismatch = 1: band = -(jump score)
                    kw = dict(mode=mode, match_score=1, mismatch_score=1, gap_open=-rng.randint(0, 3), gap_extend=-ae, default_jump_score=-band)
                    assert keyedge.terms(keyedge.scoring(kw))[3] == band
                    p = _check_plan(kw, 100, 100, strip, "reach")
                    assert (p == "insertion-chain reach") == (reach > strip), (kw, p)
    # every LB transition (need = 2^LB - 1 / 2^LB) up to LB 24 / 25, through n and through m_max
    for LB in range(5, 26):
        for m_max in ((1 << LB) - 3, (1 << LB) - 2):
            _check_plan(dict(gap_extend=-2), 1, m_max, strip, "LB via m_max")
        kw = dict(match_score=1, mismatch_score=-1, gap_open=0, gap_extend=-1, default_jump_score=-1) if strip >= 4 else \
            dict(match_score=1, mismatch_score=-1, gap_open=0, gap_extend=-4, default_jump_score=-1)
        n = keyedge.n_for_lb(kw, LB - 1, 2, strip)
        for nn in (n, n + 1):
            p = _check_plan(kw, nn, 2, strip, "LB via n")
            if keyedge.length_bits(keyedge.scoring(kw), nn, 2) > keyedge.LB_MAX:
                assert p == "length bits"
    # lim exactly 2^(SB-1) (refused: the score field would wrap) and 2^(SB-1) - 2 (accepted); lim moves by 4 per unit of gap
    # open, so pick base scorings of both residues mod 4 and solve for the gap open
    hits = {0: 0, 2: 0}
    for seed in range(400):
        r = random.Random(seed)
        base = dict(mode=r.choice([0, 2, 3]), match_score=r.randint(0, 4), mismatch_score=-r.randint(0, 6), gap_open=0,
                    default_jump_score=-r.randint(0, 12))
        band = keyedge.terms(keyedge.scoring(dict(base, gap_extend=-1)))[3]
        base["gap_extend"] = -(band // strip + 1 + r.randint(0, 2))
        for LB in range(13, 21):
            m_max = (1 << LB) - 3
            T = 1 << (27 - LB)
            lim0 = keyedge.lim(keyedge.scoring(base), strip)
            d = (T - lim0) % 4
            if T - lim0 < 8 or d not in (0, 2):
                continue
            kw = dict(base, gap_open=-((T - lim0 - d) // 4))
            assert keyedge.lim(keyedge.scoring(kw), strip) == T - d
            if keyedge.length_bits(keyedge.scoring(kw), 1, m_max) != LB:
                continue
            p = _check_plan(kw, 1, m_max, strip, f"lim = 2^(SB-1) - {d}")
            assert p == ("score range" if d == 0 else LB), (kw, p)
            hits[d] += 1
    assert hits[0] >= 20 and hits[2] >= 20, hits


def test_packed_plan_regime():
    """pk_plan (which reads run on the packed kernels, with how many length bits) against its restatement in tests/keyedge.py:
    random (scoring, n, m_max) triples, every boundary +-1 (largest accepted read length and score scale, insertion-chain reach
    exactly STRIP, LB 24 / 25), and scorings whose score range lim is exactly 2^(SB-1) (refused) or 2^(SB-1) - 2 (accepted)."""
    for strip in (1, 2, 8):
        _plan_regime(strip)


def test_yclip_guard_unreachable():
    """pk_plan's query-local y-prefix clip test (dp_packed.h) never fires for options the product accepts: gap open <= 0 and an
    insertion-chain reach within STRIP give o + e (TILE + 1) < gmin + min(submin, 0).  The guard stays; this records why."""
    rng = random.Random(5)
    for strip in (1, 2, 8):
        for _ in range(20000):
            kw = _random_scoring(rng, strip)
            kw["mode"] = 1
            p = keyedge.plan(kw, 100, 100, strip)
            assert p != "y-prefix clip", kw
        for m, x, o, e, g in itertools.product(range(0, 4), range(-4, 3), range(-3, 1), range(-6, 0), range(-6, 1)):
            kw = dict(mode=1, match_score=m, mismatch_score=x, gap_open=o, gap_extend=e, default_jump_score=g)
            assert keyedge.plan(kw, 100, 100, strip) != "y-prefix clip", kw
    # a positive gap open (the only way to reach the guard) is refused by the product as by the reference
    assert emul_lib_mod.pk_plan(make_opts(gap_open=1), 100, 100, 8) == -1
