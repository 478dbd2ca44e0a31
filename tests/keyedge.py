"""The edges of the packed fill's 32-bit key (stitch_b200/csrc/dp_packed.h), restated for the tests.

    key = [ relative score : SB bits | priority : 4 bits | alignment length : LB bits ],   SB = 28 - LB

`plan` restates pk_plan: which (scoring, read length, longest contig) the packed path accepts and with how many length bits.
`max_n` / `edge_scale` find the last accepted read length / score scale, so that a test can put a read exactly at the edge of
the score field (lim just below 2^(SB-1)) or of the length field.

Scaling every score (match, mismatch, gap open / extend, the three jump scores) by an integer k > 0 leaves the chains
unchanged apart from score * k: every decision of the DP compares sums of scores, and the clip penalties are 0 or MIN_SCORE.
lim grows about k-fold, so a short read, cheap for the oracle, can run at the edge of the score field."""
from stitch_b200._abi import make_opts

MIN_SCORE = -858993459
LB_MAX = 24
SCORE_KEYS = ("match_score", "mismatch_score", "gap_open", "gap_extend", "jump_score_same_contig_and_strand",
              "jump_score_same_contig_opposite_strand", "jump_score_inter_contig")


def scoring(kw):
    """The Scoring the product derives from option kwargs (host_common.hpp make_opts): a dict."""
    o = make_opts(**kw)
    sc = dict(match=o.match_score, mismatch=o.mismatch_score, o=o.gap_open, e=o.gap_extend,
              g_same=o.jump_same, g_opp=o.jump_opp, g_inter=o.jump_inter)
    M = MIN_SCORE
    sc.update({0: dict(xp=0, xs=0, yp=0, ys=0), 1: dict(xp=M, xs=M, yp=0, ys=0),
               2: dict(xp=0, xs=0, yp=M, ys=M)}.get(o.mode, dict(xp=M, xs=M, yp=M, ys=M)))
    return sc


def _cdiv(a, b):   # C integer division (truncates toward zero)
    q = abs(a) // abs(b)
    return q if (a >= 0) == (b > 0) else -q


def terms(sc):
    submax0 = max(sc["match"], sc["mismatch"], 0)
    submin = min(sc["match"], sc["mismatch"])
    gmin = min(sc["g_same"], sc["g_opp"], sc["g_inter"])
    band = submax0 - submin - gmin
    neg = -(band - sc["o"] - sc["e"] + 2 * submax0 + 2)
    return submax0, submin, gmin, band, neg


def lim(sc, strip):
    """Range the relative scores of a column span (pk_plan): must stay below 2^(SB-1)."""
    submax0, submin, _, band, neg = terms(sc)
    return 2 * (-neg + band + submax0 - min(submin, 0) - sc["o"] + (strip + 1) * -sc["e"]) + 16


def length_bits(sc, n, m_max):
    """LB pk_plan picks: the smallest with 2^LB > max(length bound of any cell, m_max + 2)."""
    submax0, submin, gmin, _, _ = terms(sc)
    ae = -sc["e"]
    len_bound = n * (2 + (submax0 + ae - 1) // ae) + (-gmin) - sc["o"] - min(submin, 0) + 64
    need = max(len_bound, m_max + 2)
    LB = 4
    while (1 << LB) <= need:
        LB += 1
    return LB


def plan(kw_or_sc, n, m_max, strip):
    """pk_plan restated: the length bits (an int) or why the read goes to the wide path (a str)."""
    sc = kw_or_sc if "e" in kw_or_sc else scoring(kw_or_sc)
    if sc["e"] >= 0:
        return "e >= 0"
    _, submin, gmin, band, _ = terms(sc)
    ae = -sc["e"]
    if _cdiv(band, ae) + 1 > strip:
        return "insertion-chain reach"
    if sc["yp"] != MIN_SCORE and sc["xp"] == MIN_SCORE and sc["o"] + sc["e"] * (32 * strip + 1) > gmin + min(submin, 0):
        return "y-prefix clip"
    LB = length_bits(sc, n, m_max)
    if LB > LB_MAX:
        return "length bits"
    SB = 28 - LB
    if SB < 4 or lim(sc, strip) >= 1 << (SB - 1):
        return "score range"
    return LB


def accepted(kw, n, m_max, strip):
    return isinstance(plan(kw, n, m_max, strip), int)


def max_lb(kw, strip):
    """The largest LB whose score field still holds the scoring's range (0: none)."""
    L = lim(scoring(kw), strip)
    return max([LB for LB in range(4, LB_MAX + 1) if L < 1 << (27 - LB)], default=0)


def max_n(kw, m_max, strip):
    """The largest read length the plan accepts against contigs of at most m_max bases (0: none).  Acceptance is monotone
    in n: LB never shrinks as n grows, and the score range does not depend on n."""
    if not accepted(kw, 1, m_max, strip):
        return 0
    lo, hi = 1, 1 << 25
    while lo < hi:
        mid = (lo + hi + 1) // 2
        lo, hi = (mid, hi) if accepted(kw, mid, m_max, strip) else (lo, mid - 1)
    return lo


def scale(kw, k):
    """Option kwargs with every score multiplied by k (jump scores made explicit)."""
    o = make_opts(**kw)
    out = {key: v for key, v in kw.items() if key not in SCORE_KEYS + ("default_jump_score",)}
    vals = (o.match_score, o.mismatch_score, o.gap_open, o.gap_extend, o.jump_same, o.jump_opp, o.jump_inter)
    out.update({key: v * k for key, v in zip(SCORE_KEYS, vals)})
    return out


def edge_scale(base_kw, n, m_max, strip, k_max=1 << 16):
    """The largest k at which a read of length n stays packed (0: not even k = 1).  Acceptance is monotone in k: lim and
    LB grow with k, reach and the y-clip test do not change."""
    if not accepted(base_kw, n, m_max, strip):
        return 0
    lo, hi = 1, k_max
    while lo < hi:
        mid = (lo + hi + 1) // 2
        lo, hi = (mid, hi) if accepted(scale(base_kw, mid), n, m_max, strip) else (lo, mid - 1)
    return lo


def headroom(kw, n, m_max, strip):
    """lim / 2^(SB-1) of an accepted read: how close its score field is to wrapping around."""
    LB = plan(kw, n, m_max, strip)
    return lim(scoring(kw), strip) / (1 << (27 - LB))


def unscaled_key(a, k):
    """Alignment.key() with the score divided by k (asserting that it is a multiple)."""
    key = a.key()
    assert key[0] % k == 0, (key[0], k)
    return (key[0] // k,) + key[1:]


# ---- edge cases shared by the CPU (emulator) and GPU tiers ---------------------------------------------------------------

def exact_len(rng, read, n, alphabet=b"ACGT"):
    """`read` cut or padded with random bases to exactly n bases."""
    return (read + bytes(rng.choice(alphabet) for _ in range(max(0, n - len(read)))))[:n]


def headroom_case(seed, strip, mode, n_edge=None):
    """A seeded in-regime base scoring scaled to the largest k at which a read of a few hundred bases stays packed, small
    contigs (a tie-prone alphabet for odd seeds), and noisy chimeric reads at max_n and max_n - 1 (packed, at the tightest
    score field) plus one at max_n + 1 (wide).  `n_edge`: scale for a read of this length instead (a longer one leaves the
    short reads of the case a smaller LB than the largest their scoring allows).  Returns (kw, contigs, edge reads, past-edge
    read, N)."""
    import random

    import gen
    rng = random.Random(7100 + 31 * seed + strip)
    alphabet = b"AC" if seed % 2 else b"ACGT"
    contigs = [gen.rand_seq(rng, rng.randint(40, 160), alphabet) for _ in range(rng.randint(2, 4))]
    m_max = max(len(c) for c in contigs)
    base = gen.fuzz_opts_packed(seed, strip)
    base["mode"] = mode
    n0 = rng.randint(60, 160)
    k = edge_scale(base, n_edge or n0, m_max, strip)
    assert k >= 1, base
    kw = scale(base, k)
    N = max_n(kw, m_max, strip)
    reads = [exact_len(rng, gen.chimeric_read(rng, contigs, n, rng.randint(1, 4), strands=True, wrap=True, alphabet=alphabet), n, alphabet)
             for n in (N, N - 1, N + 1)]
    return kw, contigs, reads[:2], reads[2], N


LENGTH_SCORINGS = {   # large submax0 / |e| inside the insertion-chain reach of the strip; an insertion beats a jump where it can
    8: dict(match_score=2, mismatch_score=-2, gap_open=0, gap_extend=-1, default_jump_score=-3),
    2: dict(match_score=1, mismatch_score=0, gap_open=0, gap_extend=-3, default_jump_score=-4),
    1: dict(match_score=1, mismatch_score=-1, gap_open=0, gap_extend=-4, default_jump_score=-1),
}


def n_for_lb(kw, LB, m_max, strip):
    """The largest read length whose plan takes at most LB length bits (the read fills the length field furthest)."""
    sc = scoring(kw)
    lo, hi = 1, 1 << 25
    while lo < hi:
        mid = (lo + hi + 1) // 2
        lo, hi = (mid, hi) if length_bits(sc, mid, m_max) <= LB else (lo, mid - 1)
    return lo


def dropped_read(rng, contigs, n, drop_every=3):
    """Contig segments with every `drop_every`-th base dropped from the read, so that the best path carries many
    contig-side insertions (the alignment length exceeds the read length), exactly n bases."""
    out = bytearray()
    while len(out) < n:
        c = rng.choice(contigs)
        s = rng.randrange(0, len(c) // 2)
        seg = c[s:s + rng.randint(len(c) // 3, len(c) - s)]
        out += bytes(b for i, b in enumerate(seg) if i % drop_every != drop_every - 1)
    return bytes(out[:n])


def length_case(seed, strip, mode, LB=11):
    """Reads at the largest n whose plan takes LB length bits, insertion-heavy, against a few contigs of a few hundred bases.
    Returns (kw, contigs, reads, n)."""
    import random

    import gen
    rng = random.Random(8200 + 13 * seed + strip)
    contigs = [gen.rand_seq(rng, rng.randint(200, 400)) for _ in range(3)]
    kw = dict(LENGTH_SCORINGS[strip], mode=mode, double_strand=seed % 2 == 1, circular=seed % 3 == 1)
    m_max = max(len(c) for c in contigs)
    n = n_for_lb(kw, LB, m_max, strip)
    assert plan(kw, n, m_max, strip) == LB and plan(kw, n + 1, m_max, strip) == LB + 1, (kw, n)
    reads = [dropped_read(rng, contigs, n, drop_every=3 + r) for r in range(2)]
    return kw, contigs, reads, n
