"""GPU tier: the CUDA packed fill at the edges of its 32-bit key (stitch_b200/csrc/dp_packed.h): relative scores with the
least headroom pk_plan accepts, alignment lengths filling the length field, launches that widen short jobs to the largest LB
of the launch, and full-size batches whose scores are scaled to the edge (the chains must not change apart from score * k).
The DPX forms, the bulk pass without floors, the tail, quiet tiles and cluster fills all run there.  Every case asserts
which path ran (stats.packed_cells)."""
import random

import pytest

import gen
import keyedge
from stitch_b200._abi import make_opts
from test_gpu_parity import TUNING, cluster_tuning, compare, gpu_aligners

pytestmark = pytest.mark.gpu

EDGE_TUNINGS = [None] + [cluster_tuning(s, TUNING) for s in range(4)] + [{"STITCH_QUIET": "0"}, {"STITCH_WALK_IN_KERNEL": "0"}]
STATS = ("cells", "packed_cells", "tile_columns", "quiet_tile_columns", "redo_fills")


def _named(contigs):
    return [(f"c{k}", s) for k, s in enumerate(contigs)]


def _gpu(kw, named, reads, raw, tuning=None, max_inflight=0):
    al = gpu_aligners(kw, named, max_inflight, tuning)
    try:
        got = al.custom_batch(reads) if raw else al.align_batch(reads)
        st = al.stats()
        return got, {k: getattr(st, k) for k in STATS}
    finally:
        al.close()


def _oracle(oracle, kw, named, reads, raw):
    return oracle.OracleAligners(make_opts(**kw), named).batch(reads, raw=raw)[0]


def _edge_cases():
    for seed in range(8):
        kw, contigs, edge, past, N = keyedge.headroom_case(seed, 8, seed % 4)
        yield f"headroom {seed}", kw, contigs, edge, past
    for mode in range(4):
        kw, contigs, reads, n = keyedge.length_case(mode, 8, mode)
        yield f"length {mode}", kw, contigs, reads, None


@pytest.mark.parametrize("tuning", range(len(EDGE_TUNINGS)))
def test_key_edges_vs_oracle(oracle, tuning):
    """Reads at the largest accepted length of a scaled scoring (score field nearly full) and insertion-heavy reads at the
    largest length of 11 length bits, against the oracle, with production defaults, cluster fills of 1 / 2 / 4 / 16 CTAs
    (rolling state in cluster shared memory and in global memory), quiet tiles off, separate walk kernels.  All packed at
    the edge; the read one base past it runs wide."""
    t = EDGE_TUNINGS[tuning]
    worst = 0.0
    for name, kw, contigs, reads, past in _edge_cases():
        named = _named(contigs)
        m_max = max(len(c) for c in contigs)
        worst = max([worst] + [keyedge.headroom(kw, len(r), m_max, 8) for r in reads])
        for raw in (True, False):
            exp = _oracle(oracle, kw, named, reads, raw)
            got, st = _gpu(kw, named, reads, raw, t)
            compare(got, exp, f"{name} raw {raw} {t} {kw}")
            assert st["packed_cells"] == st["cells"] > 0, (name, st)
        if past is not None:
            exp = _oracle(oracle, kw, named, [past], True)
            got, st = _gpu(kw, named, [past], True, t)
            compare(got, exp, f"{name} past the edge {t} {kw}")
            assert st["packed_cells"] == 0 and st["cells"] > 0, (name, st)
    assert worst > 0.99, worst


@pytest.mark.parametrize("seed", [1, 2, 4])
def test_mixed_length_bits_launch(oracle, seed):
    """One launch, one key layout: a read at max_n of a scaled scoring (the largest LB, the tightest score field), short reads
    whose own LB is smaller (they run widened to the launch's LB), and a read past the edge (wide).  Same chains as the oracle
    and as each read aligned alone, also with 1 and 2 reads in flight (other launch splits)."""
    kw, contigs, edge, past, N = keyedge.headroom_case(seed, 8, seed % 4, n_edge=3000)
    m_max = max(len(c) for c in contigs)
    rng = random.Random(seed)
    short = [keyedge.exact_len(rng, edge[0][rng.randrange(0, N // 2):], rng.randint(10, 200)) for _ in range(5)]
    reads = [short[0], edge[0]] + short[1:3] + [past] + short[3:]
    LB = keyedge.plan(kw, N, m_max, 8)
    assert keyedge.headroom(kw, N, m_max, 8) > 0.9
    assert all(keyedge.plan(kw, len(r), m_max, 8) < LB for r in short) and not keyedge.accepted(kw, N + 1, m_max, 8)
    named = _named(contigs)
    rows = sum(len(c) for c in contigs) * (2 if kw["double_strand"] else 1)
    for raw in (True, False):
        exp = _oracle(oracle, kw, named, reads, raw)
        alone = [_gpu(kw, named, [r], raw)[0][0] for r in reads]
        compare(alone, exp, f"alone raw {raw} {kw}")
        for inflight in (0, 1, 2):
            got, st = _gpu(kw, named, reads, raw, max_inflight=inflight)
            compare(got, exp, f"mixed raw {raw} inflight {inflight} {kw}")
            if raw:   # every read but the past-edge one packed, that one wide (a chunk re-run with a larger ops buffer counts again)
                assert st["packed_cells"] >= rows * sum(len(r) for r in reads if r is not past), st
                assert st["cells"] - st["packed_cells"] >= rows * len(past), st
            assert 0 < st["packed_cells"] < st["cells"], st


def _scaled_pair(kw, named, reads, k, raw=False):
    got1, st1 = _gpu(kw, named, reads, raw)
    gotk, stk = _gpu(keyedge.scale(kw, k), named, reads, raw)
    for r, (a, b) in enumerate(zip(got1, gotk)):
        assert len(a) == len(b), f"read {r}: {len(a)} vs {len(b)} chains at k = {k}"
        for x, y in zip(a, b):
            assert keyedge.unscaled_key(y, k) == x.key(), f"read {r} at k = {k}:\n  k = 1 {x}\n  k     {y}"
    return st1, stk


def test_full_size_scale_invariance():
    """Config 2 at full size (64 noisy 10 kb reads, --double-strand --circular, production defaults: one CTA per read, quiet
    tiles) aligned with the default scores and with every score multiplied by the largest k that keeps its longest read
    packed: the same chains apart from score * k and the same work (cells, packed cells, tile-columns, quiet tile-columns,
    window re-runs) -- every quiet-tile and tracking decision compares multiples of k.  The same for a config-4-shaped 60 kb
    read at its own edge k, and for config-2 reads at k + 1, which run on the wide kernels.  (test_full_size_config2_vs_oracle
    checks the k = 1 chains of this batch against the oracle.)"""
    from stitch_b200 import synth
    kw, named, reads = synth.config(2, 64)
    m_max = max(len(s) for _, s in named)
    n_max = max(len(r) for r in reads)
    k = keyedge.edge_scale(kw, n_max, m_max, 8)
    assert k >= 2 and keyedge.headroom(keyedge.scale(kw, k), n_max, m_max, 8) > 0.9
    st1, stk = _scaled_pair(kw, named, reads, k)
    assert st1["packed_cells"] == st1["cells"] and st1["quiet_tile_columns"] > 0, st1
    assert stk == st1, (k, st1, stk)
    # k + 1: the longest reads go wide (raw: one fill per read)
    wide = sorted(range(len(reads)), key=lambda r: -len(reads[r]))[:6]
    sub = [reads[r] for r in wide]
    assert not any(keyedge.accepted(keyedge.scale(kw, k + 1), len(r), m_max, 8) for r in sub)
    st1, stw = _scaled_pair(kw, named, sub, k + 1, raw=True)
    assert st1["packed_cells"] == st1["cells"] and stw["packed_cells"] == 0 and stw["cells"] >= st1["cells"], (st1, stw)
    # a config-4-shaped read: 60 kb, 12 exact segments of 50 x 20 kb contigs, both strands
    rng = random.Random(7)
    contigs = [gen.rand_seq(rng, 20000) for _ in range(50)]
    segs = []
    for _ in range(12):
        c = rng.randrange(50)
        s = rng.randrange(0, 20000 - 5000)
        segs.append(gen.revcomp(contigs[c][s:s + 5000]) if rng.random() < 0.5 else contigs[c][s:s + 5000])
    read = b"".join(segs)
    kw4 = dict(double_strand=True)
    k4 = keyedge.edge_scale(kw4, len(read), 20000, 8)
    assert k4 >= 2 and keyedge.headroom(keyedge.scale(kw4, k4), len(read), 20000, 8) > 0.8
    st1, stk = _scaled_pair(kw4, _named(contigs), [read], k4)
    assert st1["packed_cells"] == st1["cells"] and stk == st1, (k4, st1, stk)
