"""Pre-alignment with the banded scoring (stitch_opts.pre_align_scoring = STITCH_PREALIGN_BANDED, prealign_core.h): the
score of a contig-strand is the best local affine-gap alignment inside the band of 2 W diagonals around its best pair of
k-mer bins, not the bases its exact k-mer hits cover.

CPU tier: the definition restated independently in Python and compared with the library over the CPU emulator (whose
backend scores k-mers only, so the host layer runs the sequential statement host_common.hpp::prealign_sequential, which
calls pre_banded_score), the case the scoring exists for (a segment whose k-mers are broken up by substitutions), the
pre-alignment contract of test_prealign.py in banded mode, the option and the CLI.  GPU tier: the CUDA kernel's selections
and scores equal the emulator's for band widths from 1 to 300 and at the edges of the window, the config-3 table, and the
k-mer scoring unchanged."""
import os
import random
import subprocess

import pytest

import gen
import test_prealign as tp
from stitch_b200._abi import make_opts
from test_emul_parity import emul_lib  # noqa: F401

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "stitch_b200", "stitch-b200")
SRC = os.path.join(ROOT, "stitch_b200", "csrc", "stitch_align_cli.cpp")
NEG = float("-inf")


# ---- the definition, restated ----------------------------------------------------------------------------------------
def py_need(min_score, match, K):
    need = 1 if match <= 0 else max(1, -(-min_score // match) - K + 1)
    return need, max(1, -(-need // 2))


def py_hits(read, strand, K):
    """(read position, strand position) of every pair of equal k-mers holding only ACGT."""
    where = {}
    for p in range(len(strand) - K + 1):
        where.setdefault(strand[p:p + K], []).append(p)
    return [(j, p) for j in range(len(read) - K + 1) if set(read[j:j + K]) <= set(b"ACGT")
            for p in where.get(read[j:j + K], ())]


def py_window(hits, n, W):
    """Diagonals [dlo, dhi) of the best pair of bins (lowest bin on ties)."""
    cnt = {}
    for j, p in hits:
        b = (p - j + n) // W
        cnt[b] = cnt.get(b, 0) + 1
    best = max(cnt.get(b, 0) + cnt.get(b + 1, 0) for b in range(0, max(cnt) + 1))
    bstar = min(b for b in range(0, max(cnt) + 1) if cnt.get(b, 0) + cnt.get(b + 1, 0) == best)
    return bstar * W - n, (bstar + 2) * W - n


def py_gotoh(read, strand, dlo, dhi, match, mismatch, o, e):
    """Smith-Waterman with affine gaps (a gap of length L costs o + L e) over the cells (i, q), 1-based, with
    dlo <= q - i < dhi; cells outside are not part of any alignment."""
    n, m = len(read), len(strand)
    H, E, F = {}, {}, {}
    best = 0
    for i in range(1, n + 1):
        for q in range(max(1, i + dlo), min(m, i + dhi - 1) + 1):
            e_ = max(H[i, q - 1] + o + e, E[i, q - 1] + e) if (i, q - 1) in H else NEG
            f_ = max(H[i - 1, q] + o + e, F[i - 1, q] + e) if (i - 1, q) in H else NEG
            d = H.get((i - 1, q - 1), 0) + (match if read[i - 1] == strand[q - 1] else mismatch)
            H[i, q], E[i, q], F[i, q] = max(0, d, e_, f_), e_, f_
            best = max(best, H[i, q])
    return best


def py_prealign_score(read, strand, kw):
    """Score of the one strand under the banded scoring, or None when it is not a candidate."""
    K, W = kw["kmer_size"], kw["band_width"]
    _, need_b = py_need(kw["pre_align_min_score"], kw["match_score"], K)
    hits = py_hits(read, strand, K)
    if len(hits) < need_b:
        return None
    dlo, dhi = py_window(hits, len(read), W)
    return py_gotoh(read, strand, dlo, dhi, kw["match_score"], kw["mismatch_score"], kw["gap_open"], kw["gap_extend"])


def banded(kw):
    return dict(kw, pre_align_scoring="banded")


def test_banded_score_equals_restatement(emul_lib):
    rng = random.Random(2024)
    n_scored = 0
    for case in range(200):
        contig = gen.rand_seq(rng, rng.randint(40, 300))
        if case % 5 == 0:
            contig = contig[:10] + b"N" + contig[11:]
        kind = case % 4
        if kind == 3:
            read = gen.rand_seq(rng, rng.randint(20, 300))
        else:
            a = rng.randrange(len(contig))
            b = min(len(contig), a + rng.randint(20, 300))
            read = gen.noisy(rng, contig[a:b], sub=0.05, ins=0.02, dele=0.02) or gen.rand_seq(rng, 20)
            read = (gen.rand_seq(rng, rng.randint(0, 30)) + read) if kind == 1 else read
            read = read[:300] if len(read) >= 20 else read + gen.rand_seq(rng, 20 - len(read))
        if case % 3 == 0:
            t = rng.randrange(len(read))
            read = read[:t] + b"N" + read[t + 1:]
        kw = dict(pre_align=True, kmer_size=rng.randint(4, 8), band_width=rng.randint(1, 40), pre_align_min_score=1,
                  match_score=rng.randint(1, 3), mismatch_score=-rng.randint(1, 5), gap_open=-rng.randint(0, 6),
                  gap_extend=-rng.randint(1, 3))
        exp = py_prealign_score(read, contig, kw)
        e = emul_lib.EmulAligners(make_opts(**banded(kw)), [("c0", contig)], strip=8)
        sel, best = e.prealign_batch([read])
        e.close()
        if exp is None or exp < 1:
            assert (sel, best) == ([[]], [0]), (case, kw, exp)
        else:
            assert (sel, best) == ([[0]], [exp]), (case, kw)
            n_scored += 1
    assert n_scored >= 120


# ---- the case the banded scoring is for -------------------------------------------------------------------------------
def test_substitutions_break_kmers_but_not_the_alignment(emul_lib):
    """150 bases of a contig with a substitution every 18 bases: 48 intact 12-mers are fewer than the 89 the k-mer scoring
    needs for -s 100, but the alignment scores 142 - 8 x 4 = 110."""
    rng = random.Random(77)
    contig = gen.rand_seq(rng, 600)
    seg = bytearray(contig[200:350])
    for off in range(17, 150, 18):
        seg[off] = rng.choice([b for b in b"ACGT" if b != seg[off]])
    read = bytes(seg)
    K = 12
    assert len(range(17, 150, 18)) == 8
    kmers = [read[j:j + K] for j in range(len(read) - K + 1)]
    table = [contig[p:p + K] for p in range(len(contig) - K + 1)]
    assert sum(table.count(k) for k in kmers) == 48 and all(table.count(k) <= 1 for k in kmers)
    assert py_need(100, 1, K) == (89, 45)
    named = [("c0", contig)]
    for scoring, n_chains, xs in (("kmer", 0, None), ("banded", 1, 110)):
        e = emul_lib.EmulAligners(make_opts(pre_align=True, pre_align_scoring=scoring), named, strip=8)
        chains, sam = e.batch_sam([read], ["r"], None, None)
        assert len(chains[0]) == n_chains and e.last_prealign_scores == [xs], scoring
        if xs is None:
            assert sam[0] == ["r\t4\t*\t0\t0\t*\t*\t0\t0\t" + read.decode() + "\t*"]
        else:
            assert "\txs:i:110\t" in sam[0][0] and sam[0][0].split("\t")[2] == "c0"
        e.close()


# ---- the pre-alignment contract in banded mode ------------------------------------------------------------------------
def test_banded_subset_equals_oracle_on_the_same_subset(oracle, emul_lib):
    kw = banded(dict(double_strand=True, pre_align=True, kmer_size=8, band_width=20, pre_align_min_score=40))
    contigs, reads, truth = tp.make_case(11, 12, 300, 600, 6, 400, 3)
    tp.check_subset_mode(oracle, tp.emul_maker(emul_lib), kw, contigs, reads, truth)
    kw = banded(dict(circular=True, suboptimal=True, pre_align=True, band_width=50, pre_align_min_score=60))
    contigs, reads, truth = tp.make_case(12, 8, 300, 600, 4, 500, 2, flips=False)
    tp.check_subset_mode(oracle, tp.emul_maker(emul_lib), kw, contigs, reads, truth)


def test_banded_table_beyond_256_contig_strands(oracle, emul_lib):
    kw = banded(dict(double_strand=True, pre_align=True, kmer_size=10, band_width=30, pre_align_min_score=50))
    contigs, reads, truth = tp.make_case(13, 300, 120, 260, 5, 360, 3)
    sel, _ = tp.check_subset_mode(oracle, tp.emul_maker(emul_lib), kw, contigs, reads, truth)
    assert any(max(s) >= 256 for s in sel)


def test_banded_reads_that_reach_the_score_nowhere_are_not_aligned(emul_lib):
    rng = random.Random(5)
    contigs = [gen.rand_seq(rng, 400) for _ in range(4)]
    named = [(f"c{k}", s) for k, s in enumerate(contigs)]
    good = contigs[2][50:350]
    junk = gen.rand_seq(rng, 300)
    short = contigs[1][10:60]                                   # 50 matching bases < min score 100
    e = emul_lib.EmulAligners(make_opts(**banded(dict(double_strand=True, pre_align=True))), named, strip=8)
    chains, sam = e.batch_sam([good, junk, short], ["g", "j", "s"], None, None)
    assert [len(c) for c in chains] == [1, 0, 0]
    assert e.last_prealign_scores == [300, None, None]
    assert sam[1] == ["j\t4\t*\t0\t0\t*\t*\t0\t0\t" + junk.decode() + "\t*"]
    assert "\txs:i:300\t" in sam[0][0]
    e.close()


def test_banded_without_subset_contigs_scores_the_first_passing_target(oracle, emul_lib):
    rng = random.Random(6)
    contigs = [gen.rand_seq(rng, 500) for _ in range(5)]
    named = [(f"c{k}", s) for k, s in enumerate(contigs)]
    read = contigs[3][100:300] + gen.revcomp(contigs[1][50:400])       # targets 1 (reverse, 350 b) and 3 (forward, 200 b) pass
    kw = banded(dict(double_strand=True, pre_align=True, pre_align_subset_contigs=False))
    e = emul_lib.EmulAligners(make_opts(**kw), named, strip=8)
    got = e.batch([read, gen.rand_seq(rng, 200)])
    assert e.last_prealign_scores == [350, None] and got[1] == []
    exp, _ = oracle.OracleAligners(make_opts(double_strand=True), named).batch([read], raw=False)
    assert [a.key() for a in got[0]] == [a.key() for a in exp[0]]
    e.close()


# ---- option and CLI -------------------------------------------------------------------------------------------------
def test_scoring_option_is_validated(emul_lib):
    named = [("c0", b"ACGT" * 20)]
    with pytest.raises(emul_lib.EmulError, match=r"create failed \(-1\).*pre-alignment scoring"):
        emul_lib.EmulAligners(make_opts(pre_align=True, pre_align_scoring=2), named, strip=8)
    with pytest.raises(ValueError):
        make_opts(pre_align_scoring="smith-waterman")
    assert make_opts().pre_align_scoring == 0 and make_opts(pre_align_scoring="banded").pre_align_scoring == 1
    import stitch_b200
    assert stitch_b200.Builder(pre_align_scoring="banded").build_options().pre_align_scoring == 1
    assert stitch_b200.Builder().build_options().pre_align_scoring == 0


@pytest.fixture(scope="module")
def cli_env():
    import emul_lib
    emul_lib.build()
    if not os.path.exists(CLI) or os.path.getmtime(CLI) < os.path.getmtime(SRC):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-o", CLI, SRC, "-ldl", "-lz"])
    return dict(os.environ, STITCH_B200_LIB=os.path.join(ROOT, "tests", "emul", "libemul_s8.so"), STITCH_B200_PREFIX="emul_")


def test_cli_banded_scoring(cli_env, tmp_path):
    import emul_lib
    rng = random.Random(92)
    contigs = [gen.rand_seq(rng, rng.randint(300, 500)) for _ in range(6)]
    reads = [gen.chimeric_read(rng, contigs, rng.randint(150, 300), rng.randint(1, 2), strands=True) for _ in range(6)]
    reads.insert(2, gen.rand_seq(rng, 120))
    heads = [f"q{k}" for k in range(len(reads))]
    ref, fa = tmp_path / "ref.fa", tmp_path / "reads.fa"
    ref.write_text("".join(f">c{k}\n{c.decode()}\n" for k, c in enumerate(contigs)))
    fa.write_text("".join(f">{h}\n{r.decode()}\n" for h, r in zip(heads, reads)))
    kw = banded(dict(double_strand=True, pre_align=True, kmer_size=9, band_width=25, pre_align_min_score=45))
    e = emul_lib.EmulAligners(make_opts(**kw), [(f"c{k}", c) for k, c in enumerate(contigs)], strip=8)
    _, exp = e.batch_sam(reads, heads, None, None)
    e.close()
    args = [CLI, "align", "-a", str(fa), "-r", str(ref), "-d", "-p", "-k", "9", "-w", "25", "-s", "45", "--sam", "--batch", "3"]
    for opt in (["--pre-align-scoring", "banded"], ["--pre-align-scoring=banded"]):
        p = subprocess.run(args + opt, env=cli_env, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        assert p.returncode == 0, p.stderr.decode()
        got = [l for l in p.stdout.decode().splitlines() if not l.startswith("@")]
        assert got == [l for per_read in exp for l in per_read]
        assert any("\txs:i:" in l for l in got) and any(l.split("\t")[1] == "4" for l in got)
    p = subprocess.run(args + ["--pre-align-scoring", "sw"], env=cli_env, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert p.returncode != 0 and b"unknown --pre-align-scoring sw" in p.stderr
    p = subprocess.run([CLI, "align", "--help"], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert b"--pre-align-scoring <kmer|banded>" in p.stderr


# ---- GPU tier -------------------------------------------------------------------------------------------------------
GPU_SHAPES = ((11, dict(double_strand=True, pre_align=True, kmer_size=8, band_width=20, pre_align_min_score=40), (12, 300, 600, 6, 400, 3)),
              (13, dict(double_strand=True, pre_align=True, kmer_size=10, band_width=30, pre_align_min_score=50), (300, 120, 260, 5, 360, 3)),
              (14, dict(double_strand=True, circular=True, pre_align=True, kmer_size=15, band_width=50, pre_align_min_score=80), (40, 400, 900, 5, 900, 3)))


def _gpu_vs_emul(kw, contigs, reads):
    import emul_lib
    from test_gpu_parity import gpu_aligners
    named = [(f"c{k}", s) for k, s in enumerate(contigs)]
    al = gpu_aligners(kw, named)
    got = al.prealign_batch(reads)
    al.close()
    e = emul_lib.EmulAligners(make_opts(**kw), named, strip=8)
    exp = e.prealign_batch(reads)
    e.close()
    assert got == exp, kw
    return got


def _edge_case(seed):
    """Short contigs (shorter than the window), reads longer than their contig (the window clipped at both ends of both
    sequences), reads shorter than k, reads with N."""
    rng = random.Random(seed)
    contigs = [gen.rand_seq(rng, rng.randint(25, 70)) for _ in range(6)] + [gen.rand_seq(rng, rng.randint(200, 700)) for _ in range(6)]
    reads = []
    for k in range(12):
        c = contigs[k]
        reads.append(gen.rand_seq(rng, rng.randint(0, 40)) + gen.noisy(rng, c) + gen.rand_seq(rng, rng.randint(0, 40)))
    reads += [contigs[7][:5], contigs[8][100:104], contigs[9][:1]]          # shorter than k = 6
    for k in range(6):
        r = bytearray(gen.noisy(rng, contigs[6 + k][rng.randrange(50):]))
        for _ in range(3):
            r[rng.randrange(len(r))] = ord("N")
        reads.append(bytes(r))
    reads.append(b"N" * 60)
    return contigs, [r for r in reads if r]


@pytest.mark.gpu
@pytest.mark.parametrize("scoring", ["banded", "kmer"])
def test_kernel_equals_emulator(oracle, scoring):
    """Banded: selections and scores of the CUDA kernel equal the emulator's on the shapes of test_prealign_on_gpu, for band
    widths of one partial chunk (1, 16, 17, 50), two (100) and five (300) chunks of 128 cells, and at the window's edges.
    K-mer: the same inputs give what the k-mer kernel gives (test_prealign_on_gpu's expectations)."""
    for seed, kw, shape in GPU_SHAPES:
        kw = dict(kw, pre_align_scoring=scoring)
        contigs, reads, truth = tp.make_case(seed, *shape)
        sel, best = tp.check_subset_mode(oracle, _GpuPre, kw, contigs, reads, truth)
        assert (sel, best) == _gpu_vs_emul(kw, contigs, reads)
        for W in (1, 16, 17, 50, 100, 300):
            _gpu_vs_emul(dict(kw, band_width=W), contigs, reads)
    for W in (1, 17, 50, 100, 300):
        contigs, reads = _edge_case(W)
        sel, best = _gpu_vs_emul(dict(double_strand=True, pre_align=True, kmer_size=6, band_width=W, pre_align_min_score=15,
                                      pre_align_scoring=scoring), contigs, reads)
        assert sum(map(len, sel)) > len(reads) // 2
    if scoring == "kmer":
        rng = random.Random(5)
        from test_gpu_parity import gpu_aligners
        contigs = [gen.rand_seq(rng, 400) for _ in range(4)]
        al = gpu_aligners(dict(double_strand=True, pre_align=True), [(f"c{k}", s) for k, s in enumerate(contigs)])
        chains = al.align_batch([contigs[2][50:350], gen.rand_seq(rng, 300), contigs[1][10:60]])
        assert [len(c) for c in chains] == [1, 0, 0] and al.last_prealign_scores == [300, None, None]
        al.close()


class _GpuPre:
    """The shape tests/test_prealign.py's checks expect, over the CUDA library."""
    def __init__(self, kw, named):
        from test_gpu_parity import gpu_aligners
        self.al = gpu_aligners(kw, named)

    def batch(self, reads):
        out = self.al.align_batch(reads)
        self.last_prealign_scores = self.al.last_prealign_scores
        return out

    def prealign_batch(self, reads):
        return self.al.prealign_batch(reads)

    def close(self):
        self.al.close()


@pytest.mark.gpu
def test_config3_full_table_banded(oracle):
    """BASELINE config 3 at its stated scale (4 000 contig-strands, reads of 5-20 kb, `-d -p -x`) in banded mode: chains
    equal the oracle's on the selected subsets, and every contig-strand the k-mer scoring finds for a read's segments is
    found by the banded scoring too (recall at least the k-mer scoring's)."""
    import numpy as np
    from stitch_b200 import synth
    from test_gpu_parity import gpu_aligners
    rng = np.random.default_rng(20243)
    contigs = [c.tobytes() for c in synth.make_contigs(rng, 2000, 5000, 10000)]
    reads, truth = [], []
    for _ in range(48):
        t = []
        reads.append(synth.make_read(rng, [np.frombuffer(c, dtype=np.uint8) for c in contigs], int(rng.integers(5000, 20001)), 3, 8,
                                     strands=True, truth=t).tobytes())
        truth.append(sorted(set(t)))
    named = [(f"c{k}", s) for k, s in enumerate(contigs)]
    recall = {}
    for scoring in ("kmer", "banded"):
        kw = dict(double_strand=True, pre_align=True, pre_align_scoring=scoring)
        al = gpu_aligners(kw, named)
        got = al.align_batch(reads)
        pre = al.last_prealign_scores
        sel, best = al.prealign_batch(reads)
        al.close()
        for r in range(len(reads)):
            assert len(sel[r]) <= 32 and pre[r] == best[r] and len(got[r]) == 1
        recall[scoring] = sum(1 for r in range(len(reads)) for c in truth[r] if c in sel[r])
        if scoring == "banded":
            for r in sorted(range(len(reads)), key=lambda r: (len(reads[r]) * len(sel[r]), r))[:3]:
                oracle.set_checker_layout(True)
                try:
                    exp = tp.reduced_oracle(oracle, kw, contigs, reads[r], sel[r])
                finally:
                    oracle.set_checker_layout(False)
                assert [a.key() for a in got[r]] == [a.key() for a in exp], r
    assert recall["banded"] >= recall["kmer"], recall
