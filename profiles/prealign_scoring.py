"""Cost and recall of the two pre-alignment scorings (stitch_opts.pre_align_scoring) on BASELINE config 3.

Runs config-3 reads (synth.config(3, ...): 128 contigs x 2 strands, reads of 5-20 kb with 3-8 segments) through
stitch_prealign_batch with the k-mer and with the banded scoring and prints one JSON line per scoring:
  prealign_ms_per_read   stitch_stats.prealign_ms of one call over the reads (copies + kernel, CUDA events) / reads;
                         median, min and max over --repeats timed calls after --warmup untimed ones;
  align_ms_per_read      stitch_stats.total_ms / reads of stitch_align_batch with `-p -x` (pre-alignment, then the alignment
                         against the selected strands only) on the first --align-reads reads, after one untimed call;
  selected_per_read      mean number of selected contig-strands;
  recall                 share of the (read, contig-strand a segment was drawn from) pairs whose strand is selected.

    python profiles/prealign_scoring.py [--reads 1024] [--warmup 2] [--repeats 7] [--align-reads 128] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_name():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                           stderr=subprocess.DEVNULL, text=True, timeout=60)
        return q.stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=1024)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--align-reads", type=int, default=128)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import stitch_b200
    from stitch_b200 import synth
    truth = []
    kw, named, reads = synth.config(3, a.reads, truth=truth)
    targets = [stitch_b200.TargetSeq(n, s) for n, s in named]
    device = gpu_name()
    lines = []
    for scoring in ("kmer", "banded"):
        al = stitch_b200.Builder(**kw, pre_align=True, pre_align_scoring=scoring).build_aligners(targets)
        for _ in range(a.warmup):
            al.prealign_batch(reads)
        ms = []
        for _ in range(a.repeats):
            sel, best = al.prealign_batch(reads)   # the statistics cover the last call
            ms.append(al.stats().prealign_ms / len(reads))
        few = reads[:a.align_reads]
        al.align_batch(few)
        al.align_batch(few)
        st = al.stats()
        al.close()
        hit = sum(1 for r in range(len(reads)) for c in truth[r] if c in sel[r])
        lines.append(dict(
            scoring=scoring, config=3, reads=len(reads), contig_strands=2 * len(named), bases=sum(map(len, reads)),
            prealign_ms_per_read=statistics.median(ms), prealign_ms_per_read_min=min(ms), prealign_ms_per_read_max=max(ms),
            warmup=a.warmup, repeats=a.repeats, align_reads=len(few), align_ms_per_read=st.total_ms / len(few),
            align_prealign_ms_per_read=st.prealign_ms / len(few),
            selected_per_read=sum(map(len, sel)) / len(reads), unselected_reads=sum(1 for s in sel if not s),
            recall=hit / sum(len(t) for t in truth), device=device))
    text = "".join(json.dumps(l) + "\n" for l in lines)
    sys.stdout.write(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
