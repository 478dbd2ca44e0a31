"""stitch_b200 — B200-native drop-in for the alignment hot path of fulcrumgenomics/stitch.

The product is the CUDA library behind include/stitch_b200.h (stitch_b200/csrc).  This package is
the thin ctypes host mirror of the reference's aligner API for that path, with the reference's
names and argument meaning (fg-stitch-lib/src/align/aligners/mod.rs):

    Builder().mode("local").double_strand(True)...          # Options + derive_builder, :65-116
    aligners = builder.build_aligners(target_seqs)          # :171
    chains, prealign_score = aligners.align(record)         # :237  (one read)
    per_read = aligners.align_batch(reads)                  # the batched form the GPU wants

No compute happens in Python and nothing here touches oracle/.
"""
import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence

from . import _abi
from ._abi import (MODE_GLOBAL, MODE_LOCAL, MODE_QUERY_LOCAL, MODE_TARGET_LOCAL, StitchStats,
                   make_contigs, make_opts, pack_reads)
from .alignment import Alignment

__all__ = ["Builder", "Aligners", "TargetSeq", "FastxOwnedRecord", "Alignment", "StitchError",
           "reverse_complement", "MODE_LOCAL", "MODE_QUERY_LOCAL", "MODE_TARGET_LOCAL", "MODE_GLOBAL"]

_COMP = bytes.maketrans(b"AGCTYRWSKMDVHBNagctyrwskmdvhbn", b"TCGARYWSMKHBDVNtcgarywsmkhbdvn")


def reverse_complement(seq: bytes) -> bytes:
    """util/dna.rs:5-41 (IUPAC complement table, unknown bytes unchanged)."""
    return bytes(seq).translate(_COMP)[::-1]


class StitchError(RuntimeError):
    """Raised where the reference panics / returns Err."""


@dataclass
class TargetSeq:
    """util/target_seq.rs:15-48: upper-cased forward bases (+ revcomp derived by the library)."""
    name: str
    fwd: bytes
    circular: bool = False

    def __post_init__(self):
        self.fwd = bytes(self.fwd).upper()

    @property
    def revcomp(self) -> bytes:
        return reverse_complement(self.fwd)

    def __len__(self):
        return len(self.fwd)


@dataclass
class FastxOwnedRecord:
    """align/io.rs:39-70."""
    head: bytes
    seq: bytes
    qual: Optional[bytes] = None

    def seq_upper_case(self) -> bytes:
        return bytes(self.seq).upper()


class Builder:
    """Options builder with the reference's field names and defaults (aligners/mod.rs:65-116)."""
    _FIELDS = dict(mode=MODE_LOCAL, match_score=1, mismatch_score=-4, gap_open=-6, gap_extend=-2,
                   default_jump_score=-10, jump_score_same_contig_and_strand=None,
                   jump_score_same_contig_opposite_strand=None, jump_score_inter_contig=None,
                   double_strand=False, circular=False, circular_slop=20, suboptimal=False,
                   suboptimal_pct=20.0, pre_align=False, pre_align_subset_contigs=True, kmer_size=12, band_width=50,
                   pre_align_min_score=100, pre_align_scoring="kmer")

    def __init__(self, **kw):
        self._v = dict(self._FIELDS)
        for k, v in kw.items():
            getattr(self, k)(v)

    def __getattr__(self, name):
        if name in Builder._FIELDS:
            def setter(value):
                self._v[name] = value
                return self
            return setter
        raise AttributeError(name)

    def build_options(self) -> _abi.StitchOpts:
        return make_opts(**self._v)

    def build_aligners(self, target_seqs: Sequence[TargetSeq], device: int = 0) -> "Aligners":
        return Aligners(self.build_options(), target_seqs, device)


class Aligners:
    """One instance per host thread / GPU, like the reference's `Aligners` (mod.rs:227-234)."""

    def __init__(self, opts: _abi.StitchOpts, target_seqs: Sequence[TargetSeq], device: int = 0):
        from . import _lib
        self._lib = _lib.load()
        self.opts = opts
        self.target_seqs = list(target_seqs)
        arr, self._keep = make_contigs([(t.name, t.fwd) for t in self.target_seqs])
        h = C.c_void_p()
        rc = self._lib.stitch_create(C.byref(opts), arr, len(self.target_seqs), device, C.byref(h))
        if rc != 0:
            msg = self._lib.stitch_last_error(None)
            raise StitchError(f"stitch_create failed ({rc}): {msg.decode() if msg else ''}")
        self._h = h

    # -- batched entry points -------------------------------------------------------------
    def _run(self, fn, reads, subsets):
        from . import _lib
        buf, offs = pack_reads(reads)
        words, stride = None, 0
        if subsets is not None:
            n_strands = len(self.target_seqs) * (2 if self.opts.double_strand else 1)
            stride = (n_strands + 31) // 32
            words = (C.c_uint32 * (stride * len(reads)))()
            for r, sub in enumerate(subsets):
                for c in (sub or ()):
                    words[r * stride + c // 32] |= 1 << (c % 32)
        res = C.c_void_p()
        rc = fn(self._h, buf, offs, len(reads), words, stride, C.byref(res))
        if rc != 0:
            raise StitchError(f"{fn.__name__} failed ({rc}): {self.last_error()}")
        try:
            out = _lib.read_results(self._lib, _lib.PRODUCT_RESULTS, res)
            self.last_prealign_scores = _lib.read_prealign(self._lib, "stitch_", res, len(reads))
            return out
        finally:
            self._lib.stitch_free_results(res)

    def align_batch_sam(self, reads: Sequence[bytes], headers: Sequence[str], quals=None, sam_opts=None, subsets=None):
        """Aligners::align followed by SamRecordFormatter::format (aligners/mod.rs:622-972) for each read:
        -> (chains per read, SAM text lines per read)."""
        from . import _lib
        buf, offs = pack_reads(reads)
        res = C.c_void_p()
        words, stride = None, 0
        if subsets is not None:
            n_strands = len(self.target_seqs) * (2 if self.opts.double_strand else 1)
            stride = (n_strands + 31) // 32
            words = (C.c_uint32 * (stride * len(reads)))()
            for r, sub in enumerate(subsets):
                for c in (sub or ()):
                    words[r * stride + c // 32] |= 1 << (c % 32)
        rc = self._lib.stitch_align_batch(self._h, buf, offs, len(reads), words, stride, C.byref(res))
        if rc != 0:
            raise StitchError(f"stitch_align_batch failed ({rc}): {self.last_error()}")
        try:
            chains = _lib.read_results(self._lib, _lib.PRODUCT_RESULTS, res)
            pre = _lib.read_prealign(self._lib, "stitch_", res, len(reads))
            self.last_prealign_scores = pre
            sam = [_lib.format_sam(self._lib, "stitch_", self._h, res, r, headers[r], bytes(reads[r]),
                                   None if quals is None else quals[r], pre[r], sam_opts) for r in range(len(reads))]
            return chains, sam
        finally:
            self._lib.stitch_free_results(res)

    def align_batch(self, reads: Sequence[bytes], subsets=None) -> List[List[Alignment]]:
        """Aligners::align for each read (chains per read; empty list = unmapped)."""
        return self._run(self._lib.stitch_align_batch, reads, subsets)

    def custom_batch(self, reads: Sequence[bytes], subsets=None) -> List[List[Alignment]]:
        """MultiContigAligner::custom_with_subset for each read (one raw chain, clips kept)."""
        return self._run(self._lib.stitch_custom_batch, reads, subsets)

    # -- reference-shaped single-read call ---------------------------------------------------
    def align(self, record, target_seqs=None, target_hashes=None):
        """(Vec<Alignment>, Option<i32>) of Aligners::align (with opts.pre_align: the library's own pre-alignment)."""
        seq = record.seq if isinstance(record, FastxOwnedRecord) else bytes(record)
        chains = self.align_batch([seq])[0]
        return chains, self.last_prealign_scores[0]

    def prealign_batch(self, reads: Sequence[bytes]):
        """The pre-alignment alone: (selected contig-strands per read, best score per read)."""
        from . import _lib
        n_strands = len(self.target_seqs) * (2 if self.opts.double_strand else 1)
        return _lib.prealign_batch(self._lib, "stitch_", self._h, reads, n_strands)

    def stats(self) -> StitchStats:
        s = StitchStats()
        self._lib.stitch_get_stats(self._h, C.byref(s))
        return s

    def set_max_inflight(self, n: int):
        self._lib.stitch_set_max_inflight(self._h, int(n))

    def last_error(self) -> str:
        msg = self._lib.stitch_last_error(self._h)
        return msg.decode() if msg else ""

    def close(self):
        if getattr(self, "_h", None):
            self._lib.stitch_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
