"""ctypes mirror of include/stitch_b200.h (records only; no behaviour)."""
import ctypes as C

MODE_LOCAL, MODE_QUERY_LOCAL, MODE_TARGET_LOCAL, MODE_GLOBAL = 0, 1, 2, 3
OP_MATCH, OP_SUBST, OP_DEL, OP_INS, OP_XCLIP, OP_YCLIP, OP_XJUMP, OP_YJUMP = range(8)

PREALIGN_KMER, PREALIGN_BANDED = 0, 1
PREALIGN_SCORING = {"kmer": PREALIGN_KMER, "banded": PREALIGN_BANDED}   # stitch_opts.pre_align_scoring

MODE_NAMES = {
    # AlignmentMode::from_str, fg-stitch-lib/src/align/aligners/constants.rs:121-136
    "local": MODE_LOCAL,
    "query-local": MODE_QUERY_LOCAL, "query_local": MODE_QUERY_LOCAL, "querylocal": MODE_QUERY_LOCAL, "query": MODE_QUERY_LOCAL,
    "target-local": MODE_TARGET_LOCAL, "target_local": MODE_TARGET_LOCAL, "targetlocal": MODE_TARGET_LOCAL, "target": MODE_TARGET_LOCAL,
    "global": MODE_GLOBAL,
}


class StitchOpts(C.Structure):
    _fields_ = [
        ("mode", C.c_int32), ("match_score", C.c_int32), ("mismatch_score", C.c_int32),
        ("gap_open", C.c_int32), ("gap_extend", C.c_int32),
        ("jump_same", C.c_int32), ("jump_opp", C.c_int32), ("jump_inter", C.c_int32),
        ("double_strand", C.c_uint8), ("circular", C.c_uint8), ("suboptimal", C.c_uint8), ("reserved0", C.c_uint8),
        ("circular_slop", C.c_uint32), ("suboptimal_pct", C.c_float),
        ("pre_align", C.c_uint8), ("pre_align_subset_contigs", C.c_uint8), ("pre_align_scoring", C.c_uint8),
        ("reserved1", C.c_uint8 * 1),
        ("kmer_size", C.c_uint32), ("band_width", C.c_uint32), ("pre_align_min_score", C.c_int32),
    ]


class StitchContig(C.Structure):
    _fields_ = [("name", C.c_char_p), ("fwd", C.POINTER(C.c_uint8)), ("len", C.c_uint32)]


class StitchChain(C.Structure):
    _fields_ = [
        ("score", C.c_int32), ("xstart", C.c_uint32), ("xend", C.c_uint32), ("ystart", C.c_uint32),
        ("yend", C.c_uint32), ("xlen", C.c_uint32), ("ylen", C.c_uint32),
        ("start_contig_idx", C.c_uint32), ("end_contig_idx", C.c_uint32), ("length", C.c_uint32),
        ("n_ops", C.c_uint32), ("reserved", C.c_uint32), ("ops_offset", C.c_uint64),
    ]


class StitchOp(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("a", C.c_uint32), ("b", C.c_uint32)]


class StitchStats(C.Structure):
    _fields_ = [
        ("cells", C.c_uint64), ("fills", C.c_uint64), ("kernel_launches", C.c_uint64),
        ("fill_ms", C.c_double), ("traceback_ms", C.c_double), ("total_ms", C.c_double),
        ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("traceback_bytes", C.c_uint64),
        ("packed_fill_ms", C.c_double), ("wide_fill_ms", C.c_double), ("redo_fill_ms", C.c_double),
        ("packed_cells", C.c_uint64), ("redo_fills", C.c_uint64), ("tail_fill_ms", C.c_double), ("packed_launches", C.c_uint64),
        ("tile_columns", C.c_uint64), ("quiet_tile_columns", C.c_uint64),
        ("prealign_ms", C.c_double), ("prealign_reads", C.c_uint64),
    ]


class StitchSamOpts(C.Structure):
    _fields_ = [("soft_clip", C.c_uint8), ("use_eq_and_x", C.c_uint8), ("pick_primary", C.c_uint8), ("filter_secondary", C.c_uint8),
                ("filter_secondary_pct", C.c_float)]


def make_opts(mode=MODE_LOCAL, match_score=1, mismatch_score=-4, gap_open=-6, gap_extend=-2,
              default_jump_score=-10, jump_score_same_contig_and_strand=None,
              jump_score_same_contig_opposite_strand=None, jump_score_inter_contig=None,
              double_strand=False, circular=False, circular_slop=20, suboptimal=False,
              suboptimal_pct=20.0, pre_align=False, pre_align_subset_contigs=True, kmer_size=12, band_width=50,
              pre_align_min_score=100, pre_align_scoring="kmer") -> StitchOpts:
    """Options with the reference's defaults (aligners/mod.rs:67-116, 143-152).  `pre_align_scoring`: "kmer" (default)
    or "banded" (stitch_b200/csrc/prealign_core.h); an int is passed through as it is."""
    if isinstance(mode, str):
        mode = MODE_NAMES[mode.lower()]
    if isinstance(pre_align_scoring, str):
        if pre_align_scoring not in PREALIGN_SCORING:
            raise ValueError(f"pre_align_scoring must be one of {sorted(PREALIGN_SCORING)}, got {pre_align_scoring!r}")
        pre_align_scoring = PREALIGN_SCORING[pre_align_scoring]
    pick = lambda v: default_jump_score if v is None else v
    return StitchOpts(
        mode=mode, match_score=match_score, mismatch_score=mismatch_score, gap_open=gap_open,
        gap_extend=gap_extend, jump_same=pick(jump_score_same_contig_and_strand),
        jump_opp=pick(jump_score_same_contig_opposite_strand), jump_inter=pick(jump_score_inter_contig),
        double_strand=int(bool(double_strand)), circular=int(bool(circular)), suboptimal=int(bool(suboptimal)),
        reserved0=0, circular_slop=int(circular_slop), suboptimal_pct=float(suboptimal_pct),
        pre_align=int(bool(pre_align)), pre_align_subset_contigs=int(bool(pre_align_subset_contigs)), kmer_size=int(kmer_size),
        band_width=int(band_width), pre_align_min_score=int(pre_align_min_score), pre_align_scoring=int(pre_align_scoring))


def make_contigs(contigs):
    """contigs: list of (name, bytes).  Returns (array, keepalive)."""
    arr = (StitchContig * len(contigs))()
    keep = []
    for k, (name, seq) in enumerate(contigs):
        seq = bytes(seq)
        buf = (C.c_uint8 * max(1, len(seq))).from_buffer_copy(seq if seq else b"\0")
        nm = name.encode() if isinstance(name, str) else bytes(name)
        keep.append((buf, nm))
        arr[k].name = nm
        arr[k].fwd = C.cast(buf, C.POINTER(C.c_uint8))
        arr[k].len = len(seq)
    return arr, keep


def pack_reads(reads):
    """reads: list of bytes -> (uint8 array, uint64 offsets array)."""
    offs = (C.c_uint64 * (len(reads) + 1))()
    total = 0
    for k, r in enumerate(reads):
        offs[k] = total
        total += len(r)
    offs[len(reads)] = total
    blob = b"".join(bytes(r) for r in reads)
    buf = (C.c_uint8 * max(1, total)).from_buffer_copy(blob if blob else b"\0")
    return buf, offs
