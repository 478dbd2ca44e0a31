/*
 * stitch_b200.h — C ABI of the B200-native jump-aware aligner.
 *
 * This is the drop-in boundary for the alignment hot path of fulcrumgenomics/stitch.
 * Every entry point names the reference interface it replaces (paths relative to the
 * reference checkout; LIB = fg-stitch-lib/src):
 *
 *   stitch_create        <-> Builder::build_aligners            LIB/align/aligners/mod.rs:171-211
 *                            (Options: mod.rs:65-116; contig order: forward contigs in FASTA
 *                             order, then, with double_strand, all reverse complements)
 *   stitch_align_batch   <-> Aligners::align, once per read     LIB/align/aligners/mod.rs:237-340
 *                            (which drives MultiContigAligner::custom_with_subset
 *                             multi_contig_aligner.rs:178, traceback_all :363, traceback_from :380,
 *                             realign_origin mod.rs:442 and Alignment::split_at_y alignment.rs:207)
 *   stitch_custom_batch  <-> MultiContigAligner::custom_with_subset (raw, clips kept)
 *                            LIB/align/aligners/multi_contig_aligner.rs:178-361
 *   stitch_results_*     <-> the returned (Vec<Alignment>, Option<i32>)   LIB/align/alignment.rs:16-51
 *   stitch_destroy       <-> drop(Aligners)
 *   stitch_last_error    <-> the panic / anyhow message of the reference (never unwinds over FFI)
 *
 * Plain pointers and sizes only; no C++ or torch types cross this boundary.  One stitch_ctx
 * per host thread / per GPU (the reference builds one `Aligners` per thread,
 * fg-stitch-cli/src/commands/align.rs:345-360).  Batches preserve input order.
 */
#ifndef STITCH_B200_H
#define STITCH_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* AlignmentMode, LIB/align/aligners/constants.rs:96-108 (Custom is rejected, mod.rs:129). */
enum { STITCH_MODE_LOCAL = 0, STITCH_MODE_QUERY_LOCAL = 1, STITCH_MODE_TARGET_LOCAL = 2, STITCH_MODE_GLOBAL = 3 };

/* stitch_opts.pre_align_scoring (definitions: stitch_b200/csrc/prealign_core.h).  KMER: the bases covered by exact k-mer
 * hits in the best band of 2 band_width diagonals.  BANDED: the best local affine-gap alignment inside that band. */
enum { STITCH_PREALIGN_KMER = 0, STITCH_PREALIGN_BANDED = 1 };

/* AlignmentOperation, LIB/align/aligners/constants.rs:20-29.  Runs of Match/Subst/Del/Ins are
 * run-length encoded: `a` is the run length.  Xclip/Yclip/Yjump: `a` is the length.
 * Xjump: `a` = contig index, `b` = 0-based contig offset the chain continues at. */
enum {
    STITCH_OP_MATCH = 0, STITCH_OP_SUBST = 1, STITCH_OP_DEL = 2, STITCH_OP_INS = 3,
    STITCH_OP_XCLIP = 4, STITCH_OP_YCLIP = 5, STITCH_OP_XJUMP = 6, STITCH_OP_YJUMP = 7
};

/* Error codes (negative).  The reference panics where these are returned. */
enum {
    STITCH_OK = 0,
    STITCH_ERR_INVALID = -1,   /* bad argument / option out of the supported range        */
    STITCH_ERR_CUDA = -2,      /* CUDA runtime failure (no CPU fallback exists)            */
    STITCH_ERR_NOMEM = -3,     /* device or host allocation failed                          */
    STITCH_ERR_LIMIT = -4,     /* > 256 contig-strands for ONE read, > 65536 in the table, contig >= 2^27 */
    STITCH_ERR_INTERNAL = -5   /* traceback reached a state the reference would panic on   */
};

/* Options consumed by the path: subset of Options, LIB/align/aligners/mod.rs:67-116. */
typedef struct stitch_opts {
    int32_t mode;                 /* STITCH_MODE_*                         (default local)  */
    int32_t match_score;          /* default  1                                             */
    int32_t mismatch_score;       /* default -4                                             */
    int32_t gap_open;             /* default -6                                             */
    int32_t gap_extend;           /* default -2                                             */
    int32_t jump_same;            /* jump_score_same_contig_and_strand      (default -10)   */
    int32_t jump_opp;             /* jump_score_same_contig_opposite_strand (default -10)   */
    int32_t jump_inter;           /* jump_score_inter_contig                (default -10)   */
    uint8_t double_strand;        /* -d                                                     */
    uint8_t circular;             /* -C (applies to every contig, mod.rs:186-204)           */
    uint8_t suboptimal;           /* --suboptimal                                            */
    uint8_t reserved0;
    uint32_t circular_slop;       /* default 20                                              */
    float suboptimal_pct;         /* default 20.0                                            */
    /* Pre-alignment contig selection (Options.pre_align .. pre_align_subset_contigs, mod.rs:76-86; align.rs:119-146). */
    uint8_t pre_align;            /* -p: only reads with a pre-alignment score >= pre_align_min_score are aligned   */
    uint8_t pre_align_subset_contigs; /* -x: align such a read to the contig-strands that reached the score only     */
    uint8_t pre_align_scoring;    /* STITCH_PREALIGN_*: how a contig-strand is scored (default k-mer; 0 = k-mer)   */
    uint8_t reserved1[1];
    uint32_t kmer_size;           /* -k, default 12                                          */
    uint32_t band_width;          /* -w, default 50                                          */
    int32_t pre_align_min_score;  /* -s, default 100                                         */
} stitch_opts;

/* One target sequence (TargetSeq, LIB/util/target_seq.rs:15): upper-cased forward bases.
 * The reverse complement is derived by the library (LIB/util/dna.rs:31). */
typedef struct stitch_contig {
    const char *name;
    const uint8_t *fwd;
    uint32_t len;
} stitch_contig;

/* Alignment, LIB/align/alignment.rs:16-51 (x = contig, y = read; see SURVEY.md section 0). */
typedef struct stitch_chain {
    int32_t score;
    uint32_t xstart, xend;        /* contig coordinates */
    uint32_t ystart, yend;        /* read coordinates   */
    uint32_t xlen, ylen;          /* xlen = length of the END contig (traceback/mod.rs:250) */
    uint32_t start_contig_idx, end_contig_idx;
    uint32_t length;              /* number of Match/Subst/Ins/Del on the path */
    uint32_t n_ops;               /* run-length encoded ops                      */
    uint32_t reserved;
    uint64_t ops_offset;          /* index of this chain's first op in the ops array */
} stitch_chain;

typedef struct stitch_op { uint32_t kind, a, b; } stitch_op;

/* Device-side counters of the last batch (for bench.py / roofline). */
typedef struct stitch_stats {
    uint64_t cells;               /* DP cell updates: sum over fills of n * sum(m_c)          */
    uint64_t fills;               /* number of DP fills (re-alignment fills included)          */
    uint64_t kernel_launches;     /* kernels launched by the library for the batch             */
    double fill_ms;               /* CUDA-event time of the fill kernels                       */
    double traceback_ms;          /* CUDA-event time of fix-up + traceback kernels             */
    double total_ms;              /* CUDA-event time, first H2D to last D2H of the batch       */
    uint64_t h2d_bytes, d2h_bytes;
    uint64_t traceback_bytes;     /* bytes of checkpoints + jump records written to HBM        */
    double packed_fill_ms;        /* of fill_ms: the packed-key kernel (bulk fill + tail + in-kernel fix-up/walk phase) */
    double wide_fill_ms;          /* of fill_ms: the wide kernel (last columns / fallback)     */
    double redo_fill_ms;          /* of fill_ms: re-runs of reads whose tracking window was too narrow */
    uint64_t packed_cells;        /* cell updates done by the packed-key kernel                */
    uint64_t redo_fills;          /* number of such re-runs                                    */
    double tail_fill_ms;          /* of fill_ms: the packed tail when it ran as its own launch (0: same launch as the fill) */
    uint64_t packed_launches;     /* launches of the packed-key kernel (one per chunk of reads)        */
    uint64_t tile_columns;        /* packed bulk pass: (256-row tile, column) pairs of the batch               */
    uint64_t quiet_tile_columns;  /* of those: skipped because the tile was provably quiet (dp_packed.h)       */
    double prealign_ms;           /* CUDA-event time of the pre-alignment (copies + prealign_kernel)           */
    uint64_t prealign_reads;      /* reads that went through the pre-alignment                                   */
} stitch_stats;

typedef struct stitch_ctx stitch_ctx;
typedef struct stitch_results stitch_results;

/* Builds the aligner for `n_contigs` targets on CUDA device `device`.
 * Fails with STITCH_ERR_CUDA when no usable device exists: there is no CPU path. */
int stitch_create(const stitch_opts *opts, const stitch_contig *contigs, uint32_t n_contigs,
                  int device, stitch_ctx **out);

/* Aligners::align for every read of the batch.  `bases` holds the reads back to back
 * (already upper-cased is not required: the library upper-cases, io.rs:64), read r is
 * bases[offsets[r] .. offsets[r+1]).  `subset_words` is NULL or n_reads * subset_stride
 * 32-bit words; bit c of read r's words selects contig-strand c (the pre-align subset,
 * mod.rs:287-295); an all-zero row means "all contigs".  With opts.pre_align and subset_words == NULL the library
 * runs its own pre-alignment (k-mer seeding on the GPU, DESIGN.md section 9) and selects the contig-strands itself; a
 * read that reaches the minimum score nowhere comes back with no chain (unmapped). */
int stitch_align_batch(stitch_ctx *ctx, const uint8_t *bases, const uint64_t *offsets,
                       uint32_t n_reads, const uint32_t *subset_words, uint32_t subset_stride,
                       stitch_results **out);

/* MultiContigAligner::custom_with_subset for every read: exactly one chain per read, clip
 * operations kept, no re-alignment, no sub-optimal chains. */
int stitch_custom_batch(stitch_ctx *ctx, const uint8_t *bases, const uint64_t *offsets,
                        uint32_t n_reads, const uint32_t *subset_words, uint32_t subset_stride,
                        stitch_results **out);

/* The pre-alignment alone (needs opts.pre_align): per read the selected contig-strands as subset_words (the BitSet
 * `contigs_to_align` of mod.rs:287-295; an all-zero row: no contig-strand reached pre_align_min_score, the read would not
 * be aligned) and, in best_scores (may be NULL), the best score among them (0 when none).  Feeding the words back to
 * stitch_align_batch gives the chains stitch_align_batch computes by itself with opts.pre_align_subset_contigs. */
int stitch_prealign_batch(stitch_ctx *ctx, const uint8_t *bases, const uint64_t *offsets, uint32_t n_reads,
                          uint32_t *subset_words, uint32_t subset_stride, int32_t *best_scores);

/* Same as stitch_align_batch / stitch_custom_batch but with reads already resident in
 * device memory (device pointers); used to time the path without host copies. */
int stitch_custom_batch_device(stitch_ctx *ctx, const uint8_t *d_bases, const uint64_t *h_offsets,
                               uint32_t n_reads, stitch_results **out);

uint32_t stitch_results_n_reads(const stitch_results *r);
/* chains of read r are chains[first .. first+count) */
void stitch_results_read(const stitch_results *r, uint32_t read, uint64_t *first, uint32_t *count);
const stitch_chain *stitch_results_chains(const stitch_results *r, uint64_t *n_chains);
const stitch_op *stitch_results_ops(const stitch_results *r, uint64_t *n_ops);
void stitch_free_results(stitch_results *r);
/* The Option<i32> of Aligners::align's return value (mod.rs:338-339): the best pre-alignment score of read `read`.
 * Returns 1 and sets *score when there is one (pre_align on and the read reached pre_align_min_score on some
 * contig-strand), 0 for None. */
int stitch_results_prealign(const stitch_results *r, uint32_t read, int32_t *score);
/* A results handle holding ONE read with the given chains (copied; ops_offset of chain k indexes `ops`).  Alignment is a
 * plain public struct in the reference (LIB/align/alignment.rs:16-51) and SamRecordFormatter::format takes any
 * &[Alignment] (mod.rs:622-627): this is how a caller formats chains it built or edited itself (n_chains = 0: the
 * unmapped record). */
int stitch_results_from_chains(const stitch_chain *chains, uint32_t n_chains, const stitch_op *ops, uint64_t n_ops,
                               stitch_results **out);

/* Options of the SAM record layer: Options.{soft_clip,use_eq_and_x,pick_primary,filter_secondary,filter_secondary_pct},
 * LIB/align/aligners/mod.rs:106-115 (defaults: false, false, query-length, false, 10.0). */
typedef struct stitch_sam_opts {
    uint8_t soft_clip, use_eq_and_x, pick_primary /* 0 query-length, 1 score */, filter_secondary;
    float filter_secondary_pct;
} stitch_sam_opts;

/* SamRecordFormatter::format (LIB/align/aligners/mod.rs:622-972) with SubAlignmentBuilder::build
 * (LIB/align/sub_alignment.rs:170-241) for read `read` of `res`: one SAM text line per record (flags, RNAME, POS,
 * MAPQ, CIGAR with soft/hard clips, SEQ/QUAL orientation, the custom tags qs qe ts te as xs si sc cl ci cn, AS, NM,
 * SA), lines separated by '\n'.  `read_header` is the FASTQ header (name = first word), `quals` may be NULL; they
 * are passed through as given.  `*out_text` is malloc'ed: release it with stitch_free_text.  sopts == NULL: defaults. */
int stitch_format_sam(stitch_ctx *ctx, const stitch_results *res, uint32_t read, const char *read_header,
                      const uint8_t *bases, const uint8_t *quals, uint32_t n_bases, int has_pre_align_score,
                      int32_t pre_align_score, const stitch_sam_opts *sopts, char **out_text);
void stitch_free_text(char *text);

int stitch_get_stats(const stitch_ctx *ctx, stitch_stats *out);
/* Upper bound on reads in flight; 0 = choose from free HBM. */
int stitch_set_max_inflight(stitch_ctx *ctx, uint32_t max_reads);

void stitch_destroy(stitch_ctx *ctx);
/* Message of the last failure on this ctx (or of stitch_create when ctx is NULL). */
const char *stitch_last_error(const stitch_ctx *ctx);

/* Diagnostic for the roofline: sustained INT32 add+max issue rate of the device, in giga
 * operations per second, an add followed by a max counted as two operations (SURVEY.md 8d). */
int stitch_measure_int32_peak(int device, double *gops);

/* ABI version of this header. */
uint32_t stitch_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* STITCH_B200_H */
