// host_common.hpp — host side of the library above the DP backend.
//
// Restates the per-read driver of the reference around the DP core:
//   Builder::build_aligners   fg-stitch-lib/src/align/aligners/mod.rs:171-211
//   Aligners::align           mod.rs:237-340   (pre-alignment is not on this path)
//   remove_clipping           mod.rs:343-353
//   realign_origin & friends  mod.rs:365-553
//   Alignment::split_at_y     fg-stitch-lib/src/align/alignment.rs:207-360
// but batched: every DP fill (+ traceback request) is a Job handed to a Backend; the product's
// backend is CUDA (cuda_backend.cu).  The tests also instantiate this driver over a CPU
// emulation backend to check the host logic and the DP decomposition without a GPU.
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <set>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/stitch_b200.h"
#include "dp_core.h"
#include "prealign_core.h"

namespace stitch {
namespace host {

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string &m) : std::runtime_error(m), code(c) {}
};

struct Opts {
    int mode = STITCH_MODE_LOCAL;
    Scoring sc{};
    bool double_strand = false, circular = false, suboptimal = false;
    uint32_t slop = 20;
    float sub_pct = 20.0f;
    bool pre_align = false, pre_subset = true;   // mod.rs:76-86
    bool pre_banded = false;                     // STITCH_PREALIGN_BANDED (prealign_core.h)
    uint32_t kmer = 12, band = 50;
    int32_t pre_min_score = 100;
};

inline Opts make_opts(const stitch_opts &o) {
    Opts p;
    if (o.mode < STITCH_MODE_LOCAL || o.mode > STITCH_MODE_GLOBAL)
        throw Error(STITCH_ERR_INVALID, "Custom alignment mode not supported");   // mod.rs:129
    if (o.gap_open > 0) throw Error(STITCH_ERR_INVALID, "gap_open can't be positive");
    if (o.gap_extend > 0) throw Error(STITCH_ERR_INVALID, "gap_extend can't be positive");
    if (o.jump_same > 0 || o.jump_opp > 0 || o.jump_inter > 0)
        throw Error(STITCH_ERR_INVALID, "jump scores can't be positive");       // scoring.rs:64-75
    p.mode = o.mode;
    p.sc.match = o.match_score; p.sc.mismatch = o.mismatch_score;
    p.sc.o = o.gap_open; p.sc.e = o.gap_extend;
    p.sc.g_same = o.jump_same; p.sc.g_opp = o.jump_opp; p.sc.g_inter = o.jump_inter;
    const int32_t M = MIN_SCORE;
    switch (o.mode) {   // mod.rs:123-131
    case STITCH_MODE_LOCAL: p.sc.xp = p.sc.xs = p.sc.yp = p.sc.ys = 0; break;
    case STITCH_MODE_QUERY_LOCAL: p.sc.xp = p.sc.xs = M; p.sc.yp = p.sc.ys = 0; break;
    case STITCH_MODE_TARGET_LOCAL: p.sc.xp = p.sc.xs = 0; p.sc.yp = p.sc.ys = M; break;
    default: p.sc.xp = p.sc.xs = p.sc.yp = p.sc.ys = M; break;
    }
    p.double_strand = o.double_strand != 0; p.circular = o.circular != 0; p.suboptimal = o.suboptimal != 0;
    p.slop = o.circular_slop; p.sub_pct = o.suboptimal_pct;
    p.pre_align = o.pre_align != 0; p.pre_subset = o.pre_align_subset_contigs != 0;
    p.kmer = o.kmer_size; p.band = o.band_width; p.pre_min_score = o.pre_align_min_score;
    if (o.pre_align_scoring != STITCH_PREALIGN_KMER && o.pre_align_scoring != STITCH_PREALIGN_BANDED)
        throw Error(STITCH_ERR_INVALID, "pre-alignment scoring must be 0 (k-mer) or 1 (banded)");
    p.pre_banded = o.pre_align_scoring == STITCH_PREALIGN_BANDED;
    if (p.pre_align) {
        if (p.kmer < 4 || p.kmer > 31) throw Error(STITCH_ERR_INVALID, "k-mer size must be 4..31");
        if (p.band < 1) throw Error(STITCH_ERR_INVALID, "band width must be positive");
    }
    return p;
}

inline int64_t max_abs_score(const Scoring &s) {
    int64_t v = 0;
    for (int32_t x : {s.match, s.mismatch, s.o, s.e, s.g_same, s.g_opp, s.g_inter})
        v = std::max<int64_t>(v, x < 0 ? -(int64_t)x : x);
    return v;
}

inline std::vector<uint8_t> revcomp(const std::vector<uint8_t> &s) {   // util/dna.rs:5-41
    static const auto table = [] {
        std::vector<uint8_t> t(256);
        for (int v = 0; v < 256; ++v) t[(size_t)v] = (uint8_t)v;
        const char *a = "AGCTYRWSKMDVHBN", *b = "TCGARYWSMKHBDVN";
        for (int k = 0; k < 15; ++k) { t[(uint8_t)a[k]] = (uint8_t)b[k]; t[(uint8_t)a[k] + 32] = (uint8_t)(b[k] + 32); }
        return t;
    }();
    std::vector<uint8_t> r(s.size());
    for (size_t k = 0; k < s.size(); ++k) r[k] = table[s[s.size() - 1 - k]];
    return r;
}

// All contig-strands: forward contigs in input order, then (double_strand) their reverse
// complements in the same order (mod.rs:186-205).
struct Contigs {
    uint32_t n_targets = 0, n_strands = 0;
    std::vector<std::string> names;
    std::vector<uint32_t> len;       // per strand
    std::vector<uint32_t> seq_off;   // per strand, into blob
    std::vector<uint8_t> blob;
    uint32_t max_len = 0;

    void build(const stitch_contig *c, uint32_t n, bool double_strand) {
        if (n == 0) throw Error(STITCH_ERR_INVALID, "no contigs");
        n_targets = n; n_strands = double_strand ? 2 * n : n;
        // the reference asserts <= 256 contig-strands on the TABLE (8-bit contig index of its traceback cell,
        // packed_length_cell.rs:139-140); here the table may hold MAX_TABLE_STRANDS and the limit applies to the
        // contig-strands one read is aligned against (Layout): larger tables need a per-read subset (pre-alignment)
        if (n_strands > MAX_TABLE_STRANDS) throw Error(STITCH_ERR_LIMIT, "more than 65536 contig-strands");
        std::vector<std::vector<uint8_t>> fwd(n);
        std::set<std::string> seen_names;
        for (uint32_t k = 0; k < n; ++k) {
            if (!c[k].name || (!c[k].fwd && c[k].len)) throw Error(STITCH_ERR_INVALID, "null contig");
            if (c[k].len == 0) throw Error(STITCH_ERR_INVALID, "empty contig");
            if (c[k].len > MAX_CONTIG_LEN) throw Error(STITCH_ERR_LIMIT, "contig longer than 2^27-1");
            names.emplace_back(c[k].name);
            if (!seen_names.insert(names[k]).second) throw Error(STITCH_ERR_INVALID, "Contig already added! name: " + names[k]);   // MCA:101-104
            fwd[k].assign(c[k].fwd, c[k].fwd + c[k].len);
            for (auto &b : fwd[k]) if (b >= 'a' && b <= 'z') b = (uint8_t)(b - 32);   // target_seq.rs:111-115
        }
        auto add = [&](const std::vector<uint8_t> &s) {
            while (blob.size() % 16) blob.push_back(0);   // aligned vector loads of a lane's bases
            seq_off.push_back((uint32_t)blob.size());
            len.push_back((uint32_t)s.size());
            blob.insert(blob.end(), s.begin(), s.end());
            max_len = std::max<uint32_t>(max_len, (uint32_t)s.size());
        };
        for (uint32_t k = 0; k < n; ++k) add(fwd[k]);
        if (double_strand) for (uint32_t k = 0; k < n; ++k) add(revcomp(fwd[k]));
    }
};

// The contig subset a fill runs over (MCA::custom_with_subset keeps ascending contig order).
struct Layout {
    std::vector<ContigEntry> ent;   // ascending contig_idx
    uint32_t n_tiles = 0;
    uint64_t cells_per_col = 0;    // sum of m_c
    uint32_t PM() const { return n_tiles * (uint32_t)TILE; }
};

struct LayoutCache {
    const Contigs *contigs = nullptr;
    bool circular = false;
    std::vector<Layout> layouts;
    std::map<std::vector<uint32_t>, uint32_t> index;
    uint64_t generation = 0;       // bumped when the cache is emptied (layout ids are only valid within one batch)

    // Called between batches: with per-read subsets (pre-alignment) every batch brings new layouts.
    void trim(size_t keep_below = 4096) {
        if (layouts.size() < keep_below) return;
        layouts.clear(); index.clear(); ++generation;
    }

    uint32_t get(const std::vector<uint32_t> &strands /* ascending contig-strand indices */) {
        auto it = index.find(strands);
        if (it != index.end()) return it->second;
        if (strands.size() > MAX_STRANDS)
            throw Error(STITCH_ERR_LIMIT, "a read would be aligned against more than 256 contig-strands (the reference's limit, "
                                          "packed_length_cell.rs:139-140): select contigs per read (pre-alignment / subset_words)");
        Layout L;
        const uint32_t T = contigs->n_targets;
        std::map<uint32_t, int32_t> pos_of;
        for (uint32_t c : strands) {
            ContigEntry e{};
            e.contig_idx = c; e.m = contigs->len[c];
            e.tile_start = L.n_tiles; e.ntiles = (e.m + TILE - 1) / TILE;
            e.opp = -1; e.seq_off = contigs->seq_off[c]; e.circular = circular ? 1u : 0u;
            pos_of[c] = (int32_t)L.ent.size();
            L.n_tiles += e.ntiles; L.cells_per_col += e.m;
            L.ent.push_back(e);
        }
        for (auto &e : L.ent) {   // opposite strand = same name, other strand, if present (MCA:241-262)
            const uint32_t o = e.contig_idx < T ? e.contig_idx + T : e.contig_idx - T;
            const auto it = o < contigs->n_strands ? pos_of.find(o) : pos_of.end();
            if (it != pos_of.end()) e.opp = it->second;
        }
        layouts.push_back(std::move(L));
        const uint32_t id = (uint32_t)layouts.size() - 1;
        index.emplace(strands, id);
        return id;
    }
    uint32_t all() {
        std::vector<uint32_t> s(contigs->n_strands);
        for (uint32_t k = 0; k < contigs->n_strands; ++k) s[k] = k;
        return get(s);
    }
};

// ---------------------------------------------------------------------------------------------
// Jobs
// ---------------------------------------------------------------------------------------------
enum WalkKind : uint32_t { WALK_BEST = 0, WALK_ALL = 1, WALK_FROM = 2 };

struct Job {
    const uint8_t *read = nullptr;   // upper-cased query (host memory, owned by the caller)
    uint32_t n = 0;
    uint32_t layout = 0;
    WalkKind walk = WALK_BEST;
    uint32_t from_contig = 0;        // WALK_FROM: contig-strand index the chain must end on
};

struct RawChain { ChainHdr h{}; std::vector<OutOp> ops; };
struct JobResult { std::vector<RawChain> chains; };

struct BackendStats {
    uint64_t cells = 0, fills = 0, launches = 0, h2d = 0, d2h = 0, tb_bytes = 0, refills = 0;
    double fill_ms = 0, tb_ms = 0, total_ms = 0, packed_ms = 0, wide_ms = 0, redo_ms = 0, tail_ms = 0;
    uint64_t packed_cells = 0, packed_launches = 0, tile_columns = 0, quiet_tile_columns = 0, pre_reads = 0;
    double pre_ms = 0;
    void reset() { *this = BackendStats(); }
};

// K-mer index of every contig-strand for the pre-alignment (prealign_core.h): the positions (offsets into the contig
// blob) of every valid k-mer, grouped by bucket (counting sort).  Replaces the per-target hash maps of
// TargetSeq::build_target_hash (util/target_seq.rs:50-56).
struct KmerIndex {
    uint32_t K = 0;
    std::vector<uint32_t> off;   // [n_buckets + 1]
    std::vector<uint32_t> pos;   // blob offsets, grouped by bucket
    void build(const Contigs &c, uint32_t k) {
        K = k;
        const uint32_t nb = pre_n_buckets(K);
        off.assign((size_t)nb + 1, 0);
        auto each = [&](auto &&fn) {
            for (uint32_t s = 0; s < c.n_strands; ++s) {
                if (c.len[s] < K) continue;
                const uint8_t *b = c.blob.data() + c.seq_off[s];
                for (uint32_t p = 0; p + K <= c.len[s]; ++p) { uint64_t code; if (pre_kmer_code(b + p, K, code)) fn(pre_bucket(code, K), c.seq_off[s] + p); }
            }
        };
        each([&](uint32_t bucket, uint32_t) { ++off[(size_t)bucket + 1]; });
        for (size_t b = 0; b < nb; ++b) off[b + 1] += off[b];
        pos.assign(off[nb], 0);
        std::vector<uint32_t> cur(off.begin(), off.end() - 1);
        each([&](uint32_t bucket, uint32_t p) { pos[cur[bucket]++] = p; });
    }
};

// The pre-alignment exactly as prealign_core.h defines it, sequentially, for either scoring (opts.pre_banded): per read the
// selected contig-strands in ascending order with their scores.  The statement of the definition the backends are checked
// against; it runs for a backend that does not implement the banded scoring itself (Backend::prealign_scores_banded).
inline void prealign_sequential(const Opts &o, const Contigs &c, KmerIndex &kindex, const std::vector<Job> &reads,
                                std::vector<std::vector<PreHit>> &out) {
    if (kindex.K != o.kmer) kindex.build(c, o.kmer);
    out.assign(reads.size(), std::vector<PreHit>());
    const uint32_t K = o.kmer, W = o.band;
    for (size_t r = 0; r < reads.size(); ++r) {
        const uint8_t *read = reads[r].read; const uint32_t n = reads[r].n;
        std::vector<uint32_t> cnt(c.n_strands, 0);
        std::vector<std::pair<uint32_t, uint32_t>> hits;   // (strand, diagonal + n)
        for (uint32_t j = 0; j + K <= n; ++j) {
            uint64_t code;
            if (!pre_kmer_code(read + j, K, code)) continue;
            const uint32_t b = pre_bucket(code, K);
            for (uint32_t e = kindex.off[b]; e < kindex.off[b + 1]; ++e) {
                const uint32_t p = kindex.pos[e];
                if (K > PRE_DIRECT_K && !pre_same_kmer(c.blob.data() + p, read + j, K)) continue;
                const uint32_t s = pre_strand_of(c.seq_off.data(), c.n_strands, p);
                ++cnt[s]; hits.emplace_back(s, (p - c.seq_off[s]) + n - j);
            }
        }
        uint32_t need = o.pre_banded ? pre_need_banded(o.pre_min_score, o.sc.match, K) : pre_need(o.pre_min_score, o.sc.match, K);
        std::vector<uint32_t> cand;
        for (;;) {
            cand.clear();
            for (uint32_t s = 0; s < c.n_strands; ++s) if (cnt[s] >= need) cand.push_back(s);
            if (cand.size() <= PRE_MAX_CAND) break;
            need *= 2;
        }
        const uint32_t n_bins = (n + c.max_len) / W + 2;
        std::vector<PreHit> kept;
        for (uint32_t s : cand) {
            std::vector<uint32_t> bins(n_bins, 0);
            for (const auto &h : hits) if (h.first == s && h.second / W < n_bins) ++bins[h.second / W];
            uint32_t best = 0, bstar = 0;   // the lowest bin of the best pair
            for (uint32_t b = 0; b < n_bins; ++b) {
                const uint32_t v = bins[b] + (b + 1 < n_bins ? bins[b + 1] : 0u);
                if (v > best) { best = v; bstar = b; }
            }
            const int32_t dlo = (int32_t)(bstar * W) - (int32_t)n, dhi = dlo + 2 * (int32_t)W;
            const int32_t sc = o.pre_banded ? pre_banded_score(read, n, c.blob.data() + c.seq_off[s], c.len[s], dlo, dhi, o.sc)
                                            : pre_score_of(o.sc.match, best, K);
            if (sc >= o.pre_min_score) kept.push_back(PreHit{s, sc});
        }
        if (kept.size() > MAX_STRANDS) {
            std::stable_sort(kept.begin(), kept.end(), [](const PreHit &a, const PreHit &b) { return a.score != b.score ? a.score > b.score : a.strand < b.strand; });
            kept.resize(MAX_STRANDS);
            std::sort(kept.begin(), kept.end(), [](const PreHit &a, const PreHit &b) { return a.strand < b.strand; });
        }
        out[r] = kept;
    }
}

struct Backend {
    virtual ~Backend() {}
    // Pre-alignment (prealign_core.h): per read, the selected contig-strands in ascending order with their scores.
    virtual void prealign(const std::vector<Job> &reads, std::vector<std::vector<PreHit>> &out) = 0;
    // Whether prealign() implements the banded scoring too (the CUDA backend: kernels_prealign.cuh).  With a backend that
    // implements only the k-mer scoring (the CPU emulator the tests run), the banded scoring comes from prealign_sequential.
    virtual bool prealign_scores_banded() const { return false; }
    // `device_reads`: reads already resident on the device (d_bases base pointer + per-job offsets
    // in Job::read interpreted as offsets); only the CUDA backend supports it.
    virtual void run(const std::vector<Job> &jobs, std::vector<JobResult> &out) = 0;
    virtual void set_max_inflight(uint32_t) {}
    BackendStats stats;
};

// Debugging aid (STITCH_DUMP_DIR): raw per-job records, same format from every backend.
inline void dump_job(const char *dir, uint32_t seq, const std::vector<LastCell> &last, const std::vector<SnRec> &sn,
                     const std::vector<ColRec> &colrec, const std::vector<uint8_t> &tb) {
    auto wr = [&](const char *name, const void *p, size_t bytes) {
        std::string fn = std::string(dir) + "/job" + std::to_string(seq) + "." + name;
        if (FILE *f = std::fopen(fn.c_str(), "wb")) { std::fwrite(p, 1, bytes, f); std::fclose(f); }
    };
    wr("last", last.data(), last.size() * sizeof(LastCell));
    wr("sn", sn.data(), sn.size() * sizeof(SnRec));
    wr("colrec", colrec.data(), colrec.size() * sizeof(ColRec));
    wr("tb", tb.data(), tb.size());
}

// ---------------------------------------------------------------------------------------------
// Host alignment record with expanded operations
// ---------------------------------------------------------------------------------------------
struct HOp { uint8_t kind; uint32_t a, b; };
struct HAlign {
    int32_t score = 0;
    int64_t xstart = 0, xend = 0, ystart = 0, yend = 0, xlen = 0, ylen = 0;
    int64_t start_contig = 0, end_contig = 0, length = 0;
    std::vector<HOp> ops;   // run-length encoded exactly like stitch_op
};

inline bool is_base_op(uint32_t k) { return k <= OP_INS; }
inline int64_t op_len_y(const HOp &o) {   // constants.rs:75-84 (RLE aware)
    switch (o.kind) {
    case OP_MATCH: case OP_SUBST: case OP_DEL: case OP_YCLIP: case OP_YJUMP: return o.a;
    default: return 0;
    }
}

inline HAlign from_raw(const RawChain &r) {
    HAlign a;
    a.score = r.h.score; a.xstart = r.h.xstart; a.xend = r.h.xend; a.ystart = r.h.ystart; a.yend = r.h.yend;
    a.xlen = r.h.xlen; a.ylen = r.h.ylen; a.start_contig = r.h.start_contig_idx; a.end_contig = r.h.end_contig_idx;
    a.length = r.h.length;
    a.ops.reserve(r.ops.size());
    for (const OutOp &o : r.ops) a.ops.push_back(HOp{(uint8_t)o.kind, o.a, o.b});
    return a;
}

inline void push_rle(std::vector<HOp> &v, const HOp &o) {
    if (is_base_op(o.kind) && !v.empty() && v.back().kind == o.kind) v.back().a += o.a;
    else v.push_back(o);
}

// mod.rs:343-353: in the three local modes only Match/Subst/Ins/Del/Xjump survive.
inline HAlign remove_clipping(const Opts &opts, HAlign a) {
    if (opts.mode == STITCH_MODE_GLOBAL) return a;
    std::vector<HOp> kept;
    for (const HOp &o : a.ops) if (is_base_op(o.kind) || o.kind == OP_XJUMP) push_rle(kept, o);
    a.ops.swap(kept);
    return a;
}

// alignment.rs:207-360 for mode Custom (traceback_from always yields Custom, TB:369, so the
// clip re-insertion branches of the reference are dead on this path).  Works on single-base
// granularity by expanding the runs lazily.
inline HAlign split_at_y(const HAlign &s, int64_t y_pivot) {
    if (s.ops.empty()) return s;
    if (s.ops.front().kind == OP_XCLIP || s.ops.front().kind == OP_YCLIP || s.ops.back().kind == OP_XCLIP ||
        s.ops.back().kind == OP_YCLIP)
        throw Error(STITCH_ERR_INTERNAL, "split_at_y: leading/trailing clip");
    // expand to unit ops
    std::vector<HOp> u;
    for (const HOp &o : s.ops) {
        if (is_base_op(o.kind)) for (uint32_t t = 0; t < o.a; ++t) u.push_back(HOp{o.kind, 1, 0});
        else u.push_back(o);
    }
    auto lx = [](const HOp &o, int64_t x) -> int64_t {
        switch (o.kind) {
        case OP_MATCH: case OP_SUBST: case OP_INS: return 1;
        case OP_XCLIP: return o.a;
        case OP_XJUMP: return (int64_t)o.b - x;
        default: return 0;
        }
    };
    int64_t x = s.xstart, y = s.ystart, contig = s.start_contig;
    size_t k = 0;
    while (k < u.size() && !is_base_op(u[k].kind)) {
        if (u[k].kind == OP_XJUMP) contig = u[k].a;
        y += op_len_y(u[k]); x += lx(u[k], x); ++k;
    }
    while (k < u.size()) {
        if (y + op_len_y(u[k]) >= y_pivot) break;
        if (u[k].kind == OP_XJUMP) contig = u[k].a;
        y += op_len_y(u[k]); x += lx(u[k], x); ++k;
    }
    if (k >= u.size()) throw Error(STITCH_ERR_INTERNAL, "split_at_y: pivot beyond the alignment");
    const int64_t pre_xend = x + 1, pre_yend = y + 1, pre_end_contig = contig;
    const size_t pre_count = k + 1;
    if (y_pivot < pre_yend) throw Error(STITCH_ERR_INTERNAL, "split_at_y: y_pivot < pre.yend");
    while (k < u.size()) {
        if (y >= y_pivot && is_base_op(u[k].kind)) break;
        if (u[k].kind == OP_XJUMP) contig = u[k].a;
        y += op_len_y(u[k]); x += lx(u[k], x); ++k;
    }
    const int64_t post_xstart = x, post_ystart = y, post_start_contig = contig;
    HAlign a;
    a.start_contig = post_start_contig; a.end_contig = pre_end_contig;
    a.xstart = post_xstart; a.ystart = post_ystart - y_pivot;
    a.xend = pre_xend; a.yend = pre_yend + s.ylen - y_pivot;
    a.ylen = s.ylen; a.xlen = s.xlen; a.score = s.score; a.length = s.length;
    if (a.ystart < 0) throw Error(STITCH_ERR_INTERNAL, "split_at_y: ystart underflow");
    for (size_t t = k; t < u.size(); ++t) push_rle(a.ops, u[t]);
    // post.end_contig = s.end_contig, post.xend = s.xend; pre.start = s.start_contig, pre.xstart = s.xstart
    if (s.start_contig != s.end_contig || s.xstart != s.xend)
        a.ops.push_back(HOp{(uint8_t)OP_XJUMP, (uint32_t)s.start_contig, (uint32_t)s.xstart});
    const int64_t yjump = a.ylen + s.ystart - s.yend;
    if (yjump < 0) throw Error(STITCH_ERR_INTERNAL, "split_at_y: yjump underflow");
    if (yjump > 0) a.ops.push_back(HOp{(uint8_t)OP_YJUMP, (uint32_t)yjump, 0});
    {
        // the pre-pivot ops start a new run even if the previous op has the same kind only when
        // separated by a special op; push_rle merges adjacent equal base ops, which renders the
        // same per-base sequence.
        for (size_t t = 0; t < pre_count; ++t) push_rle(a.ops, u[t]);
    }
    return a;
}

// ---------------------------------------------------------------------------------------------
// Results container behind stitch_results
// ---------------------------------------------------------------------------------------------
struct Results {
    std::vector<stitch_chain> chains;
    std::vector<stitch_op> ops;
    std::vector<uint64_t> first;
    std::vector<uint32_t> count;
    std::vector<uint8_t> has_pre;     // per read: Some / None of the pre-alignment score (mod.rs:338-339)
    std::vector<int32_t> pre_score;
    void begin_read() { first.push_back(chains.size()); count.push_back(0); has_pre.push_back(0); pre_score.push_back(0); }
    void set_pre(int32_t score) { has_pre.back() = 1; pre_score.back() = score; }
    void add(const HAlign &a) {
        stitch_chain c{};
        c.score = a.score; c.xstart = (uint32_t)a.xstart; c.xend = (uint32_t)a.xend;
        c.ystart = (uint32_t)a.ystart; c.yend = (uint32_t)a.yend; c.xlen = (uint32_t)a.xlen; c.ylen = (uint32_t)a.ylen;
        c.start_contig_idx = (uint32_t)a.start_contig; c.end_contig_idx = (uint32_t)a.end_contig;
        c.length = (uint32_t)a.length; c.ops_offset = ops.size(); c.n_ops = (uint32_t)a.ops.size();
        for (const HOp &o : a.ops) ops.push_back(stitch_op{o.kind, o.a, o.b});
        chains.push_back(c);
        count.back() += 1;
    }
};

// ---------------------------------------------------------------------------------------------
// The per-read driver, batched
// ---------------------------------------------------------------------------------------------
struct Aligner {
    Opts opts;
    Contigs contigs;
    LayoutCache layouts;
    std::unique_ptr<Backend> backend;
    std::string last_error;
    KmerIndex seq_kindex;   // prealign_sequential's index (built on first use)

    // The pre-alignment of a batch under opts' scoring (see Backend::prealign_scores_banded).
    void prealign(const std::vector<Job> &reads, std::vector<std::vector<PreHit>> &hits) {
        if (opts.pre_banded && !backend->prealign_scores_banded()) prealign_sequential(opts, contigs, seq_kindex, reads, hits);
        else backend->prealign(reads, hits);
    }

    void init(const stitch_opts &o, const stitch_contig *c, uint32_t n) {
        opts = make_opts(o);
        contigs.build(c, n, opts.double_strand);
        layouts.contigs = &contigs;
        layouts.circular = opts.circular;
        if (contigs.n_strands <= MAX_STRANDS) layouts.all();
    }

    void check_ranges(uint64_t max_n) const {
        // i32 headroom: the reference's scores are sums of at most (n + m) per-step scores on top
        // of MIN_SCORE; outside this range the reference itself overflows.
        const int64_t span = (int64_t)std::max<uint64_t>(max_n, contigs.max_len) + 2;
        if (max_abs_score(opts.sc) * span > 400000000ll)
            throw Error(STITCH_ERR_INVALID, "scores x sequence length exceed the i32 range of the reference's DP");
        if (max_n > MAX_CONTIG_LEN) throw Error(STITCH_ERR_LIMIT, "read longer than 2^27-1");
    }

    uint32_t layout_for(const uint32_t *words, uint32_t stride) {
        if (!words) return layouts.all();
        std::vector<uint32_t> s;
        for (uint32_t w = 0; w < stride && w * 32 < contigs.n_strands; ++w)
            for (uint32_t bits = words[w]; bits; bits &= bits - 1) {
                const uint32_t c = w * 32 + (uint32_t)__builtin_ctz(bits);
                if (c < contigs.n_strands) s.push_back(c);
            }
        if (s.empty()) return layouts.all();
        return layouts.get(s);
    }

    static std::vector<uint8_t> upper(const uint8_t *p, uint64_t n) {   // io.rs:64
        std::vector<uint8_t> v(p, p + n);
        for (auto &b : v) if (b >= 'a' && b <= 'z') b = (uint8_t)(b - 32);
        return v;
    }

    // MultiContigAligner::custom_with_subset per read (raw chain, clips kept).
    void custom_batch(const uint8_t *bases, const uint64_t *offs, uint32_t n_reads, const uint32_t *subset,
                      uint32_t stride, Results &res) {
        layouts.trim();
        std::vector<std::vector<uint8_t>> q(n_reads);
        std::vector<Job> jobs(n_reads);
        uint64_t max_n = 0;
        for (uint32_t r = 0; r < n_reads; ++r) {
            q[r] = upper(bases + offs[r], offs[r + 1] - offs[r]);
            max_n = std::max<uint64_t>(max_n, q[r].size());
            jobs[r].read = q[r].data(); jobs[r].n = (uint32_t)q[r].size();
            jobs[r].layout = layout_for(subset ? subset + (size_t)r * stride : nullptr, stride);
            jobs[r].walk = WALK_BEST;
        }
        check_ranges(max_n);
        std::vector<JobResult> out;
        backend->run(jobs, out);
        for (uint32_t r = 0; r < n_reads; ++r) {
            res.begin_read();
            if (out[r].chains.size() != 1) throw Error(STITCH_ERR_INTERNAL, "traceback_from returned None");
            res.add(from_raw(out[r].chains[0]));
        }
    }

    struct RealignPlan {           // one chain's origin re-alignment (mod.rs:442-553)
        std::vector<std::vector<uint8_t>> queries;
        std::vector<int64_t> pivots;
        std::vector<int64_t> contig;   // contig the re-aligned chain must start and end on
        uint32_t layout = 0;
        size_t first_job = 0;
    };

    // mod.rs:365-410 + the query construction of mod.rs:471-549
    bool plan_realign(const std::vector<uint8_t> &query, const HAlign &al, RealignPlan &plan) {
        const int64_t slop = opts.slop;
        int64_t at_start = -1, at_end = -1;
        if (al.xstart <= slop && opts.circular) at_start = al.start_contig;
        if (al.xlen <= al.xend + slop && opts.circular) at_end = al.end_contig;
        if (at_start >= 0 && at_end >= 0 && at_start == at_end) return false;
        if (at_start < 0 && at_end < 0) return false;
        if (at_start >= 0 && al.yend == al.ylen) at_start = -1;
        if (at_end >= 0 && al.ystart == 0) at_end = -1;
        if (at_start < 0 && at_end < 0) return false;

        std::vector<bool> in(contigs.n_strands, false);
        in[(size_t)al.start_contig] = true; in[(size_t)al.end_contig] = true;
        for (const HOp &o : al.ops) if (o.kind == OP_XJUMP) in[o.a] = true;
        std::vector<uint32_t> strands;
        for (uint32_t c = 0; c < contigs.n_strands; ++c) if (in[c]) strands.push_back(c);
        plan.layout = layouts.get(strands);

        auto rotate = [&](int64_t at) {
            std::vector<uint8_t> r(query.begin() + at, query.end());
            r.insert(r.end(), query.begin(), query.begin() + at);
            return r;
        };
        auto add = [&](int64_t at, int64_t contig) {
            plan.queries.push_back(rotate(at)); plan.pivots.push_back(al.ylen - at); plan.contig.push_back(contig);
        };
        if (at_start >= 0) {
            int64_t y2 = al.ystart;
            for (const HOp &o : al.ops) {
                if (o.kind == OP_XJUMP && (int64_t)o.a != at_start) break;
                y2 += op_len_y(o);
            }
            add(al.yend, at_start);
            add(y2, at_start);
        }
        if (at_end >= 0) {
            int64_t y2 = al.ystart, ycur = al.ystart, xidx = al.start_contig;
            for (const HOp &o : al.ops) {
                if (o.kind == OP_XJUMP) {
                    if ((int64_t)o.a == at_end && xidx != at_end) y2 = ycur;
                    xidx = o.a;
                }
                ycur += op_len_y(o);
            }
            add(al.ystart, at_end);
            add(y2, at_end);
        }
        return true;
    }

    // Aligners::align per read.
    // mod.rs:243-295: which contig-strands a read is aligned against, from its pre-alignment hits.  Returns false when
    // the read is not aligned at all (no contig-strand reached the minimum score: (Vec::new(), None), mod.rs:282-284).
    bool prealign_select(const std::vector<PreHit> &hits, std::vector<uint32_t> &strands, int32_t &score) {
        strands.clear();
        if (hits.empty()) return false;
        const uint32_t T = contigs.n_targets;
        if (opts.pre_subset) {   // every contig-strand that reached the score (mod.rs:287-292)
            score = hits[0].score;
            for (const PreHit &h : hits) { strands.push_back(h.strand); score = std::max(score, h.score); }
            return true;
        }
        // all contigs are aligned anyhow: the reference stops at the first target (in input order) with a passing strand
        // and reports the best score of THAT target's strands (mod.rs:274-277, 338)
        uint32_t first_t = 0xffffffffu;
        for (const PreHit &h : hits) first_t = std::min(first_t, h.strand % T);
        bool any = false;
        for (const PreHit &h : hits) if (h.strand % T == first_t) { score = any ? std::max(score, h.score) : h.score; any = true; }
        return true;   // strands stays empty: all contigs
    }

    void prealign_batch(const uint8_t *bases, const uint64_t *offs, uint32_t n_reads, uint32_t *words, uint32_t stride, int32_t *best) {
        std::vector<std::vector<uint8_t>> q(n_reads);
        std::vector<Job> pj(n_reads);
        for (uint32_t r = 0; r < n_reads; ++r) {
            q[r] = upper(bases + offs[r], offs[r + 1] - offs[r]);
            pj[r].read = q[r].data(); pj[r].n = (uint32_t)q[r].size();
        }
        std::vector<std::vector<PreHit>> hits;
        prealign(pj, hits);
        std::fill(words, words + (size_t)n_reads * stride, 0u);
        for (uint32_t r = 0; r < n_reads; ++r) {
            int32_t b = 0;
            for (const PreHit &h : hits[r]) { words[(size_t)r * stride + h.strand / 32] |= 1u << (h.strand % 32); b = std::max(b, h.score); }
            if (best) best[r] = b;
        }
    }

    // Aligners::align per read.
    void align_batch(const uint8_t *bases, const uint64_t *offs, uint32_t n_reads, const uint32_t *subset,
                     uint32_t stride, Results &res) {
        layouts.trim();
        std::vector<std::vector<uint8_t>> q(n_reads);
        uint64_t max_n = 0;
        for (uint32_t r = 0; r < n_reads; ++r) {
            q[r] = upper(bases + offs[r], offs[r + 1] - offs[r]);
            max_n = std::max<uint64_t>(max_n, q[r].size());
        }
        check_ranges(max_n);
        // stage 0: pre-alignment contig selection (only when the caller does not bring its own subsets)
        const bool pre = opts.pre_align && !subset;
        std::vector<uint8_t> has_pre(n_reads, 0), dropped(n_reads, 0);
        std::vector<int32_t> pre_score(n_reads, 0);
        std::vector<std::vector<uint32_t>> pre_strands(n_reads);
        if (pre) {
            std::vector<Job> pj(n_reads);
            for (uint32_t r = 0; r < n_reads; ++r) { pj[r].read = q[r].data(); pj[r].n = (uint32_t)q[r].size(); }
            std::vector<std::vector<PreHit>> hits;
            prealign(pj, hits);
            for (uint32_t r = 0; r < n_reads; ++r) {
                if (prealign_select(hits[r], pre_strands[r], pre_score[r])) has_pre[r] = 1;
                else dropped[r] = 1;
            }
        }
        // stage 1: one fill + traceback per read that is aligned
        std::vector<Job> jobs;
        std::vector<int64_t> job_of(n_reads, -1);
        for (uint32_t r = 0; r < n_reads; ++r) {
            if (dropped[r]) continue;
            Job j;
            j.read = q[r].data(); j.n = (uint32_t)q[r].size();
            if (pre && !pre_strands[r].empty()) j.layout = layouts.get(pre_strands[r]);
            else j.layout = layout_for(subset ? subset + (size_t)r * stride : nullptr, stride);
            j.walk = opts.suboptimal ? WALK_ALL : WALK_BEST;
            job_of[r] = (int64_t)jobs.size();
            jobs.push_back(j);
        }
        std::vector<JobResult> out1;
        backend->run(jobs, out1);
        std::vector<JobResult> out(n_reads);
        for (uint32_t r = 0; r < n_reads; ++r) if (job_of[r] >= 0) out[r] = std::move(out1[(size_t)job_of[r]]);

        // stage 2: origin re-alignment jobs for every chain
        std::vector<std::vector<HAlign>> chains(n_reads);
        std::vector<std::vector<RealignPlan>> plans(n_reads);
        std::vector<Job> jobs2;
        for (uint32_t r = 0; r < n_reads; ++r) {
            if (dropped[r]) continue;
            if (!opts.suboptimal && out[r].chains.size() != 1) throw Error(STITCH_ERR_INTERNAL, "traceback_from returned None");
            for (const RawChain &rc : out[r].chains) chains[r].push_back(remove_clipping(opts, from_raw(rc)));
            plans[r].resize(chains[r].size());
            for (size_t c = 0; c < chains[r].size(); ++c) {
                RealignPlan &p = plans[r][c];
                if (!plan_realign(q[r], chains[r][c], p)) continue;
                p.first_job = jobs2.size();
                for (size_t t = 0; t < p.queries.size(); ++t) {
                    Job j; j.read = p.queries[t].data(); j.n = (uint32_t)p.queries[t].size(); j.layout = p.layout;
                    j.walk = WALK_FROM; j.from_contig = (uint32_t)p.contig[t];
                    jobs2.push_back(j);
                }
            }
        }
        std::vector<JobResult> out2;
        if (!jobs2.empty()) backend->run(jobs2, out2);

        // stage 3: accept / rotate back (mod.rs:412-431), then sub-optimal filtering (mod.rs:318-329)
        for (uint32_t r = 0; r < n_reads; ++r) {
            std::vector<HAlign> finals;
            for (size_t c = 0; c < chains[r].size(); ++c) {
                HAlign best = chains[r][c];
                const RealignPlan &p = plans[r][c];
                for (size_t t = 0; t < p.queries.size(); ++t) {
                    const JobResult &jr = out2[p.first_job + t];
                    if (jr.chains.empty()) continue;   // traceback_from -> None
                    HAlign na = from_raw(jr.chains[0]);
                    if (na.score > best.score && na.start_contig == p.contig[t] && best.end_contig == p.contig[t])
                        best = split_at_y(remove_clipping(opts, na), p.pivots[t]);
                }
                finals.push_back(std::move(best));
            }
            if (opts.suboptimal && finals.size() > 1) {
                std::stable_sort(finals.begin(), finals.end(), [](const HAlign &l, const HAlign &rr) { return l.score > rr.score; });
                const float min_score = (float)finals[0].score * opts.sub_pct / 100.0f;
                std::vector<HAlign> kept;
                for (auto &a : finals) if ((float)a.score >= min_score) kept.push_back(std::move(a));
                finals.swap(kept);
            }
            res.begin_read();
            for (auto &a : finals) res.add(a);
            if (has_pre[r]) res.set_pre(pre_score[r]);
        }
    }
};

}  // namespace host
}  // namespace stitch
