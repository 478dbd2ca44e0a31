// TEST INFRASTRUCTURE ONLY — CPU emulation of the CUDA kernels' tile / lane / round structure
// over the product's own __host__ __device__ DP core (stitch_b200/csrc/dp_core.h) and host driver
// (host_common.hpp).  It lets the CPU-only test tier fuzz the decomposition (pass A, insertion-chain
// scan, pass B, row-m finalize, checkpoints, windowed y-suffix tracking, fix-up, unit re-fill +
// resumable walk, re-alignment driver) against the oracle.  Exported under the emul_ prefix; the
// product library never links or loads this.
#define STITCH_API(name) emul_##name
#include "../../stitch_b200/csrc/capi_impl.hpp"
#include "../../stitch_b200/csrc/dp_packed.h"

#include <cstdio>
#include <cstdlib>
#include <vector>

// process-wide counters of the quiet-tile path (tests assert that tiles were actually skipped)
static unsigned long long g_quiet_tiles = 0, g_quiet_skipped = 0, g_quiet_mat = 0;
extern "C" void emul_quiet_counters(unsigned long long *out) { out[0] = g_quiet_tiles; out[1] = g_quiet_skipped; out[2] = g_quiet_mat; }
// process-wide counters of the path each fill took (tests assert which path ran): out[0] packed fills, out[1] wide fills,
// out[2 + LB] packed fills that ran with LB length bits (LB = 0 .. 31)
static unsigned long long g_path[2 + 32] = {0};
extern "C" void emul_path_counters(unsigned long long *out) { for (int k = 0; k < 2 + 32; ++k) out[k] = g_path[k]; }

namespace stitch {
namespace host {

#ifndef EMUL_WARPS
#define EMUL_WARPS 4
#endif

static uint32_t env_u32(const char *name, uint32_t dflt) {
    const char *v = std::getenv(name);
    return v ? (uint32_t)std::strtoul(v, nullptr, 10) : dflt;
}

// One column of a set of contigs (all contigs of the layout in the fill; one contig in a unit
// re-fill).  Mirrors fill_kernel's per-column body.
struct ColumnArgs {
    const Scoring *sc;
    const ContigEntry *ent; uint32_t C; uint32_t n_tiles;   // tile_start relative to the state arrays
    const uint8_t *bases; const uint8_t *read;
    uint32_t j, n;
    const CellState *prev; CellState *curr; CellState *ck_state;
    uint8_t *tb_col;
    ColRec *colrec_col;          // nullable
    const JumpInfo *J;           // per contig
    int32_t *Sm; uint32_t *slm, *tbm;                 // row-m summaries (in: column j-1, out: column j)
    int32_t *cm; uint32_t *cml, *cmk;                 // column best (out), nullable
    bool track; SnRec *sn; bool lastcol; LastCell *last;
};

static void emul_column(const ColumnArgs &A) {
    const Scoring &sc = *A.sc;
    const uint32_t C = A.C, j = A.j, n = A.n;
    const int W = EMUL_WARPS;
    const Row0 r0 = row0_at(sc, j, n), r0p = row0_at(sc, j - 1, n);
    ColConst cc; cc.j = j; cc.n = n; cc.q = A.read[j - 1];
    cc.xclip_score = sc.xp + std::max(sc.yp, sc.o + sc.e * (int32_t)j);
    cc.sl0j = r0.sl;
    std::vector<LaneA> la((size_t)W * 32);
    std::vector<ICarry> excl((size_t)W * 32), tileagg((size_t)W), tcarry((size_t)W);
    std::vector<XsPart> xs(C); std::vector<CmPart> cmp(C); std::vector<RowM> rowm(C);
    for (uint32_t a = 0; a < C; ++a) { xs_init(xs[a]); cm_init(cmp[a]); }
    ICarry round_carry{MIN_SCORE, 0, 0};
    for (uint32_t t0 = 0; t0 < A.n_tiles; t0 += (uint32_t)W) {
        const int nw = (int)std::min<uint32_t>((uint32_t)W, A.n_tiles - t0);
        std::vector<TileCtx> tcs((size_t)nw);
        for (int w = 0; w < nw; ++w) {   // phase A + warp scan
            const uint32_t tile = t0 + (uint32_t)w;
            uint32_t a = 0;
            while (!(tile >= A.ent[a].tile_start && tile < A.ent[a].tile_start + A.ent[a].ntiles)) ++a;
            const ContigEntry &en = A.ent[a];
            TileCtx tc; tc.a = a; tc.self_idx = en.contig_idx; tc.m = en.m; tc.tile = tile;
            tc.tile_in_contig = tile - en.tile_start; tc.J = A.J[a]; tc.circular = en.circular != 0;
            tc.wrap_src_ok = A.tbm[a] != TB_XCLIP_SUFFIX; tc.Sm_prev = A.Sm[a]; tc.slm_prev = A.slm[a];
            tcs[(size_t)w] = tc;
            for (uint32_t lane = 0; lane < 32; ++lane) {
                const uint32_t row0 = tc.tile_in_contig * TILE + lane * STRIP + 1;
                LaneA &out = la[(size_t)w * 32 + lane];
                out.has_m = 0; out.agg = ICarry{MIN_SCORE, 0, 0};
                if (row0 > en.m) continue;
                CellState up[STRIP]; uint8_t x[STRIP];
                for (int k = 0; k < STRIP; ++k) {
                    up[k] = A.prev[state_index(tile, lane, (uint32_t)k)];
                    const uint32_t i = row0 + (uint32_t)k;
                    x[k] = i <= en.m ? A.bases[en.seq_off + i - 1] : 0;
                }
                int32_t dgS; uint32_t dgsl;
                if (row0 == 1) { dgS = r0p.S; dgsl = r0p.sl; }
                else { const CellState &p = A.prev[row_index(en, row0 - 1)]; dgS = p.S; dgsl = p.sl; }
                lane_pass_a(sc, cc, tc, row0, up, dgS, dgsl, x, out, &rowm[a]);
            }
            ICarry cur[32];
            for (int l = 0; l < 32; ++l) cur[l] = la[(size_t)w * 32 + (size_t)l].agg;
            for (int d = 1; d < 32; d <<= 1) {
                ICarry nxt[32];
                for (int l = 0; l < 32; ++l)
                    nxt[l] = l >= d ? icarry_combine(cur[l - d], (uint32_t)(d * STRIP), sc.e, cur[l]) : cur[l];
                for (int l = 0; l < 32; ++l) cur[l] = nxt[l];
            }
            for (int l = 0; l < 32; ++l) excl[(size_t)w * 32 + (size_t)l] = l ? cur[l - 1] : ICarry{MIN_SCORE, 0, 0};
            tileagg[(size_t)w] = cur[31];
        }
        for (int w = 0; w < nw; ++w) {   // carry folding within the round
            const TileCtx &tc = tcs[(size_t)w];
            int w0 = w;
            while (w0 > 0 && tcs[(size_t)(w0 - 1)].a == tc.a) --w0;
            ICarry c = tcs[(size_t)w0].tile_in_contig == 0 ? icarry_row1(sc, r0) : round_carry;
            for (int u = w0; u < w; ++u) c = icarry_combine(c, TILE, sc.e, tileagg[(size_t)u]);
            tcarry[(size_t)w] = c;
        }
        round_carry = icarry_combine(tcarry[(size_t)(nw - 1)], TILE, sc.e, tileagg[(size_t)(nw - 1)]);
        for (int w = 0; w < nw; ++w) {   // phase B
            const TileCtx &tc = tcs[(size_t)w];
            const ContigEntry &en = A.ent[tc.a];
            for (uint32_t lane = 0; lane < 32; ++lane) {
                const uint32_t row0 = tc.tile_in_contig * TILE + lane * STRIP + 1;
                if (row0 > en.m) continue;
                LaneA &a_ = la[(size_t)w * 32 + lane];
                ICarry cin = lane == 0 ? tcarry[(size_t)w]
                                       : icarry_combine(tcarry[(size_t)w], lane * STRIP, sc.e, excl[(size_t)w * 32 + lane]);
                uint8_t x[STRIP];
                for (int k = 0; k < STRIP; ++k) {
                    const uint32_t i = row0 + (uint32_t)k;
                    x[k] = i <= en.m ? A.bases[en.seq_off + i - 1] : 0;
                }
                LaneB lb;
                lane_pass_b(sc, cc, tc, row0, lane, a_, cin, A.curr, A.ck_state, A.tb_col, A.track, A.sn, A.lastcol, A.last, x,
                            lb, &rowm[tc.a]);
                xs[tc.a] = xs_merge(xs[tc.a], lb.xs);
                cmp[tc.a] = cm_merge(cmp[tc.a], lb.cm);
            }
        }
    }
    for (uint32_t a = 0; a < C; ++a) {
        ContigColOut o = contig_finalize(sc, cc, A.ent[a], a, C, rowm[a], xs[a], cmp[a], r0, A.J[a], A.curr, A.ck_state, A.tb_col,
                                         A.colrec_col, A.track, A.sn, A.lastcol, A.last);
        if (A.cm) { A.cm[a] = o.cm.S; A.cmk[a] = o.cm.row; A.cml[a] = o.cm.sl; }
        A.Sm[a] = o.Sm; A.slm[a] = o.slm; A.tbm[a] = o.s_tb_m;
    }
}

struct EmulBackend : Backend {
    Aligner &al;
    uint32_t dump_seq = 0;
    uint32_t K, WINDOW, PACKED, QUIET, QUIET_EDGE, QUIET_LAST, CONE_AUDIT, CONE, LB_MIN;
    explicit EmulBackend(Aligner &a) : al(a) {
        K = std::max<uint32_t>(1, env_u32("EMUL_K", 7));          // checkpoint spacing (columns)
        WINDOW = std::max<uint32_t>(1, env_u32("EMUL_WINDOW", 6));  // columns at the end of the read filled by the wide path
        PACKED = env_u32("EMUL_PACKED", 1);                         // 0: wide path only
        QUIET = env_u32("EMUL_QUIET", 1);                           // 0: the bulk pass never skips quiet tiles
        QUIET_EDGE = env_u32("EMUL_QUIET_EDGE", 1);                 // 0: the first and last tile of a warp chunk are always computed
        QUIET_LAST = env_u32("EMUL_QUIET_LAST", 1);                 // 0: the last tile of a contig (row m) is always computed
        CONE = env_u32("EMUL_CONE", 1);                             // 0: the walk re-fills whole contigs
        CONE_AUDIT = env_u32("EMUL_CONE_AUDIT", 0);                 // 1: audit the dependency cone of the unit re-fills (experiment)
        LB_MIN = env_u32("EMUL_LB_MIN", 0);                         // packed fills take at least this many length bits (widened LB)
    }
    ~EmulBackend() {
        if (std::getenv("EMUL_UNIT_STATS")) std::fprintf(stderr, "[emul units] cone %llu full %llu\n", (unsigned long long)cone_units, (unsigned long long)full_units);
        if (CONE_AUDIT && cone_units)
            std::fprintf(stderr, "[emul cone] units %llu, cone cells %llu, differing bytes %llu, rows in the cone %.1f%% of the rows re-filled\n",
                         (unsigned long long)cone_units, (unsigned long long)cone_cells, (unsigned long long)cone_bad,
                         100.0 * (double)cone_window_rows / (double)cone_full_rows);
        g_quiet_tiles += q_tiles; g_quiet_skipped += q_skipped; g_quiet_mat += q_mat;
        if (std::getenv("EMUL_QUIET_STATS") && q_tiles) {
            std::fprintf(stderr, "   why:");
            for (int k = 0; k < 64; ++k) if (q_why[k]) std::fprintf(stderr, " %d:%llu", k, (unsigned long long)q_why[k]);
            std::fprintf(stderr, "\n   first failing cell of a tile: S %llu D-only %llu; failing cells S %llu D-only %llu", (unsigned long long)q_failS, (unsigned long long)q_failD, (unsigned long long)q_failcells[0], (unsigned long long)q_failcells[1]);
            std::fprintf(stderr, "\n   dense interior tiles by #non-boring S cells: 0:%llu 1-2:%llu 3-8:%llu 9-32:%llu 33-100:%llu >100:%llu", (unsigned long long)q_hist[0], (unsigned long long)q_hist[1], (unsigned long long)q_hist[2], (unsigned long long)q_hist[3], (unsigned long long)q_hist[4], (unsigned long long)q_hist[5]);
            std::fprintf(stderr, "\n   age (columns since the contig's last !stay) at which a dense tile turns quiet:");
            for (int k = 0; k < 12; ++k) std::fprintf(stderr, " %d:%llu", k, (unsigned long long)q_agehist[k]);
            std::fprintf(stderr, "\n   delta:");
            for (int k = 0; k < 64; ++k) if (q_delta[k]) std::fprintf(stderr, " %d:%llu", k - 32, (unsigned long long)q_delta[k]);
            std::fprintf(stderr, "\n");
        }
        if (std::getenv("EMUL_QUIET_STATS") && q_tiles)
            std::fprintf(stderr, "[emul quiet] tile-columns %llu skipped %llu (%.1f%%) materialised %llu\n", (unsigned long long)q_tiles,
                         (unsigned long long)q_skipped, 100.0 * (double)q_skipped / (double)q_tiles, (unsigned long long)q_mat),
            std::fprintf(stderr, "   skipped share by class: first tiles %.1f%% (of %llu), last tiles %.1f%% (of %llu), others %.1f%%\n", 100.0 * q_cls[0][1] / std::max<uint64_t>(q_cls[0][0], 1), (unsigned long long)q_cls[0][0], 100.0 * q_cls[1][1] / std::max<uint64_t>(q_cls[1][0], 1), (unsigned long long)q_cls[1][0], 100.0 * q_cls[2][1] / std::max<uint64_t>(q_cls[2][0], 1)),
            std::fprintf(stderr, "   dense because: special %.1f%% boundary %.1f%% !stay %.1f%% !self %.1f%% !left %.1f%%\n", 100.0 * q_special / q_tiles,
                         100.0 * q_boundary / q_tiles, 100.0 * q_nostay / q_tiles, 100.0 * q_noself / q_tiles, 100.0 * q_noleft / q_tiles);
    }

    struct Fill {
        std::vector<ColRec> colrec; std::vector<LastCell> last; std::vector<SnRec> sn;
        std::vector<CellState> ck_state; std::vector<CkSum> ck_sum; std::vector<int32_t> gcol;
        std::vector<CellState> hand_state; std::vector<CkSum> hand_sum;   // wide state at column j0 (packed -> wide hand-over)
        bool need_full_track = false;
    };

    void alloc(const Job &job, const Layout &L, Fill &F) {
        const uint32_t C = (uint32_t)L.ent.size(), PM = L.PM(), n = job.n;
        const uint32_t nb = (n + K - 1) / K;
        F.colrec.assign((size_t)(n + 1) * C, ColRec{});
        F.last.assign(PM, LastCell{});
        F.sn.assign(PM, SnRec{0x3fffffff, 7, 7, 7});   // garbage unless initialised below
        F.ck_state.assign((size_t)(nb ? nb - 1 : 0) * PM, CellState{});
        F.ck_sum.assign((size_t)(nb ? nb - 1 : 0) * C, CkSum{});
        F.gcol.assign((size_t)n + 1, MIN_SCORE);
        F.hand_state.assign(PM, CellState{MIN_SCORE, MIN_SCORE, 0, 0});
        F.hand_sum.assign(C, CkSum{});
        for (uint32_t a = 0; a < C; ++a) { int32_t t; uint32_t lx; col0_tracker(al.opts.sc, L.ent[a].m, t, lx); F.colrec[a].lx = lx; }
    }

    // Wide columns (j0, n].  j0 == 0: from column 0; else from the hand-over state at column j0 (the jump of
    // column j0 + 1 is read from colrec).  gcol[0..j0] must be filled by the caller when j0 > 0.
    void fill_wide(const Job &job, const Layout &L, uint32_t j0, uint32_t track_from, Fill &F) {
        const Scoring &sc = al.opts.sc;
        const uint32_t C = (uint32_t)L.ent.size(), PM = L.PM(), n = job.n;
        const uint8_t *bases = al.contigs.blob.data();
        std::vector<CellState> st[2];
        st[0].assign(PM, CellState{MIN_SCORE, MIN_SCORE, 0, 0}); st[1] = st[0];
        stats.cells += (uint64_t)L.cells_per_col * (n - j0);
        stats.fills += 1;
        const bool any_track = track_from <= n;
        std::vector<int32_t> cm(C), Sm(C);
        std::vector<uint32_t> cml(C), cmk(C), slm(C), tbm(C);
        for (uint32_t a = 0; a < C; ++a) {
            const ContigEntry &en = L.ent[a];
            CmPart part; cm_init(part); cm_add(part, 0, 0, 0);
            for (uint32_t i = 1; i <= en.m; ++i) {
                Col0 c0 = col0_at(sc, i, en.m);
                if (j0 == 0) st[0][row_index(en, i)] = CellState{c0.S, MIN_SCORE, c0.sl, 0};
                if (any_track) F.sn[row_index(en, i)] = sn_init(sc, c0.S, c0.sl, en.contig_idx, n);
                cm_add(part, c0.S, c0.sl, i);
            }
            if (!(part.S == 0 && part.row == 0)) throw Error(STITCH_ERR_INTERNAL, "emul: column-0 best is not (0, row 0)");
            cm[a] = 0; cmk[a] = 0; cml[a] = 0;
            Col0 cmm = col0_at(sc, en.m, en.m);
            Sm[a] = cmm.S; slm[a] = cmm.sl; tbm[a] = cmm.s_tb;
        }
        if (j0 > 0) {
            st[j0 & 1] = F.hand_state;
            for (uint32_t a = 0; a < C; ++a) { Sm[a] = F.hand_sum[a].Sm; slm[a] = F.hand_sum[a].slm; tbm[a] = F.hand_sum[a].tbm; }
        }
        std::vector<JumpInfo> J(C);
        for (uint32_t j = j0 + 1; j <= n; ++j) {
            if (j == j0 + 1 && j0 > 0) {
                for (uint32_t a = 0; a < C; ++a) { const ColRec &cr = F.colrec[(size_t)j * C + a]; J[a] = JumpInfo{cr.jscore, cr.jlen, cr.jidx, cr.jfrom}; }
            } else {
                int32_t g = cm[0];
                for (uint32_t a = 1; a < C; ++a) g = std::max(g, cm[a]);
                F.gcol[j - 1] = g;
                for (uint32_t a = 0; a < C; ++a) J[a] = select_jump(sc, L.ent.data(), C, a, cm.data(), cml.data(), cmk.data());
            }
            const bool ck = (j % K == 0) && j < n;
            ColumnArgs A{};
            A.sc = &sc; A.ent = L.ent.data(); A.C = C; A.n_tiles = L.n_tiles; A.bases = bases; A.read = job.read;
            A.j = j; A.n = n; A.prev = st[(j - 1) & 1].data(); A.curr = st[j & 1].data();
            A.ck_state = ck ? F.ck_state.data() + (size_t)(j / K - 1) * PM : nullptr;
            A.tb_col = nullptr; A.colrec_col = F.colrec.data() + (size_t)j * C; A.J = J.data();
            A.Sm = Sm.data(); A.slm = slm.data(); A.tbm = tbm.data(); A.cm = cm.data(); A.cml = cml.data(); A.cmk = cmk.data();
            A.track = j >= track_from; A.sn = F.sn.data(); A.lastcol = j == n; A.last = F.last.data();
            emul_column(A);
            if (ck) for (uint32_t a = 0; a < C; ++a) F.ck_sum[(size_t)(j / K - 1) * C + a] = CkSum{Sm[a], slm[a], tbm[a], 0};
        }
        {
            int32_t g = cm[0];
            for (uint32_t a = 1; a < C; ++a) g = std::max(g, cm[a]);
            F.gcol[n] = g;
        }
        F.need_full_track = any_track && track_from > 1 && first_candidate_column(sc, F.gcol.data(), n) < track_from;
    }

    // ---- packed path (dp_packed.h) with the kernel's structure: EMUL_WARPS warps own contiguous chunks of
    // tiles; a chunk that starts inside a contig recomputes the chain exit of the strip before it (the halo).
    struct PkState {           // rolling packed state of a set of contigs (tile_start relative to these arrays)
        std::vector<int32_t> S[2], D[2];
        std::vector<int32_t> cm, Sm, SmKey, DmKey; std::vector<uint32_t> cml, cmk, slm, tbm;   // DmKey: D key of row m (latest column)
        // quiet tiles (bulk pass only): flag per tile (state of the latest column is in the closed form), base
        // classes present in the tile (bit 0..3 = A C G T, bit 4 = anything else), closed form of the latest column
        bool quiet_on = false;
        std::vector<uint8_t> quiet, tmask; std::vector<PkQuiet> Q;
    };
    static uint32_t base_bit(uint8_t b) { return b == 'A' ? 1u : b == 'C' ? 2u : b == 'G' ? 4u : b == 'T' ? 8u : 16u; }
    static const int32_t POISON = 0x7f7f7f7f;   // what a skipped tile leaves in the state arrays (nobody may read it)
    uint64_t q_hist[6] = {0}; uint64_t q_agehist[12] = {0}; std::vector<uint32_t> q_age; uint64_t q_failS = 0, q_failD = 0, q_failcells[2] = {0, 0}; uint64_t q_why[64] = {0}, q_delta[64] = {0}; uint64_t q_cls[3][2] = {{0,0},{0,0},{0,0}}; uint64_t q_tiles = 0, q_skipped = 0, q_mat = 0, q_special = 0, q_boundary = 0, q_nostay = 0, q_noself = 0, q_noleft = 0;
    void pk_quiet_setup(const PK &pk, const ContigEntry *ent, uint32_t C, uint32_t NT, PkState &st) {
        const uint8_t *bases = al.contigs.blob.data();
        st.quiet_on = QUIET != 0;
        st.quiet.assign(NT, 0); st.tmask.assign(NT, 0); st.Q.assign(C, pk_quiet_init(pk)); st.DmKey.assign(C, pk.NEGKEY + pk.PD6);
        for (uint32_t a = 0; a < C; ++a)
            for (uint32_t i = 1; i < ent[a].m; ++i) st.tmask[ent[a].tile_start + (i - 1) / TILE] |= (uint8_t)base_bit(bases[ent[a].seq_off + i - 1]);   // ordinary rows only
    }
    struct PkCol {
        bool allow_skip = false;                            // bulk: this column may skip quiet tiles (not a checkpoint column)
        bool tail_quiet = false;                            // traceback variant (tail): quiet tiles whose cells stay below track_thr are skipped
        const ContigEntry *ent; uint32_t C, NT; const uint32_t *owner;
        const uint8_t *read; uint32_t j, n; int32_t B, Bprev; const JumpInfo *J;
        bool tb; uint8_t *tb_col; ColRec *colrec_col;       // traceback variant: packed bytes, Lx[j] per contig
        bool track; SnRec *sn; bool lastcol; LastCell *last;
        int32_t track_thr;                                  // only cells with S >= track_thr can hold a final tracker value
    };

    void pk_state_init0(const PK &pk, const ContigEntry *ent, uint32_t C, uint32_t pm, PkState &st) {
        const Scoring &sc = al.opts.sc;
        for (int b = 0; b < 2; ++b) { st.S[b].assign(pm, pk.NEGKEY); st.D[b].assign(pm, pk.NEGKEY + pk.PD6); }
        st.cm.assign(C, 0); st.cml.assign(C, 0); st.cmk.assign(C, 0); st.Sm.resize(C); st.slm.resize(C); st.tbm.resize(C); st.SmKey.resize(C);
        for (uint32_t a = 0; a < C; ++a) {
            const ContigEntry &en = ent[a];
            for (uint32_t i = 1; i <= en.m; ++i) { Col0 c0 = col0_at(sc, i, en.m); st.S[0][row_linear(en, i)] = pk_from_wide(pk, 0, c0.S, c0.sl, 0); }
            Col0 cmm = col0_at(sc, en.m, en.m);
            st.Sm[a] = cmm.S; st.slm[a] = cmm.sl; st.tbm[a] = cmm.s_tb; st.SmKey[a] = st.S[0][row_linear(en, en.m)];
        }
    }
    // from a wide checkpoint of column j0 (base Bj0); `ck` in the wide tile-transposed order of `ent_ck` positions
    void pk_state_from_ck(const PK &pk, const ContigEntry *ent, const ContigEntry *ent_ck, uint32_t C, uint32_t pm, uint32_t j0, int32_t Bj0,
                          const CellState *ck, const CkSum *sums, PkState &st) {
        for (int b = 0; b < 2; ++b) { st.S[b].assign(pm, pk.NEGKEY); st.D[b].assign(pm, pk.NEGKEY + pk.PD6); }
        st.cm.assign(C, 0); st.cml.assign(C, 0); st.cmk.assign(C, 0); st.Sm.resize(C); st.slm.resize(C); st.tbm.resize(C); st.SmKey.resize(C);
        for (uint32_t a = 0; a < C; ++a) {
            const ContigEntry &en = ent[a];
            for (uint32_t i = 1; i <= en.m; ++i) {
                const CellState &cs = ck[row_index(ent_ck[a], i)];
                st.S[j0 & 1][row_linear(en, i)] = pk_from_wide(pk, Bj0, cs.S, cs.sl, 0);
                st.D[j0 & 1][row_linear(en, i)] = pk_from_wide(pk, Bj0, cs.D, cs.dl, PP_D);
            }
            st.Sm[a] = sums[a].Sm; st.slm[a] = sums[a].slm; st.tbm[a] = sums[a].tbm;
            st.SmKey[a] = pk_from_wide(pk, Bj0, sums[a].Sm, sums[a].slm, 0);
        }
    }

    void packed_column(const PK &pk, const PkCol &A, PkState &st) {
        const Scoring &sc = al.opts.sc;
        const uint8_t *bases = al.contigs.blob.data();
        const uint32_t C = A.C, NT = A.NT, j = A.j, n = A.n;
        const int W = EMUL_WARPS;
        const int32_t B = A.B;
        const PCol pc = pk_col(pk, sc, B, A.Bprev, j, n, A.read[j - 1]);
        const Row0 r0 = row0_at(sc, j, n), r0p = row0_at(sc, j - 1, n);
        const int32_t *Sp = st.S[(j - 1) & 1].data(), *Dp = st.D[(j - 1) & 1].data();
        int32_t *Sc = st.S[j & 1].data(), *Dc = st.D[j & 1].data();
        std::vector<int32_t> tilemax(NT);
        std::vector<PkRowM> stash(C);
        const uint32_t Weff = std::min<uint32_t>((uint32_t)W, NT);
        const bool ycmode = sc.yp != MIN_SCORE && sc.xp == MIN_SCORE;
        // quiet tiles: closed form of this column per contig; sub index of a contig base against y_j, y_{j-1}, y_{j-2}, y_{j-3}
        const bool quiet_on = st.quiet_on && (!A.tb || A.tail_quiet);
        const int32_t deadrel = pk_deadrel(sc);
        // sv(xb, back, s): s[k] = sub index of contig base xb against y_{j-back-k}, k = 0 .. PKQ_L
        auto sidx = [&](uint8_t xb, int back) -> int { return ((int)j - back >= 1 && xb == A.read[j - 1 - (uint32_t)back]) ? 0 : 1; };
        auto sv = [&](uint8_t xb, int back, int *s) { for (int k = 0; k <= PKQ_L; ++k) s[k] = sidx(xb, back + k); };
        std::vector<PkQuiet> Qn(C);
        if (quiet_on) {
            const bool allow = A.allow_skip && base_bit(pc.q) != 16u;
            for (uint32_t a = 0; a < C; ++a) {
                PkFirstIn fi;
                fi.r0pkey = pk_from_wide(pk, A.Bprev, r0p.S, r0p.sl, 0);
                fi.cr1key = pk_carry_row1(pk, pc, sc, r0);
                fi.wbase = pk_wbase(pk, st.SmKey[a]);
                fi.wrap = A.ent[a].circular && st.tbm[a] != TB_XCLIP_SUFFIX;
                fi.yc1 = ycmode ? pk_key(pk, (int64_t)sc.yp + sc.o + (int64_t)sc.e - B, PP_YC, col0_slen(sc, 1, A.ent[a].m)) : pk.NEGKEY;
                Qn[a] = pk_quiet_next(pk, sc, pc, pk_jc(pk, pc, A.J[a].score, A.J[a].len), st.Q[a], allow, &fi);
                // tail: a skipped tile must not hold a cell that can still set a final y-suffix tracker (SCA:432-447)
                if (A.tb && A.track && pk_abs(pk, B, pk_max(Qn[a].bk[0], Qn[a].bk[1])) >= A.track_thr) { Qn[a].stay = 0; Qn[a].stay_first = 0; }
                ++q_why[Qn[a].why & 63]; ++q_delta[(uint32_t)(pc.delta + 32) & 63];
                if (q_age.size() < C) q_age.assign(C, 0);
                if (!Qn[a].stay) q_age[a] = 0; else if (q_age[a] < 11) ++q_age[a];
            }
        }
        std::vector<int32_t> Smat(TILE), Dmat(TILE);
        const std::vector<uint8_t> quiet_old = st.quiet;   // flags of column j-1 (what a chunk reads of its left neighbour chunk)
        const bool edge_on = quiet_on && QUIET_EDGE != 0, last_on = quiet_on && QUIET_LAST != 0;
        for (uint32_t w = 0; w < Weff; ++w) {
            const uint32_t t_lo = (uint32_t)((uint64_t)NT * w / Weff), t_hi = (uint32_t)((uint64_t)NT * (w + 1) / Weff);
            int32_t prev_exit = 0; uint32_t prev_exit_open = 0;
            bool prev_skipped = false; uint8_t qold_left = 0;
            for (uint32_t tile = t_lo; tile < t_hi; ++tile) {
                const uint32_t a = A.owner[tile];
                const ContigEntry &en = A.ent[a];
                const uint32_t tic = tile - en.tile_start;
                const bool first = tic == 0, lastt = tic + 1 == en.ntiles;
                const bool special = first || lastt;
                const int32_t Jc = pk_jc(pk, pc, A.J[a].score, A.J[a].len);
                // ---- quiet tiles: skip / materialise decisions from the flags of column j-1 ----
                const uint8_t qold = quiet_on ? st.quiet[tile] : 0;
                // tile-1 of the same contig was quiet at j-1 (across a chunk boundary: the flag its owner published)
                const uint8_t qleft = first ? 0 : (tile > t_lo ? qold_left : (edge_on ? quiet_old[tile - 1] : 0));
                qold_left = qold;
                if (quiet_on) {
                    ++q_tiles; ++q_cls[first ? 0 : (lastt ? 1 : 2)][0];
                    if ((lastt && !(last_on && !first)) || (first && !Qn[a].stay_first && Qn[a].stay)) ++q_special; else if (!edge_on && (tile == t_lo || tile + 1 == t_hi)) ++q_boundary; else if (!Qn[a].stay) ++q_nostay;
                    else if (!qold) ++q_noself; else if (!qleft) ++q_noleft;
                }
                if (quiet_on && (!lastt || (last_on && !first)) && (edge_on || (tile != t_lo && tile + 1 != t_hi)) && qold &&
                    (first ? Qn[a].stay_first != 0 : (qleft && Qn[a].stay))) {
                    const uint32_t mb = base_bit(pc.q);
                    const bool hm = (st.tmask[tile] & mb) != 0, hx = (st.tmask[tile] & ~mb) != 0;
                    tilemax[tile] = st.tmask[tile] == 0 ? pk.NEGKEY : (hm ? (hx ? pk_max(Qn[a].bk[0], Qn[a].bk[1]) : Qn[a].bk[0]) : Qn[a].bk[1]);
                    if (lastt) {   // row m: the candidates the tile would have stashed for the per-contig finish
                        int32_t dm_new;
                        stash[a] = pk_quiet_rowm(pk, pc, st.Q[a], Jc, st.SmKey[a], st.DmKey[a], sidx(bases[en.seq_off + en.m - 2], 1),
                                                 bases[en.seq_off + en.m - 1] == pc.q, &dm_new);
                        st.DmKey[a] = dm_new;
                    }
                    for (uint32_t r = 0; r < (uint32_t)TILE; ++r) { Sc[tile * TILE + r] = POISON; Dc[tile * TILE + r] = POISON; }
                    prev_skipped = true; ++q_skipped; ++q_cls[first ? 0 : (lastt ? 1 : 2)][1];
                    continue;   // stays quiet
                }
                const int32_t *SpT = Sp, *DpT = Dp;   // state of column j-1 as this tile reads it (own rows: base .. base+TILE)
                if (qold) {   // the tile's own state of column j-1 is the closed form (memory may be stale): materialise
                    ++q_mat;
                    const PkQuiet &Qp = st.Q[a];
                    for (uint32_t r = 0; r < (uint32_t)TILE; ++r) {
                        const uint8_t xb = bases[en.seq_off + tic * TILE + r];
                        int sx[PKQ_L + 1]; sv(xb, 1, sx);
                        Smat[r] = pk_quiet_S(Qp, sx[0]);
                        Dmat[r] = pk_quiet_D(pk, Qp, sx);
                    }
                    if (lastt) {   // row m is not in the closed form: its keys of column j-1 are kept per contig
                        const uint32_t rm = en.m - 1 - tic * TILE;
                        Smat[rm] = st.SmKey[a]; Dmat[rm] = st.DmKey[a];
                    }
                    SpT = Smat.data() - (size_t)tile * TILE; DpT = Dmat.data() - (size_t)tile * TILE;
                }
                const bool wrap0 = first && en.circular && st.tbm[a] != TB_XCLIP_SUFFIX;
                const int32_t wbase = pk_wbase(pk, st.SmKey[a]);
                PStrip strips[32];
                int nvs[32]; bool hasm[32];
                uint8_t xs[32][STRIP];
                auto fill_yc = [&](PStrip &ps, uint32_t row0, bool in_first) {
                    for (int k = 0; k < STRIP; ++k) {
                        ps.YC[k] = pk.NEGKEY;
                        const uint32_t i = row0 + (uint32_t)k;
                        if (in_first && ycmode && i <= en.m)
                            ps.YC[k] = pk_key(pk, (int64_t)sc.yp + sc.o + (int64_t)sc.e * i - B, PP_YC, col0_slen(sc, i, en.m));
                    }
                };
                for (uint32_t lane = 0; lane < 32; ++lane) {
                    const uint32_t row0 = tic * TILE + lane * STRIP + 1;
                    const uint32_t base = tile * TILE + lane * STRIP;
                    int32_t Sdg0;
                    if (row0 == 1) Sdg0 = pk_from_wide(pk, A.Bprev, r0p.S, r0p.sl, 0);
                    else if (lane > 0) Sdg0 = SpT[base - 1];
                    else if (qleft) Sdg0 = pk_quiet_S(st.Q[a], sidx(bases[en.seq_off + row0 - 2], 1));   // last row of a quiet tile
                    else Sdg0 = Sp[base - 1];
                    for (int k = 0; k < STRIP; ++k) xs[lane][k] = row0 + k <= en.m ? bases[en.seq_off + row0 + k - 1] : 0;
                    int nv = STRIP; bool hm = false;
                    if (special) {
                        const int64_t left = (int64_t)en.m - (int64_t)row0;
                        nv = left >= STRIP ? STRIP : (left < 0 ? 0 : (int)left);
                        hm = left >= 0 && left < STRIP;
                        fill_yc(strips[lane], row0, first);
                    }
                    nvs[lane] = nv; hasm[lane] = hm;
                    if (A.tb) {
                        if (special) pk_pass1<true, true>(pk, pc, SpT + base, DpT + base, Sdg0, xs[lane], Jc, wrap0 && lane == 0, wbase, nv, hm, strips[lane]);
                        else pk_pass1<false, true>(pk, pc, SpT + base, DpT + base, Sdg0, xs[lane], Jc, false, wbase, STRIP, false, strips[lane]);
                    } else {
                        if (special) pk_pass1<true, false>(pk, pc, SpT + base, DpT + base, Sdg0, xs[lane], Jc, wrap0 && lane == 0, wbase, nv, hm, strips[lane]);
                        else pk_pass1<false, false>(pk, pc, SpT + base, DpT + base, Sdg0, xs[lane], Jc, false, wbase, STRIP, false, strips[lane]);
                    }
                }
                int32_t tmax = pk.NEGKEY;
                bool tile_quiet = quiet_on && (!lastt || (last_on && !first)); uint32_t nfailS = 0;
                for (uint32_t lane = 0; lane < 32; ++lane) {
                    const uint32_t row0 = tic * TILE + lane * STRIP + 1;
                    const uint32_t base = tile * TILE + lane * STRIP;
                    int32_t cin; uint32_t cin_open = 0;
                    if (lane > 0) { cin = pk_carry_from_exit(pk, strips[lane - 1].exit); cin_open = strips[lane - 1].exit_open; }
                    else if (first) { cin = pk_carry_row1(pk, pc, sc, r0); cin_open = 1; }
                    else if (tile == t_lo) {   // chunk start inside a contig: the halo strip (rows row0-8 .. row0-1)
                        const uint32_t hb = tile * TILE - STRIP;
                        uint8_t x[STRIP];
                        const uint32_t hrow0 = tic * TILE - STRIP + 1;
                        for (int k = 0; k < STRIP; ++k) x[k] = bases[en.seq_off + hrow0 + k - 1];
                        PStrip h;
                        fill_yc(h, hrow0, tic == 1);
                        int32_t hs[STRIP + 1], hd[STRIP];   // S of the row before the halo rows and of the halo rows, D of the halo rows (column j-1)
                        for (int k = 0; k <= STRIP; ++k) {
                            const uint32_t row = hrow0 - 1 + (uint32_t)k;   // 1-based
                            if (qleft) {   // the neighbour chunk's last tile is quiet (its memory may be stale): closed form
                                int sx[PKQ_L + 1]; sv(bases[en.seq_off + row - 1], 1, sx);
                                hs[k] = pk_quiet_S(st.Q[a], sx[0]);
                                if (k >= 1) hd[k - 1] = pk_quiet_D(pk, st.Q[a], sx);
                            } else {
                                hs[k] = Sp[hb - 1 + (uint32_t)k];
                                if (k >= 1) hd[k - 1] = Dp[hb - 1 + (uint32_t)k];
                            }
                        }
                        pk_pass1<true, true>(pk, pc, hs + 1, hd, hs[0], x, Jc, false, wbase, STRIP, false, h);
                        cin = pk_carry_from_exit(pk, h.exit); cin_open = h.exit_open;
                    } else if (prev_skipped) { cin = pk.NEGKEY + pk.PI5; cin_open = 0; }   // chain out of a quiet tile: dead (C4)
                    else { cin = pk_carry_from_exit(pk, prev_exit); cin_open = prev_exit_open; }
                    int32_t S[STRIP], Iarr[STRIP]; uint8_t tbb[STRIP];
                    int32_t colmax = pk.NEGKEY; int32_t I_m = pk.NEGKEY; uint32_t iext_m = 0;
                    if (A.tb) {
                        if (special) pk_pass2<true, true>(pk, pc, strips[lane], cin, cin_open, nvs[lane], hasm[lane], S, colmax, tbb, Iarr, I_m, iext_m);
                        else pk_pass2<false, true>(pk, pc, strips[lane], cin, cin_open, STRIP, false, S, colmax, tbb, Iarr, I_m, iext_m);
                    } else {
                        if (special) pk_pass2<true, false>(pk, pc, strips[lane], cin, 0, nvs[lane], hasm[lane], S, colmax, nullptr, nullptr, I_m, iext_m);
                        else pk_pass2<false, false>(pk, pc, strips[lane], cin, 0, STRIP, false, S, colmax, nullptr, nullptr, I_m, iext_m);
                    }
                    for (int k = 0; k < nvs[lane]; ++k) {
                        Sc[base + k] = S[k]; Dc[base + k] = strips[lane].D6[k];
                        if (quiet_on && (!lastt || (last_on && !first))) {
                            int sx[PKQ_L + 1]; sv(xs[lane][k], 0, sx);
                            const bool okc = pk_quiet_cell(pk, Qn[a], deadrel, S[k], strips[lane].D6[k], sx);
                            if (!okc) { const bool sOK = S[k] == Qn[a].bk[sx[0]]; ++q_failcells[sOK ? 1 : 0]; if (!sOK) ++nfailS; if (tile_quiet) { if (sOK) ++q_failD; else ++q_failS; } }
                            tile_quiet = tile_quiet && okc;
                        }
                        if (A.tb) {
                            const uint32_t i = row0 + (uint32_t)k;
                            if (A.tb_col) A.tb_col[base + k] = tbb[k];
                            const bool trk = A.track && pk_abs(pk, B, S[k]) >= A.track_thr;
                            if (trk || A.lastcol)
                                pk_cell_records(pk, pc, sc, S[k], Iarr[k], tbb[k], xs[lane][k] == pc.q, en.contig_idx, i, en.m, A.J[a], j, n,
                                                trk ? &A.sn[row_index(en, i)] : nullptr, A.lastcol ? &A.last[row_index(en, i)] : nullptr);
                        }
                    }
                    if (hasm[lane]) {
                        const int km = nvs[lane];
                        stash[a] = PkRowM{strips[lane].A[km], strips[lane].D6[km], strips[lane].jp[km], I_m, A.tb ? strips[lane].fl[km] : 0u, iext_m};
                        Dc[base + km] = strips[lane].D6[km];
                        if (quiet_on) st.DmKey[a] = strips[lane].D6[km];
                    }
                    tmax = pk_max(tmax, colmax);
                }
                tilemax[tile] = tmax;
                prev_exit = strips[31].exit; prev_exit_open = strips[31].exit_open;
                prev_skipped = false;
                if (quiet_on && tile_quiet && !qold) ++q_agehist[q_age[a]];
                if (quiet_on) st.quiet[tile] = tile_quiet ? 1 : 0;
                if (quiet_on && !special) ++q_hist[nfailS == 0 ? 0 : nfailS <= 2 ? 1 : nfailS <= 8 ? 2 : nfailS <= 32 ? 3 : nfailS <= 100 ? 4 : 5];
            }
        }
        if (quiet_on) st.Q = Qn;
        // per contig: tracker / column best over rows < m, finish row m, column best
        for (uint32_t a = 0; a < C; ++a) {
            const ContigEntry &en = A.ent[a];
            int32_t kmax = pk.NEGKEY;
            for (uint32_t t = 0; t < en.ntiles; ++t) kmax = pk_max(kmax, tilemax[en.tile_start + t]);
            CmPart rows; cm_init(rows);
            XsPart tr; xs_init(tr);
            // S key of an ordinary row of column j: the closed form in a quiet tile (its memory may be stale)
            auto cell_key = [&](uint32_t a_, const ContigEntry &en_, uint32_t i) -> int32_t {
                const uint32_t tile = en_.tile_start + (i - 1) / TILE;
                if (quiet_on && st.quiet[tile]) return pk_quiet_S(Qn[a_], sidx(bases[en_.seq_off + i - 1], 0));
                return Sc[row_linear(en_, i)];
            };
            if (en.m >= 2) {
                const int32_t smax = pk_rel(pk, kmax);
                auto first_row = [&](bool full_key) -> uint32_t {
                    for (uint32_t t = 0; t < en.ntiles; ++t) {
                        const int32_t tm = tilemax[en.tile_start + t];
                        if (full_key ? tm != kmax : pk_rel(pk, tm) != smax) continue;
                        for (uint32_t r = 0; r < (uint32_t)TILE; ++r) {
                            const uint32_t i = t * TILE + r + 1;
                            if (i >= en.m) break;
                            const int32_t key = cell_key(a, en, i);
                            if (full_key ? key == kmax : pk_rel(pk, key) == smax) return i;
                        }
                    }
                    throw Error(STITCH_ERR_INTERNAL, "emul packed: column best not found");
                };
                const uint32_t frow = first_row(false);
                const int32_t fkey = cell_key(a, en, frow);
                rows.S = B + smax; rows.row = frow; rows.sl = pk_len(pk, fkey); rows.valid = 1;
                if (sc.xs != MIN_SCORE) { tr.t = B + smax + sc.xs; tr.len = pk_len(pk, kmax); tr.row = A.tb ? first_row(true) : 1; }
            }
            const PkRowMOut fo = pk_finish_rowm(pk, pc, sc, stash[a], tr, r0, A.J[a], bases[en.seq_off + en.m - 1] == pc.q, en.contig_idx, en.m, j);
            const RowMOut &ro = fo.ro;
            Sc[row_linear(en, en.m)] = fo.skey;
            if (A.tb) {
                if (A.tb_col) A.tb_col[row_linear(en, en.m)] = (uint8_t)fo.tbbyte;
                if (A.colrec_col) {
                    ColRec &cr = A.colrec_col[a];
                    cr.jscore = A.J[a].score; cr.jlen = A.J[a].len; cr.jidx = A.J[a].idx; cr.jfrom = A.J[a].from; cr.lx = ro.lx;
                }
                const uint32_t p = row_index(en, en.m);
                if (A.track && ro.c.S >= A.track_thr) sn_update(sc, A.sn[p], ro.c.S, ro.c.sl, ro.c.idx, j, n);
                if (A.lastcol) {
                    LastCell lc; lc.S = ro.c.S; lc.I = pk_abs(pk, B, stash[a].I); lc.sl = ro.c.sl; lc.il = pk_len(pk, stash[a].I);
                    lc.idx = ro.c.idx; lc.from = ro.c.from; lc.s_tb = (uint8_t)ro.s_tb; lc.i_tb = 0;
                    lc.flags = (uint8_t)((stash[a].iext ? 1 : 0) | ((stash[a].fl & 1u) ? 2 : 0)); lc.pad = 0; lc.pad2 = 0;
                    A.last[p] = lc;
                }
            }
            CmPart cmv; cm_init(cmv);
            cm_add(cmv, r0.S, r0.sl, 0);
            cmv = cm_merge(cmv, rows);
            CmPart top; top.S = ro.c.S; top.row = en.m; top.sl = ro.c.sl; top.valid = 1;
            cmv = cm_merge(cmv, top);
            st.cm[a] = cmv.S; st.cmk[a] = cmv.row; st.cml[a] = cmv.sl;
            st.Sm[a] = ro.c.S; st.slm[a] = ro.c.sl; st.tbm[a] = ro.s_tb;
            st.SmKey[a] = fo.skey;
        }
    }

    static int32_t max_of(const std::vector<int32_t> &v) { int32_t g = v[0]; for (int32_t x : v) g = std::max(g, x); return g; }
    static std::vector<uint32_t> owners_of(const ContigEntry *ent, uint32_t C, uint32_t NT) {
        std::vector<uint32_t> o(NT);
        for (uint32_t a = 0; a < C; ++a) for (uint32_t t = 0; t < ent[a].ntiles; ++t) o[ent[a].tile_start + t] = a;
        return o;
    }

    // Bulk: all n columns, no traceback outputs.  Leaves wide checkpoints, colrec[j] jump records, gcol.
    void fill_packed_bulk(const Job &job, const Layout &L, uint32_t LB, Fill &F) {
        const Scoring &sc = al.opts.sc;
        const uint32_t C = (uint32_t)L.ent.size(), PM = L.PM(), NT = L.n_tiles, n = job.n;
        const PK pk = pk_make(sc, LB);
        stats.cells += (uint64_t)L.cells_per_col * n;
        stats.fills += 1;
        PkState st;
        pk_state_init0(pk, L.ent.data(), C, PM, st);
        pk_quiet_setup(pk, L.ent.data(), C, NT, st);
        const std::vector<uint32_t> owner = owners_of(L.ent.data(), C, NT);
        F.gcol[0] = 0;
        std::vector<JumpInfo> J(C);
        int32_t B = 0;
        for (uint32_t j = 1; j <= n; ++j) {
            const int32_t Bprev = B;
            B = max_of(st.cm);
            for (uint32_t a = 0; a < C; ++a) {
                J[a] = select_jump(sc, L.ent.data(), C, a, st.cm.data(), st.cml.data(), st.cmk.data());
                ColRec &cr = F.colrec[(size_t)j * C + a];
                cr.jscore = J[a].score; cr.jlen = J[a].len; cr.jidx = J[a].idx; cr.jfrom = J[a].from;
            }
            PkCol A{};
            A.ent = L.ent.data(); A.C = C; A.NT = NT; A.owner = owner.data(); A.read = job.read; A.j = j; A.n = n;
            A.B = B; A.Bprev = Bprev; A.J = J.data();
            A.allow_skip = !((j % K == 0) && j < n);   // a checkpoint column is computed (and stored) by every tile
            packed_column(pk, A, st);
            F.gcol[j] = max_of(st.cm);
            if ((j % K == 0) && j < n) {
                const int32_t *Sc = st.S[j & 1].data(), *Dc = st.D[j & 1].data();
                for (uint32_t a = 0; a < C; ++a) {
                    const ContigEntry &en = L.ent[a];
                    for (uint32_t i = 1; i <= en.m; ++i) {
                        const int32_t s = Sc[row_linear(en, i)], d = Dc[row_linear(en, i)];
                        F.ck_state[(size_t)(j / K - 1) * PM + row_index(en, i)] = CellState{pk_abs(pk, B, s), pk_abs(pk, B, d), pk_len(pk, s), pk_len(pk, d)};
                    }
                    F.ck_sum[(size_t)(j / K - 1) * C + a] = CkSum{st.Sm[a], st.slm[a], st.tbm[a], 0};
                }
            }
        }
    }

    // Tail: columns (j0, n] again (j0 = 0 or a checkpointed column) in the traceback variant, with the
    // y-suffix trackers of every row and the column-n records the fix-up needs.
    void fill_packed_tail(const Job &job, const Layout &L, uint32_t LB, uint32_t j0, bool tracked, Fill &F) {
        const Scoring &sc = al.opts.sc;
        const uint32_t C = (uint32_t)L.ent.size(), PM = L.PM(), NT = L.n_tiles, n = job.n;
        const PK pk = pk_make(sc, LB);
        stats.cells += (uint64_t)L.cells_per_col * (n - j0);
        PkState st;
        if (j0 == 0) pk_state_init0(pk, L.ent.data(), C, PM, st);
        else pk_state_from_ck(pk, L.ent.data(), L.ent.data(), C, PM, j0, F.gcol[j0 - 1], F.ck_state.data() + (size_t)(j0 / K - 1) * PM,
                              F.ck_sum.data() + (size_t)(j0 / K - 1) * C, st);
        if (tracked)
            for (uint32_t a = 0; a < C; ++a) {
                const ContigEntry &en = L.ent[a];
                for (uint32_t i = 1; i <= en.m; ++i) { Col0 c0 = col0_at(sc, i, en.m); F.sn[row_index(en, i)] = sn_init(sc, c0.S, c0.sl, en.contig_idx, n); }
            }
        const std::vector<uint32_t> owner = owners_of(L.ent.data(), C, NT);
        std::vector<JumpInfo> J(C);
        pk_quiet_setup(pk, L.ent.data(), C, NT, st);   // quiet tiles in the tail: no tile is quiet at the checkpoint
        for (uint32_t a = 0; a < C; ++a) st.DmKey[a] = st.D[j0 & 1][row_linear(L.ent[a], L.ent[a].m)];
        // every row ends with a tracker value >= max_j G(j) - W' (dp_core.h: first_candidate_column): cells below can be skipped
        int32_t thr = MIN_SCORE;
        if (tracked) {
            thr = max_of(F.gcol) - track_margin(sc, job.walk == WALK_BEST);
        }
        for (uint32_t j = j0 + 1; j <= n; ++j) {
            for (uint32_t a = 0; a < C; ++a) { const ColRec &cr = F.colrec[(size_t)j * C + a]; J[a] = JumpInfo{cr.jscore, cr.jlen, cr.jidx, cr.jfrom}; }
            PkCol A{};
            A.ent = L.ent.data(); A.C = C; A.NT = NT; A.owner = owner.data(); A.read = job.read; A.j = j; A.n = n;
            A.B = F.gcol[j - 1]; A.Bprev = j >= 2 ? F.gcol[j - 2] : 0; A.J = J.data();
            A.tb = true; A.tb_col = nullptr; A.colrec_col = F.colrec.data() + (size_t)j * C;
            A.track = tracked; A.sn = F.sn.data(); A.lastcol = j == n; A.last = F.last.data(); A.track_thr = thr;
            A.tail_quiet = true; A.allow_skip = j != n;   // column n: every cell leaves its record for the end-of-read fix-up
            packed_column(pk, A, st);
        }
    }

    // The packed re-fill of the walk as the CUDA kernel does it (pk_refill_unit): columns (jb, j] only, and, when
    // pk_cone_plan allows, restricted to the cone of the entry cell (i_entry, j): the tiles above the window hold the lowest
    // in-band keys from the start, the tiles of the window above the cone's current top tile keep their stale values, and
    // TbUnit::has() makes the walk ask for a new unit whenever it would read outside the cone.  EMUL_CONE=0: whole contigs.
    // EMUL_CONE_AUDIT=1 additionally compares every traceback byte inside the cone with a full re-fill.
    uint64_t cone_units = 0, cone_bad = 0, cone_cells = 0, cone_window_rows = 0, cone_full_rows = 0, full_units = 0;
    void load_unit_packed(const Job &job, const Layout &L, uint32_t LB, const Fill &F, uint32_t a, uint32_t j, std::vector<uint8_t> &bytes,
                          std::vector<ColRec> &ucr, TbUnit &u, uint32_t i_entry = 0) {
        const Scoring &sc = al.opts.sc;
        const uint32_t C = (uint32_t)L.ent.size(), PM = L.PM(), n = job.n;
        const uint32_t b = (j - 1) / K, jb = b * K;
        const PK pk = pk_make(sc, LB);
        ContigEntry en = L.ent[a];
        const uint32_t pm = en.ntiles * TILE;
        const ContigEntry en_ck = en;
        en.tile_start = 0;
        PkCone cone; cone.on = false; cone.slope = 0; cone.win_lo = 0; cone.win_n = en.ntiles;
        if (CONE) cone = pk_cone_plan(sc, en, i_entry, j, jb);
        const std::vector<uint32_t> owner(en.ntiles, 0);
        auto run = [&](bool use_cone, std::vector<uint8_t> &out_bytes, std::vector<ColRec> &out_cr) {
            PkState st;
            if (b == 0) pk_state_init0(pk, &en, 1, pm, st);
            else pk_state_from_ck(pk, &en, &en_ck, 1, pm, jb, F.gcol[jb - 1], F.ck_state.data() + (size_t)(b - 1) * PM,
                                  F.ck_sum.data() + (size_t)(b - 1) * C + a, st);
            out_bytes.assign((size_t)(j - jb) * pm, 0);
            out_cr.assign(j - jb, ColRec{});
            const size_t above = use_cone ? (size_t)cone.win_lo * TILE : 0;   // rows (0-based) above the window
            for (int par = 0; par < 2 && use_cone; ++par)
                for (size_t r = 0; r < above; ++r) { st.S[par][r] = pk.NEGKEY; st.D[par][r] = pk.NEGKEY + pk.PD6; }
            for (uint32_t jj = jb + 1; jj <= j; ++jj) {
                const ColRec &cr = F.colrec[(size_t)jj * C + a];
                JumpInfo J{cr.jscore, cr.jlen, cr.jidx, cr.jfrom};
                PkCol A{};
                A.ent = &en; A.C = 1; A.NT = en.ntiles; A.owner = owner.data(); A.read = job.read; A.j = jj; A.n = n;
                A.B = F.gcol[jj - 1]; A.Bprev = jj >= 2 ? F.gcol[jj - 2] : 0; A.J = &J;
                A.tb = true; A.tb_col = out_bytes.data() + (size_t)(jj - jb - 1) * pm; A.colrec_col = out_cr.data() + (jj - jb - 1);
                packed_column(pk, A, st);
                if (use_cone) {   // the tiles above the cone's top tile are "not computed": they keep what they held
                    const size_t stale = (size_t)pk_cone_top_tile(cone, i_entry, j, jj) * TILE;
                    for (size_t r = 0; r < stale && r < (size_t)en.m; ++r) {
                        st.S[jj & 1][r] = r < above ? pk.NEGKEY : st.S[(jj - 1) & 1][r];
                        st.D[jj & 1][r] = r < above ? pk.NEGKEY + pk.PD6 : st.D[(jj - 1) & 1][r];
                    }
                }
            }
        };
        run(cone.on, bytes, ucr);
        stats.cells += (uint64_t)(cone.on ? cone.win_n * TILE : en.m) * (j - jb);
        u.bytes = bytes.data(); u.cr = ucr.data(); u.a = a; u.jb = jb; u.je = j; u.pm = pm;
        u.i_hi = cone.on ? i_entry : 0xffffffffu; u.slope = cone.slope;
        if (cone.on) ++cone_units; else ++full_units;
        if (CONE_AUDIT && cone.on) {
            std::vector<uint8_t> bytes2; std::vector<ColRec> ucr2;
            run(false, bytes2, ucr2);
            for (uint32_t jj = jb + 1; jj <= j; ++jj) {
                const int64_t top = (int64_t)i_entry - (int64_t)cone.slope * (int64_t)(j - jj);
                const uint32_t lo = top < 1 ? 1u : (uint32_t)top;
                cone_window_rows += i_entry - lo + 1; cone_full_rows += en.m;
                for (uint32_t r = lo; r <= i_entry; ++r) {
                    ++cone_cells;
                    if (bytes2[(size_t)(jj - jb - 1) * pm + r - 1] != bytes[(size_t)(jj - jb - 1) * pm + r - 1]) {
                        ++cone_bad;
                        if (std::getenv("EMUL_CONE_DEBUG"))
                            std::fprintf(stderr, "[cone diff] a %u m %u K %u jb %u j %u i_entry %u slope %u win %u+%u | cell (%u, %u): cone %u full %u\n", a, en.m, K, jb, j,
                                         i_entry, cone.slope, cone.win_lo, cone.win_n, r, jj, bytes[(size_t)(jj - jb - 1) * pm + r - 1], bytes2[(size_t)(jj - jb - 1) * pm + r - 1]);
                    }
                }
            }
        }
    }

    // Returns the length bits of the packed path, or 0 when the read ran on the wide path.
    uint32_t fill(const Job &job, const Layout &L, uint32_t track_from, Fill &F, bool allow_packed) {
        const Scoring &sc = al.opts.sc;
        const uint32_t n = job.n;
        alloc(job, L, F);
        uint32_t m_max = 0;
        for (const auto &e : L.ent) m_max = std::max(m_max, e.m);
        uint32_t LB = (allow_packed && PACKED) ? pk_plan(sc, n, m_max) : 0;
        if (!LB) { ++g_path[1]; fill_wide(job, L, 0, track_from, F); return 0; }
        LB = std::max(LB, LB_MIN);   // (cuda_backend.cu run_chunk: one LB per launch, the largest any job needs)
        ++g_path[0]; ++g_path[2 + (LB & 31u)];
        fill_packed_bulk(job, L, LB, F);
        // the tail restarts at the last checkpoint before the first column that can hold a final y-suffix
        // tracker (dp_core.h: first_candidate_column); column n is always part of it
        const bool tracked = sc.ys != MIN_SCORE;
        const uint32_t jc = tracked ? std::min(first_candidate_column(sc, F.gcol.data(), n, job.walk == WALK_BEST), n) : n;
        const uint32_t j0 = ((jc - 1) / K) * K;
        fill_packed_tail(job, L, LB, j0, tracked, F);
        F.need_full_track = false;
        ++stats.launches;
        return LB;
    }

    // Re-fills contig `a` over the block of columns holding column j.
    void load_unit(const Job &job, const Layout &L, const Fill &F, uint32_t a, uint32_t j, std::vector<uint8_t> &bytes,
                   std::vector<ColRec> &ucr, TbUnit &u) {
        const Scoring &sc = al.opts.sc;
        const uint32_t C = (uint32_t)L.ent.size(), PM = L.PM(), n = job.n;
        const uint32_t b = (j - 1) / K, jb = b * K, je = std::min(jb + K, n);
        ContigEntry en = L.ent[a];
        const uint32_t pm = en.ntiles * TILE, gbase = en.tile_start * TILE;
        en.tile_start = 0;
        std::vector<CellState> st[2];
        st[0].assign(pm, CellState{MIN_SCORE, MIN_SCORE, 0, 0}); st[1] = st[0];
        int32_t Sm; uint32_t slm, tbm;
        if (b == 0) {
            for (uint32_t i = 1; i <= en.m; ++i) { Col0 c0 = col0_at(sc, i, en.m); st[0][row_index(en, i)] = CellState{c0.S, MIN_SCORE, c0.sl, 0}; }
            Col0 cmm = col0_at(sc, en.m, en.m);
            Sm = cmm.S; slm = cmm.sl; tbm = cmm.s_tb;
        } else {
            const CellState *ck = F.ck_state.data() + (size_t)(b - 1) * PM + gbase;
            for (uint32_t p = 0; p < pm; ++p) st[jb & 1][p] = ck[p];
            const CkSum &cs = F.ck_sum[(size_t)(b - 1) * C + a];
            Sm = cs.Sm; slm = cs.slm; tbm = cs.tbm;
        }
        bytes.assign((size_t)(je - jb) * pm, 0);
        ucr.assign(je - jb, ColRec{});
        stats.cells += (uint64_t)en.m * (je - jb);
        for (uint32_t jj = jb + 1; jj <= je; ++jj) {
            const ColRec &cr = F.colrec[(size_t)jj * C + a];
            JumpInfo J{cr.jscore, cr.jlen, cr.jidx, cr.jfrom};
            ColumnArgs A{};
            A.sc = &sc; A.ent = &en; A.C = 1; A.n_tiles = en.ntiles; A.bases = al.contigs.blob.data(); A.read = job.read;
            A.j = jj; A.n = n; A.prev = st[(jj - 1) & 1].data(); A.curr = st[jj & 1].data(); A.ck_state = nullptr;
            A.tb_col = bytes.data() + (size_t)(jj - jb - 1) * pm; A.colrec_col = ucr.data() + (jj - jb - 1); A.J = &J;
            A.Sm = &Sm; A.slm = &slm; A.tbm = &tbm; A.cm = nullptr; A.cml = nullptr; A.cmk = nullptr;
            A.track = false; A.sn = nullptr; A.lastcol = false; A.last = nullptr;
            emul_column(A);
        }
        u.bytes = bytes.data(); u.cr = ucr.data(); u.a = a; u.jb = jb; u.je = je; u.pm = pm; u.i_hi = 0xffffffffu; u.slope = 0;
    }

    void run_one(const Job &job, JobResult &res) {
        const Layout &L = al.layouts.layouts[job.layout];
        const Scoring &sc = al.opts.sc;
        const uint32_t C = (uint32_t)L.ent.size(), n = job.n;
        if (n == 0) throw Error(STITCH_ERR_INVALID, "empty read");
        const bool tracked_mode = sc.ys != MIN_SCORE;   // Sn can only matter when y-suffix clipping is free
        uint32_t track_from = tracked_mode ? (n > WINDOW ? n - WINDOW + 1 : 1) : n + 1;
        Fill F;
        const uint32_t LB = fill(job, L, track_from, F, true);
        if (F.need_full_track) { ++stats.launches; fill(job, L, 1, F, false); }
        for (uint32_t a = 0; a < C; ++a)
            fixup_contig(sc, L.ent[a], n, F.last.data(), F.sn.data(), tracked_mode, &F.colrec[(size_t)n * C + a].lx);
        if (const char *dump = std::getenv("STITCH_DUMP_DIR")) dump_job(dump, dump_seq++, F.last, F.sn, F.colrec, std::vector<uint8_t>());
        ReadView v;
        v.sc = sc; v.ent = L.ent.data(); v.C = C; v.n = n; v.colrec = F.colrec.data();
        v.last = F.last.data(); v.sn = F.sn.data(); v.contig_bases = al.contigs.blob.data(); v.read = job.read;
        v.unit.bytes = nullptr; v.unit.cr = nullptr; v.unit.a = 0xffffffffu; v.unit.jb = v.unit.je = v.unit.pm = 0; v.unit.i_hi = 0xffffffffu; v.unit.slope = 0;
        std::vector<uint8_t> unit_bytes; std::vector<ColRec> unit_cr;
        const uint32_t cap = 2 * n + 4 * C + 64;
        auto do_walk = [&](uint32_t a_end, RawChain &rc) -> uint32_t {
            uint32_t c = cap;
            for (;;) {
                rc.ops.assign(c, OutOp{0, 0, 0});
                WalkState ws;
                walk_begin(v, a_end, rc.ops.data(), c, ws, rc.h);
                uint32_t s;
                while ((s = walk_run(v, ws, rc.h)) == WALK_NEED_UNIT) {
                    if (LB) load_unit_packed(job, L, LB, F, ws.a, ws.j, unit_bytes, unit_cr, v.unit, ws.i);
                    else load_unit(job, L, F, ws.a, ws.j, unit_bytes, unit_cr, v.unit);
                }
                if (s != WALK_OVERFLOW) break;
                c *= 2;
            }
            rc.ops.resize(rc.h.n_ops);
            return rc.h.status;
        };
        if (job.walk == WALK_BEST) {
            RawChain rc;
            uint32_t s = do_walk(pick_end(v, nullptr), rc);
            if (s == WALK_PANIC) throw Error(STITCH_ERR_INTERNAL, "traceback reached a state the reference panics on");
            if (s == WALK_OK) res.chains.push_back(std::move(rc));
        } else if (job.walk == WALK_FROM) {
            const int32_t a_end = v.pos_of(job.from_contig);
            if (a_end >= 0) {
                RawChain rc;
                uint32_t s = do_walk((uint32_t)a_end, rc);
                if (s == WALK_PANIC) throw Error(STITCH_ERR_INTERNAL, "traceback reached a state the reference panics on");
                if (s == WALK_OK) res.chains.push_back(std::move(rc));
            }
        } else {   // traceback_all (TB:152-217) over the layout's contigs
            std::vector<uint8_t> seen(C, 0);
            uint32_t n_seen = 0;
            auto mark = [&](uint32_t idx) {
                const int32_t p = v.pos_of(idx);
                if (p >= 0 && !seen[(size_t)p]) { seen[(size_t)p] = 1; ++n_seen; }
            };
            while (n_seen < C) {
                const uint32_t a_end = pick_end(v, seen.data());
                RawChain rc;
                uint32_t s = do_walk(a_end, rc);
                if (s == WALK_PANIC) throw Error(STITCH_ERR_INTERNAL, "traceback reached a state the reference panics on");
                if (s != WALK_OK) { mark(L.ent[a_end].contig_idx); continue; }
                mark(rc.h.start_contig_idx); mark(rc.h.end_contig_idx);
                for (const OutOp &o : rc.ops) if (o.kind == OP_XJUMP) mark(o.a);
                res.chains.push_back(std::move(rc));
            }
        }
    }

    // Pre-alignment contig selection exactly as prealign_core.h defines it (the CUDA kernel's outputs are compared with
    // these in the gpu tier), sequentially.
    KmerIndex kindex;
    void prealign(const std::vector<Job> &reads, std::vector<std::vector<PreHit>> &out) override {
        const Opts &o = al.opts;
        const Contigs &c = al.contigs;
        if (kindex.K != o.kmer) kindex.build(c, o.kmer);
        out.assign(reads.size(), std::vector<PreHit>());
        const uint32_t K = o.kmer, W = o.band;
        for (size_t r = 0; r < reads.size(); ++r) {
            const uint8_t *read = reads[r].read; const uint32_t n = reads[r].n;
            std::vector<uint32_t> cnt(c.n_strands, 0);
            std::vector<std::pair<uint32_t, uint32_t>> hits;   // (strand, shifted diagonal)
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
            uint32_t need = pre_need(o.pre_min_score, o.sc.match, K);
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
                uint32_t best = 0;
                for (uint32_t b = 0; b < n_bins; ++b) best = std::max(best, bins[b] + (b + 1 < n_bins ? bins[b + 1] : 0u));
                const int32_t sc = pre_score_of(o.sc.match, best, K);
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

    void run(const std::vector<Job> &jobs, std::vector<JobResult> &out) override {
        out.assign(jobs.size(), JobResult());
        for (size_t k = 0; k < jobs.size(); ++k) run_one(jobs[k], out[k]);
    }
};

Backend *stitch_make_backend(Aligner &al, int) { return new EmulBackend(al); }

}  // namespace host
}  // namespace stitch

// sizeof of the device structs whose sizes tests/ckplan.py uses to restate the shared-memory layouts of the CUDA kernels
// (PkColConst: kernels_packed.cuh, not compiled here; same members)
extern "C" void emul_struct_sizes(uint32_t *out) {
    using namespace stitch;
    struct PkColConst { PCol pc; int32_t r0pkey, cr1key; uint8_t yq[PKQ_L + 2]; };
    const uint32_t s[] = {sizeof(JumpInfo), sizeof(PkRowM), sizeof(PkQuiet), sizeof(ContigEntry), sizeof(PkColConst), sizeof(RowM),
                          sizeof(XsPart), sizeof(CmPart), sizeof(ICarry)};
    for (size_t k = 0; k < sizeof(s) / sizeof(s[0]); ++k) out[k] = s[k];
}

// pk_plan (dp_packed.h) of the scoring the product derives from these options: the length bits of the packed path, 0 = the
// wide path, -1 = options the product refuses
extern "C" int32_t emul_pk_plan(const stitch_opts *o, uint32_t n, uint32_t m_max) {
    try {
        return (int32_t)stitch::pk_plan(stitch::host::make_opts(*o).sc, n, m_max);
    } catch (const stitch::host::Error &) {
        return -1;
    }
}
