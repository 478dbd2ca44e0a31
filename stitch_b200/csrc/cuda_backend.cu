// cuda_backend.cu — the sm_100a implementation of the DP backend + the product's C ABI.
//
// Kernels (one launch each per chunk of reads):
//   fill_kernel    K1  column-by-column DP fill of every contig-strand of a read; persistent CTAs pull
//                      reads from a queue; replaces MCA::custom's loop body (multi_contig_aligner.rs:270-347
//                      = SCA:188-239 + 677-697 + 292-451 of the reference)
//   fixup_kernel   K2  end-of-read fix-up of column n (SCA:453-555), one thread per contig-strand
//   walk_kernel    K3  end-contig selection + pointer walk (traceback/mod.rs:129-373)
// The arithmetic lives in dp_core.h (shared with the CPU emulator the tests fuzz against the
// oracle); this file is the parallel glue: tile/lane mapping, warp-shuffle max-plus scan of the
// insertion chain, cross-warp carry folding through shared memory, per-contig reductions.
//
// There is no CPU path: every entry point fails with STITCH_ERR_CUDA when no device is usable.
#include <cuda_runtime.h>

#include <algorithm>
#include <numeric>

#define STITCH_API(name) stitch_##name
#include "capi_impl.hpp"
#include "kernels_wide.cuh"
#include "kernels_packed.cuh"
#include "kernels_walk.cuh"
#include "kernels_prealign.cuh"

namespace stitch {
namespace gpu {

using host::Error;

#define CUDA_CHECK(expr)                                                                              \
    do {                                                                                              \
        cudaError_t err__ = (expr);                                                                   \
        if (err__ != cudaSuccess)                                                                     \
            throw Error(err__ == cudaErrorMemoryAllocation ? STITCH_ERR_NOMEM : STITCH_ERR_CUDA,      \
                        std::string(#expr) + ": " + cudaGetErrorString(err__));                       \
    } while (0)

constexpr int FILL_WARPS = 8;
#ifndef STITCH_PACK_WARPS
#define STITCH_PACK_WARPS 16
#endif
constexpr int PACK_WARPS = STITCH_PACK_WARPS;   // warps of a fill CTA (build-time: -DSTITCH_PACK_WARPS=12 trades four warps for 170 registers per thread)
constexpr int WALK_WARPS = 16;

// ---------------------------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------------------------
template <typename T>
struct DevBuf {
    T *p = nullptr; size_t cap = 0;
    void reserve(size_t n) {
        if (n <= cap) return;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        const size_t want = n + n / 8 + 64;
        CUDA_CHECK(cudaMalloc(&p, want * sizeof(T)));
        cap = want;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    ~DevBuf() { release(); }
};
template <typename T>
struct PinBuf {
    T *p = nullptr; size_t cap = 0;
    void reserve(size_t n) {
        if (n <= cap) return;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        const size_t want = n + n / 8 + 64;
        CUDA_CHECK(cudaMallocHost(&p, want * sizeof(T)));
        cap = want;
    }
    ~PinBuf() { if (p) cudaFreeHost(p); }
};

static inline uint64_t round_up(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }

static uint32_t env_u32(const char *name, uint32_t dflt) {
    const char *v = std::getenv(name);
    return v && *v ? (uint32_t)std::strtoul(v, nullptr, 10) : dflt;
}

struct CudaBackend : host::Backend {
    host::Aligner &al;
    int device;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[16] = {};
    int marks[16] = {}; int n_marks = 0;
    enum { T_H2D = 0, T_PACKED, T_TAIL, T_WIDE, T_FIXUP, T_REDO, T_WALK, T_D2H, T_END };
    int num_sms = 0;
    uint32_t max_inflight = 0;
    size_t uploaded_layouts = 0;
    uint64_t uploaded_generation = ~0ull;
    uint32_t K = 256;        // checkpoint spacing (columns) of the current batch
    uint32_t K_base = 256;   // its default; STITCH_CK_EVERY overrides (tests)
    bool ck_auto = true;     // no override: a batch that fits in one launch with half the spacing uses K_base / 2
    uint32_t WINDOW = 64;    // columns at the end of the read with y-suffix tracking; STITCH_TRACK_WINDOW
    const uint8_t *device_reads = nullptr;   // set for run_device()

    DevBuf<uint8_t> d_contigs, d_reads, d_unit, d_ptbases;
    DevBuf<ContigEntry> d_ents;
    DevBuf<uint16_t> d_owners;
    DevBuf<LayoutDesc> d_layouts;
    DevBuf<JobDesc> d_jobs;
    DevBuf<uint32_t> d_order;
    DevBuf<CellState> d_state, d_ck, d_hand;
    DevBuf<CkSum> d_handsum;
    DevBuf<int32_t> d_pstate, d_wpstate, d_pck;
    DevBuf<uint32_t> d_tailj0, d_done;
    DevBuf<unsigned long long> d_dbg, d_qstats;
    bool debug_stats = false;
    DevBuf<ColRec> d_ucr;
    uint32_t use_packed = 1;   // STITCH_PACKED=0 forces the wide kernels (tests)
    uint32_t walk_in_kernel = 1;   // STITCH_WALK_IN_KERNEL=0: separate fix-up / walk kernels after the packed fill
    // STITCH_CLUSTER: CTAs per read in the packed kernel (1, 2, 4, 8, 16); 0 = automatic: one CTA per read when there are
    // enough reads to fill the GPU (measured best on config 2), a cluster per read when there are only a few (the origin
    // re-alignment fills, small batches), with the rolling state in the cluster's shared memory when it fits
    uint32_t cluster_pref = 0;
    uint32_t cluster_min_tiles = 4 * PACK_WARPS;   // STITCH_CLUSTER_MIN_TILES: smaller layouts use one CTA per read
    uint32_t cluster_smem = 1;   // STITCH_CLUSTER_SMEM=0: clusters keep the rolling state in global memory
    uint32_t quiet_tiles = 1;    // STITCH_QUIET=0: the packed bulk pass computes every tile of every column
    uint32_t quiet_tail = 1;     // STITCH_QUIET_TAIL=0: the tail columns compute every tile
    uint32_t cone_refill = 1;    // STITCH_CONE=0: the walk re-fills whole contigs (dp_packed.h: cone re-fill)
    // STITCH_STAGE_DEPTH: slots of the staging ring per warp (2 or 4).  Measured at 592 config-2 reads: 475 / 467 / 452 GCUPS
    // at 2 / 3 / 4 slots: the ring's shared memory is taken from the L1 (184 KB instead of 110 KB per CTA), which costs more
    // than the deeper prefetch brings; 2 is the default
    uint32_t stage_depth_pref = 2;
    uint32_t quiet_first = 1, quiet_edge = 1, quiet_last = 1;   // STITCH_QUIET_FIRST / _EDGE / _LAST = 0: those tiles are always computed
    DevBuf<CkSum> d_cksum;
    DevBuf<int32_t> d_gcol;
    DevBuf<ColRec> d_colrec;
    DevBuf<LastCell> d_last;
    DevBuf<SnRec> d_sn;
    DevBuf<OutOp> d_ops;
    DevBuf<ChainHdr> d_chains;
    DevBuf<JobOut> d_jobout;
    DevBuf<uint32_t> d_counter;
    PinBuf<uint8_t> h_reads;
    PinBuf<JobDesc> h_jobs;
    PinBuf<uint32_t> h_order, h_redo;
    DevBuf<uint32_t> d_redo;
    PinBuf<OutOp> h_ops;
    PinBuf<ChainHdr> h_chains;
    PinBuf<JobOut> h_jobout;

    CudaBackend(host::Aligner &a, int dev) : al(a), device(dev) {
        int count = 0;
        cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess || count == 0)
            throw Error(STITCH_ERR_CUDA, std::string("no CUDA device available (") + cudaGetErrorString(e) +
                                             "); stitch_b200 has no CPU fallback");
        if (dev < 0 || dev >= count) throw Error(STITCH_ERR_INVALID, "bad device index");
        CUDA_CHECK(cudaSetDevice(dev));
        cudaDeviceProp prop;
        CUDA_CHECK(cudaGetDeviceProperties(&prop, dev));
        num_sms = prop.multiProcessorCount;
        CUDA_CHECK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        for (auto &x : ev) CUDA_CHECK(cudaEventCreate(&x));
        d_contigs.reserve(al.contigs.blob.size() + 1024);   // strips of the last tile over-read
        CUDA_CHECK(cudaMemcpy(d_contigs.p, al.contigs.blob.data(), al.contigs.blob.size(), cudaMemcpyHostToDevice));
        d_counter.reserve(8);
        ck_auto = std::getenv("STITCH_CK_EVERY") == nullptr;
        K_base = std::max<uint32_t>(1, env_u32("STITCH_CK_EVERY", K_base));
        K = K_base;
        WINDOW = std::max<uint32_t>(1, env_u32("STITCH_TRACK_WINDOW", WINDOW));
        use_packed = env_u32("STITCH_PACKED", 1);
        walk_in_kernel = env_u32("STITCH_WALK_IN_KERNEL", 1);
        debug_stats = env_u32("STITCH_DEBUG_STATS", 0) != 0;
        cluster_pref = std::min<uint32_t>(16, env_u32("STITCH_CLUSTER", cluster_pref));
        cluster_min_tiles = env_u32("STITCH_CLUSTER_MIN_TILES", cluster_min_tiles);
        cluster_smem = env_u32("STITCH_CLUSTER_SMEM", 1);
        quiet_tiles = env_u32("STITCH_QUIET", quiet_tiles);
        cone_refill = env_u32("STITCH_CONE", 1);
        stage_depth_pref = env_u32("STITCH_STAGE_DEPTH", stage_depth_pref) >= 4 ? 4u : 2u;
        quiet_first = env_u32("STITCH_QUIET_FIRST", 1); quiet_edge = env_u32("STITCH_QUIET_EDGE", 1); quiet_last = env_u32("STITCH_QUIET_LAST", 1); quiet_tail = env_u32("STITCH_QUIET_TAIL", 1);
    }
    ~CudaBackend() override {
        cudaSetDevice(device);
        for (auto &x : ev) if (x) cudaEventDestroy(x);
        if (stream) cudaStreamDestroy(stream);
    }
    void set_max_inflight(uint32_t n) override { max_inflight = n; }

    void upload_layouts() {
        const auto &Ls = al.layouts.layouts;
        if (uploaded_layouts == Ls.size() && uploaded_generation == al.layouts.generation) return;
        uploaded_generation = al.layouts.generation;
        std::vector<ContigEntry> ents; std::vector<uint16_t> owners; std::vector<LayoutDesc> descs;
        for (const auto &L : Ls) {
            LayoutDesc d{};
            d.ent_off = (uint32_t)ents.size(); d.C = (uint32_t)L.ent.size(); d.n_tiles = L.n_tiles;
            d.owner_off = (uint32_t)owners.size(); d.PM = L.PM();
            for (uint32_t a = 0; a < d.C; ++a) {
                ents.push_back(L.ent[a]);
                d.max_ctiles = std::max(d.max_ctiles, L.ent[a].ntiles);
                for (uint32_t t = 0; t < L.ent[a].ntiles; ++t) owners.push_back((uint16_t)a);
            }
            descs.push_back(d);
        }
        d_ents.reserve(ents.size()); d_owners.reserve(owners.size()); d_layouts.reserve(descs.size());
        CUDA_CHECK(cudaMemcpy(d_ents.p, ents.data(), ents.size() * sizeof(ContigEntry), cudaMemcpyHostToDevice));
        CUDA_CHECK(cudaMemcpy(d_owners.p, owners.data(), owners.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
        CUDA_CHECK(cudaMemcpy(d_layouts.p, descs.data(), descs.size() * sizeof(LayoutDesc), cudaMemcpyHostToDevice));
        uploaded_layouts = Ls.size();
    }

    // opt-in dynamic shared memory of an sm_100 CTA (227 KB) minus the kernels' static shared memory
    static constexpr size_t SMEM_LIMIT = 227 * 1024 - 2048;
    static constexpr uint32_t K_MAX = 8192;   // the walk stages 21 bytes per column of a unit in shared memory
    uint32_t blocks_of(uint32_t n) const { return (n + K - 1) / K; }
    uint32_t plan_LB(const host::Job &j) const {   // length bits of the packed path, 0 = wide path
        if (!use_packed) return 0;
        const host::Layout &L = al.layouts.layouts[j.layout];
        uint32_t m_max = 0;
        for (const auto &e : L.ent) m_max = std::max(m_max, e.m);
        const uint32_t LB = pk_plan(al.opts.sc, j.n, m_max);
        // shared memory of the packed fill: per-contig / per-tile tables + the stage ring; otherwise the read takes the
        // (slow, exact) wide path.  The walk phase's staging is optional: run_chunk sizes it with the real K and falls back
        // to the separate walk kernel (or to unstaged contig bases) when it does not fit.
        if (LB && PackSmem::bytes((uint32_t)L.ent.size(), L.n_tiles, PACK_WARPS, PackSmem::default_stage(PACK_WARPS)) > SMEM_LIMIT) return 0;
        return LB;
    }
    // records a read holds from its fill until its walk is done (CellState/ColRec/... counts)
    // ck: wide checkpoints (CellState records); pck: packed checkpoints (raw keys, 2 per cell)
    struct Need { uint64_t colrec, cell, ck, cksum, gcol, pck; };
    Need need_of(const host::Job &j, bool packed) const {
        const host::Layout &L = al.layouts.layouts[j.layout];
        const uint64_t C = L.ent.size(), PM = L.PM(), nb = blocks_of(j.n);
        const uint64_t late = packed ? PK_LATE_CKS : 0;   // late checkpoints of the packed fill (kernels_packed.cuh)
        return Need{(uint64_t)(j.n + 1) * C, PM, packed ? 0 : (nb - 1) * PM, (nb - 1 + late) * C, (uint64_t)j.n + 1, packed ? (nb - 1 + late) * 2 * PM : 0};
    }
    static uint64_t need_bytes(const Need &n) {
        return n.colrec * sizeof(ColRec) + n.cell * (sizeof(LastCell) + sizeof(SnRec)) + n.ck * sizeof(CellState) + n.pck * 4 +
               n.cksum * sizeof(CkSum) + n.gcol * 4;
    }
    // Operation buffer of a read (run-length ops of all its chains).  It starts at (n/2 + 4C + 64) per chain for up to 8
    // chains and grows x4 per retry of its chunk (`grow`), up to a bound no chain can exceed: M/X/D records consume a column
    // each (<= n), an x-jump follows an M/X move or sits at column n (<= n + C + 1), x-clips need a jump between them
    // (<= jumps + 2), y-clips <= 2, and I runs alternate with the rest (<= the rest + 1): 6n + 4C + 13 per chain.
    static uint64_t chain_ops_bound(uint32_t n, uint32_t C) { return 6ull * n + 4ull * C + 16; }
    uint64_t ops_max_of(const host::Job &j) const {
        const uint32_t C = (uint32_t)al.layouts.layouts[j.layout].ent.size();
        return std::min<uint64_t>(chain_ops_bound(j.n, C) * (j.walk == host::WALK_ALL ? C : 1), 0xffffffffull);
    }
    uint64_t ops_cap_of(const host::Job &j, uint32_t grow) const {
        const uint32_t C = (uint32_t)al.layouts.layouts[j.layout].ent.size();
        const uint64_t per_chain = j.n / 2 + 4ull * C + 64;
        return std::min<uint64_t>((per_chain * (j.walk == host::WALK_ALL ? std::min<uint32_t>(C, 8) : 1)) << (2 * grow), ops_max_of(j));
    }
    uint64_t out_bytes(const host::Job &j) const {
        const uint64_t C = al.layouts.layouts[j.layout].ent.size();
        return ops_cap_of(j, 0) * sizeof(OutOp) + (j.walk == host::WALK_ALL ? C : 1) * sizeof(ChainHdr) + 4096;
    }

    void run(const std::vector<host::Job> &jobs, std::vector<host::JobResult> &out) override {
        CUDA_CHECK(cudaSetDevice(device));
        out.assign(jobs.size(), host::JobResult());
        if (jobs.empty()) return;
        for (const auto &j : jobs) if (j.n == 0) throw Error(STITCH_ERR_INVALID, "empty read");
        upload_layouts();
        size_t free_b = 0, total_b = 0;
        CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
        // memory our arenas may take: what is free now plus what they already hold
        const uint64_t held = d_ck.cap * sizeof(CellState) + d_colrec.cap * sizeof(ColRec) + d_last.cap * sizeof(LastCell) +
                              d_sn.cap * sizeof(SnRec) + d_ops.cap * sizeof(OutOp) + d_pck.cap * 4;
        mem_budget = (uint64_t)((double)((uint64_t)free_b + held) * 0.85);
        // equal-sized chunks (so that no chunk is a sliver) of per-read records + outputs
        std::vector<uint64_t> bytes(jobs.size());
        uint64_t total = 0;
        const uint64_t cap = mem_budget;
        auto size_up = [&]() {
            total = 0;
            for (size_t k = 0; k < jobs.size(); ++k) {
                bytes[k] = out_bytes(jobs[k]) + need_bytes(need_of(jobs[k], plan_LB(jobs[k]) != 0));
                total += bytes[k];
            }
        };
        // Checkpoint spacing: the smallest spacing that still keeps the whole batch in ONE launch.  The tail and the unit
        // re-fills of the walk shrink with K (a cone unit costs ~K^2), checkpoints grow with 1/K.  Measured on config 2: 450 vs
        // 431 GCUPS at 592 reads with K_base / 2, but 390 vs 430 when the doubled checkpoints split 1000 reads into two
        // launches; on config 4 (100 kb reads x 2 M rows, 16 MB per checkpoint) the spacing has to grow instead.  Candidates:
        // K_base / 2 .. K_base in eighths (only without an explicit STITCH_CK_EVERY), then multiples of K_base up to K_MAX.
        {
            std::vector<uint32_t> cand;
            if (ck_auto && K_base >= 64) for (uint32_t k = K_base / 2; k < K_base; k += K_base / 8) cand.push_back(k);
            for (uint32_t q : {2u, 3u, 4u, 6u, 8u, 12u, 16u, 24u, 32u, 48u, 64u}) { const uint64_t k = (uint64_t)K_base * q / 2; if (k <= K_MAX || cand.empty()) cand.push_back((uint32_t)k); }
            bool found = false;
            for (uint32_t k : cand) { K = k; size_up(); if (total <= cap) { found = true; break; } }
            if (!found) {
                // several launches: K_base, widened so that no read holds more than ~512 MB of checkpoints
                K = K_base;
                for (const auto &j : jobs) {
                    const uint64_t per_ck = (uint64_t)al.layouts.layouts[j.layout].PM() * 8;
                    const uint64_t max_cks = std::max<uint64_t>(1, (512ull << 20) / std::max<uint64_t>(per_ck, 1));
                    const uint64_t need_K = ((uint64_t)j.n + max_cks) / (max_cks + 1);
                    if (need_K > K) K = (uint32_t)((need_K + K_base - 1) / K_base * K_base);
                }
                if (K > K_MAX && K_base <= K_MAX) K = K_MAX / K_base * K_base;
            }
        }
        size_up();
        ops_grow.assign(jobs.size(), 0);
        for (size_t k = 0; k < jobs.size(); ++k)
            if (bytes[k] > mem_budget) throw Error(STITCH_ERR_NOMEM, "one read's checkpoints do not fit in device memory");
        const uint64_t n_chunks = (total + cap - 1) / cap;
        const uint64_t target = total / n_chunks + 1;
        size_t begin = 0;
        while (begin < jobs.size()) {
            size_t end = begin; uint64_t used = 0;
            while (end < jobs.size()) {
                if (end > begin && (used + bytes[end] > cap || used >= target || (max_inflight && end - begin >= max_inflight))) break;
                used += bytes[end]; ++end;
            }
            run_chunk(jobs, begin, end, out);
            begin = end;
        }
    }
    uint64_t mem_budget = 0;

    template <typename KernelT>
    void set_smem(KernelT kernel, size_t smem) {
        if (smem > SMEM_LIMIT + 2048) throw Error(STITCH_ERR_LIMIT, "shared memory of a kernel exceeds 227 KB (contig table or checkpoint spacing too large)");
        if (smem > 48 * 1024) CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }

    void run_chunk(const std::vector<host::Job> &jobs, size_t begin, size_t end, std::vector<host::JobResult> &out) {
        const uint32_t nj = (uint32_t)(end - begin);
        const auto &Ls = al.layouts.layouts;
        h_jobs.reserve(nj); h_order.reserve(4 * (size_t)nj + 16);
        const bool tracked = al.opts.sc.ys != MIN_SCORE;
        uint64_t reads_b = 0, ops_n = 0, chains_n = 0, pm_max = 0, unit_max = 0, cells = 0, handsum_n = 0, ppm_max = 0;
        Need tot{0, 0, 0, 0, 0, 0};
        uint32_t n_packed = 0, ntmax = 1, max_ctiles = 1, cmax = 1;
        // the kernels of a chunk carve their shared-memory tables for the chunk's largest contig count and tile count: packed jobs
        // whose combination does not fit (many contigs in one job, many tiles in another) go to the wide path, largest first
        std::vector<uint32_t> LBs(nj);
        for (uint32_t k = 0; k < nj; ++k) { LBs[k] = plan_LB(jobs[begin + k]); cmax = std::max<uint32_t>(cmax, (uint32_t)Ls[jobs[begin + k].layout].ent.size()); }
        for (;;) {
            uint32_t nt = 1, big = nj;
            for (uint32_t k = 0; k < nj; ++k)
                if (LBs[k] && Ls[jobs[begin + k].layout].n_tiles >= nt) { nt = Ls[jobs[begin + k].layout].n_tiles; big = k; }
            if (big == nj || PackSmem::bytes(cmax, nt, PACK_WARPS, PackSmem::default_stage(PACK_WARPS)) <= SMEM_LIMIT) break;
            LBs[big] = 0;
        }
        // one key layout per launch: every packed job takes the largest LB any of them needs (more length bits are always valid:
        // pk_plan's score-range test depends on the scoring alone and has passed for that LB), so that the kernels read the PK
        // constants from the constant bank (Params::pk) instead of rebuilding them from a per-job LB
        uint32_t LBu = 0;
        for (uint32_t k = 0; k < nj; ++k) LBu = std::max(LBu, LBs[k]);
        for (uint32_t k = 0; k < nj; ++k) if (LBs[k]) LBs[k] = LBu;
        for (uint32_t k = 0; k < nj; ++k) {
            const host::Job &j = jobs[begin + k];
            const host::Layout &L = Ls[j.layout];
            const uint32_t C = (uint32_t)L.ent.size();
            JobDesc d{};
            d.read_off = device_reads ? (uint64_t)(uintptr_t)j.read : reads_b;
            d.colrec_off = tot.colrec; d.cell_off = tot.cell; d.cksum_off = tot.cksum; d.gcol_off = tot.gcol; d.ops_off = ops_n;
            d.n = j.n; d.layout = j.layout; d.walk = j.walk; d.from_contig = j.from_contig;
            d.max_chains = j.walk == host::WALK_ALL ? C : 1;
            d.ops_cap = (uint32_t)ops_cap_of(j, ops_grow[begin + k]);
            d.chain_first = (uint32_t)chains_n;
            d.track_from = tracked ? (j.n > WINDOW ? j.n - WINDOW + 1 : 1) : j.n + 1;
            d.hand_off = tot.cell; d.handsum_off = handsum_n;
            d.LB = LBs[k]; d.j0 = 0;
            d.ck_off = d.LB ? tot.pck : tot.ck;
            const Need nd = need_of(j, d.LB != 0);
            uint32_t mct = 0;
            for (const auto &e : L.ent) mct = std::max(mct, e.ntiles);
            max_ctiles = std::max(max_ctiles, mct);
            if (d.LB) {
                stats.packed_cells += L.cells_per_col * j.n; ++n_packed;
                ntmax = std::max(ntmax, L.n_tiles); ppm_max = std::max<uint64_t>(ppm_max, L.PM());
            }
            tot.colrec += nd.colrec; tot.cell += nd.cell; tot.ck += nd.ck; tot.pck += nd.pck; tot.cksum += nd.cksum; tot.gcol += nd.gcol;
            handsum_n += C;
            pm_max = std::max<uint64_t>(pm_max, L.PM());
            h_jobs.p[k] = d;
            reads_b += round_up(j.n, 16);
            ops_n += d.ops_cap; chains_n += d.max_chains;
            unit_max = std::max<uint64_t>(unit_max, (uint64_t)mct * TILE * std::min<uint32_t>(K, j.n));
            cells += L.cells_per_col * j.n;
        }
        const uint32_t n_wide = nj - n_packed;
        std::iota(h_order.p, h_order.p + nj, 0u);
        std::stable_sort(h_order.p, h_order.p + nj, [&](uint32_t x, uint32_t y) {
            const host::Job &a = jobs[begin + x], &b = jobs[begin + y];
            return Ls[a.layout].cells_per_col * a.n > Ls[b.layout].cells_per_col * b.n;
        });
        // order lists: [0, nj) all jobs; then the packed jobs; then the wide jobs; then re-runs
        uint32_t *po = h_order.p + nj, *wo = po + n_packed, *ro = wo + n_wide;
        { uint32_t a = 0, b = 0; for (uint32_t k = 0; k < nj; ++k) { if (h_jobs.p[h_order.p[k]].LB) po[a++] = h_order.p[k]; else wo[b++] = h_order.p[k]; } }

        // grids: one CTA (or one thread-block cluster) per packed read; two 8-warp CTAs per SM for the wide fill
        const uint32_t wgrid = std::min<uint32_t>(nj, (uint32_t)num_sms);                     // walk kernel
        const uint32_t wide_grid = std::min<uint32_t>(n_wide, 2 * (uint32_t)num_sms);         // wide fill (and its re-runs: n_redo <= n_wide)
        uint32_t cluster = cluster_pref;
        if (cluster == 0) {   // automatic: the largest cluster that still gives every read its own team in one wave
            cluster = 1;
            while (cluster < 16 && (uint64_t)n_packed * cluster * 2 <= (uint64_t)num_sms * 3 / 4) cluster *= 2;
        }
        if (ntmax < cluster_min_tiles) cluster = 1;
        uint32_t pteams = 0;
        size_t cstate_bytes = 0, pstage = PackSmem::default_stage(PACK_WARPS);
        if (n_packed) {
            pteams = std::min<uint32_t>(n_packed, (uint32_t)num_sms / cluster);
            if (cluster > 1) {
                cudaLaunchConfig_t cfg = {};
                cfg.gridDim = dim3((unsigned)num_sms / cluster * cluster); cfg.blockDim = dim3(PACK_WARPS * 32);
                // rolling state in the cluster's shared memory when every CTA's slice of the largest read fits
                // (a CTA owns the chunks of its 16 warps: up to 16 tiles even when the read has fewer than 16 x cluster tiles)
                const size_t slice = std::max<size_t>(std::min<size_t>(ntmax, PACK_WARPS), (size_t)ntmax / cluster + 2) * ST * sizeof(int32_t);
                if (cluster_smem && PackSmem::bytes(cmax, ntmax, PACK_WARPS, slice) <= 220 * 1024) cstate_bytes = slice;
                pstage = cstate_bytes ? cstate_bytes : PackSmem::default_stage(PACK_WARPS);
                cfg.dynamicSmemBytes = PackSmem::bytes(cmax, ntmax, PACK_WARPS, pstage);
                set_smem(fill_packed_kernel<PACK_WARPS>, cfg.dynamicSmemBytes);
                if (cluster > 8) CUDA_CHECK(cudaFuncSetAttribute(fill_packed_kernel<PACK_WARPS>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
                cudaLaunchAttribute at[1];
                at[0].id = cudaLaunchAttributeClusterDimension;
                at[0].val.clusterDim.x = cluster; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
                cfg.attrs = at; cfg.numAttrs = 1;
                int max_clusters = 0;
                if (cudaOccupancyMaxActiveClusters(&max_clusters, fill_packed_kernel<PACK_WARPS>, &cfg) == cudaSuccess && max_clusters > 0)
                    pteams = std::min<uint32_t>(pteams, (uint32_t)max_clusters);
                else { cudaGetLastError(); cluster = 1; cstate_bytes = 0; pstage = PackSmem::default_stage(PACK_WARPS); pteams = std::min<uint32_t>(n_packed, (uint32_t)num_sms); }
                if (debug_stats) std::fprintf(stderr, "[stitch dbg] cluster %u: max active clusters %d, state in smem %zu B/CTA\n", cluster, max_clusters, cstate_bytes);
            }
        }
        // shared memory of the packed fill, and of its walk phase (per-unit staging of K columns + the unit's contig bases) when
        // that fits beside it with the real K and the longest contig of this chunk; otherwise the separate walk kernel runs
        // staging ring of the fill: as deep as shared memory allows (the walk phase's staging included when it would otherwise fit)
        uint32_t depth = 2;
        if (cluster == 1) {
            const size_t walk_extra = (walk_in_kernel && cluster == 1 && n_packed > 0) ? UnitStage::bytes(K, max_ctiles, false) : 0;
            for (depth = stage_depth_pref; depth > 2; depth /= 2)
                if ((PackSmem::bytes(cmax, ntmax, PACK_WARPS, PackSmem::default_stage(PACK_WARPS, depth)) + 15) / 16 * 16 + walk_extra <= SMEM_LIMIT) break;
            pstage = PackSmem::default_stage(PACK_WARPS, depth);
        }
        size_t psmem = (PackSmem::bytes(cmax, ntmax, PACK_WARPS, pstage) + 15) / 16 * 16;
        bool packed_walks_in_kernel = walk_in_kernel && cluster == 1 && n_packed > 0;
        bool pstage_bases = true;
        if (packed_walks_in_kernel) {
            if (psmem + UnitStage::bytes(K, max_ctiles, true) > SMEM_LIMIT) pstage_bases = false;
            if (psmem + UnitStage::bytes(K, max_ctiles, pstage_bases) > SMEM_LIMIT) packed_walks_in_kernel = false;
        }
        const uint32_t n_post = packed_walks_in_kernel ? n_wide : nj;   // reads walked by the separate fix-up / walk kernels
        const uint32_t bufgrid = std::max(n_post ? wgrid : 0u, packed_walks_in_kernel ? pteams : 0u);   // CTAs that own walk buffers
        d_jobs.reserve(nj); d_order.reserve(4 * (size_t)nj + 16);
        d_colrec.reserve(tot.colrec); d_last.reserve(tot.cell);
        d_sn.reserve(tot.cell); d_ck.reserve(tot.ck + 64); d_pck.reserve(tot.pck + 64);
        d_cksum.reserve(tot.cksum); d_gcol.reserve(tot.gcol);
        d_ops.reserve(ops_n); d_chains.reserve(chains_n); d_jobout.reserve(nj);
        // wide rolling state: one pair of column buffers per CTA of the LARGEST grid that indexes it (wide fill / re-runs by
        // blockIdx, wide unit re-fills of the walk kernel)
        d_state.reserve((uint64_t)std::max(wide_grid, n_wide ? wgrid : 0u) * 2 * pm_max + 64);
        d_hand.reserve(64); d_handsum.reserve(handsum_n + 64);   // (hand-over buffers of the retired packed -> wide tail)
        d_pstate.reserve((uint64_t)pteams * 2 * ppm_max + 64);
        const uint64_t tb_stride = round_up(ppm_max + 2 * PackSmem::STAGE_PRE, 256);   // tile-ordered bases per team (+ the 16 bytes before tile 0)
        d_ptbases.reserve((uint64_t)pteams * tb_stride + 256);
        d_tailj0.reserve(nj);
        const uint64_t wps_half = (uint64_t)max_ctiles * TILE;
        d_wpstate.reserve((uint64_t)bufgrid * 2 * wps_half + 64);
        d_ucr.reserve((uint64_t)bufgrid * K + 64);
        d_unit.reserve((uint64_t)bufgrid * round_up(unit_max, 256) + 64);
        if (!device_reads) { d_reads.reserve(reads_b); h_reads.reserve(reads_b); }
        h_ops.reserve(ops_n); h_chains.reserve(chains_n); h_jobout.reserve(nj);

        n_marks = 0;
        mark(T_H2D);
        if (!device_reads) {
            for (uint32_t k = 0; k < nj; ++k)
                std::memcpy(h_reads.p + h_jobs.p[k].read_off, jobs[begin + k].read, jobs[begin + k].n);
            CUDA_CHECK(cudaMemcpyAsync(d_reads.p, h_reads.p, reads_b, cudaMemcpyHostToDevice, stream));
            stats.h2d += reads_b;
        }
        CUDA_CHECK(cudaMemcpyAsync(d_jobs.p, h_jobs.p, nj * sizeof(JobDesc), cudaMemcpyHostToDevice, stream));
        CUDA_CHECK(cudaMemcpyAsync(d_order.p, h_order.p, 2 * (size_t)nj * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
        stats.h2d += nj * (sizeof(JobDesc) + 2 * sizeof(uint32_t));
        CUDA_CHECK(cudaMemsetAsync(d_counter.p, 0, 8 * sizeof(uint32_t), stream));

        Params P{};
        if (LBu) P.pk = pk_make(al.opts.sc, LBu);
        P.sc = al.opts.sc; P.jobs = d_jobs.p; P.order = d_order.p; P.n_jobs = nj; P.cmax = cmax;
        P.layouts = d_layouts.p; P.ents = d_ents.p; P.owners = d_owners.p;
        P.contig_bases = d_contigs.p; P.reads = device_reads ? device_reads : d_reads.p;
        P.state = d_state.p; P.state_stride = 2 * pm_max; P.state_half = pm_max;
        P.unit_bytes = d_unit.p; P.unit_stride = round_up(unit_max, 256);
        P.colrec = d_colrec.p; P.last = d_last.p; P.sn = d_sn.p; P.ck_state = d_ck.p; P.pck = d_pck.p; P.ck_sum = d_cksum.p; P.gcol = d_gcol.p;
        P.ops = d_ops.p; P.chains = d_chains.p; P.job_out = d_jobout.p; P.counter = d_counter.p;
        d_qstats.reserve(2); CUDA_CHECK(cudaMemsetAsync(d_qstats.p, 0, 2 * sizeof(unsigned long long), stream)); P.qstats = d_qstats.p;
        P.K = K; P.tracked_mode = tracked ? 1 : 0; P.force_full = 0;
        P.hand_state = d_hand.p; P.hand_sum = d_handsum.p; P.pstate = d_pstate.p; P.pstate_stride = 2 * ppm_max; P.pstate_half = ppm_max;
        P.ptbases = d_ptbases.p; P.ptbases_stride = tb_stride;
        P.ntmax = ntmax; P.tail_j0 = d_tailj0.p; P.wpstate = d_wpstate.p; P.wpstate_stride = 2 * wps_half; P.wpstate_half = wps_half;
        P.unit_cr = d_ucr.p; P.max_ctiles = max_ctiles; P.cluster_size = 1; P.cone = cone_refill;
        if (debug_stats) { d_dbg.reserve(80); CUDA_CHECK(cudaMemsetAsync(d_dbg.p, 0, 80 * sizeof(unsigned long long), stream)); P.dbg = d_dbg.p; }

        const size_t smem = WideSmem<FILL_WARPS>::bytes(cmax);
        set_smem(fill_wide_kernel<FILL_WARPS>, smem);
        mark(T_PACKED);
        if (n_packed) {
            Params Q = P; Q.order = d_order.p + nj; Q.n_jobs = n_packed; Q.counter = d_counter.p + 3;
            Q.cluster_size = cluster; Q.stage_bytes = (uint32_t)pstage; Q.cluster_state_smem = (uint32_t)cstate_bytes; Q.stage_depth = depth;
            Q.quiet = quiet_tiles; Q.quiet_first = quiet_first; Q.quiet_edge = quiet_edge; Q.quiet_last = quiet_last; Q.quiet_tail = quiet_tail;
            if (packed_walks_in_kernel) {   // second phase of the same kernel: fix-up + walk of the packed reads
                d_done.reserve(nj);
                CUDA_CHECK(cudaMemsetAsync(d_done.p, 0, nj * sizeof(uint32_t), stream));
                Q.done = d_done.p;
                Q.walk_stage_smem_off = (uint32_t)psmem; Q.unit_stage_bases = pstage_bases ? 1u : 0u;
                psmem += UnitStage::bytes(K, max_ctiles, pstage_bases);
            }
            Q.pso = PackSmem::layout(cmax, ntmax, PACK_WARPS, pstage);
            set_smem(fill_packed_kernel<PACK_WARPS>, psmem);
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(pteams * cluster); cfg.blockDim = dim3(PACK_WARPS * 32); cfg.dynamicSmemBytes = psmem; cfg.stream = stream;
            cudaLaunchAttribute at[1];
            unsigned na = 0;
            if (cluster > 1) {
                at[na].id = cudaLaunchAttributeClusterDimension;
                at[na].val.clusterDim.x = cluster; at[na].val.clusterDim.y = 1; at[na].val.clusterDim.z = 1;
                ++na;
            }
            cfg.attrs = at; cfg.numAttrs = na;
            CUDA_CHECK(cudaLaunchKernelEx(&cfg, fill_packed_kernel<PACK_WARPS>, Q));
            stats.launches += 1; stats.packed_launches += 1;
        }
        mark(T_WIDE);
        if (n_wide) {
            // jobs outside the packed regime run on the wide kernel
            Params Q = P; Q.order = d_order.p + nj + n_packed; Q.n_jobs = n_wide;
            fill_wide_kernel<FILL_WARPS><<<wide_grid, FILL_WARPS * 32, smem, stream>>>(Q);
            CUDA_CHECK(cudaGetLastError());
            stats.launches += 1;
        }
        // fix-up and walk kernels: the wide reads, plus the packed ones when their kernel did not do it itself
        const uint32_t *post_order = packed_walks_in_kernel ? d_order.p + nj + n_packed : d_order.p;
        mark(T_FIXUP);
        if (n_post) {
            Params Q = P; Q.order = post_order; Q.n_jobs = n_post;
            fixup_kernel<<<n_post, 64, 0, stream>>>(Q);
            CUDA_CHECK(cudaGetLastError());
            stats.launches += 1;
        }
        stats.fills += nj; stats.cells += cells;
        if (tracked && n_wide) {
            // wide-path reads whose tracking window was too narrow are filled again from an earlier checkpoint
            CUDA_CHECK(cudaMemcpyAsync(h_jobout.p, d_jobout.p, nj * sizeof(JobOut), cudaMemcpyDeviceToHost, stream));
            mark(T_END);
            sync("fill");
            collect_marks();
            uint32_t n_redo = 0;
            h_redo.reserve(nj); d_redo.reserve(nj);
            for (uint32_t t = 0; t < n_wide; ++t) {
                const uint32_t k = wo[t];
                if (h_jobout.p[k].status != JOB_NEED_FULL_TRACK) continue;
                ro[n_redo++] = k;
                const uint32_t first = h_jobout.p[k].n_chains;   // first column that may hold a final y-suffix tracker
                h_redo.p[k] = first > 0 ? ((first - 1) / K) * K : 0;
                stats.cells += Ls[jobs[begin + k].layout].cells_per_col * (jobs[begin + k].n - h_redo.p[k]);
            }
            mark(T_REDO);
            if (n_redo) {
                CUDA_CHECK(cudaMemcpyAsync(d_order.p + 2 * (size_t)nj, ro, n_redo * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
                CUDA_CHECK(cudaMemcpyAsync(d_redo.p, h_redo.p, nj * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
                Params Q = P; Q.order = d_order.p + 2 * (size_t)nj; Q.n_jobs = n_redo; Q.force_full = 1; Q.counter = d_counter.p + 1;
                Q.redo_j0 = d_redo.p;
                fill_wide_kernel<FILL_WARPS><<<std::min<uint32_t>(n_redo, wide_grid), FILL_WARPS * 32, smem, stream>>>(Q);
                CUDA_CHECK(cudaGetLastError());
                fixup_kernel<<<n_redo, 64, 0, stream>>>(Q);
                CUDA_CHECK(cudaGetLastError());
                stats.launches += 2; stats.fills += n_redo; stats.refills += n_redo;
            }
        }
        mark(T_WALK);
        if (n_post) {
            Params Wp = P; Wp.order = post_order; Wp.n_jobs = n_post; Wp.counter = d_counter.p + 2;
            size_t wsmem = std::max(WideSmem<WALK_WARPS>::bytes(1), PackSmem::bytes(1, max_ctiles, WALK_WARPS, 0));
            wsmem = (wsmem + 15) / 16 * 16;
            Wp.walk_stage_smem_off = (uint32_t)wsmem;
            // the per-unit staging: K columns of records always (K <= K_MAX), the contig's bases only when they fit (only packed
            // re-fills read them; a contig beyond ~190 kb is read from global memory instead)
            const bool wstage_bases = n_post > n_wide && wsmem + UnitStage::bytes(K, max_ctiles, true) <= SMEM_LIMIT;
            Wp.unit_stage_bases = wstage_bases ? 1u : 0u;
            wsmem += (UnitStage::bytes(K, max_ctiles, wstage_bases) + 15) / 16 * 16;
            const size_t state_b = 2 * wps_half * sizeof(int32_t);
            if (wsmem + state_b <= 160 * 1024) { Wp.walk_state_smem_off = (uint32_t)wsmem; wsmem += state_b; }
            set_smem(walk_kernel<WALK_WARPS>, wsmem);
            walk_kernel<WALK_WARPS><<<wgrid, WALK_WARPS * 32, wsmem, stream>>>(Wp);
            CUDA_CHECK(cudaGetLastError());
            stats.launches += 1;
        }
        mark(T_D2H);
        CUDA_CHECK(cudaMemcpyAsync(h_jobout.p, d_jobout.p, nj * sizeof(JobOut), cudaMemcpyDeviceToHost, stream));
        CUDA_CHECK(cudaMemcpyAsync(h_chains.p, d_chains.p, chains_n * sizeof(ChainHdr), cudaMemcpyDeviceToHost, stream));
        CUDA_CHECK(cudaMemcpyAsync(h_ops.p, d_ops.p, ops_n * sizeof(OutOp), cudaMemcpyDeviceToHost, stream));
        mark(T_END);
        sync("walk");
        collect_marks();
        {
            unsigned long long hq[2];
            CUDA_CHECK(cudaMemcpy(hq, d_qstats.p, sizeof(hq), cudaMemcpyDeviceToHost));
            stats.tile_columns += hq[0]; stats.quiet_tile_columns += hq[1];
        }
        if (debug_stats) {
            unsigned long long h[80];
            cudaMemcpy(h, d_dbg.p, sizeof(h), cudaMemcpyDeviceToHost);
            std::fprintf(stderr, "[stitch dbg] jobs %u (K %u): tail columns %llu, tail Mcycles %.1f, bulk Mcycles %.1f | walk units %llu, "
                         "refill columns %llu, refill Mcycles %.1f, walk-job Mcycles %.1f\n", nj, K, h[0], h[1] * 1e-6, h[2] * 1e-6, h[3], h[6],
                         h[4] * 1e-6, h[5] * 1e-6);
            std::fprintf(stderr, "[stitch dbg] bulk columns, Mcycles summed over reads: select %.1f, tile phase %.1f (mean warp busy %.1f), per-contig finish %.1f (warp 0: tile maxima reduced at %.1f, look-ups done at %.1f, row m done at %.1f)\n",
                         h[7] * 1e-6, h[8] * 1e-6, h[10] * 1e-6, h[9] * 1e-6, h[13] * 1e-6, h[11] * 1e-6, h[12] * 1e-6);
            std::fprintf(stderr, "[stitch dbg] tile phase per warp, Gcycles busy / M tiles computed:");
            for (int w = 0; w < PACK_WARPS; ++w) std::fprintf(stderr, " %.1f/%.1f", h[16 + w] * 1e-9, h[48 + w] * 1e-6);
            std::fprintf(stderr, "\n");
        }
        stats.tb_bytes += tot.ck * sizeof(CellState) + tot.pck * 4 + tot.colrec * sizeof(ColRec);
        stats.d2h += nj * sizeof(JobOut) + chains_n * sizeof(ChainHdr) + ops_n * sizeof(OutOp);

        bool overflow = false;
        for (uint32_t k = 0; k < nj; ++k) {
            if (h_jobout.p[k].status == WALK_OVERFLOW) {
                // rare: rerun the chunk with x4 the operation buffer of every read that overflowed; a buffer that already
                // holds chain_ops_bound per chain cannot have overflowed
                if (h_jobs.p[k].ops_cap >= ops_max_of(jobs[begin + k])) throw Error(STITCH_ERR_INTERNAL, "operation buffer overflow");
                ++ops_grow[begin + k];
                overflow = true;
            } else if (h_jobout.p[k].status != WALK_OK)
                throw Error(STITCH_ERR_INTERNAL, "traceback reached a state the reference panics on");
        }
        if (overflow) {
            for (size_t k = begin; k < end; ++k) out[k] = host::JobResult();
            run_chunk(jobs, begin, end, out);
            return;
        }
        for (uint32_t k = 0; k < nj; ++k) {
            const JobDesc &d = h_jobs.p[k];
            uint64_t off = d.ops_off;
            for (uint32_t c = 0; c < h_jobout.p[k].n_chains; ++c) {
                host::RawChain rc;
                rc.h = h_chains.p[d.chain_first + c];
                rc.ops.assign(h_ops.p + off, h_ops.p + off + rc.h.n_ops);
                off += rc.h.n_ops;
                out[begin + k].chains.push_back(std::move(rc));
            }
        }
    }
    // ---- pre-alignment contig selection (prealign_core.h, kernels_prealign.cuh) ----
    host::KmerIndex kindex;
    DevBuf<uint32_t> d_koff, d_kpos, d_seqoff, d_slen, d_pcnt, d_pbins, d_poutn, d_prlen;
    DevBuf<uint64_t> d_proff;
    DevBuf<PreHit> d_pout;
    void prealign(const std::vector<host::Job> &reads, std::vector<std::vector<PreHit>> &out) override {
        CUDA_CHECK(cudaSetDevice(device));
        out.assign(reads.size(), std::vector<PreHit>());
        if (reads.empty()) return;
        const host::Opts &o = al.opts;
        const host::Contigs &c = al.contigs;
        if (kindex.K != o.kmer) {   // built once per context (the reference hashes every target at start-up, align.rs:333-336)
            kindex.build(c, o.kmer);
            d_koff.reserve(kindex.off.size()); d_kpos.reserve(kindex.pos.size() + 1); d_seqoff.reserve(c.n_strands); d_slen.reserve(c.n_strands);
            CUDA_CHECK(cudaMemcpy(d_koff.p, kindex.off.data(), kindex.off.size() * 4, cudaMemcpyHostToDevice));
            CUDA_CHECK(cudaMemcpy(d_kpos.p, kindex.pos.data(), kindex.pos.size() * 4, cudaMemcpyHostToDevice));
            CUDA_CHECK(cudaMemcpy(d_seqoff.p, c.seq_off.data(), c.n_strands * 4, cudaMemcpyHostToDevice));
            CUDA_CHECK(cudaMemcpy(d_slen.p, c.len.data(), c.n_strands * 4, cudaMemcpyHostToDevice));
        }
        cudaEvent_t e0 = ev[14], e1 = ev[15];
        const size_t CH = 16384;   // reads per launch (2 KB of output each)
        std::vector<uint64_t> offs; std::vector<uint32_t> lens; std::vector<PreHit> hout; std::vector<uint32_t> hn;
        for (size_t begin = 0; begin < reads.size(); begin += CH) {
            const size_t end = std::min(reads.size(), begin + CH), nr = end - begin;
            uint64_t bytes = 0; uint32_t max_n = 1;
            offs.assign(nr, 0); lens.assign(nr, 0);
            for (size_t k = 0; k < nr; ++k) { offs[k] = bytes; lens[k] = reads[begin + k].n; bytes += round_up(reads[begin + k].n, 16); max_n = std::max(max_n, reads[begin + k].n); }
            h_reads.reserve(bytes); d_reads.reserve(bytes);
            for (size_t k = 0; k < nr; ++k) std::memcpy(h_reads.p + offs[k], reads[begin + k].read, reads[begin + k].n);
            const uint32_t grid = (uint32_t)std::min<size_t>(nr, 2 * (size_t)num_sms);
            const uint32_t n_bins = (max_n + c.max_len) / o.band + 2;
            d_proff.reserve(nr); d_prlen.reserve(nr); d_pout.reserve(nr * MAX_STRANDS); d_poutn.reserve(nr);
            d_pcnt.reserve((size_t)grid * c.n_strands); d_pbins.reserve((size_t)grid * PRE_MAX_CAND * n_bins);
            CUDA_CHECK(cudaEventRecord(e0, stream));
            CUDA_CHECK(cudaMemcpyAsync(d_reads.p, h_reads.p, bytes, cudaMemcpyHostToDevice, stream));
            CUDA_CHECK(cudaMemcpyAsync(d_proff.p, offs.data(), nr * 8, cudaMemcpyHostToDevice, stream));
            CUDA_CHECK(cudaMemcpyAsync(d_prlen.p, lens.data(), nr * 4, cudaMemcpyHostToDevice, stream));
            CUDA_CHECK(cudaMemsetAsync(d_counter.p, 0, 8 * sizeof(uint32_t), stream));
            PreKParams P{};
            P.off = d_koff.p; P.pos = d_kpos.p; P.blob = d_contigs.p; P.seq_off = d_seqoff.p; P.strand_len = d_slen.p;
            P.n_strands = c.n_strands; P.K = o.kmer; P.W = o.band; P.n_bins = n_bins; P.match = o.sc.match; P.min_score = o.pre_min_score;
            P.reads = d_reads.p; P.read_off = d_proff.p; P.read_len = d_prlen.p; P.n_reads = (uint32_t)nr;
            P.counter = d_counter.p; P.cnt = d_pcnt.p; P.bins = d_pbins.p; P.out = d_pout.p; P.out_n = d_poutn.p;
            prealign_kernel<<<grid, PRE_THREADS, 0, stream>>>(P);
            CUDA_CHECK(cudaGetLastError());
            hout.resize(nr * MAX_STRANDS); hn.resize(nr);
            CUDA_CHECK(cudaMemcpyAsync(hn.data(), d_poutn.p, nr * 4, cudaMemcpyDeviceToHost, stream));
            CUDA_CHECK(cudaMemcpyAsync(hout.data(), d_pout.p, nr * MAX_STRANDS * sizeof(PreHit), cudaMemcpyDeviceToHost, stream));
            CUDA_CHECK(cudaEventRecord(e1, stream));
            sync("prealign");
            float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
            stats.pre_ms += ms; stats.total_ms += ms; stats.launches += 1; stats.pre_reads += nr;
            stats.h2d += bytes + nr * 12; stats.d2h += nr * (4 + MAX_STRANDS * sizeof(PreHit));
            for (size_t k = 0; k < nr; ++k) out[begin + k].assign(hout.begin() + k * MAX_STRANDS, hout.begin() + k * MAX_STRANDS + hn[k]);
        }
    }

    void mark(int tag) {
        if (n_marks >= 14) return;   // (events 14 and 15 time the pre-alignment)
        CUDA_CHECK(cudaEventRecord(ev[n_marks], stream));
        marks[n_marks++] = tag;
    }
    // durations between consecutive marks, credited to the earlier mark's phase (call after a stream sync)
    void collect_marks() {
        for (int k = 0; k + 1 < n_marks; ++k) {
            float ms = 0;
            cudaEventElapsedTime(&ms, ev[k], ev[k + 1]);
            switch (marks[k]) {
            case T_PACKED: stats.packed_ms += ms; stats.fill_ms += ms; break;
            case T_TAIL: stats.tail_ms += ms; stats.fill_ms += ms; break;
            case T_WIDE: stats.wide_ms += ms; stats.fill_ms += ms; break;
            case T_REDO: stats.redo_ms += ms; stats.fill_ms += ms; break;
            case T_FIXUP: case T_WALK: stats.tb_ms += ms; break;
            default: break;
            }
            stats.total_ms += ms;
        }
        n_marks = 0;
    }
    void sync(const char *what) {
        cudaError_t se = cudaStreamSynchronize(stream);
        if (se != cudaSuccess) throw Error(STITCH_ERR_CUDA, std::string("kernel failed (") + what + "): " + cudaGetErrorString(se));
    }
    std::vector<uint32_t> ops_grow;   // per job of the current run(): x4 growths of its operation buffer (retries)
};

}  // namespace gpu

namespace host {
Backend *stitch_make_backend(Aligner &al, int device) { return new gpu::CudaBackend(al, device); }
}  // namespace host
}  // namespace stitch

// Reads already resident in device memory (upper-cased): times the path without host copies.
extern "C" int stitch_custom_batch_device(stitch_ctx *ctx, const uint8_t *d_bases, const uint64_t *h_offsets,
                                          uint32_t n_reads, stitch_results **out) {
    if (!ctx) return STITCH_ERR_INVALID;
    STITCH_GUARD_BEGIN
    if (!d_bases || !h_offsets || !out) throw stitch::host::Error(STITCH_ERR_INVALID, "null argument");
    auto *be = static_cast<stitch::gpu::CudaBackend *>(ctx->al.backend.get());
    std::vector<stitch::host::Job> jobs(n_reads);
    uint64_t max_n = 0;
    for (uint32_t r = 0; r < n_reads; ++r) {
        jobs[r].read = reinterpret_cast<const uint8_t *>((uintptr_t)h_offsets[r]);
        jobs[r].n = (uint32_t)(h_offsets[r + 1] - h_offsets[r]);
        jobs[r].layout = ctx->al.layouts.all();
        jobs[r].walk = stitch::host::WALK_BEST;
        max_n = std::max<uint64_t>(max_n, jobs[r].n);
    }
    ctx->al.check_ranges(max_n);
    be->stats.reset();
    std::vector<stitch::host::JobResult> res;
    be->device_reads = d_bases;
    try { be->run(jobs, res); } catch (...) { be->device_reads = nullptr; throw; }
    be->device_reads = nullptr;
    std::unique_ptr<stitch_results> r(new stitch_results());
    for (uint32_t k = 0; k < n_reads; ++k) {
        r->res.begin_read();
        if (res[k].chains.size() != 1) throw stitch::host::Error(STITCH_ERR_INTERNAL, "traceback_from returned None");
        r->res.add(stitch::host::from_raw(res[k].chains[0]));
    }
    *out = r.release();
    return STITCH_OK;
    STITCH_GUARD_END(ctx)
}

// ---------------------------------------------------------------------------------------------
// INT32 add+max issue-rate microbenchmark (the roofline denominator of the fill kernel)
// ---------------------------------------------------------------------------------------------
namespace stitch { namespace gpu {
__global__ void __launch_bounds__(256) int32_peak_kernel(int32_t *out, int iters, int32_t c, int32_t w) {
    int32_t v[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) v[k] = (int32_t)(threadIdx.x * 16 + k);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
#pragma unroll
            for (int k = 0; k < 16; ++k) v[k] = max(v[k] + c, w + k);   // one add + one max per element
        }
    }
    int32_t acc = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) acc ^= v[k];
    out[blockIdx.x * blockDim.x + threadIdx.x] = acc;
}
}}  // namespace stitch::gpu

extern "C" int stitch_measure_int32_peak(int device, double *gops) {
    if (!gops) return STITCH_ERR_INVALID;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return STITCH_ERR_CUDA;
    if (cudaSetDevice(device) != cudaSuccess) return STITCH_ERR_CUDA;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return STITCH_ERR_CUDA;
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 2048;
    int32_t *d = nullptr;
    if (cudaMalloc(&d, (size_t)blocks * threads * sizeof(int32_t)) != cudaSuccess) return STITCH_ERR_NOMEM;
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    double best = 0;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(a);
        stitch::gpu::int32_peak_kernel<<<blocks, threads>>>(d, iters, -3, -1000000 + rep);
        cudaEventRecord(b);
        if (cudaEventSynchronize(b) != cudaSuccess) { cudaFree(d); return STITCH_ERR_CUDA; }
        float ms = 0;
        cudaEventElapsedTime(&ms, a, b);
        const double ops = 2.0 * 16 * 4 * (double)iters * blocks * threads;
        if (rep > 0) best = std::max(best, ops / (ms * 1e-3) / 1e9);
    }
    cudaEventDestroy(a); cudaEventDestroy(b); cudaFree(d);
    *gops = best;
    return STITCH_OK;
}
