"""The checkpoint spacing K of the CUDA path and what depends on it (stitch_b200/csrc/cuda_backend.cu, kernels_packed.cuh),
restated for the tests.

`CudaBackend::run` picks K per batch (k_candidates); `run_chunk` sizes the shared memory of the packed fill and of the walk
with it and decides whether the walk runs inside the packed kernel (plan_chunk).  The packed fill stores regular checkpoints
every K columns and up to PK_LATE_CKS late ones at n - 32 k (late_ck, ck_index), and its tail restarts from the last of them
before the first column that can hold a final y-suffix tracker (tail_start).  Walk units longer than PK_CONE_MAX_COLS columns
build their per-column constants per column.  Every read gets an operation buffer that grows x4 per retry of its chunk up to
a bound no chain exceeds (ops_cap).

The tests use the restatement to put inputs on both sides of each branch and to predict the kernel launches of a batch."""

TILE = 256                      # rows per warp tile of the CUDA build (STRIP = 8)
PACK_WARPS = WALK_WARPS = 16
SMEM_LIMIT = 227 * 1024 - 2048
K_MAX = 8192
K_BASE = 256
PK_LATE_CKS, PK_LATE_STEP = 3, 32
PK_CONE_MAX_COLS = 384
WALK_STATE_SMEM_MAX = 160 * 1024   # walk kernel: the re-fill state of one contig in shared memory below this
CLUSTER_MIN_TILES = 4 * PACK_WARPS

# sizeof of the device structs the shared-memory layouts are carved from (test_emul_traceback_spacing checks them against
# the headers)
SIZES = dict(JumpInfo=16, PkRowM=24, PkQuiet=44, ContigEntry=32, PkColConst=56, RowM=68, XsPart=12, CmPart=16, ICarry=12)
STAGE_BYTES = 2 * TILE * 4 + 16 + TILE


def r16(v):
    return (v + 15) // 16 * 16


# ---- checkpoint spacing ---------------------------------------------------------------------------------------------------

def k_candidates(k_base=K_BASE, auto=True):
    """Spacings run() tries in order, the first that keeps the batch in one launch wins: K_base/2 .. K_base in eighths (no
    STITCH_CK_EVERY), then K_base * q / 2 up to K_MAX."""
    cand = []
    if auto and k_base >= 64:
        cand += list(range(k_base // 2, k_base, k_base // 8))
    for q in (2, 3, 4, 6, 8, 12, 16, 24, 32, 48, 64):
        k = k_base * q // 2
        if k <= K_MAX or not cand:
            cand.append(k)
    return cand


def regular_cks(n, K):
    """Regular checkpoint columns K, 2K, ... < n."""
    return (n - 1) // K


def late_ck(j, n, K):
    """k (1 .. PK_LATE_CKS) when column j is a late checkpoint column of a read of n columns, else 0."""
    if j >= n or j % K == 0:
        return 0
    d = n - j
    return d // PK_LATE_STEP if d % PK_LATE_STEP == 0 and d // PK_LATE_STEP <= PK_LATE_CKS else 0


def ck_index(j0, n, K):
    """Index among the read's stored checkpoints of the one at column j0 > 0."""
    return j0 // K - 1 if j0 % K == 0 else regular_cks(n, K) + (n - j0) // PK_LATE_STEP - 1


def ck_columns(n, K):
    """{column: index} of every checkpoint the packed bulk pass stores."""
    return {j: ck_index(j, n, K) for j in range(1, n) if (j % K == 0) or late_ck(j, n, K)}


def tail_start(first, n, K):
    """Column the packed tail restarts from: the last checkpoint (regular or late) before `first`, the first column that
    can hold a final y-suffix tracker (n when nothing is tracked)."""
    j0 = (first - 1) // K * K
    for k in range(1, PK_LATE_CKS + 1):
        if n <= PK_LATE_STEP * k:
            break
        jl = n - PK_LATE_STEP * k
        if jl % K == 0:
            continue
        if jl < first:
            j0 = max(j0, jl)
            break
    return j0


def redo_start(first, K):
    """Column a wide-path re-run (tracking window too narrow) restarts from."""
    return (first - 1) // K * K if first > 0 else 0


def cone_unit_cols(j, K):
    """Columns of the walk unit entered at column j: (jb, j], jb = the checkpoint column before j."""
    return j - (j - 1) // K * K


# ---- shared memory ---------------------------------------------------------------------------------------------------------

def default_stage(W=PACK_WARPS, depth=2):
    return W * depth * STAGE_BYTES


def pack_smem_bytes(cmax, ntmax, W=PACK_WARPS, stage=None):
    s = SIZES
    stage = default_stage(W) if stage is None else stage
    return (stage + 4 * (cmax * 9 + ntmax + 2 * W * 18) +
            (s["PkRowM"] + s["JumpInfo"] + 2 * s["PkQuiet"] + s["ContigEntry"]) * cmax + 5 * ntmax + 4 * 8 + 64 + 36 * W + 8)


def unit_stage_bytes(K, max_ctiles, stage_bases):
    s = SIZES
    cone = r16(s["PkColConst"] * K) + r16(4 * K) if K <= PK_CONE_MAX_COLS else 0
    return r16(s["JumpInfo"] * K) + r16(4 * (K + 1)) + r16(K) + cone + (r16(max_ctiles * TILE + 16) if stage_bases else 0)


def wide_smem_bytes(W, cmax):
    s = SIZES
    return (s["JumpInfo"] * cmax + s["RowM"] * cmax + (s["XsPart"] + s["CmPart"]) * cmax * W + 4 * cmax * 6 +
            s["ICarry"] * (2 * W + 2) + 64)


# ---- layouts and the decisions of run_chunk --------------------------------------------------------------------------------

def layout(contig_lens, double_strand=False):
    """(C, n_tiles, max_ctiles) of the layout holding every contig-strand."""
    ms = [m for m in contig_lens for _ in range(2 if double_strand else 1)]
    nt = [(m + TILE - 1) // TILE for m in ms]
    return len(ms), sum(nt), max(nt)


def plan_chunk(jobs, K, num_sms, walk_in_kernel=True, cluster_pref=0, cluster_min_tiles=CLUSTER_MIN_TILES, packed=True):
    """run_chunk for one chunk: `jobs` is a list of (layout, LB) with LB = 0 for a read on the wide path (keyedge.plan).
    Returns the decisions and the kernel launches of the chunk without window re-runs (each re-run adds 2)."""
    cmax = max(L[0] for L, _ in jobs)
    LBs = [LB if packed else 0 for _, LB in jobs]
    while True:   # packed jobs whose tables do not fit beside the chunk's largest contig count go wide, largest first
        nt, big = 1, None
        for k, (L, _) in enumerate(jobs):
            if LBs[k] and L[1] >= nt:
                nt, big = L[1], k
        if big is None or pack_smem_bytes(cmax, nt) <= SMEM_LIMIT:
            break
        LBs[big] = 0
    n_packed = sum(1 for LB in LBs if LB)
    n_wide = len(jobs) - n_packed
    ntmax = max([L[1] for (L, _), LB in zip(jobs, LBs) if LB], default=1)
    max_ctiles = max(L[2] for L, _ in jobs)
    cluster = cluster_pref
    if cluster == 0:
        cluster = 1
        while cluster < 16 and n_packed * cluster * 2 <= num_sms * 3 // 4:
            cluster *= 2
    if ntmax < cluster_min_tiles:
        cluster = 1
    psmem = r16(pack_smem_bytes(cmax, ntmax))
    in_kernel = bool(walk_in_kernel) and cluster == 1 and n_packed > 0
    pstage_bases = True
    if in_kernel:
        if psmem + unit_stage_bytes(K, max_ctiles, True) > SMEM_LIMIT:
            pstage_bases = False
        if psmem + unit_stage_bytes(K, max_ctiles, pstage_bases) > SMEM_LIMIT:
            in_kernel = False
    n_post = n_wide if in_kernel else len(jobs)
    wstage_bases = wstate_smem = None
    if n_post:
        wsmem = r16(max(wide_smem_bytes(WALK_WARPS, 1), pack_smem_bytes(1, max_ctiles, WALK_WARPS, 0)))
        wstage_bases = n_post > n_wide and wsmem + unit_stage_bytes(K, max_ctiles, True) <= SMEM_LIMIT
        wsmem += r16(unit_stage_bytes(K, max_ctiles, wstage_bases))
        wstate_smem = wsmem + 2 * max_ctiles * TILE * 4 <= WALK_STATE_SMEM_MAX
    launches = (1 if n_packed else 0) + (1 if n_wide else 0) + (2 if n_post else 0)
    return dict(n_packed=n_packed, n_wide=n_wide, cluster=cluster, in_kernel=in_kernel, pstage_bases=pstage_bases if in_kernel else None,
                wstage_bases=wstage_bases, wstate_smem=wstate_smem, launches=launches)


# ---- operation buffer ------------------------------------------------------------------------------------------------------

def chain_ops_bound(n, C):
    """No chain of a read of n columns against C contig-strands has more run-length ops (cuda_backend.cu)."""
    return 6 * n + 4 * C + 16


def ops_cap(n, C, walk_all, grow=0):
    """Operation buffer of a read after `grow` x4 growths (retries of its chunk)."""
    bound = chain_ops_bound(n, C) * (C if walk_all else 1)
    return min((n // 2 + 4 * C + 64) * (min(C, 8) if walk_all else 1) * 4 ** grow, bound, 0xffffffff)


def retries(n, C, walk_all, need):
    """Retries a read whose chains take `need` ops in all causes; None when the bound itself is exceeded (an error)."""
    g = 0
    while ops_cap(n, C, walk_all, g) < need:
        if ops_cap(n, C, walk_all, g) >= min(chain_ops_bound(n, C) * (C if walk_all else 1), 0xffffffff):
            return None
        g += 1
    return g


# ---- inputs shared by the CPU (emulator) and GPU tiers ---------------------------------------------------------------------

SWEEP_K = (7, 31, 32, 33, 96, 128, 160, 192, 224, 256, 383, 384, 385, 512, 1024, 2048, 8192)


def edge_read(rng, contig, L, n):
    """An exact copy of L contig bases followed by n - L N's: in local mode the best chain ends at column L, which is also the
    first column whose best cell reaches the best score (dp_core.h first_candidate_column, margin 0): the packed tail and the
    wide re-run must restart before it."""
    s = rng.randrange(0, len(contig) - L + 1)
    return contig[s:s + L] + b"N" * (n - L)


def spacing_case(seed=0):
    """Contigs of a few kb and noisy chimeric reads of 0.2-4 kb whose lengths sit on and around multiples of the swept spacings
    (mK - 1, mK, mK + 1, K = n, K > n), plus two edge reads of 1600 columns whose best chain ends at n - 64 (a late checkpoint
    column, or a regular one for the K that divide 1536) and at n - 80 (restart from the late checkpoint at n - 96)."""
    import random

    import gen
    rng = random.Random(5150 + seed)
    contigs = [gen.rand_seq(rng, rng.randint(1600, 2200)) for _ in range(3)] + [gen.rand_seq(rng, 700)]   # < 64 tiles: one CTA per read
    lengths = (224, 383, 384, 385, 672, 1023, 1024, 1025, 2048, 4000)
    reads = []
    for n in lengths:
        r = gen.chimeric_read(rng, contigs, n, 1 + n // 900, strands=True, wrap=True, noise=True)
        reads.append((r + gen.rand_seq(rng, n))[:n])
    reads.append(edge_read(rng, contigs[0], 1536, 1600))
    reads.append(edge_read(rng, contigs[1], 1520, 1600))
    return contigs, reads


def skip_case(n, C, k=1, seed=0):
    """C copies of one single-strand contig built as blocks of k bases from {A, C} followed by one base from {G, T}, and a read
    of n bases that is the contig with every G / T dropped.  Under SKIP_SCORING (match 2, mismatch -1, gap open 0, extend -1,
    jumps -4) the only optimal chain against each copy is k '=' and one contig-side gap (I) in turn from the contig's first
    base: score 2n - (blocks - 1), 2 * blocks - 1 run-length ops, where blocks = ceil(n / k); a suboptimal batch returns one
    such chain per copy."""
    import random
    rng = random.Random(77 + 1000 * k + seed)
    blocks = (n + k - 1) // k
    x, y = bytearray(), bytearray()
    for b in range(blocks + 8):
        block = bytes(rng.choice(b"AC") for _ in range(k))
        x += block + bytes([rng.choice(b"GT")])
        if b < blocks:
            y += block
    return [bytes(x)] * C, bytes(y[:n]), blocks


SKIP_SCORING = dict(match_score=2, mismatch_score=-1, gap_open=0, gap_extend=-1, default_jump_score=-4)


def skip_chain_ok(a, n, k, blocks, contig_idx):
    """The closed form of skip_case's chain (clips removed, as align_batch returns it)."""
    ops = [(0, min(k, n - b * k), 0) if t == 0 else (3, 1, 0) for b in range(blocks) for t in ((0, 1) if b + 1 < blocks else (0,))]
    return (a.score == 2 * n - (blocks - 1) and a.start_contig_idx == contig_idx and a.end_contig_idx == contig_idx and
            a.xstart == 0 and a.ystart == 0 and a.yend == n and [tuple(o) for o in a.ops] == ops)
