// K1b -- causal prior on a tensor grid:  m(x) = u(x).w ,  v(x) = s2 + noise - u(x)^T M u(x).
//
// Replaces DoCalculus.update_do_function / compute_do (reference DoCalculus.py:34-89): the reference
// rebuilds an (N x D) design per candidate and runs a full GP predict (O(N^2 D + N^3)); here the
// Monte-Carlo average has been folded into w and M once per observation (K1a) and each candidate costs a
// dense symmetric quadratic form in its N-vector u(x) = prod_k tab_k[i_k(x)][:].
//
// Shape of the work: T = U (G x N) * M (N x N) followed by a row-wise dot with U.  Only M's lower
// block triangle is visited: for column block J the k-blocks below the diagonal block are accumulated,
// doubled, and the (full, symmetric) diagonal block is added.  One work item = 128 candidates.
//
// Persistent kernel, one CTA per SM, work items claimed from an atomic counter.  Per item:
//   phase 1 (all warps)   : materialise the item's U tile (128 x Npad) ONCE, in DMMA fragment order, in the CTA's
//                           private global scratch (d table loads + (d-1) multiplies per element).  Doing the FP64
//                           multiplies here -- and not inside the k loop -- matters: DMUL shares the FP64 pipe with
//                           DMMA, and a producer warp issuing even 2 % of the pipe's work in the steady state stalled
//                           on math-pipe throttle long enough to starve the consumers (77 % -> 96 % of DMMA peak).
//   phase 2, producer     : one elected thread of a producer warpgroup (setmaxnreg 40); per 16-deep stage two contiguous
//   (warps 8-11)            16 KB TMA bulk copies (cp.async.bulk, SASS UBLKCP): the M slab (K1a stores M blocked in
//                           fragment order) and the U slab, both completing on the stage's "full" mbarrier (32 KB).
//   phase 2, consumers    : (setmaxnreg 232) wait "full", 4 x (12 LDS.64 + 32 DMMA.8x8x4), arrive on "empty".  They
//   (warps 0-7)             never touch global memory inside the k loop; after each J block a short epilogue dots the
//                           accumulators with u (re-read from the scratch) and w.  Warps whose rows are partly or wholly
//                           padding (last tile of a slice, small explicit-point batches) run instantiations with fewer
//                           live row blocks; a last column block with few live columns (N = 128 k + Lc, Lc <= 64) is
//                           consumed with all warps re-tiled over those columns (consume_ragged_block).
// Launches with too few tiles to fill the GPU (explicit points, small grids) are cut into segments of M's triangle
// (template SPLIT); the interventional rows (cbo_prior_eval which == 1) are evaluated by prior_rows.cu.
// Roofline: FP64 pipe.  Executed flops per candidate = N^2 (+ lower order); the dense-counted figure of
// SURVEY.md §8(d) is 2 N^2 + 2 N + d N.  Scratch traffic: each U slab is re-read once per J block
// (~N/256 times), about 1 TB/s of L2/HBM reads chip-wide at N = 1e4 -- 15 % of HBM bandwidth.
#include "m_triangle_pass.cuh"
#include "prior_pair.cuh"

namespace cbo {

constexpr int kPriorWsHeader = 256;  // bytes reserved at the start of the workspace (work counter)

constexpr int kPartialDoubles = 2 * CBO_PRIOR_TILE;   // one (q, m) partial per row of a work item
constexpr int kPartialFloor = 1024;                    // partial slots every workspace holds, besides 4 per CTA

// (this file is the grid / explicit-point evaluation, cbo_prior_eval which == 0; the interventional rows, which == 1,
// are evaluated in compensated arithmetic by prior_rows.cu)
// split = {chunk, nsplit}: chunk > 0 -> segments; else nsplit > 1 -> folded column blocks; else one item per tile.
// skip_pair: the launch leaves the sets of the small-N tensor-grid path (prior_pair.cu) alone -- they count no tiles here.
struct PriorSplit { int chunk, nsplit, skip_pair; };
__host__ __device__ inline long long prior_tiles(const cbo_set_desc& S, PriorSplit sp) {
    if (!computes_prior(S) || (sp.skip_pair && pair_eligible(S))) return 0;
    return (S.g_count + CBO_PRIOR_TILE - 1) / CBO_PRIOR_TILE;
}

// Work decomposition.  chunk == 0 (the grid): one item per 128-candidate tile walks every (jb, kt) of M's lower block
// triangle.  chunk > 0 (too few tiles to fill the GPU: small grids, small explicit-point batches): the
// triangle of each tile is cut into segments -- for column block jb, its strictly-lower k range in pieces of `chunk`
// column blocks (ceil(jb / chunk) of them, each counted twice in u^T M u) and its diagonal block -- one item per segment,
// so that M is streamed once by the WHOLE GPU and the launch is bound by HBM (or by the few rows' flops), not by one
// SM per tile.  The per-item partial row sums are combined in item order by prior_finalize_kernel (deterministic).
//   G(n) = sum_{x=0..n} ceil(x / chunk)   (closed form: decoding an item is O(sets) + O(log nJ))
__host__ __device__ inline long long prior_G(int n, int chunk) {
    if (n <= 0) return 0;
    const long long q = n / chunk, r = n - q * chunk;
    return (long long)chunk * q * (q + 1) / 2 + r * (q + 1);
}
// segments of column blocks [0, jb): F(jb) = sum_{x<jb} (ceil(x/chunk) + 1)
__host__ __device__ inline long long prior_F(int jb, int chunk) { return prior_G(jb - 1, chunk) + jb; }
// Fallback when a launch has too few tiles to fill the GPU but too many for segments to fit the partial buffer: the
// column blocks are dealt to `ns` items per tile, folded (jb mod 2ns in {sp, 2ns-1-sp}) so the triangular cost balances.
__host__ __device__ inline int prior_nsplit(const cbo_set_desc& S, int nsplit) {
    const int nJ = m_row_blocks(S), cap = nJ / 2 > 1 ? nJ / 2 : 1;
    return nsplit < cap ? nsplit : cap;
}
__host__ __device__ inline long long prior_items_per_tile(const cbo_set_desc& S, PriorSplit sp) {
    return sp.chunk > 0 ? prior_F(m_row_blocks(S), sp.chunk) : prior_nsplit(S, sp.nsplit);
}
__host__ __device__ inline long long prior_items(const cbo_set_desc& S, PriorSplit sp) {
    return prior_tiles(S, sp) * prior_items_per_tile(S, sp);
}

template <int WM_, int WN_, int MA_, int NB_, int STAGES_>
struct PriorCfg {
    static constexpr int WM = WM_, WN = WN_, MA = MA_, NB = NB_, STAGES = STAGES_;
    static constexpr int BM = WM * MA * 8;  // candidates per work item
    static constexpr int BN = WN * NB * 8;  // columns of M per J block
    static constexpr int NCONS = WM * WN * 32;   // consumer warps first ...
    static constexpr int NT = NCONS + 128;       // ... then one producer warpgroup (registers are allocated per warpgroup)
    static constexpr int A_TILE = BM * kBK;
    static constexpr int B_TILE = BN * kBK;
    static constexpr unsigned STAGE_BYTES = (A_TILE + B_TILE) * sizeof(double);
    static constexpr size_t SMEM = (size_t)STAGES * STAGE_BYTES + 2 * WN * BM * sizeof(double) +
                                   (CBO_MAX_D + 1) * BM * sizeof(int32_t) + 2 * STAGES * sizeof(uint64_t) + 16;
    // setmaxnreg redistributes the CTA's own allocation: NT x (registers per thread at launch, pinned by ptxas to the
    // __launch_bounds__ ceiling).  Asking for more than the pool deadlocks the consumers on the inc.
    static constexpr int LAUNCH_REGS = (65536 / NT) / 8 * 8;
    static constexpr int PROD_REGS = 40, CONS_REGS = 232;
    static_assert(BM == CBO_PRIOR_TILE, "host item count assumes CBO_PRIOR_TILE points per work item");
    static_assert(BN == kMBlkRows, "the J block must match the row block of M's blocked layout");
    static_assert(NCONS % 128 == 0, "setmaxnreg works on whole warpgroups");
    static_assert(128 * PROD_REGS + NCONS * CONS_REGS <= NT * LAUNCH_REGS, "setmaxnreg budget exceeds the CTA's register pool");
};

// One decoded work item (everything both roles need); decoded redundantly by every thread from the descriptors.
// It covers column blocks [jb0, jb1); a split item is one segment: a single column block and the k range [kt0, kt1)
// (in 16-deep slabs), which lies either wholly below the diagonal block or is the diagonal block.
struct PriorItem {
    const cbo_set_desc* S;
    int tile, nJ, jb0, jb1, kt0, kt1, sp, ns;
    int kmax;        // 16-deep k slabs that hold live rows of M: ceil(n_obs / 16); the slabs past them are zero padding
    bool split;      // a segment item
    bool partial;    // the item's row sums are partial (segments or folded column blocks): they go to the partial buffer
    __device__ __forceinline__ bool mine(int jb) const { const int r = jb % (2 * ns); return r == sp || r == 2 * ns - 1 - sp; }
    // SPLIT is a compile-time copy of `split` (kernel-uniform): the grid path keeps its loop bounds free of item state
    template <bool SPLIT> __device__ __forceinline__ int kbeg(int jb) const { return SPLIT ? kt0 : 0; }
    // end of the k loop: padding slabs are skipped by the producer and the consumers alike (U and M are exactly zero there,
    // so nothing changes but the stage count: 7 instead of 8 at N = 100); phase 1 still fills them for the epilogue's reads
    template <bool SPLIT> __device__ __forceinline__ int kend(int jb) const {
        const int e = SPLIT ? kt1 : (jb + 1) * kSlabsPerBlock;
        return e < kmax ? e : kmax;
    }
};

// First work item of every set, computed on the host and passed as a kernel parameter: finding an item's set is a scan
// over constants instead of a walk over the descriptors in global memory (which cost 5 us per item with coral's 25 sets --
// as much as a quarter of a 128-column item's DMMA time).  Launches with more sets than fit fall back to the walk.
constexpr int kMaxBases = 32;
struct PriorBases { int n; int base[kMaxBases + 1]; };

__device__ __forceinline__ PriorItem decode_prior_item(const cbo_set_desc* __restrict__ sets, int num_sets, PriorSplit split,
                                                       const PriorBases& pb, int item) {
    const int chunk = split.chunk;
    int local = item, s = 0;
    if (pb.n == num_sets) {
#pragma unroll 1
        for (; s < num_sets - 1; ++s)
            if (item < pb.base[s + 1]) break;
        local = item - pb.base[s];
    } else {
        for (; s < num_sets - 1; ++s) {
            const int cnt = (int)prior_items(sets[s], split);
            if (local < cnt) break;
            local -= cnt;
        }
    }
    PriorItem it;
    it.S = sets + s;
    it.nJ = m_row_blocks(sets[s]);
    it.kmax = (sets[s].n_obs + kBK - 1) / kBK;
    it.split = chunk > 0;
    it.sp = 0, it.ns = 1;
    if (!it.split) {
        it.ns = prior_nsplit(sets[s], split.nsplit);
        it.tile = local / it.ns, it.sp = local % it.ns;
        it.jb0 = 0, it.jb1 = it.nJ, it.kt0 = it.kt1 = 0;
        it.partial = it.ns > 1;
        return it;
    }
    it.partial = prior_F(it.nJ, chunk) > 1;
    const int per_tile = (int)prior_F(it.nJ, chunk);
    it.tile = local / per_tile;
    const int seg = local - it.tile * per_tile;
    int lo = 0, hi = it.nJ - 1;                  // largest jb with F(jb) <= seg
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (prior_F(mid, chunk) <= seg) lo = mid; else hi = mid - 1;
    }
    const int jb = lo, piece = seg - (int)prior_F(jb, chunk), lower = (jb + chunk - 1) / chunk;
    it.jb0 = jb, it.jb1 = jb + 1;
    if (piece < lower) {                         // strictly-lower piece: column blocks [piece*chunk, min(jb, (piece+1)*chunk))
        const int b1 = (piece + 1) * chunk < jb ? (piece + 1) * chunk : jb;
        it.kt0 = piece * chunk * kSlabsPerBlock, it.kt1 = b1 * kSlabsPerBlock;
    } else {                                     // the diagonal block
        it.kt0 = jb * kSlabsPerBlock, it.kt1 = (jb + 1) * kSlabsPerBlock;
    }
    return it;
}

__device__ __forceinline__ void bar_all(int nthreads) { asm volatile("bar.sync 0, %0;" ::"r"(nthreads) : "memory"); }
__device__ __forceinline__ void bar_consumers(int nthreads) { asm volatile("bar.sync 1, %0;" ::"r"(nthreads) : "memory"); }

// The LAST column block of M when few of its 128 columns are live (n_obs = 128 (nJ - 1) + Lc with Lc <= 64; config 5 has
// Lc = 16).  In the regular warp tiling only the warps that own the live columns would do useful DMMAs while the block
// still costs a full 1/nJ-th of the item's longest k loop (2.5 % of an item at nJ = 79).  Here the 8 consumer warps are
// re-tiled over (128 rows) x (NW * NB2 * 8 live columns): MW x NW warps of MA2 x NB2 blocks each, so the block costs
// Lc/128 of a full one (it then runs at the speed the slabs arrive).  Same ring protocol: every warp waits on every
// stage and arrives once.
template <class Cfg, int MW, int NW, int MA2, int NB2>
__device__ __forceinline__ void consume_ragged_block(const PriorItem& it, const double* __restrict__ sA, const double* __restrict__ sB,
                                                     double* __restrict__ sRed, uint64_t* full, uint64_t* empty, int& stage,
                                                     unsigned& phase, const double* __restrict__ scratch, const double* __restrict__ w,
                                                     int warp, int lane) {
    constexpr int BM = Cfg::BM, BN = Cfg::BN, WN = Cfg::WN, STAGES = Cfg::STAGES;
    static_assert(MW * NW * 32 == Cfg::NCONS && MW * MA2 * 8 == BM && NW <= WN, "re-tiling must cover the 128 rows with all consumer warps");
    const int jb = it.nJ - 1, noff = jb * kSlabsPerBlock, ke = it.kmax;   // (kmax <= nJ * 8: the padding slabs are skipped)
    const int row0 = (warp / NW) * MA2 * 8, wn2 = warp % NW, col0 = wn2 * NB2 * 8;
    double acc[MA2][NB2][2];
#pragma unroll
    for (int mi = 0; mi < MA2; ++mi)
#pragma unroll
        for (int ni = 0; ni < NB2; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
    auto run = [&](int k0, int k1) {
#pragma unroll 1
        for (int kt = k0; kt < k1; ++kt) {
            mbar_wait(&full[stage], phase);
            mma_stage<BM, BN, MA2, NB2, MA2>(sA + stage * Cfg::A_TILE, sB + stage * Cfg::B_TILE, acc, row0, col0, lane);
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[stage]);
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
    };
    run(0, noff);
#pragma unroll
    for (int mi = 0; mi < MA2; ++mi)
#pragma unroll
        for (int ni = 0; ni < NB2; ++ni) { acc[mi][ni][0] *= 2.0; acc[mi][ni][1] *= 2.0; }
    run(noff, ke);
    // the row sums of this block go into slots that other warps own in the regular tiling: wait until every consumer
    // warp is past its earlier epilogues (the producer takes no part in barrier 1)
    bar_consumers(Cfg::NCONS);
#pragma unroll
    for (int mi = 0; mi < MA2; ++mi) {
        const int r = row0 + mi * 8 + (lane >> 2);
        double q = 0.0, mm = 0.0;
#pragma unroll
        for (int ni = 0; ni < NB2; ++ni) {
            const int j = jb * BN + col0 + ni * 8 + (lane & 3) * 2;
            const double2 u = __ldcg(reinterpret_cast<const double2*>(scratch + (size_t)(j >> 4) * Cfg::A_TILE + frag_off(BM, (j & 15) >> 2, r, j & 3)));
            const double2 ww = ldg_nc_d2(w + j);
            q = fma(acc[mi][ni][0], u.x, q);
            q = fma(acc[mi][ni][1], u.y, q);
            mm = fma(u.x, ww.x, mm);
            mm = fma(u.y, ww.y, mm);
        }
        q += __shfl_xor_sync(0xffffffffu, q, 1);
        q += __shfl_xor_sync(0xffffffffu, q, 2);
        mm += __shfl_xor_sync(0xffffffffu, mm, 1);
        mm += __shfl_xor_sync(0xffffffffu, mm, 2);
        if ((lane & 3) == 0) {  // (wn2, r) has exactly one owner in this tiling
            sRed[wn2 * BM + r] += q;
            sRed[(WN + wn2) * BM + r] += mm;
        }
    }
}

// Consumer k loop + J-block epilogues of one work item for a warp whose first LIVE row blocks (of MA) hold live rows.
// LIVE == 0: the warp owns only padding rows; it still walks the ring (wait full / arrive empty) so the counts match.
template <class Cfg, int LIVE, bool SPLIT>
__device__ __forceinline__ void consume_item(const PriorItem& it, const double* __restrict__ sA, const double* __restrict__ sB,
                                             double* __restrict__ sRed, uint64_t* full, uint64_t* empty, int& stage, unsigned& phase,
                                             const double* __restrict__ scratch, const double* __restrict__ w, int warp, int lane,
                                             int ragged_cols) {
    constexpr int BM = Cfg::BM, BN = Cfg::BN, MA = Cfg::MA, NB = Cfg::NB, WN = Cfg::WN, STAGES = Cfg::STAGES;
    static_assert(BN / kBK == kSlabsPerBlock, "J block width");
    const int wm = warp / WN, wn = warp % WN;
    const int row0 = wm * MA * 8, col0 = wn * NB * 8;
    if constexpr (LIVE == 0) {
#pragma unroll 1
        for (int jb = it.jb0; jb < it.jb1; ++jb) {
            if (!it.mine(jb)) continue;
#pragma unroll 1
            for (int kt = it.template kbeg<SPLIT>(jb); kt < it.template kend<SPLIT>(jb); ++kt) {
                mbar_wait(&full[stage], phase);
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[stage]);
                if (++stage == STAGES) { stage = 0; phase ^= 1u; }
            }
        }
        return;
    }
    constexpr int LV = LIVE > 0 ? LIVE : 1;
    double acc[MA][NB][2];
#pragma unroll
    for (int mi = 0; mi < MA; ++mi)
#pragma unroll
        for (int ni = 0; ni < NB; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;

    // full tiles of the grid path hand the last column block to consume_ragged_block when at most 64 of its columns are live
    const int jend = (!SPLIT && LIVE == MA && ragged_cols > 0) ? it.nJ - 1 : it.jb1;
#pragma unroll 1
    for (int jb = it.jb0; jb < jend; ++jb) {
        if (!it.mine(jb)) continue;
        const int kb = it.template kbeg<SPLIT>(jb), ke = it.template kend<SPLIT>(jb), noff = jb * kSlabsPerBlock;   // noff: first slab of the diagonal block
        auto double_acc = [&]() {   // strictly-lower blocks appear twice in u^T M u
#pragma unroll
            for (int mi = 0; mi < LV; ++mi)
#pragma unroll
                for (int ni = 0; ni < NB; ++ni) { acc[mi][ni][0] *= 2.0; acc[mi][ni][1] *= 2.0; }
        };
        auto run = [&](int k0, int k1) {    // the steady state: wait full, 4 x (12 LDS.64 + 32 DMMA), arrive empty
#pragma unroll 1
            for (int kt = k0; kt < k1; ++kt) {
                mbar_wait(&full[stage], phase);
                mma_stage<BM, BN, MA, NB, LV>(sA + stage * Cfg::A_TILE, sB + stage * Cfg::B_TILE, acc, row0, col0, lane);
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[stage]);
                if (++stage == STAGES) { stage = 0; phase ^= 1u; }
            }
        };
        if constexpr (SPLIT) {
            run(kb, ke);                     // a segment lies wholly below the diagonal block or is the diagonal block
        } else {
            run(kb, noff);                   // strictly-lower blocks ...
            double_acc();                    // ... count twice (doubling the zeros of jb == 0 is harmless) ...
            run(noff, ke);                   // ... the diagonal block once; the doubling stays out of the k loop
        }
        if (ke <= noff) double_acc();        // a split item's segment that lies wholly below the diagonal block
        const bool with_m = ke > noff;        // the segment holding the diagonal block also carries the block's share of u.w
        // J-block epilogue: q_g += sum_{j in J} T[g][j] u[g][j] ; m_g += sum_{j in J} u[g][j] w[j]
        // (u of column block jb sits in the scratch at slab jb*8 - ubase: a lower segment keeps it after its k slabs)
        const int ubase = !SPLIT ? 0 : (ke <= noff ? noff - (ke - kb) : kb);
#pragma unroll
        for (int mi = 0; mi < LV; ++mi) {
            const int r = row0 + mi * 8 + (lane >> 2);
            double q = 0.0, mm = 0.0;
#pragma unroll
            for (int ni = 0; ni < NB; ++ni) {
                const int j = jb * BN + col0 + ni * 8 + (lane & 3) * 2;
                const double2 u = __ldcg(reinterpret_cast<const double2*>(   // L2: never a stale L1 line of an earlier item
                    scratch + (size_t)((j >> 4) - ubase) * Cfg::A_TILE + frag_off(BM, (j & 15) >> 2, r, j & 3)));
                const double2 ww = ldg_nc_d2(w + j);   // unconditional: the loads of the whole epilogue stay batched
                q = fma(acc[mi][ni][0], u.x, q);
                q = fma(acc[mi][ni][1], u.y, q);
                mm = fma(u.x, ww.x, mm);
                mm = fma(u.y, ww.y, mm);
                acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
            }
            q += __shfl_xor_sync(0xffffffffu, q, 1);
            q += __shfl_xor_sync(0xffffffffu, q, 2);
            mm += __shfl_xor_sync(0xffffffffu, mm, 1);
            mm += __shfl_xor_sync(0xffffffffu, mm, 2);
            if ((lane & 3) == 0) {  // (wn, r) has exactly one owner: no race, fixed order -> deterministic
                sRed[wn * BM + r] += q;
                if (with_m) sRed[(WN + wn) * BM + r] += mm;
            }
        }
    }
    if constexpr (!SPLIT && LIVE == MA) {
        if (ragged_cols > 32) consume_ragged_block<Cfg, 4, 2, 4, 4>(it, sA, sB, sRed, full, empty, stage, phase, scratch, w, warp, lane);
        else if (ragged_cols > 16) consume_ragged_block<Cfg, 8, 1, 2, 4>(it, sA, sB, sRed, full, empty, stage, phase, scratch, w, warp, lane);
        else if (ragged_cols > 0) consume_ragged_block<Cfg, 8, 1, 2, 2>(it, sA, sB, sRed, full, empty, stage, phase, scratch, w, warp, lane);
    }
}

template <class Cfg, bool SPLIT>
__global__ void __launch_bounds__(Cfg::NT, 1)
prior_eval_kernel(const cbo_set_desc* __restrict__ sets, int num_sets, PriorSplit split, const PriorBases pb, int total_items,
                  int* __restrict__ counter, double* __restrict__ partials, double* __restrict__ scratch_base, size_t slot_doubles) {
    constexpr int BM = Cfg::BM, BN = Cfg::BN, WN = Cfg::WN, NT = Cfg::NT, NCONS = Cfg::NCONS;
    constexpr int STAGES = Cfg::STAGES;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* sA = reinterpret_cast<double*>(smem_raw);
    double* sB = sA + STAGES * Cfg::A_TILE;
    double* sRed = sB + STAGES * Cfg::B_TILE;                          // [2][WN][BM] running q and m partial sums
    uint64_t* bars = reinterpret_cast<uint64_t*>(sRed + 2 * WN * BM);  // full[STAGES], empty[STAGES]
    int32_t* sRow = reinterpret_cast<int32_t*>(bars + 2 * STAGES);     // [CBO_MAX_D + 1][BM]: table row offsets, live flag
    volatile int32_t* sItem = sRow + (CBO_MAX_D + 1) * BM;
    uint64_t* full = bars;
    uint64_t* empty = bars + STAGES;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double* __restrict__ scratch = scratch_base + (size_t)blockIdx.x * slot_doubles;

    if (tid == 0) {
        for (int i = 0; i < STAGES; ++i) {
            mbar_init(&full[i], 1);               // the producer's arrive.expect_tx; the bytes come from the TMA
            mbar_init(&empty[i], Cfg::WM * WN);  // one arrive per consumer warp
        }
        mbar_fence_init();
        *sItem = atomicAdd(counter, 1);
    }
    __syncthreads();
    int stage = 0;        // ring position, carried across work items (producer and consumers advance identically)
    unsigned phase = 0;

    // Per item, three CTA-wide barriers (bar 0, all NT threads) in both roles:
    //   A  the item id in sItem is valid                B  the U scratch of the item is complete (TMA may read it)
    //   C  the item is retired (sItem / sRow / sRed / scratch may be overwritten)
    if (warp >= NCONS / 32) {
        // =============================== PRODUCER WARPGROUP (one elected thread works) ===============================
        setmaxnreg_dec<Cfg::PROD_REGS>();
        for (;;) {
            const int item = *sItem;                                   // barrier A happened (kernel start / end of last item)
            if (item >= total_items) break;
            const PriorItem it = decode_prior_item(sets, num_sets, split, pb, item);
            const double* __restrict__ M = it.S->M;
            const int Npad = it.S->n_obs_pad;
            bar_all(NT);                                               // B
            if (warp == NCONS / 32 && lane == 0) {
#pragma unroll 1
                for (int jb = it.jb0; jb < it.jb1; ++jb) {
                    if (!it.mine(jb)) continue;
                    const int kb = it.template kbeg<SPLIT>(jb), ke = it.template kend<SPLIT>(jb);
#pragma unroll 1
                    for (int kt = kb; kt < ke; ++kt) {
                        mbar_wait(&empty[stage], phase ^ 1u);
                        mbar_arrive_expect_tx(&full[stage], Cfg::STAGE_BYTES);
                        bulk_g2s(sB + stage * Cfg::B_TILE, M + mblk_base(jb, kt, Npad), Cfg::B_TILE * sizeof(double), &full[stage]);
                        bulk_g2s(sA + stage * Cfg::A_TILE, scratch + (size_t)(kt - kb) * Cfg::A_TILE, Cfg::A_TILE * sizeof(double), &full[stage]);
                        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                    }
                }
            }
            __syncwarp();
            bar_all(NT);                                               // C (+ A of the next item: consumer thread 0 wrote sItem before it)
        }
    } else {
        // =============================== CONSUMER WARPGROUPS ===============================
        setmaxnreg_inc<Cfg::CONS_REGS>();
        for (;;) {
            const int item = *sItem;
            if (item >= total_items) break;
            const PriorItem it = decode_prior_item(sets, num_sets, split, pb, item);
            const cbo_set_desc& S = *it.S;
            // effective problem: the tensor grid, or explicit points (one table with a row per candidate)
            const int d = S.points ? 1 : S.d;
            const long long gbeg = S.g_begin, gcnt = S.g_count;
            const int Npad = S.n_obs_pad;
            // 16-wide column slabs of U the item touches: all of them, or (split item) its k range [kt0, kt1) followed,
            // for a segment below the diagonal, by the 8 slabs of column block jb that the epilogue dots with
            const int nk_item = SPLIT ? it.kt1 - it.kt0 : it.nJ * kSlabsPerBlock;
            const bool extra = SPLIT && it.kt1 <= it.jb0 * kSlabsPerBlock;
            const int nKT = nk_item + (extra ? kSlabsPerBlock : 0);
            // live rows of this item (the last tile of a slice and the interventional rows fill only part of the 128):
            // rows past them are never generated, multiplied or stored (rows of U are independent in U*M)
            const long long left = gcnt - (long long)it.tile * BM;
            const int nlive = left < BM ? (int)left : BM;

            // per-row table offsets (C-order decomposition of the flat grid index, last dim fastest)
            const bool small_grid = S.g_total < 0x7fffffffLL;   // 32-bit index arithmetic (64-bit div/mod is a long emulated sequence)
            for (int r = tid; r < BM; r += NCONS) {
                const bool live = r < nlive;
                const long long g0 = gbeg + (live ? (long long)it.tile * BM + r : 0);
                if (small_grid) {
                    unsigned gg = (unsigned)g0;
#pragma unroll
                    for (int k = CBO_MAX_D - 1; k >= 0; --k) {
                        if (k < d) {
                            const unsigned pk = S.points ? (unsigned)S.g_total : (unsigned)S.p[k], q = gg / pk;
                            sRow[k * BM + r] = (int)(gg - q * pk) * Npad;
                            gg = q;
                        }
                    }
                } else {
                    long long gg = g0;
#pragma unroll
                    for (int k = CBO_MAX_D - 1; k >= 0; --k) {
                        if (k < d) {
                            const long long pk = S.points ? S.g_total : (long long)S.p[k];
                            sRow[k * BM + r] = (int)(gg % pk) * Npad;
                            gg /= pk;
                        }
                    }
                }
                sRow[CBO_MAX_D * BM + r] = live ? 1 : 0;
            }
            for (int i = tid; i < 2 * WN * BM; i += NCONS) sRed[i] = 0.0;
            bar_consumers(NCONS);

            // ---- phase 1: U tile -> scratch, fragment order [kt][k4 group][row][4] -------------------------------
            {
                const double* tab[CBO_MAX_D];
#pragma unroll
                for (int k = 0; k < CBO_MAX_D; ++k) tab[k] = S.tab[k < d ? k : 0];
                // unit = one 16-byte pair of one row; a warp's 32 units are 4 rows x 128 bytes of one slab: the table
                // reads are four full lines and the scratch writes four full lines.  A thread owns the SAME (row, k pair)
                // positions in every slab, so its row offsets, live flags and scratch offsets are set up once per item and
                // the slab loop is loads, multiplies and a store -- no index arithmetic, no division.
                const int per_slab = ((nlive + 3) >> 2) * 32;   // 16-byte units of the live rows in one slab
                constexpr int UW = (BM / 4 * 32 + NCONS - 1) / NCONS;
                int roff[UW][CBO_MAX_D], dst0[UW], j0[UW];
                bool valid[UW], live[UW];
#pragma unroll
                for (int x = 0; x < UW; ++x) {
                    const int wi = tid + x * NCONS, l = wi & 31;
                    const int kb = l >> 3, half = l & 1, row = (wi >> 5) * 4 + ((l & 7) >> 1);
                    valid[x] = wi < per_slab;
                    live[x] = valid[x] && sRow[CBO_MAX_D * BM + row] != 0;
                    j0[x] = kb * 4 + half * 2;
                    dst0[x] = frag_off(BM, kb, row, half * 2);
#pragma unroll
                    for (int k = 0; k < CBO_MAX_D; ++k) roff[x][k] = (k < d && valid[x]) ? sRow[k * BM + row] : 0;
                }
#pragma unroll 1
                for (int ks = 0; ks < nKT; ++ks) {                  // ks: slab inside the scratch
                    const int kt = !SPLIT ? ks : (ks < nk_item ? it.kt0 + ks : it.jb0 * kSlabsPerBlock + (ks - nk_item));
                    double2 v[UW];
#pragma unroll
                    for (int x = 0; x < UW; ++x) {
                        v[x] = make_double2(0.0, 0.0);
                        if (live[x]) {
                            const int j = kt * kBK + j0[x];
                            v[x] = ldg_nc_d2(tab[0] + roff[x][0] + j);
#pragma unroll
                            for (int k = 1; k < CBO_MAX_D; ++k) {
                                if (k < d) {
                                    const double2 t = ldg_nc_d2(tab[k] + roff[x][k] + j);
                                    v[x].x *= t.x; v[x].y *= t.y;
                                }
                            }
                        }
                    }
#pragma unroll
                    for (int x = 0; x < UW; ++x)
                        if (valid[x]) *reinterpret_cast<double2*>(scratch + (size_t)ks * Cfg::A_TILE + dst0[x]) = v[x];
                }
                fence_proxy_async();  // generic-proxy writes above -> visible to the TMA (async proxy) reads below
            }
            bar_all(NT);                                               // B

            {   // live row blocks of THIS warp (warp-uniform), rounded up to an instantiated count
                const int live_here = nlive - (warp / WN) * Cfg::MA * 8;
                const int need = live_here <= 0 ? 0 : (live_here + 7) >> 3;
                // live columns of the last column block when they are few (<= 64) and the item is a full tile of a grid
                // launch with more than one column block; 0 = regular tiling throughout.  CTA-uniform: every consumer
                // warp of a full tile runs the LIVE == MA instantiation.
                const int lc = S.n_obs - (it.nJ - 1) * BN;
                // (the item must own that block: when the column blocks are dealt to several items per tile -- nsplit > 1, a
                // grid with too few tiles for segments -- most items do not, and the producer streams nothing for it)
                const int ragged_cols = (!SPLIT && nlive == BM && it.nJ > 1 && lc <= 64 && it.mine(it.nJ - 1)) ? lc : 0;
#define CBO_CONSUME(LIVE) consume_item<Cfg, LIVE, SPLIT>(it, sA, sB, sRed, full, empty, stage, phase, scratch, S.w, warp, lane, ragged_cols)
                if (need >= 7) CBO_CONSUME(8);
                else if (need == 6) CBO_CONSUME(6);
                else if (need == 5) CBO_CONSUME(5);
                else if (need == 4) CBO_CONSUME(4);
                else if (need == 3) CBO_CONSUME(3);
                else if (need == 2) CBO_CONSUME(2);
                else if (need == 1) CBO_CONSUME(1);
                else CBO_CONSUME(0);
#undef CBO_CONSUME
            }
            bar_consumers(NCONS);

            double* out_m = S.m;
            double* out_v = S.v;
            for (int r = tid; r < nlive; r += NCONS) {
                const long long loc = (long long)it.tile * BM + r;
                double qs = 0.0, ms = 0.0;
#pragma unroll
                for (int x = 0; x < WN; ++x) { qs += sRed[x * BM + r]; ms += sRed[(WN + x) * BM + r]; }
                if (it.partial) {             // partial sums of this segment / column-block share; prior_finalize_kernel adds them up
                    partials[(size_t)item * kPartialDoubles + r] = qs;
                    partials[(size_t)item * kPartialDoubles + BM + r] = ms;
                } else {
                    out_m[loc] = ms;
                    out_v[loc] = (S.s2 + S.noise) - qs;
                }
            }
            bar_consumers(NCONS);                                      // everyone has read this item's sItem / sRed
            if (tid == 0) *sItem = atomicAdd(counter, 1);
            bar_all(NT);                                               // C / A
        }
    }
}

// Adds the partial row sums of every (set, tile) in item order (deterministic) and writes m, v.
__global__ void __launch_bounds__(CBO_PRIOR_TILE)
prior_finalize_kernel(const cbo_set_desc* __restrict__ sets, int num_sets, PriorSplit split,
                      const double* __restrict__ partials) {
    long long base = 0;
    for (int s = 0; s < num_sets; ++s) {
        const cbo_set_desc& S = sets[s];
        const int tiles = (int)prior_tiles(S, split);
        if (tiles == 0) continue;
        const int per = (int)prior_items_per_tile(S, split);
        if (per > 1) {
            const long long gcnt = S.g_count;
            double* out_m = S.m;
            double* out_v = S.v;
            for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
                const int r = threadIdx.x;
                const long long loc = (long long)tile * CBO_PRIOR_TILE + r;
                if (loc < gcnt) {
                    double qs = 0.0, ms = 0.0;
                    const double* p = partials + (size_t)(base + (long long)tile * per) * kPartialDoubles;
                    for (int i = 0; i < per; ++i, p += kPartialDoubles) {
                        qs += p[r];
                        ms += p[CBO_PRIOR_TILE + r];
                    }
                    out_m[loc] = ms;
                    out_v[loc] = (S.s2 + S.noise) - qs;
                }
            }
        }
        base += (long long)tiles * per;
    }
}

// ---- host side ----------------------------------------------------------------------------------------
using PriorCfgA = PriorCfg<2, 4, 8, 4, 4>;   // 8 consumer warps + 1 producer warp, 128 x 128 tile, 64 accumulators/thread

static size_t prior_slot_doubles(const cbo_set_desc* h_sets, int num_sets) {
    int npad = 0;
    for (int s = 0; s < num_sets; ++s)
        if (computes_prior(h_sets[s]) && h_sets[s].n_obs_pad > npad) npad = h_sets[s].n_obs_pad;
    return (size_t)CBO_PRIOR_TILE * npad;
}

static size_t prior_partial_items(long long ctas) { return (size_t)(4 * ctas + kPartialFloor); }

size_t prior_rows_workspace_bytes(const cbo_set_desc* h_sets, int num_sets);
int prior_rows_impl(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, void* d_ws, size_t ws_bytes,
                    size_t ws_offset, cudaStream_t st);

// workspace = [256 B header][pair tables of the small-N tensor-grid sets (prior_pair.cu)][partials][ctas scratch slots];
// the interventional-rows kernel (which == 1, prior_rows.cu) runs stream-ordered with the grid kernels and reuses
// everything behind the header for its own partials (the pair tables are rebuilt by every which == 0 call)
static size_t pair_area_bytes(const cbo_set_desc* h_sets, int num_sets) {
    return (pair_area_doubles(h_sets, num_sets) * sizeof(double) + 255) / 256 * 256;
}

size_t prior_workspace_bytes_impl(const cbo_set_desc* h_sets, int num_sets, int num_ctas) {
    const size_t grid = pair_area_bytes(h_sets, num_sets) + prior_partial_items(num_ctas) * kPartialDoubles * sizeof(double) +
                        (size_t)num_ctas * prior_slot_doubles(h_sets, num_sets) * sizeof(double);
    const size_t rows = prior_rows_workspace_bytes(h_sets, num_sets);
    return kPriorWsHeader + (grid > rows ? grid : rows);
}

// FP64 flops issued through DMMA by one which == 0 call (cbo_prior_eval_flops): the pair-table sets when the call takes
// that path (at least one item per SM), everything else through the general kernel's lower block triangle.
double prior_eval_flops_impl(const cbo_set_desc* h_sets, int num_sets, int num_sms) {
    const bool pair = pair_items_total(h_sets, num_sets) >= num_sms;
    double fl = 0.0;
    for (int s = 0; s < num_sets; ++s) {
        const cbo_set_desc& S = h_sets[s];
        if (!computes_prior(S) || S.g_count == 0) continue;
        if (pair && pair_eligible(S)) {
            const PairGeom g = pair_geom(S);
            double blocks = 0.0;    // live 8 x 8 blocks of all tiles of one plane
            for (int ca = 0; ca < g.nchA; ++ca)
                for (int cb = 0; cb < g.nchB; ++cb) {
                    const int ra = g.pa - ca * g.CRa, rb = g.pb - cb * g.CRb;
                    blocks += (double)(((ra < g.CRa ? ra : g.CRa) + 7) / 8) * (((rb < g.CRb ? rb : g.CRb) + 7) / 8);
                }
            fl += 2.0 * 64.0 * blocks * g.s_count * (double)g.Kslabs * kBK;
        } else {
            const int nJ = m_row_blocks(S), lc = S.n_obs - (nJ - 1) * kMBlkRows;
            const int last_cols = (nJ == 1 || lc > 64) ? 128 : (lc <= 16 ? 16 : (lc <= 32 ? 32 : 64));
            const double n16 = (double)((S.n_obs + kBK - 1) / kBK * kBK);
            fl += (double)S.g_count * 2.0 * (128.0 * 128.0 * (nJ - 1) * nJ / 2.0 + last_cols * n16);
        }
    }
    return fl;
}

int prior_eval_impl(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, int which, void* d_ws,
                    size_t ws_bytes, cudaStream_t st) {
    if (which == 1) return prior_rows_impl(h_sets, d_sets, num_sets, d_ws, ws_bytes, kPriorWsHeader, st);
    int dev = 0, sms = 0;
    CBO_CUDA(cudaGetDevice(&dev));
    CBO_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const size_t slot = prior_slot_doubles(h_sets, num_sets);
    const size_t fixed = kPriorWsHeader + (size_t)kPartialFloor * kPartialDoubles * sizeof(double);
    const size_t per_cta = 4 * kPartialDoubles * sizeof(double) + slot * sizeof(double);
    // the pair area is part of the layout whenever the workspace has room for it next to one scratch slot (it always has
    // when it was sized with cbo_prior_workspace_bytes); a smaller workspace runs every set through the general kernel
    size_t pair_bytes = pair_area_bytes(h_sets, num_sets);
    if (d_ws == nullptr || ws_bytes < fixed + per_cta + pair_bytes) pair_bytes = 0;
    // The small-N path needs enough (scale row, tile) items to occupy the GPU: a launch with fewer items than SMs (one or
    // two small 2-D grids, e.g. the complete graph's six sets) is served better by the general kernel's segment split.
    PriorSplit split{0, 1, 0};
    if (pair_bytes > 0 && pair_items_total(h_sets, num_sets) >= sms) split.skip_pair = 1;
    if (split.skip_pair) {
        const int rc = prior_pair_impl(h_sets, d_sets, num_sets, reinterpret_cast<double*>(static_cast<unsigned char*>(d_ws) + kPriorWsHeader),
                                       sms, st);
        if (rc != 0) return rc;
    }
    long long tiles = 0;
    for (int s = 0; s < num_sets; ++s) {
        const cbo_set_desc& S = h_sets[s];
        if (prior_tiles(S, split) == 0) continue;
        for (int k = 0; k < (S.points ? 1 : S.d); ++k) {
            const long long pk = S.points ? S.g_total : (long long)S.p[k];
            CBO_REQUIRE(pk * (long long)S.n_obs_pad < 2147483647LL, "cbo_prior_eval: table %d of set %d too large", k, s);
        }
        CBO_REQUIRE((long long)CBO_PRIOR_TILE * S.n_obs_pad < 2147483647LL, "cbo_prior_eval: set %d n_obs_pad too large", s);
        tiles += prior_tiles(S, split);
    }
    if (tiles == 0) return 0;
    CBO_REQUIRE(d_ws != nullptr && ws_bytes >= fixed + per_cta + pair_bytes,
                "cbo_prior_eval: workspace of %zu bytes cannot hold one scratch slot (%zu bytes needed); see cbo_prior_workspace_bytes",
                ws_bytes, fixed + per_cta + pair_bytes);
    long long ctas = (long long)((ws_bytes - fixed - pair_bytes) / per_cta);
    if (ctas > sms) ctas = sms;      // one CTA per SM (shared memory bound); more slots than SMs are not used
    // too few tiles to fill the GPU twice over: cut every tile's triangle of M into segments (as fine as the partial
    // buffer and a 4-items-per-CTA budget allow); when even the coarsest segments do not fit, deal out column blocks
    auto count = [&](PriorSplit sp) {
        long long t = 0;
        for (int s = 0; s < num_sets; ++s) t += prior_items(h_sets[s], sp);
        return t;
    };
    if (tiles < 2 * ctas) {
        int nJmax = 1;
        for (int s = 0; s < num_sets; ++s)
            if (prior_tiles(h_sets[s], split) > 0 && m_row_blocks(h_sets[s]) > nJmax) nJmax = m_row_blocks(h_sets[s]);
        const long long budget = (long long)prior_partial_items(ctas) < 4 * ctas ? (long long)prior_partial_items(ctas) : 4 * ctas;
        for (int c = 1; c <= nJmax && nJmax > 1; ++c)
            if (count(PriorSplit{c, 1, split.skip_pair}) <= budget) { split.chunk = c; break; }
        if (split.chunk == 0) {
            split.nsplit = (int)((2 * ctas + tiles - 1) / tiles);
            while (split.nsplit > 1 && count(split) > (long long)prior_partial_items(ctas)) --split.nsplit;
        }
    }
    const long long total = count(split);
    const bool partial = split.chunk > 0 || split.nsplit > 1;
    CBO_REQUIRE(total < 2147483647LL, "cbo_prior_eval: too many work items");
    CBO_REQUIRE(!partial || (size_t)total <= prior_partial_items(ctas), "cbo_prior_eval: internal: partial buffer too small");
    const long long grid = ctas < total ? ctas : total;
    unsigned char* ws = reinterpret_cast<unsigned char*>(d_ws);
    double* partials = reinterpret_cast<double*>(ws + kPriorWsHeader + pair_bytes);
    double* scratch = partials + prior_partial_items(ctas) * kPartialDoubles;
    auto kern = split.chunk > 0 ? prior_eval_kernel<PriorCfgA, true> : prior_eval_kernel<PriorCfgA, false>;
    CBO_CUDA(allow_dynamic_smem(prior_eval_kernel<PriorCfgA, true>, PriorCfgA::SMEM));
    CBO_CUDA(allow_dynamic_smem(prior_eval_kernel<PriorCfgA, false>, PriorCfgA::SMEM));
    CBO_CUDA(cudaMemsetAsync(d_ws, 0, kPriorWsHeader, st));
    PriorBases pb;
    pb.n = num_sets <= kMaxBases ? num_sets : 0;
    pb.base[0] = 0;
    for (int s = 0; s < kMaxBases; ++s)
        pb.base[s + 1] = pb.base[s] + (s < pb.n ? (int)prior_items(h_sets[s], split) : 0);
    kern<<<(unsigned)grid, PriorCfgA::NT, PriorCfgA::SMEM, st>>>(d_sets, num_sets, split, pb, (int)total,
                                                                 reinterpret_cast<int*>(ws), partials, scratch, slot);
    note_launch();
    CBO_CUDA(cudaGetLastError());
    if (partial) {
        prior_finalize_kernel<<<(unsigned)(tiles < 1024 ? tiles : 1024), CBO_PRIOR_TILE, 0, st>>>(d_sets, num_sets, split, partials);
        note_launch();
        CBO_CUDA(cudaGetLastError());
    }
    return 0;
}

}  // namespace cbo
