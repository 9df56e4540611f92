// The pass over the lower block triangle of the prior matrix M shared by K1c (prior_rows.cu, the prior at a set's
// interventional rows) and K7's prior-gradient pass (refine.cu).  Grid = (k chunk c, row block I, set x what the kernel
// repeats per set).  A CTA of 128 threads owns the rows of block I (thread n: row I * 128 + n) and chunk c: <= kPassSlabs of
// the block's 16-deep column slabs inside the triangle; those left of the diagonal block appear twice in u^T M u and are
// consumed with scale 2 (exact).  Each (I, c) item writes its own partials (no atomics); reducers add them in index order.
// M arrives by TMA bulk copies (one contiguous 16 KB slab of K1a's blocked layout each) in a kPassStages-deep ring in the
// kernel's dynamic shared memory (kPassRingBytes), issued ahead by thread 0: the bytes in flight do not depend on the
// register budget, which is what an HBM-bound pass needs.
#pragma once
#include "dmma_tile.cuh"

namespace cbo {

constexpr int kPassThreads = kMBlkRows;                 // thread n owns row n of a row block
constexpr int kSlabsPerBlock = kMBlkRows / kBK;         // 16-deep slabs per 128-row block of M
constexpr int kPassSlabs = 32;                          // slabs per CTA
constexpr int kPassStages = 3;                          // 16 KB slabs of M in flight per CTA
constexpr size_t kPassRingBytes = (size_t)kPassStages * kMBlkDoubles * sizeof(double);

__host__ __device__ inline int m_row_blocks(const cbo_set_desc& S) { return (S.n_obs + kMBlkRows - 1) / kMBlkRows; }
__host__ __device__ inline int m_chunks(const cbo_set_desc& S) { return (m_row_blocks(S) * kSlabsPerBlock + kPassSlabs - 1) / kPassSlabs; }
// does chunk c of row block I (< m_row_blocks) hold a slab of the triangle?  If not, nothing was written to its slots.
__host__ __device__ inline bool m_item_exists(int I, int c) { return c * kPassSlabs < (I + 1) * kSlabsPerBlock; }

struct MPassItem { int I, c, kt0, kt1, diag0, nsl; };    // diag0: first slab of the diagonal block; nsl = kt1 - kt0

// this CTA's item (blockIdx.x = chunk, blockIdx.y = row block); false: it has no work for set S
__device__ __forceinline__ bool m_pass_item(const cbo_set_desc& S, MPassItem& it) {
    const int I = blockIdx.y, c = blockIdx.x, nslab = (I + 1) * kSlabsPerBlock, kt0 = c * kPassSlabs;
    const int kt1 = kt0 + kPassSlabs < nslab ? kt0 + kPassSlabs : nslab;
    it = MPassItem{I, c, kt0, kt1, I * kSlabsPerBlock, kt1 - kt0};
    return I < m_row_blocks(S) && m_item_exists(I, c);
}

// Streams the item's slabs of M (row pitch Npad) through the ring.  The kernel's own operands of a slab (u_r in K1c, u and
// a_k of 8 points in K7) are double-buffered in shared memory: fetch(kt) loads those of slab kt into registers (for the
// next slab, before the wait), store(buf) writes them into buffer buf, and consume(slab, scale, cur) consumes one slab
// (fragment order) with its operands in buffer cur.  Every thread calls it; on return every buffer has been read.
template <class Fetch, class Store, class Consume>
__device__ __forceinline__ void m_pass_stream(const MPassItem& it, const double* M, int Npad, Fetch&& fetch,
                                              Store&& store, Consume&& consume) {
    extern __shared__ __align__(128) unsigned char ring_raw[];
    double* sM = reinterpret_cast<double*>(ring_raw);     // [kPassStages][128 x 16 slab, fragment order]
    __shared__ uint64_t full[kPassStages];
    const int tid = threadIdx.x;
    auto issue = [&](int idx) {
        const int st = idx % kPassStages;
        mbar_arrive_expect_tx(&full[st], (unsigned)(kMBlkDoubles * sizeof(double)));
        bulk_g2s(sM + (size_t)st * kMBlkDoubles, M + mblk_base(it.I, it.kt0 + idx, Npad), (unsigned)(kMBlkDoubles * sizeof(double)), &full[st]);
    };
    if (tid == 0) {
        for (int st = 0; st < kPassStages; ++st) mbar_init(&full[st], 1);
        mbar_fence_init();
    }
    __syncthreads();
    if (tid == 0)
        for (int idx = 0; idx < kPassStages && idx < it.nsl; ++idx) issue(idx);
    fetch(it.kt0);
    store(0);
    __syncthreads();
#pragma unroll 1
    for (int idx = 0; idx < it.nsl; ++idx) {
        const int kt = it.kt0 + idx, cur = idx & 1, st = idx % kPassStages;
        const bool more = idx + 1 < it.nsl;
        if (more) fetch(kt + 1);            // next slab's operands in flight while this slab is consumed
        mbar_wait(&full[st], (unsigned)(idx / kPassStages) & 1u);
        consume(sM + (size_t)st * kMBlkDoubles, kt < it.diag0 ? 2.0 : 1.0, cur);
        if (more) store(cur ^ 1);           // the other buffer was last read one iteration ago, before that iteration's barrier
        __syncthreads();                    // every thread has read ring stage st and buffer cur
        if (tid == 0 && idx + kPassStages < it.nsl) issue(idx + kPassStages);
    }
}

// ---- host ----------------------------------------------------------------------------------------------------------------
// Grid of a pass: x = the most chunks of a set, y = the most row blocks, z = num_sets * per_set, over the sets that compute
// a prior (x == y == 0 when none does).  CTAs past a smaller set's extent find no item.
inline dim3 m_pass_grid(const cbo_set_desc* h_sets, int num_sets, int per_set) {
    dim3 g(0, 0, (unsigned)(num_sets * per_set));
    for (int s = 0; s < num_sets; ++s) {
        if (!computes_prior(h_sets[s])) continue;
        if ((unsigned)m_chunks(h_sets[s]) > g.x) g.x = m_chunks(h_sets[s]);
        if ((unsigned)m_row_blocks(h_sets[s]) > g.y) g.y = m_row_blocks(h_sets[s]);
    }
    return g;
}

// Checks the launch limits of `grid` and opts `kernel` into the ring's dynamic shared memory.
template <class K>
inline int m_pass_prepare(K kernel, dim3 grid, const char* who) {
    CBO_REQUIRE(grid.y <= 65535 && grid.z <= 65535, "%s: too many sets or rows for one launch", who);
    CBO_CUDA(allow_dynamic_smem(kernel, kPassRingBytes));
    return 0;
}

}  // namespace cbo
