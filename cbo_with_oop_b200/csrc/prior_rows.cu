// K1c -- causal prior at the INTERVENTIONAL ROWS:  m_int[r] = u_r.w ,  v_int[r] = s2 + noise - u_r^T M u_r,
// evaluated in compensated (twice-the-working-precision) arithmetic.
//
// Replaces DoCalculus.update_do_function (reference DoCalculus.py:34-66) for the n_s training inputs of a set's GP:
// the values the reference feeds into Mapping.f / CausalRBF.K when it fits that GP (GaussianProcessFactory.py:63-73,
// causal_kernels.py:58-59).
//
// Why a second kernel beside the DMMA one (prior_eval.cu):
//  * accuracy.  u^T M u sums N^2 products of mixed sign (M carries Ky^-1); when the observational GP is confident,
//    s2 + noise - u^T M u cancels almost completely (shipped coral data: s2 = 20, v = 0.0126, sum of |terms| = 4.8e6,
//    i.e. a condition number of 4e8).  On the grid that costs 1e-8 of relative accuracy in v, harmless.  At the
//    interventional rows the error is AMPLIFIED by the per-set fit (the Gram contains sqrt(v_i v_j), condition numbers
//    up to 1e10 on the shipped data) and reaches 1e-6 in the posterior mean.  The reference does not have the problem:
//    GPy evaluates the variance as Kdiag - |L^-1 k|^2, a sum of squares.  Here every product is split exactly
//    (TwoProd, one DFMA) and every sum carries its rounding error along (TwoSum) -- the Dot2 scheme of Ogita, Rump and
//    Oishi -- so m_int and v_int are as accurate as if accumulated with a 106-bit significand and rounded once;
//  * shape.  There are at most 128 rows: the work is one pass over M (HBM-bound for the single row a post-intervention
//    trial appends: 8 N^2 / 2 bytes), not a GEMM.
//
// The pass over M is the shared one of m_triangle_pass.cuh, with grid z = set x row pass.  Thread n accumulates
// s_n[r] = sum_k M[n][k] u_r[k] for up to RMAX interventional rows r in registers, then the CTA reduces sum_n u_r[n] s_n[r]
// and writes one (q, m) double-double partial per row; prior_rows_finalize_kernel adds the partials in index order.
#include "m_triangle_pass.cuh"

namespace cbo {

constexpr int kRowsPartial = 4;    // doubles per (item, row): q_hi, q_lo, m_hi, m_lo
// interventional rows whose accumulators live in registers at once: 32 for a whole set (register-bound, 2 CTAs per SM, the
// arithmetic dominates), 4 for the row or two a post-intervention trial appends (6+ CTAs per SM: enough slabs in flight
// to stream M at HBM speed)
constexpr int kRowsWide = 32, kRowsNarrow = 4;

// error-free transformations; the intrinsics keep the compiler from contracting or re-associating them
__device__ __forceinline__ void two_sum(double a, double b, double& s, double& e) {
    s = __dadd_rn(a, b);
    const double bb = __dsub_rn(s, a);
    e = __dadd_rn(__dsub_rn(a, __dsub_rn(s, bb)), __dsub_rn(b, bb));
}
__device__ __forceinline__ void two_prod(double a, double b, double& p, double& e) {
    p = __dmul_rn(a, b);
    e = __fma_rn(a, b, -p);
}
// (s, c) += a * b, s the running sum, c the running sum of every rounding error
__device__ __forceinline__ void dot2_step(double a, double b, double& s, double& c) {
    double p, pe, t, te;
    two_prod(a, b, p, pe);
    two_sum(s, p, t, te);
    s = t;
    c = __dadd_rn(c, __dadd_rn(te, pe));
}
// (s, c) += (h, l)
__device__ __forceinline__ void dd_add(double h, double l, double& s, double& c) {
    double t, te;
    two_sum(s, h, t, te);
    s = t;
    c = __dadd_rn(c, __dadd_rn(te, l));
}

__host__ __device__ inline int rows_first(const cbo_set_desc& S) {
    return (S.int_row_begin > 0 && S.int_row_begin < S.n_int) ? S.int_row_begin : 0;
}

struct RowsShape { int passes, nJ, chunks, rmax; };   // grid extents shared by every set of a launch (maxima); rows per pass
__host__ __device__ inline size_t rows_partial_index(const RowsShape& sh, int set, int pass, int I, int c) {
    return ((((size_t)set * sh.passes + pass) * sh.nJ + I) * sh.chunks + c) * (size_t)(sh.rmax * kRowsPartial);
}

template <int RMAX>
__global__ void __launch_bounds__(kPassThreads)
prior_rows_kernel(const cbo_set_desc* __restrict__ sets, RowsShape sh, double* __restrict__ partials) {
    const int set = blockIdx.z / sh.passes, pass = blockIdx.z % sh.passes;
    const cbo_set_desc& S = sets[set];
    if (!computes_prior(S)) return;
    const int r0 = rows_first(S) + pass * RMAX;
    MPassItem it;
    if (!m_pass_item(S, it) || r0 >= S.n_int) return;
    const int R = S.n_int - r0 < RMAX ? S.n_int - r0 : RMAX;
    const int Npad = S.n_obs_pad, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double* __restrict__ U = S.u_int + (size_t)r0 * Npad;

    __shared__ double su[2][RMAX][kBK];                      // u_r[k] of the current / next slab
    __shared__ double sred[kPassThreads / 32][RMAX][kRowsPartial];

    double acc_s[RMAX], acc_c[RMAX];
#pragma unroll
    for (int r = 0; r < RMAX; ++r) acc_s[r] = acc_c[r] = 0.0;

    // this thread's share of a slab's u columns (R x 16 doubles over 128 threads)
    constexpr int UPT = (RMAX * kBK + kPassThreads - 1) / kPassThreads;
    double un[UPT];
    auto load_u = [&](int kt) {
#pragma unroll
        for (int x = 0; x < UPT; ++x) {
            const int i = tid + x * kPassThreads;
            un[x] = i < R * kBK ? U[(size_t)(i / kBK) * Npad + kt * kBK + (i % kBK)] : 0.0;
        }
    };
    auto store_u = [&](int buf) {
#pragma unroll
        for (int x = 0; x < UPT; ++x) {
            const int i = tid + x * kPassThreads;
            if (i < RMAX * kBK) su[buf][i / kBK][i % kBK] = un[x];
        }
    };
    // this thread's row of the slab, one k4-group (32 bytes; consecutive threads -> consecutive 32-byte units) at a time:
    // the group loop is NOT unrolled, so the fully unrolled body (RMAX rows x 4 products of ~10 instructions) stays
    // inside the instruction cache -- unrolled over all 16 columns it was 37 % "no instruction" stalls
    auto consume = [&](const double* slab, double scale, int cur) {
#pragma unroll 1
        for (int g = 0; g < kBK / 4; ++g) {
            const double2 a = *reinterpret_cast<const double2*>(slab + ((g * kMBlkRows + tid) << 2));
            const double2 b = *reinterpret_cast<const double2*>(slab + ((g * kMBlkRows + tid) << 2) + 2);
            const double mv[4] = {a.x * scale, a.y * scale, b.x * scale, b.y * scale};
#pragma unroll
            for (int r = 0; r < RMAX; ++r) {
                if (r < R) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) dot2_step(mv[k], su[cur][r][g * 4 + k], acc_s[r], acc_c[r]);
                }
            }
        }
    };
    m_pass_stream(it, S.M, Npad, load_u, store_u, consume);

    // q partial of row r: sum over the block's rows n of u_r[n] * s_n[r]; m partial (once per row block: the CTA that
    // owns the first slab of the diagonal block): sum_n u_r[n] w[n]
    const bool with_m = it.kt0 <= it.diag0 && it.diag0 < it.kt1;
    const int n = it.I * kMBlkRows + tid;
    const double wn = with_m ? S.w[n] : 0.0;
#pragma unroll
    for (int r = 0; r < RMAX; ++r) {
        double qh = 0.0, ql = 0.0, mh = 0.0, ml = 0.0;
        if (r < R) {
            const double ur = U[(size_t)r * Npad + n];
            two_prod(ur, acc_s[r], qh, ql);
            ql = __fma_rn(ur, acc_c[r], ql);
            if (with_m) two_prod(ur, wn, mh, ml);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {   // fixed butterfly: deterministic
            const double oh = __shfl_xor_sync(0xffffffffu, qh, o), ol = __shfl_xor_sync(0xffffffffu, ql, o);
            const double ph = __shfl_xor_sync(0xffffffffu, mh, o), pl = __shfl_xor_sync(0xffffffffu, ml, o);
            dd_add(oh, ol, qh, ql);
            dd_add(ph, pl, mh, ml);
        }
        if (lane == 0) { sred[warp][r][0] = qh, sred[warp][r][1] = ql, sred[warp][r][2] = mh, sred[warp][r][3] = ml; }
    }
    __syncthreads();
    if (tid < RMAX) {
        double qh = 0.0, ql = 0.0, mh = 0.0, ml = 0.0;
#pragma unroll
        for (int wq = 0; wq < kPassThreads / 32; ++wq) {
            dd_add(sred[wq][tid][0], sred[wq][tid][1], qh, ql);
            dd_add(sred[wq][tid][2], sred[wq][tid][3], mh, ml);
        }
        double* out = partials + rows_partial_index(sh, set, pass, it.I, it.c) + tid * kRowsPartial;
        out[0] = qh, out[1] = ql, out[2] = mh, out[3] = ml;
    }
}

// one CTA of 32 warps per (set, pass), 32 / rmax warps per row (1 for a whole set, 8 for the row or two a post-intervention
// trial appends: with one warp its 1580 partials at N = 1e4 were a 36 us chain of dependent loads): thread t of a row's
// warps adds the partials of items t, t + T, ... (a fixed assignment), a fixed butterfly combines the lanes and the row's
// first lane adds its warps' sums in warp order -- the order of the additions never depends on scheduling
__global__ void __launch_bounds__(32 * kRowsWide)
prior_rows_finalize_kernel(const cbo_set_desc* __restrict__ sets, RowsShape sh, const double* __restrict__ partials) {
    __shared__ double warp_sums[kRowsWide][4];
    const int set = blockIdx.x / sh.passes, pass = blockIdx.x % sh.passes;
    const cbo_set_desc& S = sets[set];
    const int lane = threadIdx.x, warp = threadIdx.y, wpr = kRowsWide / sh.rmax;     // warps per row
    const int row = warp / wpr, sub = warp - row * wpr;
    if (!computes_prior(S)) return;      // CTA-uniform
    const int r = rows_first(S) + pass * sh.rmax + row;
    double qh = 0.0, ql = 0.0, mh = 0.0, ml = 0.0;
    const int nJ = m_row_blocks(S);
    if (r < S.n_int) {                   // warp-uniform
        for (int e = sub * 32 + lane; e < nJ * sh.chunks; e += 32 * wpr) {
            const int I = e / sh.chunks, c = e - I * sh.chunks;
            if (!m_item_exists(I, c)) continue;
            const double* p = partials + rows_partial_index(sh, set, pass, I, c) + row * kRowsPartial;
            dd_add(p[0], p[1], qh, ql);
            dd_add(p[2], p[3], mh, ml);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double oh = __shfl_xor_sync(0xffffffffu, qh, o), ol = __shfl_xor_sync(0xffffffffu, ql, o);
            const double ph = __shfl_xor_sync(0xffffffffu, mh, o), pl = __shfl_xor_sync(0xffffffffu, ml, o);
            dd_add(oh, ol, qh, ql);
            dd_add(ph, pl, mh, ml);
        }
    }
    if (lane == 0) { warp_sums[warp][0] = qh; warp_sums[warp][1] = ql; warp_sums[warp][2] = mh; warp_sums[warp][3] = ml; }
    __syncthreads();
    if (lane == 0 && sub == 0 && r < S.n_int) {
        for (int w = 1; w < wpr; ++w) {
            dd_add(warp_sums[warp + w][0], warp_sums[warp + w][1], qh, ql);
            dd_add(warp_sums[warp + w][2], warp_sums[warp + w][3], mh, ml);
        }
        S.m_int[r] = mh + ml;
        S.v_int[r] = ((S.s2 + S.noise) - qh) - ql;
    }
}

static RowsShape rows_shape(const cbo_set_desc* h_sets, int num_sets) {
    const dim3 g = m_pass_grid(h_sets, num_sets, 1);
    RowsShape sh{0, (int)g.y, (int)g.x, kRowsWide};
    int rows_max = 0;
    for (int s = 0; s < num_sets; ++s) {
        const int rows = h_sets[s].n_int - rows_first(h_sets[s]);
        if (computes_prior(h_sets[s]) && rows > rows_max) rows_max = rows;
    }
    if (rows_max == 0) return sh;
    sh.rmax = rows_max <= kRowsNarrow ? kRowsNarrow : kRowsWide;
    sh.passes = (rows_max + sh.rmax - 1) / sh.rmax;
    return sh;
}

// workspace the rows kernel needs for `num_sets` sets at the row capacity (every interventional row, CBO_MAX_NINT at most)
size_t prior_rows_workspace_bytes(const cbo_set_desc* h_sets, int num_sets) {
    RowsShape sh = rows_shape(h_sets, num_sets);
    if (sh.passes == 0) return 0;
    sh.rmax = kRowsWide;
    sh.passes = (CBO_MAX_NINT + kRowsWide - 1) / kRowsWide;
    return rows_partial_index(sh, num_sets, 0, 0, 0) * sizeof(double);
}

int prior_rows_impl(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, void* d_ws, size_t ws_bytes,
                    size_t ws_offset, cudaStream_t st) {
    const RowsShape sh = rows_shape(h_sets, num_sets);
    if (sh.passes == 0) return 0;
    const size_t need = rows_partial_index(sh, num_sets, 0, 0, 0) * sizeof(double);
    CBO_REQUIRE(d_ws != nullptr && ws_bytes >= ws_offset + need,
                "cbo_prior_eval: workspace of %zu bytes is too small for the interventional rows (%zu needed); see "
                "cbo_prior_workspace_bytes", ws_bytes, ws_offset + need);
    double* partials = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(d_ws) + ws_offset);
    const dim3 grid(sh.chunks, sh.nJ, num_sets * sh.passes);
    const auto kernel = sh.rmax == kRowsNarrow ? prior_rows_kernel<kRowsNarrow> : prior_rows_kernel<kRowsWide>;
    if (int rc = m_pass_prepare(kernel, grid, "cbo_prior_eval")) return rc;
    kernel<<<grid, kPassThreads, kPassRingBytes, st>>>(d_sets, sh, partials);
    note_launch();
    CBO_CUDA(cudaGetLastError());
    prior_rows_finalize_kernel<<<num_sets * sh.passes, dim3(32, kRowsWide), 0, st>>>(d_sets, sh, partials);
    note_launch();
    CBO_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace cbo
