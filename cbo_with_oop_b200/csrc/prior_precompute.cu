// K1a -- fold the Monte-Carlo average of the causal prior into (w, M), once per observation.
//
// The reference averages observational-GP predictions over the conditioning samples for EVERY candidate
// (DoCalculus.py:50-66 -> compute_do :68-78).  With P_ji = prod_{k not intervened} exp(-.5 ((C_ik - X_jk)/l_k)^2)
// (train row j, conditioning sample i) that average is a fixed linear / quadratic form in u(x):
//     pbar = mean_i P           w = s2 * alpha * pbar
//     M    = s2^2 * Kyinv o (P P^T / S_mc)
// so it is computed once here (SURVEY.md App. A.5).  Two stream-ordered stages, each set read from the device descriptors:
//   pgen : P (N x S) with one exp per element, coalesced along i, deterministic row sums -> pbar, w
//   syrk : lower block triangle of P P^T on the FP64 tensor pipe (DMMA), fused Hadamard with Kyinv,
//          mirrored store so M is a full symmetric matrix, written in the blocked fragment-order layout of
//          dmma_tile.cuh (mblk_off) that K1b streams with one TMA bulk copy per pipeline stage.
// Roofline: FP64 pipe, 2 N^2 S_mc dense-counted flops (N^2 S_mc executed).  No conditioning columns (c == 0)
// degenerates to M = s2^2 Kyinv.
#include "dmma_tma_tile.cuh"

namespace cbo {

// One CTA per row j of P (blockIdx.x; the grid covers every set's n_obs_pad) of set blockIdx.y.
__global__ void __launch_bounds__(256)
pgen_kernel(const cbo_set_desc* __restrict__ sets) {
    __shared__ double red[8];
    const cbo_set_desc& S = sets[blockIdx.y];
    const int j = blockIdx.x;
    if (!computes_prior(S) || S.c == 0 || j >= S.n_obs_pad) return;
    const int c = S.c, n_obs = S.n_obs, n_mc = S.n_mc, n_mc_pad = S.n_mc_pad;
    double* __restrict__ row = S.P + (size_t)j * n_mc_pad;
    const bool live = j < n_obs;
    double il[CBO_MAX_C], xj[CBO_MAX_C];
#pragma unroll
    for (int k = 0; k < CBO_MAX_C; ++k) {
        il[k] = k < c ? 1.0 / S.ls_cond[k] : 0.0;
        xj[k] = (live && k < c) ? S.x_obs_cond[(size_t)k * n_obs + j] : 0.0;
    }
    double sum = 0.0;
    for (int i = threadIdx.x; i < n_mc_pad; i += 256) {
        double val = 0.0;
        if (live && i < n_mc) {
            double r2 = 0.0;
#pragma unroll
            for (int k = 0; k < CBO_MAX_C; ++k) {
                if (k < c) {
                    const double t = (S.mc_cond[(size_t)k * n_mc + i] - xj[k]) * il[k];
                    r2 += t * t;
                }
            }
            val = exp(-0.5 * r2);
        }
        row[i] = val;
        sum += val;
    }
    sum = warp_sum(sum);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
#pragma unroll
        for (int x = 0; x < 8; ++x) t += red[x];
        const double pb = live ? t / (double)n_mc : 0.0;
        S.pbar[j] = pb;
        S.w[j] = live ? S.s2 * S.alpha_obs[j] * pb : 0.0;
    }
}

// c == 0: P == 1, pbar == 1, Q == 1.  Row j = blockIdx.y of the blockIdx.z-th set without conditioning columns (the grid
// covers those sets only: they are usually few among many).
__global__ void __launch_bounds__(256)
nocond_kernel(const cbo_set_desc* __restrict__ sets, int num_sets) {
    int s = 0;
    for (int z = blockIdx.z; s < num_sets; ++s) {
        if (computes_prior(sets[s]) && sets[s].c == 0 && z-- == 0) break;
    }
    if (s >= num_sets) return;
    const cbo_set_desc& S = sets[s];
    const int j = blockIdx.y, n_obs = S.n_obs, n_obs_pad = S.n_obs_pad;
    if (j >= n_obs_pad) return;
    const double s2 = S.s2;
    const double* __restrict__ kyinv = S.kyinv;
    double* __restrict__ M = S.M;
    const bool lj = j < n_obs;
    for (int k = blockIdx.x * 256 + threadIdx.x; k < n_obs_pad; k += gridDim.x * 256) {
        M[mblk_off(j, k, n_obs_pad)] = (lj && k < n_obs) ? (s2 * s2) * kyinv[(size_t)j * n_obs + k] : 0.0;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        S.pbar[j] = lj ? 1.0 : 0.0;
        S.w[j] = lj ? s2 * S.alpha_obs[j] : 0.0;
    }
}

// The epilogue of both syrk pipelines for the accumulator pair (r, cidx), (r, cidx + 1) of P P^T: M = coef * Kyinv o Q, zero
// outside the live N x N corner, mirrored into the upper triangle for a tile below the diagonal.
__device__ __forceinline__ void store_m_pair(double* __restrict__ M, const double* __restrict__ kyinv, double coef, int n_obs,
                                             int n_obs_pad, int r, int cidx, bool mirror, double a0, double a1) {
    double v0 = 0.0, v1 = 0.0;
    if (r < n_obs) {
        if (cidx < n_obs) v0 = coef * kyinv[(size_t)r * n_obs + cidx] * a0;
        if (cidx + 1 < n_obs) v1 = coef * kyinv[(size_t)r * n_obs + cidx + 1] * a1;
    }
    *reinterpret_cast<double2*>(M + mblk_off(r, cidx, n_obs_pad)) = make_double2(v0, v1);
    if (mirror) {
        M[mblk_off(cidx, r, n_obs_pad)] = v0;
        M[mblk_off(cidx + 1, r, n_obs_pad)] = v1;
    }
}

// One CTA per (set, lower-triangle tile), tiles in set order, on the cp.async mainloop of dmma_tile.cuh.
template <int WM, int WN, int MA, int NB, int STAGES>
__global__ void __launch_bounds__(WM * WN * 32, 1)
syrk_kernel(const cbo_set_desc* __restrict__ sets, int num_sets) {
    constexpr int BM = WM * MA * 8, BN = WN * NB * 8;
    static_assert(BM == BN && BM == CBO_NPAD, "square tiles of CBO_NPAD");
    constexpr int TILE = BM * kBK;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* sA = reinterpret_cast<double*>(smem_raw);
    double* sB = sA + STAGES * TILE;
    // (set, lower-triangle tile) of this CTA: sets with conditioning columns only
    int s = 0, t = blockIdx.x;
    for (; s < num_sets; ++s) {
        if (!computes_prior(sets[s]) || sets[s].c == 0) continue;
        const int nT = sets[s].n_obs_pad / CBO_NPAD, cnt = nT * (nT + 1) / 2;
        if (t < cnt) break;
        t -= cnt;
    }
    if (s >= num_sets) return;
    const cbo_set_desc& S = sets[s];
    const double* __restrict__ P = S.P;
    const double* __restrict__ kyinv = S.kyinv;
    double* __restrict__ M = S.M;
    const int n_mc_pad = S.n_mc_pad, n_obs = S.n_obs, n_obs_pad = S.n_obs_pad;
    const double coef = (S.s2 * S.s2) / (double)S.n_mc;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = warp / WN, wn = warp % WN;
    const int row0 = wm * MA * 8, col0 = wn * NB * 8;
    int bi, bj;
    tri_tile(t, bi, bj);
    double acc[MA][NB][2];
#pragma unroll
    for (int mi = 0; mi < MA; ++mi)
#pragma unroll
        for (int ni = 0; ni < NB; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
    abt_mainloop<WM, WN, MA, NB, STAGES>(P + (size_t)bi * BM * n_mc_pad, n_mc_pad, P + (size_t)bj * BN * n_mc_pad, n_mc_pad,
                                         n_mc_pad / kBK, sA, sB, acc, tid);
#pragma unroll
    for (int mi = 0; mi < MA; ++mi) {
        const int r = bi * BM + row0 + mi * 8 + (lane >> 2);
#pragma unroll
        for (int ni = 0; ni < NB; ++ni)
            store_m_pair(M, kyinv, coef, n_obs, n_obs_pad, r, bj * BN + col0 + ni * 8 + (lane & 3) * 2, bi != bj, acc[mi][ni][0],
                         acc[mi][ni][1]);
    }
}

// The same product for a set whose block triangle covers the GPU (n_obs_pad (n_obs_pad / 128 + 1) / 256 tiles >= SMs): persistent
// CTAs on the tensor-map TMA pipeline of dmma_tma_tile.cuh (P is a plain row-major matrix), same epilogue.
struct PriorSyrkPlan {
    const double* kyinv;
    double* M;
    double coef;
    int n_obs, n_obs_pad, nT, nk;
    __device__ int count() const { return nT * (nT + 1) / 2; }
    __device__ TileJob job(int t) const {
        int bi, bj;
        tri_tile(t, bi, bj);
        return TileJob{bi * CBO_NPAD, bj * CBO_NPAD, 0, nk, bi, bj};
    }
    __device__ void store(const TileJob& j, const double (&acc)[8][4][2], int tid) const {
        tma_for_each_acc(acc, tid, [&](int rr, int cc, double a0, double a1) {
            store_m_pair(M, kyinv, coef, n_obs, n_obs_pad, j.ti * CBO_NPAD + rr, j.tj * CBO_NPAD + cc, j.ti != j.tj, a0, a1);
        });
    }
};

// Does set s (with conditioning columns) need launches of its own?  Yes when its block triangle fills the GPU (it takes the
// TMA pipeline) or when its P scratch overlaps another set's (the two must run one after the other).
static bool own_launches(const cbo_set_desc* h_sets, int num_sets, int s, int sms) {
    const cbo_set_desc& S = h_sets[s];
    const int nT = S.n_obs_pad / CBO_NPAD;
    if (nT * (nT + 1) / 2 >= sms) return true;
    const double* e0 = S.P + (size_t)S.n_obs_pad * S.n_mc_pad;
    for (int t = 0; t < num_sets; ++t) {
        const cbo_set_desc& T = h_sets[t];
        if (t == s || !computes_prior(T) || T.c == 0) continue;
        if (S.P < T.P + (size_t)T.n_obs_pad * T.n_mc_pad && T.P < e0) return true;
    }
    return false;
}

int prior_precompute_impl(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, cudaStream_t st) {
    constexpr int STAGES = 4;
    constexpr size_t SMEM = (size_t)STAGES * 2 * CBO_NPAD * kBK * sizeof(double);
    auto syrk = syrk_kernel<2, 4, 8, 4, STAGES>;
    CBO_CUDA(allow_dynamic_smem(syrk, SMEM));
    int dev = 0, sms = 0;
    CBO_CUDA(cudaGetDevice(&dev));
    CBO_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    int nocond = 0, npad_nocond = 0;
    for (int s = 0; s < num_sets; ++s) {
        const cbo_set_desc& S = h_sets[s];
        if (!computes_prior(S)) continue;
        CBO_REQUIRE(S.kyinv && S.alpha_obs && S.M && S.w && S.pbar, "cbo_prior_precompute: set %d has a NULL pointer", s);
        if (S.c == 0) {
            ++nocond;
            if (S.n_obs_pad > npad_nocond) npad_nocond = S.n_obs_pad;
            continue;
        }
        CBO_REQUIRE(S.P && S.x_obs_cond && S.mc_cond, "cbo_prior_precompute: set %d has a NULL P/x_obs_cond/mc_cond", s);
    }
    if (nocond > 0) {
        const int kx = (npad_nocond + 255) / 256;       // CTAs per row, up to 8
        nocond_kernel<<<dim3(kx < 8 ? kx : 8, npad_nocond, nocond), 256, 0, st>>>(d_sets, num_sets);
        note_launch();
        CBO_CUDA(cudaGetLastError());
    }
    // pgen -> syrk on sets [first, first + count); the kernels skip the sets without conditioning columns
    auto pgen_launch = [&](int first, int count, int npad) -> int {
        pgen_kernel<<<dim3(npad, count), 256, 0, st>>>(d_sets + first);
        note_launch();
        CBO_CUDA(cudaGetLastError());
        return 0;
    };
    auto syrk_launch = [&](int first, int count, int tiles) -> int {
        syrk<<<tiles, 256, SMEM, st>>>(d_sets + first, count);
        note_launch();
        CBO_CUDA(cudaGetLastError());
        return 0;
    };
    // A run of sets that need no launches of their own shares one launch per stage (the reference's shipped sizes are 25
    // sets of N = 100..200: per-set launches would cost more than the work).  The others run one after the other.
    int first = -1, npad = 0, tiles = 0;
    for (int s = 0; s <= num_sets; ++s) {
        const bool cond = s < num_sets && computes_prior(h_sets[s]) && h_sets[s].c > 0;
        const bool own = cond && own_launches(h_sets, num_sets, s, sms);
        if (first >= 0 && (own || s == num_sets)) {
            if (int rc = pgen_launch(first, s - first, npad)) return rc;
            if (int rc = syrk_launch(first, s - first, tiles)) return rc;
            first = -1, npad = tiles = 0;
        }
        if (!cond) continue;
        const cbo_set_desc& S = h_sets[s];
        const int nT = S.n_obs_pad / CBO_NPAD, t = nT * (nT + 1) / 2;
        if (!own) {
            if (first < 0) first = s;
            if (S.n_obs_pad > npad) npad = S.n_obs_pad;
            tiles += t;
            continue;
        }
        if (int rc = pgen_launch(s, 1, S.n_obs_pad)) return rc;
        if (t < sms) {
            if (int rc = syrk_launch(s, 1, t)) return rc;
            continue;
        }
        CUtensorMap mapP;
        if (make_f64_rowmajor_map(&mapP, S.P, S.n_obs_pad, S.n_mc_pad, S.n_mc_pad)) return -1;
        CBO_CUDA(launch_tma_tiles(mapP, mapP, PriorSyrkPlan{S.kyinv, S.M, (S.s2 * S.s2) / (double)S.n_mc, S.n_obs, S.n_obs_pad, nT,
                                                           S.n_mc_pad / kBK}, t, sms, st));
    }
    return 0;
}

}  // namespace cbo
