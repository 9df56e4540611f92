// K7 -- value and gradient of acq(x) = EI(x) / cost(x) at arbitrary points, and a projected quasi-Newton ascent of acq
// that refines each exploration set's grid maximum inside the set's interventional box.
//
// Replaces the reference's continuous search: CausalGradientAcquisitionOptimizer's L-BFGS polish of the best anchor
// (causal_optimizer.py:52-62) and the gradients it consumes (causal_acquisition_functions.py:45-67).
//
// Arithmetic (x in R^d, d <= 4; the observational GP has N rows X_.j and intervened lengthscales l_k):
//   causal prior    u_j = prod_k exp(-.5 ((x_k - X_kj) / l_k)^2),  m = u.w,  v = s2 + noise - u^T M u
//                   a_kj = u_j (x_k - X_kj) / l_k^2,  dm/dx_k = -sum_j a_kj w_j,  dv/dx_k = 2 a_k^T M u
//                   (each sum is accumulated with the weights a_kj themselves: no x_k u^T M u - sum_j X_kj ... cancellation)
//   per-set GP      e_i = s2 exp(-.5 |x - x_i|^2 / l^2),  k*_i = e_i + sv_i sqrt(v) (non-causal: e_i, m = v = 0)
//                   dk*_i = -e_i (x - x_i) / l^2 + sv_i dv / (2 sqrt v)     ((s2, l) = hyper, (1, 1) when NULL)
//                   mu = m + k*.alpha,  var = (s2 + v) - |L^-1 k*|^2 + noise   (k*, var, EI and cost: surrogate.cuh)
//                   dmu = dm + sum_i alpha_i dk*_i,  dvar = dv - 2 beta^T dk*,  beta = L^-T L^-1 k*
//   acquisition     u = (best - mu) / sd,  ei = sign sd (u Phi + phi),  dei = -sign Phi dmu + sign phi dvar / (2 sd)
//                   c = cost_fix + cost_variable sum |x_k|,  acq = ei / c,  dacq = (dei - acq dc) / c
//
// Prior-gradient pass (refine_prior_kernel): the model is K1c (prior_rows.cu).  A CTA owns the 128 rows n of a row block
// of M and a run of <= kRefSlabs of the block's 16-deep column slabs of M's lower block triangle, streamed by TMA bulk
// copies through a 3-stage ring.  For each of the 8 points of a set, thread n accumulates
//   S_u[n] = sum_k sc M_nk u_k  and  S_a,i[n] = sum_k sc M_nk a_ik      (sc = 2 left of the diagonal block, 1 inside it)
// and the CTA reduces  q = sum_n u_n S_u[n],  dv_i = sum_n (a_in S_u[n] + u_n S_a,i[n])  (the symmetric form of 2 a_i^T M u
// over the lower block triangle) and, once per row block, u.w and a_i.w.  That is 1 + d FMAs per element of M and point;
// the u / a columns of the current slab are built in shared memory from x_obs_int (no per-point table in HBM).  Partials
// go to fixed slots of the workspace and are added in index order by the step kernel: no atomics, and the slots of a set
// depend on that set alone.
//
// Step kernel (refine_step_kernel): one CTA per set, one warp per trial point (posterior by column-oriented substitutions
// with L in shared memory), then thread 0 takes one projected quasi-Newton step on -acq: BFGS on <= 4 variables (update
// skipped when s^T y <= 0), an active set for coordinates pinned at a bound, and a parallel backtracking line search --
// the 8 trial points of the next pass are clamp(x + 2^-j p), j = 0..7, accepted by Armijo's rule.  The first direction is
// the gradient scaled so that its largest move is one grid spacing.
#include <float.h>
#include "dmma_tile.cuh"
#include "surrogate.cuh"

namespace cbo {

constexpr int kRefB = 8;                       // trial points per set and pass
constexpr int kRefSlabs = 32;                  // 16-deep slabs of M per CTA of the prior pass
constexpr int kRefStages = 3;                  // 16 KB slabs in flight per CTA
constexpr int kRefThreads = kMBlkRows;         // prior pass: thread n owns row n of a row block
constexpr int kRefPF = 2 + 2 * CBO_MAX_D;      // partial per (item, point): m, q, a.w [4], dv [4]
constexpr int kStepThreads = 32 * kRefB;       // step / gradient kernels: one warp per point
constexpr size_t kRefRingBytes = (size_t)kRefStages * kMBlkDoubles * sizeof(double);
constexpr double kArmijo = 1e-4;

struct RefineState {                           // one per set, in the workspace
    double x[CBO_MAX_D], g[CBO_MAX_D], p[CBO_MAX_D];
    double H[CBO_MAX_D * CBO_MAX_D];           // inverse-Hessian approximation of -acq
    double lo[CBO_MAX_D], hi[CBO_MAX_D], h[CBO_MAX_D];
    double x0[CBO_MAX_D];
    double xt[kRefB][CBO_MAX_D];               // points of the next prior pass
    double f, f0;
    long long part_base;                       // first double of the set's partials
    int32_t running, iter, status, ntrial, qn, max_iter;
};

__host__ __device__ inline int ref_nJ(const cbo_set_desc& S) { return (S.n_obs + kMBlkRows - 1) / kMBlkRows; }
__host__ __device__ inline int ref_chunks(const cbo_set_desc& S) { return (ref_nJ(S) * (kMBlkRows / kBK) + kRefSlabs - 1) / kRefSlabs; }
// partial slots of one batch of 8 points of a set
__host__ __device__ inline long long ref_items(const cbo_set_desc& S) {
    return computes_prior(S) ? (long long)ref_nJ(S) * ref_chunks(S) : 0;
}
constexpr long long kRefItemDoubles = (long long)kRefB * kRefPF;
constexpr size_t kRefHeader = 256;             // [0]: sets still running (int32)
inline size_t ref_state_bytes(int num_sets) { return ((size_t)num_sets * sizeof(RefineState) + 255) / 256 * 256; }

// ---- prior-gradient pass -------------------------------------------------------------------------------------------------
struct PassArgs {
    const double* pts;       // point q of set s, batch b: pts[s * set_stride + (b * kRefB + q) * pt_stride + k]
    long long set_stride;
    int pt_stride, npts, nbatch;
    const RefineState* state;   // refine: the running flags and partial bases; NULL: one set, partials at 0
    double* partials;
};

template <int D>
__global__ void __launch_bounds__(kRefThreads)
refine_prior_kernel(const cbo_set_desc* __restrict__ sets, PassArgs a) {
    const int set = blockIdx.z / a.nbatch, batch = blockIdx.z % a.nbatch;
    const cbo_set_desc& S = sets[set];
    if (S.d != D || !computes_prior(S)) return;
    if (a.state && !a.state[set].running) return;
    const int nJ = ref_nJ(S), chunks = ref_chunks(S);
    const int I = blockIdx.y, c = blockIdx.x;
    const int nslab = (I + 1) * (kMBlkRows / kBK), kt0 = c * kRefSlabs;
    if (I >= nJ || c >= chunks || kt0 >= nslab) return;
    const int kt1 = kt0 + kRefSlabs < nslab ? kt0 + kRefSlabs : nslab;
    const int nsl = kt1 - kt0, diag0 = I * (kMBlkRows / kBK);
    const int N = S.n_obs, Npad = S.n_obs_pad, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    extern __shared__ __align__(128) unsigned char ring_raw[];
    double* sM = reinterpret_cast<double*>(ring_raw);
    __shared__ uint64_t full[kRefStages];
    __shared__ __align__(16) double tab[2][kRefB][1 + D][kBK];      // u (row 0) and a_k (rows 1..D) of the slab's columns
    __shared__ double sx[kRefB][D];
    __shared__ double sred[kRefThreads / 32][kRefB][2 + 2 * D];
    double il[D];
#pragma unroll
    for (int k = 0; k < D; ++k) il[k] = 1.0 / S.ls_int[k];

    if (tid < kRefB * D) {
        const int q = tid / D, k = tid % D;
        int pi = batch * kRefB + q;
        if (pi >= a.npts) pi = a.npts - 1;          // padding points repeat the last one (their partials are not read)
        sx[q][k] = a.pts[a.set_stride * set + (long long)pi * a.pt_stride + k];
    }
    if (tid == 0) {
        for (int st = 0; st < kRefStages; ++st) mbar_init(&full[st], 1);
        mbar_fence_init();
    }
    __syncthreads();
    auto issue = [&](int idx) {
        const int st = idx % kRefStages;
        mbar_arrive_expect_tx(&full[st], (unsigned)(kMBlkDoubles * sizeof(double)));
        bulk_g2s(sM + (size_t)st * kMBlkDoubles, S.M + mblk_base(I, kt0 + idx, Npad), (unsigned)(kMBlkDoubles * sizeof(double)), &full[st]);
    };
    if (tid == 0)
        for (int idx = 0; idx < kRefStages && idx < nsl; ++idx) issue(idx);

    // table entry of this thread: point tid / 16, column tid % 16 of slab kt
    const int tq = tid >> 4, tc = tid & 15;
    auto entry = [&](int kt, double (&e)[1 + D]) {
        const int col = kt * kBK + tc;
        if (col < N) {
            double r2 = 0.0, z[D];
#pragma unroll
            for (int k = 0; k < D; ++k) {
                z[k] = (sx[tq][k] - S.x_obs_int[(size_t)k * N + col]) * il[k];
                r2 = fma(z[k], z[k], r2);
            }
            e[0] = exp(-0.5 * r2);
#pragma unroll
            for (int k = 0; k < D; ++k) e[1 + k] = e[0] * z[k] * il[k];
        } else {
#pragma unroll
            for (int k = 0; k <= D; ++k) e[k] = 0.0;
        }
    };
    auto store = [&](int buf, const double (&e)[1 + D]) {
#pragma unroll
        for (int k = 0; k <= D; ++k) tab[buf][tq][k][tc] = e[k];
    };
    double acc[kRefB][1 + D];
#pragma unroll
    for (int q = 0; q < kRefB; ++q)
#pragma unroll
        for (int k = 0; k <= D; ++k) acc[q][k] = 0.0;
    double en[1 + D];
    entry(kt0, en);
    store(0, en);
    __syncthreads();
#pragma unroll 1
    for (int idx = 0; idx < nsl; ++idx) {
        const int kt = kt0 + idx, cur = idx & 1, st = idx % kRefStages;
        const bool more = idx + 1 < nsl;
        if (more) entry(kt + 1, en);
        mbar_wait(&full[st], (unsigned)(idx / kRefStages) & 1u);
        const double* slab = sM + (size_t)st * kMBlkDoubles;
        const double scale = kt < diag0 ? 2.0 : 1.0;
#pragma unroll 1
        for (int g = 0; g < kBK / 4; ++g) {
            const double2 m01 = *reinterpret_cast<const double2*>(slab + ((g * kMBlkRows + tid) << 2));
            const double2 m23 = *reinterpret_cast<const double2*>(slab + ((g * kMBlkRows + tid) << 2) + 2);
            const double m0 = m01.x * scale, m1 = m01.y * scale, m2 = m23.x * scale, m3 = m23.y * scale;
#pragma unroll
            for (int q = 0; q < kRefB; ++q) {
#pragma unroll
                for (int k = 0; k <= D; ++k) {
                    const double2 t01 = *reinterpret_cast<const double2*>(&tab[cur][q][k][g * 4]);
                    const double2 t23 = *reinterpret_cast<const double2*>(&tab[cur][q][k][g * 4 + 2]);
                    double s = acc[q][k];
                    s = fma(m0, t01.x, s);
                    s = fma(m1, t01.y, s);
                    s = fma(m2, t23.x, s);
                    s = fma(m3, t23.y, s);
                    acc[q][k] = s;
                }
            }
        }
        if (more) store(cur ^ 1, en);
        __syncthreads();
        if (tid == 0 && idx + kRefStages < nsl) issue(idx + kRefStages);
    }

    // row n's share: q = u_n S_u, dv_i = a_in S_u + u_n S_a,i; once per row block (c == 0): m = u_n w_n, a_in w_n
    const int n = I * kMBlkRows + tid;
    const bool with_m = c == 0;
    const double wn = (with_m && n < N) ? S.w[n] : 0.0;
#pragma unroll
    for (int q = 0; q < kRefB; ++q) {
        double un = 0.0, an[D];
#pragma unroll
        for (int k = 0; k < D; ++k) an[k] = 0.0;
        if (n < N) {
            double r2 = 0.0, z[D];
#pragma unroll
            for (int k = 0; k < D; ++k) {
                z[k] = (sx[q][k] - S.x_obs_int[(size_t)k * N + n]) * il[k];
                r2 = fma(z[k], z[k], r2);
            }
            un = exp(-0.5 * r2);
#pragma unroll
            for (int k = 0; k < D; ++k) an[k] = un * z[k] * il[k];
        }
        double v[2 + 2 * D];
        v[0] = un * wn;
        v[1] = un * acc[q][0];
#pragma unroll
        for (int k = 0; k < D; ++k) {
            v[2 + k] = an[k] * wn;
            v[2 + D + k] = fma(an[k], acc[q][0], un * acc[q][1 + k]);
        }
#pragma unroll
        for (int e = 0; e < 2 + 2 * D; ++e) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v[e] += __shfl_xor_sync(0xffffffffu, v[e], o);   // fixed butterfly
            if (lane == 0) sred[warp][q][e] = v[e];
        }
    }
    __syncthreads();
    double* out = a.partials + (a.state ? a.state[set].part_base : 0) +
                  (((long long)batch * nJ + I) * chunks + c) * kRefItemDoubles;
    for (int e = tid; e < kRefB * kRefPF; e += kRefThreads) {
        const int q = e / kRefPF, f = e % kRefPF;
        // slot layout per point: m, q, a.w[CBO_MAX_D], dv[CBO_MAX_D]
        double s = 0.0;
        int src = -1;
        if (f < 2) src = f;
        else if (f < 2 + CBO_MAX_D) src = (f - 2 < D) ? f : -1;
        else src = (f - 2 - CBO_MAX_D < D) ? f - CBO_MAX_D + D : -1;
        if (src >= 0) s = ((sred[0][q][src] + sred[1][q][src]) + sred[2][q][src]) + sred[3][q][src];
        out[e] = s;
    }
}

// ---- per-point posterior, EI and gradients: one warp per point -------------------------------------------------------------
struct RefSmem {
    double* Lp;     // packed lower triangle of L, row i at i (i + 1) / 2
    double* al;     // alpha
    double* sv;     // sqrt(v_int) (0 for a non-causal set)
    double* xs;     // x_int / l, n x d
    double s2, il;  // per-set GP variance and 1 / lengthscale
};
inline size_t ref_smem_bytes(int n) { return ((size_t)n * (n + 1) / 2 + 2 * (size_t)n + (size_t)n * CBO_MAX_D) * sizeof(double); }

__device__ void stage_posterior(const cbo_set_desc& S, RefSmem& sm, double* base) {
    const int n = S.n_int, d = S.d;
    sm.Lp = base;
    sm.al = sm.Lp + (size_t)n * (n + 1) / 2;
    sm.sv = sm.al + n;
    sm.xs = sm.sv + n;
    const SurrogateHyper h = surrogate_hyper(S);
    sm.s2 = h.s2;
    sm.il = h.il;
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
        const int i = e / n, j = e % n;
        if (j <= i) sm.Lp[i * (i + 1) / 2 + j] = S.L[e];
    }
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        sm.al[i] = S.alpha[i];
        sm.sv[i] = S.causal ? S.sqrt_v_int[i] : 0.0;
    }
    for (int i = threadIdx.x; i < n * d; i += blockDim.x) sm.xs[i] = S.x_int[i] * sm.il;
}

// partials: the set's slots of this point's batch (NULL when the set has no device prior); q = point within the batch
__device__ void eval_point(const cbo_set_desc& S, const RefSmem& sm, const double* __restrict__ partials, int q,
                           const double (&x)[CBO_MAX_D], double best, double task_sign, cbo_acq_grad_out& o) {
    const int lane = threadIdx.x & 31, n = S.n_int, d = S.d;
    const unsigned FULL = 0xffffffffu;
    double m = 0.0, v = 0.0, dm[CBO_MAX_D] = {0.0, 0.0, 0.0, 0.0}, dv[CBO_MAX_D] = {0.0, 0.0, 0.0, 0.0};
    if (partials) {
        // partial slots in index order per lane, then a fixed butterfly: the same additions on every run
        const int chunks = ref_chunks(S), items = ref_nJ(S) * chunks;
        double acc[kRefPF];
#pragma unroll
        for (int f = 0; f < kRefPF; ++f) acc[f] = 0.0;
        for (int e = lane; e < items; e += 32) {
            const int I = e / chunks, c = e - I * chunks;
            if (c * kRefSlabs >= (I + 1) * (kMBlkRows / kBK)) continue;
            const double* p = partials + (long long)e * kRefItemDoubles + q * kRefPF;
#pragma unroll
            for (int f = 0; f < kRefPF; ++f) acc[f] += p[f];
        }
#pragma unroll
        for (int f = 0; f < kRefPF; ++f) acc[f] = warp_sum(acc[f]);
        m = acc[0];
        v = (S.s2 + S.noise) - acc[1];
#pragma unroll
        for (int k = 0; k < CBO_MAX_D; ++k) {
            dm[k] = k < d ? -acc[2 + k] : 0.0;
            dv[k] = k < d ? acc[2 + CBO_MAX_D + k] : 0.0;
        }
    }
    const bool causal = S.causal != 0;
    const double sqv = causal ? sqrt(v) : 0.0;
    const double hv = causal ? 0.5 / sqv : 0.0;
    // rows i = lane + 32 r of k*, dk*
    double ks[4], dks[4][CBO_MAX_D], rr[4];
    double mu_p = 0.0, dmu_p[CBO_MAX_D] = {0.0, 0.0, 0.0, 0.0};
    double xl[CBO_MAX_D];
#pragma unroll
    for (int k = 0; k < CBO_MAX_D; ++k) xl[k] = x[k] * sm.il;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int i = lane + 32 * r;
        ks[r] = 0.0;
#pragma unroll
        for (int k = 0; k < CBO_MAX_D; ++k) dks[r][k] = 0.0;
        if (i < n) {
            double r2 = 0.0, z[CBO_MAX_D];
#pragma unroll
            for (int k = 0; k < CBO_MAX_D; ++k) {
                z[k] = k < d ? xl[k] - sm.xs[i * d + k] : 0.0;
                r2 = fma(z[k], z[k], r2);
            }
            const double e = surrogate_rbf(r2, sm.s2);
            ks[r] = surrogate_k(r2, sm.sv[i], sqv, sm.s2);
#pragma unroll
            for (int k = 0; k < CBO_MAX_D; ++k) dks[r][k] = fma(-e, __dmul_rn(z[k], sm.il), sm.sv[i] * dv[k] * hv);
            mu_p = fma(ks[r], sm.al[i], mu_p);
#pragma unroll
            for (int k = 0; k < CBO_MAX_D; ++k) dmu_p[k] = fma(sm.al[i], dks[r][k], dmu_p[k]);
        }
        rr[r] = ks[r];
    }
    const double mu = m + warp_sum(mu_p);
    double dmu[CBO_MAX_D];
#pragma unroll
    for (int k = 0; k < CBO_MAX_D; ++k) dmu[k] = dm[k] + warp_sum(dmu_p[k]);

    // t = L^-1 k* (column-oriented forward substitution; lane j % 32 owns t_j)
#pragma unroll
    for (int rb = 0; rb < 4; ++rb) {
        const int jn = n - 32 * rb < 32 ? n - 32 * rb : 32;
        for (int jj = 0; jj < jn; ++jj) {
            const int j = 32 * rb + jj;
            const double tj = __shfl_sync(FULL, rr[rb], jj) / sm.Lp[j * (j + 1) / 2 + j];
            if (lane == jj) rr[rb] = tj;
#pragma unroll
            for (int r = rb; r < 4; ++r) {
                const int i = lane + 32 * r;
                if (i > j && i < n) rr[r] = fma(-sm.Lp[i * (i + 1) / 2 + j], tj, rr[r]);
            }
        }
    }
    double ss = 0.0;
#pragma unroll
    for (int r = 0; r < 4; ++r) ss = fma(rr[r], rr[r], ss);
    ss = warp_sum(ss);
    const double var = surrogate_var(sm.s2, v, ss);
    // beta = L^-T t (backward substitution; lane j % 32 owns beta_j)
#pragma unroll
    for (int rb = 3; rb >= 0; --rb) {
        const int jn = n - 32 * rb < 32 ? n - 32 * rb : 32;
        for (int jj = jn - 1; jj >= 0; --jj) {
            const int j = 32 * rb + jj;
            const double* Lj = sm.Lp + j * (j + 1) / 2;
            const double bj = __shfl_sync(FULL, rr[rb], jj) / Lj[j];
            if (lane == jj) rr[rb] = bj;
#pragma unroll
            for (int r = 0; r <= rb; ++r) {
                const int i = lane + 32 * r;
                if (i < j) rr[r] = fma(-Lj[i], bj, rr[r]);
            }
        }
    }
    double dvar[CBO_MAX_D];
#pragma unroll
    for (int k = 0; k < CBO_MAX_D; ++k) {
        double s = 0.0;
#pragma unroll
        for (int r = 0; r < 4; ++r) s = fma(rr[r], dks[r][k], s);
        dvar[k] = dv[k] - 2.0 * warp_sum(s);
    }
    const ExpectedImprovement e = expected_improvement(best, mu, var, task_sign);
    const double cost = candidate_cost(S, d, x);
    const double acq = e.ei / cost;
    o.m = m; o.v = v; o.mu = mu; o.var = var; o.ei = e.ei; o.acq = acq;
#pragma unroll
    for (int k = 0; k < CBO_MAX_D; ++k) {
        const double dc = (S.cost_variable && k < d) ? (x[k] > 0.0 ? 1.0 : (x[k] < 0.0 ? -1.0 : 0.0)) : 0.0;
        const double dei = task_sign * (e.pdf * dvar[k] / (2.0 * e.sd) - e.cdf * dmu[k]);
        o.dm[k] = dm[k]; o.dv[k] = dv[k]; o.dmu[k] = dmu[k]; o.dvar[k] = dvar[k]; o.dei[k] = dei;
        o.dacq[k] = (dei - acq * dc) / cost;
    }
}

__global__ void __launch_bounds__(kStepThreads)
acq_grad_kernel(const cbo_set_desc* __restrict__ set, const double* __restrict__ pts, int num_points, int batch0, double best,
                double task_sign, const double* __restrict__ partials, long long batch_stride, cbo_acq_grad_out* __restrict__ out) {
    extern __shared__ __align__(16) double smem_d[];
    const cbo_set_desc& S = *set;
    RefSmem sm;
    stage_posterior(S, sm, smem_d);
    __syncthreads();
    const int q = threadIdx.x >> 5, lb = blockIdx.x, pi = (batch0 + lb) * kRefB + q;
    if (pi >= num_points) return;                      // warp-uniform; no barrier follows
    double x[CBO_MAX_D];
#pragma unroll
    for (int k = 0; k < CBO_MAX_D; ++k) x[k] = k < S.d ? pts[(long long)pi * S.d + k] : 0.0;
    cbo_acq_grad_out o;
    eval_point(S, sm, computes_prior(S) ? partials + lb * batch_stride : nullptr, q, x, best, task_sign, o);
    if ((threadIdx.x & 31) == 0) out[pi] = o;
}

// ---- refinement --------------------------------------------------------------------------------------------------------
__global__ void refine_init_kernel(const cbo_set_desc* __restrict__ sets, int num_sets, const double* __restrict__ x0, int max_iter,
                                   RefineState* __restrict__ state, int* __restrict__ running) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= num_sets) return;
    const cbo_set_desc& S = sets[s];
    RefineState& R = state[s];
    long long base = 0;
    for (int t = 0; t < s; ++t) base += ref_items(sets[t]) * kRefItemDoubles;
    R.part_base = base;
    R.iter = 0; R.qn = 0; R.ntrial = 1; R.max_iter = max_iter;
    R.f = R.f0 = __longlong_as_double(0x7ff8000000000000LL);   // NaN until evaluated
    bool finite = true;
    for (int k = 0; k < CBO_MAX_D; ++k) {
        R.x0[k] = k < S.d ? x0[(size_t)s * CBO_MAX_D + k] : 0.0;
        finite &= !isnan(R.x0[k]);
        R.g[k] = R.p[k] = 0.0;
        for (int j = 0; j < CBO_MAX_D; ++j) R.H[k * CBO_MAX_D + j] = 0.0;
    }
    R.status = S.causal && S.prior_external ? CBO_REFINE_SKIPPED_EXTERNAL
             : S.points ? CBO_REFINE_SKIPPED_POINTS
             : !finite ? CBO_REFINE_SKIPPED_NONFINITE : CBO_REFINE_CONVERGED;
    R.running = R.status == CBO_REFINE_CONVERGED;
    for (int k = 0; k < CBO_MAX_D; ++k) {
        double lo = 0.0, hi = 0.0, h = 0.0;
        if (k < S.d && R.running) {
            lo = hi = S.grid[k][0];
            for (int i = 1; i < S.p[k]; ++i) { lo = fmin(lo, S.grid[k][i]); hi = fmax(hi, S.grid[k][i]); }
            h = S.p[k] > 1 ? (hi - lo) / (S.p[k] - 1) : 0.0;
        }
        R.lo[k] = lo; R.hi[k] = hi; R.h[k] = h;
        R.x[k] = k < S.d ? fmin(fmax(R.x0[k], lo), hi) : 0.0;
        if (!R.running) R.x[k] = R.x0[k];
    }
    for (int j = 0; j < kRefB; ++j)
        for (int k = 0; k < CBO_MAX_D; ++k) R.xt[j][k] = R.x[k];
    if (R.running) atomicAdd(running, 1);
}

// New search direction from (x, g, H) and the 8 trial points; returns false when the projected gradient is small.
__device__ bool refine_direction(RefineState& R, int d, double gtol) {
    double pg[CBO_MAX_D], gmax = 0.0, rel = 0.0;
    bool fr[CBO_MAX_D];
    for (int k = 0; k < CBO_MAX_D; ++k) {
        fr[k] = k < d && R.h[k] > 0.0 && !(R.x[k] <= R.lo[k] && R.g[k] < 0.0) && !(R.x[k] >= R.hi[k] && R.g[k] > 0.0);
        pg[k] = fr[k] ? R.g[k] : 0.0;
        if (fr[k]) {
            gmax = fmax(gmax, fabs(pg[k]) / R.h[k]);
            rel = fmax(rel, fabs(pg[k]) * (R.hi[k] - R.lo[k]));
        }
    }
    if (!(rel > gtol * fabs(R.f))) return false;
    double p[CBO_MAX_D], slope = 0.0;
    if (R.qn) {
        for (int k = 0; k < CBO_MAX_D; ++k) {
            p[k] = 0.0;
            if (fr[k])
                for (int j = 0; j < CBO_MAX_D; ++j) p[k] = fma(R.H[k * CBO_MAX_D + j], pg[j], p[k]);
            slope = fma(p[k], pg[k], slope);
        }
        if (!(slope > 0.0)) R.qn = 0;                 // not an ascent direction: restart from the scaled gradient
    }
    if (!R.qn)
        for (int k = 0; k < CBO_MAX_D; ++k) p[k] = pg[k] / gmax;   // largest move: one grid spacing
    for (int k = 0; k < CBO_MAX_D; ++k) R.p[k] = p[k];
    for (int j = 0; j < kRefB; ++j) {
        const double t = ldexp(1.0, -j);
        for (int k = 0; k < CBO_MAX_D; ++k)
            R.xt[j][k] = k < d ? fmin(fmax(fma(t, p[k], R.x[k]), R.lo[k]), R.hi[k]) : 0.0;
    }
    R.ntrial = kRefB;
    return true;
}

__global__ void __launch_bounds__(kStepThreads)
refine_step_kernel(const cbo_set_desc* __restrict__ sets, double best, double task_sign, double gtol, RefineState* __restrict__ state,
                   const double* __restrict__ partials, int* __restrict__ running) {
    extern __shared__ __align__(16) double smem_d[];
    __shared__ double sf[kRefB], sg[kRefB][CBO_MAX_D];
    const int s = blockIdx.x;
    const cbo_set_desc& S = sets[s];
    RefineState& R = state[s];
    if (!R.running) return;                           // CTA-uniform
    RefSmem sm;
    stage_posterior(S, sm, smem_d);
    __syncthreads();
    const int q = threadIdx.x >> 5, d = S.d;
    if (q < R.ntrial) {
        double x[CBO_MAX_D];
#pragma unroll
        for (int k = 0; k < CBO_MAX_D; ++k) x[k] = R.xt[q][k];
        cbo_acq_grad_out o;
        eval_point(S, sm, computes_prior(S) ? partials + R.part_base : nullptr, q, x, best, task_sign, o);
        if ((threadIdx.x & 31) == 0) {
            sf[q] = o.acq;
#pragma unroll
            for (int k = 0; k < CBO_MAX_D; ++k) sg[q][k] = o.dacq[k];
        }
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    bool go = true;
    if (R.ntrial == 1) {                              // the start point
        R.f = R.f0 = sf[0];
        for (int k = 0; k < CBO_MAX_D; ++k) R.g[k] = sg[0][k];
        bool ok = isfinite(R.f);
        for (int k = 0; k < d; ++k) ok &= isfinite(R.g[k]);
        if (!ok) { R.status = isfinite(R.f) ? CBO_REFINE_LINE_SEARCH_FAILED : CBO_REFINE_SKIPPED_NONFINITE; go = false; }
    } else {                                          // a line search: the largest step that passes Armijo's test
        ++R.iter;
        int acc = -1;
        for (int j = 0; j < kRefB && acc < 0; ++j) {
            double gain = 0.0;
            for (int k = 0; k < d; ++k) gain = fma(R.g[k], R.xt[j][k] - R.x[k], gain);
            bool ok = sf[j] > R.f && sf[j] >= R.f + kArmijo * gain;     // NaN fails both
            for (int k = 0; k < d; ++k) ok &= isfinite(sg[j][k]);
            if (ok) acc = j;
        }
        if (acc < 0) {
            if (R.qn) R.qn = 0;                       // retry along the scaled gradient
            else { R.status = CBO_REFINE_LINE_SEARCH_FAILED; go = false; }
        } else {
            double sv[CBO_MAX_D], yv[CBO_MAX_D], sy = 0.0, yy = 0.0, smax = 0.0;
            for (int k = 0; k < CBO_MAX_D; ++k) {
                sv[k] = k < d ? R.xt[acc][k] - R.x[k] : 0.0;
                yv[k] = k < d ? -(sg[acc][k] - R.g[k]) : 0.0;    // gradient change of -acq
                sy = fma(sv[k], yv[k], sy);
                yy = fma(yv[k], yv[k], yy);
                if (k < d && R.hi[k] > R.lo[k]) smax = fmax(smax, fabs(sv[k]) / (R.hi[k] - R.lo[k]));
            }
            if (sy > 0.0) {                           // BFGS update of the inverse Hessian of -acq
                if (!R.qn) {
                    for (int k = 0; k < CBO_MAX_D; ++k)
                        for (int j = 0; j < CBO_MAX_D; ++j) R.H[k * CBO_MAX_D + j] = k == j && k < d ? sy / yy : 0.0;
                    R.qn = 1;
                }
                const double rho = 1.0 / sy;
                double Hy[CBO_MAX_D], yHy = 0.0;
                for (int k = 0; k < CBO_MAX_D; ++k) {
                    Hy[k] = 0.0;
                    for (int j = 0; j < CBO_MAX_D; ++j) Hy[k] = fma(R.H[k * CBO_MAX_D + j], yv[j], Hy[k]);
                    yHy = fma(yv[k], Hy[k], yHy);
                }
                for (int k = 0; k < CBO_MAX_D; ++k)
                    for (int j = 0; j < CBO_MAX_D; ++j)
                        R.H[k * CBO_MAX_D + j] += (1.0 + rho * yHy) * rho * sv[k] * sv[j] - rho * (Hy[k] * sv[j] + sv[k] * Hy[j]);
            }
            for (int k = 0; k < CBO_MAX_D; ++k) { R.x[k] = R.xt[acc][k]; R.g[k] = sg[acc][k]; }
            R.f = sf[acc];
            if (smax <= 1e-12) { R.status = CBO_REFINE_CONVERGED; go = false; }
        }
    }
    if (go) {
        if (!refine_direction(R, d, gtol)) { R.status = CBO_REFINE_CONVERGED; go = false; }
        else if (R.iter >= R.max_iter) { R.status = CBO_REFINE_MAX_ITER; go = false; }
    }
    if (!go) {
        R.running = 0;
        atomicSub(running, 1);
    }
}

__global__ void refine_finish_kernel(const RefineState* __restrict__ state, int num_sets, cbo_refine_result* __restrict__ out) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= num_sets) return;
    const RefineState& R = state[s];
    cbo_refine_result r;
    const bool better = R.f > R.f0;
    for (int k = 0; k < CBO_MAX_D; ++k) r.x[k] = better ? R.x[k] : R.x0[k];
    r.value = better ? R.f : R.f0;
    r.start_value = R.f0;
    r.iterations = R.iter;
    r.status = R.status;
    out[s] = r;
}

// ---- host side -----------------------------------------------------------------------------------------------------------
static size_t ref_partial_bytes(const cbo_set_desc* h_sets, int num_sets) {
    long long t = 0;
    for (int s = 0; s < num_sets; ++s) t += ref_items(h_sets[s]);
    return (size_t)t * kRefItemDoubles * sizeof(double);
}

size_t refine_workspace_bytes_impl(const cbo_set_desc* h_sets, int num_sets) {
    return kRefHeader + ref_state_bytes(num_sets) + ref_partial_bytes(h_sets, num_sets);
}

// one prior-gradient pass: a launch per dimension count present among the sets with a device prior
static int launch_prior_pass(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, const PassArgs& a, cudaStream_t st) {
    int nJ = 0, chunks = 0;
    bool dims[CBO_MAX_D + 1] = {};
    for (int s = 0; s < num_sets; ++s) {
        const cbo_set_desc& S = h_sets[s];
        if (!computes_prior(S)) continue;
        dims[S.d] = true;
        if (ref_nJ(S) > nJ) nJ = ref_nJ(S);
        if (ref_chunks(S) > chunks) chunks = ref_chunks(S);
    }
    if (!nJ) return 0;
    CBO_REQUIRE((long long)num_sets * a.nbatch <= 65535 && nJ <= 65535, "K7: too many sets or rows for one launch");
    const dim3 grid(chunks, nJ, num_sets * a.nbatch);
#define CBO_REF_PASS(D)                                                                                   \
    if (dims[D]) {                                                                                        \
        CBO_CUDA(allow_dynamic_smem(refine_prior_kernel<D>, kRefRingBytes));                              \
        refine_prior_kernel<D><<<grid, kRefThreads, kRefRingBytes, st>>>(d_sets, a);                      \
        note_launch();                                                                                    \
        CBO_CUDA(cudaGetLastError());                                                                     \
    }
    CBO_REF_PASS(1) CBO_REF_PASS(2) CBO_REF_PASS(3) CBO_REF_PASS(4)
#undef CBO_REF_PASS
    return 0;
}

static int check_posterior_ptrs(const cbo_set_desc& S, int s, const char* who) {
    CBO_REQUIRE(S.L && S.alpha && S.x_int, "%s: set %d has a NULL posterior pointer", who, s);
    CBO_REQUIRE(!S.causal || S.prior_external || S.sqrt_v_int, "%s: causal set %d needs sqrt_v_int", who, s);
    if (computes_prior(S)) CBO_REQUIRE(S.M && S.w && S.x_obs_int, "%s: set %d has NULL M/w/x_obs_int", who, s);
    return 0;
}

int acq_grad_impl(const cbo_set_desc* h_set, const cbo_set_desc* d_set, const double* d_points, int num_points, double best, int task_sign,
                  void* d_ws, size_t ws_bytes, cbo_acq_grad_out* d_out, cudaStream_t st) {
    const cbo_set_desc& S = *h_set;
    CBO_REQUIRE(d_set != nullptr, "cbo_acq_grad: d_set is NULL");
    CBO_REQUIRE(task_sign == 1 || task_sign == -1, "cbo_acq_grad: task_sign must be +1 ('min') or -1 ('max')");
    CBO_REQUIRE(num_points >= 0, "cbo_acq_grad: num_points=%d is negative", num_points);
    CBO_REQUIRE(num_points == 0 || (d_points && d_out), "cbo_acq_grad: NULL points or output");
    CBO_REQUIRE(!(S.causal && S.prior_external), "cbo_acq_grad: the set's prior is supplied by the caller; there is no device prior to differentiate");
    if (int rc = check_posterior_ptrs(S, 0, "cbo_acq_grad")) return rc;
    const long long per_batch = ref_items(S) * kRefItemDoubles;
    const size_t need = kRefHeader + ref_state_bytes(1) + (size_t)per_batch * sizeof(double);
    CBO_REQUIRE(d_ws != nullptr && ws_bytes >= need, "cbo_acq_grad: workspace of %zu bytes is too small (%zu needed; see cbo_refine_workspace_bytes)",
                ws_bytes, need);
    if (num_points == 0) return 0;
    double* partials = reinterpret_cast<double*>(static_cast<unsigned char*>(d_ws) + kRefHeader + ref_state_bytes(1));
    const int nbatch = (num_points + kRefB - 1) / kRefB;
    const long long room = per_batch ? (long long)((ws_bytes - kRefHeader - ref_state_bytes(1)) / sizeof(double)) / per_batch : nbatch;
    const int per_launch = (int)(room < nbatch ? (room < 65535 ? room : 65535) : (nbatch < 65535 ? nbatch : 65535));
    const size_t smem = ref_smem_bytes(S.n_int);
    if (smem > 48 * 1024) CBO_CUDA(allow_dynamic_smem(acq_grad_kernel, smem));
    for (int b0 = 0; b0 < nbatch; b0 += per_launch) {
        const int nb = nbatch - b0 < per_launch ? nbatch - b0 : per_launch;
        PassArgs a{d_points + (long long)b0 * kRefB * S.d, 0, S.d, num_points - b0 * kRefB, nb, nullptr, partials};
        if (int rc = launch_prior_pass(h_set, d_set, 1, a, st)) return rc;
        acq_grad_kernel<<<nb, kStepThreads, smem, st>>>(d_set, d_points, num_points, b0, best, (double)task_sign, partials, per_batch, d_out);
        note_launch();
        CBO_CUDA(cudaGetLastError());
    }
    return 0;
}

int refine_impl(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, double best, int task_sign, const double* d_x0,
                int max_iter, double gtol, void* d_ws, size_t ws_bytes, cbo_refine_result* d_out, cudaStream_t st) {
    CBO_REQUIRE(d_sets != nullptr, "cbo_refine: d_sets is NULL");
    CBO_REQUIRE(task_sign == 1 || task_sign == -1, "cbo_refine: task_sign must be +1 ('min') or -1 ('max')");
    CBO_REQUIRE(d_x0 && d_out, "cbo_refine: NULL start points or output");
    CBO_REQUIRE(max_iter >= 0 && max_iter <= 100000, "cbo_refine: max_iter=%d outside [0,100000]", max_iter);
    CBO_REQUIRE(gtol >= 0.0 && gtol < 1.0, "cbo_refine: gtol must lie in [0, 1)");
    int nmax = 1;
    for (int s = 0; s < num_sets; ++s) {
        const cbo_set_desc& S = h_sets[s];
        if ((S.causal && S.prior_external) || S.points) continue;      // skipped: read nothing of them
        if (int rc = check_posterior_ptrs(S, s, "cbo_refine")) return rc;
        for (int k = 0; k < S.d; ++k) CBO_REQUIRE(S.grid[k], "cbo_refine: set %d grid[%d] is NULL", s, k);
        if (S.n_int > nmax) nmax = S.n_int;
    }
    const size_t need = refine_workspace_bytes_impl(h_sets, num_sets);
    CBO_REQUIRE(d_ws != nullptr && ws_bytes >= need, "cbo_refine: workspace of %zu bytes is too small (%zu needed; see cbo_refine_workspace_bytes)",
                ws_bytes, need);
    unsigned char* ws = static_cast<unsigned char*>(d_ws);
    int* running = reinterpret_cast<int*>(ws);
    RefineState* state = reinterpret_cast<RefineState*>(ws + kRefHeader);
    double* partials = reinterpret_cast<double*>(ws + kRefHeader + ref_state_bytes(num_sets));
    CBO_CUDA(cudaMemsetAsync(running, 0, sizeof(int), st));
    refine_init_kernel<<<(num_sets + 127) / 128, 128, 0, st>>>(d_sets, num_sets, d_x0, max_iter, state, running);
    note_launch();
    CBO_CUDA(cudaGetLastError());
    const size_t smem = ref_smem_bytes(nmax);
    if (smem > 48 * 1024) CBO_CUDA(allow_dynamic_smem(refine_step_kernel, smem));
    const PassArgs a{&state[0].xt[0][0], (long long)(sizeof(RefineState) / sizeof(double)), CBO_MAX_D, kRefB, 1, state, partials};
    // pass 0 evaluates the start point; every later pass one line search.  The host polls the running count every
    // kRefPoll passes (4 bytes) so that a call whose sets have all stopped launches nothing more.
    constexpr int kRefPoll = 4;
    for (int it = 0; it <= max_iter; ++it) {
        if (it > 0 && it % kRefPoll == 0) {
            int left = 0;
            CBO_CUDA(cudaMemcpyAsync(&left, running, sizeof(int), cudaMemcpyDeviceToHost, st));
            CBO_CUDA(cudaStreamSynchronize(st));
            if (left == 0) break;
        }
        if (int rc = launch_prior_pass(h_sets, d_sets, num_sets, a, st)) return rc;
        refine_step_kernel<<<num_sets, kStepThreads, smem, st>>>(d_sets, best, (double)task_sign, gtol, state, partials, running);
        note_launch();
        CBO_CUDA(cudaGetLastError());
    }
    refine_finish_kernel<<<(num_sets + 127) / 128, 128, 0, st>>>(state, num_sets, d_out);
    note_launch();
    CBO_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace cbo
