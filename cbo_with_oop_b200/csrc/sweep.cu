// K3 + K4 -- posterior predict, Expected Improvement / cost and the first-argmax over every candidate.
//
// Per candidate x of set s (one thread each; L, alpha, X_I staged once per CTA in shared memory):
//   k*_i = s2 exp(-.5 |x - X_I,i|^2 / l^2) + sqrt(v_I,i) sqrt(v(x))   CausalRBF.K(X_I, x), causal_kernels.py:55-62
//   mu   = m(x) + k*.alpha                                           GPy PosteriorExact._raw_predict + mean function
//   t    = L^-1 k* ; var = (s2 + v(x)) - |t|^2 + noise               Kdiag :64-79, dtrtrs, Gaussian noise
//   (s2, l) = surrogate_hyper(S).  1 / l scales the staged coordinates (x_int, the candidate, the
//   differences behind the separable tables) once, s2 is folded into the leading-dimension table and the A fragments: the
//   per-candidate arithmetic is unchanged, and at (1, 1) every product is by 1.0, so the results are those of l = s2 = 1.
//          (forward substitution for n <= 16 and n > 48; a DMMA product with L^-1 for 16 < n <= 48: sweep_mma_kernel)
//   EI   = sd (u Phi(u) + phi(u)), u = (best - mu) / sd, negated for task 'max'   causal_acquisition_functions.py:33-43,85-87
//   acq  = EI / cost(x)                                              utils.py:34, cost_functions.py:11-17
// then a (value, index) max-reduction with np.argmax semantics (first maximum; NaN counts as -inf and is
// tallied), per tile -> per set -> global (CBO.select_next_intervention, CBO.py:269-277: first set attaining the max).
// The variance is not clipped (the reference does not clip either); a negative variance gives NaN.
// Sets whose posterior is cached (cbo_set_desc.posterior_cached) only refresh EI from mu / var: ei_refresh_kernel.
// k*, var, EI, the cost, the candidate's coordinates and the argmax reduction are surrogate.cuh's (shared with K2, K7, K8);
// the separable k* tables below are a different factorisation of k* and keep their own form.
// Roofline: with the prior cached this pass is 16 B/candidate of HBM reads plus n^2/2 FMAs; it is a few
// per cent of a post-observation sweep and half of a post-intervention trial.
#include <float.h>
#include "surrogate.cuh"

namespace cbo {

constexpr int kSweepThreads = 128;     // a work item is CBO_SWEEP_TILE consecutive candidates, kSweepThreads at a time

// Shared-memory image of one set's posterior: L^-1 is NOT formed; the forward substitution reads L rows (packed lower
// triangle) as warp-wide broadcasts.
struct SweepSmem {
    double* Lp;    // packed lower triangle, row i at i(i+1)/2, diagonal entries inverted
    double* al;    // alpha
    double* sv;    // sqrt(v_int)
    double* xs;    // x_int, n x d
    double* tcol;  // [n][kSweepThreads] workspace of the generic path
};

// Posterior mean and |L^-1 k*|^2 of one candidate.  NREG > 0: n <= NREG and the solution vector lives in registers
// (fully unrolled, one broadcast LDS per FMA); NREG == 0: any n <= CBO_MAX_NINT, the vector lives in a shared-memory
// column owned by the thread.
template <int NREG>
__device__ __forceinline__ void posterior_at(const SweepSmem& sm, int n, int d, const double (&x)[CBO_MAX_D], double svg, double s2,
                                             int tid, double& mu, double& ss) {
    mu = 0.0; ss = 0.0;
    if constexpr (NREG > 0) {
        double t[NREG];
#pragma unroll
        for (int i = 0; i < NREG; ++i) {
            if (i < n) {
                double r2 = 0.0;
#pragma unroll
                for (int k = 0; k < CBO_MAX_D; ++k) {
                    if (k < d) { const double q = x[k] - sm.xs[i * d + k]; r2 = fma(q, q, r2); }
                }
                const double ks = surrogate_k(r2, sm.sv[i], svg, s2);
                mu = fma(ks, sm.al[i], mu);
                const double* __restrict__ Li = sm.Lp + i * (i + 1) / 2;
                // four interleaved partial sums: the row's dot product is a dependent FMA chain, and with 3-5 CTAs per SM
                // the FP64 latency, not the pipe, set the pace (1e3 dependent FMAs per candidate at n = 45)
                double a0 = ks, a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll
                for (int j = 0; j < i; ++j) {
                    if ((j & 3) == 0) a0 = fma(-Li[j], t[j], a0);
                    else if ((j & 3) == 1) a1 = fma(-Li[j], t[j], a1);
                    else if ((j & 3) == 2) a2 = fma(-Li[j], t[j], a2);
                    else a3 = fma(-Li[j], t[j], a3);
                }
                t[i] = ((a0 + a1) + (a2 + a3)) * Li[i];     // Li[i] = 1 / L[i][i]: staged once per item, no division per candidate and row
                ss = fma(t[i], t[i], ss);
            }
        }
    } else {
        for (int i = 0; i < n; ++i) {
            double r2 = 0.0;
#pragma unroll
            for (int k = 0; k < CBO_MAX_D; ++k) {
                if (k < d) { const double q = x[k] - sm.xs[i * d + k]; r2 = fma(q, q, r2); }
            }
            const double ks = surrogate_k(r2, sm.sv[i], svg, s2);
            mu = fma(ks, sm.al[i], mu);
            const double* __restrict__ Li = sm.Lp + i * (i + 1) / 2;
            double a = ks;
            for (int j = 0; j < i; ++j) a = fma(-Li[j], sm.tcol[j * kSweepThreads + tid], a);
            const double tt = a * Li[i];
            sm.tcol[i * kSweepThreads + tid] = tt;
            ss = fma(tt, tt, ss);
        }
    }
}

// Separable form of k* on a tensor grid: exp(-.5 |x - X_I,i|^2) = E_lead[row][i] * E_last[j][i], the product of the
// leading dimensions' factor (constant along a run of the fastest grid dimension) and the fastest dimension's factor.
// A work item of CBO_SWEEP_TILE consecutive candidates touches at most CBO_SWEEP_TILE / p_last + 2 leading rows and
// p_last values of the fastest index, so the CTA evaluates (rows + p_last) * n exponentials once, in shared memory,
// instead of n per candidate (9x fewer at p = 100, n = 10).  Used when n <= 48 and p_last <= kSepMaxP; otherwise
// every candidate evaluates its own exponentials (explicit points, very long last dimensions, n > 48).
constexpr int kSepMaxP = 256;
__host__ __device__ inline bool sweep_separable(const cbo_set_desc& S) {
    return !S.points && S.n_int <= 48 && S.p[S.d - 1] <= kSepMaxP && S.p[S.d - 1] >= 16;   // (>= 16: at most 66 leading rows per item)
}
__host__ __device__ inline int sweep_lead_rows(const cbo_set_desc& S) { return CBO_SWEEP_TILE / S.p[S.d - 1] + 2; }

// Which launch evaluates a set (decided by the set alone, never by its neighbours in the call):
//   0  sweep_kernel<16, false>   n <= 16 without separable tables; cached posterior with a variable cost
//   1  sweep_kernel<16, true>    n <= 16 on a tensor grid
//   2  sweep_mma_kernel<true>    16 < n <= 48 on a tensor grid      (|L^-1 k*|^2 on the FP64 tensor pipe)
//   3  sweep_mma_kernel<false>   16 < n <= 48, explicit points / very short or long last dimension
//   4  sweep_kernel<0, false>    n > 48
//   5  ei_refresh_kernel         cached posterior, fixed cost: EI refresh from mu / var (16 B per candidate)
enum { kClsFma = 0, kClsFmaSep = 1, kClsMmaSep = 2, kClsMma = 3, kClsGeneric = 4, kClsCached = 5, kNumSweepClasses = 6 };
__host__ __device__ inline int sweep_class(const cbo_set_desc& S) {
    if (S.posterior_cached) return S.cost_variable ? kClsFma : kClsCached;
    if (S.n_int <= kSweepFmaMaxN) return sweep_separable(S) ? kClsFmaSep : kClsFma;
    if (S.n_int <= kSweepMmaMaxN) return sweep_separable(S) ? kClsMmaSep : kClsMma;
    return kClsGeneric;
}

template <int NREG>
__device__ __forceinline__ void posterior_sep(const SweepSmem& sm, int n, const double* __restrict__ eLast, int ldl,
                                              const double* __restrict__ eLead, int ldr, double svg, double& mu, double& ss) {
    mu = 0.0; ss = 0.0;
    double t[NREG];
#pragma unroll
    for (int i = 0; i < NREG; ++i) {
        if (i < n) {
            const double ks = fma(eLead[i * ldr], eLast[i * ldl], sm.sv[i] * svg);
            mu = fma(ks, sm.al[i], mu);
            const double* __restrict__ Li = sm.Lp + i * (i + 1) / 2;
            double a0 = ks, a1 = 0.0, a2 = 0.0, a3 = 0.0;      // (four interleaved partial sums, as in posterior_at)
#pragma unroll
            for (int j = 0; j < i; ++j) {
                if ((j & 3) == 0) a0 = fma(-Li[j], t[j], a0);
                else if ((j & 3) == 1) a1 = fma(-Li[j], t[j], a1);
                else if ((j & 3) == 2) a2 = fma(-Li[j], t[j], a2);
                else a3 = fma(-Li[j], t[j], a3);
            }
            t[i] = ((a0 + a1) + (a2 + a3)) * Li[i];
            ss = fma(t[i], t[i], ss);
        }
    }
}

// NREG = 16: n <= 16, the forward substitution runs in registers; NREG = 0: n > 48, the solution vector lives in shared
// memory (16 < n <= 48 is sweep_mma_kernel's).  SEP: the sets whose posterior is evaluated through the separable k* tables.
// Which launch takes a set is decided by the set alone (sweep_class), so a set's arithmetic never depends on which other sets
// share the call (ranks that hold different subsets must produce the same bits), and each instantiation carries one path
// only (less code, fewer live registers).
template <int NREG, bool SEP>
__global__ void __launch_bounds__(kSweepThreads, 5)
sweep_kernel(const cbo_set_desc* __restrict__ sets, int num_sets, double best, double task_sign,
             cbo_set_best* __restrict__ tile_best) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    int tile;
    const int s = find_item(sets, num_sets, kItemsSweep, blockIdx.x, tile);
    const cbo_set_desc& S = sets[s];
    const int n = S.n_int, d = S.d, tid = threadIdx.x;
    const bool causal = S.causal != 0;
    const bool cached = S.posterior_cached != 0;   // mu / var of an earlier sweep are still valid: EI refresh only
    const auto [s2, il] = surrogate_hyper(S);
    if (sweep_class(S) != (NREG == 0 ? kClsGeneric : (SEP ? kClsFmaSep : kClsFma))) return;       // another launch's set
    const bool sep = SEP;
    const int p_last = S.points ? 1 : S.p[d - 1];

    SweepSmem sm;
    sm.Lp = reinterpret_cast<double*>(smem_raw);
    sm.al = sm.Lp + (size_t)n * (n + 1) / 2;
    sm.sv = sm.al + n;
    sm.xs = sm.sv + n;
    sm.tcol = sm.xs + (size_t)n * CBO_MAX_D;      // generic path (n > 48): [n][threads]; separable path: the two tables
    const int ldl = p_last | 1, ldr = sweep_lead_rows(S) | 1;          // odd pitches: no bank conflicts
    double* eLast = sm.tcol;                       // [n][ldl]
    double* eLead = eLast + (size_t)n * ldl;       // [n][ldr]

    const long long loc0 = (long long)tile * CBO_SWEEP_TILE;
    const long long left = S.g_count - loc0;
    const int cnt = left < CBO_SWEEP_TILE ? (int)left : CBO_SWEEP_TILE;
    const long long gidx0 = S.g_begin + loc0;
    const long long row_first = S.points ? gidx0 : gidx0 / p_last;   // first leading row of the item

    if (!cached) {
        for (int e = tid; e < n * n; e += kSweepThreads) {
            const int i = e / n, j = e % n;
            if (j <= i) sm.Lp[i * (i + 1) / 2 + j] = j < i ? S.L[e] : 1.0 / S.L[e];   // the diagonal is staged as its reciprocal
        }
        for (int i = tid; i < n; i += kSweepThreads) {
            sm.al[i] = S.alpha[i];
            sm.sv[i] = causal ? S.sqrt_v_int[i] : 0.0;
        }
        for (int i = tid; i < n * d; i += kSweepThreads) sm.xs[i] = S.x_int[i] * il;
        if (sep) {
            const double* __restrict__ gl = S.grid[d - 1];
            for (int e = tid; e < n * p_last; e += kSweepThreads) {
                const int i = e / p_last, j = e - i * p_last;
                const double q = (gl[j] - S.x_int[i * d + d - 1]) * il;
                eLast[i * ldl + j] = exp(-0.5 * (q * q));
            }
            const long long last_row = (gidx0 + cnt - 1) / p_last;
            const int nrows = (int)(last_row - row_first) + 1;
            for (int e = tid; e < n * nrows; e += kSweepThreads) {
                const int i = e / nrows, r = e - i * nrows;
                long long rr = row_first + r;
                double r2 = 0.0;
                for (int k = d - 2; k >= 0; --k) {
                    const long long pk = S.p[k];
                    const double q = (S.grid[k][(int)(rr % pk)] - S.x_int[i * d + k]) * il;
                    r2 = fma(q, q, r2);
                    rr /= pk;
                }
                eLead[i * ldr + r] = __dmul_rn(s2, exp(-0.5 * r2));
            }
        }
        __syncthreads();
    }

    double val = -DBL_MAX * 2.0;  // -inf
    long long idx = LLONG_MAX;
    int n_nan = 0;
    // this thread's candidates: loc0 + tid, + 128, ...; (row, j) = (leading row, fastest index) advance without divisions
    long long row = row_first;
    int jj = 0;
    if (!S.points) {
        const long long g = gidx0 + tid;
        row = g / p_last;
        jj = (int)(g - row * p_last);
    }
    const bool need_x = (!cached && !sep) || S.cost_variable;
#pragma unroll 1
    for (int c = tid; c < cnt; c += kSweepThreads) {
        const long long loc = loc0 + c, gidx = gidx0 + c;
        double x[CBO_MAX_D];
#pragma unroll
        for (int k = 0; k < CBO_MAX_D; ++k) x[k] = 0.0;
        if (need_x) candidate_x(S, d, gidx, row, jj, x);
        double mu, var;
        if (cached) {
            mu = S.mu[loc];
            var = S.var[loc];
        } else {
            const double vg = causal ? S.v[loc] : 0.0;
            const double mg = causal ? S.m[loc] : 0.0;
            const double svg = causal ? sqrt(vg) : 0.0;
            double ss;
            if constexpr (SEP) posterior_sep<NREG>(sm, n, eLast + jj, ldl, eLead + (int)(row - row_first), ldr, svg, mu, ss);
            else {
                double xl[CBO_MAX_D];
#pragma unroll
                for (int k = 0; k < CBO_MAX_D; ++k) xl[k] = x[k] * il;
                posterior_at<NREG>(sm, n, d, xl, svg, s2, tid, mu, ss);
            }
            mu += mg;
            var = surrogate_var(s2, vg, ss);
            if (S.mu) S.mu[loc] = mu;
            if (S.var) S.var[loc] = var;
        }
        const double ei = expected_improvement(best, mu, var, task_sign).ei;
        const double acq = ei / candidate_cost(S, d, x);
        if (S.ei) S.ei[loc] = ei;
        if (S.acq) S.acq[loc] = acq;
        if (acq != acq) ++n_nan;
        else if (better(acq, gidx, val, idx)) { val = acq; idx = gidx; }
        jj += kSweepThreads;
        while (jj >= p_last && !S.points) { jj -= p_last; ++row; }
    }
    // first-argmax over the tile
    cta_first_argmax<kSweepThreads>(val, idx, n_nan);
    if (tid == 0) {
        cbo_set_best b;
        b.value = val; b.index = idx; b.n_nan = n_nan; b.reserved = 0;
        tile_best[blockIdx.x] = b;
    }
}

// ---- 16 < n <= 48: |L^-1 k*|^2 on the FP64 tensor pipe --------------------------------------------------------------------
// The forward substitution costs n^2/2 FMAs per candidate with one broadcast LDS each: at n = 45 the LSU, not the FP64 pipe,
// set the pace (ncu, profiles/r02_k3_sweep_refresh_*: FP64 pipe 29 %, LSU wavefronts 33 %, 3 warps per scheduler waiting on
// each other's loads).  Here t = W k*, W = L^-1 (K2 leaves L^-T in the upper triangle of `L`), is a GEMM over candidates on
// DMMA.8x8x4: a warp takes 32 consecutive candidates as four groups of 8 rows; per group the A fragments are the candidate's
// k* values (lane (r, q) evaluates k*_j for j = 4 ks + q: two table loads and one FMA on a tensor grid), the B fragments are
// the 8 x 4 blocks of W on and below the diagonal, staged once per item in fragment order (conflict-free LDS.64, one per TWO
// DMMAs: two groups share each load), and the accumulators are t itself: ss = sum of squares, reduced over the 4 lanes of a
// row; mu = k*.alpha rides along as 12 FMAs.  42 DMMAs per 8 candidates at n = 48 (36.75 if the triangle were cut exactly).
// Lane 4 r + q then finishes candidate 8 q + r of the warp's 32 (EI, cost, argmax): the group results it needs are already
// in its own registers.  L^-1 k* has the forward error of a triangular solve with the same factor (n eps |W| |k*|); on the
// shipped data the variance moves by <= 5e-9 of its parity floor against substitution (measured in NumPy on the golden
// fixtures, DESIGN.md K3).
constexpr int kMmaNB = kSweepMmaMaxN / 8;             // 8-row output blocks of t
constexpr int kMmaKS = kSweepMmaMaxN / 4;             // k4 steps
constexpr int kMmaSlots = kMmaNB * (kMmaNB + 1);      // fragments of W's block lower triangle: block ib has 2 ib + 2 of them
__host__ __device__ inline int sweep_mma_lead_rows(int p_last, int chunk) { return chunk * CBO_SWEEP_TILE / p_last + 2; }
constexpr int kMmaMaxChunk = 64;                      // <= kMmaThreads (one thread per neutral slot), bounds the lead-row table
__host__ __device__ inline int sweep_mma_ldl(int p_last) { return ((p_last + 3) / 8) * 8 + 4; }   // = 4 (mod 8): 4 rows x 4 columns of a half-warp hit 16 banks

constexpr int kMmaThreads = 512;                     // 16 warps, one CTA per SM: an item is two rounds of 16 warp passes
template <bool SEP>
__global__ void __launch_bounds__(kMmaThreads, 1)
sweep_mma_kernel(const cbo_set_desc* __restrict__ sets, int num_sets, double best, double task_sign,
                 cbo_set_best* __restrict__ tile_best, int chunk) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    int tile;
    const int s = find_item(sets, num_sets, kItemsSweep, blockIdx.x, tile);
    const cbo_set_desc& S = sets[s];
    if (sweep_class(S) != (SEP ? kClsMmaSep : kClsMma)) return;       // another launch's set
    // `chunk` consecutive items of a set are swept by the CTA of the first one: the per-item staging (n (p_last + rows) exp for
    // the k* tables, the fragments of L^-1) was 14 % of the kernel with one item per CTA, and a launch of few long-lived CTAs
    // has no wave quantisation.  The chunk's argmax goes to its first item's slot, the other slots get the neutral element.
    if (tile % chunk != 0) return;
    const int n = S.n_int, d = S.d, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int r = lane >> 2, q = lane & 3;
    const bool causal = S.causal != 0;
    const auto [s2, il] = surrogate_hyper(S);
    const int p_last = S.points ? 1 : S.p[d - 1];
    const int nb = (n + 7) >> 3, ksn = (n + 3) >> 2;

    double* Wf = reinterpret_cast<double*>(smem_raw);          // [slot][lane]
    double* al = Wf + kMmaSlots * 32;
    double* sv = al + kSweepMmaMaxN;
    double* xs = sv + kSweepMmaMaxN;                            // n x d
    double* eLast = xs + kSweepMmaMaxN * CBO_MAX_D;             // [n][ldl]
    const int ldl = sweep_mma_ldl(p_last), ldr = sweep_mma_lead_rows(p_last, chunk) | 1;
    const int n4 = 4 * ksn;                                     // table rows: n rounded up to whole k4 steps, the extra rows zero
    double* eLead = eLast + (size_t)n4 * ldl;                   // [n4][ldr]

    const long long loc0 = (long long)tile * CBO_SWEEP_TILE;
    const long long left = S.g_count - loc0;
    const int cnt = left < (long long)chunk * CBO_SWEEP_TILE ? (int)left : chunk * CBO_SWEEP_TILE;
    const long long gidx0 = S.g_begin + loc0;
    const long long row_first = S.points ? gidx0 : gidx0 / p_last;
    const int off0 = S.points ? 0 : (int)(gidx0 - row_first * p_last);

    for (int e = tid; e < nb * (nb + 1) * 32; e += kMmaThreads) {
        const int slot = e >> 5, l = e & 31;
        int ib = 0;
        while ((ib + 1) * (ib + 2) <= slot) ++ib;
        const int i = 8 * ib + (l >> 2), j = 4 * (slot - ib * (ib + 1)) + (l & 3);
        double w = 0.0;
        if (i < n && j <= i) w = (j == i) ? 1.0 / S.L[(size_t)i * n + i] : S.L[(size_t)j * n + i];
        Wf[e] = w;
    }
    for (int i = tid; i < n4; i += kMmaThreads) {
        al[i] = i < n ? S.alpha[i] : 0.0;
        sv[i] = (causal && i < n) ? S.sqrt_v_int[i] : 0.0;
    }
    for (int i = tid; i < n * d; i += kMmaThreads) xs[i] = S.x_int[i] * il;
    if (SEP) {
        const double* __restrict__ gl = S.grid[d - 1];
        for (int e = tid; e < n4 * p_last; e += kMmaThreads) {
            const int i = e / p_last, j = e - i * p_last;
            double v = 0.0;
            if (i < n) {
                const double t = (gl[j] - S.x_int[i * d + d - 1]) * il;
                v = exp(-0.5 * (t * t));
            }
            eLast[i * ldl + j] = v;
        }
        const long long last_row = (gidx0 + cnt - 1) / p_last;
        const int nrows = (int)(last_row - row_first) + 1;
        for (int e = tid; e < n4 * nrows; e += kMmaThreads) {
            const int i = e / nrows, rw = e - i * nrows;
            double v = 0.0;
            if (i < n) {
                long long rr = row_first + rw;
                double r2 = 0.0;
                for (int k = d - 2; k >= 0; --k) {
                    const long long pk = S.p[k];
                    const double t = (S.grid[k][(int)(rr % pk)] - S.x_int[i * d + k]) * il;
                    r2 = fma(t, t, r2);
                    rr /= pk;
                }
                v = __dmul_rn(s2, exp(-0.5 * r2));
            }
            eLead[i * ldr + rw] = v;
        }
    }
    __syncthreads();

    double val = -DBL_MAX * 2.0;  // -inf
    long long idx = LLONG_MAX;
    int n_nan = 0;
#pragma unroll 1
    for (int c0 = warp * 32; c0 < cnt; c0 += kMmaThreads) {
        // this lane's own candidate (the one it finishes): 8 q + r of the warp's 32; a dead tail lane shadows the last live one
        const int c_own = c0 + 8 * q + r;
        const bool live = c_own < cnt;
        const int c = live ? c_own : cnt - 1;
        const long long loc = loc0 + c, gidx = gidx0 + c;
        const double vg = causal ? S.v[loc] : 0.0;
        const double mg = causal ? S.m[loc] : 0.0;
        const double svg = causal ? sqrt(vg) : 0.0;
        int lrow = 0, jj = 0;
        double x[CBO_MAX_D];
#pragma unroll
        for (int k = 0; k < CBO_MAX_D; ++k) x[k] = 0.0;
        if (!S.points) {
            const unsigned off = (unsigned)(off0 + c);
            lrow = (int)(off / (unsigned)p_last);
            jj = (int)(off - (unsigned)lrow * (unsigned)p_last);
        }
        if (!SEP || S.cost_variable) candidate_x(S, d, gidx, row_first + lrow, jj, x);
        double mu = 0.0, ss = 0.0;
#pragma unroll 1
        for (int g = 0; g < 4; ++g) {
            double a[kMmaKS], acc[kMmaNB][2];
            const int src = (lane & ~3) | g;      // the lane that owns candidate 8 g + r
            const double svg_g = __shfl_sync(0xffffffffu, svg, src);
            double mp = 0.0;
            if (SEP) {
                const double* __restrict__ eR = eLead + __shfl_sync(0xffffffffu, lrow, src);
                const double* __restrict__ eL = eLast + __shfl_sync(0xffffffffu, jj, src);
#pragma unroll
                for (int ks = 0; ks < kMmaKS; ++ks) {
                    a[ks] = 0.0;
                    if (ks < ksn) {       // rows n .. n4 - 1 of the tables, of sv and of alpha are zero: k*_j = 0 there
                        const int j = 4 * ks + q;
                        a[ks] = fma(eR[j * ldr], eL[j * ldl], sv[j] * svg_g);
                        mp = fma(a[ks], al[j], mp);
                    }
                }
            } else {
                double xg[CBO_MAX_D];
#pragma unroll
                for (int k = 0; k < CBO_MAX_D; ++k) xg[k] = __shfl_sync(0xffffffffu, x[k], src) * il;
#pragma unroll
                for (int ks = 0; ks < kMmaKS; ++ks) {
                    a[ks] = 0.0;
                    if (ks < ksn) {
                        const int j = 4 * ks + q, jc = j < n ? j : n - 1;
                        double r2 = 0.0;
#pragma unroll
                        for (int k = 0; k < CBO_MAX_D; ++k) {
                            if (k < d) { const double t = xg[k] - xs[jc * d + k]; r2 = fma(t, t, r2); }
                        }
                        const double kv = surrogate_k(r2, sv[jc], svg_g, s2);
                        a[ks] = j < n ? kv : 0.0;
                        mp = fma(a[ks], al[jc], mp);
                    }
                }
            }
            double sp = 0.0;
#pragma unroll
            for (int ib = 0; ib < kMmaNB; ++ib) acc[ib][0] = acc[ib][1] = 0.0;
            // k4 step outermost: consecutive DMMAs go to different accumulators (issued block by block they formed dependent
            // chains of up to 12 and the warp waited out the pipe latency 42 times per group: DMMA pipe 38 % active)
            // (the B fragments of step ks + 1 are loaded before the DMMAs of step ks are issued)
            double bn[kMmaNB];
#pragma unroll
            for (int ib = 0; ib < kMmaNB; ++ib) bn[ib] = ib < nb ? Wf[(ib * (ib + 1)) * 32 + lane] : 0.0;
#pragma unroll
            for (int ks = 0; ks < kMmaKS; ++ks) {
                if (ks < ksn) {
                    double bc[kMmaNB];
#pragma unroll
                    for (int ib = 0; ib < kMmaNB; ++ib) bc[ib] = bn[ib];
                    if (ks + 1 < ksn) {
#pragma unroll
                        for (int ib = (ks + 1) >> 1; ib < kMmaNB; ++ib)
                            if (ib < nb) bn[ib] = Wf[(ib * (ib + 1) + ks + 1) * 32 + lane];
                    }
#pragma unroll
                    for (int ib = ks >> 1; ib < kMmaNB; ++ib)
                        if (ib < nb) dmma884(acc[ib][0], acc[ib][1], a[ks], bc[ib]);
                }
            }
#pragma unroll
            for (int ib = 0; ib < kMmaNB; ++ib) sp = fma(acc[ib][0], acc[ib][0], fma(acc[ib][1], acc[ib][1], sp));
            mp += __shfl_xor_sync(0xffffffffu, mp, 1);
            sp += __shfl_xor_sync(0xffffffffu, sp, 1);
            mp += __shfl_xor_sync(0xffffffffu, mp, 2);
            sp += __shfl_xor_sync(0xffffffffu, sp, 2);
            if (q == g) { mu = mp; ss = sp; }
        }
        mu += mg;
        const double var = surrogate_var(s2, vg, ss);
        if (live) {
            if (S.mu) S.mu[loc] = mu;
            if (S.var) S.var[loc] = var;
        }
        const double ei = expected_improvement(best, mu, var, task_sign).ei;
        const double acq = ei / candidate_cost(S, d, x);
        if (live) {
            if (S.ei) S.ei[loc] = ei;
            if (S.acq) S.acq[loc] = acq;
            if (acq != acq) ++n_nan;
            else if (better(acq, gidx, val, idx)) { val = acq; idx = gidx; }
        }
    }
    // first-argmax over the tile
    cta_first_argmax<kMmaThreads>(val, idx, n_nan);
    if (tid == 0) {
        cbo_set_best b;
        b.value = val; b.index = idx; b.n_nan = n_nan; b.reserved = 0;
        tile_best[blockIdx.x] = b;
    }
    const int items_here = (cnt + CBO_SWEEP_TILE - 1) / CBO_SWEEP_TILE;
    if (tid > 0 && tid < items_here) {
        cbo_set_best b;
        b.value = -DBL_MAX * 2.0; b.index = LLONG_MAX; b.n_nan = 0; b.reserved = 0;
        tile_best[blockIdx.x + tid] = b;
    }
}

// ---- cached posterior: EI refresh only ------------------------------------------------------------------------------------
// After an intervention every set but the refitted one keeps mu / var (cbo_set_desc.posterior_cached) and only EI moves with
// the incumbent: 16 B per candidate and ~150 FP64 operations (sqrt, two divisions, exp, erfc).  Inside sweep_kernel's
// one-candidate-at-a-time loop that chain was latency-bound (32 us per 1e6 candidates, 0.5 TB/s); here a thread carries
// kEiUnroll independent candidates through it.  EI is surrogate.cuh's expected_improvement(), as in sweep_kernel: the same bits.
constexpr int kEiUnroll = 4;
__global__ void __launch_bounds__(kSweepThreads, 6)
ei_refresh_kernel(const cbo_set_desc* __restrict__ sets, int num_sets, double best, double task_sign,
                  cbo_set_best* __restrict__ tile_best) {
    int tile;
    const int s = find_item(sets, num_sets, kItemsSweep, blockIdx.x, tile);
    const cbo_set_desc& S = sets[s];
    if (sweep_class(S) != kClsCached) return;
    const int tid = threadIdx.x;
    const long long loc0 = (long long)tile * CBO_SWEEP_TILE;
    const long long left = S.g_count - loc0;
    const int cnt = left < CBO_SWEEP_TILE ? (int)left : CBO_SWEEP_TILE;
    const long long gidx0 = S.g_begin + loc0;
    const double* __restrict__ gmu = S.mu + loc0;
    const double* __restrict__ gvar = S.var + loc0;
    double* __restrict__ gei = S.ei ? S.ei + loc0 : nullptr;
    double* __restrict__ gacq = S.acq ? S.acq + loc0 : nullptr;
    const double cost = S.cost_fix;
    double val = -DBL_MAX * 2.0;  // -inf
    long long idx = LLONG_MAX;
    int n_nan = 0;
#pragma unroll 1
    for (int c0 = tid; c0 < cnt; c0 += kSweepThreads * kEiUnroll) {
        double mu[kEiUnroll], var[kEiUnroll], ei[kEiUnroll], acq[kEiUnroll];
#pragma unroll
        for (int u = 0; u < kEiUnroll; ++u) {
            const int c = c0 + u * kSweepThreads;
            mu[u] = c < cnt ? gmu[c] : 0.0;
            var[u] = c < cnt ? gvar[c] : 1.0;
        }
#pragma unroll
        for (int u = 0; u < kEiUnroll; ++u) {
            ei[u] = expected_improvement(best, mu[u], var[u], task_sign).ei;
            acq[u] = ei[u] / cost;
        }
#pragma unroll
        for (int u = 0; u < kEiUnroll; ++u) {
            const int c = c0 + u * kSweepThreads;
            if (c < cnt) {
                if (gei) gei[c] = ei[u];
                if (gacq) gacq[c] = acq[u];
                if (acq[u] != acq[u]) ++n_nan;
                else if (better(acq[u], gidx0 + c, val, idx)) { val = acq[u]; idx = gidx0 + c; }
            }
        }
    }
    cta_first_argmax<kSweepThreads>(val, idx, n_nan);
    if (tid == 0) {
        cbo_set_best b;
        b.value = val; b.index = idx; b.n_nan = n_nan; b.reserved = 0;
        tile_best[blockIdx.x] = b;
    }
}

// per-set reduction over the set's tiles (one CTA per set, fixed order)
__global__ void __launch_bounds__(256)
set_reduce_kernel(const cbo_set_desc* __restrict__ sets, int num_sets, const cbo_set_best* __restrict__ tile_best,
                  cbo_set_best* __restrict__ set_best) {
    const int s = blockIdx.x, tid = threadIdx.x;
    long long base = 0;
    for (int x = 0; x < s; ++x) base += host_items(sets[x], kItemsSweep);
    const long long cnt = host_items(sets[s], kItemsSweep);
    double val = -DBL_MAX * 2.0;
    long long idx = LLONG_MAX;
    int nn = 0;
    for (long long t = tid; t < cnt; t += 256) {
        const cbo_set_best b = tile_best[base + t];
        if (better(b.value, b.index, val, idx)) { val = b.value; idx = b.index; }
        nn += b.n_nan;
    }
    cta_first_argmax<256>(val, idx, nn);
    if (tid == 0) {
        cbo_set_best b;
        b.value = val; b.index = (idx == LLONG_MAX) ? -1 : idx; b.n_nan = nn; b.reserved = 0;
        set_best[s] = b;
    }
}

// gathered[rank][set] -> set_best[set] (when num_ranks > 0) and the global result.
// CBO.select_next_intervention (CBO.py:275-276): first set attaining the maximum.
__global__ void __launch_bounds__(128)
combine_kernel(const cbo_set_best* __restrict__ gathered, int num_ranks, int num_sets, cbo_set_best* __restrict__ set_best,
               cbo_sweep_result* __restrict__ result) {
    for (int s = threadIdx.x; s < num_sets && num_ranks > 0; s += blockDim.x) {
        double val = -DBL_MAX * 2.0;
        long long idx = LLONG_MAX;
        int nn = 0;
        for (int r = 0; r < num_ranks; ++r) {
            const cbo_set_best b = gathered[(size_t)r * num_sets + s];
            const long long bi = b.index < 0 ? LLONG_MAX : b.index;
            if (better(b.value, bi, val, idx)) { val = b.value; idx = bi; }
            nn += b.n_nan;
        }
        cbo_set_best o;
        o.value = val; o.index = (idx == LLONG_MAX) ? -1 : idx; o.n_nan = nn; o.reserved = 0;
        set_best[s] = o;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        cbo_sweep_result r;
        r.value = -DBL_MAX * 2.0; r.index = -1; r.set = -1; r.n_nan = 0;
        for (int s = 0; s < num_sets; ++s) {
            const cbo_set_best b = set_best[s];
            r.n_nan += b.n_nan;
            if (b.index >= 0 && (r.set < 0 || b.value > r.value)) { r.value = b.value; r.index = b.index; r.set = s; }
        }
        *result = r;
    }
}

int sweep_impl(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, double best, int task_sign,
               cbo_set_best* d_tile_best, cbo_set_best* d_set_best, cbo_sweep_result* d_result, cudaStream_t st) {
    CBO_REQUIRE(task_sign == 1 || task_sign == -1, "cbo_sweep: task_sign must be +1 ('min') or -1 ('max')");
    CBO_REQUIRE(d_tile_best && d_set_best && d_result, "cbo_sweep: NULL output pointer");
    long long total = 0;
    // per launch class (sweep_class): is there a set for it, its largest n_int, and its k* tables / workspace in doubles
    bool any[kNumSweepClasses] = {};
    int nmax[kNumSweepClasses];
    size_t tab[kNumSweepClasses] = {};
    for (int c = 0; c < kNumSweepClasses; ++c) nmax[c] = 1;
    for (int s = 0; s < num_sets; ++s) {
        const cbo_set_desc& S = h_sets[s];
        CBO_REQUIRE(S.n_int >= 1 && S.n_int <= CBO_MAX_NINT, "cbo_sweep: set %d n_int=%d outside [1,%d]", s, S.n_int, CBO_MAX_NINT);
        CBO_REQUIRE(S.L && S.alpha && S.x_int, "cbo_sweep: set %d has a NULL posterior pointer", s);
        CBO_REQUIRE(!S.posterior_cached || (S.mu && S.var), "cbo_sweep: set %d is marked posterior_cached without mu/var arrays", s);
        CBO_REQUIRE(!S.causal || (S.m && S.v && S.sqrt_v_int), "cbo_sweep: causal set %d needs m/v/sqrt_v_int", s);
        for (int k = 0; k < (S.points ? 0 : S.d); ++k) CBO_REQUIRE(S.grid[k], "cbo_sweep: set %d grid[%d] is NULL", s, k);
        total += host_items(S, kItemsSweep);
        if (S.g_count <= 0) continue;
        const int c = sweep_class(S);
        any[c] = true;
        if (!S.posterior_cached && S.n_int > nmax[c]) nmax[c] = S.n_int;
        size_t t = 0;
        if (c == kClsFmaSep) t = (size_t)S.n_int * ((S.p[S.d - 1] | 1) + (sweep_lead_rows(S) | 1));
        if (c == kClsGeneric) t = (size_t)S.n_int * kSweepThreads;
        if (t > tab[c]) tab[c] = t;
    }
    CBO_REQUIRE(total < 2147483647LL, "cbo_sweep: too many work items");
    // chunk length of the tensor-pipe launch: its items spread once over the SMs, within the shared memory the longest
    // lead-row table needs
    int chunk = 1;
    const size_t mma_base = ((size_t)kMmaSlots * 32 + 2 * kSweepMmaMaxN + (size_t)kSweepMmaMaxN * CBO_MAX_D) * sizeof(double);
    if (any[kClsMmaSep]) {
        int dev = 0, sms = 0;
        CBO_CUDA(cudaGetDevice(&dev));
        CBO_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        long long items = 0;
        for (int s = 0; s < num_sets; ++s)
            if (h_sets[s].g_count > 0 && sweep_class(h_sets[s]) == kClsMmaSep) items += host_items(h_sets[s], kItemsSweep);
        chunk = (int)((items + sms - 1) / sms);
        if (chunk > kMmaMaxChunk) chunk = kMmaMaxChunk;
        for (;; --chunk) {
            tab[kClsMmaSep] = 0;
            for (int s = 0; s < num_sets; ++s) {
                const cbo_set_desc& S = h_sets[s];
                if (S.g_count <= 0 || sweep_class(S) != kClsMmaSep) continue;
                const int pl = S.p[S.d - 1];
                const size_t t = (size_t)((S.n_int + 3) & ~3) * (sweep_mma_ldl(pl) + (sweep_mma_lead_rows(pl, chunk) | 1));
                if (t > tab[kClsMmaSep]) tab[kClsMmaSep] = t;
            }
            if (chunk == 1 || mma_base + tab[kClsMmaSep] * sizeof(double) <= 160 * 1024) break;
        }
    }
    if (total > 0) {
        auto fma_smem = [&](int c) {
            return ((size_t)nmax[c] * (nmax[c] + 1) / 2 + 2 * (size_t)nmax[c] + (size_t)nmax[c] * CBO_MAX_D + tab[c]) * sizeof(double);
        };
#define CBO_SWEEP_LAUNCH(kern, threads, smem, ...)                                                                           \
    do {                                                                                                       \
        if ((smem) > 48 * 1024) CBO_CUDA(allow_dynamic_smem(kern, (smem)));                                    \
        kern<<<(unsigned)total, (threads), (smem), st>>>(d_sets, num_sets, best, (double)task_sign, d_tile_best __VA_ARGS__); \
        note_launch();                                                                                         \
        CBO_CUDA(cudaGetLastError());                                                                          \
    } while (0)
        if (any[kClsFmaSep]) CBO_SWEEP_LAUNCH((sweep_kernel<16, true>), kSweepThreads, fma_smem(kClsFmaSep));
        if (any[kClsMmaSep]) CBO_SWEEP_LAUNCH((sweep_mma_kernel<true>), kMmaThreads, mma_base + tab[kClsMmaSep] * sizeof(double), , chunk);
        if (any[kClsFma]) CBO_SWEEP_LAUNCH((sweep_kernel<16, false>), kSweepThreads, fma_smem(kClsFma));
        if (any[kClsMma]) CBO_SWEEP_LAUNCH((sweep_mma_kernel<false>), kMmaThreads, mma_base, , 1);
        if (any[kClsGeneric]) CBO_SWEEP_LAUNCH((sweep_kernel<0, false>), kSweepThreads, fma_smem(kClsGeneric));
        if (any[kClsCached]) CBO_SWEEP_LAUNCH(ei_refresh_kernel, kSweepThreads, (size_t)0);
#undef CBO_SWEEP_LAUNCH
    }
    set_reduce_kernel<<<num_sets, 256, 0, st>>>(d_sets, num_sets, d_tile_best, d_set_best);
    note_launch();
    CBO_CUDA(cudaGetLastError());
    combine_kernel<<<1, 128, 0, st>>>(nullptr, 0, num_sets, d_set_best, d_result);
    note_launch();
    CBO_CUDA(cudaGetLastError());
    return 0;
}

int argmax_combine_impl(const cbo_set_best* d_gathered, int num_ranks, int num_sets, cbo_set_best* d_set_best,
                        cbo_sweep_result* d_result, cudaStream_t st) {
    CBO_REQUIRE(d_gathered && num_ranks >= 1 && num_sets >= 1, "cbo_argmax_combine: bad arguments");
    combine_kernel<<<1, 128, 0, st>>>(d_gathered, num_ranks, num_sets, d_set_best, d_result);
    note_launch();
    CBO_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace cbo
