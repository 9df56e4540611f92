// The per-set surrogate GP, defined once for every kernel that evaluates it: the fit (K2, posterior_fit.cu), the sweep
// (K3 / K4, sweep.cu), the gradients and refinement (K7, refine.cu) and the hyper-parameter search (K8, posterior_hyper.cu).
//   k(x_i, x_j) = s2 exp(-.5 |x_i - x_j|^2 / l^2) + sv_i sv_j     sv = sqrt(v) of the causal prior, 0 for a non-causal set
//   Ky          = K + kSurrogateDiag I,  L = jitchol(Ky)            (the likelihood's noise 1e-10 and the 1e-8 GPy's exact inference adds)
//   var(x)      = (s2 + v(x)) - |L^-1 k*|^2 + noise
//   EI          = sd (u Phi(u) + phi(u)),  u = (best - mu) / sd, negated for task 'max';  acq = EI / cost(x)
// A change to the model (its noise, another kernel) is made here and reaches every kernel at once.
// K8 runs the Gram and jitchol below.  For speed it keeps its own substitutions (by 1 / L_ii) and its own L^-1 loop: its
// alpha and L^-1 may differ from what K2's routines would give at rounding level.
#pragma once
#include "cbo_common.cuh"

namespace cbo {

// ---- model -----------------------------------------------------------------------------------------------------------------
struct SurrogateHyper {
    double s2, il;     // variance and 1 / lengthscale
};
// cbo_set_desc.hyper = (s2, l), or the reference's (1, 1) when it is NULL (a scaling by 1.0 is exact: the same bits as l = s2 = 1)
__device__ __forceinline__ SurrogateHyper surrogate_hyper(const cbo_set_desc& S) {
    return S.hyper ? SurrogateHyper{S.hyper[0], 1.0 / S.hyper[1]} : SurrogateHyper{1.0, 1.0};
}

// r^2 / l^2 between rows i and j of the n x d coordinates xs, from coordinate differences (no cancellation)
__device__ __forceinline__ double surrogate_r2(const double* xs, int i, int j, int d, double il) {
    double r2 = 0.0;
    for (int k = 0; k < d; ++k) {
        const double t = (xs[i * d + k] - xs[j * d + k]) * il;
        r2 += t * t;
    }
    return r2;
}
// s2 exp(-.5 r^2), r^2 already scaled by 1 / l^2
__device__ __forceinline__ double surrogate_rbf(double r2, double s2) { return __dmul_rn(s2, exp(-0.5 * r2)); }
__device__ __forceinline__ double surrogate_k(double r2, double svi, double svj, double s2) {
    return fma(svi, svj, surrogate_rbf(r2, s2));
}
constexpr double kSurrogateDiag = 1e-10 + 1e-8;     // added to the diagonal of the Gram
// posterior variance from the prior variance v(x) (0 for a non-causal set) and ss = |L^-1 k*|^2
__device__ __forceinline__ double surrogate_var(double s2, double v, double ss) { return ((s2 + v) - ss) + 1e-10; }

// ---- fit: Gram, Cholesky, solves, L^-T (one CTA of THREADS threads; A is n x n with row pitch ld, n <= 128) ------------------
// Ky into the lower triangle of A, then L = jitchol(Ky) in place with GPy's rule: plain Cholesky first; on a non-positive pivot
// retry with jitter = mean(diag Ky) 1e-6 10^t, t = 0..4.  Returns the retries (0..5), or -1 when Ky is not positive definite
// even then.  On success A's lower triangle is L, dsq[i] = L_ii and rinv[i] = 1 / L_ii.  xs are the n x d coordinates, sv the
// sqrt(v) factors.  Every thread reads the same pivot, so the failure branch is uniform over the CTA.
template <int THREADS>
__device__ __forceinline__ int surrogate_jitchol(double* A, int ld, const double* xs, const double* sv, int n, int d,
                                                 SurrogateHyper h, double* dsq, double* rinv) {
    __shared__ double diag_mean;
    const int tid = threadIdx.x;
    int tries = 0;
    double jitter = 0.0;
    for (;;) {
        for (int e = tid; e < n * n; e += THREADS) {
            const int i = e / n, j = e - i * n;
            if (j > i) continue;
            double kij = surrogate_k(surrogate_r2(xs, i, j, d, h.il), sv[i], sv[j], h.s2);
            if (i == j) kij += kSurrogateDiag + jitter;
            A[i * ld + j] = kij;
        }
        __syncthreads();
        if (tries == 0) {  // mean of the diagonal of Ky, the scale of GPy's jitter
            if (tid == 0) {
                double t = 0.0;
                for (int i = 0; i < n; ++i) t += A[i * ld + i];
                diag_mean = t / n;
            }
            __syncthreads();
        }
        // Right-looking Cholesky, lower.  Every thread forms 1 / sqrt(pivot) itself; the diagonal is written after the loop
        // (nobody waits for thread 0, two barriers per column instead of three); the trailing update walks a 16 x 16 thread
        // grid (no integer division per element).  The arithmetic is LAPACK's: scale the column, then subtract products of
        // scaled entries.
        bool failed = false;
        for (int j = 0; j < n; ++j) {
            const double piv = A[j * ld + j];
            if (!(piv > 0.0)) { failed = true; break; }
            const double sq = sqrt(piv);
            const double inv = 1.0 / sq;
            if (tid == 0) dsq[j] = sq;
            for (int i = j + 1 + tid; i < n; i += THREADS) A[i * ld + j] *= inv;
            __syncthreads();
            for (int i = j + 1 + (tid >> 4); i < n; i += THREADS / 16)
                for (int k = j + 1 + (tid & 15); k <= i; k += 16) A[i * ld + k] -= A[i * ld + j] * A[k * ld + j];
            __syncthreads();
        }
        if (!failed) break;
        __syncthreads();     // (a thread may still be reading the failing pivot while the next Gram is written)
        if (tries == 5) return -1;
        jitter = (tries == 0) ? diag_mean * 1e-6 : jitter * 10.0;
        ++tries;
    }
    for (int j = tid; j < n; j += THREADS) {
        A[j * ld + j] = dsq[j];
        rinv[j] = 1.0 / dsq[j];
    }
    __syncthreads();
    return tries;
}

// z <- L^-1 z and z <- L^-T z in one warp with no CTA barriers: lane l owns rows l, l + 32, l + 64, l + 96 in registers, the
// pivot row's value travels by shuffle.  L is the lower triangle of A, dsq[j] = L_jj.
__device__ __forceinline__ double warp_own_row(const double (&z)[4], int j) {
    const int slot = j >> 5;
    return slot == 0 ? z[0] : slot == 1 ? z[1] : slot == 2 ? z[2] : z[3];
}
__device__ __forceinline__ void warp_solve_lower(const double* A, int ld, const double* dsq, int n, double (&z)[4]) {
    const int lane = threadIdx.x & 31;
    for (int j = 0; j < n; ++j) {
        const double zj = __shfl_sync(0xffffffffu, warp_own_row(z, j) / dsq[j], j & 31);
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int i = lane + 32 * r;
            if (i == j) z[r] = zj;
            else if (i > j && i < n) z[r] = fma(-A[i * ld + j], zj, z[r]);
        }
    }
}
__device__ __forceinline__ void warp_solve_upper(const double* A, int ld, const double* dsq, int n, double (&z)[4]) {
    const int lane = threadIdx.x & 31;
    for (int j = n - 1; j >= 0; --j) {
        const double aj = __shfl_sync(0xffffffffu, warp_own_row(z, j) / dsq[j], j & 31);
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int i = lane + 32 * r;
            if (i == j) z[r] = aj;
            else if (i < j) z[r] = fma(-A[j * ld + i], aj, z[r]);
        }
    }
}

// W = L^-1 into the strict upper triangle of A, transposed (column c of W is row c of the upper triangle; the diagonal of W is
// rinv): W[i][c] = -(sum_{c <= j < i} L[i][j] W[j][c]) / L[i][i].  Four lanes per column split every dot product and combine by a
// fixed butterfly, THREADS / 4 columns at once (a single thread per column made the inverse a 20 us chain at n = 45).
template <int THREADS>
__device__ __forceinline__ void surrogate_lower_inverse(double* A, int ld, const double* rinv, int n) {
    constexpr int kCols = THREADS / 4;
    const int tid = threadIdx.x, sub = tid & 3;
    for (int c = tid >> 2; c < (n + kCols - 1) / kCols * kCols; c += kCols) {        // warp-uniform trip count
        const bool col = c < n;
        const double wcc = col ? rinv[c] : 0.0;
        for (int i = (c & ~7) + 1; i < n; ++i) {      // row i of column c, i > c (a warp holds columns 8 w .. 8 w + 7)
            double a0 = 0.0;
            if (col && i > c) {
                for (int j = c + 1 + sub; j < i; j += 4) a0 = fma(A[i * ld + j], A[c * ld + j], a0);
                if (sub == 0) a0 = fma(A[i * ld + c], wcc, a0);
            }
            a0 += __shfl_xor_sync(0xffffffffu, a0, 1);
            a0 += __shfl_xor_sync(0xffffffffu, a0, 2);
            if (col && i > c && sub == 0) A[c * ld + i] = -a0 * rinv[i];
            __syncwarp();
        }
    }
    __syncthreads();
}

// ---- acquisition -----------------------------------------------------------------------------------------------------------
// acq = ei / cost.  The caller divides, so that it can form the cost after EI: a cost formed first stays live across EI's
// division and spills in the sweep kernels.
struct ExpectedImprovement {
    double sd, u, pdf, cdf, ei;
};
__device__ __forceinline__ ExpectedImprovement expected_improvement(double best, double mu, double var, double task_sign) {
    ExpectedImprovement e;
    e.sd = sqrt(var);
    e.u = (best - mu) / e.sd;
    e.pdf = 0.3989422804014326779 * exp(-0.5 * e.u * e.u);
    e.cdf = 0.5 * erfc(-e.u * 0.7071067811865475244);
    e.ei = task_sign * (e.sd * (e.u * e.cdf + e.pdf));
    return e;
}
// cost_functions.py:11-17: a fixed cost, plus sum |x_k| when the cost is variable (d = S.d)
__device__ __forceinline__ double candidate_cost(const cbo_set_desc& S, int d, const double (&x)[CBO_MAX_D]) {
    double cost = S.cost_fix;
    if (S.cost_variable) {
#pragma unroll
        for (int k = 0; k < CBO_MAX_D; ++k)
            if (k < d) cost += fabs(x[k]);
    }
    return cost;
}

// Coordinates of a candidate: explicit point gidx, or the grid point whose leading dimensions are at flat row `row` and whose
// fastest dimension is at index jj (d = S.d).  Entries k >= d are left as they are.
__device__ __forceinline__ void candidate_x(const cbo_set_desc& S, int d, long long gidx, long long row, int jj,
                                            double (&x)[CBO_MAX_D]) {
    if (S.points) {
#pragma unroll
        for (int k = 0; k < CBO_MAX_D; ++k) x[k] = k < d ? S.points[gidx * d + k] : 0.0;
    } else {
        x[d - 1] = S.grid[d - 1][jj];
        for (int k = d - 2; k >= 0; --k) {
            const long long pk = S.p[k];
            x[k] = S.grid[k][(int)(row % pk)];
            row /= pk;
        }
    }
}

// First argmax (np.argmax: larger value, then smaller index; see better()) and NaN tally over a CTA of THREADS threads, by a
// fixed butterfly per warp and warp order on thread 0.  The result is valid on thread 0 only.
template <int THREADS>
__device__ __forceinline__ void cta_first_argmax(double& val, long long& idx, int& n_nan) {
    __shared__ double red_v[THREADS / 32];
    __shared__ long long red_i[THREADS / 32];
    __shared__ int red_n[THREADS / 32];
    const int tid = threadIdx.x;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, val, o);
        const long long oi = __shfl_xor_sync(0xffffffffu, idx, o);
        n_nan += __shfl_xor_sync(0xffffffffu, n_nan, o);
        if (better(ov, oi, val, idx)) { val = ov; idx = oi; }
    }
    if ((tid & 31) == 0) { red_v[tid >> 5] = val; red_i[tid >> 5] = idx; red_n[tid >> 5] = n_nan; }
    __syncthreads();
    if (tid == 0) {
        n_nan = red_n[0];
        for (int w = 1; w < THREADS / 32; ++w) {
            if (better(red_v[w], red_i[w], val, idx)) { val = red_v[w]; idx = red_i[w]; }
            n_nan += red_n[w];
        }
    }
}

}  // namespace cbo
