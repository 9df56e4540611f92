// K8 -- marginal-likelihood fit of the per-set GP's variance s2 and lengthscale l (opt-in), one CTA per (set, start), the
// Gram resident in shared memory (n <= 128, as in K2).
//
// The model, its Gram and jitchol are surrogate.cuh's, the same code K2 runs, so K8 optimises the model K2 then factors:
//   Ky = s2 exp(-.5 r^2 / l^2) + sqrt(v) sqrt(v)^T [causal only] + (kSurrogateDiag + jitter) I ,  res = y - m_int (or y)
//   NLL = .5 res^T alpha + sum log L_ii + .5 n log(2 pi) ,  alpha = Ky^-1 res
//   dNLL / dtheta = .5 sum_ij (W - alpha alpha^T)_ij dK_ij / dtheta ,  W = Ky^-1 = L^-T L^-1 ,  theta = (log s2, log l)
//   dK / dlog s2 = s2 E ,  dK / dlog l = s2 E o (r^2 / l^2) ,  E = exp(-.5 r^2 / l^2)
// The gradient needs L^-1 (n^3 / 6, written transposed into the strict upper triangle, which the Cholesky
// leaves free) and one pass over the pairs i >= j for W_ij = sum_{k >= i} X_ki X_kj (another n^3 / 6): no second n x n array,
// so n = 128 fits in 132 KB.  The row pitch is odd (n | 1): every access walks rows or columns without bank conflicts.
//
// Search: CBO_HYPER_STARTS starts per set (start 0 = (1, 1), the reference's model, clipped to the box; starts 1..8 the
// lattice log s2 in {log var(res), log var(res) + log 10} x four log l at the centres of quarters of [log l_lo, log l_hi]),
// each a projected BFGS in the log box: coordinates at a bound whose gradient points outwards are held, the first direction
// (and every restart) is the projected steepest descent scaled to a largest move of 1 in log units, and the line search
// backtracks over 1, 1/2, .., 1/128 with Armijo's test (as K7), evaluating the gradient only at the accepted point.  Every
// thread of the CTA runs the same optimiser arithmetic on the same broadcast values (no divergence, no shared control
// state); reductions are fixed trees, so a result depends on its set and start alone: bit-identical across runs, across
// calls that group the sets differently, and across ranks that run K8 redundantly on a split set.
#include <float.h>
#include "surrogate.cuh"

namespace cbo {

constexpr int kHypThreads = 256;
constexpr int kHypWarps = kHypThreads / 32;
constexpr int kHypTrials = 8;            // backtracking steps 1, 1/2, ..., 1/128
constexpr double kHypArmijo = 1e-4;
constexpr double kHalfLog2Pi = 0.91893853320467274178;

struct HypSmem {
    double* A;     // [n][ld]: Gram, then L in the lower triangle (diagonal in dsq), L^-1 transposed in the strict upper one
    double* xs;    // x_int, n x d
    double* sv;    // sqrt(v_int); 0 for a non-causal set
    double* res;   // y - m_int (or y)
    double* al;    // alpha
    double* dsq;   // L_ii
    double* rinv;  // 1 / L_ii
    double* red;   // 2 kHypWarps reduction slots, then the NLL
    int ld;
};
inline size_t hyp_smem_bytes(int n) {
    return ((size_t)n * (n | 1) + (size_t)n * CBO_MAX_D + 5 * (size_t)n + 2 * kHypWarps + 1) * sizeof(double);
}

__device__ void hyp_stage(const cbo_set_desc& S, HypSmem& sm, double* base) {
    const int n = S.n_int, d = S.d;
    sm.ld = n | 1;
    sm.A = base;
    sm.xs = sm.A + (size_t)n * sm.ld;
    sm.sv = sm.xs + (size_t)n * CBO_MAX_D;
    sm.res = sm.sv + n;
    sm.al = sm.res + n;
    sm.dsq = sm.al + n;
    sm.rinv = sm.dsq + n;
    sm.red = sm.rinv + n;
    for (int i = threadIdx.x; i < n; i += kHypThreads) {
        sm.sv[i] = S.causal ? sqrt(S.v_int[i]) : 0.0;
        sm.res[i] = S.causal ? S.y_int[i] - S.m_int[i] : S.y_int[i];
    }
    for (int i = threadIdx.x; i < n * d; i += kHypThreads) sm.xs[i] = S.x_int[i];
}

// CTA-wide sums of two values, the same fixed tree on every call; every thread receives the result
__device__ __forceinline__ void hyp_sum2(double& a, double& b, double* red) {
    a = warp_sum(a);
    b = warp_sum(b);
    const int w = threadIdx.x >> 5;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) { red[2 * w] = a; red[2 * w + 1] = b; }
    __syncthreads();
    a = 0.0; b = 0.0;
#pragma unroll
    for (int k = 0; k < kHypWarps; ++k) { a += red[2 * k]; b += red[2 * k + 1]; }
}

// NLL at h: K2's Gram and jitchol (surrogate.cuh), then alpha.  Returns the jitter retries (0..5), or -1 when Ky is not
// positive definite even with jitter (f = +inf).  Leaves L, dsq, rinv and alpha in shared memory for hyp_grad.
__device__ int hyp_nll(const HypSmem& sm, int n, int d, SurrogateHyper h, double& f) {
    const int tid = threadIdx.x, ld = sm.ld;
    double* nll = sm.red + 2 * kHypWarps;
    const int tries = surrogate_jitchol<kHypThreads>(sm.A, ld, sm.xs, sm.sv, n, d, h, sm.dsq, sm.rinv);
    if (tries < 0) { f = __longlong_as_double(0x7ff0000000000000LL); return -1; }
    // z = L^-1 res, alpha = L^-T z in one warp as K2's warp_solve_lower / _upper, but multiplying by 1 / L_ii where K2
    // divides by L_ii: the division lies on the dependent chain of every row, and with it the fit of a shipped configuration
    // took up to 1.4x as long.  |z|^2 and sum log L_ii by fixed butterflies.
    if (tid < 32) {
        double z[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) z[r] = (tid + 32 * r < n) ? sm.res[tid + 32 * r] : 0.0;
        for (int j = 0; j < n; ++j) {
            const double zj = __shfl_sync(0xffffffffu, warp_own_row(z, j) * sm.rinv[j], j & 31);
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int i = tid + 32 * r;
                if (i == j) z[r] = zj;
                else if (i > j && i < n) z[r] = fma(-sm.A[i * ld + j], zj, z[r]);
            }
        }
        double zz = 0.0, lg = 0.0;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            zz = fma(z[r], z[r], zz);
            if (tid + 32 * r < n) lg += log(sm.dsq[tid + 32 * r]);
        }
        zz = warp_sum(zz);
        lg = warp_sum(lg);
        for (int j = n - 1; j >= 0; --j) {
            const double aj = __shfl_sync(0xffffffffu, warp_own_row(z, j) * sm.rinv[j], j & 31);
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int i = tid + 32 * r;
                if (i == j) z[r] = aj;
                else if (i < j) z[r] = fma(-sm.A[j * ld + i], aj, z[r]);
            }
        }
#pragma unroll
        for (int r = 0; r < 4; ++r)
            if (tid + 32 * r < n) sm.al[tid + 32 * r] = z[r];
        if (tid == 0) *nll = (0.5 * zz + lg) + n * kHalfLog2Pi;
    }
    __syncthreads();
    f = *nll;
    return tries;
}

// Gradient of the NLL in (log s2, log l) from the state hyp_nll left (same h).
__device__ void hyp_grad(const HypSmem& sm, int n, int d, SurrogateHyper h, double& g0, double& g1) {
    const int tid = threadIdx.x, ld = sm.ld;
    // X = L^-1, column by column from the right: X_ij = -(sum_{j < k <= i} X_ik L_kj) / L_jj, stored at A[j][i].  (K2's
    // surrogate_lower_inverse, which walks each column down its rows, made the fit 2-3.5 % slower here, 1.7 % at n = 128.)
    for (int j = n - 2; j >= 0; --j) {
        for (int i = j + 1 + tid; i < n; i += kHypThreads) {
            double a = sm.A[i * ld + j] * sm.rinv[i];
            for (int k = j + 1; k < i; ++k) a = fma(sm.A[k * ld + i], sm.A[k * ld + j], a);
            sm.A[j * ld + i] = -a * sm.rinv[j];
        }
        __syncthreads();
    }
    // .5 sum_ij (W - alpha alpha^T)_ij G_ij over the pairs i >= j (off-diagonal pairs twice)
    double t0 = 0.0, t1 = 0.0;
    for (int e = tid; e < n * n; e += kHypThreads) {
        const int i = e / n, j = e - i * n;
        if (j > i) continue;
        const double xij = (i == j) ? sm.rinv[i] : sm.A[j * ld + i];
        double w = xij * sm.rinv[i];
        for (int k = i + 1; k < n; ++k) w = fma(sm.A[i * ld + k], sm.A[j * ld + k], w);
        const double r2 = surrogate_r2(sm.xs, i, j, d, h.il);
        const double c = (i == j ? 0.5 : 1.0) * (w - sm.al[i] * sm.al[j]) * surrogate_rbf(r2, h.s2);
        t0 += c;
        t1 = fma(c, r2, t1);
    }
    hyp_sum2(t0, t1, sm.red);
    g0 = t0;
    g1 = t1;
}

struct HypStart {
    double th[2];     // (log s2, log l) at the end of the search
    double f;         // NLL there (+inf when the start failed)
    double f11;       // NLL at (1, 1) (start 0 only)
    int32_t iter, status, tries, ok;
};

__global__ void __launch_bounds__(kHypThreads)
hyper_fit_kernel(const cbo_set_desc* __restrict__ sets, const double* __restrict__ bounds, int max_iter, double gtol,
                 HypStart* __restrict__ out) {
    extern __shared__ __align__(16) double smem_d[];
    const int s = blockIdx.x / CBO_HYPER_STARTS, k0 = blockIdx.x % CBO_HYPER_STARTS;
    const cbo_set_desc& S = sets[s];
    const int n = S.n_int, d = S.d;
    HypSmem sm;
    hyp_stage(S, sm, smem_d);
    __syncthreads();
    const double lb[2] = {log(bounds[4 * s + 0]), log(bounds[4 * s + 2])};
    const double ub[2] = {log(bounds[4 * s + 1]), log(bounds[4 * s + 3])};
    double th[2];
    if (k0 == 0) {
        th[0] = 0.0; th[1] = 0.0;
    } else {
        double mean = 0.0, var = 0.0;
        for (int i = 0; i < n; ++i) mean += sm.res[i];
        mean /= n;
        for (int i = 0; i < n; ++i) var = fma(sm.res[i] - mean, sm.res[i] - mean, var);
        var /= n;
        const int a = (k0 - 1) & 3, b = (k0 - 1) >> 2;
        th[0] = (var > 0.0 ? log(var) : lb[0]) + b * 2.302585092994045684;
        th[1] = lb[1] + (a + 0.5) * 0.25 * (ub[1] - lb[1]);
    }
    for (int k = 0; k < 2; ++k) th[k] = fmin(fmax(th[k], lb[k]), ub[k]);
    auto at = [](const double (&t)[2]) { return SurrogateHyper{exp(t[0]), 1.0 / exp(t[1])}; };     // (log s2, log l) -> (s2, 1 / l)
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    double f, f11 = nan, g[2] = {0.0, 0.0};
    int tries = hyp_nll(sm, n, d, at(th), f);
    if (k0 == 0) {
        if (th[0] == 0.0 && th[1] == 0.0) f11 = tries >= 0 ? f : nan;
        else {
            double f1;
            const int t1 = hyp_nll(sm, n, d, SurrogateHyper{1.0, 1.0}, f1);
            f11 = t1 >= 0 ? f1 : nan;
            tries = hyp_nll(sm, n, d, at(th), f);     // L of the start point again, for its gradient
        }
    }
    int status = CBO_HYPER_MAX_ITER, iter = 0;
    if (tries < 0) status = CBO_HYPER_NOT_PD;
    else {
        hyp_grad(sm, n, d, at(th), g[0], g[1]);
        if (!(isfinite(g[0]) && isfinite(g[1]))) status = CBO_HYPER_LINE_SEARCH_FAILED;
    }
    double H[4] = {1.0, 0.0, 0.0, 1.0};
    bool qn = false;
    while (status == CBO_HYPER_MAX_ITER) {
        double pg[2], gmax = 0.0;
        bool fr[2];
        for (int k = 0; k < 2; ++k) {
            fr[k] = ub[k] > lb[k] && !(th[k] <= lb[k] && g[k] > 0.0) && !(th[k] >= ub[k] && g[k] < 0.0);
            pg[k] = fr[k] ? g[k] : 0.0;
            gmax = fmax(gmax, fabs(pg[k]));
        }
        if (gmax <= gtol) { status = CBO_HYPER_CONVERGED; break; }
        if (iter >= max_iter) break;
        double p[2];
        if (qn) {
            double slope = 0.0;
            for (int k = 0; k < 2; ++k) {
                p[k] = fr[k] ? -fma(H[2 * k], pg[0], H[2 * k + 1] * pg[1]) : 0.0;
                slope = fma(p[k], pg[k], slope);
            }
            if (!(slope < 0.0)) qn = false;       // not a descent direction: restart from the scaled gradient
        }
        if (!qn)
            for (int k = 0; k < 2; ++k) p[k] = -pg[k] / gmax;
        double tt[2], ft = 0.0;
        int tr = -1;
        bool acc = false;
        for (int j = 0; j < kHypTrials && !acc; ++j) {
            const double t = ldexp(1.0, -j);
            for (int k = 0; k < 2; ++k) tt[k] = fmin(fmax(fma(t, p[k], th[k]), lb[k]), ub[k]);
            tr = hyp_nll(sm, n, d, at(tt), ft);
            const double gain = fma(g[0], tt[0] - th[0], g[1] * (tt[1] - th[1]));
            acc = tr >= 0 && ft < f && ft <= fma(kHypArmijo, gain, f);     // NaN fails
        }
        ++iter;
        if (!acc) {
            if (qn) { qn = false; continue; }    // retry along the scaled gradient
            status = CBO_HYPER_LINE_SEARCH_FAILED;
            break;
        }
        double gt[2];
        hyp_grad(sm, n, d, at(tt), gt[0], gt[1]);
        if (!(isfinite(gt[0]) && isfinite(gt[1]))) { status = CBO_HYPER_LINE_SEARCH_FAILED; break; }
        const double sv[2] = {tt[0] - th[0], tt[1] - th[1]};
        const double yv[2] = {gt[0] - g[0], gt[1] - g[1]};
        const double sy = fma(sv[0], yv[0], sv[1] * yv[1]);
        if (sy > 0.0) {                            // BFGS update of the inverse Hessian
            if (!qn) {
                const double yy = fma(yv[0], yv[0], yv[1] * yv[1]);
                H[0] = H[3] = sy / yy;
                H[1] = H[2] = 0.0;
                qn = true;
            }
            const double rho = 1.0 / sy;
            const double Hy[2] = {fma(H[0], yv[0], H[1] * yv[1]), fma(H[2], yv[0], H[3] * yv[1])};
            const double yHy = fma(yv[0], Hy[0], yv[1] * Hy[1]);
            for (int k = 0; k < 2; ++k)
                for (int j = 0; j < 2; ++j)
                    H[2 * k + j] += (1.0 + rho * yHy) * rho * sv[k] * sv[j] - rho * (Hy[k] * sv[j] + sv[k] * Hy[j]);
        }
        th[0] = tt[0]; th[1] = tt[1];
        g[0] = gt[0]; g[1] = gt[1];
        f = ft;
        tries = tr;
    }
    if (threadIdx.x == 0) {
        HypStart r;
        r.th[0] = th[0]; r.th[1] = th[1];
        r.f = f; r.f11 = f11;
        r.iter = iter; r.status = status; r.tries = tries; r.ok = status != CBO_HYPER_NOT_PD;
        out[blockIdx.x] = r;
    }
}

// per set: the start with the lowest NLL (NaN = +inf, ties to the lowest start) is written through `hyper`
__global__ void hyper_reduce_kernel(const cbo_set_desc* __restrict__ sets, int num_sets, const HypStart* __restrict__ starts,
                                    cbo_hyper_result* __restrict__ out) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= num_sets) return;
    const cbo_set_desc& S = sets[s];
    const HypStart* st = starts + (size_t)s * CBO_HYPER_STARTS;
    int win = -1;
    double fb = __longlong_as_double(0x7ff0000000000000LL);
    for (int k = 0; k < CBO_HYPER_STARTS; ++k)
        if (st[k].ok && st[k].f < fb) { fb = st[k].f; win = k; }
    cbo_hyper_result r;
    r.nll_start = st[0].f11;
    if (win >= 0) {
        const HypStart& w = st[win];
        r.variance = exp(w.th[0]);
        r.lengthscale = exp(w.th[1]);
        S.hyper[0] = r.variance;
        S.hyper[1] = r.lengthscale;
        r.nll = w.f;
        r.iterations = w.iter; r.status = w.status; r.start = win; r.jitter_tries = w.tries;
    } else {
        r.variance = S.hyper[0];
        r.lengthscale = S.hyper[1];
        r.nll = __longlong_as_double(0x7ff8000000000000LL);
        r.iterations = 0; r.status = CBO_HYPER_NOT_PD; r.start = -1; r.jitter_tries = -1;
    }
    out[s] = r;
}

// NLL and gradient at each set's current hyper-parameters
__global__ void __launch_bounds__(kHypThreads)
posterior_nll_kernel(const cbo_set_desc* __restrict__ sets, double* __restrict__ out) {
    extern __shared__ __align__(16) double smem_d[];
    const cbo_set_desc& S = sets[blockIdx.x];
    const int n = S.n_int, d = S.d;
    HypSmem sm;
    hyp_stage(S, sm, smem_d);
    __syncthreads();
    const SurrogateHyper h = surrogate_hyper(S);
    double f, g0 = 0.0, g1 = 0.0;
    const int tries = hyp_nll(sm, n, d, h, f);
    if (tries >= 0) hyp_grad(sm, n, d, h, g0, g1);
    else f = g0 = g1 = __longlong_as_double(0x7ff8000000000000LL);
    if (threadIdx.x == 0) {
        out[3 * blockIdx.x] = f;
        out[3 * blockIdx.x + 1] = g0;
        out[3 * blockIdx.x + 2] = g1;
    }
}

// ---- host side -----------------------------------------------------------------------------------------------------------
static int hyp_check_sets(const cbo_set_desc* h_sets, int num_sets, const char* who, int& nmax) {
    nmax = 1;
    for (int s = 0; s < num_sets; ++s) {
        const cbo_set_desc& S = h_sets[s];
        CBO_REQUIRE(S.x_int && S.y_int, "%s: set %d has a NULL x_int/y_int", who, s);
        CBO_REQUIRE(!S.causal || (S.m_int && S.v_int), "%s: causal set %d needs m_int/v_int", who, s);
        if (S.n_int > nmax) nmax = S.n_int;
    }
    return 0;
}

static size_t hyp_bounds_bytes(int num_sets) { return ((size_t)num_sets * 4 * sizeof(double) + 255) & ~(size_t)255; }

size_t hyper_workspace_bytes_impl(int num_sets) {
    return hyp_bounds_bytes(num_sets) + (size_t)num_sets * CBO_HYPER_STARTS * sizeof(HypStart);
}

int posterior_nll_impl(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, double* d_out, cudaStream_t st) {
    int nmax;
    if (int rc = hyp_check_sets(h_sets, num_sets, "cbo_posterior_nll", nmax)) return rc;
    const size_t smem = hyp_smem_bytes(nmax);
    if (smem > 48 * 1024) CBO_CUDA(allow_dynamic_smem(posterior_nll_kernel, smem));
    posterior_nll_kernel<<<num_sets, kHypThreads, smem, st>>>(d_sets, d_out);
    note_launch();
    CBO_CUDA(cudaGetLastError());
    return 0;
}

int hyper_fit_impl(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, const double* h_bounds, int max_iter,
                   double gtol, void* d_ws, size_t ws_bytes, cbo_hyper_result* d_out, cudaStream_t st) {
    CBO_REQUIRE(h_bounds != nullptr, "cbo_posterior_hyper_fit: h_bounds is NULL");
    CBO_REQUIRE(d_out != nullptr, "cbo_posterior_hyper_fit: d_out is NULL");
    CBO_REQUIRE(max_iter >= 0 && max_iter <= 100000, "cbo_posterior_hyper_fit: max_iter=%d outside [0,100000]", max_iter);
    CBO_REQUIRE(gtol >= 0.0 && isfinite(gtol), "cbo_posterior_hyper_fit: gtol must be finite and non-negative");
    int nmax;
    if (int rc = hyp_check_sets(h_sets, num_sets, "cbo_posterior_hyper_fit", nmax)) return rc;
    for (int s = 0; s < num_sets; ++s) {
        CBO_REQUIRE(h_sets[s].hyper != nullptr, "cbo_posterior_hyper_fit: set %d has hyper == NULL (nowhere to write the fit)", s);
        const double* b = h_bounds + 4 * s;
        bool ok = true;
        for (int k = 0; k < 4; ++k) ok &= isfinite(b[k]) && b[k] > 0.0;
        CBO_REQUIRE(ok && b[0] <= b[1] && b[2] <= b[3],
                    "cbo_posterior_hyper_fit: set %d bounds s2 [%g, %g], l [%g, %g] must be finite and positive with lo <= hi", s,
                    b[0], b[1], b[2], b[3]);
    }
    const size_t need = hyper_workspace_bytes_impl(num_sets);
    CBO_REQUIRE(d_ws != nullptr && ws_bytes >= need,
                "cbo_posterior_hyper_fit: workspace of %zu bytes is too small (%zu needed; see cbo_posterior_hyper_workspace_bytes)",
                ws_bytes, need);
    double* d_bounds = static_cast<double*>(d_ws);
    HypStart* starts = reinterpret_cast<HypStart*>(static_cast<unsigned char*>(d_ws) + hyp_bounds_bytes(num_sets));
    CBO_CUDA(cudaMemcpyAsync(d_bounds, h_bounds, (size_t)num_sets * 4 * sizeof(double), cudaMemcpyHostToDevice, st));
    const size_t smem = hyp_smem_bytes(nmax);
    if (smem > 48 * 1024) CBO_CUDA(allow_dynamic_smem(hyper_fit_kernel, smem));
    hyper_fit_kernel<<<num_sets * CBO_HYPER_STARTS, kHypThreads, smem, st>>>(d_sets, d_bounds, max_iter, gtol, starts);
    note_launch();
    CBO_CUDA(cudaGetLastError());
    hyper_reduce_kernel<<<(num_sets + 127) / 128, 128, 0, st>>>(d_sets, num_sets, starts, d_out);
    note_launch();
    CBO_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace cbo
