// K2 -- batched exact-GP fit of the per-set surrogate, one CTA per exploration set, everything resident in
// shared memory.
//
// Replaces GPRegression(...) at GaussianProcessFactory.py:57-73, i.e. GPy's ExactGaussianInference:
//   causal     : K = s2 exp(-.5 r^2 / l^2) + sqrt(v(X)) sqrt(v(X))^T   (CausalRBF.K, causal_kernels.py:45-62)
//                resid = y - m(X)                              (Mapping.f = mean function, :65-68)
//   non-causal : K = s2 exp(-.5 r^2 / l^2), resid = y          (:57-60)
//   (s2, l) = hyper[0..1], or the reference's (1, 1) when `hyper` is NULL (the scaling by 1 is exact: same bits)
//   Ky = K + kSurrogateDiag I ; L = jitchol(Ky) ; alpha = Ky^-1 resid
// The model, GPy's jitchol rule, the solves and L^-1 are those of surrogate.cuh, which K3, K7 and K8 share.
// Output `L`: the factor in the lower triangle; for n <= 48 the strict upper triangle carries L^-T (for K3), else zeros.
// After 5 jitter retries the fit gives up (fit_info[1] = 1, outputs NaN).
// n <= 128, so the matrix (<= 128 KB) lives in shared memory; latency-bound by construction (n is tiny),
// its cost is microseconds per trial.  r^2 is formed from coordinate differences (no cancellation).
#include "surrogate.cuh"

namespace cbo {

constexpr int kFitThreads = 256;

__global__ void __launch_bounds__(kFitThreads, 1)
posterior_fit_kernel(const cbo_set_desc* __restrict__ sets) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const cbo_set_desc& S = sets[blockIdx.x];
    const int n = S.n_int, d = S.d, tid = threadIdx.x;
    if (n <= 0) return;
    double* A = reinterpret_cast<double*>(smem_raw);  // n x n, row-major, lower triangle becomes L
    double* sv = A + (size_t)n * n;                   // sqrt(v_int)
    double* rhs = sv + n;                             // y - m, then the solution
    double* xs = rhs + n;                             // x_int copy, n x d
    double* rinv = xs + (size_t)n * CBO_MAX_D;        // 1 / L_ii
    double* dsq = rinv + n;                           // L_ii

    for (int i = tid; i < n; i += kFitThreads) {
        sv[i] = S.causal ? sqrt(S.v_int[i]) : 0.0;
        rhs[i] = S.causal ? S.y_int[i] - S.m_int[i] : S.y_int[i];
    }
    for (int i = tid; i < n * d; i += kFitThreads) xs[i] = S.x_int[i];
    __syncthreads();

    const int tries = surrogate_jitchol<kFitThreads>(A, n, xs, sv, n, d, surrogate_hyper(S), dsq, rinv);
    const bool bad = tries < 0;
    if (!bad) {
        // alpha = L^-T L^-1 rhs in one warp
        if (tid < 32) {
            double z[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) z[r] = (tid + 32 * r < n) ? rhs[tid + 32 * r] : 0.0;
            warp_solve_lower(A, n, dsq, n, z);
            warp_solve_upper(A, n, dsq, n, z);
#pragma unroll
            for (int r = 0; r < 4; ++r)
                if (tid + 32 * r < n) rhs[tid + 32 * r] = z[r];
        }
        __syncthreads();
    }
    // n <= kSweepMmaMaxN: L^-T goes into the strict upper triangle.  K3's tensor-pipe path multiplies k* by L^-1 (a GEMM over
    // candidates) instead of substituting per candidate.
    const bool with_inv = n <= kSweepMmaMaxN;
    if (!bad && with_inv) surrogate_lower_inverse<kFitThreads>(A, n, rinv, n);
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    for (int e = tid; e < n * n; e += kFitThreads) {
        const int i = e / n, j = e % n;
        S.L[e] = bad ? nan : ((j <= i || with_inv) ? A[e] : 0.0);
    }
    for (int i = tid; i < n; i += kFitThreads) {
        S.alpha[i] = bad ? nan : rhs[i];
        S.sqrt_v_int[i] = sv[i];
    }
    if (tid == 0) {
        S.fit_info[0] = bad ? 5 : tries;
        S.fit_info[1] = bad ? 1 : 0;
    }
}

int posterior_fit_impl(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, cudaStream_t st) {
    int nmax = 0;
    for (int s = 0; s < num_sets; ++s) {
        const cbo_set_desc& S = h_sets[s];
        CBO_REQUIRE(S.n_int >= 1 && S.n_int <= CBO_MAX_NINT, "cbo_posterior_fit: set %d n_int=%d outside [1,%d]", s, S.n_int, CBO_MAX_NINT);
        CBO_REQUIRE(S.x_int && S.y_int && S.L && S.alpha && S.sqrt_v_int && S.fit_info, "cbo_posterior_fit: set %d has a NULL pointer", s);
        CBO_REQUIRE(!S.causal || (S.m_int && S.v_int), "cbo_posterior_fit: causal set %d needs m_int/v_int", s);
        if (S.n_int > nmax) nmax = S.n_int;
    }
    const size_t smem = ((size_t)nmax * nmax + 4 * (size_t)nmax + (size_t)nmax * CBO_MAX_D) * sizeof(double);
    if (smem > 48 * 1024) CBO_CUDA(allow_dynamic_smem(posterior_fit_kernel, smem));
    posterior_fit_kernel<<<num_sets, kFitThreads, smem, st>>>(d_sets);
    note_launch();
    CBO_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace cbo
