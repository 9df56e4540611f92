// K2 -- batched exact-GP fit of the per-set surrogate, one CTA per exploration set, everything resident in
// shared memory.
//
// Replaces GPRegression(...) at GaussianProcessFactory.py:57-73, i.e. GPy's ExactGaussianInference:
//   causal     : K = s2 exp(-.5 r^2 / l^2) + sqrt(v(X)) sqrt(v(X))^T   (CausalRBF.K, causal_kernels.py:45-62)
//                resid = y - m(X)                              (Mapping.f = mean function, :65-68)
//   non-causal : K = s2 exp(-.5 r^2 / l^2), resid = y          (:57-60)
//   (s2, l) = hyper[0..1], or the reference's (1, 1) when `hyper` is NULL (the scaling by 1 is exact: same bits)
//   Ky = K + (1e-10 + 1e-8) I ; L = jitchol(Ky) ; alpha = Ky^-1 resid
// Output `L`: the factor in the lower triangle; for n <= 48 the strict upper triangle carries L^-T (for K3), else zeros.
// jitchol rule (GPy util.linalg): plain Cholesky first; on a non-positive pivot retry with
// jitter = mean(diag Ky) * 1e-6 * 10^t, t = 0..4; give up after 5 retries (fit_info[1] = 1, outputs NaN).
// n <= 128, so the matrix (<= 128 KB) lives in shared memory; latency-bound by construction (n is tiny),
// its cost is microseconds per trial.  r^2 is formed from coordinate differences (no cancellation).
#include "cbo_common.cuh"

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
    bool failed = false;
    __shared__ double diag_mean;
    const double s2 = S.hyper ? S.hyper[0] : 1.0, il = S.hyper ? 1.0 / S.hyper[1] : 1.0;

    for (int i = tid; i < n; i += kFitThreads) {
        sv[i] = S.causal ? sqrt(S.v_int[i]) : 0.0;
        rhs[i] = S.causal ? S.y_int[i] - S.m_int[i] : S.y_int[i];
    }
    for (int i = tid; i < n * d; i += kFitThreads) xs[i] = S.x_int[i];
    __syncthreads();

    int tries = 0;
    double jitter = 0.0;
    for (;;) {
        // Gram matrix + noise (+ jitter on retries)
        for (int e = tid; e < n * n; e += kFitThreads) {
            const int i = e / n, j = e % n;
            double r2 = 0.0;
            for (int k = 0; k < d; ++k) {
                const double t = (xs[i * d + k] - xs[j * d + k]) * il;
                r2 += t * t;
            }
            double kij = fma(sv[i], sv[j], __dmul_rn(s2, exp(-0.5 * r2)));
            if (i == j) kij += (1e-10 + 1e-8) + jitter;
            A[e] = kij;
        }
        __syncthreads();
        if (tries == 0) {  // mean of the diagonal of Ky, the scale of GPy's jitter
            if (tid == 0) {
                double t = 0.0;
                for (int i = 0; i < n; ++i) t += A[i * n + i];
                diag_mean = t / n;
            }
            __syncthreads();
        }
        // Right-looking Cholesky, lower.  Every thread reads the same pivot (so the failure branch is uniform) and forms
        // 1 / sqrt(pivot) itself; the diagonal is written after the loop (nobody waits for thread 0, two barriers per column
        // instead of three); the trailing update walks a 16 x 16 thread grid (no integer division per element).  The
        // arithmetic is LAPACK's: scale the column, then subtract products of scaled entries.
        failed = false;
        for (int j = 0; j < n; ++j) {
            const double piv = A[j * n + j];
            if (!(piv > 0.0)) { failed = true; break; }
            const double sq = sqrt(piv);
            const double inv = 1.0 / sq;
            if (tid == 0) dsq[j] = sq;
            for (int i = j + 1 + tid; i < n; i += kFitThreads) A[i * n + j] *= inv;
            __syncthreads();
            for (int i = j + 1 + (tid >> 4); i < n; i += kFitThreads / 16)
                for (int k = j + 1 + (tid & 15); k <= i; k += 16) A[i * n + k] -= A[i * n + j] * A[k * n + j];
            __syncthreads();
        }
        if (!failed) break;
        __syncthreads();     // (a thread may still be reading the failing pivot while the next Gram is written)
        if (tries == 5) break;
        jitter = (tries == 0) ? diag_mean * 1e-6 : jitter * 10.0;
        ++tries;
    }
    const bool bad = failed;

    if (!bad) {
        for (int j = tid; j < n; j += kFitThreads) {
            A[j * n + j] = dsq[j];
            rinv[j] = 1.0 / dsq[j];
        }
        __syncthreads();
        // forward L z = rhs, backward L^T a = z in ONE warp, no CTA barriers: lane l owns rows l, l + 32, l + 64, l + 96 in
        // registers, the pivot row's value travels by shuffle (two barriers per row and a division by thread 0 before)
        if (tid < 32) {
            double z[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) z[r] = (tid + 32 * r < n) ? rhs[tid + 32 * r] : 0.0;
            for (int j = 0; j < n; ++j) {
                const int slot = j >> 5;
                const double own = (slot == 0 ? z[0] : slot == 1 ? z[1] : slot == 2 ? z[2] : z[3]) / dsq[j];
                const double zj = __shfl_sync(0xffffffffu, own, j & 31);
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const int i = tid + 32 * r;
                    if (i == j) z[r] = zj;
                    else if (i > j && i < n) z[r] = fma(-A[i * n + j], zj, z[r]);
                }
            }
            for (int j = n - 1; j >= 0; --j) {
                const int slot = j >> 5;
                const double own = (slot == 0 ? z[0] : slot == 1 ? z[1] : slot == 2 ? z[2] : z[3]) / dsq[j];
                const double aj = __shfl_sync(0xffffffffu, own, j & 31);
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const int i = tid + 32 * r;
                    if (i == j) z[r] = aj;
                    else if (i < j) z[r] = fma(-A[j * n + i], aj, z[r]);
                }
            }
#pragma unroll
            for (int r = 0; r < 4; ++r)
                if (tid + 32 * r < n) rhs[tid + 32 * r] = z[r];
        }
        __syncthreads();
    }
    // n <= kSweepMmaMaxN: L^-T goes into the strict upper triangle (the diagonal of L^-1 is 1 / L_ii).  K3's tensor-pipe path
    // multiplies k* by L^-1 (a GEMM over candidates) instead of substituting per candidate.  Column c of
    // W = L^-1 is stored as row c of the upper triangle: W[i][c] = -(sum_{c <= j < i} L[i][j] W[j][c]) / L[i][i].
    const bool with_inv = n <= kSweepMmaMaxN;
    if (!bad && with_inv) {
        // four lanes per column split every dot product and combine by a fixed butterfly: 64 columns at once, one round for
        // n <= 48 (a single thread per column made the inverse a 20 us chain at n = 45).  Lane sub = 0 stores.
        const int sub = tid & 3;
        for (int c = tid >> 2; c < ((n + 63) & ~63); c += kFitThreads / 4) {        // warp-uniform trip count
            const bool col = c < n;
            const double wcc = col ? rinv[c] : 0.0;
            for (int i = (c & ~7) + 1; i < n; ++i) {      // row i of column c, i > c (a warp holds columns 8 w .. 8 w + 7)
                double a0 = 0.0;
                if (col && i > c) {
                    for (int j = c + 1 + sub; j < i; j += 4) a0 = fma(A[i * n + j], A[c * n + j], a0);
                    if (sub == 0) a0 = fma(A[i * n + c], wcc, a0);
                }
                a0 += __shfl_xor_sync(0xffffffffu, a0, 1);
                a0 += __shfl_xor_sync(0xffffffffu, a0, 2);
                if (col && i > c && sub == 0) A[c * n + i] = -a0 * rinv[i];
                __syncwarp();
            }
        }
        __syncthreads();
    }
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
        S.fit_info[0] = tries;
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
