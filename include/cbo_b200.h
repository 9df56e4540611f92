/* cbo_b200.h -- C ABI of libcbo_b200.so: the B200-native (sm_100a) per-trial acquisition sweep of
 * Causal Bayesian Optimisation (causal prior -> per-set GP posterior -> EI / cost -> argmax).
 *
 * The reference (ChampiB/CBO_with_OOP) is pure Python and has no FFI; each entry point below names the
 * reference call site whose arithmetic it replaces (paths relative to the reference checkout).  The
 * reference-side binding a maintainer would add is shown in INTEGRATION.md.
 *
 * Conventions
 *  - every pointer inside cbo_set_desc is a CUDA DEVICE pointer to float64 unless stated otherwise;
 *    the caller owns every allocation (PyTorch tensors in the shipped host code), the library allocates
 *    nothing and keeps no global state besides a thread-local error string;
 *  - `h_sets` is a HOST array of descriptors, `d_sets` the same bytes resident on the device;
 *  - `stream` is a cudaStream_t passed as void*; calls are asynchronous on it and re-entrant per stream;
 *  - return value: 0 ok, <0 invalid argument (see cbo_last_error), >0 a cudaError_t;
 *  - there is NO CPU fallback: without a CUDA device every compute entry point returns an error.
 */
#ifndef CBO_B200_H
#define CBO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define CBO_API __attribute__((visibility("default")))
#else
#define CBO_API
#endif

#define CBO_ABI_VERSION 9
#define CBO_MAX_D 4          /* intervened dimensions per exploration set (reference uses 1..3) */
#define CBO_MAX_C 8          /* conditioning dimensions of an observational GP */
#define CBO_MAX_NINT 128     /* interventional rows per set (reference: 10 .. ~50) */
#define CBO_NPAD 128         /* n_obs_pad must be a multiple of this */
#define CBO_SPAD 16          /* n_mc_pad must be a multiple of this */
#define CBO_PRIOR_TILE 128   /* grid points per prior-eval work item */
#define CBO_SWEEP_TILE 1024  /* grid points per sweep work item (128 threads, 8 candidates each) */

/* One exploration set.  Index conventions follow SURVEY.md §8(d): the candidate grid is the tensor
 * product of per-dimension coordinate tables, flattened C-order (last dimension fastest). */
typedef struct cbo_set_desc {
    /* ---- sizes ------------------------------------------------------------------------------- */
    int32_t d;            /* intervened dims */
    int32_t c;            /* conditioning dims */
    int32_t n_obs;        /* N: training rows of the observational GP */
    int32_t n_obs_pad;    /* leading dimension of tab/u_int/M/w/pbar/P rows; multiple of CBO_NPAD */
    int32_t n_mc;         /* S_mc: conditioning samples averaged over (reference: = n_obs) */
    int32_t n_mc_pad;     /* leading dimension of P; multiple of CBO_SPAD */
    int32_t n_int;        /* n: interventional rows */
    int32_t causal;       /* 1: causal prior mean + CausalRBF; 0: zero mean + RBF (NON_CAUSAL_GP) */
    int32_t p[CBO_MAX_D]; /* grid points per intervened dim */
    int64_t g_total;      /* prod p[k] */
    int64_t g_begin;      /* this rank evaluates flat grid indices [g_begin, g_begin + g_count) */
    int64_t g_count;
    /* ---- observational GP: inputs (utils.py:40-45 fit, hyper-parameters frozen) ---------------- */
    const double* x_obs_int;   /* (d, n_obs)   intervened columns of the training design, one row per dim */
    const double* x_obs_cond;  /* (c, n_obs)   conditioning columns of the training design */
    const double* mc_cond;     /* (c, n_mc)    conditioning samples (DoCalculus.py:85-88 non-intervened columns) */
    const double* alpha_obs;   /* (n_obs)      Ky^-1 y */
    const double* kyinv;       /* (n_obs, n_obs) row-major, Ky^-1 */
    double ls_int[CBO_MAX_D];  /* lengthscale per intervened dim */
    double ls_cond[CBO_MAX_C]; /* lengthscale per conditioning dim */
    double s2;                 /* RBF variance */
    double noise;              /* likelihood variance (1e-2, utils.py:43) */
    /* ---- causal prior: work buffers written by the library --------------------------------------- */
    double* tab[CBO_MAX_D];    /* (p[k], n_obs_pad) exp tables, zero for j >= n_obs */
    double* u_int;             /* (n_int, n_obs_pad) exp table of the interventional rows */
    double* P;                 /* (n_obs_pad, n_mc_pad) scratch; may be shared between sets (stream-ordered) */
    double* pbar;              /* (n_obs_pad) */
    double* w;                 /* (n_obs_pad) s2 * alpha * pbar, zero padded */
    double* M;                 /* n_obs_pad^2 doubles: s2^2 Kyinv o (P P^T / S_mc), symmetric, zero padded, stored BLOCKED:
                                  element (n,k) at ((n/128)*(n_obs_pad/16) + k/16)*2048 + (((k%16)/4)*128 + n%128)*4 + k%4,
                                  i.e. every 128-row x 16-column slab is contiguous and in DMMA fragment order */
    /* ---- interventional data and the per-set GP ------------------------------------------------ */
    const double* grid[CBO_MAX_D]; /* (p[k]) candidate coordinates per dim (np.linspace tables from the host) */
    const double* x_int;       /* (n_int, d) row-major */
    const double* y_int;       /* (n_int) */
    double* m_int;             /* (n_int) prior mean at x_int      [written by cbo_prior_eval which=1] */
    double* v_int;             /* (n_int) prior variance at x_int  */
    double* L;                 /* (n_int, n_int) row-major lower Cholesky factor [cbo_posterior_fit]; for n_int <= 48 its strict upper
                                  triangle carries L^-T, which cbo_sweep multiplies by on the FP64 tensor pipe (16 < n_int <= 48) */
    double* alpha;             /* (n_int) Ky^-1 (y - m) */
    double* sqrt_v_int;        /* (n_int) sqrt(v_int) */
    int32_t* fit_info;         /* [0] jitter retries used (0..5), [1] 0 ok / 1 not positive definite */
    /* ---- acquisition ----------------------------------------------------------------------------- */
    double cost_fix;           /* sum of the fixed costs of the set's variables (cost_functions.py:11-17) */
    int32_t cost_variable;     /* 1: add sum_k |x_k| per candidate (GraphInterface.py:46-50) */
    int32_t prior_external;    /* 1: m_int, v_int, m, v are supplied by the caller (e.g. produced by the mean/variance
                                  closures of DoCalculus); build_tables / prior_precompute / prior_eval skip the set */
    /* ---- per-candidate arrays, indexed by (g - g_begin) ----------------------------------------- */
    double* m;                 /* (g_count) prior mean       [cbo_prior_eval which=0]; required when causal */
    double* v;                 /* (g_count) prior variance */
    double* mu;                /* optional (may be NULL): posterior mean */
    double* var;               /* optional: posterior variance incl. 1e-10 noise */
    double* ei;                /* optional: expected improvement */
    double* acq;               /* optional: ei / cost */
    /* ---- explicit candidates instead of a tensor grid (model.predict(X) / acquisition.evaluate(X) on arbitrary X) ---- */
    int32_t posterior_cached;  /* 1: cbo_sweep reads this set's mu / var arrays (written by an earlier sweep with the same
                                  interventional data) instead of recomputing them: the 16 B/candidate EI refresh of a
                                  post-intervention trial for the sets that were not intervened on */
    int32_t int_row_begin;     /* cbo_prior_eval which=1 evaluates the interventional rows [int_row_begin, n_int) and leaves
                                  m_int / v_int of the earlier rows untouched (a post-intervention trial appends one row);
                                  0 = all rows */
    const double* y_obs;       /* (n_obs) training targets of the observational GP; only read by cbo_obs_gp_fit, which WRITES
                                  alpha_obs and kyinv from them (NULL: the caller supplies alpha_obs / kyinv itself) */
    const double* points;      /* NULL: tensor grid.  Otherwise (g_total, d) row-major candidates; then p[0] = g_total,
                                  p[1..] = 1, grid[] is unused and tab[0] is the (g_total, n_obs_pad) exp table of the points */
    /* ---- hyper-parameters of the per-set GP (ABI 9) ------------------------------------------------ */
    double* hyper;             /* NULL: the reference's RBF variance 1 and lengthscale 1.  Otherwise two device doubles
                                  (s2, l) read by cbo_posterior_fit, cbo_sweep, cbo_acq_grad and cbo_refine, and written by
                                  cbo_posterior_hyper_fit:  k(x, x') = s2 exp(-.5 |x - x'|^2 / l^2) [+ sqrt(v(x)) sqrt(v(x'))] */
} cbo_set_desc;

/* Result of one sweep on one rank. */
typedef struct cbo_set_best {
    double value;     /* max acquisition over the rank's slice of the set; -inf when the slice is empty */
    int64_t index;    /* flat grid index of the first maximiser; -1 when empty */
    int32_t n_nan;    /* candidates of the slice whose acquisition was NaN */
    int32_t reserved;
} cbo_set_best;

typedef struct cbo_sweep_result {
    double value;      /* best acquisition over all sets (ties: lowest set, then lowest index; NaN = -inf) */
    int64_t index;     /* flat grid index inside the set */
    int32_t set;       /* exploration-set index; -1 when nothing was evaluated */
    int32_t n_nan;     /* candidates whose acquisition was NaN (negative predictive variance) */
} cbo_sweep_result;

CBO_API int cbo_abi_version(void);
CBO_API size_t cbo_sizeof_set_desc(void);
/* Offset of a named field of cbo_set_desc, or -1: lets a foreign-language binding verify its mirror. */
CBO_API long cbo_offsetof_set_desc(const char* field);
CBO_API const char* cbo_last_error(void);
/* Kernels launched by this library from the calling thread since it was loaded (diagnostic; bench.py's gpu_launches). */
CBO_API unsigned long long cbo_launch_count(void);

/* Number of sweep work items (tiles of CBO_SWEEP_TILE candidates) for this descriptor list; host-side
 * arithmetic only.  Callers size `d_tile_best` with it. */
CBO_API long cbo_sweep_num_items(const cbo_set_desc* h_sets, int num_sets);

/* K5. exact-inference state of the observational GPs on the device: for every set with y_obs != NULL,
 *   Ky = s2 exp(-.5 r^2) + (noise + 1e-8 + jitter) I ,  L = chol(Ky) ,  alpha_obs = Ky^-1 y_obs ,  kyinv = Ky^-1
 * written through the descriptor's alpha_obs / kyinv pointers (blocked Cholesky, triangular inverse and L^-T L^-1 on the
 * FP64 tensor pipe).  Replaces the GPRegression(...) inside fit_gaussian_process (utils.py:40-45; GPy exact inference with
 * dpotrs / dpotri) for frozen hyper-parameters.  d_info[s] = 0 ok, 1 + panel index when a pivot was not positive: the
 * caller retries with jitter = mean(diag Ky) * 1e-6 * 10^t (GPy's jitchol rule).  Sets are processed one after the other
 * in the same workspace (cbo_obs_gp_workspace_bytes: the largest set's 2 Npad^2 + O(Npad) doubles). */
CBO_API size_t cbo_obs_gp_workspace_bytes(const cbo_set_desc* h_sets, int num_sets);
CBO_API int cbo_obs_gp_fit(const cbo_set_desc* h_sets, int num_sets, double jitter, void* d_workspace, size_t workspace_bytes,
                           int32_t* d_info, void* stream);

/* Objective of the hyper-parameter search around K5 (gp.optimize() in fit_gaussian_process, utils.py:44), for ONE set whose
 * state was just produced by cbo_obs_gp_fit in the same workspace:
 *   d_out[0] = -log p(y | X, s2, l) = 0.5 y.alpha + sum log L_ii + 0.5 N log(2 pi)
 *   d_out[1] = d/d log s2 ,  d_out[2 + k] = d/d log l_k  (k over the intervened, then the conditioning columns; sum them
 *   for a shared lengthscale); the noise is fixed (utils.py:43).  d_out: 2 + d + c device doubles. */
CBO_API int cbo_obs_gp_nll(const cbo_set_desc* h_set, void* d_workspace, size_t workspace_bytes, double* d_out, void* stream);

/* K0. exp tables: tab[k][i][j] = exp(-.5 ((grid[k][i] - x_obs_int[k][j]) / ls_int[k])^2) and
 * u_int[i][j] = exp(-.5 sum_k ((x_int[i][k] - x_obs_int[k][j]) / ls_int[k])^2).
 * Replaces the kernel evaluations inside gp.predict at DoCalculus.py:77 for the intervened columns.
 * `d_sets` (required) is read by the kernel: every table of every set is written by ONE launch. */
CBO_API int cbo_build_tables(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, void* stream);

/* K1a. P, pbar, w, M from the observational GP state and the conditioning samples.
 * Replaces the per-candidate np.hstack + gp.predict set-up of DoCalculus.py:68-89 (done once per
 * observation instead of once per candidate; SURVEY.md App. A.5).
 * `d_sets` (required) is read by the kernels.  Sets without conditioning columns share one launch.  The others run two
 * stages, P then M; consecutive sets share one launch per stage unless a set's P overlaps another set's (such sets run
 * one after the other) or its N is large enough to fill the GPU on its own (then it runs alone, on the TMA pipeline). */
CBO_API int cbo_prior_precompute(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, void* stream);

/* K1b. causal prior m(x) = u.w, v(x) = s2 + noise - u^T M u.
 * which = 0: on the rank's slice of the tensor grid, or on explicit points (writes m, v).  FP64 tensor pipe (DMMA);
 *            persistent kernel, one CTA per SM; each CTA materialises the 128 x n_obs_pad table product of its current
 *            128 candidates in a private slot of `d_workspace`.  Launches with too few 128-candidate tiles to fill the
 *            GPU cut every tile's triangle of M into segments (deterministic partial sums).
 *            Small observational sets on 2-D / 3-D tensor grids (n_obs <= 256: the reference's shipped data, 100..200
 *            rows) take a different decomposition when the call holds at least one work item per SM: u^T M u is
 *            regrouped over the n_obs (n_obs + 1) / 2 index pairs of the symmetric M, so that a whole plane of the
 *            grid is one GEMM between two small per-dimension "pair tables" kept in `d_workspace`
 *            (csrc/prior_pair.cu); cbo_prior_pair_items tells which decomposition a call will use.
 * which = 1: on the interventional rows x_int[int_row_begin .. n_int) (writes m_int, v_int).  These values are the
 *            inputs of the per-set fit, which amplifies their error by the Gram's condition number, so they are
 *            accumulated in compensated (double-double) arithmetic; one pass over M, HBM-bound for a single appended row.
 * Replaces DoCalculus.update_do_function (DoCalculus.py:34-66), index 0 and 1 together.
 * `d_workspace`: device memory, 256-byte aligned, sized with cbo_prior_workspace_bytes(h_sets, num_sets, num_ctas);
 * num_ctas = the SM count uses the whole GPU, fewer slots run fewer CTAs, at least one slot is required. */
CBO_API size_t cbo_prior_workspace_bytes(const cbo_set_desc* h_sets, int num_sets, int num_ctas);
CBO_API int cbo_prior_eval(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, int which,
                           void* d_workspace, size_t workspace_bytes, void* stream);
/* Host-side arithmetic only: the number of (scale row, tile) work items the pair-table decomposition of
 * cbo_prior_eval(which = 0) would run for this descriptor list on a device with `num_sms` SMs and a workspace sized
 * by cbo_prior_workspace_bytes; 0 when every set goes through the general kernel. */
CBO_API long cbo_prior_pair_items(const cbo_set_desc* h_sets, int num_sets, int num_sms);
/* Host-side arithmetic only: FP64 flops (2 per multiply-add) that the DMMA instructions of ONE cbo_prior_eval(which = 0)
 * call issue for this descriptor list -- the numerator of the kernel's FP64-pipe utilisation (bench.py's roofline).
 * General kernel: per candidate, the lower block triangle of M in 128 x 128 blocks (ragged last column block re-tiled);
 * pair-table kernel: per work item, (live 8 x 8 blocks of the tile) x (pair + mean columns, padded to 16). */
CBO_API double cbo_prior_eval_flops(const cbo_set_desc* h_sets, int num_sets, int num_sms);

/* K2. one CTA per set: Gram of the interventional rows (CausalRBF.K, causal_kernels.py:45-62, or RBF; variance and
 * lengthscale from `hyper`, 1 when it is NULL),
 * + (1e-10 + 1e-8) I, Cholesky with GPy's jitter-retry rule, alpha = Ky^-1 (y - m).
 * Replaces GPRegression(...) at GaussianProcessFactory.py:57-73 (GPy ExactGaussianInference). */
CBO_API int cbo_posterior_fit(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, void* stream);

/* K3 + K4. per candidate: k*, mu, forward substitution, var, EI, / cost; per-tile first-argmax; then a
 * deterministic reduction to per-set bests and the global best.
 * Replaces model.predict + CausalExpectedImprovement.evaluate + Cost.evaluate + the anchor top-1
 * (causal_acquisition_functions.py:27-43, utils.py:29-37, causal_optimizer.py:52-55) and
 * CBO.select_next_intervention (CBO.py:269-277).
 * task_sign: +1 for task 'min', -1 for 'max' (causal_acquisition_functions.py:38-41).
 * d_tile_best: device scratch of cbo_sweep_num_items() cbo_set_best entries; outputs: d_set_best
 * (num_sets entries), d_result (1 entry). */
CBO_API int cbo_sweep(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, double best,
              int task_sign, cbo_set_best* d_tile_best, cbo_set_best* d_set_best,
              cbo_sweep_result* d_result, void* stream);

/* A whole post-intervention trial in ONE call (CBO.update_gaussian_process_of_last_intervention + compute_best_acquisition_values,
 * CBO.py:224-260, after Monitor.add_intervention_data :148-160 appended one row to set `refit_set`): uploads the descriptor
 * array (it carries the trial's n_int / int_row_begin / posterior_cached flags), evaluates the interventional-row table and
 * the prior of the rows [int_row_begin, n_int) of that set only, refits it, and sweeps every set -- sets marked
 * posterior_cached only refresh EI from their mu / var arrays (16 B per candidate).  refit_set = -1: sweep only.
 * Six launches and one 488 B x num_sets copy; the per-stage entry points above remain for callers that time the stages. */
CBO_API int cbo_refresh_trial(const cbo_set_desc* h_sets, cbo_set_desc* d_sets, int num_sets, int refit_set, double best,
                              int task_sign, void* d_workspace, size_t workspace_bytes, cbo_set_best* d_tile_best,
                              cbo_set_best* d_set_best, cbo_sweep_result* d_result, void* stream);

/* K8. Marginal-likelihood fit of the per-set GP's hyper-parameters (opt-in).
 * The reference calls models[i].optimize() after every intervention (CBO.py:173) and then rebuilds the model with l = 1,
 * s2 = 1 (SURVEY.md App. B #16); this is the fit it meant to keep, of exactly the model cbo_posterior_fit then builds:
 *   Ky = s2 exp(-.5 r^2 / l^2) [+ sqrt(v_int) sqrt(v_int)^T] + (1e-10 + 1e-8 + jitter) I ,  r = y - m_int (or y)
 *   NLL = .5 r^T Ky^-1 r + sum log L_ii + .5 n log(2 pi)   (jitter: K2's rule, mean(diag) 1e-6 10^t, t = 0..4)
 * cbo_posterior_nll: d_out[3 s .. 3 s + 2] = NLL and its derivatives in log s2 and log l at the set's current `hyper`
 * (NULL = (1, 1)); one CTA per set, every set needs m_int / v_int (causal) and x_int / y_int on the device.
 * cbo_posterior_hyper_fit: per set, CBO_HYPER_STARTS deterministic starts (start 0 = (1, 1) clipped to the box, the others
 * a lattice from the bounds and var(r)), one CTA each, a projected BFGS in (log s2, log l) inside
 * h_bounds[4 s .. 4 s + 3] = (s2_lo, s2_hi, l_lo, l_hi) (HOST memory: checked, then copied into the workspace) with Armijo backtracking (steps 1, 1/2, .., 1/128); stop when
 * max |projected gradient| <= gtol or after max_iter line searches.  A reduction keeps each set's lowest NLL (ties: lowest
 * start; NaN = +inf) and writes it through `hyper`; a set none of whose starts has a positive-definite Gram keeps its
 * `hyper`.  Bit-identical across runs and independent of the other sets of the call.  Every set needs hyper != NULL. */
#define CBO_HYPER_STARTS 9
enum {
    CBO_HYPER_CONVERGED = 0,          /* max |projected gradient| <= gtol */
    CBO_HYPER_MAX_ITER = 1,           /* max_iter line searches done */
    CBO_HYPER_LINE_SEARCH_FAILED = 2, /* no backtracking step lowered the NLL (Armijo) */
    CBO_HYPER_NOT_PD = 3              /* the Gram was not positive definite, even with jitter, at every start: hyper unchanged */
};
typedef struct cbo_hyper_result {
    double variance, lengthscale;  /* the set's (s2, l) after the call */
    double nll;                    /* -log p(y) there */
    double nll_start;              /* -log p(y) at (1, 1) (NaN if not positive definite there) */
    int32_t iterations;            /* line searches of the winning start */
    int32_t status;                /* CBO_HYPER_* of the winning start */
    int32_t start;                 /* index of the winning start, -1 when none succeeded */
    int32_t jitter_tries;          /* jitter retries of the Cholesky at the result */
} cbo_hyper_result;
CBO_API int cbo_posterior_nll(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, double* d_out, void* stream);
CBO_API size_t cbo_posterior_hyper_workspace_bytes(const cbo_set_desc* h_sets, int num_sets);
CBO_API int cbo_posterior_hyper_fit(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, const double* h_bounds,
                                    int max_iter, double gtol, void* d_workspace, size_t workspace_bytes, cbo_hyper_result* d_out,
                                    void* stream);

/* K4 (multi-GPU). Combine `num_ranks` gathered per-set bests (rank-major: [rank][set]) into the global
 * per-set bests and the global result with the same rule on every rank.  Runs on the device so the
 * all-gathered buffer never leaves it. */
CBO_API int cbo_argmax_combine(const cbo_set_best* d_gathered, int num_ranks, int num_sets,
                       cbo_set_best* d_set_best, cbo_sweep_result* d_result, void* stream);

/* K7. Continuous refinement of each exploration set's acquisition maximum (opt-in).
 * Replaces the reference's L-BFGS polish of the best anchor, causal_optimizer.py:52-62, and the gradient it consumes,
 * CausalExpectedImprovement.evaluate_with_gradients / Cost (causal_acquisition_functions.py:45-67): the value and gradient
 * of acq(x) = EI(x) / cost(x) for one set at arbitrary points, and a projected quasi-Newton ascent of acq inside the box
 * [min grid[k], max grid[k]] that starts at a caller-given point (the grid argmax of a preceding cbo_sweep).
 * Every iteration is one pass over M's lower block triangle for the set's 8 trial points (value and gradient of the
 * causal prior, csrc/refine.cu) and one step kernel per set; no host synchronisation except a 4-byte poll of the sets
 * still running every few iterations.  Results are bit-identical across runs and do not depend on which other sets share
 * the call.  The device state the sweep left behind is read, never written: M, w, x_obs_int, L, alpha, sqrt_v_int, x_int,
 * grid. */
enum {
    CBO_REFINE_CONVERGED = 0,         /* small projected gradient or a negligible step */
    CBO_REFINE_MAX_ITER = 1,          /* max_iter iterations done */
    CBO_REFINE_LINE_SEARCH_FAILED = 2, /* none of the 8 trial steps along the gradient direction raised acq (Armijo) */
    CBO_REFINE_SKIPPED_EXTERNAL = 3,  /* prior_external: no device prior to differentiate */
    CBO_REFINE_SKIPPED_POINTS = 4,    /* explicit candidate points (points != NULL): no box */
    CBO_REFINE_SKIPPED_NONFINITE = 5  /* the start point has a NaN coordinate, or acq there is NaN / +-inf */
};
typedef struct cbo_acq_grad_out {      /* one explicit point; d* = gradient with respect to x (entries >= d are 0) */
    double m, v, mu, var, ei, acq;     /* prior mean / variance, posterior mean / variance (incl. 1e-10), EI, EI / cost */
    double dm[CBO_MAX_D], dv[CBO_MAX_D], dmu[CBO_MAX_D], dvar[CBO_MAX_D], dei[CBO_MAX_D], dacq[CBO_MAX_D];
} cbo_acq_grad_out;
typedef struct cbo_refine_result {     /* one set */
    double x[CBO_MAX_D];  /* refined point; the start point itself when value <= start_value or the set was skipped */
    double value;         /* acq(x) (refinement arithmetic); equals start_value when no step improved it */
    double start_value;   /* acq at the start point in the same arithmetic (NaN when skipped) */
    int32_t iterations;   /* line searches performed */
    int32_t status;       /* CBO_REFINE_* */
} cbo_refine_result;
/* Workspace of cbo_refine for this descriptor list, and of cbo_acq_grad for one set (which then evaluates its points 8 at
 * a time, more per launch when the workspace is larger). */
CBO_API size_t cbo_refine_workspace_bytes(const cbo_set_desc* h_sets, int num_sets);
/* Value and gradient of the prior, posterior, EI and acq of ONE set at d_points (num_points, d) row-major, with the set's
 * current device state (causal sets need the prior precompute, every set the posterior fit).  d_out: num_points entries. */
CBO_API int cbo_acq_grad(const cbo_set_desc* h_set, const cbo_set_desc* d_set, const double* d_points, int num_points,
                         double best, int task_sign, void* d_workspace, size_t workspace_bytes,
                         cbo_acq_grad_out* d_out, void* stream);
/* Refine every set from d_x0 (num_sets, CBO_MAX_D) device doubles; a row holding a NaN skips its set.  max_iter line
 * searches at most; gtol: stop when max_k |projected d acq / dx_k| (max grid[k] - min grid[k]) <= gtol |acq|.
 * d_out: num_sets entries.  Sets with prior_external or explicit points are skipped (status says why). */
CBO_API int cbo_refine(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, double best, int task_sign,
                       const double* d_x0, int max_iter, double gtol,
                       void* d_workspace, size_t workspace_bytes, cbo_refine_result* d_out, void* stream);

/* K6. Ground truth of an intervention: E[target | do(...)] of a structural equation model by Monte Carlo.
 * Replaces compute_interventions / sample_from_model / intervene_dict (graph_functions.py:8-77: 100 000 samples in a Python
 * loop per intervention; the function reseeds with seed 1 on every call, so the noise matrix is a constant of the run and
 * stays on the device).  The SEM is a program over nodes in topological order:
 *   value[i] = constant_i + sum_t coef_t * f_t(scale_t * source_t) ,  source_t = noise[src] when src < num_noise, else
 *   value[src - num_noise] (an earlier node);  an intervened node (do_mask) takes do_value instead.
 * d_noise: (num_noise, num_samples) row-major; d_do_mask / d_do_value: (batch, num_nodes); d_partials: scratch of
 * batch * CBO_SEM_BLOCKS doubles; d_mean: (batch) Monte-Carlo means of the target node (deterministic summation order). */
#define CBO_SEM_MAX_NODES 16
#define CBO_SEM_MAX_TERMS 96
#define CBO_SEM_BLOCKS 64
enum { CBO_SEM_ID = 0, CBO_SEM_EXP = 1, CBO_SEM_COS = 2, CBO_SEM_SIN = 3, CBO_SEM_SQUARE = 4 };
typedef struct cbo_sem_term { int32_t src; int32_t func; double coef; double scale; } cbo_sem_term;
typedef struct cbo_sem_node { int32_t first_term; int32_t num_terms; double constant; } cbo_sem_node;
CBO_API int cbo_sem_eval(const cbo_sem_node* d_nodes, int num_nodes, const cbo_sem_term* d_terms, int num_terms,
                         const double* d_noise, int num_noise, long long num_samples, const int32_t* d_do_mask,
                         const double* d_do_value, int batch, int target_node, double* d_partials, double* d_mean, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CBO_B200_H */
