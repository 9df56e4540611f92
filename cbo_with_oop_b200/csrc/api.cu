// extern "C" surface of libcbo_b200.so (declared in include/cbo_b200.h).  No torch types, no exceptions, no
// allocation: plain pointers and sizes in, status code out.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>
#include <stddef.h>

#include "cbo_common.cuh"

namespace cbo {

static thread_local char g_error[512] = "";
static thread_local unsigned long long g_launches = 0;

void note_launch(int n) { g_launches += (unsigned long long)n; }
unsigned long long launch_count() { return g_launches; }

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
    set_error("%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
    return (int)e;
}

int validate_sets(const cbo_set_desc* h_sets, int num_sets) {
    CBO_REQUIRE(h_sets != nullptr, "descriptor array is NULL");
    CBO_REQUIRE(num_sets >= 1 && num_sets <= 4096, "num_sets=%d outside [1,4096]", num_sets);
    for (int s = 0; s < num_sets; ++s) {
        const cbo_set_desc& S = h_sets[s];
        CBO_REQUIRE(S.d >= 1 && S.d <= CBO_MAX_D, "set %d: d=%d outside [1,%d]", s, S.d, CBO_MAX_D);
        CBO_REQUIRE(S.c >= 0 && S.c <= CBO_MAX_C, "set %d: c=%d outside [0,%d]", s, S.c, CBO_MAX_C);
        CBO_REQUIRE(S.n_int >= 1 && S.n_int <= CBO_MAX_NINT, "set %d: n_int=%d outside [1,%d]", s, S.n_int, CBO_MAX_NINT);
        long long g = 1;
        for (int k = 0; k < S.d; ++k) {
            CBO_REQUIRE(S.p[k] >= 1, "set %d: p[%d]=%d < 1", s, k, S.p[k]);
            g *= S.p[k];
        }
        CBO_REQUIRE(g == S.g_total, "set %d: g_total=%lld != prod p = %lld", s, (long long)S.g_total, g);
        CBO_REQUIRE(S.g_begin >= 0 && S.g_count >= 0 && S.g_begin + S.g_count <= S.g_total,
                    "set %d: slice [%lld,+%lld) outside the grid of %lld", s, (long long)S.g_begin, (long long)S.g_count, g);
        CBO_REQUIRE(!S.points || (S.p[0] == S.g_total), "set %d: explicit points need p[0] == g_total", s);
        if (S.causal && !S.prior_external) {
            CBO_REQUIRE(S.n_obs >= 1 && S.n_obs_pad >= S.n_obs && S.n_obs_pad % CBO_NPAD == 0,
                        "set %d: n_obs=%d n_obs_pad=%d (pad must be a multiple of %d)", s, S.n_obs, S.n_obs_pad, CBO_NPAD);
            CBO_REQUIRE(S.c == 0 || (S.n_mc >= 1 && S.n_mc_pad >= S.n_mc && S.n_mc_pad % CBO_SPAD == 0),
                        "set %d: n_mc=%d n_mc_pad=%d (pad must be a multiple of %d)", s, S.n_mc, S.n_mc_pad, CBO_SPAD);
            for (int k = 0; k < S.d; ++k) CBO_REQUIRE(S.ls_int[k] > 0.0, "set %d: ls_int[%d] must be positive", s, k);
            for (int k = 0; k < S.c; ++k) CBO_REQUIRE(S.ls_cond[k] > 0.0, "set %d: ls_cond[%d] must be positive", s, k);
        }
        CBO_REQUIRE(S.cost_fix > 0.0 || S.cost_variable, "set %d: cost would be zero", s);
    }
    return 0;
}

int build_tables_impl(const cbo_set_desc*, const cbo_set_desc*, int, cudaStream_t);
int prior_precompute_impl(const cbo_set_desc*, const cbo_set_desc*, int, cudaStream_t);
int prior_eval_impl(const cbo_set_desc*, const cbo_set_desc*, int, int, void*, size_t, cudaStream_t);
size_t prior_workspace_bytes_impl(const cbo_set_desc*, int, int);
long long pair_items_total(const cbo_set_desc*, int);
double prior_eval_flops_impl(const cbo_set_desc*, int, int);
int posterior_fit_impl(const cbo_set_desc*, const cbo_set_desc*, int, cudaStream_t);
int sweep_impl(const cbo_set_desc*, const cbo_set_desc*, int, double, int, cbo_set_best*, cbo_set_best*, cbo_sweep_result*,
               cudaStream_t);
int argmax_combine_impl(const cbo_set_best*, int, int, cbo_set_best*, cbo_sweep_result*, cudaStream_t);
size_t obs_gp_workspace_bytes_impl(const cbo_set_desc*, int);
int obs_gp_fit_impl(const cbo_set_desc*, int, double, void*, size_t, int32_t*, cudaStream_t);
int obs_gp_nll_impl(const cbo_set_desc*, void*, size_t, double*, cudaStream_t);
int int_rows_table_impl(const cbo_set_desc&, const cbo_set_desc*, cudaStream_t);
size_t refine_workspace_bytes_impl(const cbo_set_desc*, int);
int acq_grad_impl(const cbo_set_desc*, const cbo_set_desc*, const double*, int, double, int, void*, size_t, cbo_acq_grad_out*, cudaStream_t);
int refine_impl(const cbo_set_desc*, const cbo_set_desc*, int, double, int, const double*, int, double, void*, size_t, cbo_refine_result*,
                cudaStream_t);
int posterior_nll_impl(const cbo_set_desc*, const cbo_set_desc*, int, double*, cudaStream_t);
size_t hyper_workspace_bytes_impl(int);
int hyper_fit_impl(const cbo_set_desc*, const cbo_set_desc*, int, const double*, int, double, void*, size_t, cbo_hyper_result*,
                   cudaStream_t);
int sem_eval_impl(const cbo_sem_node*, int, const cbo_sem_term*, int, const double*, int, long long, const int32_t*, const double*, int,
                  int, double*, double*, cudaStream_t);

}  // namespace cbo

using namespace cbo;

extern "C" {

int cbo_abi_version(void) { return CBO_ABI_VERSION; }
unsigned long long cbo_launch_count(void) { return launch_count(); }
size_t cbo_sizeof_set_desc(void) { return sizeof(cbo_set_desc); }
const char* cbo_last_error(void) { return g_error; }

long cbo_offsetof_set_desc(const char* field) {
    if (!field) return -1;
#define F(name) if (strcmp(field, #name) == 0) return (long)offsetof(cbo_set_desc, name);
    F(d) F(c) F(n_obs) F(n_obs_pad) F(n_mc) F(n_mc_pad) F(n_int) F(causal) F(p) F(g_total) F(g_begin) F(g_count)
    F(x_obs_int) F(x_obs_cond) F(mc_cond) F(alpha_obs) F(kyinv) F(ls_int) F(ls_cond) F(s2) F(noise)
    F(tab) F(u_int) F(P) F(pbar) F(w) F(M) F(grid) F(x_int) F(y_int) F(m_int) F(v_int) F(L) F(alpha) F(sqrt_v_int)
    F(fit_info) F(cost_fix) F(cost_variable) F(prior_external) F(m) F(v) F(mu) F(var) F(ei) F(acq) F(posterior_cached) F(int_row_begin) F(y_obs) F(points) F(hyper)
#undef F
    return -1;
}

long cbo_sweep_num_items(const cbo_set_desc* h_sets, int num_sets) {
    if (!h_sets || num_sets < 0) return -1;
    long long t = 0;
    for (int s = 0; s < num_sets; ++s) t += host_items(h_sets[s], kItemsSweep);
    return (long)t;
}

size_t cbo_obs_gp_workspace_bytes(const cbo_set_desc* h_sets, int num_sets) {
    if (!h_sets || num_sets < 1) return 0;
    return obs_gp_workspace_bytes_impl(h_sets, num_sets);
}

int cbo_obs_gp_fit(const cbo_set_desc* h_sets, int num_sets, double jitter, void* d_workspace, size_t workspace_bytes,
                   int32_t* d_info, void* stream) {
    if (int rc = validate_sets(h_sets, num_sets)) return rc;
    CBO_REQUIRE(jitter >= 0.0, "cbo_obs_gp_fit: jitter must be non-negative");
    return obs_gp_fit_impl(h_sets, num_sets, jitter, d_workspace, workspace_bytes, d_info, (cudaStream_t)stream);
}

int cbo_obs_gp_nll(const cbo_set_desc* h_set, void* d_workspace, size_t workspace_bytes, double* d_out, void* stream) {
    if (int rc = validate_sets(h_set, 1)) return rc;
    return obs_gp_nll_impl(h_set, d_workspace, workspace_bytes, d_out, (cudaStream_t)stream);
}

int cbo_build_tables(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, void* stream) {
    if (int rc = validate_sets(h_sets, num_sets)) return rc;
    CBO_REQUIRE(d_sets != nullptr, "cbo_build_tables: d_sets is NULL");
    return build_tables_impl(h_sets, d_sets, num_sets, (cudaStream_t)stream);
}

int cbo_prior_precompute(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, void* stream) {
    if (int rc = validate_sets(h_sets, num_sets)) return rc;
    CBO_REQUIRE(d_sets != nullptr, "cbo_prior_precompute: d_sets is NULL");
    return prior_precompute_impl(h_sets, d_sets, num_sets, (cudaStream_t)stream);
}

size_t cbo_prior_workspace_bytes(const cbo_set_desc* h_sets, int num_sets, int num_ctas) {
    if (!h_sets || num_sets < 1 || num_ctas < 1) return 0;
    return prior_workspace_bytes_impl(h_sets, num_sets, num_ctas);
}

long cbo_prior_pair_items(const cbo_set_desc* h_sets, int num_sets, int num_sms) {
    if (!h_sets || num_sets < 1 || num_sms < 1) return 0;
    const long long t = pair_items_total(h_sets, num_sets);
    return t >= num_sms ? (long)t : 0;
}

double cbo_prior_eval_flops(const cbo_set_desc* h_sets, int num_sets, int num_sms) {
    if (!h_sets || num_sets < 1 || num_sms < 1) return 0.0;
    return prior_eval_flops_impl(h_sets, num_sets, num_sms);
}

int cbo_prior_eval(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, int which, void* d_workspace,
                   size_t workspace_bytes, void* stream) {
    if (int rc = validate_sets(h_sets, num_sets)) return rc;
    CBO_REQUIRE(d_sets != nullptr, "cbo_prior_eval: d_sets is NULL");
    CBO_REQUIRE(which == 0 || which == 1, "cbo_prior_eval: which=%d must be 0 (grid) or 1 (x_int)", which);
    for (int s = 0; s < num_sets; ++s) {
        const cbo_set_desc& S = h_sets[s];
        if (!computes_prior(S)) continue;
        CBO_REQUIRE(S.M && S.w, "cbo_prior_eval: set %d has NULL M/w", s);
        if (which == 0) {
            CBO_REQUIRE(S.g_count == 0 || (S.m && S.v), "cbo_prior_eval: set %d has NULL m/v", s);
            for (int k = 0; k < (S.points ? 1 : S.d); ++k) CBO_REQUIRE(S.tab[k], "cbo_prior_eval: set %d tab[%d] is NULL", s, k);
        } else {
            CBO_REQUIRE(S.u_int && S.m_int && S.v_int, "cbo_prior_eval: set %d has NULL u_int/m_int/v_int", s);
        }
    }
    return prior_eval_impl(h_sets, d_sets, num_sets, which, d_workspace, workspace_bytes, (cudaStream_t)stream);
}

int cbo_posterior_fit(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, void* stream) {
    if (int rc = validate_sets(h_sets, num_sets)) return rc;
    CBO_REQUIRE(d_sets != nullptr, "cbo_posterior_fit: d_sets is NULL");
    return posterior_fit_impl(h_sets, d_sets, num_sets, (cudaStream_t)stream);
}

int cbo_sweep(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, double best, int task_sign,
              cbo_set_best* d_tile_best, cbo_set_best* d_set_best, cbo_sweep_result* d_result, void* stream) {
    if (int rc = validate_sets(h_sets, num_sets)) return rc;
    CBO_REQUIRE(d_sets != nullptr, "cbo_sweep: d_sets is NULL");
    return sweep_impl(h_sets, d_sets, num_sets, best, task_sign, d_tile_best, d_set_best, d_result, (cudaStream_t)stream);
}

int cbo_refresh_trial(const cbo_set_desc* h_sets, cbo_set_desc* d_sets, int num_sets, int refit_set, double best, int task_sign,
                      void* d_workspace, size_t workspace_bytes, cbo_set_best* d_tile_best, cbo_set_best* d_set_best,
                      cbo_sweep_result* d_result, void* stream) {
    if (int rc = validate_sets(h_sets, num_sets)) return rc;
    CBO_REQUIRE(d_sets != nullptr, "cbo_refresh_trial: d_sets is NULL");
    CBO_REQUIRE(refit_set >= -1 && refit_set < num_sets, "cbo_refresh_trial: refit_set=%d outside [-1,%d)", refit_set, num_sets);
    cudaStream_t st = (cudaStream_t)stream;
    // the descriptors carry this trial's flags (n_int, int_row_begin, posterior_cached): one small host -> device copy
    CBO_CUDA(cudaMemcpyAsync(d_sets, h_sets, (size_t)num_sets * sizeof(cbo_set_desc), cudaMemcpyHostToDevice, st));
    if (refit_set >= 0) {
        const cbo_set_desc* h = h_sets + refit_set;
        const cbo_set_desc* d = d_sets + refit_set;
        CBO_REQUIRE(!h->posterior_cached, "cbo_refresh_trial: the refitted set cannot be marked posterior_cached");
        if (computes_prior(*h)) {
            if (int rc = int_rows_table_impl(*h, d, st)) return rc;
            if (int rc = prior_eval_impl(h, d, 1, 1, d_workspace, workspace_bytes, st)) return rc;
        }
        if (int rc = posterior_fit_impl(h, d, 1, st)) return rc;
    }
    return sweep_impl(h_sets, d_sets, num_sets, best, task_sign, d_tile_best, d_set_best, d_result, st);
}

int cbo_argmax_combine(const cbo_set_best* d_gathered, int num_ranks, int num_sets, cbo_set_best* d_set_best,
                       cbo_sweep_result* d_result, void* stream) {
    CBO_REQUIRE(d_set_best && d_result, "cbo_argmax_combine: NULL output pointer");
    return argmax_combine_impl(d_gathered, num_ranks, num_sets, d_set_best, d_result, (cudaStream_t)stream);
}

size_t cbo_refine_workspace_bytes(const cbo_set_desc* h_sets, int num_sets) {
    if (!h_sets || num_sets < 1) return 0;
    return refine_workspace_bytes_impl(h_sets, num_sets);
}

int cbo_acq_grad(const cbo_set_desc* h_set, const cbo_set_desc* d_set, const double* d_points, int num_points, double best, int task_sign,
                 void* d_workspace, size_t workspace_bytes, cbo_acq_grad_out* d_out, void* stream) {
    if (int rc = validate_sets(h_set, 1)) return rc;
    return acq_grad_impl(h_set, d_set, d_points, num_points, best, task_sign, d_workspace, workspace_bytes, d_out, (cudaStream_t)stream);
}

int cbo_refine(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, double best, int task_sign, const double* d_x0,
               int max_iter, double gtol, void* d_workspace, size_t workspace_bytes, cbo_refine_result* d_out, void* stream) {
    if (int rc = validate_sets(h_sets, num_sets)) return rc;
    return refine_impl(h_sets, d_sets, num_sets, best, task_sign, d_x0, max_iter, gtol, d_workspace, workspace_bytes, d_out,
                       (cudaStream_t)stream);
}

int cbo_posterior_nll(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, double* d_out, void* stream) {
    if (int rc = validate_sets(h_sets, num_sets)) return rc;
    CBO_REQUIRE(d_sets != nullptr, "cbo_posterior_nll: d_sets is NULL");
    CBO_REQUIRE(d_out != nullptr, "cbo_posterior_nll: d_out is NULL");
    return posterior_nll_impl(h_sets, d_sets, num_sets, d_out, (cudaStream_t)stream);
}

size_t cbo_posterior_hyper_workspace_bytes(const cbo_set_desc* h_sets, int num_sets) {
    if (!h_sets || num_sets < 1) return 0;
    return hyper_workspace_bytes_impl(num_sets);
}

int cbo_posterior_hyper_fit(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, const double* h_bounds, int max_iter,
                            double gtol, void* d_workspace, size_t workspace_bytes, cbo_hyper_result* d_out, void* stream) {
    if (int rc = validate_sets(h_sets, num_sets)) return rc;
    CBO_REQUIRE(d_sets != nullptr, "cbo_posterior_hyper_fit: d_sets is NULL");
    return hyper_fit_impl(h_sets, d_sets, num_sets, h_bounds, max_iter, gtol, d_workspace, workspace_bytes, d_out, (cudaStream_t)stream);
}

int cbo_sem_eval(const cbo_sem_node* d_nodes, int num_nodes, const cbo_sem_term* d_terms, int num_terms, const double* d_noise,
                 int num_noise, long long num_samples, const int32_t* d_do_mask, const double* d_do_value, int batch, int target_node,
                 double* d_partials, double* d_mean, void* stream) {
    return sem_eval_impl(d_nodes, num_nodes, d_terms, num_terms, d_noise, num_noise, num_samples, d_do_mask, d_do_value, batch,
                         target_node, d_partials, d_mean, (cudaStream_t)stream);
}

}  // extern "C"
