// K0 -- separable RBF factors of the observational GP's cross-covariance on the intervened columns.
//
//   tab[k][i][j] = exp(-.5 ((grid_k[i] - X_obs[j, k]) / l_k)^2)          i < p_k, j < N   (0 for N <= j < Npad)
//   u_int[i][j]  = exp(-.5 sum_k ((x_int[i, k] - X_obs[j, k]) / l_k)^2)   i < n_int
//
// These are the k(Z_i(x), X_j) factors that the reference evaluates inside gp.predict for every candidate
// (DoCalculus.py:77 via get_intervened_inputs :80-89).  On a tensor grid u(x) is the elementwise product of one
// row per table, so the quadratic-form kernel never calls exp.  HBM-bound (one 8-byte store per exp),
// coalesced along j; a negligible share of a sweep.
#include "cbo_common.cuh"

namespace cbo {

// Every table of every set in one launch: blockIdx.z = set * (CBO_MAX_D + 1) + table.  Table k < d is the grid table of
// dimension k, table d is u_int.  A set with explicit points has no grid tables: its table 0 is tab[0] with one row per
// point, formed like a row of u_int.  int_rows_only: blockIdx.z = set, and only the rows [int_row_begin, n_int) of u_int.
__global__ void __launch_bounds__(256)
tables_kernel(const cbo_set_desc* __restrict__ sets, bool int_rows_only) {
    const cbo_set_desc& S = sets[int_rows_only ? blockIdx.z : blockIdx.z / (CBO_MAX_D + 1)];
    const int d = S.d, k = int_rows_only ? d : blockIdx.z % (CBO_MAX_D + 1);
    if (!computes_prior(S) || k > d || (S.points && k > 0 && k < d)) return;
    const int n_obs = S.n_obs, n_obs_pad = S.n_obs_pad;
    const int j = blockIdx.x * 256 + threadIdx.x;
    if (j >= n_obs_pad) return;
    const bool live = j < n_obs;
    if (k < d && !S.points) {
        const double x = live ? S.x_obs_int[(size_t)k * n_obs + j] : 0.0, inv_l = 1.0 / S.ls_int[k];
        const double* __restrict__ coords = S.grid[k];
        double* __restrict__ out = S.tab[k];
        for (int i = blockIdx.y; i < S.p[k]; i += gridDim.y) {
            const double t = (coords[i] - x) * inv_l;
            out[(size_t)i * n_obs_pad + j] = live ? exp(-0.5 * (t * t)) : 0.0;
        }
        return;
    }
    // rows of d coordinates: the explicit points (table 0) or the interventional rows (table d)
    const bool points = k < d;
    const double* __restrict__ src = points ? S.points : S.x_int;
    double* __restrict__ out = points ? S.tab[0] : S.u_int;
    const int r0 = int_rows_only ? S.int_row_begin : 0, rows = points ? (int)S.g_total : S.n_int;
    double x[CBO_MAX_D], il[CBO_MAX_D];
#pragma unroll
    for (int q = 0; q < CBO_MAX_D; ++q) {
        x[q] = (live && q < d) ? S.x_obs_int[(size_t)q * n_obs + j] : 0.0;
        il[q] = q < d ? 1.0 / S.ls_int[q] : 0.0;
    }
    for (int i = r0 + blockIdx.y; i < rows; i += gridDim.y) {
        double r2 = 0.0;
#pragma unroll
        for (int q = 0; q < CBO_MAX_D; ++q) {
            if (q < d) {
                const double t = (src[i * d + q] - x[q]) * il[q];
                r2 += t * t;
            }
        }
        out[(size_t)i * n_obs_pad + j] = live ? exp(-0.5 * r2) : 0.0;
    }
}

static unsigned row_blocks(int rows) { return (unsigned)(rows < 1024 ? rows : 1024); }

// The interventional-row table of the refitted set of a post-intervention trial, rows [int_row_begin, n_int) only (the grid
// tables do not depend on x_int).  `d_set`: the set's descriptor on the device.
int int_rows_table_impl(const cbo_set_desc& S, const cbo_set_desc* d_set, cudaStream_t st) {
    if (!computes_prior(S) || S.int_row_begin >= S.n_int) return 0;
    CBO_REQUIRE(S.u_int && S.x_int && S.x_obs_int, "cbo_refresh_trial: NULL u_int/x_int/x_obs_int pointer");
    tables_kernel<<<dim3((S.n_obs_pad + 255) / 256, row_blocks(S.n_int - S.int_row_begin)), 256, 0, st>>>(d_set, true);
    note_launch();
    CBO_CUDA(cudaGetLastError());
    return 0;
}

int build_tables_impl(const cbo_set_desc* h_sets, const cbo_set_desc* d_sets, int num_sets, cudaStream_t st) {
    int npad_max = 0, rows_max = 1;
    for (int s = 0; s < num_sets; ++s) {
        const cbo_set_desc& S = h_sets[s];
        if (!computes_prior(S)) continue;
        if (S.points) {
            CBO_REQUIRE(S.tab[0] && S.x_obs_int, "cbo_build_tables: set %d has a NULL table pointer", s);
            CBO_REQUIRE(S.g_total < 2147483647LL / CBO_MAX_D, "cbo_build_tables: set %d has too many explicit points", s);
            if (S.g_total > rows_max) rows_max = (int)S.g_total;
        }
        for (int k = 0; k < (S.points ? 0 : S.d); ++k) {
            CBO_REQUIRE(S.tab[k] && S.grid[k] && S.x_obs_int, "cbo_build_tables: set %d has a NULL table/grid pointer", s);
            if (S.p[k] > rows_max) rows_max = S.p[k];
        }
        CBO_REQUIRE(S.u_int && S.x_int, "cbo_build_tables: set %d has a NULL u_int/x_int pointer", s);
        if (S.n_int > rows_max) rows_max = S.n_int;
        if (S.n_obs_pad > npad_max) npad_max = S.n_obs_pad;
    }
    if (npad_max == 0) return 0;
    // num_sets <= 4096 (validate_sets): the grid's z extent stays within 65535
    tables_kernel<<<dim3((npad_max + 255) / 256, row_blocks(rows_max), num_sets * (CBO_MAX_D + 1)), 256, 0, st>>>(d_sets, false);
    note_launch();
    CBO_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace cbo
