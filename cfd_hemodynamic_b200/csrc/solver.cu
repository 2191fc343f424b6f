// Block-Schur preconditioner and right-preconditioned FGMRES.
//
// Replaces KSP(fgmres) + PC(fieldsplit, SCHUR) configured by the reference at
// src/solvers/stabilized_schur.py:226-275.  Differences by design (DESIGN.md §5):
//   * upper block-triangular factorisation (one A00^-1 per application) instead of FULL;
//   * A00^-1 ~ AMG V-cycle(s) instead of GMRES(30)+ASM/ILU(0);
//   * S^-1 ~ c_m diag(Mp)^-1 + c_L Lp^-1 (Cahouet–Chabard) with an AMG V-cycle on
//     the pressure Laplacian instead of ILU(0) on SELFP.
// Parity with the reference is therefore on the converged solution, never on
// iteration counts.
#include <math.h>
#include <stdlib.h>

#include "hemo_internal.cuh"

int hemo_spmv_block(hemo_ctx* ctx, int rows, int cols, const double* vals, const double* xu, const double* xp,
                    double alpha, const double* bu, const double* bp, double* yu, double* yp);
int hemo_scale_copy(hemo_ctx* ctx, int64_t n, double a, const double* x, double* y);
int hemo_mdot(hemo_ctx* ctx, int64_t n, int k, const double* V, int64_t ldv, const double* w, double* h_host);
int hemo_maxpy(hemo_ctx* ctx, int64_t n, int k, const double* V, int64_t ldv, const double* hcoef_dev, double sign,
               double* w, double* norm_host);
int hemo_remove_mean(hemo_ctx* ctx, int64_t n, double* x);
int hemo_copy_remove_mean(hemo_ctx* ctx, int64_t n, const double* src, double* x);
int hemo_amg_numeric_shift(hemo_ctx* ctx, HemoAmg* amg, double coarse_shift);

// A00 (2x2 node blocks) out of the monolithic CSR values
__global__ void __launch_bounds__(256)
k_extract_a00(int64_t nnz_node, const int32_t* __restrict__ nrowptr, const int32_t* __restrict__ rowof,
              const int32_t* __restrict__ ncol, const uint8_t* __restrict__ mask,
              const double* __restrict__ vals, areal* __restrict__ out, areal2* __restrict__ a01) {
    const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= nnz_node) return;
    const int i = rowof[s];
    {
        // compact single-precision copy of A01 (rows u_x, u_y of node i, pressure column of node j)
        const int r0 = nrowptr[i];
        const int deg = nrowptr[i + 1] - r0;
        const int t = (int)(s - r0);
        const int64_t ru0 = 6 * (int64_t)r0, ru1 = ru0 + 3 * deg;
        areal2 g;
        g.x = (areal)vals[ru0 + 2 * deg + t];
        g.y = (areal)vals[ru1 + 2 * deg + t];
        a01[s] = g;
    }
    if (mask) {
        const int j = ncol[s];
        if (mask[i] || mask[j]) {      // ghost node of a partition: identity row/column in the local PC
            const areal d = (i == j) ? (areal)1 : (areal)0;
            areal2 r0v, r1v;
            r0v.x = d; r0v.y = 0; r1v.x = 0; r1v.y = d;
            reinterpret_cast<areal2*>(out)[2 * s] = r0v;
            reinterpret_cast<areal2*>(out)[2 * s + 1] = r1v;
            return;
        }
    }
    const int r0 = nrowptr[i];
    const int deg = nrowptr[i + 1] - r0;
    const int t = (int)(s - r0);
    const int64_t ru0 = 6 * (int64_t)r0, ru1 = ru0 + 3 * deg;
    areal2 a, b;
    a.x = (areal)vals[ru0 + 2 * t]; a.y = (areal)vals[ru0 + 2 * t + 1];
    b.x = (areal)vals[ru1 + 2 * t]; b.y = (areal)vals[ru1 + 2 * t + 1];
    reinterpret_cast<areal2*>(out)[2 * s] = a;
    reinterpret_cast<areal2*>(out)[2 * s + 1] = b;
}

// pressure Laplacian with identity rows/cols on Dirichlet pressure dofs
__global__ void __launch_bounds__(256)
k_lap_with_bc(int n, int64_t nnz_node, const int32_t* __restrict__ rowof, const int32_t* __restrict__ ncol,
              const double* __restrict__ lap, const uint8_t* __restrict__ dofflag /* pressure part, n */,
              areal* __restrict__ out) {
    const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= nnz_node) return;
    double v = lap[s];
    if (dofflag) {
        const int i = rowof[s], j = ncol[s];
        const bool fi = dofflag[i] != 0, fj = dofflag[j] != 0;
        if (fi || fj) v = (i == j) ? 1.0 : 0.0;
    }
    out[s] = (areal)v;
}

__global__ void k_areal_to_double(int64_t n, const areal* __restrict__ x, double* __restrict__ y) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) y[i] = (double)x[i];
}

// x[node*bs + k] = 0 on masked nodes
__global__ void k_mask_nodes(int n, int bs, const uint8_t* __restrict__ mask, double* __restrict__ x) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool masked = i < n && mask[i];
    hemo_pdl_wait();
    hemo_pdl_trigger();
    if (!masked) return;
    for (int k = 0; k < bs; ++k) x[(int64_t)i * bs + k] = 0.0;
}

// t_u = r_u - A01 z_p on the compact single-precision copy of A01 (4 lanes per node row)
__global__ void __launch_bounds__(256)
k_a01_residual(int n, const int32_t* __restrict__ nrowptr, const int32_t* __restrict__ ncol,
               const areal2* __restrict__ a01, const double* __restrict__ zp, const double* __restrict__ ru,
               double* __restrict__ tu) {
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = gt >> 2, lane = gt & 3;
    const bool ok = i < n;
    const int r0 = ok ? nrowptr[i] : 0, r1 = ok ? nrowptr[i + 1] : 0;
    // first entry of the lane (constant during the solve) before the wait
    areal2 g;
    g.x = g.y = 0;
    int c = 0;
    if (r0 + lane < r1) { g = a01[r0 + lane]; c = ncol[r0 + lane]; }
    hemo_pdl_wait();
    hemo_pdl_trigger();
    double a0 = 0.0, a1 = 0.0;
    for (int s = r0 + lane; s < r1; s += 4) {
        if (s != r0 + lane) { g = a01[s]; c = ncol[s]; }
        const double z = zp[c];
        a0 = fma((double)g.x, z, a0);
        a1 = fma((double)g.y, z, a1);
    }
#pragma unroll
    for (int o = 2; o > 0; o >>= 1) {
        a0 += __shfl_down_sync(0xffffffffu, a0, o, 4);
        a1 += __shfl_down_sync(0xffffffffu, a1, o, 4);
    }
    if (ok && lane == 0) {
        tu[2 * (int64_t)i] = ru[2 * (int64_t)i] - a0;
        tu[2 * (int64_t)i + 1] = ru[2 * (int64_t)i + 1] - a1;
    }
}

// the same with one thread per node row: the 7-9 entries of a fine-mesh row are requested four at a time before the
// first use (see sell_row_product in amg.cu for the scheduling fences)
__global__ void __launch_bounds__(256)
k_a01_residual_row(int n, const int32_t* __restrict__ nrowptr, const int32_t* __restrict__ ncol,
                   const areal2* __restrict__ a01, const double* __restrict__ zp, const double* __restrict__ ru,
                   double* __restrict__ tu) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool ok = i < n;
    const int r0 = ok ? nrowptr[i] : 0, r1 = ok ? nrowptr[i + 1] : 0;
    int j[4];
    areal2 g[4];
    // column indices and A01 entries of the first four (constant during the solve) before the wait
    auto fetch = [&](int s) {
        int t[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) t[u] = s + u < r1 ? s + u : r1 - 1;
#pragma unroll
        for (int u = 0; u < 4; ++u) j[u] = ncol[t[u]];
#pragma unroll
        for (int u = 0; u < 4; ++u) g[u] = a01[t[u]];
    };
    if (r0 < r1) fetch(r0);
    hemo_pdl_wait();
    hemo_pdl_trigger();
    if (!ok) return;
    double a0 = 0.0, a1 = 0.0;
    for (int s = r0; s < r1; s += 4) {
        double z[4];
        if (s != r0) fetch(s);
        __syncwarp(__activemask());
#pragma unroll
        for (int u = 0; u < 4; ++u) z[u] = zp[j[u]];
        __syncwarp(__activemask());
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const double m = s + u < r1 ? z[u] : 0.0;
            a0 = fma((double)g[u].x, m, a0);
            a1 = fma((double)g[u].y, m, a1);
        }
    }
    tu[2 * (int64_t)i] = ru[2 * (int64_t)i] - a0;          // (r_u may be a Krylov column: 8-byte alignment only)
    tu[2 * (int64_t)i + 1] = ru[2 * (int64_t)i + 1] - a1;
}

// z_p = c_m t_p / mass + c_L q_p ; Dirichlet pressure dofs: z_p = r_p
__global__ void k_schur_combine(int n, double cm, double cl, const double* __restrict__ tp, const double* __restrict__ mass,
                                const double* __restrict__ qp, const uint8_t* __restrict__ dofflag /* pressure part, n */,
                                const double* __restrict__ rp, double* __restrict__ zp) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    hemo_pdl_wait();
    hemo_pdl_trigger();
    if (i >= n) return;
    double v = cm * tp[i] / mass[i] + cl * qp[i];
    if (dofflag && dofflag[i]) v = rp[i];
    zp[i] = v;
}

static int pc_build_graph(hemo_ctx* ctx, const double* vals_dev);

// y (+)= A x for a CSR matrix with fp64 values on fp64 vectors, 4 lanes per row (coarse-space transfers)
template <bool ADD>
__global__ void __launch_bounds__(256)
k_csr_apply_d(int nrows, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const double* __restrict__ val,
              const double* __restrict__ x, double scale, double* __restrict__ y) {
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = gt >> 2, lane = gt & 3;
    const bool ok = i < nrows;
    const int r0 = ok ? rowptr[i] : 0, r1 = ok ? rowptr[i + 1] : 0;
    double a = 0.0;
    for (int t = r0 + lane; t < r1; t += 4) a = fma(val[t], x[col[t]], a);
    a += __shfl_xor_sync(0xffffffffu, a, 1, 4);
    a += __shfl_xor_sync(0xffffffffu, a, 2, 4);
    if (ok && lane == 0) y[i] = ADD ? y[i] + scale * a : scale * a;
}

// Two-level Schwarz for the pressure operator of the Schur approximation on a partitioned mesh: the rank-local
// V-cycle sees only its subdomain, so the global low modes come from a coarse space — the level-k operator of the
// global pressure hierarchy, replicated on every rank (a few 10^4 unknowns).  P0 / R0 are host CSR arrays (copied).
extern "C" int hemo_pc_set_coarse_pressure(hemo_ctx* ctx, hemo_ctx* coarse_ctx, int coarse_n, const int32_t* p_rowptr,
                                           const int32_t* p_col, const double* p_val, const int32_t* r_rowptr,
                                           const int32_t* r_col, const double* r_val, int cycles) {
    if (!ctx) return HEMO_EINVAL;
    cudaFree(ctx->cp_rowptr); cudaFree(ctx->cp_col); cudaFree(ctx->cp_val);
    cudaFree(ctx->cr_rowptr); cudaFree(ctx->cr_col); cudaFree(ctx->cr_val);
    cudaFree(ctx->coarse_rhs); cudaFree(ctx->coarse_sol);
    ctx->cp_rowptr = ctx->cp_col = ctx->cr_rowptr = ctx->cr_col = nullptr;
    ctx->cp_val = ctx->cr_val = ctx->coarse_rhs = ctx->coarse_sol = nullptr;
    ctx->coarse_ctx = nullptr;
    ctx->coarse_n = 0;
    hemo_krylov_invalidate(ctx);
    ctx->pc_graph_dirty = true;
    if (!coarse_ctx) return 0;
    if (coarse_n <= 0 || !p_rowptr || !p_col || !p_val || !r_rowptr || !r_col || !r_val) return HEMO_EINVAL;
    if (!ctx->cells) HEMO_FAIL(ctx, HEMO_ESTATE, "hemo_set_mesh must precede hemo_pc_set_coarse_pressure");
    if (coarse_ctx->n != coarse_n || !coarse_ctx->amg[1].ready)
        HEMO_FAIL(ctx, HEMO_ESTATE, "coarse context: graph / pressure hierarchy not set up");
    const int n = ctx->n;
    int rc;
    if ((rc = hemo_upload(ctx, &ctx->cp_rowptr, p_rowptr, (size_t)n + 1, false))) return rc;
    if ((rc = hemo_upload(ctx, &ctx->cp_col, p_col, (size_t)p_rowptr[n], false))) return rc;
    if ((rc = hemo_upload(ctx, &ctx->cp_val, p_val, (size_t)p_rowptr[n], false))) return rc;
    if ((rc = hemo_upload(ctx, &ctx->cr_rowptr, r_rowptr, (size_t)coarse_n + 1, false))) return rc;
    if ((rc = hemo_upload(ctx, &ctx->cr_col, r_col, (size_t)r_rowptr[coarse_n], false))) return rc;
    if ((rc = hemo_upload(ctx, &ctx->cr_val, r_val, (size_t)r_rowptr[coarse_n], false))) return rc;
    if ((rc = hemo_alloc(ctx, &ctx->coarse_rhs, (size_t)coarse_n))) return rc;
    if ((rc = hemo_alloc(ctx, &ctx->coarse_sol, (size_t)coarse_n))) return rc;
    HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->coarse_ctx = coarse_ctx;
    ctx->coarse_n = coarse_n;
    ctx->coarse_cycles = cycles > 0 ? cycles : 1;
    return 0;
}

// The additive coarse correction q += P0 Ac^-1 sum_ranks(R0 t) in two halves: the branch (restriction, allreduce,
// replicated coarse V-cycle) is enqueued on a side stream forked from the solver's stream, so it runs beside the
// rank-local V-cycle (and its allreduce latency hides behind it); the join adds the prolongated correction.
// Fork / join are event dependencies, which stream capture records as graph edges.
static int coarse_pressure_fork(hemo_ctx* ctx, const double* t_dev) {
    hemo_ctx* cc = ctx->coarse_ctx;
    const int nc = ctx->coarse_n;
    int rc = 0;
    if (!ctx->side_stream) {
        HEMO_CHECK_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->side_stream, cudaStreamNonBlocking));
        HEMO_CHECK_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
        HEMO_CHECK_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
    }
    cudaStream_t main_st = ctx->stream, side = ctx->side_stream;
    HEMO_CHECK_CUDA(ctx, cudaEventRecord(ctx->ev_fork, main_st));
    HEMO_CHECK_CUDA(ctx, cudaStreamWaitEvent(side, ctx->ev_fork, 0));
    ctx->stream = side;                       // everything below is enqueued on the side stream
    do {
        k_csr_apply_d<false><<<hemo_grid((int64_t)nc * 4, 256), 256, 0, side>>>(nc, ctx->cr_rowptr, ctx->cr_col, ctx->cr_val, t_dev,
                                                                               1.0, ctx->coarse_rhs);
        ctx->launches++;
        if (cudaGetLastError() != cudaSuccess) { rc = HEMO_ESTATE; ctx->err = "coarse restriction launch failed"; break; }
        if ((rc = hemo_comm_allreduce_j(ctx, ctx->coarse_rhs, nc))) break;
        cudaStream_t saved = cc->stream;
        const bool saved_cap = cc->capturing;
        const int saved_pdl = cc->pdl;
        const int64_t before = cc->launches;
        cc->stream = side;
        cc->capturing = ctx->capturing;
        cc->pdl = ctx->pdl;
        cc->opts.cheb_degree = ctx->opts.cheb_degree;
        cc->opts.cheb_degree_pre = ctx->opts.cheb_degree_pre;
        cc->opts.cheb_ratio = ctx->opts.cheb_ratio;
        rc = hemo_amg_vcycle(cc, &cc->amg[1], ctx->coarse_rhs, ctx->coarse_sol, ctx->coarse_cycles);
        ctx->launches += cc->launches - before;
        cc->stream = saved;
        cc->capturing = saved_cap;
        cc->pdl = saved_pdl;
        if (rc) ctx->err = cc->err;
    } while (0);
    ctx->stream = main_st;
    if (rc) return rc;
    HEMO_CHECK_CUDA(ctx, cudaEventRecord(ctx->ev_join, side));
    return 0;
}

static int coarse_pressure_join(hemo_ctx* ctx, double* q_dev) {
    const int n = ctx->n;
    cudaStream_t st = ctx->stream;
    HEMO_CHECK_CUDA(ctx, cudaStreamWaitEvent(st, ctx->ev_join, 0));
    k_csr_apply_d<true><<<hemo_grid((int64_t)n * 4, 256), 256, 0, st>>>(n, ctx->cp_rowptr, ctx->cp_col, ctx->cp_val, ctx->coarse_sol,
                                                                       1.0, q_dev);
    HEMO_LAUNCH_CHECK(ctx);
    return 0;
}

// Dirichlet flags of the pressure dofs: the tail of dofflag in the [u (dim n) | p (n)] layout
static inline const uint8_t* pressure_flags(const hemo_ctx* ctx) {
    return ctx->have_bc ? ctx->dofflag + (size_t)ctx->dim * ctx->n : nullptr;
}

extern "C" int hemo_remove_mean_vec(hemo_ctx* ctx, int64_t n, double* x_dev) {
    if (!ctx || !x_dev || n <= 0) return HEMO_EINVAL;
    return hemo_remove_mean(ctx, n, x_dev);
}

extern "C" int hemo_set_external_schur(hemo_ctx* ctx, int on) {
    if (!ctx) return HEMO_EINVAL;
    ctx->external_schur = on != 0;
    return 0;
}

// Numeric setup of the scalar (pressure Laplacian) hierarchy alone: used by a context that
// only serves the replicated global pressure solve of the multi-GPU driver.
extern "C" int hemo_amg_setup_scalar(hemo_ctx* ctx, const double* lap_vals_dev, double coarse_shift) {
    if (!ctx || !lap_vals_dev) return HEMO_EINVAL;
    if (!ctx->amg[1].ready) HEMO_FAIL(ctx, HEMO_ESTATE, "pressure AMG hierarchy not finalized");
    k_lap_with_bc<<<hemo_grid(ctx->nnz_node, 256), 256, 0, ctx->stream>>>(ctx->n, ctx->nnz_node, ctx->rowof, ctx->ncol,
                                                                          lap_vals_dev, pressure_flags(ctx),
                                                                          ctx->amg[1].op[0].val);
    HEMO_LAUNCH_CHECK(ctx);
    return hemo_amg_numeric_shift(ctx, &ctx->amg[1], coarse_shift);
}

extern "C" int hemo_set_pc_mask(hemo_ctx* ctx, const uint8_t* node_mask_dev) {
    if (!ctx) return HEMO_EINVAL;
    if (!ctx->cells) HEMO_FAIL(ctx, HEMO_ESTATE, "hemo_set_mesh must precede hemo_set_pc_mask");
    if (!node_mask_dev) {
        cudaFree(ctx->pc_mask);
        ctx->pc_mask = nullptr;
        return 0;
    }
    return hemo_upload(ctx, &ctx->pc_mask, node_mask_dev, (size_t)ctx->n, true);
}

extern "C" int hemo_mask_nodes(hemo_ctx* ctx, const uint8_t* node_mask_dev, double* x_dev) {
    if (!ctx || !node_mask_dev || !x_dev) return HEMO_EINVAL;
    const int n = ctx->n;
    k_mask_nodes<<<hemo_grid(n, 256), 256, 0, ctx->stream>>>(n, 2, node_mask_dev, x_dev);
    HEMO_LAUNCH_CHECK(ctx);
    k_mask_nodes<<<hemo_grid(n, 256), 256, 0, ctx->stream>>>(n, 1, node_mask_dev, x_dev + 2 * (int64_t)n);
    HEMO_LAUNCH_CHECK(ctx);
    return 0;
}

extern "C" int hemo_vec_mdot(hemo_ctx* ctx, int64_t n, int k, const double* V_dev, int64_t ldv, const double* w_dev,
                             double* h_host) {
    if (!ctx || !V_dev || !w_dev || !h_host || k < 1 || k > 400 || n < 1) return HEMO_EINVAL;
    return hemo_mdot(ctx, n, k, V_dev, ldv, w_dev, h_host);
}

extern "C" int hemo_vec_maxpy(hemo_ctx* ctx, int64_t n, int k, const double* V_dev, int64_t ldv,
                              const double* coef_host, double sign, double* w_dev, double* normsq_host) {
    if (!ctx || !V_dev || !w_dev || !coef_host || k < 1 || k > 400 || n < 1) return HEMO_EINVAL;
    int rc = hemo_ensure_reduce(ctx, (size_t)1184 * 2, 512);
    if (rc) return rc;
    if (!ctx->kry_coef && (rc = hemo_alloc(ctx, &ctx->kry_coef, 512))) return rc;
    for (int i = 0; i < k; ++i) ctx->red_host[i] = coef_host[i];
    HEMO_CHECK_CUDA(ctx, cudaMemcpyAsync(ctx->kry_coef, ctx->red_host, sizeof(double) * k, cudaMemcpyHostToDevice,
                                         ctx->stream));
    double nrm = 0.0;
    rc = hemo_maxpy(ctx, n, k, V_dev, ldv, ctx->kry_coef, sign, w_dev, normsq_host ? &nrm : nullptr);
    if (rc) return rc;
    if (normsq_host) *normsq_host = nrm * nrm;      // local ||w||^2, to be summed over ranks
    else HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // red_host is reused by the next call
    return 0;
}

extern "C" int hemo_vec_scale(hemo_ctx* ctx, int64_t n, double a, const double* x_dev, double* y_dev) {
    if (!ctx || !x_dev || !y_dev || n < 1) return HEMO_EINVAL;
    return hemo_scale_copy(ctx, n, a, x_dev, y_dev);
}

extern "C" int hemo_use_graph(hemo_ctx* ctx, int on) {
    if (!ctx) return HEMO_EINVAL;
    ctx->use_graph = on != 0;
    return 0;
}

extern "C" int hemo_set_solver_opts(hemo_ctx* ctx, const hemo_solver_opts* o) {
    if (!ctx || !o) return HEMO_EINVAL;
    if (o->restart < 1 || o->restart > 400 || o->max_it < 1) return HEMO_EINVAL;
    // fields the captured graphs (FGMRES iteration, preconditioner, hemo_amg_apply) bake in as launch arguments or
    // launch sequence: a change re-captures them at their next use
    const hemo_solver_opts& p = ctx->opts;
    const bool baked = p.amg_cycles_u != o->amg_cycles_u || p.amg_cycles_p != o->amg_cycles_p ||
                       p.cheb_degree != o->cheb_degree || p.cheb_degree_pre != o->cheb_degree_pre ||
                       p.cheb_ratio != o->cheb_ratio || p.project_pressure != o->project_pressure ||
                       p.pc_mode != o->pc_mode || p.schur_mass_coef != o->schur_mass_coef ||
                       p.schur_lap_coef != o->schur_lap_coef;
    ctx->opts = *o;
    if (baked) {
        hemo_krylov_invalidate(ctx);
        ctx->pc_graph_dirty = true;
        ctx->amg[0].apply_valid = ctx->amg[1].apply_valid = false;
    }
    return 0;
}

extern "C" int hemo_pc_setup(hemo_ctx* ctx, const double* vals_dev, const double* lap_vals_dev,
                             const double* mass_dev) {
    if (!ctx || !vals_dev) return HEMO_EINVAL;
    const bool tet = ctx->dim == 3;    // 3-D: block-Jacobi sweeps on A00 instead of the velocity hierarchy (DESIGN.md §5b)
    if ((!tet && !ctx->amg[0].ready) || !ctx->amg[1].ready) HEMO_FAIL(ctx, HEMO_ESTATE, "AMG hierarchies not finalized");
    if (tet && (ctx->pc_mask || ctx->external_schur))
        HEMO_FAIL(ctx, HEMO_ESTATE, "partition masks / external Schur solves are not implemented for tetrahedra yet");
    const int n = ctx->n;
    const size_t gd = (size_t)ctx->dim;
    cudaStream_t st = ctx->stream;
    int rc;
    if (!ctx->pc_tmp_u) {
        if ((rc = hemo_alloc(ctx, &ctx->pc_tmp_u, gd * n))) return rc;
        if ((rc = hemo_alloc(ctx, &ctx->pc_tmp_u2, gd * n))) return rc;
        if ((rc = hemo_alloc(ctx, &ctx->pc_tmp_p, (size_t)n))) return rc;
        if ((rc = hemo_alloc(ctx, &ctx->pc_tmp_p2, (size_t)n))) return rc;
        if (!tet && (rc = hemo_alloc(ctx, &ctx->a01, (size_t)ctx->nnz_node))) return rc;
        if ((rc = hemo_alloc(ctx, &ctx->pc_in, (gd + 1) * n + 32))) return rc;
        if ((rc = hemo_alloc(ctx, &ctx->pc_out, (gd + 1) * n + 32))) return rc;
    }
    if (tet) {
        if ((rc = hemo_tet_pc_setup(ctx, vals_dev))) return rc;
    } else {
        k_extract_a00<<<hemo_grid(ctx->nnz_node, 256), 256, 0, st>>>(ctx->nnz_node, ctx->nrowptr, ctx->rowof, ctx->ncol,
                                                                     ctx->pc_mask, vals_dev, ctx->amg[0].op[0].val, ctx->a01);
        HEMO_LAUNCH_CHECK(ctx);
        if ((rc = hemo_amg_numeric_shift(ctx, &ctx->amg[0], 0.0))) return rc;
    }
    if (mass_dev) ctx->mass = mass_dev;
    if (lap_vals_dev) {
        if (!ctx->mass) return HEMO_EINVAL;
        k_lap_with_bc<<<hemo_grid(ctx->nnz_node, 256), 256, 0, st>>>(n, ctx->nnz_node, ctx->rowof, ctx->ncol, lap_vals_dev,
                                                                     pressure_flags(ctx), ctx->amg[1].op[0].val);
        HEMO_LAUNCH_CHECK(ctx);
        if ((rc = hemo_amg_numeric_shift(ctx, &ctx->amg[1], ctx->opts.project_pressure ? 1e-8 : 0.0))) return rc;
    }
    if (!ctx->mass) HEMO_FAIL(ctx, HEMO_ESTATE, "first hemo_pc_setup call needs lap_vals and mass");
    hemo_krylov_invalidate(ctx);     // smoother coefficients are baked into the captured iteration
    ctx->pc_graph_dirty = true;      // ... and into the stand-alone preconditioner graph (re-captured on demand)
    return 0;
}

extern "C" int hemo_amg_apply(hemo_ctx* ctx, int which, const double* b_dev, double* x_dev, int ncycles) {
    if (!ctx || which < 0 || which > 1 || !b_dev || !x_dev) return HEMO_EINVAL;
    HemoAmg& amg = ctx->amg[which];
    if (!ctx->use_graph || ctx->stream == 0 || ctx->capturing)
        return hemo_amg_vcycle(ctx, &amg, b_dev, x_dev, ncycles);
    // repeated applications with the same buffers (the replicated global pressure solve of the
    // multi-GPU driver) replay a captured graph
    if (amg.apply_valid && amg.apply_exec && amg.apply_b == b_dev && amg.apply_x == x_dev && amg.apply_cycles == ncycles) {
        HEMO_CHECK_CUDA(ctx, cudaGraphLaunch(amg.apply_exec, ctx->stream));
        ctx->launches += amg.apply_nodes;
        return 0;
    }
    cudaStream_t st = ctx->stream;
    HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(st));
    const int64_t before = ctx->launches;
    ctx->capturing = true;
    if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
        ctx->capturing = false;
        cudaGetLastError();
        return hemo_amg_vcycle(ctx, &amg, b_dev, x_dev, ncycles);
    }
    int rc = hemo_amg_vcycle(ctx, &amg, b_dev, x_dev, ncycles);
    cudaGraph_t g = nullptr;
    cudaError_t e = cudaStreamEndCapture(st, &g);
    ctx->capturing = false;
    amg.apply_nodes = ctx->launches - before;
    ctx->launches = before;
    if (rc != 0 || e != cudaSuccess || !g) {
        cudaGetLastError();
        if (g) cudaGraphDestroy(g);
        if (rc) return rc;
        return hemo_amg_vcycle(ctx, &amg, b_dev, x_dev, ncycles);
    }
    if (amg.apply_exec) { cudaGraphExecDestroy(amg.apply_exec); amg.apply_exec = nullptr; }
    HEMO_CHECK_CUDA(ctx, cudaGraphInstantiate(&amg.apply_exec, g, 0));
    cudaGraphDestroy(g);
    amg.apply_b = b_dev; amg.apply_x = x_dev; amg.apply_cycles = ncycles; amg.apply_valid = true;
    HEMO_CHECK_CUDA(ctx, cudaGraphLaunch(amg.apply_exec, st));
    ctx->launches += amg.apply_nodes;
    return 0;
}

extern "C" int hemo_amg_get_level_values(hemo_ctx* ctx, int which, int level, double* vals_dev, int64_t capacity) {
    if (!ctx || which < 0 || which > 1 || !vals_dev) return HEMO_EINVAL;
    HemoAmg& amg = ctx->amg[which];
    if (!amg.ready || level < 0 || level >= amg.nlev) return HEMO_EINVAL;
    const int64_t cnt = amg.op[level].nnzb * amg.bs * amg.bs;
    if (capacity < cnt) return HEMO_EINVAL;
    k_areal_to_double<<<hemo_grid(cnt, 256), 256, 0, ctx->stream>>>(cnt, amg.op[level].val, vals_dev);
    HEMO_LAUNCH_CHECK(ctx);
    return 0;
}

extern "C" int hemo_amg_level_info(hemo_ctx* ctx, int which, int level, int64_t* out) {
    if (!ctx || which < 0 || which > 1 || !out) return HEMO_EINVAL;
    const HemoAmg& amg = ctx->amg[which];
    if (!amg.ready || level < 0 || level >= amg.nlev) return HEMO_EINVAL;
    const HemoAmgOp& o = amg.op[level];
    out[0] = o.n;
    out[1] = o.nnzb;
    out[2] = o.sell_ptr ? o.sell_entries : 0;
    out[3] = level >= amg.fuse_level ? HEMO_AMG_SCOPE_CTA : HEMO_AMG_SCOPE_LEVEL;
    return 0;
}

int hemo_pc_apply_body(hemo_ctx* ctx, const double* vals_dev, const double* r_dev, double* z_dev) {
    const int n = ctx->n;
    cudaStream_t st = ctx->stream;
    const double* ru = r_dev;
    const double* rp = r_dev + ctx->dim * (int64_t)n;
    double* zu = z_dev;
    double* zp = z_dev + ctx->dim * (int64_t)n;
    double* tp = ctx->pc_tmp_p;
    double* qp = ctx->pc_tmp_p2;
    double* tu = ctx->pc_tmp_u;
    int rc;
    if (!ctx->external_schur) {
    if (ctx->opts.project_pressure && !ctx->pc_mask) {
        if ((rc = hemo_copy_remove_mean(ctx, n, rp, tp))) return rc;      // the copy rides on the summation pass
    } else {
        HEMO_CHECK_CUDA(ctx, cudaMemcpyAsync(tp, rp, sizeof(double) * n, cudaMemcpyDeviceToDevice, st));
        if (ctx->pc_mask) HEMO_LAUNCH(ctx, k_mask_nodes, hemo_grid(n, 256), 256, 0, st, n, 1, ctx->pc_mask, tp);
        if (ctx->opts.project_pressure && (rc = hemo_remove_mean(ctx, n, tp))) return rc;
    }
    if (ctx->coarse_ctx && (rc = coarse_pressure_fork(ctx, tp))) return rc;
    if ((rc = hemo_amg_vcycle(ctx, &ctx->amg[1], tp, qp, ctx->opts.amg_cycles_p))) return rc;
    if (ctx->coarse_ctx) {
        HEMO_PROF_BEGIN(ctx, HEMO_PROF_COARSE);          // what is left on the critical path: the join
        if ((rc = coarse_pressure_join(ctx, qp))) return rc;
        HEMO_PROF_END(ctx, HEMO_PROF_COARSE);
    }
    HEMO_LAUNCH(ctx, k_schur_combine, hemo_grid(n, 256), 256, 0, st, n, ctx->opts.schur_mass_coef, ctx->opts.schur_lap_coef, tp,
                ctx->mass, qp, pressure_flags(ctx), rp, zp);
    if (ctx->opts.project_pressure && (rc = hemo_remove_mean(ctx, n, zp))) return rc;
    }   // else: z_p was provided by the caller (global pressure solve of the multi-GPU driver)
    if (ctx->dim == 3)    // t_u = r_u - A01 z_p, then damped block-Jacobi sweeps on A00 (amg_cycles_u * 4 sweeps)
        return hemo_tet_velocity_solve(ctx, vals_dev, ru, zp, tu, ctx->pc_tmp_u2, zu, 4 * ctx->opts.amg_cycles_u, 2.0 / 3.0);
    // t_u = r_u - A01 z_p
    if (n >= 32768 && ctx->nnz_node <= 12 * (int64_t)n)
        HEMO_LAUNCH(ctx, k_a01_residual_row, hemo_grid(n, 256), 256, 0, st, n, ctx->nrowptr, ctx->ncol, ctx->a01, zp, ru, tu);
    else
        HEMO_LAUNCH(ctx, k_a01_residual, hemo_grid((int64_t)n * 4, 256), 256, 0, st, n, ctx->nrowptr, ctx->ncol, ctx->a01, zp, ru,
                    tu);
    if (ctx->pc_mask) HEMO_LAUNCH(ctx, k_mask_nodes, hemo_grid(n, 256), 256, 0, st, n, 2, ctx->pc_mask, tu);
    if ((rc = hemo_amg_vcycle(ctx, &ctx->amg[0], tu, zu, ctx->opts.amg_cycles_u))) return rc;
    return 0;
}

// (Re)capture the preconditioner application as a CUDA graph on ctx->stream:
// ~100 small kernels per application replay with one launch.  Needs a
// non-default stream; on the legacy default stream the direct path is used.
static int pc_build_graph(hemo_ctx* ctx, const double* vals_dev) {
    if (!ctx->use_graph || ctx->stream == 0) return 0;
    cudaStream_t st = ctx->stream;
    int rc = hemo_ensure_reduce(ctx, (size_t)1184 * 8, 512);   // no allocation may happen while capturing
    if (rc) return rc;
    HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(st));
    const int64_t before = ctx->launches;
    ctx->capturing = true;
    cudaError_t e = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal);
    if (e != cudaSuccess) {
        ctx->capturing = false;
        cudaGetLastError();
        ctx->use_graph = 0;            // capture unsupported here: fall back to direct launches
        return 0;
    }
    rc = hemo_pc_apply_body(ctx, vals_dev, ctx->pc_in, ctx->pc_out);
    cudaGraph_t g = nullptr;
    e = cudaStreamEndCapture(st, &g);
    ctx->capturing = false;
    ctx->pc_graph_nodes = ctx->launches - before;
    ctx->launches = before;
    if (rc != 0 || e != cudaSuccess || !g) {
        cudaGetLastError();
        if (g) cudaGraphDestroy(g);
        ctx->use_graph = 0;
        if (rc) return rc;
        return 0;
    }
    bool updated = false;
    if (ctx->pc_graph_exec) {
        cudaGraphExecUpdateResultInfo info;
        if (cudaGraphExecUpdate(ctx->pc_graph_exec, g, &info) == cudaSuccess) updated = true;
        else { cudaGetLastError(); cudaGraphExecDestroy(ctx->pc_graph_exec); ctx->pc_graph_exec = nullptr; }
    }
    if (!updated) HEMO_CHECK_CUDA(ctx, cudaGraphInstantiate(&ctx->pc_graph_exec, g, 0));
    if (ctx->pc_graph) cudaGraphDestroy(ctx->pc_graph);
    ctx->pc_graph = g;
    return 0;
}

extern "C" int hemo_pc_apply(hemo_ctx* ctx, const double* vals_dev, const double* r_dev, double* z_dev) {
    if (!ctx || !vals_dev || !r_dev || !z_dev) return HEMO_EINVAL;
    if (!ctx->mass || !ctx->pc_tmp_u) HEMO_FAIL(ctx, HEMO_ESTATE, "hemo_pc_setup not called");
    if (ctx->use_graph && ctx->stream != 0 && ctx->pc_graph_dirty) {
        int rc = pc_build_graph(ctx, vals_dev);
        if (rc) return rc;
        ctx->pc_graph_dirty = false;
    }
    if (ctx->use_graph && ctx->pc_graph_exec && ctx->stream != 0) {
        const size_t bytes = sizeof(double) * (size_t)(ctx->dim + 1) * (size_t)ctx->n;
        cudaStream_t st = ctx->stream;
        HEMO_CHECK_CUDA(ctx, cudaMemcpyAsync(ctx->pc_in, r_dev, bytes, cudaMemcpyDeviceToDevice, st));
        if (ctx->external_schur)
            HEMO_CHECK_CUDA(ctx, cudaMemcpyAsync(ctx->pc_out + (size_t)ctx->dim * ctx->n, z_dev + (size_t)ctx->dim * ctx->n,
                                                 sizeof(double) * ctx->n, cudaMemcpyDeviceToDevice, st));
        HEMO_CHECK_CUDA(ctx, cudaGraphLaunch(ctx->pc_graph_exec, st));
        HEMO_CHECK_CUDA(ctx, cudaMemcpyAsync(z_dev, ctx->pc_out, bytes, cudaMemcpyDeviceToDevice, st));
        ctx->launches += ctx->pc_graph_nodes;
        return 0;
    }
    return hemo_pc_apply_body(ctx, vals_dev, r_dev, z_dev);
}

// ---------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------
extern "C" int hemo_ctx_create(int device, hemo_ctx** out) {
    if (!out) return HEMO_EINVAL;
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return (int)e;
    hemo_ctx* ctx = new hemo_ctx();
    ctx->device = device;
    ctx->opts.restart = 60;
    ctx->opts.max_it = 1000;
    ctx->opts.rtol = 1e-5;
    ctx->opts.atol = 1e-50;
    ctx->opts.amg_cycles_u = 1;
    ctx->opts.amg_cycles_p = 1;
    ctx->opts.cheb_degree = 2;
    ctx->opts.project_pressure = 0;
    ctx->opts.pc_mode = 0;
    ctx->opts.schur_mass_coef = 0.0;
    ctx->opts.schur_lap_coef = 1.0;
    ctx->opts.cheb_ratio = 4.0;
    ctx->opts.cheb_degree_pre = 0;
    const char* pdl = getenv("HEMO_PDL");
    ctx->pdl = pdl && atoi(pdl) == 0 ? 0 : 1;
    *out = ctx;
    return 0;
}

extern "C" int hemo_ctx_destroy(hemo_ctx* ctx) {
    if (!ctx) return HEMO_EINVAL;
    cudaSetDevice(ctx->device);
    cudaFree(ctx->cellpos); cudaFree(ctx->mseg_ptr); cudaFree(ctx->mseg_src); cudaFree(ctx->vseg_ptr);
    cudaFree(ctx->vseg_src); cudaFree(ctx->diagslot); cudaFree(ctx->rowof); cudaFree(ctx->Ae); cudaFree(ctx->Fe);
    cudaFree(ctx->dvec); cudaFree(ctx->dofflag); cudaFree(ctx->dofmult); cudaFree(ctx->cellflag);
    for (int s = 0; s < HEMO_MAX_FACET_SETS; ++s) { cudaFree(ctx->fsets[s].cells); cudaFree(ctx->fsets[s].mask); }
    cudaFree(ctx->red_partial); cudaFree(ctx->red_out);
    if (ctx->red_host) cudaFreeHost(ctx->red_host);
    hemo_amg_free(&ctx->amg[0]); hemo_amg_free(&ctx->amg[1]);
    if (ctx->pc_graph_exec) cudaGraphExecDestroy(ctx->pc_graph_exec);
    if (ctx->pc_graph) cudaGraphDestroy(ctx->pc_graph);
    cudaFree(ctx->wss_cell2t); cudaFree(ctx->wss_tmp);
    free(ctx->qrules);
    free(ctx->p2rules);
    hemo_tet_free(ctx);
    hemo_cc_free(ctx);
    cudaFree(ctx->pc_in); cudaFree(ctx->pc_out); cudaFree(ctx->pc_mask); cudaFree(ctx->kry_coef); cudaFree(ctx->a01);
    cudaFree(ctx->pc_tmp_u); cudaFree(ctx->pc_tmp_u2); cudaFree(ctx->pc_tmp_p); cudaFree(ctx->pc_tmp_p2);
    cudaFree(ctx->kry_V); cudaFree(ctx->kry_Z); cudaFree(ctx->kry_w);
    cudaFree(ctx->cp_rowptr); cudaFree(ctx->cp_col); cudaFree(ctx->cp_val);
    cudaFree(ctx->cr_rowptr); cudaFree(ctx->cr_col); cudaFree(ctx->cr_val);
    cudaFree(ctx->coarse_rhs); cudaFree(ctx->coarse_sol);
    if (ctx->side_stream) cudaStreamDestroy(ctx->side_stream);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    hemo_krylov_free(ctx);
    hemo_comm_free(ctx);
    delete ctx;
    return 0;
}

extern "C" const char* hemo_last_error(hemo_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

extern "C" int hemo_set_stream(hemo_ctx* ctx, void* cuda_stream) {
    if (!ctx) return HEMO_EINVAL;
    ctx->stream = (cudaStream_t)cuda_stream;
    return 0;
}

extern "C" int hemo_prof_enable(hemo_ctx* ctx, int on) {
    if (!ctx) return HEMO_EINVAL;
    ctx->prof.on = on != 0;
    for (int c = 0; c < HEMO_PROF_NCLASS; ++c) ctx->prof.used[c] = 0;
    return 0;
}

extern "C" int hemo_prof_get(hemo_ctx* ctx, int cls, double* ms_total, int64_t* launches) {
    if (!ctx || cls < 0 || cls >= HEMO_PROF_NCLASS || !ms_total || !launches) return HEMO_EINVAL;
    HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    HemoProf& p = ctx->prof;
    double tot = 0.0;
    const size_t pairs = p.used[cls] / 2;
    for (size_t i = 0; i < pairs; ++i) {
        float ms = 0.f;
        HEMO_CHECK_CUDA(ctx, cudaEventElapsedTime(&ms, p.ev[cls][2 * i], p.ev[cls][2 * i + 1]));
        tot += ms;
    }
    *ms_total = tot;
    *launches = (int64_t)pairs;
    return 0;
}

extern "C" int64_t hemo_launch_count(hemo_ctx* ctx) { return ctx ? ctx->launches : 0; }
