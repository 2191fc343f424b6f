// Sparse matrix-vector products and Krylov vector kernels (fp64, HBM-bound).
//
// Replaces PETSc MatMult / VecMDot / VecMAXPY / VecNorm used inside
// KSPSolve(fgmres) configured at reference src/solvers/stabilized_schur.py:226-229.
//
// The monolithic Jacobian keeps the reference CSR layout (rows [u|p], columns
// ascending), but all three rows of a mesh node share one column structure,
// so the SpMV walks the *node graph*: 4 bytes of index per 72 bytes of values.
// All reductions are two-stage with a fixed grid and a fixed summation order
// (bitwise reproducible, no atomics).
#include "hemo_internal.cuh"

#define RED_BLOCKS 1184   // 148 SMs * 8
#define RED_THREADS 256

// Captured CUDA graphs (preconditioner application, V-cycle) hold the raw addresses of these
// buffers in their kernel nodes.  The scratch is therefore allocated once at the size of the largest
// request any entry point makes (restart <= 400: RED_BLOCKS * (400 + 4) partial sums, 1024 results);
// should a larger request ever arrive, every captured graph is dropped before the buffers move.
static void drop_graphs(hemo_ctx* ctx) {
    hemo_krylov_invalidate(ctx);
    if (ctx->pc_graph_exec) { cudaGraphExecDestroy(ctx->pc_graph_exec); ctx->pc_graph_exec = nullptr; }
    if (ctx->pc_graph) { cudaGraphDestroy(ctx->pc_graph); ctx->pc_graph = nullptr; }
    ctx->pc_graph_dirty = true;
    for (int w = 0; w < 2; ++w) {
        HemoAmg& a = ctx->amg[w];
        if (a.apply_exec) { cudaGraphExecDestroy(a.apply_exec); a.apply_exec = nullptr; }
        a.apply_valid = false;
    }
}

int hemo_ensure_reduce(hemo_ctx* ctx, size_t partial_n, size_t out_n) {
    const size_t min_partial = (size_t)RED_BLOCKS * 404, min_out = 1024;
    if (partial_n < min_partial) partial_n = min_partial;
    if (out_n < min_out) out_n = min_out;
    if (partial_n > ctx->red_partial_n) {
        if (ctx->red_partial) {
            HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            drop_graphs(ctx);
        }
        int rc = hemo_alloc(ctx, &ctx->red_partial, partial_n);
        if (rc) return rc;
        ctx->red_partial_n = partial_n;
    }
    if (out_n > ctx->red_out_n) {
        if (ctx->red_out) {
            HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            drop_graphs(ctx);
        }
        int rc = hemo_alloc(ctx, &ctx->red_out, out_n);
        if (rc) return rc;
        if (ctx->red_host) cudaFreeHost(ctx->red_host);
        HEMO_CHECK_CUDA(ctx, cudaMallocHost((void**)&ctx->red_host, out_n * sizeof(double)));
        ctx->red_out_n = out_n;
    }
    return 0;
}

void hemo_drop_solver_state(hemo_ctx* ctx) {
    cudaStreamSynchronize(ctx->stream);
    drop_graphs(ctx);
    cudaFree(ctx->pc_tmp_u); cudaFree(ctx->pc_tmp_u2); cudaFree(ctx->pc_tmp_p); cudaFree(ctx->pc_tmp_p2);
    cudaFree(ctx->pc_in); cudaFree(ctx->pc_out); cudaFree(ctx->a01);
    ctx->pc_tmp_u = ctx->pc_tmp_u2 = ctx->pc_tmp_p = ctx->pc_tmp_p2 = ctx->pc_in = ctx->pc_out = nullptr;
    ctx->a01 = nullptr;
    cudaFree(ctx->kry_V); cudaFree(ctx->kry_Z); cudaFree(ctx->kry_w);
    ctx->kry_V = ctx->kry_Z = ctx->kry_w = nullptr;
    ctx->kry_restart = 0;
    hemo_krylov_invalidate(ctx);
    ctx->kry.m = 0; ctx->kry.last_its = 0;
    cudaFree(ctx->pc_mask);
    ctx->pc_mask = nullptr;
    ctx->mass = nullptr;
    ctx->amg[0].ready = ctx->amg[1].ready = false;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ double block_sum(double v, double* sh) {
    // blockDim.x == RED_THREADS (8 warps); result valid in thread 0
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) sh[wid] = v;
    __syncthreads();
    double r = 0.0;
    if (wid == 0) {
        r = (lane < (blockDim.x >> 5)) ? sh[lane] : 0.0;
        r = warp_sum(r);
    }
    __syncthreads();
    return r;
}

// ---------------------------------------------------------------------------
// node-structured SpMV on the monolithic matrix:  y = b + alpha * A[rows, cols] x
// 8 lanes per node row-group.
// ---------------------------------------------------------------------------
template <bool RU, bool RP, bool CU, bool CP>
__global__ void __launch_bounds__(256)
k_spmv_node(int n, int64_t nnz_node, const int32_t* __restrict__ nrowptr, const int32_t* __restrict__ ncol,
            const double* __restrict__ vals, const double* __restrict__ xu, const double* __restrict__ xp,
            double alpha, const double* __restrict__ bu, const double* __restrict__ bp,
            double* __restrict__ yu, double* __restrict__ yp) {
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = gt >> 3;
    const int lane = gt & 7;
    const bool ok = i < n;   // no early return: full-mask shuffles below
    const int r0 = ok ? nrowptr[i] : 0;
    const int deg = ok ? nrowptr[i + 1] - r0 : 0;
    const int64_t ru0 = 6 * (int64_t)r0, ru1 = ru0 + 3 * deg, rp = 6 * nnz_node + 3 * (int64_t)r0;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0;
    for (int t = lane; t < deg; t += 8) {
        const int j = ncol[r0 + t];
        double x0 = 0.0, x1 = 0.0, x2 = 0.0;
        if (CU) {
            const double2 xv = reinterpret_cast<const double2*>(xu)[j];
            x0 = xv.x; x1 = xv.y;
        }
        if (CP) x2 = xp[j];
        if (RU) {
            if (CU) {
                a0 += vals[ru0 + 2 * t] * x0 + vals[ru0 + 2 * t + 1] * x1;
                a1 += vals[ru1 + 2 * t] * x0 + vals[ru1 + 2 * t + 1] * x1;
            }
            if (CP) {
                a0 += vals[ru0 + 2 * deg + t] * x2;
                a1 += vals[ru1 + 2 * deg + t] * x2;
            }
        }
        if (RP) {
            if (CU) a2 += vals[rp + 2 * t] * x0 + vals[rp + 2 * t + 1] * x1;
            if (CP) a2 += vals[rp + 2 * deg + t] * x2;
        }
    }
    // reduce over the 8 lanes of the group
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) {
        a0 += __shfl_down_sync(0xffffffffu, a0, o, 8);
        a1 += __shfl_down_sync(0xffffffffu, a1, o, 8);
        a2 += __shfl_down_sync(0xffffffffu, a2, o, 8);
    }
    if (ok && lane == 0) {
        if (RU) {
            double r0v = alpha * a0, r1v = alpha * a1;
            if (bu) { r0v += bu[2 * (int64_t)i]; r1v += bu[2 * (int64_t)i + 1]; }
            yu[2 * (int64_t)i] = r0v;
            yu[2 * (int64_t)i + 1] = r1v;
        }
        if (RP) {
            double r2v = alpha * a2;
            if (bp) r2v += bp[i];
            yp[i] = r2v;
        }
    }
}

// sub-block dispatch used by the preconditioner (rows/cols: 1 = u, 2 = p, 3 = both)
int hemo_spmv_block(hemo_ctx* ctx, int rows, int cols, const double* vals, const double* xu, const double* xp,
                    double alpha, const double* bu, const double* bp, double* yu, double* yp) {
    const int n = ctx->n;
    const int grid = hemo_grid((int64_t)n * 8, 256);
    cudaStream_t st = ctx->stream;
#define LAUNCH(RU, RP, CU, CP)                                                                        \
    k_spmv_node<RU, RP, CU, CP><<<grid, 256, 0, st>>>(n, ctx->nnz_node, ctx->nrowptr, ctx->ncol, vals, \
                                                      xu, xp, alpha, bu, bp, yu, yp)
    if (rows == 3 && cols == 3) LAUNCH(true, true, true, true);
    else if (rows == 1 && cols == 1) LAUNCH(true, false, true, false);
    else if (rows == 1 && cols == 2) LAUNCH(true, false, false, true);
    else if (rows == 2 && cols == 1) LAUNCH(false, true, true, false);
    else if (rows == 2 && cols == 2) LAUNCH(false, true, false, true);
    else HEMO_FAIL(ctx, HEMO_EINVAL, "unsupported sub-block");
#undef LAUNCH
    HEMO_LAUNCH_CHECK(ctx);
    return 0;
}

extern "C" int hemo_spmv(hemo_ctx* ctx, const double* vals_dev, const double* x_dev, double* y_dev) {
    if (!ctx || !vals_dev || !x_dev || !y_dev) return HEMO_EINVAL;
    if (!ctx->nrowptr) HEMO_FAIL(ctx, HEMO_ESTATE, "node graph not set");
    if (ctx->dim == 3) return hemo_tet_spmv(ctx, vals_dev, x_dev, y_dev);
    const int64_t n = ctx->n;
    return hemo_spmv_block(ctx, 3, 3, vals_dev, x_dev, x_dev + 2 * n, 1.0, nullptr, nullptr, y_dev, y_dev + 2 * n);
}

// ---------------------------------------------------------------------------
// BSR SpMV for multigrid operators: y = b + alpha * A x (bs = 1 or 2), hierarchy storage
// type `areal`, fp64 accumulation
// ---------------------------------------------------------------------------
template <int BS>
__global__ void __launch_bounds__(256)
k_bsr_spmv(int n, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
           const areal* __restrict__ val, const areal* __restrict__ x, double alpha,
           const areal* __restrict__ b, areal* __restrict__ y) {
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = gt >> 2;        // 4 lanes per block row
    const int lane = gt & 3;
    const bool ok = i < n;
    const int r0 = ok ? rowptr[i] : 0, r1 = ok ? rowptr[i + 1] : 0;
    hemo_pdl_wait();
    hemo_pdl_trigger();
    double a0 = 0.0, a1 = 0.0;
    // column loads of three strided entries first (the col -> x chain bounds short rows)
    for (int t = r0 + lane; t < r1; t += 12) {
        const int t1 = t + 4, t2 = t + 8;
        const bool p1 = t1 < r1, p2 = t2 < r1;
        const int j0 = col[t];
        const int j1 = p1 ? col[t1] : j0;
        const int j2 = p2 ? col[t2] : j0;
        if (BS == 1) {
            const double v0 = (double)val[t], x0 = (double)x[j0];
            const double v1 = p1 ? (double)val[t1] : 0.0, x1 = (double)x[j1];
            const double v2 = p2 ? (double)val[t2] : 0.0, x2 = (double)x[j2];
            a0 = fma(v0, x0, a0);
            a0 = fma(v1, x1, a0);
            a0 = fma(v2, x2, a0);
        } else {
            const areal2* v2p = reinterpret_cast<const areal2*>(val);
            const areal2* x2p = reinterpret_cast<const areal2*>(x);
            const areal2 c0 = v2p[2 * (int64_t)t], d0 = v2p[2 * (int64_t)t + 1], xa = x2p[j0];
            areal2 c1, d1, c2, d2;
            c1.x = c1.y = d1.x = d1.y = c2.x = c2.y = d2.x = d2.y = 0;
            if (p1) { c1 = v2p[2 * (int64_t)t1]; d1 = v2p[2 * (int64_t)t1 + 1]; }
            if (p2) { c2 = v2p[2 * (int64_t)t2]; d2 = v2p[2 * (int64_t)t2 + 1]; }
            const areal2 xb = x2p[j1], xc = x2p[j2];
            a0 += (double)c0.x * xa.x + (double)c0.y * xa.y + (double)c1.x * xb.x + (double)c1.y * xb.y +
                  (double)c2.x * xc.x + (double)c2.y * xc.y;
            a1 += (double)d0.x * xa.x + (double)d0.y * xa.y + (double)d1.x * xb.x + (double)d1.y * xb.y +
                  (double)d2.x * xc.x + (double)d2.y * xc.y;
        }
    }
#pragma unroll
    for (int o = 2; o > 0; o >>= 1) {
        a0 += __shfl_down_sync(0xffffffffu, a0, o, 4);
        if (BS == 2) a1 += __shfl_down_sync(0xffffffffu, a1, o, 4);
    }
    if (ok && lane == 0) {
        if (BS == 1) {
            y[i] = (areal)((b ? (double)b[i] : 0.0) + alpha * a0);
        } else {
            y[2 * (int64_t)i] = (areal)((b ? (double)b[2 * (int64_t)i] : 0.0) + alpha * a0);
            y[2 * (int64_t)i + 1] = (areal)((b ? (double)b[2 * (int64_t)i + 1] : 0.0) + alpha * a1);
        }
    }
}

int hemo_bsr_spmv_ex(hemo_ctx* ctx, int bs, int n, const int32_t* rowptr, const int32_t* col, const areal* val,
                     const areal* x, double alpha, const areal* b, areal* y) {
    const int grid = hemo_grid((int64_t)n * 4, 256);
    if (bs == 1) HEMO_LAUNCH(ctx, k_bsr_spmv<1>, grid, 256, 0, ctx->stream, n, rowptr, col, val, x, alpha, b, y);
    else HEMO_LAUNCH(ctx, k_bsr_spmv<2>, grid, 256, 0, ctx->stream, n, rowptr, col, val, x, alpha, b, y);
    return 0;
}

int hemo_bsr_spmv(hemo_ctx* ctx, int bs, int n, const int32_t* rowptr, const int32_t* col, const areal* val,
                  const areal* x, areal* y) {
    return hemo_bsr_spmv_ex(ctx, bs, n, rowptr, col, val, x, 1.0, nullptr, y);
}

// ---------------------------------------------------------------------------
// vector kernels
// ---------------------------------------------------------------------------
__global__ void k_axpy(int64_t n, double a, const double* __restrict__ x, double* __restrict__ y) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        y[i] = fma(a, x[i], y[i]);
}

__global__ void k_scale_copy(int64_t n, double a, const double* __restrict__ x, double* __restrict__ y) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        y[i] = a * x[i];
}

// y = x * (1 / s[0]) with s on the device
__global__ void k_scale_inv_dev(int64_t n, const double* __restrict__ s, const double* __restrict__ x,
                                double* __restrict__ y) {
    const double a = 1.0 / s[0];
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        y[i] = a * x[i];
}

__global__ void __launch_bounds__(RED_THREADS)
k_dot_partial(int64_t n, const double* __restrict__ x, const double* __restrict__ y, double* __restrict__ partial) {
    __shared__ double sh[32];
    double acc = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        acc = fma(x[i], y[i], acc);
    acc = block_sum(acc, sh);
    if (threadIdx.x == 0) partial[blockIdx.x] = acc;
}

// out[k] = sum_b partial[k * nblk + b], one block per k, fixed order
__global__ void __launch_bounds__(RED_THREADS)
k_reduce_final(int nblk, const double* __restrict__ partial, double* __restrict__ out, int sqrt_last_k) {
    __shared__ double sh[32];
    const int k = blockIdx.x;
    double acc = 0.0;
    for (int b = threadIdx.x; b < nblk; b += blockDim.x) acc += partial[(int64_t)k * nblk + b];
    acc = block_sum(acc, sh);
    if (threadIdx.x == 0) out[k] = (sqrt_last_k >= 0 && k == sqrt_last_k) ? sqrt(acc) : acc;
}

static int grid_for(int64_t n) {
    int64_t g = (n + RED_THREADS - 1) / RED_THREADS;
    if (g > RED_BLOCKS) g = RED_BLOCKS;
    if (g < 1) g = 1;
    return (int)g;
}

extern "C" int hemo_axpy(hemo_ctx* ctx, int64_t n, double a, const double* x_dev, double* y_dev) {
    if (!ctx || !x_dev || !y_dev || n < 0) return HEMO_EINVAL;
    k_axpy<<<grid_for(n), RED_THREADS, 0, ctx->stream>>>(n, a, x_dev, y_dev);
    HEMO_LAUNCH_CHECK(ctx);
    return 0;
}

int hemo_scale_copy(hemo_ctx* ctx, int64_t n, double a, const double* x, double* y) {
    k_scale_copy<<<grid_for(n), RED_THREADS, 0, ctx->stream>>>(n, a, x, y);
    HEMO_LAUNCH_CHECK(ctx);
    return 0;
}

int hemo_scale_inv_dev(hemo_ctx* ctx, int64_t n, const double* s_dev, const double* x, double* y) {
    k_scale_inv_dev<<<grid_for(n), RED_THREADS, 0, ctx->stream>>>(n, s_dev, x, y);
    HEMO_LAUNCH_CHECK(ctx);
    return 0;
}

// dot product left on the device in ctx->red_out[slot]
int hemo_dot_to_slot(hemo_ctx* ctx, int64_t n, const double* x, const double* y, int slot, bool take_sqrt) {
    int rc = hemo_ensure_reduce(ctx, RED_BLOCKS * 8, 512);
    if (rc) return rc;
    const int g = grid_for(n);
    k_dot_partial<<<g, RED_THREADS, 0, ctx->stream>>>(n, x, y, ctx->red_partial);
    HEMO_LAUNCH_CHECK(ctx);
    k_reduce_final<<<1, RED_THREADS, 0, ctx->stream>>>(g, ctx->red_partial, ctx->red_out + slot, take_sqrt ? 0 : -1);
    HEMO_LAUNCH_CHECK(ctx);
    return 0;
}

int hemo_dot_dev(hemo_ctx* ctx, int64_t n, const double* x, const double* y, double* out_host) {
    int rc = hemo_dot_to_slot(ctx, n, x, y, 0, false);
    if (rc) return rc;
    HEMO_CHECK_CUDA(ctx, cudaMemcpyAsync(ctx->red_host, ctx->red_out, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *out_host = ctx->red_host[0];
    return 0;
}

extern "C" int hemo_dot(hemo_ctx* ctx, int64_t n, const double* x_dev, const double* y_dev, double* out_host) {
    if (!ctx || !x_dev || !y_dev || !out_host || n < 0) return HEMO_EINVAL;
    return hemo_dot_dev(ctx, n, x_dev, y_dev, out_host);
}

// dot product over the owned entries of two local [u | p] vectors, summed over the ranks (VecDot under MPI)
__global__ void __launch_bounds__(RED_THREADS)
k_dot_seg_partial(int64_t len0, int64_t off1, int64_t len1, const double* __restrict__ x, const double* __restrict__ y,
                  double* __restrict__ partial) {
    __shared__ double sh[32];
    double acc = 0.0;
    const int64_t n = len0 + len1;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t q = i < len0 ? i : i - len0 + off1;
        acc = fma(x[q], y[q], acc);
    }
    acc = block_sum(acc, sh);
    if (threadIdx.x == 0) partial[blockIdx.x] = acc;
}

extern "C" int hemo_global_dot(hemo_ctx* ctx, const double* x_dev, const double* y_dev, double* out_host) {
    if (!ctx || !x_dev || !y_dev || !out_host) return HEMO_EINVAL;
    if (!ctx->cells) HEMO_FAIL(ctx, HEMO_ESTATE, "mesh not set");
    const int64_t N = (int64_t)(ctx->dim + 1) * ctx->n;
    if (!ctx->comm || ctx->kry.seg_len0 == 0) return hemo_dot_dev(ctx, N, x_dev, y_dev, out_host);
    int rc = hemo_ensure_reduce(ctx, RED_BLOCKS * 8, 512);
    if (rc) return rc;
    const HemoKrylov& K = ctx->kry;
    const int g = grid_for(K.seg_len0 + K.seg_len1);
    k_dot_seg_partial<<<g, RED_THREADS, 0, ctx->stream>>>(K.seg_len0, K.seg_off1, K.seg_len1, x_dev, y_dev, ctx->red_partial);
    HEMO_LAUNCH_CHECK(ctx);
    k_reduce_final<<<1, RED_THREADS, 0, ctx->stream>>>(g, ctx->red_partial, ctx->red_out + 502, -1);
    HEMO_LAUNCH_CHECK(ctx);
    if ((rc = hemo_comm_allreduce_j(ctx, ctx->red_out + 502, 1))) return rc;
    HEMO_CHECK_CUDA(ctx, cudaMemcpyAsync(ctx->red_host + 502, ctx->red_out + 502, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *out_host = ctx->red_host[502];
    return 0;
}

extern "C" int hemo_norm2(hemo_ctx* ctx, int64_t n, const double* x_dev, double* out_host) {
    if (!ctx || !x_dev || !out_host || n < 0) return HEMO_EINVAL;
    double d = 0.0;
    int rc = hemo_dot_dev(ctx, n, x_dev, x_dev, &d);
    if (rc) return rc;
    *out_host = sqrt(d);
    return 0;
}

// ---------------------------------------------------------------------------
// Gram–Schmidt kernels for (F)GMRES: classical GS, one pass each
//   mdot:  h[i] = V_i . w  for i < k  (w read once per tile, V streamed)
//   maxpy: w -= sum_i h[i] V_i ; partial ||w||^2 in the same pass
// ---------------------------------------------------------------------------
#define MD_TILE 8   // elements per thread held in registers

__global__ void __launch_bounds__(RED_THREADS)
k_mdot_partial(int64_t n, int k, const double* __restrict__ V, int64_t ldv, const double* __restrict__ w,
               double* __restrict__ partial /*[k][gridDim.x]*/) {
    __shared__ double sh[32];
    extern __shared__ double acc_sh[];   // k running sums of this block (thread 0 only)
    const int64_t tile = (int64_t)RED_THREADS * MD_TILE;
    const int64_t ntiles = (n + tile - 1) / tile;
    for (int i = threadIdx.x; i < k; i += blockDim.x) acc_sh[i] = 0.0;
    __syncthreads();
    for (int64_t tl = blockIdx.x; tl < ntiles; tl += gridDim.x) {
        const int64_t base = tl * tile + threadIdx.x;
        double wr[MD_TILE];
#pragma unroll
        for (int e = 0; e < MD_TILE; ++e) {
            const int64_t idx = base + (int64_t)e * RED_THREADS;
            wr[e] = (idx < n) ? w[idx] : 0.0;
        }
        for (int i = 0; i < k; ++i) {
            const double* Vi = V + (int64_t)i * ldv;
            double a = 0.0;
#pragma unroll
            for (int e = 0; e < MD_TILE; ++e) {
                const int64_t idx = base + (int64_t)e * RED_THREADS;
                if (idx < n) a = fma(Vi[idx], wr[e], a);
            }
            a = block_sum(a, sh);
            if (threadIdx.x == 0) acc_sh[i] += a;   // fixed tile order per block
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < k; i += blockDim.x) partial[(int64_t)i * gridDim.x + blockIdx.x] = acc_sh[i];
}

__global__ void __launch_bounds__(RED_THREADS)
k_maxpy_norm(int64_t n, int k, const double* __restrict__ V, int64_t ldv, const double* __restrict__ hcoef,
             double sign, double* __restrict__ w, double* __restrict__ partial) {
    __shared__ double sh[32];
    extern __shared__ double hsh[];
    for (int i = threadIdx.x; i < k; i += blockDim.x) hsh[i] = hcoef[i];
    __syncthreads();
    double nrm = 0.0;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < n; idx += (int64_t)gridDim.x * blockDim.x) {
        double acc = w[idx];
        for (int i = 0; i < k; ++i) acc = fma(sign * hsh[i], V[(int64_t)i * ldv + idx], acc);
        w[idx] = acc;
        nrm = fma(acc, acc, nrm);
    }
    nrm = block_sum(nrm, sh);
    if (threadIdx.x == 0 && partial) partial[blockIdx.x] = nrm;
}

// h (device, ctx->red_out[0..k)) = V^T w ; copies h to red_host and syncs
int hemo_mdot(hemo_ctx* ctx, int64_t n, int k, const double* V, int64_t ldv, const double* w, double* h_host) {
    int rc = hemo_ensure_reduce(ctx, (size_t)RED_BLOCKS * (size_t)(k + 2), 512 > k + 2 ? 512 : (size_t)k + 2);
    if (rc) return rc;
    // w is re-read once per basis vector from L2/HBM; V dominates the traffic.
    int g = grid_for((n + MD_TILE - 1) / MD_TILE);
    HEMO_PROF_BEGIN(ctx, HEMO_PROF_MDOT);
    k_mdot_partial<<<g, RED_THREADS, sizeof(double) * k, ctx->stream>>>(n, k, V, ldv, w, ctx->red_partial);
    HEMO_LAUNCH_CHECK(ctx);
    HEMO_PROF_END(ctx, HEMO_PROF_MDOT);
    k_reduce_final<<<k, RED_THREADS, 0, ctx->stream>>>(g, ctx->red_partial, ctx->red_out, -1);
    HEMO_LAUNCH_CHECK(ctx);
    HEMO_CHECK_CUDA(ctx, cudaMemcpyAsync(ctx->red_host, ctx->red_out, sizeof(double) * k, cudaMemcpyDeviceToHost, ctx->stream));
    HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < k; ++i) h_host[i] = ctx->red_host[i];
    return 0;
}

// w += sign * sum_i h[i] V_i using the coefficients in hcoef_dev; returns ||w|| if norm_host
int hemo_maxpy(hemo_ctx* ctx, int64_t n, int k, const double* V, int64_t ldv, const double* hcoef_dev, double sign,
               double* w, double* norm_host) {
    int rc = hemo_ensure_reduce(ctx, (size_t)RED_BLOCKS * 2, 512);
    if (rc) return rc;
    const int g = grid_for(n);
    HEMO_PROF_BEGIN(ctx, HEMO_PROF_MAXPY);
    k_maxpy_norm<<<g, RED_THREADS, sizeof(double) * (k > 0 ? k : 1), ctx->stream>>>(
        n, k, V, ldv, hcoef_dev, sign, w, norm_host ? ctx->red_partial : nullptr);
    HEMO_LAUNCH_CHECK(ctx);
    HEMO_PROF_END(ctx, HEMO_PROF_MAXPY);
    if (norm_host) {
        k_reduce_final<<<1, RED_THREADS, 0, ctx->stream>>>(g, ctx->red_partial, ctx->red_out + 500, 0);
        HEMO_LAUNCH_CHECK(ctx);
        HEMO_CHECK_CUDA(ctx, cudaMemcpyAsync(ctx->red_host + 500, ctx->red_out + 500, sizeof(double),
                                             cudaMemcpyDeviceToHost, ctx->stream));
        HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        *norm_host = ctx->red_host[500];
    }
    return 0;
}

// mean removal on the device (constant-pressure null space): x -= sum(x)/n.  Two launches: per-block partial sums
// (optionally copying src -> x on the way), then every block re-reduces the partials in the same fixed order and
// subtracts (no single-block reduction kernel in between).
__global__ void __launch_bounds__(RED_THREADS)
k_sub_mean_partials(int64_t n, int nparts, const double* __restrict__ partial, double* __restrict__ x) {
    __shared__ double sh[32];
    __shared__ double mean;
    hemo_pdl_wait();
    hemo_pdl_trigger();
    double acc = 0.0;
    for (int t = threadIdx.x; t < nparts; t += blockDim.x) acc += partial[t];
    acc = block_sum(acc, sh);
    if (threadIdx.x == 0) mean = acc / (double)n;
    __syncthreads();
    const double m = mean;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        x[i] -= m;
}

// partial[b] = sum of this block's entries of src; dst = src when they differ
__global__ void __launch_bounds__(RED_THREADS)
k_sum_partial(int64_t n, const double* src, double* dst, double* __restrict__ partial) {
    __shared__ double sh[32];
    hemo_pdl_wait();
    hemo_pdl_trigger();
    double acc = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double v = src[i];
        if (dst != src) dst[i] = v;
        acc += v;
    }
    acc = block_sum(acc, sh);
    if (threadIdx.x == 0) partial[blockIdx.x] = acc;
}

// x = src - mean(src)  (src == x: in place)
int hemo_copy_remove_mean(hemo_ctx* ctx, int64_t n, const double* src, double* x) {
    int rc = hemo_ensure_reduce(ctx, (size_t)RED_BLOCKS * 2, 512);
    if (rc) return rc;
    const int g = grid_for(n);
    HEMO_LAUNCH(ctx, k_sum_partial, g, RED_THREADS, 0, ctx->stream, n, src, x, ctx->red_partial);
    HEMO_LAUNCH(ctx, k_sub_mean_partials, g, RED_THREADS, 0, ctx->stream, n, g, ctx->red_partial, x);
    return 0;
}

int hemo_remove_mean(hemo_ctx* ctx, int64_t n, double* x) { return hemo_copy_remove_mean(ctx, n, x, x); }
