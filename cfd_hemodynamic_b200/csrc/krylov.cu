// Device-resident right-preconditioned FGMRES(restart).
//
// Replaces KSPSolve(fgmres) as configured by the reference at src/solvers/stabilized_schur.py:226-229,272-273
// (flexible GMRES, right preconditioning, classical Gram-Schmidt without refinement, restart, rtol / atol / max_it).
//
// B200 design: the whole Arnoldi recurrence lives on the device.  The Hessenberg column, the Givens rotations, the
// residual estimate and the convergence flag are updated by the last block of the update kernel; every kernel reads
// the column index j from the device state, so the arguments of one iteration never change and the iteration
// (preconditioner + SpMV + multi-dot + multi-axpy/norm/Givens) replays as ONE CUDA graph.  The host only polls the
// state at the iteration count it expects from the previous solve; the k_fg_* kernels queued beyond convergence exit at
// once (the preconditioner's kernels run again on the stale input, and nothing reads their output).
//
// Basis vectors are stored unnormalised with their scale s_j = 1/||w_j|| (device array): the SpMV writes w straight
// into slot j+1, the update kernel orthogonalises it in place, and the "normalise" pass of textbook GMRES disappears
// (the preconditioner input is scaled while it is staged).
//
// Multi-GPU (one partition per GPU, hemo_comm_init): vectors are local [owned | ghost]; reductions run over the owned
// entries and are summed with one ncclAllReduce each (PETSc VecMDot / VecNorm), the search direction gets a forward
// ghost update (ghostUpdate(INSERT, FORWARD), stabilized_schur.py:137-142) before the operator is applied.
#include <math.h>

#include "hemo_internal.cuh"

#define FG_BLOCKS 1184   // 148 SMs * 8
#define FG_THREADS 256
#define FG_TILE 8

int hemo_remove_mean(hemo_ctx* ctx, int64_t n, double* x);
int hemo_pc_apply_body(hemo_ctx* ctx, const double* vals_dev, const double* r_dev, double* z_dev);

struct FgState {
    int j;           // column of the current cycle
    int its;         // iterations done
    int converged;   // 0 running, 1 res <= tol, 2 happy breakdown, -1 non-finite
    int cycle_full;  // j reached restart
    double res, tol, bnorm, beta;
    unsigned int ticket_mdot, ticket_maxpy, ticket_misc, pad;
};

// owned entries of a local [u | p] vector: [0, len0) and [off1, off1 + len1)
struct FgSeg {
    int64_t len0, off1, len1;
};
__device__ __forceinline__ int64_t seg_index(const FgSeg& s, int64_t i) { return i < s.len0 ? i : i - s.len0 + s.off1; }
__device__ __forceinline__ bool seg_owned(const FgSeg& s, int64_t q) { return q < s.len0 || (q >= s.off1 && q < s.off1 + s.len1); }

__device__ __forceinline__ double fg_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double fg_block_sum(double v, double* sh) {
    v = fg_warp_sum(v);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) sh[wid] = v;
    __syncthreads();
    double r = 0.0;
    if (wid == 0) {
        r = (lane < (blockDim.x >> 5)) ? sh[lane] : 0.0;
        r = fg_warp_sum(r);
    }
    __syncthreads();
    return r;
}

// the last block to arrive gets true (all other blocks' global writes are visible to it)
__device__ __forceinline__ bool fg_last_block(unsigned int* ticket) {
    __shared__ bool last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int t = atomicAdd(ticket, 1u);
        last = (t == gridDim.x - 1);
        if (last) *ticket = 0;
    }
    __syncthreads();
    if (last) __threadfence();
    return last;
}

// ---- start of a solve / of a restart cycle ------------------------------------------------------------------------
// V_0 = r (unnormalised), partial ||r||^2
__global__ void __launch_bounds__(FG_THREADS)
k_fg_start(FgState* st, FgSeg seg, int64_t nloc, const double* __restrict__ r, double* __restrict__ V0,
           double* __restrict__ partial, double* __restrict__ out, int first) {
    __shared__ double sh[32];
    if (!first && st->converged) return;
    // every local entry is kept (the rows of the overlap region are complete: their values equal the owners' up to
    // rounding, so the overlapping Schwarz preconditioner needs no ghost update of its input); owned entries are reduced
    double acc = 0.0;
    for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < nloc; q += (int64_t)gridDim.x * blockDim.x) {
        const double v = r[q];
        V0[q] = v;
        if (seg_owned(seg, q)) acc = fma(v, v, acc);
    }
    acc = fg_block_sum(acc, sh);
    if (threadIdx.x == 0) partial[blockIdx.x] = acc;
    if (!fg_last_block(&st->ticket_misc)) return;
    double s = 0.0;
    for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) s += partial[b];
    s = fg_block_sum(s, sh);
    if (threadIdx.x == 0) out[0] = s;     // local ||r||^2 (summed over ranks before k_fg_begin_cycle)
}

__global__ void k_fg_begin_cycle(FgState* st, const double* __restrict__ normsq, int first, double rtol, double atol,
                                 double* __restrict__ g, double* __restrict__ scale, int m) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if (!first && st->converged) return;
    // a sum of squares: no fmax clamp, which would turn a NaN (a non-finite entry) into a zero norm
    const double beta = sqrt(normsq[0]);
    if (first) {
        st->its = 0;
        st->converged = 0;
        st->bnorm = beta;
        st->tol = fmax(rtol * beta, atol);
        st->res = beta;
        if (beta == 0.0 || beta <= atol) st->converged = 1;
        else if (!isfinite(beta)) st->converged = -1;
    } else {
        st->res = beta;
        if (beta <= st->tol) st->converged = 1;
        else if (!isfinite(beta)) st->converged = -1;
    }
    st->beta = beta;
    st->j = 0;
    st->cycle_full = 0;
    for (int i = 0; i <= m; ++i) g[i] = 0.0;
    g[0] = beta;
    scale[0] = beta > 0.0 ? 1.0 / beta : 0.0;
}

// ---- one iteration ---------------------------------------------------------------------------------------------------
// stage the preconditioner input: pc_in = s_j V_j (all local entries: ghosts are refreshed by the halo update)
__global__ void __launch_bounds__(FG_THREADS)
k_fg_load(const FgState* __restrict__ st, int64_t n, const double* __restrict__ V, int64_t ldv,
          const double* __restrict__ scale, double* __restrict__ pc_in) {
    hemo_pdl_wait();
    hemo_pdl_trigger();
    if (st->converged || st->cycle_full) return;
    const int j = st->j;
    const double s = scale[j];
    const double* v = V + (int64_t)j * ldv;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        pc_in[i] = s * v[i];
}

// w = A z with z = pc_out; the same pass stores z as Z_j (node-structured monolithic Jacobian, 8 lanes per node)
__global__ void __launch_bounds__(256)
k_fg_spmv_node(const FgState* __restrict__ st, int n, int64_t nnz_node, const int32_t* __restrict__ nrowptr,
               const int32_t* __restrict__ ncol, const double* __restrict__ vals, const double* __restrict__ z,
               double* __restrict__ V, double* __restrict__ Z, int64_t ldv) {
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = gt >> 3;
    const int lane = gt & 7;
    const bool ok = i < n;
    const int r0 = ok ? nrowptr[i] : 0;
    const int deg = ok ? nrowptr[i + 1] - r0 : 0;
    const int64_t ru0 = 6 * (int64_t)r0, ru1 = ru0 + 3 * deg, rp = 6 * nnz_node + 3 * (int64_t)r0;
    // the first trip's column index and Jacobian entries (constant during the solve) load before the wait
    int c = 0;
    double v[9];
    auto fetch = [&](int t) {
        c = ncol[r0 + t];
        v[0] = vals[ru0 + 2 * t]; v[1] = vals[ru0 + 2 * t + 1]; v[2] = vals[ru0 + 2 * deg + t];
        v[3] = vals[ru1 + 2 * t]; v[4] = vals[ru1 + 2 * t + 1]; v[5] = vals[ru1 + 2 * deg + t];
        v[6] = vals[rp + 2 * t];  v[7] = vals[rp + 2 * t + 1];  v[8] = vals[rp + 2 * deg + t];
    };
    if (lane < deg) fetch(lane);
    hemo_pdl_wait();
    hemo_pdl_trigger();
    if (st->converged || st->cycle_full) return;
    const int j = st->j;
    const double* xu = z;
    const double* xp = z + 2 * (int64_t)n;
    double* w = V + (int64_t)(j + 1) * ldv;
    double* zj = Z + (int64_t)j * ldv;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0;
    for (int t = lane; t < deg; t += 8) {
        if (t != lane) fetch(t);
        const double2 xv = reinterpret_cast<const double2*>(xu)[c];
        const double x2 = xp[c];
        a0 += v[0] * xv.x + v[1] * xv.y + v[2] * x2;
        a1 += v[3] * xv.x + v[4] * xv.y + v[5] * x2;
        a2 += v[6] * xv.x + v[7] * xv.y + v[8] * x2;
    }
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) {
        a0 += __shfl_down_sync(0xffffffffu, a0, o, 8);
        a1 += __shfl_down_sync(0xffffffffu, a1, o, 8);
        a2 += __shfl_down_sync(0xffffffffu, a2, o, 8);
    }
    if (ok && lane == 0) {
        reinterpret_cast<double2*>(w)[i] = make_double2(a0, a1);
        w[2 * (int64_t)n + i] = a2;
        reinterpret_cast<double2*>(zj)[i] = reinterpret_cast<const double2*>(xu)[i];
        zj[2 * (int64_t)n + i] = xp[i];
    }
}

// generic variant: w was produced by another SpMV routine (tetrahedra); only stores Z_j = z and moves w into slot j+1
__global__ void __launch_bounds__(FG_THREADS)
k_fg_store(const FgState* __restrict__ st, int64_t n, const double* __restrict__ z, const double* __restrict__ w,
           double* __restrict__ V, double* __restrict__ Z, int64_t ldv) {
    hemo_pdl_wait();
    hemo_pdl_trigger();
    if (st->converged || st->cycle_full) return;
    const int j = st->j;
    double* wj = V + (int64_t)(j + 1) * ldv;
    double* zj = Z + (int64_t)j * ldv;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        zj[i] = z[i];
        wj[i] = w[i];
    }
}

// h_i = s_i (V_i . w), i <= j  (VecMDot): the w tile is held in registers and V streamed once, four basis vectors
// in flight per pass; partial sums go warp -> per-warp shared accumulators (no block barrier inside the loop) ->
// one partial per block and vector.  k_fg_mdot_final sums the partials in a fixed order (bitwise reproducible).
template <bool SEG>
__global__ void __launch_bounds__(FG_THREADS)
k_fg_mdot(const FgState* __restrict__ st, FgSeg seg, const double* __restrict__ V, int64_t ldv,
          double* __restrict__ partial /*[m+1][gridDim.x]*/, int kpad) {
    extern __shared__ double acc_sh[];       // (FG_THREADS / 32) x kpad
    hemo_pdl_wait();
    hemo_pdl_trigger();
    if (st->converged || st->cycle_full) return;
    const int j = st->j, k = j + 1;
    const double* w = V + (int64_t)k * ldv;
    const int64_t n = seg.len0 + seg.len1;
    const int64_t tile = (int64_t)FG_THREADS * FG_TILE;
    const int64_t ntiles = (n + tile - 1) / tile;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = FG_THREADS / 32;
    for (int i = threadIdx.x; i < nw * kpad; i += blockDim.x) acc_sh[i] = 0.0;
    __syncthreads();
    double* acc = acc_sh + wid * kpad;
    for (int64_t tl = blockIdx.x; tl < ntiles; tl += gridDim.x) {
        const int64_t base = tl * tile + threadIdx.x;
        double wr[FG_TILE];
        int64_t qi[FG_TILE];
#pragma unroll
        for (int e = 0; e < FG_TILE; ++e) {
            const int64_t idx = base + (int64_t)e * FG_THREADS;
            const bool ok = idx < n;
            qi[e] = ok ? (SEG ? seg_index(seg, idx) : idx) : 0;
            wr[e] = ok ? w[qi[e]] : 0.0;          // out-of-range lanes multiply entry 0 by zero
        }
        for (int i = 0; i < k; i += 4) {
            const double* V0 = V + (int64_t)i * ldv;
            const double* V1 = V + (int64_t)min(i + 1, k - 1) * ldv;
            const double* V2 = V + (int64_t)min(i + 2, k - 1) * ldv;
            const double* V3 = V + (int64_t)min(i + 3, k - 1) * ldv;
            double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll
            for (int e = 0; e < FG_TILE; ++e) {
                a0 = fma(V0[qi[e]], wr[e], a0);
                a1 = fma(V1[qi[e]], wr[e], a1);
                a2 = fma(V2[qi[e]], wr[e], a2);
                a3 = fma(V3[qi[e]], wr[e], a3);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                a0 += __shfl_down_sync(0xffffffffu, a0, o);
                a1 += __shfl_down_sync(0xffffffffu, a1, o);
                a2 += __shfl_down_sync(0xffffffffu, a2, o);
                a3 += __shfl_down_sync(0xffffffffu, a3, o);
            }
            if (lane == 0) {
                acc[i] += a0;
                if (i + 1 < k) acc[i + 1] += a1;
                if (i + 2 < k) acc[i + 2] += a2;
                if (i + 3 < k) acc[i + 3] += a3;
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < k; i += blockDim.x) {
        double s = 0.0;
#pragma unroll
        for (int q = 0; q < nw; ++q) s += acc_sh[q * kpad + i];
        partial[(int64_t)i * gridDim.x + blockIdx.x] = s;
    }
}

// one block per basis vector (blocks beyond the current column leave at once: the grid is fixed for the graph)
__global__ void __launch_bounds__(128)
k_fg_mdot_final(const FgState* __restrict__ st, int nblk, const double* __restrict__ partial,
                const double* __restrict__ scale, double* __restrict__ hcol) {
    __shared__ double sh[32];
    hemo_pdl_wait();
    hemo_pdl_trigger();
    if (st->converged || st->cycle_full) return;
    const int i = blockIdx.x;
    if (i > st->j) return;
    double s = 0.0;
    for (int b = threadIdx.x; b < nblk; b += blockDim.x) s += partial[(int64_t)i * nblk + b];
    s = fg_block_sum(s, sh);
    if (threadIdx.x == 0) hcol[i] = scale[i] * s;
}

// Givens update of column j from h (hcol[0..j]) and hn.  Called by a whole block: the previous rotations and the
// column are staged in shared memory by all threads (one coalesced pass), then thread 0 runs the dependent chain out
// of shared memory (a chain of global loads would cost one L2 round trip per rotation).
__device__ void fg_givens(FgState* st, int m, const double* __restrict__ hcol, double hn, double* __restrict__ H,
                          double* __restrict__ cs, double* __restrict__ sn, double* __restrict__ g,
                          double* __restrict__ scale, double* __restrict__ smem /* 3 (m + 2) */) {
    const int j = st->j;
    double* hs = smem;
    double* cs_s = smem + (m + 2);
    double* sn_s = smem + 2 * (m + 2);
    for (int i = threadIdx.x; i <= j; i += blockDim.x) {
        hs[i] = hcol[i];
        if (i < j) { cs_s[i] = cs[i]; sn_s[i] = sn[i]; }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        hs[j + 1] = hn;
        for (int i = 0; i < j; ++i) {
            const double a = hs[i], b = hs[i + 1];
            hs[i] = cs_s[i] * a + sn_s[i] * b;
            hs[i + 1] = -sn_s[i] * a + cs_s[i] * b;
        }
        const double a = hs[j], b = hs[j + 1];
        const double d = hypot(a, b);
        const double c = d > 0.0 ? a / d : 1.0, sgn = d > 0.0 ? b / d : 0.0;
        cs[j] = c;
        sn[j] = sgn;
        hs[j] = d;
        hs[j + 1] = 0.0;
        const double gj = g[j];
        g[j + 1] = -sgn * gj;
        g[j] = c * gj;
        const double res = fabs(sgn * gj);
        st->res = res;
        st->its += 1;
        scale[j + 1] = hn > 0.0 ? 1.0 / hn : 0.0;
        if (!isfinite(res) || !isfinite(d)) st->converged = -1;     // d: a non-finite column gives c = 1, s = 0
        else if (res <= st->tol) st->converged = 1;
        else if (hn == 0.0) st->converged = 2;
        if (j + 1 >= m) st->cycle_full = 1;
    }
    __syncthreads();
    double* Hj = H + (int64_t)j * (m + 1);
    for (int i = threadIdx.x; i <= j + 1; i += blockDim.x) Hj[i] = hs[i];
    __syncthreads();
    if (threadIdx.x == 0) st->j = j + 1;
}

// w -= sum_i (s_i h_i) V_i ; ||w||^2 ; (single GPU) Givens by the last block
__global__ void __launch_bounds__(FG_THREADS)
k_fg_maxpy(FgState* st, FgSeg seg, int64_t nloc, double* __restrict__ V, int64_t ldv, const double* __restrict__ hcol, int m,
           double* __restrict__ partial, double* __restrict__ normsq_out, int do_givens, double* __restrict__ H,
           double* __restrict__ cs, double* __restrict__ sn, double* __restrict__ g, double* __restrict__ scale) {
    __shared__ double sh[32];
    extern __shared__ double hsh[];
    hemo_pdl_wait();
    hemo_pdl_trigger();
    if (st->converged || st->cycle_full) return;
    const int j = st->j, k = j + 1;
    double* w = V + (int64_t)k * ldv;
    for (int i = threadIdx.x; i < k; i += blockDim.x) hsh[i] = hcol[i] * scale[i];
    __syncthreads();
    double nrm = 0.0;
    for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < nloc; q += (int64_t)gridDim.x * blockDim.x) {
        double acc = w[q];
        for (int i = 0; i < k; ++i) acc = fma(-hsh[i], V[(int64_t)i * ldv + q], acc);
        w[q] = acc;
        if (seg_owned(seg, q)) nrm = fma(acc, acc, nrm);
    }
    nrm = fg_block_sum(nrm, sh);
    if (threadIdx.x == 0) partial[blockIdx.x] = nrm;
    if (!fg_last_block(&st->ticket_maxpy)) return;
    __shared__ double total;
    double s = 0.0;
    for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) s += partial[b];
    s = fg_block_sum(s, sh);
    if (threadIdx.x == 0) {
        normsq_out[0] = s;
        total = s;
    }
    __syncthreads();
    if (do_givens) fg_givens(st, m, hcol, sqrt(total), H, cs, sn, g, scale, hsh);
}

// multi-GPU: Givens after the norm has been summed over the ranks
__global__ void k_fg_givens(FgState* st, int m, const double* __restrict__ hcol, const double* __restrict__ normsq,
                            double* __restrict__ H, double* __restrict__ cs, double* __restrict__ sn,
                            double* __restrict__ g, double* __restrict__ scale) {
    extern __shared__ double gsh[];
    hemo_pdl_wait();
    hemo_pdl_trigger();
    if (st->converged || st->cycle_full) return;
    fg_givens(st, m, hcol, sqrt(normsq[0]), H, cs, sn, g, scale, gsh);
}

// ---- end of a cycle: y += Z_k (H_k^-1 g_k) ------------------------------------------------------------------------
__global__ void k_fg_backsolve(FgState* st, int m, const double* __restrict__ H, const double* __restrict__ g,
                               double* __restrict__ ycoef, int* __restrict__ kout) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const int k = st->j;
    for (int i = k - 1; i >= 0; --i) {
        double s = g[i];
        for (int l = i + 1; l < k; ++l) s -= H[(int64_t)l * (m + 1) + i] * ycoef[l];
        ycoef[i] = s / H[(int64_t)i * (m + 1) + i];
    }
    *kout = k;
}

__global__ void __launch_bounds__(FG_THREADS)
k_fg_update(const int* __restrict__ kptr, int64_t n, const double* __restrict__ Z, int64_t ldv,
            const double* __restrict__ ycoef, double* __restrict__ y) {
    extern __shared__ double csh[];
    const int k = *kptr;
    for (int i = threadIdx.x; i < k; i += blockDim.x) csh[i] = ycoef[i];
    __syncthreads();
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < n; idx += (int64_t)gridDim.x * blockDim.x) {
        double acc = y[idx];
        for (int i = 0; i < k; ++i) acc = fma(csh[i], Z[(int64_t)i * ldv + idx], acc);
        y[idx] = acc;
    }
}

// r = b - A y for a restart is formed by the caller's SpMV; this kernel only combines
__global__ void __launch_bounds__(FG_THREADS)
k_fg_residual(const FgState* __restrict__ st, int64_t n, const double* __restrict__ b, const double* __restrict__ Ay,
              double* __restrict__ r) {
    if (st->converged) return;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        r[i] = b[i] - Ay[i];
}

// ---------------------------------------------------------------------------------------------------------------------
static int fg_grid(int64_t n, int per_thread) {
    int64_t g = (n + (int64_t)FG_THREADS * per_thread - 1) / ((int64_t)FG_THREADS * per_thread);
    if (g > FG_BLOCKS) g = FG_BLOCKS;
    if (g < 1) g = 1;
    return (int)g;
}

static int fg_ensure(hemo_ctx* ctx, int m, int64_t ldv) {
    HemoKrylov& K = ctx->kry;
    int rc;
    if (K.m != m || K.ldv != ldv || !ctx->kry_V) {
        if ((rc = hemo_alloc(ctx, &ctx->kry_V, (size_t)(m + 1) * ldv))) return rc;
        if ((rc = hemo_alloc(ctx, &ctx->kry_Z, (size_t)m * ldv))) return rc;
        if ((rc = hemo_alloc(ctx, &ctx->kry_w, (size_t)ldv + 512))) return rc;
        // ghost entries of the basis are never written by the owned-entry kernels: start from defined values
        HEMO_CHECK_CUDA(ctx, cudaMemsetAsync(ctx->kry_V, 0, sizeof(double) * (size_t)(m + 1) * ldv, ctx->stream));
        HEMO_CHECK_CUDA(ctx, cudaMemsetAsync(ctx->kry_Z, 0, sizeof(double) * (size_t)m * ldv, ctx->stream));
        if ((rc = hemo_alloc(ctx, &K.H, (size_t)(m + 1) * m))) return rc;
        if ((rc = hemo_alloc(ctx, &K.small, (size_t)6 * (m + 2)))) return rc;
        if ((rc = hemo_alloc(ctx, &K.partial, (size_t)FG_BLOCKS * (m + 2)))) return rc;
        if ((rc = hemo_alloc(ctx, &K.state, (size_t)64))) return rc;
        if (!K.state_host) HEMO_CHECK_CUDA(ctx, cudaMallocHost((void**)&K.state_host, 64 * sizeof(double)));
        HEMO_CHECK_CUDA(ctx, cudaMemsetAsync(K.state, 0, 64 * sizeof(double), ctx->stream));
        K.m = m; K.ldv = ldv;
        ctx->kry_restart = m;
        if (K.iter_exec) { cudaGraphExecDestroy(K.iter_exec); K.iter_exec = nullptr; }
        K.iter_valid = false;
    }
    return 0;
}

void hemo_krylov_free(hemo_ctx* ctx) {
    HemoKrylov& K = ctx->kry;
    cudaFree(K.H); cudaFree(K.small); cudaFree(K.partial); cudaFree(K.state);
    if (K.state_host) cudaFreeHost(K.state_host);
    if (K.iter_exec) cudaGraphExecDestroy(K.iter_exec);
    K = HemoKrylov();
}

void hemo_krylov_invalidate(hemo_ctx* ctx) {
    HemoKrylov& K = ctx->kry;
    if (K.iter_exec) { cudaGraphExecDestroy(K.iter_exec); K.iter_exec = nullptr; }
    K.iter_valid = false;
}

struct FgPtrs {
    FgState* st;
    double *H, *cs, *sn, *g, *ycoef, *hcol, *scale, *normsq;
    int* kout;
};

static FgPtrs fg_ptrs(hemo_ctx* ctx) {
    HemoKrylov& K = ctx->kry;
    const int m = K.m;
    FgPtrs p;
    p.st = reinterpret_cast<FgState*>(K.state);
    p.normsq = K.state + 16;
    p.kout = reinterpret_cast<int*>(K.state + 24);
    p.H = K.H;
    p.cs = K.small;
    p.sn = K.small + (m + 2);
    p.g = K.small + 2 * (m + 2);
    p.ycoef = K.small + 3 * (m + 2);
    p.hcol = K.small + 4 * (m + 2);
    p.scale = K.small + 5 * (m + 2);
    return p;
}

// one FGMRES iteration enqueued on the stream (identical arguments for every j)
static int fg_iteration_body(hemo_ctx* ctx, const double* vals_dev) {
    HemoKrylov& K = ctx->kry;
    const FgPtrs p = fg_ptrs(ctx);
    const int n = ctx->n, m = K.m;
    const int64_t N = (int64_t)(ctx->dim + 1) * n, ldv = K.ldv;
    cudaStream_t st = ctx->stream;
    const FgSeg seg = {K.seg_len0 ? K.seg_len0 : N, K.seg_off1, K.seg_len0 ? K.seg_len1 : 0};
    int rc;
    HEMO_LAUNCH(ctx, k_fg_load, fg_grid(N, 4), FG_THREADS, 0, st, p.st, N, ctx->kry_V, ldv, p.scale, ctx->pc_in);
    if (ctx->comm && ctx->comm_ras_overlap && (rc = hemo_comm_halo(ctx, ctx->pc_in))) return rc;
    HEMO_PROF_BEGIN(ctx, HEMO_PROF_PC);
    if ((rc = hemo_pc_apply_body(ctx, vals_dev, ctx->pc_in, ctx->pc_out))) return rc;
    HEMO_PROF_END(ctx, HEMO_PROF_PC);
    if (ctx->comm && (rc = hemo_comm_halo(ctx, ctx->pc_out))) return rc;
    HEMO_PROF_BEGIN(ctx, HEMO_PROF_SPMV);
    if (ctx->dim == 3) {
        if ((rc = hemo_tet_spmv(ctx, vals_dev, ctx->pc_out, ctx->kry_w))) return rc;
        HEMO_LAUNCH(ctx, k_fg_store, fg_grid(N, 4), FG_THREADS, 0, st, p.st, N, ctx->pc_out, ctx->kry_w, ctx->kry_V, ctx->kry_Z,
                    ldv);
    } else {
        HEMO_LAUNCH(ctx, k_fg_spmv_node, hemo_grid((int64_t)n * 8, 256), 256, 0, st, p.st, n, ctx->nnz_node, ctx->nrowptr,
                    ctx->ncol, vals_dev, ctx->pc_out, ctx->kry_V, ctx->kry_Z, ldv);
    }
    HEMO_PROF_END(ctx, HEMO_PROF_SPMV);
    const int64_t nown = seg.len0 + seg.len1;
    HEMO_PROF_BEGIN(ctx, HEMO_PROF_MDOT);
    {
        const int kpad = m + 4;
        const int gm = fg_grid(nown, FG_TILE);
        const size_t smem = sizeof(double) * (FG_THREADS / 32) * kpad;
        if (seg.len1 > 0) HEMO_LAUNCH(ctx, k_fg_mdot<true>, gm, FG_THREADS, smem, st, p.st, seg, ctx->kry_V, ldv, K.partial, kpad);
        else HEMO_LAUNCH(ctx, k_fg_mdot<false>, gm, FG_THREADS, smem, st, p.st, seg, ctx->kry_V, ldv, K.partial, kpad);
        HEMO_LAUNCH(ctx, k_fg_mdot_final, m, 128, 0, st, p.st, gm, K.partial, p.scale, p.hcol);
    }
    HEMO_PROF_END(ctx, HEMO_PROF_MDOT);
    if (ctx->comm && (rc = hemo_comm_allreduce_j(ctx, p.hcol, m + 1))) return rc;
    HEMO_PROF_BEGIN(ctx, HEMO_PROF_MAXPY);
    HEMO_LAUNCH(ctx, k_fg_maxpy, fg_grid(N, 1), FG_THREADS, sizeof(double) * 3 * (m + 2), st, p.st, seg, N, ctx->kry_V, ldv,
                p.hcol, m, K.partial, p.normsq, ctx->comm ? 0 : 1, p.H, p.cs, p.sn, p.g, p.scale);
    HEMO_PROF_END(ctx, HEMO_PROF_MAXPY);
    if (ctx->comm) {
        if ((rc = hemo_comm_allreduce_j(ctx, p.normsq, 1))) return rc;
        HEMO_LAUNCH(ctx, k_fg_givens, 1, 64, sizeof(double) * 3 * (m + 2), st, p.st, m, p.hcol, p.normsq, p.H, p.cs, p.sn, p.g,
                    p.scale);
    }
    return 0;
}

// kernel nodes and programmatic-dependency edges of a captured graph
static void fg_graph_stats(cudaGraph_t g, int64_t* kernels, int64_t* prog) {
    *kernels = *prog = 0;
    size_t nn = 0, ne = 0;
    if (cudaGraphGetNodes(g, nullptr, &nn) != cudaSuccess || cudaGraphGetEdges_v2(g, nullptr, nullptr, nullptr, &ne) != cudaSuccess) {
        cudaGetLastError();
        return;
    }
    std::vector<cudaGraphNode_t> nodes(nn), from(ne), to(ne);
    std::vector<cudaGraphEdgeData> data(ne);
    if (cudaGraphGetNodes(g, nodes.data(), &nn) != cudaSuccess ||
        cudaGraphGetEdges_v2(g, from.data(), to.data(), data.data(), &ne) != cudaSuccess) {
        cudaGetLastError();
        return;
    }
    for (cudaGraphNode_t v : nodes) {
        cudaGraphNodeType t;
        if (cudaGraphNodeGetType(v, &t) == cudaSuccess && t == cudaGraphNodeTypeKernel) ++*kernels;
    }
    for (const cudaGraphEdgeData& d : data)
        if (d.type == cudaGraphDependencyTypeProgrammatic) ++*prog;
}

// The iteration replays as one CUDA graph (captured once per preconditioner set-up: the kernel arguments do not
// depend on j).  Needs a non-default stream; otherwise, or with profiling events on, direct launches.
static int fg_iteration(hemo_ctx* ctx, const double* vals_dev) {
    HemoKrylov& K = ctx->kry;
    const bool graph_ok = ctx->use_graph && ctx->stream != 0 && !ctx->prof.on;
    if (!graph_ok) return fg_iteration_body(ctx, vals_dev);
    if (K.iter_valid && K.iter_exec && K.iter_vals == vals_dev) {
        HEMO_CHECK_CUDA(ctx, cudaGraphLaunch(K.iter_exec, ctx->stream));
        ctx->launches += K.iter_nodes;
        return 0;
    }
    cudaStream_t st = ctx->stream;
    const int64_t before = ctx->launches;
    ctx->capturing = true;
    if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
        ctx->capturing = false;
        cudaGetLastError();
        return fg_iteration_body(ctx, vals_dev);
    }
    int rc = fg_iteration_body(ctx, vals_dev);
    cudaGraph_t g = nullptr;
    cudaError_t e = cudaStreamEndCapture(st, &g);
    ctx->capturing = false;
    K.iter_nodes = ctx->launches - before;
    ctx->launches = before;
    if (rc != 0 || e != cudaSuccess || !g) {
        cudaGetLastError();
        if (g) cudaGraphDestroy(g);
        if (rc) return rc;
        ctx->use_graph = 0;
        return fg_iteration_body(ctx, vals_dev);
    }
    fg_graph_stats(g, &K.iter_kernel_nodes, &K.iter_prog_edges);
    bool updated = false;
    if (K.iter_exec) {
        cudaGraphExecUpdateResultInfo info;
        if (cudaGraphExecUpdate(K.iter_exec, g, &info) == cudaSuccess) updated = true;
        else { cudaGetLastError(); cudaGraphExecDestroy(K.iter_exec); K.iter_exec = nullptr; }
    }
    if (!updated) {
        e = cudaGraphInstantiate(&K.iter_exec, g, 0);
        if (e != cudaSuccess) { cudaGraphDestroy(g); HEMO_CHECK_CUDA(ctx, e); }
    }
    cudaGraphDestroy(g);
    K.iter_valid = true;
    K.iter_vals = vals_dev;
    HEMO_CHECK_CUDA(ctx, cudaGraphLaunch(K.iter_exec, st));
    ctx->launches += K.iter_nodes;
    return 0;
}

extern "C" int hemo_krylov_graph_info(hemo_ctx* ctx, int64_t* kernel_nodes, int64_t* programmatic_edges) {
    if (!ctx || !kernel_nodes || !programmatic_edges) return HEMO_EINVAL;
    if (!ctx->kry.iter_valid) HEMO_FAIL(ctx, HEMO_ESTATE, "no FGMRES iteration graph has been captured");
    *kernel_nodes = ctx->kry.iter_kernel_nodes;
    *programmatic_edges = ctx->kry.iter_prog_edges;
    return 0;
}

static int fg_poll(hemo_ctx* ctx, FgState* out) {
    HemoKrylov& K = ctx->kry;
    HEMO_CHECK_CUDA(ctx, cudaMemcpyAsync(K.state_host, K.state, sizeof(FgState), cudaMemcpyDeviceToHost, ctx->stream));
    HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *out = *reinterpret_cast<FgState*>(K.state_host);
    K.polls++;
    return 0;
}

extern "C" int hemo_set_poll_interval(hemo_ctx* ctx, int every) {
    if (!ctx || every < 1) return HEMO_EINVAL;
    ctx->kry.poll_every = every;
    return 0;
}

extern "C" int hemo_fgmres(hemo_ctx* ctx, const double* vals_dev, const double* b_dev, double* y_dev, int* its_out,
                           double* rel_resid_out) {
    if (!ctx || !vals_dev || !b_dev || !y_dev) return HEMO_EINVAL;
    if (!ctx->mass || !ctx->pc_tmp_u) HEMO_FAIL(ctx, HEMO_ESTATE, "hemo_pc_setup not called");
    const int n = ctx->n;
    const int64_t N = (int64_t)(ctx->dim + 1) * n;
    const int64_t ldv = (N + 31) / 32 * 32;
    const int m = ctx->opts.restart;
    cudaStream_t st = ctx->stream;
    int rc;
    if ((rc = fg_ensure(ctx, m, ldv))) return rc;
    HemoKrylov& K = ctx->kry;
    const FgPtrs p = fg_ptrs(ctx);
    const FgSeg seg = {K.seg_len0 ? K.seg_len0 : N, K.seg_off1, K.seg_len0 ? K.seg_len1 : 0};
    const int64_t nown = seg.len0 + seg.len1;
    HEMO_CHECK_CUDA(ctx, cudaMemsetAsync(y_dev, 0, sizeof(double) * N, st));
    k_fg_start<<<fg_grid(N, 4), FG_THREADS, 0, st>>>(p.st, seg, N, b_dev, ctx->kry_V, K.partial, p.normsq, 1);
    HEMO_LAUNCH_CHECK(ctx);
    if (ctx->comm && (rc = hemo_comm_allreduce_j(ctx, p.normsq, 1))) return rc;
    k_fg_begin_cycle<<<1, 32, 0, st>>>(p.st, p.normsq, 1, ctx->opts.rtol, ctx->opts.atol, p.g, p.scale, m);
    HEMO_LAUNCH_CHECK(ctx);

    FgState hs;
    memset(&hs, 0, sizeof hs);
    int queued = 0;                 // iterations enqueued in total
    // the iteration count of the previous solve tells when to look at the state for the first time
    int next_poll = K.last_its > 2 ? K.last_its - 1 : 1;
    bool done = false;
    while (!done) {
        int jc = 0;                 // iterations enqueued in this cycle
        while (jc < m && queued < ctx->opts.max_it) {
            if ((rc = fg_iteration(ctx, vals_dev))) return rc;
            ++jc; ++queued;
            if (queued >= next_poll) {
                if ((rc = fg_poll(ctx, &hs))) return rc;
                if (hs.converged) { done = true; break; }
                next_poll = queued + (K.poll_every > 0 ? K.poll_every : 1);
            }
        }
        // y += Z_k (H_k^-1 g_k) with k = columns completed in this cycle (device value)
        k_fg_backsolve<<<1, 32, 0, st>>>(p.st, m, p.H, p.g, p.ycoef, p.kout);
        HEMO_LAUNCH_CHECK(ctx);
        k_fg_update<<<fg_grid(N, 1), FG_THREADS, sizeof(double) * (m + 2), st>>>(p.kout, N, ctx->kry_Z, ldv, p.ycoef, y_dev);
        HEMO_LAUNCH_CHECK(ctx);
        if (done) break;
        if ((rc = fg_poll(ctx, &hs))) return rc;
        if (hs.converged || queued >= ctx->opts.max_it) break;
        // restart: r = b - A y
        if (ctx->comm && (rc = hemo_comm_halo(ctx, y_dev))) return rc;
        if ((rc = hemo_spmv(ctx, vals_dev, y_dev, ctx->kry_w))) return rc;
        k_fg_residual<<<fg_grid(N, 4), FG_THREADS, 0, st>>>(p.st, N, b_dev, ctx->kry_w, ctx->kry_w);
        HEMO_LAUNCH_CHECK(ctx);
        k_fg_start<<<fg_grid(N, 4), FG_THREADS, 0, st>>>(p.st, seg, N, ctx->kry_w, ctx->kry_V, K.partial, p.normsq, 0);
        HEMO_LAUNCH_CHECK(ctx);
        if (ctx->comm && (rc = hemo_comm_allreduce_j(ctx, p.normsq, 1))) return rc;
        k_fg_begin_cycle<<<1, 32, 0, st>>>(p.st, p.normsq, 0, ctx->opts.rtol, ctx->opts.atol, p.g, p.scale, m);
        HEMO_LAUNCH_CHECK(ctx);
    }
    if (!done && (rc = fg_poll(ctx, &hs))) return rc;
    if (ctx->comm && (rc = hemo_comm_halo(ctx, y_dev))) return rc;
    K.last_its = hs.its;
    if (its_out) *its_out = hs.its;
    if (rel_resid_out) *rel_resid_out = hs.bnorm > 0.0 ? hs.res / hs.bnorm : 0.0;
    if (hs.converged < 0) HEMO_FAIL(ctx, HEMO_DIVERGED, "FGMRES residual is not finite");
    if (!hs.converged) HEMO_FAIL(ctx, HEMO_DIVERGED, "FGMRES reached max_it without converging");
    return 0;
}
