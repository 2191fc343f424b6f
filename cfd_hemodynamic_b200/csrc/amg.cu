// Aggregation-AMG V-cycle on node-block CSR operators (bs = 2: velocity block
// A00, bs = 1: pressure Laplacian of the Schur-complement approximation).
//
// Replaces, by design with a different algorithm, the PETSc sub-solvers
// `gmres + asm/ilu(0)` on A00 and `preonly + asm/ilu(0)` on Sp configured at
// reference src/solvers/stabilized_schur.py:256-267 (ILU triangular solves are
// sequential; a multigrid cycle is all SpMV-shaped, HBM-bound work).
//
// The prolongators (aggregates, optional Jacobi smoothing) depend only on the
// mesh graph and are built once by the host; what runs here every Newton
// iteration is the numeric Galerkin product R*A*P on fixed patterns, the
// smoother set-up, and the cycles.
#include <type_traits>
#include <cub/device/device_scan.cuh>

#include "hemo_internal.cuh"

int hemo_bsr_spmv_ex(hemo_ctx* ctx, int bs, int n, const int32_t* rowptr, const int32_t* col, const areal* val,
                     const areal* x, double alpha, const areal* b, areal* y);

// ---------------------------------------------------------------------------
// Numeric Galerkin product through precomputed gather lists: one thread per
// output block, contributions summed in a fixed order, no searches at run time.
// The lists are built once on the device.
// ---------------------------------------------------------------------------
__device__ __forceinline__ int find_col(const int32_t* __restrict__ col, int lo, int hi, int key) {
    // binary search in col[lo, hi)
    int a = lo, b = hi - 1;
    while (a <= b) {
        const int m = (a + b) >> 1;
        const int c = col[m];
        if (c == key) return m;
        if (c < key) a = m + 1; else b = m - 1;
    }
    return -1;
}

// count / fill pass over "rows x inner entries x outer entries":
//   AP:  row i,  t in A-row(i),  u in P-row(a_col[t])  -> slot of p_col[u] in AP-row(i);  src = (u, t)
//   RAP: row I,  t in R-row(I),  u in AP-row(r_col[t]) -> slot of ap_col[u] in C-row(I);  src = (t, u)
template <bool FILL, bool SWAP>
__global__ void k_product_lists(int nrows, const int32_t* __restrict__ a_rowptr, const int32_t* __restrict__ a_col,
                                const int32_t* __restrict__ b_rowptr, const int32_t* __restrict__ b_col,
                                const int32_t* __restrict__ o_rowptr, const int32_t* __restrict__ o_col,
                                int32_t* __restrict__ count, const int32_t* __restrict__ seg_ptr,
                                int2* __restrict__ seg_src, int* __restrict__ bad) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nrows) return;
    const int o0 = o_rowptr[i], o1 = o_rowptr[i + 1];
    for (int t = a_rowptr[i]; t < a_rowptr[i + 1]; ++t) {
        const int j = a_col[t];
        for (int u = b_rowptr[j]; u < b_rowptr[j + 1]; ++u) {
            const int pos = find_col(o_col, o0, o1, b_col[u]);
            if (pos < 0) { atomicExch(bad, 1); continue; }
            const int k = atomicAdd(&count[pos], 1);
            if (FILL) seg_src[seg_ptr[pos] + k] = SWAP ? make_int2(u, t) : make_int2(t, u);
        }
    }
}

__global__ void k_sort_pairs(int64_t nseg, const int32_t* __restrict__ ptr, int2* __restrict__ src) {
    const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= nseg) return;
    const int b0 = ptr[s], b1 = ptr[s + 1];
    for (int i = b0 + 1; i < b1; ++i) {
        const int2 key = src[i];
        int j = i - 1;
        while (j >= b0 && (src[j].y > key.y || (src[j].y == key.y && src[j].x > key.x))) { src[j + 1] = src[j]; --j; }
        src[j + 1] = key;
    }
}

template <int BS>
__global__ void __launch_bounds__(256)
k_gather_product(int64_t nseg, const int32_t* __restrict__ seg_ptr, const int2* __restrict__ seg_src,
                 const double* __restrict__ w, const areal* __restrict__ blk, areal* __restrict__ out) {
    const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= nseg) return;
    double acc[BS * BS];
#pragma unroll
    for (int k = 0; k < BS * BS; ++k) acc[k] = 0.0;
    const int b1 = seg_ptr[s + 1];
    for (int q = seg_ptr[s]; q < b1; ++q) {
        const int2 src = seg_src[q];
        const double wt = w[src.x];
        if (BS == 2) {
            const areal2 v0 = reinterpret_cast<const areal2*>(blk)[2 * (int64_t)src.y];
            const areal2 v1 = reinterpret_cast<const areal2*>(blk)[2 * (int64_t)src.y + 1];
            acc[0] = fma(wt, (double)v0.x, acc[0]); acc[1] = fma(wt, (double)v0.y, acc[1]);
            acc[BS * BS - 2] = fma(wt, (double)v1.x, acc[BS * BS - 2]);
            acc[BS * BS - 1] = fma(wt, (double)v1.y, acc[BS * BS - 1]);
        } else {
            acc[0] = fma(wt, (double)blk[src.y], acc[0]);
        }
    }
    if (BS == 2) {
        areal2 o0, o1;
        o0.x = (areal)acc[0]; o0.y = (areal)acc[1];
        o1.x = (areal)acc[BS * BS - 2]; o1.y = (areal)acc[BS * BS - 1];
        reinterpret_cast<areal2*>(out)[2 * s] = o0;
        reinterpret_cast<areal2*>(out)[2 * s + 1] = o1;
    } else {
        out[s] = (areal)acc[0];
    }
}

static int build_one_list(hemo_ctx* ctx, bool swap, int nrows, const int32_t* a_rowptr, const int32_t* a_col,
                          const int32_t* b_rowptr, const int32_t* b_col, const int32_t* o_rowptr, const int32_t* o_col,
                          int64_t nseg, int32_t** seg_ptr, int2** seg_src) {
    cudaStream_t st = ctx->stream;
    int rc;
    int32_t* count = nullptr;
    int* bad = nullptr;
    if ((rc = hemo_alloc(ctx, &count, (size_t)nseg + 1))) return rc;
    if ((rc = hemo_alloc(ctx, &bad, 1))) return rc;
    if ((rc = hemo_alloc(ctx, seg_ptr, (size_t)nseg + 1))) return rc;
    HEMO_CHECK_CUDA(ctx, cudaMemsetAsync(count, 0, sizeof(int32_t) * (nseg + 1), st));
    HEMO_CHECK_CUDA(ctx, cudaMemsetAsync(bad, 0, sizeof(int), st));
    const int g = hemo_grid(nrows, 128);
    if (swap) k_product_lists<false, true><<<g, 128, 0, st>>>(nrows, a_rowptr, a_col, b_rowptr, b_col, o_rowptr, o_col, count, nullptr, nullptr, bad);
    else k_product_lists<false, false><<<g, 128, 0, st>>>(nrows, a_rowptr, a_col, b_rowptr, b_col, o_rowptr, o_col, count, nullptr, nullptr, bad);
    HEMO_LAUNCH_CHECK(ctx);
    void* tmp = nullptr;
    size_t tmp_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, count, *seg_ptr, (int)(nseg + 1), st);
    HEMO_CHECK_CUDA(ctx, cudaMalloc(&tmp, tmp_bytes));
    HEMO_CHECK_CUDA(ctx, cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, count, *seg_ptr, (int)(nseg + 1), st));
    int32_t total = 0;
    HEMO_CHECK_CUDA(ctx, cudaMemcpyAsync(&total, *seg_ptr + nseg, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(st));
    cudaFree(tmp);
    if (total < 0) { cudaFree(count); cudaFree(bad); HEMO_FAIL(ctx, HEMO_EINVAL, "Galerkin gather list exceeds int32"); }
    if ((rc = hemo_alloc(ctx, seg_src, (size_t)total))) return rc;
    HEMO_CHECK_CUDA(ctx, cudaMemsetAsync(count, 0, sizeof(int32_t) * (nseg + 1), st));
    if (swap) k_product_lists<true, true><<<g, 128, 0, st>>>(nrows, a_rowptr, a_col, b_rowptr, b_col, o_rowptr, o_col, count, *seg_ptr, *seg_src, bad);
    else k_product_lists<true, false><<<g, 128, 0, st>>>(nrows, a_rowptr, a_col, b_rowptr, b_col, o_rowptr, o_col, count, *seg_ptr, *seg_src, bad);
    HEMO_LAUNCH_CHECK(ctx);
    k_sort_pairs<<<hemo_grid(nseg, 256), 256, 0, st>>>(nseg, *seg_ptr, *seg_src);
    HEMO_LAUNCH_CHECK(ctx);
    int bad_h = 0;
    HEMO_CHECK_CUDA(ctx, cudaMemcpyAsync(&bad_h, bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(st));
    cudaFree(count); cudaFree(bad);
    if (bad_h) HEMO_FAIL(ctx, HEMO_EINVAL, "AMG product pattern does not cover the product");
    return 0;
}

// inverse diagonal and Gershgorin bound of D^-1 A (per-block max)
template <int BS>
__global__ void __launch_bounds__(256)
k_diag_bound(int n, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
             const areal* __restrict__ val, areal* __restrict__ dinv, double* __restrict__ partial_max) {
    __shared__ double sh[256];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    double bound = 0.0;
    if (i < n) {
        double diag[BS], rs[BS];
#pragma unroll
        for (int k = 0; k < BS; ++k) { diag[k] = 0.0; rs[k] = 0.0; }
        for (int t = rowptr[i]; t < rowptr[i + 1]; ++t) {
            const int j = col[t];
#pragma unroll
            for (int k = 0; k < BS; ++k)
#pragma unroll
                for (int l = 0; l < BS; ++l) {
                    const double v = val[(int64_t)t * BS * BS + k * BS + l];
                    rs[k] += fabs(v);
                    if (j == i && k == l) diag[k] = v;
                }
        }
#pragma unroll
        for (int k = 0; k < BS; ++k) {
            const double d = (diag[k] != 0.0) ? diag[k] : 1.0;
            dinv[(int64_t)i * BS + k] = 1.0 / d;
            bound = fmax(bound, rs[k] / fabs(d));
        }
    }
    sh[threadIdx.x] = bound;
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) sh[threadIdx.x] = fmax(sh[threadIdx.x], sh[threadIdx.x + s]);
        __syncthreads();
    }
    if (threadIdx.x == 0) partial_max[blockIdx.x] = sh[0];
}

__global__ void k_max_final(int m, const double* __restrict__ partial, double* __restrict__ out) {
    __shared__ double sh[256];
    double v = 0.0;
    for (int i = threadIdx.x; i < m; i += blockDim.x) v = fmax(v, partial[i]);
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) sh[threadIdx.x] = fmax(sh[threadIdx.x], sh[threadIdx.x + s]);
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = sh[0];
}

__global__ void k_axpy_areal(int64_t n, double a, const areal* __restrict__ x, areal* __restrict__ y) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    hemo_pdl_wait();
    hemo_pdl_trigger();
    if (i < n) y[i] = (areal)fma(a, (double)x[i], (double)y[i]);
}

__global__ void k_to_areal(int64_t n, const double* __restrict__ x, areal* __restrict__ y) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    hemo_pdl_wait();
    hemo_pdl_trigger();
    if (i < n) y[i] = (areal)x[i];
}

__global__ void k_from_areal(int64_t n, const areal* __restrict__ x, double* __restrict__ y) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    hemo_pdl_wait();
    hemo_pdl_trigger();
    if (i < n) y[i] = (double)x[i];
}

// ---------------------------------------------------------------------------
// Chebyshev smoother on D^-1 A (fused SpMV + three-term update per step)
// ---------------------------------------------------------------------------
// start from x = 0:  r = D^-1 b ; d = r / theta ; x = d
template <int BS>
__global__ void k_cheb_start_zero(int64_t N, const areal* __restrict__ dinv, const areal* __restrict__ b,
                                  double inv_theta, areal* __restrict__ r, areal* __restrict__ d,
                                  areal* __restrict__ x) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    hemo_pdl_wait();
    hemo_pdl_trigger();
    if (i >= N) return;
    const double rv = dinv[i] * b[i];
    r[i] = rv;
    const double dv = rv * inv_theta;
    d[i] = dv;
    x[i] = dv;
}

// Column indices and blocks of the three strided entries a lane of a 4-lane row group handles per trip (entries beyond
// the row end: column of the first, zero block).  The operator is constant during a solve: the first trip's chunk is
// loaded before hemo_pdl_wait, so only the vector gathers wait for the predecessor.
template <int BS>
struct CsrChunk {
    int j0, j1, j2;
    areal2 a0, a1, a2, b0, b1, b2;   // BS == 2: the two rows of each 2x2 block
    areal v0, v1, v2;                // BS == 1
    __device__ __forceinline__ void load(const int32_t* __restrict__ col, const areal* __restrict__ val, int t, int r1) {
        const int t1 = t + 4, t2 = t + 8;
        const bool p1 = t1 < r1, p2 = t2 < r1;
        j0 = col[t];
        j1 = p1 ? col[t1] : j0;
        j2 = p2 ? col[t2] : j0;
        if (BS == 1) {
            v0 = val[t];
            v1 = p1 ? val[t1] : (areal)0;
            v2 = p2 ? val[t2] : (areal)0;
        } else {
            const areal2* v2p = reinterpret_cast<const areal2*>(val);
            a0 = v2p[2 * (int64_t)t]; b0 = v2p[2 * (int64_t)t + 1];
            a1.x = a1.y = b1.x = b1.y = a2.x = a2.y = b2.x = b2.y = 0;
            if (p1) { a1 = v2p[2 * (int64_t)t1]; b1 = v2p[2 * (int64_t)t1 + 1]; }
            if (p2) { a2 = v2p[2 * (int64_t)t2]; b2 = v2p[2 * (int64_t)t2 + 1]; }
        }
    }
};

// (A x)_i for block row i, computed by the 4 lanes of a row group; every lane
// of the group returns the full sum.  `ch` holds the lane's first chunk (when the row has one).
template <int BS>
__device__ __forceinline__ void row_product(const int32_t* __restrict__ col, const areal* __restrict__ val,
                                            const areal* __restrict__ x, int r0, int r1, int lane, CsrChunk<BS>& ch,
                                            double acc[BS]) {
#pragma unroll
    for (int k = 0; k < BS; ++k) acc[k] = 0.0;
    // The dependent chain col -> x is what bounds this kernel (rows are short): the column
    // loads of three strided entries are issued first, then the value / vector loads.
    for (int t = r0 + lane; t < r1; t += 12) {
        if (t != r0 + lane) ch.load(col, val, t, r1);
        if (BS == 1) {
            const double x0 = (double)x[ch.j0], x1 = (double)x[ch.j1], x2 = (double)x[ch.j2];
            acc[0] = fma((double)ch.v0, x0, acc[0]);
            acc[0] = fma((double)ch.v1, x1, acc[0]);
            acc[0] = fma((double)ch.v2, x2, acc[0]);
        } else {
            const areal2* x2p = reinterpret_cast<const areal2*>(x);
            const areal2 xa = x2p[ch.j0], xb = x2p[ch.j1], xc = x2p[ch.j2];
            const areal2 a0 = ch.a0, a1 = ch.a1, a2 = ch.a2, b0 = ch.b0, b1 = ch.b1, b2 = ch.b2;
            acc[0] += (double)a0.x * xa.x + (double)a0.y * xa.y + (double)a1.x * xb.x + (double)a1.y * xb.y +
                      (double)a2.x * xc.x + (double)a2.y * xc.y;
            acc[BS - 1] += (double)b0.x * xa.x + (double)b0.y * xa.y + (double)b1.x * xb.x + (double)b1.y * xb.y +
                           (double)b2.x * xc.x + (double)b2.y * xc.y;
        }
    }
#pragma unroll
    for (int k = 0; k < BS; ++k) {
        acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], 1, 4);
        acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], 2, 4);
    }
}

// start from x != 0: r = D^-1 (b - A x) ; d = r / theta   (4 lanes per block row).
// x is NOT updated here (other rows still read it); the update x += d is folded
// into the first k_cheb_step (add_old) or done by an axpy when degree == 1.
template <int BS>
__global__ void __launch_bounds__(256)
k_cheb_start(int n, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
             const areal* __restrict__ val, const areal* __restrict__ dinv, const areal* __restrict__ b,
             double inv_theta, const areal* __restrict__ xin, areal* __restrict__ r, areal* __restrict__ d) {
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = gt >> 2, lane = gt & 3;
    const bool ok = i < n;
    const int r0 = ok ? rowptr[i] : 0, r1 = ok ? rowptr[i + 1] : 0;
    CsrChunk<BS> ch;
    if (r0 + lane < r1) ch.load(col, val, r0 + lane, r1);
    hemo_pdl_wait();
    hemo_pdl_trigger();
    double acc[BS];
    row_product<BS>(col, val, xin, r0, r1, lane, ch, acc);
    if (ok && lane < BS) {
        const int64_t q = (int64_t)i * BS + lane;
        const double rv = dinv[q] * (b[q] - (lane == 0 ? acc[0] : acc[BS - 1]));
        r[q] = rv;
        d[q] = rv * inv_theta;
    }
}

// Pre-smoothing from a zero iterate with one Chebyshev step, fused with the residual that follows it:
//   x = D^-1 b / theta ;  r = b - A x
// x_j is formed on the fly from (dinv_j, b_j) inside the row product, so the separate start kernel and its round trip
// through x disappear (one launch less per level and cycle).  TB = double at the top level of the first cycle: the
// fp64 right-hand side is read directly and its storage-precision copy written as a by-product (no conversion kernel).
template <int BS, typename TB>
__global__ void __launch_bounds__(256)
k_presmooth_residual(int n, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                     const areal* __restrict__ val, const areal* __restrict__ dinv, const TB* __restrict__ b,
                     double inv_theta, areal* __restrict__ x, areal* __restrict__ r, areal* __restrict__ bcopy) {
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = gt >> 2, lane = gt & 3;
    const bool ok = i < n;
    const int r0 = ok ? rowptr[i] : 0, r1 = ok ? rowptr[i + 1] : 0;
    // columns, blocks and inverse diagonals of two strided entries per trip; the first trip's (constant during the solve)
    // are loaded before the wait, only the right-hand side gathers wait for the predecessor
    int j0 = 0, j1 = 0;
    areal2 a0, b0, a1, b1;    // BS == 2
    areal v0 = 0, v1 = 0;     // BS == 1
    areal d[2 * BS];
    auto fetch = [&](int t) {
        const int t1 = t + 4;
        const bool p1 = t1 < r1;
        j0 = col[t];
        j1 = p1 ? col[t1] : j0;
        if (BS == 1) {
            v0 = val[t];
            v1 = p1 ? val[t1] : (areal)0;
        } else {
            const areal2* v2p = reinterpret_cast<const areal2*>(val);
            a0 = v2p[2 * (int64_t)t]; b0 = v2p[2 * (int64_t)t + 1];
            a1.x = a1.y = b1.x = b1.y = 0;
            if (p1) { a1 = v2p[2 * (int64_t)t1]; b1 = v2p[2 * (int64_t)t1 + 1]; }
        }
#pragma unroll
        for (int k = 0; k < BS; ++k) {
            d[k] = dinv[(int64_t)j0 * BS + k];
            d[BS + k] = dinv[(int64_t)j1 * BS + k];
        }
    };
    if (r0 + lane < r1) fetch(r0 + lane);
    hemo_pdl_wait();
    hemo_pdl_trigger();
    double acc[BS];
#pragma unroll
    for (int k = 0; k < BS; ++k) acc[k] = 0.0;
    for (int t = r0 + lane; t < r1; t += 8) {
        if (t != r0 + lane) fetch(t);
        if (BS == 1) {
            const double x0 = (double)d[0] * (double)b[j0] * inv_theta;
            const double x1 = (double)d[BS] * (double)b[j1] * inv_theta;
            acc[0] = fma((double)v0, x0, acc[0]);
            acc[0] = fma((double)v1, x1, acc[0]);
        } else {
            const double xa0 = (double)d[0] * (double)b[2 * (int64_t)j0] * inv_theta;
            const double xa1 = (double)d[1] * (double)b[2 * (int64_t)j0 + 1] * inv_theta;
            const double xb0 = (double)d[BS] * (double)b[2 * (int64_t)j1] * inv_theta;
            const double xb1 = (double)d[BS + 1] * (double)b[2 * (int64_t)j1 + 1] * inv_theta;
            acc[0] += (double)a0.x * xa0 + (double)a0.y * xa1 + (double)a1.x * xb0 + (double)a1.y * xb1;
            acc[BS - 1] += (double)b0.x * xa0 + (double)b0.y * xa1 + (double)b1.x * xb0 + (double)b1.y * xb1;
        }
    }
#pragma unroll
    for (int k = 0; k < BS; ++k) {
        acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], 1, 4);
        acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], 2, 4);
    }
    if (ok && lane < BS) {
        const int64_t q = (int64_t)i * BS + lane;
        const double bv = (double)b[q];
        x[q] = (areal)((double)dinv[q] * bv * inv_theta);
        r[q] = (areal)(bv - (lane == 0 ? acc[0] : acc[BS - 1]));
        if (bcopy) bcopy[q] = (areal)bv;
    }
}

// one step: r -= D^-1 A d_old ; d_new = c1 d_old + c2 r ; x += d_new (+ d_old)
template <int BS>
__global__ void __launch_bounds__(256)
k_cheb_step(int n, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
            const areal* __restrict__ val, const areal* __restrict__ dinv, double c1, double c2,
            const areal* __restrict__ dold, areal* __restrict__ dnew, areal* __restrict__ r,
            areal* __restrict__ x, int add_old, double* __restrict__ x64 /* optional fp64 copy of the result */) {
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = gt >> 2, lane = gt & 3;
    const bool ok = i < n;
    const int r0 = ok ? rowptr[i] : 0, r1 = ok ? rowptr[i + 1] : 0;
    CsrChunk<BS> ch;
    if (r0 + lane < r1) ch.load(col, val, r0 + lane, r1);
    hemo_pdl_wait();
    hemo_pdl_trigger();
    double acc[BS];
    row_product<BS>(col, val, dold, r0, r1, lane, ch, acc);
    if (ok && lane < BS) {
        const int64_t q = (int64_t)i * BS + lane;
        const double rv = r[q] - dinv[q] * (lane == 0 ? acc[0] : acc[BS - 1]);
        r[q] = rv;
        const double dv = c1 * dold[q] + c2 * rv;
        dnew[q] = dv;
        const double xn = (double)x[q] + (add_old ? (dv + (double)dold[q]) : dv);
        x[q] = (areal)xn;
        if (x64) x64[q] = xn;
    }
}

// ---------------------------------------------------------------------------
// Sliced-ELL versions of the same kernels (HemoAmgOp::sell_*): ONE thread per block row.  The finest operators have
// 7-9 blocks per row; with 4 lanes per CSR row half the lanes idle in the second trip and every thread has two loads
// in flight (ncu: 33-47 % of DRAM peak).  Here a warp reads 32 consecutive column indices / blocks per trip (one
// 128 B / 512 B run) and every thread has its whole row in flight.
// ---------------------------------------------------------------------------
// Loads as volatile asm: the compiler keeps their program order, so the column indices, blocks and vector entries of
// four trips are requested back to back before the first use (left to itself nvcc interleaves load and use to save
// registers and the dependent chain col -> x is paid once per trip).  Non-coherent path: none of the arrays read this
// way is written by the kernel that reads it.
__device__ __forceinline__ int ldg_nc(const int32_t* p) {
    int v;
    asm volatile("ld.global.nc.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float ldg_nc(const float* p) {
    float v;
    asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ double ldg_nc(const double* p) {
    double v;
    asm volatile("ld.global.nc.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float2 ldg_nc(const float2* p) {
    float2 v;
    asm volatile("ld.global.nc.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ double2 ldg_nc(const double2* p) {
    double2 v;
    asm volatile("ld.global.nc.v2.f64 {%0,%1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ float4 ldg_nc(const float4* p) {
    float4 v;
    asm volatile("ld.global.nc.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ double4 ldg_nc(const double4* p) {
    double4 v;
    const double2 lo = ldg_nc(reinterpret_cast<const double2*>(p)), hi = ldg_nc(reinterpret_cast<const double2*>(p) + 1);
    v.x = lo.x; v.y = lo.y; v.z = hi.x; v.w = hi.y;
    return v;
}

// gathered vector entry of block column j (BS components, storage type)
template <int BS>
struct VecLoad {
    typedef typename std::conditional<BS == 1, areal, areal2>::type raw;
    const areal* __restrict__ x;
    __device__ __forceinline__ raw load(int j) const { return ldg_nc(reinterpret_cast<const raw*>(x) + j); }
    __device__ __forceinline__ void value(const raw& t, double* out) const {
        if constexpr (BS == 1) out[0] = (double)t;
        else { out[0] = (double)t.x; out[1] = (double)t.y; }
    }
};

// x_j = D_j^-1 b_j / theta formed on the fly (pre-smoothing from zero fused with the residual)
template <int BS, typename TB>
struct JacobiLoad {
    struct raw { areal d[BS]; TB b[BS]; };
    const areal* __restrict__ dinv;
    const TB* __restrict__ b;
    double inv_theta;
    __device__ __forceinline__ raw load(int j) const {
        raw t;
#pragma unroll
        for (int k = 0; k < BS; ++k) {
            t.d[k] = ldg_nc(dinv + (int64_t)j * BS + k);
            t.b[k] = ldg_nc(b + (int64_t)j * BS + k);
        }
        return t;
    }
    __device__ __forceinline__ void value(const raw& t, double* out) const {
#pragma unroll
        for (int k = 0; k < BS; ++k) out[k] = (double)t.d[k] * (double)t.b[k] * inv_theta;
    }
};

// Row i of a sliced-ELL operator, consumed four trips at a time.  begin() loads the slice bounds and, with GROUP, the
// column indices and blocks of the first four trips: the operator is constant during a solve, so a kernel issues them
// before hemo_pdl_wait and only the vector gathers of product() wait for the predecessor.  (The pre-smoothing kernels
// gather two vectors per entry and load nothing before the wait: holding the first group across it costs them
// occupancy.)
template <int BS>
struct SellRow {
    typedef typename std::conditional<BS == 1, areal, areal4>::type blk;
    const int32_t* __restrict__ c;
    const blk* __restrict__ v;
    int W;
    bool group;       // first group loaded by begin()
    int j[4];
    blk a[4];
    template <bool GROUP>
    __device__ __forceinline__ void begin(const int32_t* __restrict__ sptr, const int32_t* __restrict__ scol,
                                          const areal* __restrict__ sval, int i) {
        const int s = i >> 5, lane = i & 31;
        const int base = sptr[s];
        W = (sptr[s + 1] - base) >> 5;         // uniform over the warp
        c = scol + base + lane;
        v = reinterpret_cast<const blk*>(sval) + base + lane;
        group = GROUP;
        if (GROUP && W > 0) fetch(0);
    }
    // trips beyond the row end repeat the last one (product gives them a zero weight)
    __device__ __forceinline__ void fetch(int k) {
        int kk[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) kk[u] = 32 * (k + u < W ? k + u : W - 1);
#pragma unroll
        for (int u = 0; u < 4; ++u) j[u] = ldg_nc(c + kk[u]);
#pragma unroll
        for (int u = 0; u < 4; ++u) a[u] = ldg_nc(v + kk[u]);
    }
    template <typename XF>
    __device__ __forceinline__ void product(const XF xf, double acc[BS]) {
#pragma unroll
        for (int k = 0; k < BS; ++k) acc[k] = 0.0;
        for (int k = 0; k < W; k += 4) {
            bool ok[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) ok[u] = k + u < W;
            if (k > 0 || !group) fetch(k);
            typename XF::raw xr[4];
            __syncwarp();                    // scheduling fence: the eight loads above are in flight before the first use
#pragma unroll
            for (int u = 0; u < 4; ++u) xr[u] = xf.load(j[u]);
            __syncwarp();
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                double xv[BS];
                xf.value(xr[u], xv);
                if constexpr (BS == 1) {
                    acc[0] = fma(ok[u] ? (double)a[u] : 0.0, xv[0], acc[0]);
                } else {
                    const double m = ok[u] ? 1.0 : 0.0;
                    acc[0] += m * ((double)a[u].x * xv[0] + (double)a[u].y * xv[1]);
                    acc[1] += m * ((double)a[u].z * xv[0] + (double)a[u].w * xv[1]);
                }
            }
        }
    }
};

template <int BS>
__global__ void __launch_bounds__(256)
k_sell_cheb_start(int n, const int32_t* __restrict__ sptr, const int32_t* __restrict__ scol, const areal* __restrict__ sval,
                  const areal* __restrict__ dinv, const areal* __restrict__ b, double inv_theta,
                  const areal* __restrict__ xin, areal* __restrict__ r, areal* __restrict__ d) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    SellRow<BS> row;
    if (i < n) row.template begin<true>(sptr, scol, sval, i);
    hemo_pdl_wait();
    hemo_pdl_trigger();
    if (i >= n) return;
    double acc[BS];
    row.product(VecLoad<BS>{xin}, acc);
#pragma unroll
    for (int k = 0; k < BS; ++k) {
        const int64_t q = (int64_t)i * BS + k;
        const double rv = (double)dinv[q] * ((double)b[q] - acc[k]);
        r[q] = (areal)rv;
        d[q] = (areal)(rv * inv_theta);
    }
}

template <int BS, typename TB>
__global__ void __launch_bounds__(256)
k_sell_presmooth_residual(int n, const int32_t* __restrict__ sptr, const int32_t* __restrict__ scol,
                          const areal* __restrict__ sval, const areal* __restrict__ dinv, const TB* __restrict__ b,
                          double inv_theta, areal* __restrict__ x, areal* __restrict__ r, areal* __restrict__ bcopy) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    hemo_pdl_wait();
    hemo_pdl_trigger();
    if (i >= n) return;
    SellRow<BS> row;
    row.template begin<false>(sptr, scol, sval, i);
    double acc[BS];
    row.product(JacobiLoad<BS, TB>{dinv, b, inv_theta}, acc);
#pragma unroll
    for (int k = 0; k < BS; ++k) {
        const int64_t q = (int64_t)i * BS + k;
        const double bv = (double)b[q];
        x[q] = (areal)((double)dinv[q] * bv * inv_theta);
        r[q] = (areal)(bv - acc[k]);
        if (bcopy) bcopy[q] = (areal)bv;
    }
}

template <int BS>
__global__ void __launch_bounds__(256)
k_sell_cheb_step(int n, const int32_t* __restrict__ sptr, const int32_t* __restrict__ scol, const areal* __restrict__ sval,
                 const areal* __restrict__ dinv, double c1, double c2, const areal* __restrict__ dold,
                 areal* __restrict__ dnew, areal* __restrict__ r, areal* __restrict__ x, int add_old,
                 double* __restrict__ x64) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    SellRow<BS> row;
    if (i < n) row.template begin<true>(sptr, scol, sval, i);
    hemo_pdl_wait();
    hemo_pdl_trigger();
    if (i >= n) return;
    double acc[BS];
    row.product(VecLoad<BS>{dold}, acc);
#pragma unroll
    for (int k = 0; k < BS; ++k) {
        const int64_t q = (int64_t)i * BS + k;
        const double dq = (double)dold[q];
        const double rv = (double)r[q] - (double)dinv[q] * acc[k];
        r[q] = (areal)rv;
        const double dv = c1 * dq + c2 * rv;
        dnew[q] = (areal)dv;
        const double xn = (double)x[q] + (add_old ? (dv + dq) : dv);
        x[q] = (areal)xn;
        if (x64) x64[q] = xn;
    }
}

// y = b - A x
template <int BS>
__global__ void __launch_bounds__(256)
k_sell_residual(int n, const int32_t* __restrict__ sptr, const int32_t* __restrict__ scol, const areal* __restrict__ sval,
                const areal* __restrict__ x, const areal* __restrict__ b, areal* __restrict__ y) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    SellRow<BS> row;
    if (i < n) row.template begin<true>(sptr, scol, sval, i);
    hemo_pdl_wait();
    hemo_pdl_trigger();
    if (i >= n) return;
    double acc[BS];
    row.product(VecLoad<BS>{x}, acc);
#pragma unroll
    for (int k = 0; k < BS; ++k) {
        const int64_t q = (int64_t)i * BS + k;
        y[q] = (areal)((double)b[q] - acc[k]);
    }
}

// pattern of the sliced-ELL copy: one thread per (padded) row
__global__ void k_sell_fill_col(int n, int nrows_padded, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                const int32_t* __restrict__ sptr, int32_t* __restrict__ scol) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nrows_padded) return;
    const int s = i >> 5, lane = i & 31;
    const int base = sptr[s], W = (sptr[s + 1] - base) >> 5;
    const int r0 = i < n ? rowptr[i] : 0, deg = i < n ? rowptr[i + 1] - r0 : 0;
    const int self = i < n ? i : n - 1;
    for (int k = 0; k < W; ++k) scol[base + 32 * k + lane] = k < deg ? col[r0 + k] : self;
}

// values of the sliced-ELL copy from the CSR values (padding stays zero): 4 lanes per row
template <int BS>
__global__ void __launch_bounds__(256)
k_sell_fill_val(int n, const int32_t* __restrict__ rowptr, const areal* __restrict__ val,
                const int32_t* __restrict__ sptr, areal* __restrict__ sval) {
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = gt >> 2, sub = gt & 3;
    if (i >= n) return;
    const int base = sptr[i >> 5] + (i & 31);
    const int r0 = rowptr[i], deg = rowptr[i + 1] - r0;
    for (int k = sub; k < deg; k += 4) {
#pragma unroll
        for (int c = 0; c < BS * BS; ++c)
            sval[((int64_t)base + 32 * k) * (BS * BS) + c] = val[((int64_t)r0 + k) * (BS * BS) + c];
    }
}

// y[i] += sum_t w_t x[col_t]: prolongation rows are 1-4 entries long — one thread per row
template <int BS>
__global__ void __launch_bounds__(256)
k_prolong_add_row(int nrows, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                  const double* __restrict__ w, const areal* __restrict__ x, areal* __restrict__ y) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool ok = i < nrows;
    const int r0 = ok ? rowptr[i] : 0, r1 = ok ? rowptr[i + 1] : 0;
    int j = 0;
    double wt = 0.0;
    if (r0 < r1) { j = col[r0]; wt = w[r0]; }       // first entry (constant) before the wait
    hemo_pdl_wait();
    hemo_pdl_trigger();
    if (!ok) return;
    double acc[BS];
#pragma unroll
    for (int k = 0; k < BS; ++k) acc[k] = 0.0;
    for (int t = r0; t < r1; ++t) {
        if (t != r0) { j = col[t]; wt = w[t]; }
#pragma unroll
        for (int k = 0; k < BS; ++k) acc[k] = fma(wt, (double)x[(int64_t)j * BS + k], acc[k]);
    }
#pragma unroll
    for (int k = 0; k < BS; ++k) {
        const int64_t q = (int64_t)i * BS + k;
        y[q] = (areal)((double)y[q] + acc[k]);
    }
}

// y[I] (+)= sum_t w_t x[col_t]  with bs components per node (restriction / prolongation);
// 4 lanes per row, column loads of three strided entries issued first
template <int BS, bool ADD>
__global__ void __launch_bounds__(256)
k_transfer(int nrows, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
           const double* __restrict__ w, const areal* __restrict__ x, areal* __restrict__ y) {
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;
    const int I = gt >> 2, lane = gt & 3;
    const bool ok = I < nrows;
    const int r0 = ok ? rowptr[I] : 0, r1 = ok ? rowptr[I + 1] : 0;
    // the first trip's columns and weights (constant) before the wait
    int j0 = 0, j1 = 0, j2 = 0;
    double w0 = 0.0, w1 = 0.0, w2 = 0.0;
    auto fetch = [&](int t) {
        const int t1 = t + 4, t2 = t + 8;
        const bool p1 = t1 < r1, p2 = t2 < r1;
        j0 = col[t];
        j1 = p1 ? col[t1] : j0;
        j2 = p2 ? col[t2] : j0;
        w0 = w[t]; w1 = p1 ? w[t1] : 0.0; w2 = p2 ? w[t2] : 0.0;
    };
    if (r0 + lane < r1) fetch(r0 + lane);
    hemo_pdl_wait();
    hemo_pdl_trigger();
    double acc[BS];
#pragma unroll
    for (int k = 0; k < BS; ++k) acc[k] = 0.0;
    for (int t = r0 + lane; t < r1; t += 12) {
        if (t != r0 + lane) fetch(t);
#pragma unroll
        for (int k = 0; k < BS; ++k) {
            const double x0 = (double)x[(int64_t)j0 * BS + k], x1 = (double)x[(int64_t)j1 * BS + k],
                         x2 = (double)x[(int64_t)j2 * BS + k];
            acc[k] += w0 * x0 + w1 * x1 + w2 * x2;
        }
    }
#pragma unroll
    for (int k = 0; k < BS; ++k) {
        acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], 1, 4);
        acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], 2, 4);
    }
    if (ok && lane < BS) {
        const double v = (lane == 0) ? acc[0] : acc[BS - 1];
        const int64_t q = (int64_t)I * BS + lane;
        if (ADD) y[q] = (areal)((double)y[q] + v);
        else y[q] = (areal)v;
    }
}

// ---------------------------------------------------------------------------
// fused coarse V-cycle: every level from `fuse_level` down (at most HEMO_FUSE_MAX_NODES nodes each) runs inside ONE
// CTA, phases separated by __syncthreads, replacing ~7 launches per level.
// ---------------------------------------------------------------------------
// Row loops: 8 lanes cooperate on one block row (coarse Galerkin rows hold 20-60 blocks; a thread-serial
// walk makes every phase a ~50-deep dependent load chain).  All lanes of a warp execute the same number of
// outer iterations, so full-mask shuffles are legal.
template <int BS, typename Epi>
__device__ __forceinline__ void rows_matvec(const HemoCoarseLevel& L, const areal* __restrict__ x, Epi epi) {
    const int lane = threadIdx.x & 7, group = threadIdx.x >> 3, ngroups = blockDim.x >> 3;
    for (int base = 0; base < L.n; base += ngroups) {
        const int i = base + group;
        const bool ok = i < L.n;
        double acc[BS];
#pragma unroll
        for (int k = 0; k < BS; ++k) acc[k] = 0.0;
        if (ok) {
            const int r1 = L.rowptr[i + 1];
            for (int t = L.rowptr[i] + lane; t < r1; t += 8) {
                const int j = L.col[t];
#pragma unroll
                for (int k = 0; k < BS; ++k)
#pragma unroll
                    for (int l = 0; l < BS; ++l)
                        acc[k] = fma((double)L.val[(int64_t)t * BS * BS + k * BS + l], (double)x[(int64_t)j * BS + l], acc[k]);
            }
        }
#pragma unroll
        for (int k = 0; k < BS; ++k) {
            acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], 1, 8);
            acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], 2, 8);
            acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], 4, 8);
        }
        if (ok && lane == 0) epi(i, acc);
    }
}

// y-rows of a transfer operator (CSR with fp64 weights) applied to a BS-component vector
template <int BS, typename Epi>
__device__ __forceinline__ void rows_transfer(int nrows, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                              const double* __restrict__ w, const areal* __restrict__ x, Epi epi) {
    const int lane = threadIdx.x & 7, group = threadIdx.x >> 3, ngroups = blockDim.x >> 3;
    for (int base = 0; base < nrows; base += ngroups) {
        const int i = base + group;
        const bool ok = i < nrows;
        double acc[BS];
#pragma unroll
        for (int k = 0; k < BS; ++k) acc[k] = 0.0;
        if (ok) {
            const int r1 = rowptr[i + 1];
            for (int t = rowptr[i] + lane; t < r1; t += 8) {
                const int j = col[t];
                const double wt = w[t];
#pragma unroll
                for (int k = 0; k < BS; ++k) acc[k] = fma(wt, (double)x[(int64_t)j * BS + k], acc[k]);
            }
        }
#pragma unroll
        for (int k = 0; k < BS; ++k) {
            acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], 1, 8);
            acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], 2, 8);
            acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], 4, 8);
        }
        if (ok && lane == 0) epi(i, acc);
    }
}

template <int BS>
__device__ void fused_smooth(const HemoCoarseLevel& L, const areal* __restrict__ b, areal* __restrict__ x, bool x_is_zero,
                             int degree, double ratio) {
    const int tid = threadIdx.x, T = blockDim.x;
    const int N = L.n * BS;
    const double lmax = *L.lmax, lmin = lmax / ratio;
    const double theta = 0.5 * (lmax + lmin), delta = 0.5 * (lmax - lmin), sigma = theta / delta;
    double rho = 1.0 / sigma;
    areal* dold = L.d0;
    areal* dnew = L.d1;
    if (x_is_zero) {
        for (int q = tid; q < N; q += T) {
            const double rv = (double)L.dinv[q] * (double)b[q];
            L.r[q] = (areal)rv;
            dold[q] = (areal)(rv / theta);
            x[q] = (areal)(rv / theta);
        }
    } else {
        rows_matvec<BS>(L, x, [&](int i, const double* acc) {
#pragma unroll
            for (int k = 0; k < BS; ++k) {
                const int q = i * BS + k;
                const double rv = (double)L.dinv[q] * ((double)b[q] - acc[k]);
                L.r[q] = (areal)rv;
                dold[q] = (areal)(rv / theta);
            }
        });
    }
    __syncthreads();
    bool pending = !x_is_zero;
    for (int s = 1; s < degree; ++s) {
        const double rho_new = 1.0 / (2.0 * sigma - rho);
        const double c1 = rho_new * rho, c2 = 2.0 * rho_new / delta;
        const areal* dcur = dold;
        areal* dnext = dnew;
        const bool add_old = pending;
        rows_matvec<BS>(L, dcur, [&](int i, const double* acc) {
#pragma unroll
            for (int k = 0; k < BS; ++k) {
                const int q = i * BS + k;
                const double rv = (double)L.r[q] - (double)L.dinv[q] * acc[k];
                L.r[q] = (areal)rv;
                const double dv = c1 * (double)dcur[q] + c2 * rv;
                dnext[q] = (areal)dv;
                x[q] = (areal)((double)x[q] + (add_old ? (dv + (double)dcur[q]) : dv));
            }
        });
        __syncthreads();
        pending = false;
        areal* t = dold; dold = dnew; dnew = t;
        rho = rho_new;
    }
    if (pending) {
        for (int q = tid; q < N; q += T) x[q] = (areal)((double)x[q] + (double)dold[q]);
        __syncthreads();
    }
}

template <int BS>
__global__ void __launch_bounds__(1024)
k_coarse_vcycle(const HemoCoarseLevel* __restrict__ desc, int nl, const areal* __restrict__ b0, areal* __restrict__ x0,
                int x0_is_zero, int degree, double ratio, const double* __restrict__ dense_inv, int dense_n) {
    hemo_pdl_wait();
    hemo_pdl_trigger();
    const int tid = threadIdx.x, T = blockDim.x;
    // down sweep
    for (int l = 0; l < nl - 1; ++l) {
        const HemoCoarseLevel L = desc[l];
        const areal* b = (l == 0) ? b0 : L.b;
        areal* x = (l == 0) ? x0 : L.x;
        // every level pre-smooths with the full Chebyshev degree; the top level of a second or later cycle smooths its
        // previous iterate, every coarser level starts from zero
        fused_smooth<BS>(L, b, x, l > 0 || x0_is_zero, degree, ratio);
        rows_matvec<BS>(L, x, [&](int i, const double* acc) {
#pragma unroll
            for (int k = 0; k < BS; ++k) L.r[i * BS + k] = (areal)((double)b[i * BS + k] - acc[k]);
        });
        __syncthreads();
        areal* bc = desc[l + 1].b;
        rows_transfer<BS>(L.nc, L.r_rowptr, L.r_col, L.r_val, L.r, [&](int I, const double* acc) {
#pragma unroll
            for (int k = 0; k < BS; ++k) bc[I * BS + k] = (areal)acc[k];
        });
        __syncthreads();
    }
    // coarsest: dense inverse, 8 lanes per row
    {
        const areal* b = (nl == 1) ? b0 : desc[nl - 1].b;
        areal* x = (nl == 1) ? x0 : desc[nl - 1].x;
        const int lane = tid & 7, group = tid >> 3, ngroups = T >> 3;
        for (int base = 0; base < dense_n; base += ngroups) {
            const int row = base + group;
            const bool ok = row < dense_n;
            double acc = 0.0;
            if (ok)
                for (int c = lane; c < dense_n; c += 8) acc = fma(dense_inv[(int64_t)row * dense_n + c], (double)b[c], acc);
            acc += __shfl_xor_sync(0xffffffffu, acc, 1, 8);
            acc += __shfl_xor_sync(0xffffffffu, acc, 2, 8);
            acc += __shfl_xor_sync(0xffffffffu, acc, 4, 8);
            if (ok && lane == 0) x[row] = (areal)acc;
        }
        __syncthreads();
    }
    // up sweep
    for (int l = nl - 2; l >= 0; --l) {
        const HemoCoarseLevel L = desc[l];
        const areal* b = (l == 0) ? b0 : L.b;
        areal* x = (l == 0) ? x0 : L.x;
        const areal* xc = desc[l + 1].x;
        rows_transfer<BS>(L.n, L.p_rowptr, L.p_col, L.p_val, xc, [&](int i, const double* acc) {
#pragma unroll
            for (int k = 0; k < BS; ++k) x[i * BS + k] = (areal)((double)x[i * BS + k] + acc[k]);
        });
        __syncthreads();
        fused_smooth<BS>(L, b, x, false, degree, ratio);
    }
}

// ---------------------------------------------------------------------------
// dense inverse of the coarsest level (applied by k_coarse_vcycle): Gauss–Jordan,
// one CTA (N <= HEMO_DENSE_MAX)
// ---------------------------------------------------------------------------
template <int BS>
__global__ void k_dense_fill(int n, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                             const areal* __restrict__ val, int N, double shift_rel, double* __restrict__ M /*N x N*/) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int t = rowptr[i]; t < rowptr[i + 1]; ++t) {
        const int j = col[t];
#pragma unroll
        for (int k = 0; k < BS; ++k)
#pragma unroll
            for (int l = 0; l < BS; ++l) {
                double v = val[(int64_t)t * BS * BS + k * BS + l];
                // optional relative diagonal shift (singular Neumann operator)
                if (i == j && k == l) v *= (1.0 + shift_rel);
                M[(int64_t)(i * BS + k) * N + (j * BS + l)] = v;
            }
    }
}

// In-place Gauss–Jordan inversion of an N x N matrix held in shared memory by
// one CTA (N <= HEMO_DENSE_MAX).  No pivoting: the coarsest Galerkin operators
// are (shifted) M-matrix-like / diagonally dominated; a vanishing pivot sets *fail.
__global__ void __launch_bounds__(1024)
k_dense_invert(int N, const double* __restrict__ Min, double* __restrict__ inv, int* __restrict__ fail) {
    extern __shared__ double A[];          // N*N
    __shared__ double fcol[HEMO_DENSE_MAX];
    __shared__ double pivinv;
    const int tid = threadIdx.x;
    const int total = N * N;
    for (int q = tid; q < total; q += blockDim.x) A[q] = Min[q];
    __syncthreads();
    for (int p = 0; p < N; ++p) {
        if (tid == 0) {
            const double piv = A[p * N + p];
            if (!(fabs(piv) > 0.0) || !isfinite(piv)) *fail = 1;
            pivinv = 1.0 / piv;
            A[p * N + p] = 1.0;
        }
        __syncthreads();
        const double pi = pivinv;
        for (int c = tid; c < N; c += blockDim.x) A[p * N + c] *= pi;
        for (int r = tid; r < N; r += blockDim.x) {
            if (r != p) { fcol[r] = A[r * N + p]; A[r * N + p] = 0.0; }
            else fcol[r] = 0.0;
        }
        __syncthreads();
        for (int q = tid; q < total; q += blockDim.x) {
            const int r = q / N;
            const int c = q - r * N;
            const double f = fcol[r];
            if (f != 0.0) A[q] -= f * A[p * N + c];
        }
        __syncthreads();
    }
    for (int q = tid; q < total; q += blockDim.x) inv[q] = A[q];
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
static void free_level(HemoAmgLevel& L) {
    cudaFree(L.p_rowptr); cudaFree(L.p_col); cudaFree(L.p_val);
    cudaFree(L.r_rowptr); cudaFree(L.r_col); cudaFree(L.r_val);
    cudaFree(L.ap_rowptr); cudaFree(L.ap_col); cudaFree(L.ap_val);
    cudaFree(L.c_rowptr); cudaFree(L.c_col);
    cudaFree(L.ap_seg_ptr); cudaFree(L.ap_seg_src); cudaFree(L.c_seg_ptr); cudaFree(L.c_seg_src);
    L = HemoAmgLevel();
}

void hemo_amg_free(HemoAmg* amg) {
    for (int l = 0; l < HEMO_MAX_LEVELS; ++l) {
        free_level(amg->lev[l]);
        HemoAmgOp& o = amg->op[l];
        cudaFree(o.val); cudaFree(o.dinv); cudaFree(o.x); cudaFree(o.b); cudaFree(o.r); cudaFree(o.d);
        cudaFree(o.sell_ptr); cudaFree(o.sell_col); cudaFree(o.sell_val);
        o = HemoAmgOp();
    }
    if (amg->apply_exec) { cudaGraphExecDestroy(amg->apply_exec); amg->apply_exec = nullptr; }
    amg->apply_valid = false;
    cudaFree(amg->fine_rowptr); cudaFree(amg->fine_col); cudaFree(amg->fine_rowof);
    amg->fine_rowptr = amg->fine_col = amg->fine_rowof = nullptr; amg->fine_nnz = 0;
    cudaFree(amg->dense_inv); cudaFree(amg->dense_work); cudaFree(amg->fuse_desc); cudaFree(amg->lmax_dev);
    amg->fuse_desc = nullptr; amg->lmax_dev = nullptr; amg->fuse_level = -1;
    amg->dense_inv = amg->dense_work = nullptr;
    amg->nlev = 0;
    amg->ready = false;
}

extern "C" int hemo_amg_set_level(hemo_ctx* ctx, int which, int level, int n_fine, int n_coarse,
                                  const int32_t* p_rowptr, const int32_t* p_col, const double* p_val,
                                  const int32_t* r_rowptr, const int32_t* r_col, const double* r_val,
                                  const int32_t* ap_rowptr, const int32_t* ap_col,
                                  const int32_t* c_rowptr, const int32_t* c_col) {
    if (!ctx || which < 0 || which > 1 || level < 0 || level >= HEMO_MAX_LEVELS - 1) return HEMO_EINVAL;
    if (!p_rowptr || !p_col || !p_val || !r_rowptr || !r_col || !r_val || !ap_rowptr || !ap_col || !c_rowptr || !c_col)
        return HEMO_EINVAL;
    HemoAmg& amg = ctx->amg[which];
    amg.bs = (which == 0) ? 2 : 1;
    amg.ready = false;
    HemoAmgLevel& L = amg.lev[level];
    free_level(L);
    L.n_fine = n_fine; L.n_coarse = n_coarse;
    L.nnz_p = p_rowptr[n_fine];
    L.nnz_ap = ap_rowptr[n_fine];
    L.nnz_c = c_rowptr[n_coarse];
    if (r_rowptr[n_coarse] != L.nnz_p) HEMO_FAIL(ctx, HEMO_EINVAL, "R is not the transpose pattern of P");
    int rc;
    if ((rc = hemo_upload(ctx, &L.p_rowptr, p_rowptr, (size_t)n_fine + 1, false))) return rc;
    if ((rc = hemo_upload(ctx, &L.p_col, p_col, (size_t)L.nnz_p, false))) return rc;
    if ((rc = hemo_upload(ctx, &L.p_val, p_val, (size_t)L.nnz_p, false))) return rc;
    if ((rc = hemo_upload(ctx, &L.r_rowptr, r_rowptr, (size_t)n_coarse + 1, false))) return rc;
    if ((rc = hemo_upload(ctx, &L.r_col, r_col, (size_t)L.nnz_p, false))) return rc;
    if ((rc = hemo_upload(ctx, &L.r_val, r_val, (size_t)L.nnz_p, false))) return rc;
    if ((rc = hemo_upload(ctx, &L.ap_rowptr, ap_rowptr, (size_t)n_fine + 1, false))) return rc;
    if ((rc = hemo_upload(ctx, &L.ap_col, ap_col, (size_t)L.nnz_ap, false))) return rc;
    if ((rc = hemo_upload(ctx, &L.c_rowptr, c_rowptr, (size_t)n_coarse + 1, false))) return rc;
    if ((rc = hemo_upload(ctx, &L.c_col, c_col, (size_t)L.nnz_c, false))) return rc;
    if ((rc = hemo_alloc(ctx, &L.ap_val, (size_t)L.nnz_ap * amg.bs * amg.bs))) return rc;
    // host arrays may be released by the caller as soon as we return
    HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

__global__ void k_rowof_generic(int n, const int32_t* __restrict__ rowptr, int32_t* __restrict__ rowof) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int s = rowptr[i]; s < rowptr[i + 1]; ++s) rowof[s] = i;
}

extern "C" int hemo_amg_set_fine_pattern(hemo_ctx* ctx, int which, const int32_t* rowptr_host, const int32_t* col_host) {
    if (!ctx || which < 0 || which > 1) return HEMO_EINVAL;
    if (!ctx->nrowptr) HEMO_FAIL(ctx, HEMO_ESTATE, "node graph not set");
    HemoAmg& amg = ctx->amg[which];
    cudaFree(amg.fine_rowptr); cudaFree(amg.fine_col); cudaFree(amg.fine_rowof);
    amg.fine_rowptr = amg.fine_col = amg.fine_rowof = nullptr;
    amg.fine_nnz = 0;
    amg.ready = false;
    if (!rowptr_host || !col_host) return 0;
    const int n = ctx->n;
    const int64_t nnz = rowptr_host[n];
    int rc;
    if ((rc = hemo_upload(ctx, &amg.fine_rowptr, rowptr_host, (size_t)n + 1, false))) return rc;
    if ((rc = hemo_upload(ctx, &amg.fine_col, col_host, (size_t)nnz, false))) return rc;
    if ((rc = hemo_alloc(ctx, &amg.fine_rowof, (size_t)nnz))) return rc;
    k_rowof_generic<<<hemo_grid(n, 256), 256, 0, ctx->stream>>>(n, amg.fine_rowptr, amg.fine_rowof);
    HEMO_LAUNCH_CHECK(ctx);
    HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    amg.fine_nnz = nnz;
    return 0;
}

// sliced-ELL pattern of one operator (kept when the padding stays below half of the entries)
static int build_sell(hemo_ctx* ctx, HemoAmgOp& o, int bs) {
    cudaFree(o.sell_ptr); cudaFree(o.sell_col); cudaFree(o.sell_val);
    o.sell_ptr = o.sell_col = nullptr; o.sell_val = nullptr; o.sell_entries = 0;
    const char* env = getenv("HEMO_SELL");
    if (env && atoi(env) == 0) return 0;
    const int n = o.n;
    // long rows / small levels: thread-serial rows lose against 4 lanes per row (measured: 10-11 us against 5.5-6 us
    // per kernel at 9.6 k nodes with ~25 blocks per row)
    if (n < 32768 || o.nnzb > 24 * (int64_t)n) return 0;
    std::vector<int32_t> rp((size_t)n + 1);
    HEMO_CHECK_CUDA(ctx, cudaMemcpy(rp.data(), o.rowptr, sizeof(int32_t) * ((size_t)n + 1), cudaMemcpyDeviceToHost));
    const int nsl = (n + 31) / 32;
    std::vector<int32_t> sp((size_t)nsl + 1);
    int64_t total = 0;
    sp[0] = 0;
    for (int s = 0; s < nsl; ++s) {
        int w = 0;
        const int hi = std::min(n, 32 * s + 32);
        for (int i = 32 * s; i < hi; ++i) w = std::max(w, rp[i + 1] - rp[i]);
        total += 32 * (int64_t)w;
        if (total > 0x7fffffffLL) return 0;
        sp[s + 1] = (int32_t)total;
    }
    if (total > o.nnzb + o.nnzb / 2) return 0;
    int rc;
    if ((rc = hemo_upload(ctx, &o.sell_ptr, sp.data(), (size_t)nsl + 1, false))) return rc;
    if ((rc = hemo_alloc(ctx, &o.sell_col, (size_t)total))) return rc;
    if ((rc = hemo_alloc(ctx, &o.sell_val, (size_t)total * bs * bs))) return rc;
    HEMO_CHECK_CUDA(ctx, cudaMemsetAsync(o.sell_val, 0, sizeof(areal) * (size_t)total * bs * bs, ctx->stream));
    k_sell_fill_col<<<hemo_grid((int64_t)nsl * 32, 256), 256, 0, ctx->stream>>>(n, nsl * 32, o.rowptr, o.col, o.sell_ptr, o.sell_col);
    HEMO_LAUNCH_CHECK(ctx);
    HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    o.sell_entries = total;
    return 0;
}

extern "C" int hemo_amg_finalize(hemo_ctx* ctx, int which, int n_levels) {
    if (!ctx || which < 0 || which > 1 || n_levels < 1 || n_levels > HEMO_MAX_LEVELS) return HEMO_EINVAL;
    if (!ctx->nrowptr) HEMO_FAIL(ctx, HEMO_ESTATE, "node graph not set");
    HemoAmg& amg = ctx->amg[which];
    amg.bs = (which == 0) ? 2 : 1;
    const int bs = amg.bs;
    amg.nlev = n_levels;
    int rc;
    for (int l = 0; l < n_levels; ++l) {
        HemoAmgOp& o = amg.op[l];
        if (l == 0) {
            o.n = ctx->n; o.nnzb = ctx->nnz_node; o.rowptr = ctx->nrowptr; o.col = ctx->ncol;
            if (amg.fine_rowptr) { o.nnzb = amg.fine_nnz; o.rowptr = amg.fine_rowptr; o.col = amg.fine_col; }
        } else {
            const HemoAmgLevel& L = amg.lev[l - 1];
            if (L.n_coarse <= 0) HEMO_FAIL(ctx, HEMO_ESTATE, "missing AMG level");
            if (l == 1 ? (L.n_fine != ctx->n) : (L.n_fine != amg.lev[l - 2].n_coarse))
                HEMO_FAIL(ctx, HEMO_EINVAL, "AMG level sizes do not chain");
            o.n = L.n_coarse; o.nnzb = L.nnz_c; o.rowptr = L.c_rowptr; o.col = L.c_col;
        }
        if ((rc = hemo_alloc(ctx, &o.val, (size_t)o.nnzb * bs * bs))) return rc;
        if ((rc = hemo_alloc(ctx, &o.dinv, (size_t)o.n * bs))) return rc;
        if ((rc = hemo_alloc(ctx, &o.x, (size_t)o.n * bs))) return rc;
        if ((rc = hemo_alloc(ctx, &o.b, (size_t)o.n * bs))) return rc;
        if ((rc = hemo_alloc(ctx, &o.r, (size_t)o.n * bs))) return rc;
        if ((rc = hemo_alloc(ctx, &o.d, (size_t)o.n * bs * 2))) return rc;   // ping-pong
    }
    const int Nc = amg.op[n_levels - 1].n * bs;
    if (Nc > HEMO_DENSE_MAX) HEMO_FAIL(ctx, HEMO_EINVAL, "coarsest AMG level too large for the dense solve");
    amg.dense_n = Nc;
    if ((rc = hemo_alloc(ctx, &amg.dense_inv, (size_t)Nc * Nc))) return rc;
    if ((rc = hemo_alloc(ctx, &amg.dense_work, (size_t)Nc * Nc + 8))) return rc;
    if ((rc = hemo_ensure_reduce(ctx, (size_t)hemo_grid(ctx->n, 256) + 1184 * 8, 512))) return rc;
    if ((rc = hemo_alloc(ctx, &amg.lmax_dev, (size_t)HEMO_MAX_LEVELS))) return rc;
    {
        // hierarchies are re-formed for every new Jacobian: precompute their gather lists
        for (int l = 0; l + 1 < n_levels; ++l) {
            HemoAmgLevel& L = amg.lev[l];
            const HemoAmgOp& A = amg.op[l];
            if ((rc = build_one_list(ctx, true, A.n, A.rowptr, A.col, L.p_rowptr, L.p_col, L.ap_rowptr, L.ap_col,
                                     L.nnz_ap, &L.ap_seg_ptr, &L.ap_seg_src))) return rc;
            if ((rc = build_one_list(ctx, false, L.n_coarse, L.r_rowptr, L.r_col, L.ap_rowptr, L.ap_col, L.c_rowptr,
                                     L.c_col, L.nnz_c, &L.c_seg_ptr, &L.c_seg_src))) return rc;
        }
    }
    // every level from `fuse_level` down runs inside the one-CTA kernel; the coarsest level always does, as it holds at
    // most HEMO_DENSE_MAX dofs
    static_assert(HEMO_DENSE_MAX <= HEMO_FUSE_MAX_NODES, "the coarsest level must fit the one-CTA kernel");
    amg.fuse_level = -1;
    for (int l = 0; l < n_levels; ++l)
        if (amg.op[l].n <= HEMO_FUSE_MAX_NODES) { amg.fuse_level = l; break; }
    // the levels that keep per-level kernels get the sliced-ELL copy
    for (int l = 0; l < amg.fuse_level; ++l)
        if ((rc = build_sell(ctx, amg.op[l], bs))) return rc;
    std::vector<HemoCoarseLevel> d;
    for (int l = amg.fuse_level; l < n_levels; ++l) {
        const HemoAmgOp& o = amg.op[l];
        HemoCoarseLevel c{};
        c.n = o.n; c.rowptr = o.rowptr; c.col = o.col; c.val = o.val; c.dinv = o.dinv;
        c.x = o.x; c.b = o.b; c.r = o.r; c.d0 = o.d; c.d1 = o.d + (size_t)o.n * bs;
        c.lmax = amg.lmax_dev + l;
        if (l + 1 < n_levels) {
            const HemoAmgLevel& L = amg.lev[l];
            c.nc = L.n_coarse;
            c.p_rowptr = L.p_rowptr; c.p_col = L.p_col; c.p_val = L.p_val;
            c.r_rowptr = L.r_rowptr; c.r_col = L.r_col; c.r_val = L.r_val;
        }
        d.push_back(c);
    }
    if ((rc = hemo_alloc(ctx, &amg.fuse_desc, d.size()))) return rc;
    HEMO_CHECK_CUDA(ctx, cudaMemcpyAsync(amg.fuse_desc, d.data(), sizeof(HemoCoarseLevel) * d.size(), cudaMemcpyHostToDevice,
                                         ctx->stream));
    HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    amg.ready = true;
    return 0;
}

template <int BS>
static int amg_numeric_t(hemo_ctx* ctx, HemoAmg* amg, double coarse_shift) {
    cudaStream_t st = ctx->stream;
#define HEMO_FILL_SELL(A)                                                                                                  \
    if ((A).sell_ptr) {                                                                                                    \
        k_sell_fill_val<BS><<<hemo_grid((int64_t)(A).n * 4, 256), 256, 0, st>>>((A).n, (A).rowptr, (A).val, (A).sell_ptr,   \
                                                                                 (A).sell_val);                            \
        HEMO_LAUNCH_CHECK(ctx);                                                                                            \
    }
    HEMO_FILL_SELL(amg->op[0]);
    for (int l = 0; l + 1 < amg->nlev; ++l) {
        const HemoAmgOp& A = amg->op[l];
        HemoAmgOp& C = amg->op[l + 1];
        const HemoAmgLevel& L = amg->lev[l];
        if (l == 0) HEMO_PROF_BEGIN(ctx, HEMO_PROF_RAP);
        k_gather_product<BS><<<hemo_grid(L.nnz_ap, 256), 256, 0, st>>>(L.nnz_ap, L.ap_seg_ptr, L.ap_seg_src, L.p_val, A.val,
                                                                        L.ap_val);
        HEMO_LAUNCH_CHECK(ctx);
        k_gather_product<BS><<<hemo_grid(L.nnz_c, 256), 256, 0, st>>>(L.nnz_c, L.c_seg_ptr, L.c_seg_src, L.r_val, L.ap_val,
                                                                       C.val);
        HEMO_LAUNCH_CHECK(ctx);
        if (l == 0) HEMO_PROF_END(ctx, HEMO_PROF_RAP);
        HEMO_FILL_SELL(C);
    }
#undef HEMO_FILL_SELL
    // smoother data; bounds are read back in one copy
    for (int l = 0; l + 1 < amg->nlev; ++l) {
        HemoAmgOp& A = amg->op[l];
        const int g = hemo_grid(A.n, 256);
        k_diag_bound<BS><<<g, 256, 0, st>>>(A.n, A.rowptr, A.col, A.val, A.dinv, ctx->red_partial);
        HEMO_LAUNCH_CHECK(ctx);
        k_max_final<<<1, 256, 0, st>>>(g, ctx->red_partial, amg->lmax_dev + l);
        HEMO_LAUNCH_CHECK(ctx);
    }
    if (amg->nlev > 1) {
        HEMO_CHECK_CUDA(ctx, cudaMemcpyAsync(ctx->red_host + 64, amg->lmax_dev, sizeof(double) * (amg->nlev - 1),
                                             cudaMemcpyDeviceToHost, st));
    }
    // dense inverse of the coarsest operator
    {
        const HemoAmgOp& A = amg->op[amg->nlev - 1];
        const int N = amg->dense_n;
        int* fail = reinterpret_cast<int*>(amg->dense_work + (size_t)N * N);
        HEMO_CHECK_CUDA(ctx, cudaMemsetAsync(amg->dense_work, 0, sizeof(double) * ((size_t)N * N + 8), st));
        k_dense_fill<BS><<<hemo_grid(A.n, 128), 128, 0, st>>>(A.n, A.rowptr, A.col, A.val, N, coarse_shift, amg->dense_work);
        HEMO_LAUNCH_CHECK(ctx);
        const size_t smem = sizeof(double) * (size_t)N * N;
        HEMO_CHECK_CUDA(ctx, cudaFuncSetAttribute(k_dense_invert, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_dense_invert<<<1, 1024, smem, st>>>(N, amg->dense_work, amg->dense_inv, fail);
        HEMO_LAUNCH_CHECK(ctx);
        int fail_h = 0;
        HEMO_CHECK_CUDA(ctx, cudaMemcpyAsync(&fail_h, fail, sizeof(int), cudaMemcpyDeviceToHost, st));
        HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(st));
        if (fail_h) HEMO_FAIL(ctx, HEMO_DIVERGED, "coarsest AMG operator is singular");
    }
    for (int l = 0; l + 1 < amg->nlev; ++l) {
        double b = ctx->red_host[64 + l];
        if (!(b > 0.0) || !isfinite(b)) HEMO_FAIL(ctx, HEMO_DIVERGED, "AMG operator has a non-finite Gershgorin bound");
        amg->op[l].lmax = b;
    }
    return 0;
}

// coarse_shift is carried in amg via dense_n sign-free field; passed explicitly by the caller
int hemo_amg_numeric_shift(hemo_ctx* ctx, HemoAmg* amg, double coarse_shift) {
    if (!amg->ready) HEMO_FAIL(ctx, HEMO_ESTATE, "AMG hierarchy not finalized");
    amg->apply_valid = false;      // smoother coefficients are baked into a captured cycle
    if (amg->bs == 2) return amg_numeric_t<2>(ctx, amg, coarse_shift);
    return amg_numeric_t<1>(ctx, amg, coarse_shift);
}

int hemo_amg_numeric(hemo_ctx* ctx, HemoAmg* amg) { return hemo_amg_numeric_shift(ctx, amg, 0.0); }

template <int BS>
static int smooth_t(hemo_ctx* ctx, const HemoAmgOp& A, const areal* b, areal* x, bool x_is_zero, int degree,
                    double ratio, double* x64 = nullptr, bool* wrote64 = nullptr) {
    cudaStream_t st = ctx->stream;
    const double lmax = A.lmax, lmin = lmax / ratio;
    const double theta = 0.5 * (lmax + lmin), delta = 0.5 * (lmax - lmin);
    const double sigma = theta / delta;
    double rho = 1.0 / sigma;
    const int64_t N = (int64_t)A.n * BS;
    areal* d0 = A.d;
    areal* d1 = A.d + N;
    if (x_is_zero) {
        HEMO_LAUNCH(ctx, k_cheb_start_zero<BS>, hemo_grid(N, 256), 256, 0, st, N, A.dinv, b, 1.0 / theta, A.r, d0, x);
    } else if (A.sell_ptr) {
        HEMO_LAUNCH(ctx, k_sell_cheb_start<BS>, hemo_grid(A.n, 256), 256, 0, st, A.n, A.sell_ptr, A.sell_col, A.sell_val, A.dinv, b,
                    1.0 / theta, x, A.r, d0);
    } else {
        HEMO_LAUNCH(ctx, k_cheb_start<BS>, hemo_grid((int64_t)A.n * 4, 256), 256, 0, st, A.n, A.rowptr, A.col, A.val, A.dinv, b,
                    1.0 / theta, x, A.r, d0);
    }
    bool pending = !x_is_zero;   // x += d0 still to be applied
    for (int k = 1; k < degree; ++k) {
        const double rho_new = 1.0 / (2.0 * sigma - rho);
        const double c1 = rho_new * rho, c2 = 2.0 * rho_new / delta;
        const bool fine = (A.n == ctx->n);
        if (fine) HEMO_PROF_BEGIN(ctx, BS == 2 ? HEMO_PROF_CHEB_U0 : HEMO_PROF_CHEB_P0);
        const bool last = (k == degree - 1);
        if (A.sell_ptr)
            HEMO_LAUNCH(ctx, k_sell_cheb_step<BS>, hemo_grid(A.n, 256), 256, 0, st, A.n, A.sell_ptr, A.sell_col, A.sell_val, A.dinv, c1,
                        c2, d0, d1, A.r, x, pending ? 1 : 0, last ? x64 : nullptr);
        else
            HEMO_LAUNCH(ctx, k_cheb_step<BS>, hemo_grid((int64_t)A.n * 4, 256), 256, 0, st, A.n, A.rowptr, A.col, A.val, A.dinv, c1, c2,
                        d0, d1, A.r, x, pending ? 1 : 0, last ? x64 : nullptr);
        if (last && x64 && wrote64) *wrote64 = true;
        if (fine) HEMO_PROF_END(ctx, BS == 2 ? HEMO_PROF_CHEB_U0 : HEMO_PROF_CHEB_P0);
        pending = false;
        areal* t = d0; d0 = d1; d1 = t;
        rho = rho_new;
    }
    if (pending) HEMO_LAUNCH(ctx, k_axpy_areal, hemo_grid(N, 256), 256, 0, st, N, 1.0, d0, x);
    return 0;
}

template <int BS>
static int vcycle_t(hemo_ctx* ctx, HemoAmg* amg, int l, const areal* b, areal* x, bool x_is_zero,
                    const double* b64 = nullptr, double* x64 = nullptr, bool* wrote64 = nullptr) {
    cudaStream_t st = ctx->stream;
    const HemoAmgOp& A = amg->op[l];
    const int degree = ctx->opts.cheb_degree > 0 ? ctx->opts.cheb_degree : 2;
    const int degree_pre = ctx->opts.cheb_degree_pre > 0 ? ctx->opts.cheb_degree_pre : degree;
    const double ratio = ctx->opts.cheb_ratio > 1.0 ? ctx->opts.cheb_ratio : 4.0;
    if (l == amg->fuse_level) {
        // every remaining level fits one CTA
        HEMO_LAUNCH(ctx, k_coarse_vcycle<BS>, 1, 1024, 0, st, amg->fuse_desc, amg->nlev - l, b, x, x_is_zero ? 1 : 0, degree, ratio,
                    amg->dense_inv, amg->dense_n);
        return 0;
    }
    int rc;
    if (x_is_zero && degree_pre == 1) {
        // one Chebyshev step from zero + residual in one kernel
        const double lmax = A.lmax, lmin = lmax / ratio;
        const double inv_theta = 1.0 / (0.5 * (lmax + lmin));
        const int g = hemo_grid((int64_t)A.n * 4, 256);
        areal* const no_copy = nullptr;
        if (A.sell_ptr) {
            const int gs = hemo_grid(A.n, 256);
            if (b64) HEMO_LAUNCH(ctx, (k_sell_presmooth_residual<BS, double>), gs, 256, 0, st, A.n, A.sell_ptr, A.sell_col, A.sell_val,
                                 A.dinv, b64, inv_theta, x, A.r, const_cast<areal*>(b));
            else HEMO_LAUNCH(ctx, (k_sell_presmooth_residual<BS, areal>), gs, 256, 0, st, A.n, A.sell_ptr, A.sell_col, A.sell_val, A.dinv,
                             b, inv_theta, x, A.r, no_copy);
        } else if (b64) HEMO_LAUNCH(ctx, (k_presmooth_residual<BS, double>), g, 256, 0, st, A.n, A.rowptr, A.col, A.val, A.dinv, b64,
                                    inv_theta, x, A.r, const_cast<areal*>(b));
        else HEMO_LAUNCH(ctx, (k_presmooth_residual<BS, areal>), g, 256, 0, st, A.n, A.rowptr, A.col, A.val, A.dinv, b, inv_theta, x,
                         A.r, no_copy);
    } else {
        if (b64) {          // the fused kernel is not used: convert the right-hand side first
            const int64_t N = (int64_t)A.n * BS;
            HEMO_LAUNCH(ctx, k_to_areal, hemo_grid(N, 256), 256, 0, st, N, b64, const_cast<areal*>(b));
        }
        if ((rc = smooth_t<BS>(ctx, A, b, x, x_is_zero, degree_pre, ratio))) return rc;
        // residual and restriction
        if (A.sell_ptr) {
            HEMO_LAUNCH(ctx, k_sell_residual<BS>, hemo_grid(A.n, 256), 256, 0, st, A.n, A.sell_ptr, A.sell_col, A.sell_val, x, b, A.r);
        } else if ((rc = hemo_bsr_spmv_ex(ctx, BS, A.n, A.rowptr, A.col, A.val, x, -1.0, b, A.r))) return rc;
    }
    const HemoAmgLevel& L = amg->lev[l];
    HemoAmgOp& C = amg->op[l + 1];
    HEMO_LAUNCH(ctx, (k_transfer<BS, false>), hemo_grid((int64_t)C.n * 4, 256), 256, 0, st, C.n, L.r_rowptr, L.r_col, L.r_val, A.r,
                C.b);
    if ((rc = vcycle_t<BS>(ctx, amg, l + 1, C.b, C.x, true))) return rc;
    if (L.nnz_p <= 6 * (int64_t)A.n && A.n >= 32768)
        HEMO_LAUNCH(ctx, k_prolong_add_row<BS>, hemo_grid(A.n, 256), 256, 0, st, A.n, L.p_rowptr, L.p_col, L.p_val, C.x, x);
    else
        HEMO_LAUNCH(ctx, (k_transfer<BS, true>), hemo_grid((int64_t)A.n * 4, 256), 256, 0, st, A.n, L.p_rowptr, L.p_col, L.p_val, C.x,
                    x);
    if ((rc = smooth_t<BS>(ctx, A, b, x, false, degree, ratio, x64, wrote64))) return rc;
    return 0;
}

// x = (ncycles V-cycles applied to A x = b, zero initial guess); fp64 in / out, the
// cycle itself runs on the hierarchy's storage type
int hemo_amg_vcycle(hemo_ctx* ctx, HemoAmg* amg, const double* b, double* x, int ncycles) {
    if (!amg->ready) HEMO_FAIL(ctx, HEMO_ESTATE, "AMG hierarchy not finalized");
    int rc;
    HemoAmgOp& top = amg->op[0];
    const int64_t N = (int64_t)top.n * amg->bs;
    const int nc = ncycles > 0 ? ncycles : 1;
    // the top level runs per-level kernels (it is not inside the fused kernel): its first kernel reads the fp64
    // right-hand side and its last one writes the fp64 result — no conversion kernels
    const bool per_level_top = amg->fuse_level > 0;
    if (!per_level_top) HEMO_LAUNCH(ctx, k_to_areal, hemo_grid(N, 256), 256, 0, ctx->stream, N, b, top.b);
    bool wrote64 = false;
    for (int c = 0; c < nc; ++c) {
        const double* b64 = (per_level_top && c == 0) ? b : nullptr;
        double* x64 = (per_level_top && c == nc - 1) ? x : nullptr;
        if (amg->bs == 2) rc = vcycle_t<2>(ctx, amg, 0, top.b, top.x, c == 0, b64, x64, &wrote64);
        else rc = vcycle_t<1>(ctx, amg, 0, top.b, top.x, c == 0, b64, x64, &wrote64);
        if (rc) return rc;
    }
    if (!wrote64) HEMO_LAUNCH(ctx, k_from_areal, hemo_grid(N, 256), 256, 0, ctx->stream, N, top.x, x);
    return 0;
}
