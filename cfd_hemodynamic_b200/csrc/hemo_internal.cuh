// Internal declarations shared by the translation units of libhemo_sm100.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/hemo.h"
#include "hemo_rules.h"

#define HEMO_MAXQ 80          // max cell quadrature points per rule (P2 needs 79)
#define HEMO_NRULES 6
#define HEMO_MAX_FACET_SETS 8
#define HEMO_MAX_LEVELS 16
#define HEMO_DENSE_MAX 160    // max dofs of the dense coarsest-level solve (N*N doubles in shared memory)

// Storage type of the multigrid hierarchies (operators, smoother data, cycle vectors).
// The preconditioner only has to be a good approximate inverse: single-precision storage
// halves its HBM traffic, accumulation stays in fp64 registers, and the outer FGMRES,
// the Jacobian, the residuals and every reduction remain fp64 (results are unchanged to the
// solver tolerance; -DHEMO_AMG_FP64 switches back).
#ifdef HEMO_AMG_FP64
typedef double areal;
typedef double2 areal2;
typedef double4 areal4;
#else
typedef float areal;
typedef float2 areal2;
typedef float4 areal4;
#endif

struct HemoRule {
    int nq;
    int alias;                // lowest block id with an identical rule
    double phi[HEMO_MAXQ][3];
    double w[HEMO_MAXQ];
    double m0, m1[3], m2[6];  // polynomial moments of the rule (reference cell)
};

struct HemoFacetSet {
    int m = 0;
    int32_t* cells = nullptr;
    int32_t* mask = nullptr;
    hemo_facet_coef coef{};
};

// One operator of a multigrid hierarchy in node-block CSR (BSR with bs x bs blocks).
struct HemoAmgOp {
    int n = 0;                 // nodes
    int64_t nnzb = 0;          // blocks
    const int32_t* rowptr = nullptr;
    const int32_t* col = nullptr;
    areal* val = nullptr;      // nnzb*bs*bs
    areal* dinv = nullptr;     // n*bs   inverse diagonal
    double lmax = 2.0;         // bound of spectrum of D^-1 A
    areal *x = nullptr, *b = nullptr, *r = nullptr, *d = nullptr;  // n*bs work vectors
    // Sliced-ELL copy of the operator for the smoother / residual kernels of the large levels: slices of 32 block rows,
    // entries of a slice stored column-major (entry k of lane's row at sell_ptr[slice] + 32 k + lane), padded to the
    // longest row of the slice with zero blocks.  One thread per row, every load of a warp is one contiguous run.
    int32_t* sell_ptr = nullptr;   // nslices + 1
    int32_t* sell_col = nullptr;
    areal* sell_val = nullptr;     // sell_entries*bs*bs
    int64_t sell_entries = 0;
};

struct HemoAmgLevel {
    int n_fine = 0, n_coarse = 0;
    int32_t *p_rowptr = nullptr, *p_col = nullptr; double* p_val = nullptr;
    int32_t *r_rowptr = nullptr, *r_col = nullptr; double* r_val = nullptr;
    int32_t *ap_rowptr = nullptr, *ap_col = nullptr; areal* ap_val = nullptr;
    int32_t *c_rowptr = nullptr, *c_col = nullptr;
    int64_t nnz_p = 0, nnz_ap = 0, nnz_c = 0;
    // precomputed gather lists of the numeric Galerkin product:
    // AP[s] = sum_k p_val[src.x] * A[src.y],  C[s] = sum_k r_val[src.x] * AP[src.y]
    int32_t* ap_seg_ptr = nullptr; int2* ap_seg_src = nullptr;
    int32_t* c_seg_ptr = nullptr;  int2* c_seg_src = nullptr;
};

// device-visible descriptor of one level for the fused coarse V-cycle kernel
struct HemoCoarseLevel {
    int n, nc;
    const int32_t *rowptr, *col;
    const areal *val, *dinv;
    areal *x, *b, *r, *d0, *d1;
    const int32_t *p_rowptr, *p_col; const double* p_val;
    const int32_t *r_rowptr, *r_col; const double* r_val;
    const double* lmax;
};

#define HEMO_FUSE_MAX_NODES 256    // levels at or below this size run inside one CTA (k_coarse_vcycle)

struct HemoAmg {
    // cached CUDA graph of hemo_amg_apply(b, x, ncycles) (replicated global pressure solve)
    cudaGraphExec_t apply_exec = nullptr;
    const double* apply_b = nullptr;
    double* apply_x = nullptr;
    int apply_cycles = 0;
    int64_t apply_nodes = 0;
    bool apply_valid = false;
    // optional level-0 pattern that differs from the mesh node graph (SELFP: distance-2 graph)
    int32_t *fine_rowptr = nullptr, *fine_col = nullptr, *fine_rowof = nullptr;
    int64_t fine_nnz = 0;
    int fuse_level = -1;           // first level handled by the one-CTA fused kernel (-1: not finalized)
    HemoCoarseLevel* fuse_desc = nullptr;   // device array, one per level from fuse_level
    double* lmax_dev = nullptr;    // HEMO_MAX_LEVELS Gershgorin bounds kept on the device
    int bs = 1;
    int nlev = 0;              // number of operators (levels); nlev-1 transfer levels
    bool ready = false;
    HemoAmgLevel lev[HEMO_MAX_LEVELS];
    HemoAmgOp op[HEMO_MAX_LEVELS];
    double* dense_inv = nullptr;   // (nc*bs)^2 inverse of the coarsest operator
    double* dense_work = nullptr;
    int dense_n = 0;
};

// kernel classes timed by the optional CUDA-event profiler (hemo_prof_*)
enum { HEMO_PROF_SPMV = 0, HEMO_PROF_CELL_JAC = 1, HEMO_PROF_GATHER_MAT = 2, HEMO_PROF_CELL_RES = 3,
       HEMO_PROF_CHEB_U0 = 4, HEMO_PROF_CHEB_P0 = 5, HEMO_PROF_MDOT = 6, HEMO_PROF_MAXPY = 7,
       HEMO_PROF_RAP = 8, HEMO_PROF_HALO = 9, HEMO_PROF_ALLREDUCE = 10, HEMO_PROF_COARSE = 11, HEMO_PROF_PC = 12,
       HEMO_PROF_NCLASS = 13 };

struct HemoProf {
    bool on = false;
    std::vector<cudaEvent_t> ev[HEMO_PROF_NCLASS];   // begin/end pairs
    size_t used[HEMO_PROF_NCLASS] = {0};
};

struct hemo_tet_state;      // assembly_tet.cu
struct hemo_cc_state;       // assembly_curlcurl.cu
struct HemoComm;            // comm.cu (NCCL communicator + halo plan of a mesh partition)

// device-resident FGMRES (krylov.cu)
struct HemoKrylov {
    int m = 0;                      // restart the buffers are sized for
    int64_t ldv = 0;                // leading dimension of the basis
    double* H = nullptr;            // (m+1) x m Hessenberg / triangular factor, column-major
    double* small = nullptr;        // cs, sn, g, ycoef, hcol, scale: 6 x (m+2)
    double* partial = nullptr;      // per-block partial sums of the multi-dot
    double* state = nullptr;        // FgState + scalars (64 doubles)
    double* state_host = nullptr;   // pinned copy
    int last_its = 0;               // iterations of the previous solve (first poll)
    int poll_every = 1;
    int64_t polls = 0;
    // owned entries of a local vector (multi-GPU): [0, seg_len0) and [seg_off1, seg_off1 + seg_len1); 0 = all
    int64_t seg_len0 = 0, seg_off1 = 0, seg_len1 = 0;
    // CUDA graph of one iteration
    cudaGraphExec_t iter_exec = nullptr;
    bool iter_valid = false;
    const double* iter_vals = nullptr;
    int64_t iter_nodes = 0;
    // kernel nodes and programmatic (PDL) edges of the last captured iteration graph (hemo_krylov_graph_info)
    int64_t iter_kernel_nodes = 0, iter_prog_edges = 0;
};

struct hemo_ctx {
    HemoProf prof;
    hemo_tet_state* tet = nullptr;   // tetrahedron rule tables (allocated on first use)
    hemo_cc_state* cc = nullptr;     // rule tables of the curl-curl formulation (allocated on first use)
    int formulation = 0;             // HEMO_FORM_STANDARD | HEMO_FORM_CURLCURL (hemo_set_formulation)
    int64_t rule_version = 0;        // bumped by every quadrature setter
    int device = 0;
    cudaStream_t stream = 0;
    std::string err;
    int64_t launches = 0;
    int pdl = 1;                     // programmatic dependent launch of the iteration kernels (HEMO_PDL=0 turns it off)

    // mesh (borrowed)
    int nv = 3;                     // nodes per cell: 3 = P1 triangle, 4 = Q1 quadrilateral (tensor-ordered) | P1 tetrahedron,
                                    // 6 = P2 triangle (3 vertex + 3 edge nodes)
    int dim = 2;                    // geometric dimension: 3 only for tetrahedra (include/hemo.h lists what works in 3-D)
    double fz = 0.0;                // third component of the body force (hemo_set_body_force3)
    const double* x = nullptr;
    const int32_t* cells = nullptr;
    const double* h = nullptr;
    int n = 0, E = 0;
    // node graph (borrowed) and derived maps (owned)
    const int32_t* nrowptr = nullptr;
    const int32_t* ncol = nullptr;
    int64_t nnz_node = 0;
    int32_t* cellpos = nullptr;     // E*nv*nv: slot of node b in row of node a
    int32_t* mseg_ptr = nullptr;    // nnz_node+1 gather segments (matrix)
    int32_t* mseg_src = nullptr;    // nv*nv*E: c*nv*nv + a*nv + b
    int32_t* vseg_ptr = nullptr;    // n+1 gather segments (vector)
    int32_t* vseg_src = nullptr;    // nv*E: c*nv + a
    int32_t* diagslot = nullptr;    // n: slot of node i in its own row
    int32_t* rowof = nullptr;       // nnz_node: row (node) of each slot
    double* Ae = nullptr;           // 9*nv*nv*E element matrices, SoA [(a*nv+b)*9 + ri*3+ci][E] (allocated on first use)
    double* Fe = nullptr;           // 3*nv*E element vectors, SoA [a*3 + comp][E]
    size_t Ae_count = 0, Fe_count = 0;
    int external_schur = 0;         // 1: hemo_pc_apply takes z_p from the caller (multi-GPU global pressure solve)
    double* dvec = nullptr;         // 3n lifting vector (g - x on bc dofs)

    // forms
    HemoForm par{0, 0, 0, {0, 0}, 0, 0.5, 1.0, 0, 0, 0, 0};
    bool have_par = false;
    const double* uh = nullptr;     // history vector of the time derivative (borrowed, 2n); null: u_n
    HemoRule rules[HEMO_NRULES];
    bool have_rule[HEMO_NRULES] = {false, false, false, false, false, false};
    bool rules_dirty = true;
    HemoQuadRule* qrules = nullptr; // HEMO_NRULES host-side rules of the quadrilateral path (allocated on first use)
    bool qrules_dirty = true;
    void* p2rules = nullptr;        // HEMO_NRULES host-side HemoP2Rule tables of the P2 triangle path (allocated on first use)
    HemoFacetRule frule{};
    HemoFacetSet fsets[HEMO_MAX_FACET_SETS];
    int64_t fset_version = 0;        // bumped by every hemo_set_facet_set (caches keyed on a set's cells check it)
    // deterministic 3-D wall-shear-stress gather (postproc.cu): cell -> index in the tagged set, per-cell contributions
    int32_t* wss_cell2t = nullptr; double* wss_tmp = nullptr; int wss_set = -1; int64_t wss_version = -1;
    uint8_t* dofflag = nullptr;
    double* dofmult = nullptr;
    uint8_t* cellflag = nullptr;
    bool have_bc = false;

    // reductions
    double* red_partial = nullptr;  // device partial sums
    size_t red_partial_n = 0;
    double* red_out = nullptr;      // device results
    double* red_host = nullptr;     // pinned host staging
    size_t red_out_n = 0;

    // solver
    hemo_solver_opts opts{};
    double schur_mass_coef = 0.0, schur_lap_coef = 0.0;
    HemoAmg amg[2];
    const double* mass = nullptr;   // lumped pressure mass (borrowed, n)
    areal2* a01 = nullptr;          // nnz_node: compact copy of the A01 block (u rows x p cols) for the PC
    uint8_t* pc_mask = nullptr;     // n: nodes excluded from the local preconditioner (ghosts)
    double* kry_coef = nullptr;     // device scratch for hemo_vec_maxpy coefficients (512)
    // CUDA graph of one preconditioner application (captured per hemo_pc_setup)
    cudaGraph_t pc_graph = nullptr;
    cudaGraphExec_t pc_graph_exec = nullptr;
    int64_t pc_graph_nodes = 0;
    bool pc_graph_dirty = true;     // re-captured lazily by the next hemo_pc_apply (hemo_fgmres captures whole iterations)
    bool capturing = false;
    int use_graph = 1;
    double* pc_in = nullptr;        // 3n (padded) staging of the graph's input / output
    double* pc_out = nullptr;
    double* pc_tmp_u = nullptr;     // 2n
    double* pc_tmp_u2 = nullptr;    // 2n
    double* pc_tmp_p = nullptr;     // n
    double* pc_tmp_p2 = nullptr;    // n
    double* kry_V = nullptr;        // (restart+1)*N
    double* kry_Z = nullptr;        // restart*N
    double* kry_w = nullptr;        // N
    int kry_restart = 0;
    HemoKrylov kry;
    // multi-GPU (comm.cu): null = single GPU
    // coarse space of the two-level Schwarz pressure solve (hemo_pc_set_coarse_pressure): replicated hierarchy in
    // another context, P0 rows of the local nodes, R0 = P0^T restricted to the owned nodes
    hemo_ctx* coarse_ctx = nullptr;
    int coarse_n = 0;
    int32_t *cp_rowptr = nullptr, *cp_col = nullptr; double* cp_val = nullptr;     // P0: n x coarse_n
    int32_t *cr_rowptr = nullptr, *cr_col = nullptr; double* cr_val = nullptr;     // R0: coarse_n x n (owned columns)
    double *coarse_rhs = nullptr, *coarse_sol = nullptr;
    int coarse_cycles = 1;
    cudaStream_t side_stream = nullptr;   // the coarse-space branch runs beside the local V-cycle (fork / join by events)
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    HemoComm* comm = nullptr;
    int comm_ras_overlap = 0;       // 1: the preconditioner input needs valid ghost values (overlapping Schwarz)
};

#define HEMO_CHECK_CUDA(ctx, expr)                                                     \
    do {                                                                               \
        cudaError_t _e = (expr);                                                       \
        if (_e != cudaSuccess) {                                                       \
            (ctx)->err = std::string(#expr) + ": " + cudaGetErrorString(_e);           \
            return (int)_e;                                                            \
        }                                                                              \
    } while (0)

#define HEMO_FAIL(ctx, code, msg)  \
    do {                           \
        (ctx)->err = (msg);        \
        return (code);             \
    } while (0)

// entry points that only exist for the 2-D cell types fail loudly on tetrahedra
#define HEMO_2D_ONLY(ctx, what)                                                                      \
    do {                                                                                             \
        if ((ctx)->dim == 3) HEMO_FAIL(ctx, HEMO_ESTATE, what " is not implemented for tetrahedra yet"); \
    } while (0)

#define HEMO_LAUNCH_CHECK(ctx)                                       \
    do {                                                             \
        (ctx)->launches++;                                           \
        cudaError_t _e = cudaGetLastError();                         \
        if (_e != cudaSuccess) {                                     \
            (ctx)->err = std::string("kernel launch: ") +            \
                         cudaGetErrorString(_e) + " at " + __FILE__ + ":" + std::to_string(__LINE__); \
            return (int)_e;                                          \
        }                                                            \
    } while (0)

// Programmatic dependent launch (PDL).  A kernel launched by HEMO_LAUNCH on a context with `pdl` set may be dispatched
// while its stream predecessor still runs.  Such a kernel follows one protocol:
//   1. optionally, loads of operands no kernel of the solve writes (operator values, indices, transfer weights);
//   2. hemo_pdl_wait(), unconditionally and before any early return: it blocks until the predecessor grid has completed
//      and its writes are visible, so the grid never completes ahead of its predecessor;
//   3. hemo_pdl_trigger(), which lets the successor's CTAs be dispatched (wait before trigger keeps at most two grids
//      of the chain live, so step 1 only ever overlaps the immediate predecessor);
//   4. the body.
// Both are no-ops in a kernel launched without the attribute.
__device__ __forceinline__ void hemo_pdl_wait() {
#if defined(__CUDA_ARCH__) && __CUDA_ARCH__ >= 900
    asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
}
__device__ __forceinline__ void hemo_pdl_trigger() {
#if defined(__CUDA_ARCH__) && __CUDA_ARCH__ >= 900
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
}

// Whether a launch on `st` may carry the programmatic-serialization attribute.  During stream capture the attribute
// becomes a programmatic graph edge, which only exists between kernel nodes: after a memcpy, an event join (several
// dependencies) or the start of the capture the launch stays plain.
static inline bool hemo_pdl_allowed(cudaStream_t st) {
    if (st == 0) return false;
    cudaStreamCaptureStatus cs;
    const cudaGraphNode_t* deps = nullptr;
    size_t nd = 0;
    if (cudaStreamGetCaptureInfo(st, &cs, nullptr, nullptr, &deps, &nd) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    if (cs != cudaStreamCaptureStatusActive) return true;
    cudaGraphNodeType t;
    return nd == 1 && cudaGraphNodeGetType(deps[0], &t) == cudaSuccess && t == cudaGraphNodeTypeKernel;
}

template <typename... P, typename... A>
static inline cudaError_t hemo_launch_kernel(hemo_ctx* ctx, void (*kernel)(P...), dim3 grid, dim3 block, size_t smem,
                                             cudaStream_t st, A... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    if (ctx->pdl && hemo_pdl_allowed(st)) {
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
    }
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, args...);
    const cudaError_t last = cudaGetLastError();
    return e != cudaSuccess ? e : last;
}

// kernel<<<grid, block, smem, st>>>(args...) followed by HEMO_LAUNCH_CHECK, for kernels that follow the PDL protocol
// above.  A template-id with a comma goes in parentheses: HEMO_LAUNCH(ctx, (k<BS, double>), ...).
#define HEMO_LAUNCH(ctx, kernel, grid, block, smem, st, ...)                                                        \
    do {                                                                                                            \
        (ctx)->launches++;                                                                                          \
        cudaError_t _e = hemo_launch_kernel((ctx), kernel, dim3(grid), dim3(block), (size_t)(smem), (st), __VA_ARGS__); \
        if (_e != cudaSuccess) {                                                                                    \
            (ctx)->err = std::string("kernel launch: ") +                                                           \
                         cudaGetErrorString(_e) + " at " + __FILE__ + ":" + std::to_string(__LINE__);              \
            return (int)_e;                                                                                         \
        }                                                                                                           \
    } while (0)

static inline void hemo_prof_mark(hemo_ctx* ctx, int cls) {
    if (!ctx->prof.on || ctx->capturing) return;
    HemoProf& p = ctx->prof;
    if (p.used[cls] == p.ev[cls].size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        p.ev[cls].push_back(e);
    }
    cudaEventRecord(p.ev[cls][p.used[cls]++], ctx->stream);
}
#define HEMO_PROF_BEGIN(ctx, cls) hemo_prof_mark(ctx, cls)
#define HEMO_PROF_END(ctx, cls) hemo_prof_mark(ctx, cls)

template <typename T>
static inline int hemo_alloc(hemo_ctx* ctx, T** p, size_t count) {
    if (*p) { cudaFree(*p); *p = nullptr; }
    if (count == 0) return 0;
    HEMO_CHECK_CUDA(ctx, cudaMalloc((void**)p, count * sizeof(T)));
    return 0;
}

template <typename T>
static inline int hemo_upload(hemo_ctx* ctx, T** p, const T* src, size_t count, bool src_is_device) {
    int rc = hemo_alloc(ctx, p, count);
    if (rc) return rc;
    if (count == 0) return 0;
    HEMO_CHECK_CUDA(ctx, cudaMemcpyAsync(*p, src, count * sizeof(T),
                                         src_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice,
                                         ctx->stream));
    return 0;
}

static inline int hemo_grid(int64_t n, int block) {
    int64_t g = (n + block - 1) / block;
    if (g < 1) g = 1;
    return (int)g;
}

// implemented in assembly_q1.cu (Q1 quadrilateral cell / facet kernels)
int hemo_q1_cell_jacobian(hemo_ctx* ctx, const double* x_dev, const double* un_dev);
int hemo_q1_cell_residual(hemo_ctx* ctx, const double* x_dev, const double* un_dev, const uint8_t* cellflag);
int hemo_q1_facets(hemo_ctx* ctx, int mode, const HemoFacetSet& fs, const double* x_dev, const double* un_dev,
                   const uint8_t* cellflag);
int hemo_q1_facet_flux(hemo_ctx* ctx, const HemoFacetSet& fs, const double* un_dev, double* partial);
int hemo_q1_laplace_mass(hemo_ctx* ctx);
// implemented in assembly_p2.cu (P2-P2 triangle cell / facet kernels, nv = 6)
int hemo_p2_set_quadrature(hemo_ctx* ctx, int block, const double* pts, const double* wts, int nq);
int hemo_p2_cell_jacobian(hemo_ctx* ctx, const double* x_dev, const double* un_dev);
int hemo_p2_cell_residual(hemo_ctx* ctx, const double* x_dev, const double* un_dev, const uint8_t* cellflag);
int hemo_p2_facets(hemo_ctx* ctx, int mode, const HemoFacetSet& fs, const double* x_dev, const double* un_dev,
                   const uint8_t* cellflag);
int hemo_p2_facet_flux(hemo_ctx* ctx, const HemoFacetSet& fs, const double* un_dev, double* partial);
int hemo_p2_laplace_mass(hemo_ctx* ctx);
// implemented in assembly_tet.cu
void hemo_tet_free(hemo_ctx* ctx);
void hemo_cc_free(hemo_ctx* ctx);
int hemo_tet_pattern(hemo_ctx* ctx, int64_t* rowptr_dev, int32_t* colind_dev);
int hemo_tet_assemble_jacobian(hemo_ctx* ctx, const double* x_dev, const double* un_dev, double* vals_dev);
int hemo_tet_assemble_residual(hemo_ctx* ctx, const double* x_dev, const double* un_dev, const double* g_dev,
                               double* b_dev);
int hemo_tet_set_facet_quadrature(hemo_ctx* ctx, const double* pts, const double* wts, int nq);
int hemo_tet_facet_flux(hemo_ctx* ctx, const HemoFacetSet& fs, const double* un_dev, double* partial);
int hemo_tet_laplace_mass(hemo_ctx* ctx);
int hemo_tet_pc_setup(hemo_ctx* ctx, const double* vals_dev);
int hemo_tet_selfp(hemo_ctx* ctx, const double* vals_dev);
int hemo_tet_velocity_solve(hemo_ctx* ctx, const double* vals_dev, const double* ru, const double* zp, double* tu,
                            double* tmp, double* zu, int sweeps, double omega);
int hemo_tet_spmv(hemo_ctx* ctx, const double* vals_dev, const double* x_dev, double* y_dev);
// implemented in linalg.cu
int hemo_ensure_reduce(hemo_ctx* ctx, size_t partial_n, size_t out_n);
// Drops everything sized by (dim, n, nnz_node) in the solver part of the context: Krylov basis,
// preconditioner work vectors, the compact A01 copy and every captured CUDA graph (their nodes
// hold raw pointers).  Called when the mesh or the cell type changes; the next hemo_pc_setup /
// hemo_fgmres reallocates.
void hemo_drop_solver_state(hemo_ctx* ctx);
int hemo_dot_dev(hemo_ctx* ctx, int64_t n, const double* x, const double* y, double* out_host);
int hemo_bsr_spmv(hemo_ctx* ctx, int bs, int n, const int32_t* rowptr, const int32_t* col,
                  const areal* val, const areal* x, areal* y);
// implemented in krylov.cu
void hemo_krylov_free(hemo_ctx* ctx);
void hemo_krylov_invalidate(hemo_ctx* ctx);
// implemented in comm.cu
int hemo_comm_halo(hemo_ctx* ctx, double* v_dev);                 // forward ghost update of a local [u | p] vector
int hemo_comm_allreduce_j(hemo_ctx* ctx, double* buf_dev, int count);   // in-place sum over the ranks (device buffer)
void hemo_comm_free(hemo_ctx* ctx);
// implemented in amg.cu
int hemo_amg_numeric(hemo_ctx* ctx, HemoAmg* amg);
int hemo_amg_vcycle(hemo_ctx* ctx, HemoAmg* amg, const double* b, double* x, int ncycles);
void hemo_amg_free(HemoAmg* amg);
