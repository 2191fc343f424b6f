/*
 * hemo.h — C-ABI of libhemo_sm100.so: the B200-native replacement for the
 * DOLFINx/PETSc calls made by the reference's `stabilized_schur` solvers.
 *
 * Every entry point names the reference interface it replaces (file:line
 * relative to the reference repository root).  Conventions:
 *   - plain pointers and sizes only; "dev" pointers are CUDA device addresses
 *     owned by the caller (torch tensors: tensor.data_ptr()); "host" pointers
 *     are ordinary host memory.  The library keeps the pointer, not a copy,
 *     for arrays documented as "borrowed".
 *   - every function returns 0 on success, <0 for an invalid argument or
 *     call order, >0 for a CUDA error (the cudaError_t), HEMO_DIVERGED for a
 *     linear solve that hit max iterations; hemo_last_error() gives the text.
 *   - work is enqueued on the stream given to hemo_set_stream (default 0);
 *     functions that return scalars to the host synchronise that stream.
 *   - one context per GPU per host thread; a context is not re-entrant.
 *
 * Global dof layout (3P `create_vector_block`, trigger
 * src/solvers/stabilized_schur.py:191-193): x = [u interleaved (2*n) | p (n)].
 * Matrix: one CSR, rows in that order, columns ascending, full FE pattern
 * (explicit zeros kept), int32 indices (nnz = 9 * nnz_node).  P1 triangles and Q1
 * quadrilaterals share this layout: one (u_x, u_y, p) triple per mesh vertex.
 */
#ifndef HEMO_H
#define HEMO_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hemo_ctx hemo_ctx;

#define HEMO_OK 0
#define HEMO_EINVAL (-1)
#define HEMO_ESTATE (-2)
#define HEMO_DIVERGED (-100)

/* Constants of the weak form: SolverBase.__init__ (src/solverBase.py:36-40)
 * and eps (src/solvers/stabilized_schur.py:100). */
typedef struct hemo_params {
    double dt, rho, mu;
    double f[2];
    double eps0;
} hemo_params;

/* Coefficients of one tagged exterior-facet integral; see FacetSet in
 * oracle/ns_oracle.py for the term each one multiplies
 * (src/solvers/stabilized_schur.py:79;
 *  src/solvers/stabilized_schur_pressure_backflow.py:192-217). */
typedef struct hemo_facet_coef {
    double a_p, pconst, a_g, a_s, a_n, beta_n, a_b, beta_b;
} hemo_facet_coef;

/* Block-form ids for hemo_set_quadrature: each block of
 * form(extract_blocks(F)) / form(extract_blocks(J)) is its own UFL form with
 * its own estimated degree (src/solvers/stabilized_schur.py:188-189). */
enum { HEMO_Q_FU = 0, HEMO_Q_FP = 1, HEMO_Q_UU = 2, HEMO_Q_UP = 3, HEMO_Q_PU = 4, HEMO_Q_PP = 5 };

/* Krylov / preconditioner options (mirrors the PETSc options set at
 * src/solvers/stabilized_schur.py:226-275). */
typedef struct hemo_solver_opts {
    int restart;          /* ksp_gmres_restart (reference: 200) */
    int max_it;           /* ksp_max_it (reference: 1000) */
    double rtol;          /* ksp_rtol (PETSc default 1e-5) */
    double atol;          /* ksp_atol (1e-50) */
    int amg_cycles_u;     /* V-cycles per A00^{-1} application */
    int amg_cycles_p;     /* V-cycles per Lp^{-1} application */
    int cheb_degree;      /* Chebyshev smoother degree per pre/post smoothing */
    int project_pressure; /* 1: remove the constant-pressure mode (nullsp attached,
                             src/solvers/stabilized_schur.py:314-317) */
    int pc_mode;          /* 0: upper block-triangular Schur (only mode implemented) */
    /* Schur-complement approximation S^-1 ~ schur_mass_coef * diag(Mp)^-1
     *                                       + schur_lap_coef * Lp^-1
     * (replaces SELFP, src/solvers/stabilized_schur.py:235; see DESIGN.md §5) */
    double schur_mass_coef;
    double schur_lap_coef;
    double cheb_ratio;    /* Chebyshev smoothing interval [lmax/ratio, lmax] (default 4) */
    int cheb_degree_pre;  /* degree of the pre-smoother (0: same as cheb_degree) */
} hemo_solver_opts;

/* ---- context ----------------------------------------------------------- */
int hemo_ctx_create(int device, hemo_ctx** out);
int hemo_ctx_destroy(hemo_ctx* ctx);
const char* hemo_last_error(hemo_ctx* ctx);
int hemo_set_stream(hemo_ctx* ctx, void* cuda_stream);
/* number of kernels this context has launched so far (bench.py gpu_launches) */
int64_t hemo_launch_count(hemo_ctx* ctx);

/* Optional CUDA-event timing of selected kernel classes on the context's
 * stream (bench.py roofline): 0 SpMV(J), 1 cell Jacobian, 2 matrix gather,
 * 3 cell residual, 4 Chebyshev step A00 level 0, 5 Chebyshev step Lp level 0,
 * 6 multi-dot, 7 multi-axpy+norm, 8 Galerkin R*AP level 0, 9 halo exchange, 10 allreduce, 11 coarse-space pressure
 * correction, 12 whole preconditioner application (nested classes overlap).  enable(on) resets
 * the counters; get() synchronises the stream. */
int hemo_prof_enable(hemo_ctx* ctx, int on);
int hemo_prof_get(hemo_ctx* ctx, int kernel_class, double* ms_total, int64_t* launches);

/* ---- mesh, spaces, pattern ---------------------------------------------- */
/* mesh.topology.cell_name() (src/solvers/stabilized_schur.py:55-58): P1 triangles (default)
 * or Q1 quadrilaterals with tensor-ordered vertices (0,0),(1,0),(0,1),(1,1) — the cells of the
 * recombined transfinite mesh, src/scenarios/stenosis_pressure_structured.py:379-386.  Call
 * before hemo_set_mesh; changing the type drops the mesh, the node graph and the quadrature
 * rules set earlier (rules belong to a cell type: triangle rules have weights summing to 1/2,
 * quadrilateral rules live on [0,1]^2 and sum to 1). */
/* HEMO_CELL_TRIANGLE_P2: P2-P2 triangles, `p_grade = 2` of src/solvers/stabilized_schur_pressure_backflow.py:71,102-106 and
 * stabilized_schur_backflow.py:63,85-87.  "Nodes" are then the P2 dof points: cells are n_cells*6 int32 (three vertex nodes,
 * then the nodes of the edges opposite local vertices 0, 1, 2 — the Basix dof order), x holds the coordinates of all nodes
 * (the affine geometry is read from the vertex nodes), every nodal array / the node graph / the CSR layout works as for P1
 * with one (u_x, u_y, p) triple per node; rules: points on the reference triangle, weights sum to 1/2, nq <= 128;
 * facet rule on [0,1], nq <= 8.  The per-step post-processing kernels are P1 / Q1 only. */
enum { HEMO_CELL_TRIANGLE = 0, HEMO_CELL_QUADRILATERAL = 1, HEMO_CELL_TETRAHEDRON = 2, HEMO_CELL_TRIANGLE_P2 = 3 };
int hemo_set_cell_type(hemo_ctx* ctx, int cell_type);

/* Weak form assembled by hemo_assemble_jacobian / hemo_assemble_residual.
 * HEMO_FORM_STANDARD: src/solvers/stabilized_schur.py:69-121 (and the boundary terms of its variants).
 * HEMO_FORM_CURLCURL: the rotational form of src/solvers/stabilized_schur_pressurebc.py:85-160 — curl-curl viscous
 *   term, (curl u x u) + grad(|u|^2/2) convection, SUPG/PSPG/LSIC with the viscous part of the strong residual
 *   dropped — with its boundary terms (:189-201): facet sets use pconst (weak pressure, the reference passes
 *   p/2) and a_n / beta_n (Nitsche for u_T = 0 written with curl x n).  P1 triangles and tetrahedra, default time
 *   scheme only. */
#define HEMO_FORM_STANDARD 0
#define HEMO_FORM_CURLCURL 1
int hemo_set_formulation(hemo_ctx* ctx, int formulation);
/* mesh.geometry.x / .dofmap / mesh.h (src/solvers/stabilized_schur.py:55-58,83-88).
 * x: n_nodes*2 doubles, cells: n_cells*(3|4) int32, h: n_cells doubles; borrowed. */
int hemo_set_mesh(hemo_ctx* ctx, const double* x_dev, int n_nodes,
                  const int32_t* cells_dev, int n_cells, const double* h_dev);
/* Node adjacency (CSR, sorted, diagonal included) = scalar P1 sparsity graph;
 * borrowed.  From it the library derives the block CSR pattern that
 * create_matrix_block builds (src/solvers/stabilized_schur.py:191), the
 * cell->nnz map and the atomic-free gather segments. */
int hemo_set_node_graph(hemo_ctx* ctx, const int32_t* nrowptr_dev, const int32_t* ncol_dev,
                        int64_t nnz_node);
int hemo_matrix_nnz(hemo_ctx* ctx, int64_t* nnz);
/* A.getValuesCSR() pattern part: rowptr (3n+1 int64) and colind (nnz int32), device. */
int hemo_get_pattern(hemo_ctx* ctx, int64_t* rowptr_dev, int32_t* colind_dev);

/* ---- forms ---------------------------------------------------------------- */
/* Quadrature rule of one block form (host arrays; pts = nq*2 reference coords; triangles:
 * wts sum to 1/2, nq <= 80; quadrilaterals: points on [0,1]^2, wts sum to 1, nq <= 256).
 * Basix rule selected by FFCx at form() (:188-189). */
int hemo_set_quadrature(hemo_ctx* ctx, int block, const double* pts_host,
                        const double* wts_host, int nq);
/* Facet rule shared by all exterior-facet integrals: points on [0,1] (2-D cells) or (s, t) pairs on the
 * reference triangle (tetrahedra). */
int hemo_set_facet_quadrature(hemo_ctx* ctx, const double* pts_host, const double* wts_host, int nq);
int hemo_set_params(hemo_ctx* ctx, const hemo_params* p);
/* Time scheme of the forms: they are evaluated at u_e = theta*u + (1-theta)*u_prev with the time
 * derivative (a0*u - u_h)/dt.  Default theta = 1/2, a0 = 1, u_h = u_prev: the mid-point scheme of
 * src/solvers/stabilized_schur.py:69-80.  theta = 1 with u_h = -(a1*u_prev + a2*u_prev2) is the
 * BDF1/BDF2 scheme of src/solvers/stabilized_schur_bdf2.py:76-110, 300-310 (bdf_a0/a1/a2 Constants).
 * uh_dev: 2n doubles, borrowed; NULL = u_prev.  tau_supg / tau_lsic always use u_prev (:101-103). */
int hemo_set_time_scheme(hemo_ctx* ctx, double theta, double a0, const double* uh_dev);
/* One tagged ds integral: unique boundary cells with a 3-bit (triangle) or 4-bit
 * (quadrilateral: facets (0,1),(0,2),(1,3),(2,3)) mask of the
 * local facets that carry the tag (Measure("ds", subdomain_id=...),
 * src/solvers/stabilized_schur_pressure_backflow.py:170-181).  m = 0 removes
 * the set.  Arrays are copied. */
int hemo_set_facet_set(hemo_ctx* ctx, int set_id, const int32_t* cells_dev,
                       const int32_t* facet_mask_dev, int m, const hemo_facet_coef* coef);
int hemo_set_facet_coef(hemo_ctx* ctx, int set_id, const hemo_facet_coef* coef);
/* Dirichlet data (src/solvers/stabilized_schur.py:198-199): per global dof a
 * flag (1 = constrained) and the diagonal multiplicity (number of DirichletBC
 * objects containing the dof); per cell a flag (1 = touches a constrained dof).
 * Copied. */
int hemo_set_bc(hemo_ctx* ctx, const uint8_t* dofflag_dev, const double* dofmult_dev,
                const uint8_t* cellflag_dev);

/* ---- assembly --------------------------------------------------------------- */
/* assembleJacobian → assemble_matrix_block (src/solvers/stabilized_schur.py:144-155):
 * vals (nnz doubles, device) receives J(x) with Dirichlet rows/cols zeroed and
 * the diagonal multiplicity set.  x = [u|p] (3n), un = u_prev (2n). */
int hemo_assemble_jacobian(hemo_ctx* ctx, const double* x_dev, const double* un_dev,
                           double* vals_dev);
/* assembleResidual → assemble_vector_block(..., x0=x, alpha=-1) (:157-175):
 * b = F(x) + lifting; b[bc] = x[bc] - g[bc].  g: 3n Dirichlet values. */
int hemo_assemble_residual(hemo_ctx* ctx, const double* x_dev, const double* un_dev,
                           const double* g_dev, double* b_dev);
/* assemble_scalar(dot(u_prev, n) * ds_out)
 * (src/solvers/stabilized_schur_pressure_backflow.py:383-385). */
int hemo_outlet_flux(hemo_ctx* ctx, int set_id, const double* un_dev, double* q_host);
/* Pressure Laplacian (node-graph CSR values, nnz_node doubles) and lumped
 * pressure mass (n doubles) for the Schur-complement approximation. */
int hemo_assemble_laplace_mass(hemo_ctx* ctx, double* lap_vals_dev, double* mass_dev);

/* ---- tetrahedra ------------------------------------------------------------------------------
 * FFCx tetrahedron kernels of the same forms (src/solvers/stabilized_schur.py:60-123 with
 * `mesh.topology.cell_name() == "tetrahedron"`, e.g. src/scenarios/taylor_green.py:34).  Element
 * tensors only: Ae SoA [(a*4+b)*16 + ri*4+ci][E], Fe SoA [a*4+comp][E] with ri/ci/comp in
 * (u_x, u_y, u_z, p) (hemo_tet_element_tensors: the cell kernel alone).  Uses hemo_set_params (dt, rho, mu,
 * eps0; f from f3_host) and hemo_set_time_scheme (theta, a0).  x: 3n, cells: 4E, sol = [u (3n) | p (n)],
 * un / uh: 3n (uh NULL = un).  Rules: points on the reference tetrahedron, weights sum to 1/6,
 * nq <= 343; one per block form like hemo_set_quadrature. */
/* With hemo_set_cell_type(HEMO_CELL_TETRAHEDRON) (x: 3n doubles, cells: 4E, sol = [u (3n) | p (n)], all
 * dof-sized arrays 4n) the generic entry points work on tetrahedra:
 *   hemo_set_mesh, hemo_set_node_graph, hemo_set_quadrature, hemo_matrix_nnz (16 * nnz_node),
 *   hemo_get_pattern (4n+1 row pointers; the CSR create_matrix_block builds, :191-193),
 *   hemo_set_facet_quadrature (points (s, t) on the reference triangle, nq*2 doubles, weights sum 1/2,
 *   nq <= 16), hemo_set_facet_set (4-bit mask, local facet i opposite local vertex i), hemo_set_bc,
 *   hemo_assemble_jacobian / hemo_assemble_residual (cell + exterior-facet integrals, Dirichlet rows and
 *   columns, lifting, set_bc), hemo_outlet_flux, hemo_spmv, hemo_assemble_laplace_mass,
 *   hemo_pc_setup / hemo_pc_apply / hemo_fgmres with the first 3-D preconditioner (DESIGN.md §5b: only the
 *   scalar pressure hierarchy `which = 1` is needed; the velocity block runs 4 * amg_cycles_u damped
 *   block-Jacobi sweeps).
 *   hemo_pc_set_schur_selfp (SELFP from the 3-D CSR values), hemo_wall_shear_stress (3n output; per-vertex
 *   gather in a fixed order, bitwise reproducible), hemo_early_stop_norms, hemo_l2_norm_sq (bs = 1 or 3).
 * Still 2-D only (HEMO_ESTATE on tetrahedra): hemo_boundary_force, partition masks. */
int hemo_set_body_force3(hemo_ctx* ctx, const double* f3_host);
int hemo_tet_set_quadrature(hemo_ctx* ctx, int block, const double* pts_host, const double* wts_host, int nq);
int hemo_tet_element_tensors(hemo_ctx* ctx, int n_nodes, int n_cells, const double* x_dev,
                             const int32_t* cells_dev, const double* h_dev, const double* sol_dev,
                             const double* un_dev, const double* uh_dev, const double* f3_host,
                             double* Ae_dev, double* Fe_dev);

/* ---- per-step post-processing on the device (SURVEY §8(f) rank 2) ------------------------
 * What Scenario.solve computes on the host after every solveStep (src/scenario.py:258-304,
 * 315-324) and the DFG force integrals (src/scenarios/dfg_1.py:183-211), for a device-resident
 * time loop.  Facet sets come from hemo_set_facet_set (a set with all-zero coefficients only
 * tags facets: the assembly skips it). */
/* solver.assemble_wss() (src/solverBase.py:144-195): wss (2n, device) =
 * sum over the set's facets of (1/|F|) int_F phi_i (T - (T.n) n) ds, T = -2 mu eps(u) n. */
int hemo_wall_shear_stress(hemo_ctx* ctx, int set_id, const double* x_dev, double* wss_dev);
/* force_host[0] = int mu d(u.t)/dn n_y - p n_x ds, force_host[1] = -int mu d(u.t)/dn n_x + p n_y ds
 * over the set, n = -FacetNormal, t = (n_y, -n_x) (drag / lift forms, dfg_1.py:189-202). */
int hemo_boundary_force(hemo_ctx* ctx, int set_id, const double* x_dev, double* force_host);
/* norms_host = { max|u - u_prev|, max|u| } over n entries (early stop, scenario.py:268-304). */
int hemo_early_stop_norms(hemo_ctx* ctx, int64_t n, const double* u_dev, const double* un_dev, double* norms_host);
/* assemble_scalar(inner(f, f) * dx) for a nodal field with bs = 1 | 2 components (scenario.py:315-324). */
int hemo_l2_norm_sq(hemo_ctx* ctx, int bs, const double* f_dev, double* out_host);

/* ---- linear algebra ----------------------------------------------------------- */
/* MatMult on the monolithic Jacobian (PETSc KSP inner loop, :226-229). */
int hemo_spmv(hemo_ctx* ctx, const double* vals_dev, const double* x_dev, double* y_dev);
/* y = a*x + y ; dot ; 2-norm on n-vectors (VecAXPY / VecDot / VecNorm). */
int hemo_axpy(hemo_ctx* ctx, int64_t n, double a, const double* x_dev, double* y_dev);
int hemo_dot(hemo_ctx* ctx, int64_t n, const double* x_dev, const double* y_dev, double* out_host);
int hemo_norm2(hemo_ctx* ctx, int64_t n, const double* x_dev, double* out_host);

/* MatNullSpaceRemove for the constant vector on an n-vector: x -= mean(x)
 * (nullsp.remove(x_n), src/solvers/stabilized_schur.py:319). */
int hemo_remove_mean_vec(hemo_ctx* ctx, int64_t n, double* x_dev);

/* ---- algebraic multigrid hierarchy -------------------------------------------- */
/* One level of a prolongator chain built by the host from the node graph
 * (aggregation + optional smoothing); all arrays here are HOST pointers.  which: 0 = velocity block A00 (2 dofs
 * per node, P (x) I2), 1 = pressure Laplacian.  Level l maps n_l → n_{l+1}
 * nodes.  All CSR arrays are copied.  The coarse node graph (pattern of
 * R*A*P) and the pattern of A*P are given so the numeric Galerkin product
 * runs with fixed structure each Newton iteration. */
int hemo_amg_set_level(hemo_ctx* ctx, int which, int level, int n_fine, int n_coarse,
                       const int32_t* p_rowptr, const int32_t* p_col, const double* p_val,
                       const int32_t* r_rowptr, const int32_t* r_col, const double* r_val,
                       const int32_t* ap_rowptr, const int32_t* ap_col,
                       const int32_t* c_rowptr, const int32_t* c_col);
int hemo_amg_finalize(hemo_ctx* ctx, int which, int n_levels);

/* Host (CPU) helper, one-time setup: greedy aggregation on a strength graph
 * (CSR without diagonal, host arrays).  exclude[i] != 0 leaves node i out
 * (agg[i] = -1).  No reference equivalent (PETSc builds ILU factors instead). */
int hemo_host_aggregate(int n, const int32_t* rowptr, const int32_t* col, const uint8_t* exclude,
                        int32_t* agg, int32_t* n_agg_out);

/* ---- solve ------------------------------------------------------------------------ */
/* Takes effect at the next hemo_pc_apply / hemo_amg_apply / hemo_fgmres: a change of the cycles, Chebyshev
 * parameters, Schur coefficients, project_pressure or pc_mode re-captures the graphs that bake them in. */
int hemo_set_solver_opts(hemo_ctx* ctx, const hemo_solver_opts* o);
/* PCSetUp (pc.setUp(), src/solvers/stabilized_schur.py:253 and every Newton
 * iteration): numeric Galerkin products of the A00 hierarchy from the current
 * Jacobian values, smoother bounds, pressure hierarchy from lap_vals (first
 * call or when lap_vals changes). */
int hemo_pc_setup(hemo_ctx* ctx, const double* vals_dev, const double* lap_vals_dev,
                  const double* mass_dev);
/* One V-cycle solve with hierarchy `which` (0: A00, 2n values; 1: Lp, n values):
 * x = V^ncycles(b) from a zero initial guess.  Exposed for the parity tests. */
int hemo_amg_apply(hemo_ctx* ctx, int which, const double* b_dev, double* x_dev, int ncycles);
/* Level operator of hierarchy `which` after hemo_pc_setup (device copy out;
 * nnzb*bs*bs doubles).  Exposed for the Galerkin-product parity test. */
int hemo_amg_get_level_values(hemo_ctx* ctx, int which, int level, double* vals_dev, int64_t capacity);
/* Which kernels run level `level` of hierarchy `which` (read-only, after hemo_amg_finalize):
 * out[0] = block rows n, out[1] = blocks nnzb, out[2] = entries of the sliced-ELL copy (0: CSR kernels),
 * out[3] = HEMO_AMG_SCOPE_*: the per-level kernels or the fused coarse V-cycle kernel (one CTA, which also
 * applies the dense inverse of the coarsest level). */
enum { HEMO_AMG_SCOPE_LEVEL = 0, HEMO_AMG_SCOPE_CTA = 1 };
int hemo_amg_level_info(hemo_ctx* ctx, int which, int level, int64_t out[4]);
/* ---- multi-GPU building blocks (domain decomposition, one partition per GPU) ----------
 * The host driver (cfd_hemodynamic_b200/parallel.py) exchanges ghost values and sums the
 * Krylov reductions with torch.distributed (NCCL); these entry points are the local,
 * per-partition pieces: PETSc VecMDot / VecMAXPY / VecScale before their MPI_Allreduce
 * (KSPSolve inside SNES, src/solvers/stabilized_schur.py:321), and the restriction of the
 * preconditioner to the partition (PCASM-like: ghost nodes are excluded, :256-267). */
int hemo_set_pc_mask(hemo_ctx* ctx, const uint8_t* node_mask_dev);
/* 1: hemo_pc_apply reads z_p from the pressure part of z (computed by the caller with a
 * global pressure solve) and only performs the velocity block solve. */
int hemo_set_external_schur(hemo_ctx* ctx, int on);
/* Numeric setup of the pressure-Laplacian hierarchy alone (contexts that only serve the
 * replicated global pressure solve). */
int hemo_amg_setup_scalar(hemo_ctx* ctx, const double* lap_vals_dev, double coarse_shift);
int hemo_mask_nodes(hemo_ctx* ctx, const uint8_t* node_mask_dev, double* x_dev);
int hemo_vec_mdot(hemo_ctx* ctx, int64_t n, int k, const double* V_dev, int64_t ldv, const double* w_dev,
                  double* h_host);
int hemo_vec_maxpy(hemo_ctx* ctx, int64_t n, int k, const double* V_dev, int64_t ldv,
                   const double* coef_host, double sign, double* w_dev, double* normsq_host);
int hemo_vec_scale(hemo_ctx* ctx, int64_t n, double a, const double* x_dev, double* y_dev);

/* ---- multi-GPU inside the library: one mesh partition per GPU, NCCL over NVLink ------------------
 * What PETSc/MPI does for the reference under `mpirun -n N` (SURVEY.md §2.4): after hemo_comm_init and
 * hemo_comm_set_partition, hemo_fgmres runs the distributed Krylov iteration itself — forward ghost
 * update of the search direction before the operator (ghostUpdate(INSERT, FORWARD),
 * src/solvers/stabilized_schur.py:137-142,168), one ncclAllReduce for the Gram-Schmidt coefficients and
 * one for the norm per iteration (VecMDot / VecNorm), Givens rotations and the convergence flag on the
 * device — captured in the same per-iteration CUDA graph as on one GPU.
 * Local numbering: owned nodes first, then ghost nodes grouped by owner rank in the order of `peers`.
 * hemo_comm_unique_id: ncclGetUniqueId on rank 0 (128 bytes, broadcast by the caller, e.g. through the
 * torch.distributed store).  NCCL is dlopen'ed (libnccl.so.2), the single-GPU path does not need it. */
int hemo_comm_unique_id(char* out128);
int hemo_comm_init(hemo_ctx* ctx, const char* uid128, int rank, int nranks);
int hemo_comm_info(hemo_ctx* ctx, int* rank, int* nranks, int* nccl_version, int64_t* halo_updates,
                   int64_t* allreduces);
/* Halo plan (host arrays): for neighbour k = peers[k], the owned local nodes send_nodes[send_ptr[k] ..
 * send_ptr[k+1]) are sent, and its values arrive in the ghost nodes n_owned + recv_ptr[k] .. n_owned +
 * recv_ptr[k+1]) — both sides list the nodes in ascending global id.  ras_overlap = 1: the preconditioner
 * input gets a ghost update too (overlapping restricted additive Schwarz, PCASM-like, :256-267). */
int hemo_comm_set_partition(hemo_ctx* ctx, int n_owned, int nneigh, const int32_t* peers_host,
                            const int32_t* send_ptr_host, const int32_t* send_nodes_host,
                            const int32_t* recv_ptr_host, int ras_overlap);
/* A context that carries only a scalar operator on an abstract graph (CSR, device, borrowed) — the replicated
 * coarse space below; only hemo_amg_set_level / hemo_amg_finalize / hemo_amg_setup_scalar / hemo_amg_apply work on it. */
int hemo_set_graph(hemo_ctx* ctx, int n, const int32_t* rowptr_dev, const int32_t* col_dev, int64_t nnz);
/* Two-level Schwarz for the pressure operator of the Schur approximation on a partitioned mesh (what PCASM lacks and
 * the reason its iteration count grows with the rank count, src/solvers/stabilized_schur.py:256-267): the rank-local
 * V-cycle is complemented by  P0 Ac^-1 sum_ranks(R0 r)  with Ac the level-k operator of the global pressure hierarchy,
 * replicated in `coarse_ctx` (hemo_set_graph + hierarchy).  P0: n x coarse_n (rows of the local nodes), R0: coarse_n x n
 * with the owned columns only; host CSR arrays, copied.  coarse_ctx = NULL removes the correction. */
int hemo_pc_set_coarse_pressure(hemo_ctx* ctx, hemo_ctx* coarse_ctx, int coarse_n, const int32_t* p_rowptr,
                                const int32_t* p_col, const double* p_val, const int32_t* r_rowptr,
                                const int32_t* r_col, const double* r_val, int cycles);
/* x.ghostUpdate(INSERT, FORWARD) of a local [u | p] vector (device). */
int hemo_comm_halo_update(hemo_ctx* ctx, double* v_dev);
/* comm.allreduce(SUM) of `count` doubles in place on the device (asynchronous on the stream). */
int hemo_comm_allreduce(hemo_ctx* ctx, double* buf_dev, int count);
/* VecDot of two local [u | p] vectors over the owned entries, summed over the ranks (plain dot
 * product without a communicator); synchronises the stream. */
int hemo_global_dot(hemo_ctx* ctx, const double* x_dev, const double* y_dev, double* out_host);
/* Iterations between two looks at the device-side convergence flag of hemo_fgmres once the iteration
 * count of the previous solve has been reached (default 1). */
int hemo_set_poll_interval(hemo_ctx* ctx, int every);

/* 1 (default): hemo_pc_setup captures one preconditioner application as a CUDA
 * graph (needs a non-default stream) and hemo_pc_apply replays it; 0: direct launches. */
int hemo_use_graph(hemo_ctx* ctx, int on);
/* SELFP Schur preconditioning matrix like the reference's (src/solvers/stabilized_schur.py:235):
 * Sp = A11 - A10 diag(A00)^-1 A01, formed on the device from the monolithic Jacobian on the
 * distance-2 node graph given with hemo_amg_set_fine_pattern(which = 1) (host CSR arrays, before
 * hemo_amg_set_level / hemo_amg_finalize), then the pressure hierarchy is re-formed numerically.
 * Use with schur_mass_coef = 0, schur_lap_coef = 1. */
int hemo_amg_set_fine_pattern(hemo_ctx* ctx, int which, const int32_t* rowptr_host, const int32_t* col_host);
int hemo_pc_set_schur_selfp(hemo_ctx* ctx, const double* vals_dev, double coarse_shift);
/* z = M^{-1} r (one application of the block preconditioner). */
int hemo_pc_apply(hemo_ctx* ctx, const double* vals_dev, const double* r_dev, double* z_dev);
/* KSPSolve: right-preconditioned FGMRES(restart) on J y = b with zero initial
 * guess (:226-229,272-273).  Device-resident: Hessenberg column, Givens rotations, residual estimate and
 * convergence flag live on the device, one iteration replays as one CUDA graph (non-default stream), the
 * host looks at the flag when the iteration count of the previous solve is reached.  its_out/resid_out on
 * host.  With a communicator (hemo_comm_init) b and y are local vectors; y returns with valid ghosts. */
int hemo_fgmres(hemo_ctx* ctx, const double* vals_dev, const double* b_dev, double* y_dev,
                int* its_out, double* rel_resid_out);
/* Kernel nodes and programmatic-dependent-launch edges of the most recently captured FGMRES iteration
 * graph (HEMO_PDL=0 in the environment at hemo_ctx_create launches every kernel plainly: no such edges).
 * HEMO_ESTATE before the first graph has been captured. */
int hemo_krylov_graph_info(hemo_ctx* ctx, int64_t* kernel_nodes, int64_t* programmatic_edges);

#ifdef __cplusplus
}
#endif
#endif /* HEMO_H */
