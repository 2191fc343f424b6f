// Finite-element assembly of the stabilized Navier–Stokes residual and Jacobian
// (P1–P1 triangles) for sm_100a.
//
// Replaces, for this path, the FFCx `tabulate_tensor` kernels + DOLFINx
// assembler triggered by the reference at src/solvers/stabilized_schur.py:154
// (assemble_matrix_block) and :172-174 (assemble_vector_block).
//
// Design (see DESIGN.md §3):
//   * one thread per cell; all quadrature dependence enters through the
//     moments  T2_ab = sum_q w_q tau(q) phi_a phi_b  and  L0 = sum_q w_q tau_lsic(q)
//     of each block form's own rule (rules live in __constant__ memory and are
//     a run-time input), the element tensors follow in closed form;
//   * element tensors are written SoA ([81][E] / [9][E]) so that every store of
//     a warp is one coalesced 256-byte line;
//   * a second kernel owns one CSR node-block (3x3 scalars) per thread and sums
//     the contributing cells in a fixed, precomputed order: no atomics, bitwise
//     reproducible; Dirichlet row/column zeroing and the diagonal multiplicity
//     are applied in the same pass.
#include <cub/device/device_scan.cuh>

#include "hemo_internal.cuh"

int hemo_amg_numeric_shift(hemo_ctx* ctx, HemoAmg* amg, double coarse_shift);

__constant__ HemoRule c_rules[HEMO_NRULES];
__constant__ HemoFacetRule c_frule;
__constant__ HemoForm c_par;

// symmetric 3x3 index: (0,0)=0 (1,1)=1 (2,2)=2 (0,1)=3 (0,2)=4 (1,2)=5
__device__ __forceinline__ constexpr int sym3(int a, int b) {
    return a == b ? a : (a + b + 2);
}

struct CellData {
    double g[3][2];    // grad phi_a
    double detJ;       // |det J|
    double U[3][2], N[3][2], P[3];
    double H[3][2];    // history of the time derivative: dudt = (a0 U - H) / dt
    double h;
};

__device__ __forceinline__ void load_cell(CellData& cd, int c, int E, const int32_t* __restrict__ cells,
                                          const double* __restrict__ x, const double* __restrict__ h,
                                          const double* __restrict__ sol, const double* __restrict__ un,
                                          const double* __restrict__ uh, int n, int v[3]) {
    v[0] = cells[3 * (int64_t)c + 0];
    v[1] = cells[3 * (int64_t)c + 1];
    v[2] = cells[3 * (int64_t)c + 2];
    double X[3][2];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const double2 xv = reinterpret_cast<const double2*>(x)[v[a]];
        X[a][0] = xv.x; X[a][1] = xv.y;
        const double2 uv = reinterpret_cast<const double2*>(sol)[v[a]];
        cd.U[a][0] = uv.x; cd.U[a][1] = uv.y;
        const double2 nv = reinterpret_cast<const double2*>(un)[v[a]];
        cd.N[a][0] = nv.x; cd.N[a][1] = nv.y;
        const double2 hv = reinterpret_cast<const double2*>(uh)[v[a]];
        cd.H[a][0] = hv.x; cd.H[a][1] = hv.y;
        cd.P[a] = sol[2 * (int64_t)n + v[a]];
    }
    const double j00 = X[1][0] - X[0][0], j01 = X[2][0] - X[0][0];
    const double j10 = X[1][1] - X[0][1], j11 = X[2][1] - X[0][1];
    const double det = j00 * j11 - j01 * j10;
    const double i00 = j11 / det, i01 = -j01 / det, i10 = -j10 / det, i11 = j00 / det;
    // grad phi_a = J^{-T} ghat_a, ghat = (-1,-1),(1,0),(0,1)
    cd.g[1][0] = i00; cd.g[1][1] = i01;
    cd.g[2][0] = i10; cd.g[2][1] = i11;
    cd.g[0][0] = -(i00 + i10); cd.g[0][1] = -(i01 + i11);
    cd.detJ = fabs(det);
    cd.h = h[c];
}

// Moments of rule r: T2[6] = detJ * sum_q w tau phi_a phi_b, L0 = detJ * sum_q w tau_lsic.
__device__ __forceinline__ void rule_moments(int r, const CellData& cd, double T2[6], double& L0) {
    const double nu = c_par.mu / c_par.rho;
    const double h = cd.h;
    const double inv_h2 = 1.0 / (h * h);
    const double t2inv = 2.0 / c_par.dt;
    const double t3inv = 4.0 * nu * inv_h2;
    const double c23 = t2inv * t2inv + t3inv * t3inv;
    const double eps2 = c_par.eps0 * c_par.eps0;
    const double re_fac = h / (2.0 * nu);
#pragma unroll
    for (int i = 0; i < 6; ++i) T2[i] = 0.0;
    L0 = 0.0;
    const int nq = c_rules[r].nq;
    for (int q = 0; q < nq; ++q) {
        const double p0 = c_rules[r].phi[q][0], p1 = c_rules[r].phi[q][1], p2 = c_rules[r].phi[q][2];
        const double w = c_rules[r].w[q];
        const double ux = p0 * cd.N[0][0] + p1 * cd.N[1][0] + p2 * cd.N[2][0];
        const double uy = p0 * cd.N[0][1] + p1 * cd.N[1][1] + p2 * cd.N[2][1];
        const double v2 = ux * ux + uy * uy;
        const double t1 = fmax(4.0 * v2, eps2) * inv_h2;   // (max(2|u_n|, eps)/h)^2
        const double tau = rsqrt(t1 + c23);
        const double v = sqrt(v2);
        const double Re = v * re_fac;
        const double z = (Re <= 3.0) ? Re / 3.0 : 1.0;
        const double tl = 0.5 * v * h * z;
        const double wt = w * tau;
        T2[0] = fma(wt * p0, p0, T2[0]);
        T2[1] = fma(wt * p1, p1, T2[1]);
        T2[2] = fma(wt * p2, p2, T2[2]);
        T2[3] = fma(wt * p0, p1, T2[3]);
        T2[4] = fma(wt * p0, p2, T2[4]);
        T2[5] = fma(wt * p1, p2, T2[5]);
        L0 = fma(w, tl, L0);
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) T2[i] *= cd.detJ;
    L0 *= cd.detJ;
}

__device__ __forceinline__ void moments_T1(const double T2[6], double T1[3]) {
    T1[0] = T2[0] + T2[3] + T2[4];
    T1[1] = T2[3] + T2[1] + T2[5];
    T1[2] = T2[4] + T2[5] + T2[2];
}

// Derived per-cell quantities shared by residual and Jacobian.
struct CellDerived {
    double M[3][2];   // u_mid nodal
    double G[2][2];   // G_ij = d_i u_mj
    double gp[2];     // grad p
    double s[3][3];   // s[c][a] = M_c . g_a
    double R[3][2];   // nodal values of the strong residual R (linear in phi)
    double A[3][2];   // nodal values of (u-u_n)/dt + (u_m.grad)u_m - f
    double divu;
};

__device__ __forceinline__ void derive_cell(const CellData& cd, CellDerived& d) {
    const double idt = 1.0 / c_par.dt, th = c_par.theta, a0 = c_par.a0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        d.M[a][0] = th * cd.U[a][0] + (1.0 - th) * cd.N[a][0];
        d.M[a][1] = th * cd.U[a][1] + (1.0 - th) * cd.N[a][1];
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
#pragma unroll
        for (int j = 0; j < 2; ++j)
            d.G[i][j] = cd.g[0][i] * d.M[0][j] + cd.g[1][i] * d.M[1][j] + cd.g[2][i] * d.M[2][j];
        d.gp[i] = cd.g[0][i] * cd.P[0] + cd.g[1][i] * cd.P[1] + cd.g[2][i] * cd.P[2];
    }
    d.divu = d.G[0][0] + d.G[1][1];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
#pragma unroll
        for (int a = 0; a < 3; ++a) d.s[c][a] = d.M[c][0] * cd.g[a][0] + d.M[c][1] * cd.g[a][1];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const double conv = d.M[c][0] * d.G[0][k] + d.M[c][1] * d.G[1][k];
            d.A[c][k] = (a0 * cd.U[c][k] - cd.H[c][k]) * idt + conv - c_par.f[k];
            d.R[c][k] = c_par.rho * d.A[c][k] + d.gp[k];
        }
    }
}

// Element residual: Fu[a][k], Fp[a].  Rule ids: HEMO_Q_FU, HEMO_Q_FP.
__device__ __forceinline__ void element_residual(const CellData& cd, const CellDerived& d,
                                                 double Fu[3][2], double Fp[3]) {
    const double rho = c_par.rho, mu = c_par.mu;
    double T2[6], L0, T2p[6], L0p, T1p[3];
    rule_moments(HEMO_Q_FU, cd, T2, L0);
    if (c_rules[HEMO_Q_FP].alias == HEMO_Q_FU) moments_T1(T2, T1p);
    else { rule_moments(HEMO_Q_FP, cd, T2p, L0p); moments_T1(T2p, T1p); }
    const HemoRule& ru = c_rules[HEMO_Q_FU];
    const HemoRule& rp = c_rules[HEMO_Q_FP];
    const double m0 = ru.m0 * cd.detJ;
    // eps = sym(G)
    const double e00 = d.G[0][0], e11 = d.G[1][1], e01 = 0.5 * (d.G[0][1] + d.G[1][0]);
    const double pbar = cd.detJ * (ru.m1[0] * cd.P[0] + ru.m1[1] * cd.P[1] + ru.m1[2] * cd.P[2]);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        // SUPG weights  W_d = sum_c T2_cd s_ca
        double Wd[3];
#pragma unroll
        for (int dd = 0; dd < 3; ++dd)
            Wd[dd] = T2[sym3(0, dd)] * d.s[0][a] + T2[sym3(1, dd)] * d.s[1][a] + T2[sym3(2, dd)] * d.s[2][a];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            double v = 0.0;
#pragma unroll
            for (int c = 0; c < 3; ++c) v += rho * cd.detJ * ru.m2[sym3(a, c)] * d.A[c][k];
            const double sig_g = 2.0 * mu * (k == 0 ? (cd.g[a][0] * e00 + cd.g[a][1] * e01)
                                                    : (cd.g[a][0] * e01 + cd.g[a][1] * e11));
            v += m0 * sig_g - cd.g[a][k] * pbar;
            v += Wd[0] * d.R[0][k] + Wd[1] * d.R[1][k] + Wd[2] * d.R[2][k];
            v += L0 * rho * d.divu * cd.g[a][k];
            Fu[a][k] = v;
        }
        double pv = cd.detJ * rp.m1[a] * d.divu;
        double acc = 0.0;
#pragma unroll
        for (int dd = 0; dd < 3; ++dd) acc += T1p[dd] * (d.R[dd][0] * cd.g[a][0] + d.R[dd][1] * cd.g[a][1]);
        Fp[a] = pv + acc / rho;
    }
}

// Element Jacobian, emitted entry by entry through `emit(slot, value)` with
// slot = (a*3+b)*9 + ri*3 + ci; ri/ci in (u_x, u_y, p).
template <typename Emit>
__device__ __forceinline__ void element_jacobian(const CellData& cd, const CellDerived& d, Emit emit) {
    // th = d(u_e)/du and idt = d(dudt)/du carry the time scheme (1/2 and 1/dt for the mid-point rule)
    const double rho = c_par.rho, mu = c_par.mu, idt = c_par.a0 / c_par.dt, th = c_par.theta;
    double T2[6], L0, T1up[3], T1pu[3], T0pp;
    rule_moments(HEMO_Q_UU, cd, T2, L0);
    {
        // rules shared between block forms are integrated once (alias = first
        // identical rule, resolved on the host)
        double t[6], l, t1[3];
        if (c_rules[HEMO_Q_UP].alias == HEMO_Q_UU) moments_T1(T2, T1up);
        else { rule_moments(HEMO_Q_UP, cd, t, l); moments_T1(t, T1up); }
        if (c_rules[HEMO_Q_PU].alias == HEMO_Q_UU) moments_T1(T2, T1pu);
        else if (c_rules[HEMO_Q_PU].alias == HEMO_Q_UP) { T1pu[0] = T1up[0]; T1pu[1] = T1up[1]; T1pu[2] = T1up[2]; }
        else { rule_moments(HEMO_Q_PU, cd, t, l); moments_T1(t, T1pu); }
        if (c_rules[HEMO_Q_PP].alias == HEMO_Q_UU) moments_T1(T2, t1);
        else if (c_rules[HEMO_Q_PP].alias == HEMO_Q_UP) { t1[0] = T1up[0]; t1[1] = T1up[1]; t1[2] = T1up[2]; }
        else if (c_rules[HEMO_Q_PP].alias == HEMO_Q_PU) { t1[0] = T1pu[0]; t1[1] = T1pu[1]; t1[2] = T1pu[2]; }
        else { rule_moments(HEMO_Q_PP, cd, t, l); moments_T1(t, t1); }
        T0pp = t1[0] + t1[1] + t1[2];
    }
    const HemoRule& ruu = c_rules[HEMO_Q_UU];
    const double m0 = ruu.m0 * cd.detJ;
    // RT[b][k] = sum_d T2_db R_dk
    double RT[3][2];
#pragma unroll
    for (int b = 0; b < 3; ++b)
#pragma unroll
        for (int k = 0; k < 2; ++k)
            RT[b][k] = T2[sym3(0, b)] * d.R[0][k] + T2[sym3(1, b)] * d.R[1][k] + T2[sym3(2, b)] * d.R[2][k];
    // Y_b = sum_d T1pu_d s_db ; V_a = sum_c T1up_c s_ca
    double Y[3], V[3];
#pragma unroll
    for (int b = 0; b < 3; ++b) {
        Y[b] = T1pu[0] * d.s[0][b] + T1pu[1] * d.s[1][b] + T1pu[2] * d.s[2][b];
        V[b] = T1up[0] * d.s[0][b] + T1up[1] * d.s[1][b] + T1up[2] * d.s[2][b];
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        // TS[c] = sum_d T2_cd s_da  (used for Z_ab)
        double TS[3];
#pragma unroll
        for (int c = 0; c < 3; ++c)
            TS[c] = T2[sym3(c, 0)] * d.s[0][a] + T2[sym3(c, 1)] * d.s[1][a] + T2[sym3(c, 2)] * d.s[2][a];
        // (G g_a)_l = sum_k G_lk g_ak
        const double Gga[2] = {d.G[0][0] * cd.g[a][0] + d.G[0][1] * cd.g[a][1],
                               d.G[1][0] * cd.g[a][0] + d.G[1][1] * cd.g[a][1]};
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            const int base = (a * 3 + b) * 9;
            const double m2ab = cd.detJ * ruu.m2[sym3(a, b)];
            const double gab = cd.g[a][0] * cd.g[b][0] + cd.g[a][1] * cd.g[b][1];
            // W_ab = sum_c T2_cb s_ca = TS[b] ;  Z_ab = sum_d TS[d] s_db
            const double Wab = TS[b];
            const double Zab = TS[0] * d.s[0][b] + TS[1] * d.s[1][b] + TS[2] * d.s[2][b];
            double Qab = 0.0;
#pragma unroll
            for (int c = 0; c < 3; ++c) Qab += cd.detJ * ruu.m2[sym3(a, c)] * d.s[c][b];
            const double diag = rho * m2ab * idt + th * rho * Qab + th * mu * m0 * gab +
                                rho * Wab * idt + th * rho * Zab;
            const double cG = th * rho * (m2ab + Wab);
#pragma unroll
            for (int k = 0; k < 2; ++k)
#pragma unroll
                for (int l = 0; l < 2; ++l) {
                    double v = cG * d.G[l][k] + th * mu * m0 * cd.g[a][l] * cd.g[b][k] +
                               th * cd.g[a][l] * RT[b][k] + th * L0 * rho * cd.g[a][k] * cd.g[b][l];
                    if (k == l) v += diag;
                    emit(base + k * 3 + l, v);
                }
            const double m1b_up = cd.detJ * c_rules[HEMO_Q_UP].m1[b];
            const double m1a_pu = cd.detJ * c_rules[HEMO_Q_PU].m1[a];
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                emit(base + k * 3 + 2, -m1b_up * cd.g[a][k] + cd.g[b][k] * V[a]);              // J_up
                emit(base + 6 + k, th * m1a_pu * cd.g[b][k] +
                                       cd.g[a][k] * (T1pu[b] * idt + th * Y[b]) +
                                       th * T1pu[b] * Gga[k]);                                   // J_pu
            }
            emit(base + 8, T0pp / rho * gab);                                                    // J_pp
        }
    }
}

// ---------------------------------------------------------------------------
// cell kernels
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
k_cell_jacobian(int E, int n, const int32_t* __restrict__ cells, const double* __restrict__ x,
                const double* __restrict__ h, const double* __restrict__ sol,
                const double* __restrict__ un, const double* __restrict__ uh, double* __restrict__ Ae) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= E) return;
    CellData cd;
    int v[3];
    load_cell(cd, c, E, cells, x, h, sol, un, uh, n, v);
    CellDerived d;
    derive_cell(cd, d);
    double* out = Ae + c;
    const int64_t stride = E;
    element_jacobian(cd, d, [&](int slot, double val) { out[slot * stride] = val; });
}

// lifting: be += Ae[:, j] * (g - x)_j over constrained dofs j (3P apply_lifting with
// x0 = x, alpha = -1; reference src/solvers/stabilized_schur.py:172-174).  Kept out of line:
// only boundary-adjacent cells take this path and it would otherwise set the register
// count of the whole residual kernel.
// Self-contained (reloads the cell, adds into Fe after the residual has been stored) so that no
// array of k_cell_residual has its address taken: its hot path stays in registers.
__device__ __noinline__ void lift_cell(int c, int E, int n, const int32_t* __restrict__ cells,
                                       const double* __restrict__ x, const double* __restrict__ h,
                                       const double* __restrict__ sol, const double* __restrict__ un,
                                       const double* __restrict__ uh, const double* __restrict__ dvec,
                                       double* __restrict__ Fe) {
    CellData cd;
    int v[3];
    load_cell(cd, c, E, cells, x, h, sol, un, uh, n, v);
    double dl[3][3];
    bool any = false;
#pragma unroll
    for (int b = 0; b < 3; ++b) {
        dl[b][0] = dvec[2 * (int64_t)v[b]];
        dl[b][1] = dvec[2 * (int64_t)v[b] + 1];
        dl[b][2] = dvec[2 * (int64_t)n + v[b]];
        any = any || dl[b][0] != 0.0 || dl[b][1] != 0.0 || dl[b][2] != 0.0;
    }
    if (!any) return;
    CellDerived d;
    derive_cell(cd, d);
    double lift[3][3];
#pragma unroll
    for (int a = 0; a < 3; ++a) lift[a][0] = lift[a][1] = lift[a][2] = 0.0;
    element_jacobian(cd, d, [&](int slot, double val) {
        const int ab = slot / 9, rc = slot % 9;
        const int a = ab / 3, b = ab % 3, ri = rc / 3, ci = rc % 3;
        lift[a][ri] += val * dl[b][ci];
    });
    const int64_t stride = E;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        Fe[(a * 3 + 0) * stride + c] += lift[a][0];
        Fe[(a * 3 + 1) * stride + c] += lift[a][1];
        Fe[(a * 3 + 2) * stride + c] += lift[a][2];
    }
}

__global__ void __launch_bounds__(128)
k_cell_residual(int E, int n, const int32_t* __restrict__ cells, const double* __restrict__ x,
                const double* __restrict__ h, const double* __restrict__ sol,
                const double* __restrict__ un, const double* __restrict__ uh,
                const uint8_t* __restrict__ cellflag, const double* __restrict__ dvec, double* __restrict__ Fe) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= E) return;
    {
        CellData cd;
        int v[3];
        load_cell(cd, c, E, cells, x, h, sol, un, uh, n, v);
        CellDerived d;
        derive_cell(cd, d);
        double Fu[3][2], Fp[3];
        element_residual(cd, d, Fu, Fp);
        const int64_t stride = E;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            Fe[(a * 3 + 0) * stride + c] = Fu[a][0];
            Fe[(a * 3 + 1) * stride + c] = Fu[a][1];
            Fe[(a * 3 + 2) * stride + c] = Fp[a];
        }
    }
    if (cellflag != nullptr && cellflag[c]) lift_cell(c, E, n, cells, x, h, sol, un, uh, dvec, Fe);
}

// ---------------------------------------------------------------------------
// exterior-facet kernel: one thread per boundary cell of a tagged set; adds
// the facet terms into the element tensors of that cell (mode 0: residual
// into Fe (+ lifting), mode 1: Jacobian into Ae).
// ---------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(128)
k_facets(int m, int E, int n, const int32_t* __restrict__ fcells, const int32_t* __restrict__ fmask,
         hemo_facet_coef co, const int32_t* __restrict__ cells, const double* __restrict__ x,
         const double* __restrict__ h, const double* __restrict__ sol, const double* __restrict__ un,
         const double* __restrict__ uh, const uint8_t* __restrict__ cellflag, const double* __restrict__ dvec,
         double* __restrict__ out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m) return;
    const int c = fcells[t];
    const int mask = fmask[t];
    CellData cd;
    int v[3];
    load_cell(cd, c, E, cells, x, h, sol, un, uh, n, v);
    double X[3][2];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        X[a][0] = x[2 * (int64_t)v[a]];
        X[a][1] = x[2 * (int64_t)v[a] + 1];
    }
    const double th = c_par.theta;     // d(u_e)/du of the time scheme (1/2: mid-point rule)
    double M[3][2];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        M[a][0] = th * cd.U[a][0] + (1.0 - th) * cd.N[a][0];
        M[a][1] = th * cd.U[a][1] + (1.0 - th) * cd.N[a][1];
    }
    double G[2][2];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j)
            G[i][j] = cd.g[0][i] * M[0][j] + cd.g[1][i] * M[1][j] + cd.g[2][i] * M[2][j];
    const double mu = c_par.mu, rho = c_par.rho;
    const int64_t stride = E;

    double dl[3][3];
    bool lift = false;
    if (MODE == 0 && cellflag != nullptr && cellflag[c]) {
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            dl[b][0] = dvec[2 * (int64_t)v[b]];
            dl[b][1] = dvec[2 * (int64_t)v[b] + 1];
            dl[b][2] = dvec[2 * (int64_t)n + v[b]];
            lift = lift || dl[b][0] != 0.0 || dl[b][1] != 0.0 || dl[b][2] != 0.0;
        }
    }

    for (int lf = 0; lf < 3; ++lf) {
        if (!(mask & (1 << lf))) continue;
        const int va = (lf == 0) ? 1 : 0;
        const int vb = (lf == 2) ? 1 : 2;
        const double tx = X[vb][0] - X[va][0], ty = X[vb][1] - X[va][1];
        const double len = sqrt(tx * tx + ty * ty);
        double nx = ty / len, ny = -tx / len;
        const double side = nx * (X[va][0] - X[lf][0]) + ny * (X[va][1] - X[lf][1]);
        if (side < 0.0) { nx = -nx; ny = -ny; }
        const double nr[2] = {nx, ny};
        const double Pn[2][2] = {{1.0 - nx * nx, -nx * ny}, {-nx * ny, 1.0 - ny * ny}};
        // facet moments via the facet rule: Phi_a, Phi_ab, B_ab (backflow)
        double Ph[3] = {0, 0, 0}, Ph2[3][3], B[3][3];
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b) { Ph2[a][b] = 0.0; B[a][b] = 0.0; }
        for (int q = 0; q < c_frule.nq; ++q) {
            const double s = c_frule.s[q], w = c_frule.w[q] * len;
            double phi[3] = {0, 0, 0};
            phi[va] = 1.0 - s;
            phi[vb] = s;
            const double unx = phi[0] * cd.N[0][0] + phi[1] * cd.N[1][0] + phi[2] * cd.N[2][0];
            const double uny = phi[0] * cd.N[0][1] + phi[1] * cd.N[1][1] + phi[2] * cd.N[2][1];
            const double unn = unx * nx + uny * ny;
            const double unm = 0.5 * (unn - fabs(unn));
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                Ph[a] += w * phi[a];
#pragma unroll
                for (int b = 0; b < 3; ++b) {
                    Ph2[a][b] += w * phi[a] * phi[b];
                    B[a][b] += w * unm * phi[a] * phi[b];
                }
            }
        }
        double dn[3], Png[3][2];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            dn[a] = cd.g[a][0] * nx + cd.g[a][1] * ny;
            Png[a][0] = Pn[0][0] * cd.g[a][0] + Pn[0][1] * cd.g[a][1];
            Png[a][1] = Pn[1][0] * cd.g[a][0] + Pn[1][1] * cd.g[a][1];
        }
        const double pen = co.a_n * co.beta_n * mu / cd.h;
        const double bf = co.a_b * co.beta_b * rho;

        if (MODE == 1 || lift) {
            // d(Fu[a][k]) / d(U[b][l]) and / d(P[b])
#pragma unroll
            for (int a = 0; a < 3; ++a)
#pragma unroll
                for (int b = 0; b < 3; ++b) {
                    double juu[2][2], jup[2];
#pragma unroll
                    for (int k = 0; k < 2; ++k) {
                        jup[k] = co.a_p * nr[k] * Ph2[a][b];
#pragma unroll
                        for (int l = 0; l < 2; ++l) {
                            const double dkl = (k == l) ? 1.0 : 0.0;
                            double vv = -th * co.a_g * mu * cd.g[b][k] * nr[l] * Ph[a];
                            vv -= th * co.a_s * mu * (cd.g[b][k] * nr[l] + dn[b] * dkl) * Ph[a];
                            vv -= th * co.a_n * mu * (Png[b][k] * nr[l] + dn[b] * Pn[k][l]) * Ph[a];
                            vv -= th * co.a_n * mu * (Png[a][l] * nr[k] + dn[a] * Pn[k][l]) * Ph[b];
                            vv += th * pen * Pn[k][l] * Ph2[a][b];
                            vv -= th * bf * B[a][b] * dkl;
                            juu[k][l] = vv;
                        }
                    }
                    if (MODE == 1) {
                        const int base = (a * 3 + b) * 9;
#pragma unroll
                        for (int k = 0; k < 2; ++k) {
#pragma unroll
                            for (int l = 0; l < 2; ++l) out[(base + k * 3 + l) * stride + c] += juu[k][l];
                            out[(base + k * 3 + 2) * stride + c] += jup[k];
                        }
                    } else {
#pragma unroll
                        for (int k = 0; k < 2; ++k) {
                            const double add = juu[k][0] * dl[b][0] + juu[k][1] * dl[b][1] + jup[k] * dl[b][2];
                            out[(a * 3 + k) * stride + c] += add;
                        }
                    }
                }
        }
        if (MODE == 0) {
            // residual
            const double Gn[2] = {G[0][0] * nx + G[0][1] * ny, G[1][0] * nx + G[1][1] * ny};
            const double e01 = 0.5 * (G[0][1] + G[1][0]);
            const double en[2] = {G[0][0] * nx + e01 * ny, e01 * nx + G[1][1] * ny};
            const double enT[2] = {Pn[0][0] * en[0] + Pn[0][1] * en[1], Pn[1][0] * en[0] + Pn[1][1] * en[1]};
            // int u_m ds (vector) and projected
            double Mi[2] = {0, 0};
#pragma unroll
            for (int cc = 0; cc < 3; ++cc) { Mi[0] += Ph[cc] * M[cc][0]; Mi[1] += Ph[cc] * M[cc][1]; }
            const double MiT[2] = {Pn[0][0] * Mi[0] + Pn[0][1] * Mi[1], Pn[1][0] * Mi[0] + Pn[1][1] * Mi[1]};
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                double pa = 0.0, Ma[2] = {0, 0}, Ba[2] = {0, 0};
#pragma unroll
                for (int b = 0; b < 3; ++b) {
                    pa += Ph2[a][b] * cd.P[b];
                    Ma[0] += Ph2[a][b] * M[b][0]; Ma[1] += Ph2[a][b] * M[b][1];
                    Ba[0] += B[a][b] * M[b][0];   Ba[1] += B[a][b] * M[b][1];
                }
                const double MaT[2] = {Pn[0][0] * Ma[0] + Pn[0][1] * Ma[1], Pn[1][0] * Ma[0] + Pn[1][1] * Ma[1]};
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    double vv = (co.a_p * pa + co.pconst * Ph[a]) * nr[k];
                    vv -= co.a_g * mu * Gn[k] * Ph[a];
                    vv -= co.a_s * 2.0 * mu * en[k] * Ph[a];
                    vv -= co.a_n * 2.0 * mu * enT[k] * Ph[a];
                    // -(2 mu eps(v) n).u_T : eps(v)n_i = 1/2 (g_ai n_k + dn_a d_ik)
                    vv -= co.a_n * mu * ((cd.g[a][0] * MiT[0] + cd.g[a][1] * MiT[1]) * nr[k] + dn[a] * MiT[k]);
                    vv += pen * MaT[k];
                    vv -= bf * Ba[k];
                    out[(a * 3 + k) * stride + c] += vv;
                }
            }
        }
    }
}

// outlet flux  Q = int u_prev . n ds  over one facet set: per-cell partials
__global__ void k_facet_flux(int m, const int32_t* __restrict__ fcells, const int32_t* __restrict__ fmask,
                             const int32_t* __restrict__ cells, const double* __restrict__ x,
                             const double* __restrict__ un, double* __restrict__ partial) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m) return;
    const int c = fcells[t];
    const int mask = fmask[t];
    int v[3];
    double X[3][2], N[3][2];
    for (int a = 0; a < 3; ++a) {
        v[a] = cells[3 * (int64_t)c + a];
        X[a][0] = x[2 * (int64_t)v[a]]; X[a][1] = x[2 * (int64_t)v[a] + 1];
        N[a][0] = un[2 * (int64_t)v[a]]; N[a][1] = un[2 * (int64_t)v[a] + 1];
    }
    double q = 0.0;
    for (int lf = 0; lf < 3; ++lf) {
        if (!(mask & (1 << lf))) continue;
        const int va = (lf == 0) ? 1 : 0;
        const int vb = (lf == 2) ? 1 : 2;
        const double tx = X[vb][0] - X[va][0], ty = X[vb][1] - X[va][1];
        double nx = ty, ny = -tx;   // |n| = len
        const double side = nx * (X[va][0] - X[lf][0]) + ny * (X[va][1] - X[lf][1]);
        if (side < 0.0) { nx = -nx; ny = -ny; }
        q += 0.5 * ((N[va][0] + N[vb][0]) * nx + (N[va][1] + N[vb][1]) * ny);
    }
    partial[t] = q;
}

__global__ void k_sum_serial(int m, const double* __restrict__ partial, double* __restrict__ out) {
    // deterministic single-block tree sum (boundary-sized input)
    __shared__ double sh[256];
    double acc = 0.0;
    for (int i = threadIdx.x; i < m; i += blockDim.x) acc += partial[i];
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = sh[0];
}

// ---------------------------------------------------------------------------
// gather (atomic-free scatter) kernels
// ---------------------------------------------------------------------------
// One thread per node pair (i, j) = one 3x3 scalar block of the CSR matrix.
__global__ void __launch_bounds__(256)
k_gather_matrix(int n, int nv2, int64_t nnz_node, int64_t E, const int32_t* __restrict__ nrowptr,
                const int32_t* __restrict__ ncol, const int32_t* __restrict__ rowof,
                const int32_t* __restrict__ seg_ptr, const int32_t* __restrict__ seg_src,
                const double* __restrict__ Ae, const uint8_t* __restrict__ dofflag,
                const double* __restrict__ dofmult, double* __restrict__ vals) {
    const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= nnz_node) return;
    const int i = rowof[s];
    const int j = ncol[s];
    double acc[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) acc[k] = 0.0;
    const int b0 = seg_ptr[s], b1 = seg_ptr[s + 1];
    for (int t = b0; t < b1; ++t) {
        const int src = seg_src[t];
        const int64_t c = src / nv2;
        const int ab = src - (int)c * nv2;
        const double* p = Ae + (int64_t)ab * 9 * E + c;
#pragma unroll
        for (int k = 0; k < 9; ++k) acc[k] += p[k * E];
    }
    const int r0 = nrowptr[i];
    const int deg = nrowptr[i + 1] - r0;
    const int tpos = (int)(s - r0);
    if (dofflag != nullptr) {
        const bool fr[3] = {dofflag[2 * (int64_t)i] != 0, dofflag[2 * (int64_t)i + 1] != 0,
                            dofflag[2 * (int64_t)n + i] != 0};
        const bool fc[3] = {dofflag[2 * (int64_t)j] != 0, dofflag[2 * (int64_t)j + 1] != 0,
                            dofflag[2 * (int64_t)n + j] != 0};
#pragma unroll
        for (int ri = 0; ri < 3; ++ri)
#pragma unroll
            for (int ci = 0; ci < 3; ++ci)
                if (fr[ri] || fc[ci]) acc[ri * 3 + ci] = 0.0;
        if (i == j) {
            if (fr[0]) acc[0] = dofmult[2 * (int64_t)i];
            if (fr[1]) acc[4] = dofmult[2 * (int64_t)i + 1];
            if (fr[2]) acc[8] = dofmult[2 * (int64_t)n + i];
        }
    }
    // rows 2i, 2i+1 start at 6*r0 and 6*r0+3*deg; p-row at 6*nnz_node + 3*r0
    const int64_t ru0 = 6 * (int64_t)r0, ru1 = ru0 + 3 * deg, rp = 6 * nnz_node + 3 * (int64_t)r0;
    vals[ru0 + 2 * tpos] = acc[0];
    vals[ru0 + 2 * tpos + 1] = acc[1];
    vals[ru0 + 2 * deg + tpos] = acc[2];
    vals[ru1 + 2 * tpos] = acc[3];
    vals[ru1 + 2 * tpos + 1] = acc[4];
    vals[ru1 + 2 * deg + tpos] = acc[5];
    vals[rp + 2 * tpos] = acc[6];
    vals[rp + 2 * tpos + 1] = acc[7];
    vals[rp + 2 * deg + tpos] = acc[8];
}

// One thread per node: b[2i], b[2i+1], b[2n+i]; then set_bc.
__global__ void __launch_bounds__(256)
k_gather_vector(int n, int nv, int64_t E, const int32_t* __restrict__ seg_ptr, const int32_t* __restrict__ seg_src,
                const double* __restrict__ Fe, const uint8_t* __restrict__ dofflag,
                const double* __restrict__ x, const double* __restrict__ g, double* __restrict__ b) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double a0 = 0, a1 = 0, a2 = 0;
    for (int t = seg_ptr[i]; t < seg_ptr[i + 1]; ++t) {
        const int src = seg_src[t];
        const int64_t c = src / nv;
        const int a = src - (int)c * nv;
        a0 += Fe[(a * 3 + 0) * E + c];
        a1 += Fe[(a * 3 + 1) * E + c];
        a2 += Fe[(a * 3 + 2) * E + c];
    }
    const int64_t d0 = 2 * (int64_t)i, d1 = d0 + 1, d2 = 2 * (int64_t)n + i;
    if (dofflag != nullptr) {
        if (dofflag[d0]) a0 = x[d0] - g[d0];
        if (dofflag[d1]) a1 = x[d1] - g[d1];
        if (dofflag[d2]) a2 = x[d2] - g[d2];
    }
    b[d0] = a0; b[d1] = a1; b[d2] = a2;
}

__global__ void k_lift_vector(int64_t N, const uint8_t* __restrict__ dofflag, const double* __restrict__ x,
                              const double* __restrict__ g, double* __restrict__ d) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= N) return;
    d[i] = dofflag[i] ? (g[i] - x[i]) : 0.0;
}

// ---------------------------------------------------------------------------
// pressure Laplacian + lumped mass (Schur-complement approximation operators)
// ---------------------------------------------------------------------------
__global__ void k_cell_laplace(int E, const int32_t* __restrict__ cells, const double* __restrict__ x,
                               double* __restrict__ Ke /*[9][E]*/, double* __restrict__ Me /*[3][E]*/) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= E) return;
    double X[3][2];
    for (int a = 0; a < 3; ++a) {
        const int v = cells[3 * (int64_t)c + a];
        X[a][0] = x[2 * (int64_t)v]; X[a][1] = x[2 * (int64_t)v + 1];
    }
    const double j00 = X[1][0] - X[0][0], j01 = X[2][0] - X[0][0];
    const double j10 = X[1][1] - X[0][1], j11 = X[2][1] - X[0][1];
    const double det = j00 * j11 - j01 * j10;
    const double i00 = j11 / det, i01 = -j01 / det, i10 = -j10 / det, i11 = j00 / det;
    double g[3][2];
    g[1][0] = i00; g[1][1] = i01; g[2][0] = i10; g[2][1] = i11;
    g[0][0] = -(i00 + i10); g[0][1] = -(i01 + i11);
    const double area = 0.5 * fabs(det);
    for (int a = 0; a < 3; ++a) {
        for (int b = 0; b < 3; ++b) Ke[(int64_t)(a * 3 + b) * E + c] = area * (g[a][0] * g[b][0] + g[a][1] * g[b][1]);
        Me[(int64_t)a * E + c] = area / 3.0;
    }
}

__global__ void k_gather_scalar_matrix(int nv2, int64_t nnz_node, int64_t E, const int32_t* __restrict__ seg_ptr,
                                       const int32_t* __restrict__ seg_src, const double* __restrict__ Ke,
                                       double* __restrict__ vals) {
    const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= nnz_node) return;
    double acc = 0.0;
    for (int t = seg_ptr[s]; t < seg_ptr[s + 1]; ++t) {
        const int src = seg_src[t];
        const int64_t c = src / nv2;
        const int ab = src - (int)c * nv2;
        acc += Ke[(int64_t)ab * E + c];
    }
    vals[s] = acc;
}

__global__ void k_gather_scalar_vector(int n, int nv, int64_t E, const int32_t* __restrict__ seg_ptr,
                                       const int32_t* __restrict__ seg_src, const double* __restrict__ Me,
                                       double* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double acc = 0.0;
    for (int t = seg_ptr[i]; t < seg_ptr[i + 1]; ++t) {
        const int src = seg_src[t];
        const int64_t c = src / nv;
        const int a = src - (int)c * nv;
        acc += Me[(int64_t)a * E + c];
    }
    out[i] = acc;
}

// ---------------------------------------------------------------------------
// setup kernels: cell->slot positions, gather segments
// ---------------------------------------------------------------------------
__global__ void k_rowof(int n, const int32_t* __restrict__ nrowptr, int32_t* __restrict__ rowof,
                        const int32_t* __restrict__ ncol, int32_t* __restrict__ diagslot) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int s = nrowptr[i]; s < nrowptr[i + 1]; ++s) {
        rowof[s] = i;
        if (ncol[s] == i) diagslot[i] = s;
    }
}

__global__ void k_cellpos(int E, int nv, const int32_t* __restrict__ cells, const int32_t* __restrict__ nrowptr,
                          const int32_t* __restrict__ ncol, int32_t* __restrict__ cellpos,
                          int32_t* __restrict__ mcount, int32_t* __restrict__ vcount, int* __restrict__ bad) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= E) return;
    int v[4];
    for (int a = 0; a < nv; ++a) v[a] = cells[nv * (int64_t)c + a];
    for (int a = 0; a < nv; ++a) {
        const int r0 = nrowptr[v[a]], r1 = nrowptr[v[a] + 1];
        atomicAdd(&vcount[v[a]], 1);
        for (int b = 0; b < nv; ++b) {
            int lo = r0, hi = r1 - 1, pos = -1;
            while (lo <= hi) {
                const int mid = (lo + hi) >> 1;
                const int cv = ncol[mid];
                if (cv == v[b]) { pos = mid; break; }
                if (cv < v[b]) lo = mid + 1; else hi = mid - 1;
            }
            if (pos < 0) { atomicExch(bad, 1); pos = r0; }
            cellpos[(int64_t)c * nv * nv + a * nv + b] = pos;
            atomicAdd(&mcount[pos], 1);
        }
    }
}

__global__ void k_fill_segments(int E, int nv, const int32_t* __restrict__ cells, const int32_t* __restrict__ cellpos,
                                const int32_t* __restrict__ mptr, const int32_t* __restrict__ vptr,
                                int32_t* __restrict__ mfill, int32_t* __restrict__ vfill,
                                int32_t* __restrict__ msrc, int32_t* __restrict__ vsrc) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= E) return;
    const int nv2 = nv * nv;
    for (int a = 0; a < nv; ++a) {
        const int va = cells[nv * (int64_t)c + a];
        const int k = atomicAdd(&vfill[va], 1);
        vsrc[vptr[va] + k] = c * nv + a;
        for (int b = 0; b < nv; ++b) {
            const int pos = cellpos[(int64_t)c * nv2 + a * nv + b];
            const int kk = atomicAdd(&mfill[pos], 1);
            msrc[mptr[pos] + kk] = c * nv2 + a * nv + b;
        }
    }
}

// sort each (short) segment so that the summation order is fixed
__global__ void k_sort_segments(int64_t nseg, const int32_t* __restrict__ ptr, int32_t* __restrict__ src) {
    const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= nseg) return;
    const int b0 = ptr[s], b1 = ptr[s + 1];
    for (int i = b0 + 1; i < b1; ++i) {
        const int key = src[i];
        int j = i - 1;
        while (j >= b0 && src[j] > key) { src[j + 1] = src[j]; --j; }
        src[j + 1] = key;
    }
}

__global__ void k_pattern(int n, int64_t nnz_node, const int32_t* __restrict__ nrowptr,
                          const int32_t* __restrict__ ncol, int64_t* __restrict__ rowptr,
                          int32_t* __restrict__ colind) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    if (i == n) { rowptr[3 * (int64_t)n] = 9 * nnz_node; return; }
    const int r0 = nrowptr[i];
    const int deg = nrowptr[i + 1] - r0;
    const int64_t ru0 = 6 * (int64_t)r0, ru1 = ru0 + 3 * deg, rp = 6 * nnz_node + 3 * (int64_t)r0;
    rowptr[2 * (int64_t)i] = ru0;
    rowptr[2 * (int64_t)i + 1] = ru1;
    rowptr[2 * (int64_t)n + i] = rp;
    for (int t = 0; t < deg; ++t) {
        const int j = ncol[r0 + t];
        colind[ru0 + 2 * t] = 2 * j;     colind[ru0 + 2 * t + 1] = 2 * j + 1; colind[ru0 + 2 * deg + t] = 2 * n + j;
        colind[ru1 + 2 * t] = 2 * j;     colind[ru1 + 2 * t + 1] = 2 * j + 1; colind[ru1 + 2 * deg + t] = 2 * n + j;
        colind[rp + 2 * t] = 2 * j;      colind[rp + 2 * t + 1] = 2 * j + 1;  colind[rp + 2 * deg + t] = 2 * n + j;
    }
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
static int upload_constants(hemo_ctx* ctx) {
    if (!ctx->rules_dirty) return 0;
    for (int r = 0; r < HEMO_NRULES; ++r)
        if (!ctx->have_rule[r]) HEMO_FAIL(ctx, HEMO_ESTATE, "quadrature rule missing for a block form");
    if (!ctx->have_par) HEMO_FAIL(ctx, HEMO_ESTATE, "hemo_set_params not called");
    HEMO_CHECK_CUDA(ctx, cudaMemcpyToSymbolAsync(c_rules, ctx->rules, sizeof(HemoRule) * HEMO_NRULES, 0,
                                                 cudaMemcpyHostToDevice, ctx->stream));
    HEMO_CHECK_CUDA(ctx, cudaMemcpyToSymbolAsync(c_frule, &ctx->frule, sizeof(HemoFacetRule), 0,
                                                 cudaMemcpyHostToDevice, ctx->stream));
    hemo_form_finalize(ctx->par);
    HEMO_CHECK_CUDA(ctx, cudaMemcpyToSymbolAsync(c_par, &ctx->par, sizeof(HemoForm), 0,
                                                 cudaMemcpyHostToDevice, ctx->stream));
    // constants are read by kernels on the same stream, in order
    ctx->rules_dirty = false;
    return 0;
}

int hemo_cc_cells(hemo_ctx* ctx, const double* x_dev, const double* un_dev, int jac_mode);   // assembly_curlcurl.cu
int hemo_cc_lift2d(hemo_ctx* ctx);

extern "C" int hemo_set_formulation(hemo_ctx* ctx, int formulation) {
    if (!ctx || (formulation != HEMO_FORM_STANDARD && formulation != HEMO_FORM_CURLCURL)) return HEMO_EINVAL;
    ctx->formulation = formulation;
    return 0;
}

extern "C" int hemo_set_cell_type(hemo_ctx* ctx, int cell_type) {
    if (!ctx || (cell_type != HEMO_CELL_TRIANGLE && cell_type != HEMO_CELL_QUADRILATERAL &&
                 cell_type != HEMO_CELL_TETRAHEDRON && cell_type != HEMO_CELL_TRIANGLE_P2))
        return HEMO_EINVAL;
    const int nv = (cell_type == HEMO_CELL_TRIANGLE) ? 3 : (cell_type == HEMO_CELL_TRIANGLE_P2 ? 6 : 4);
    const int dim = (cell_type == HEMO_CELL_TETRAHEDRON) ? 3 : 2;
    if (nv == ctx->nv && dim == ctx->dim) return 0;
    // a different cell type invalidates the mesh, the node graph tables and the rules
    ctx->nv = nv;
    ctx->dim = dim;
    ctx->cells = nullptr; ctx->x = nullptr; ctx->h = nullptr; ctx->nrowptr = nullptr; ctx->ncol = nullptr;
    ctx->n = ctx->E = 0;
    for (int r = 0; r < HEMO_NRULES; ++r) ctx->have_rule[r] = false;
    ctx->rules_dirty = ctx->qrules_dirty = true;
    // facet sets (local facet numbering) and Dirichlet cell flags belong to the old mesh
    for (int s = 0; s < HEMO_MAX_FACET_SETS; ++s) {
        HemoFacetSet& fs = ctx->fsets[s];
        cudaFree(fs.cells); cudaFree(fs.mask);
        fs.cells = fs.mask = nullptr;
        fs.m = 0;
    }
    ctx->have_bc = false;
    // solver buffers and captured graphs are sized by (dim, n): reallocated by the next hemo_pc_setup / hemo_fgmres
    hemo_drop_solver_state(ctx);
    return 0;
}

extern "C" int hemo_set_mesh(hemo_ctx* ctx, const double* x_dev, int n_nodes, const int32_t* cells_dev,
                             int n_cells, const double* h_dev) {
    if (!ctx || !x_dev || !cells_dev || !h_dev || n_nodes <= 0 || n_cells <= 0)
        return HEMO_EINVAL;
    const int64_t nv2 = (int64_t)ctx->nv * ctx->nv;
    if ((int64_t)n_cells * 9 * nv2 >= ((int64_t)1 << 40)) HEMO_FAIL(ctx, HEMO_EINVAL, "mesh too large");
    if ((int64_t)n_cells * nv2 >= ((int64_t)1 << 31)) HEMO_FAIL(ctx, HEMO_EINVAL, "n_cells*nv^2 exceeds int32 gather index");
    if (ctx->n != n_nodes || ctx->E != n_cells) {
        // a context re-used with another mesh: nothing sized by the old one may survive (Krylov basis,
        // preconditioner vectors, captured graphs, node-graph tables, Dirichlet flags, facet sets)
        hemo_drop_solver_state(ctx);
        ctx->nrowptr = nullptr; ctx->ncol = nullptr; ctx->nnz_node = 0;
        ctx->have_bc = false;
        for (int s = 0; s < HEMO_MAX_FACET_SETS; ++s) {
            HemoFacetSet& fs = ctx->fsets[s];
            cudaFree(fs.cells); cudaFree(fs.mask);
            fs.cells = fs.mask = nullptr;
            fs.m = 0;
        }
    }
    ctx->x = x_dev; ctx->cells = cells_dev; ctx->h = h_dev;
    ctx->n = n_nodes; ctx->E = n_cells;
    int rc;
    cudaFree(ctx->Ae); cudaFree(ctx->Fe);
    ctx->Ae = ctx->Fe = nullptr;
    ctx->Ae_count = ctx->Fe_count = 0;
    const size_t ndof = (size_t)(ctx->dim + 1) * n_nodes;
    if ((rc = hemo_alloc(ctx, &ctx->dvec, ndof))) return rc;
    HEMO_CHECK_CUDA(ctx, cudaMemsetAsync(ctx->dvec, 0, sizeof(double) * ndof, ctx->stream));
    return 0;
}

// A context that only carries a scalar operator on an abstract graph (no mesh): the replicated coarse space of the
// multi-GPU pressure preconditioner.  Only the pressure-hierarchy entry points work on it.
extern "C" int hemo_set_graph(hemo_ctx* ctx, int n, const int32_t* rowptr_dev, const int32_t* col_dev, int64_t nnz) {
    if (!ctx || n <= 0 || !rowptr_dev || !col_dev || nnz <= 0 || nnz >= ((int64_t)1 << 31)) return HEMO_EINVAL;
    if (ctx->n != n) hemo_drop_solver_state(ctx);
    ctx->x = nullptr; ctx->cells = nullptr; ctx->h = nullptr; ctx->E = 0;
    ctx->n = n;
    ctx->nrowptr = rowptr_dev; ctx->ncol = col_dev; ctx->nnz_node = nnz;
    ctx->have_bc = false;
    int rc;
    if ((rc = hemo_alloc(ctx, &ctx->rowof, (size_t)nnz))) return rc;
    if ((rc = hemo_alloc(ctx, &ctx->diagslot, (size_t)n))) return rc;
    HEMO_CHECK_CUDA(ctx, cudaMemsetAsync(ctx->diagslot, 0xff, sizeof(int32_t) * n, ctx->stream));
    k_rowof<<<hemo_grid(n, 256), 256, 0, ctx->stream>>>(n, rowptr_dev, ctx->rowof, col_dev, ctx->diagslot);
    HEMO_LAUNCH_CHECK(ctx);
    return 0;
}

extern "C" int hemo_set_node_graph(hemo_ctx* ctx, const int32_t* nrowptr_dev, const int32_t* ncol_dev,
                                   int64_t nnz_node) {
    if (!ctx || !nrowptr_dev || !ncol_dev || nnz_node <= 0) return HEMO_EINVAL;
    if (!ctx->cells) HEMO_FAIL(ctx, HEMO_ESTATE, "hemo_set_mesh must precede hemo_set_node_graph");
    if (nnz_node * 9 >= ((int64_t)1 << 40) || nnz_node >= ((int64_t)1 << 31))
        HEMO_FAIL(ctx, HEMO_EINVAL, "node graph too large for int32 slots");
    ctx->nrowptr = nrowptr_dev; ctx->ncol = ncol_dev; ctx->nnz_node = nnz_node;
    const int n = ctx->n, E = ctx->E, nv = ctx->nv;
    const size_t nv2 = (size_t)nv * nv;
    int rc;
    if ((rc = hemo_alloc(ctx, &ctx->rowof, (size_t)nnz_node))) return rc;
    if ((rc = hemo_alloc(ctx, &ctx->diagslot, (size_t)n))) return rc;
    if ((rc = hemo_alloc(ctx, &ctx->cellpos, nv2 * E))) return rc;
    if ((rc = hemo_alloc(ctx, &ctx->mseg_ptr, (size_t)nnz_node + 1))) return rc;
    if ((rc = hemo_alloc(ctx, &ctx->mseg_src, nv2 * E))) return rc;
    if ((rc = hemo_alloc(ctx, &ctx->vseg_ptr, (size_t)n + 1))) return rc;
    if ((rc = hemo_alloc(ctx, &ctx->vseg_src, (size_t)nv * E))) return rc;
    int32_t *mcount = nullptr, *vcount = nullptr;
    int* bad = nullptr;
    if ((rc = hemo_alloc(ctx, &mcount, (size_t)nnz_node + 1))) return rc;
    if ((rc = hemo_alloc(ctx, &vcount, (size_t)n + 1))) return rc;
    if ((rc = hemo_alloc(ctx, &bad, 1))) return rc;
    cudaStream_t st = ctx->stream;
    HEMO_CHECK_CUDA(ctx, cudaMemsetAsync(mcount, 0, sizeof(int32_t) * (nnz_node + 1), st));
    HEMO_CHECK_CUDA(ctx, cudaMemsetAsync(vcount, 0, sizeof(int32_t) * (n + 1), st));
    HEMO_CHECK_CUDA(ctx, cudaMemsetAsync(bad, 0, sizeof(int), st));
    HEMO_CHECK_CUDA(ctx, cudaMemsetAsync(ctx->diagslot, 0xff, sizeof(int32_t) * n, st));
    k_rowof<<<hemo_grid(n, 256), 256, 0, st>>>(n, nrowptr_dev, ctx->rowof, ncol_dev, ctx->diagslot);
    HEMO_LAUNCH_CHECK(ctx);
    k_cellpos<<<hemo_grid(E, 256), 256, 0, st>>>(E, nv, ctx->cells, nrowptr_dev, ncol_dev, ctx->cellpos, mcount, vcount, bad);
    HEMO_LAUNCH_CHECK(ctx);
    // exclusive scans
    void* tmp = nullptr;
    size_t tmp_bytes = 0, tb2 = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, mcount, ctx->mseg_ptr, (int)(nnz_node + 1), st);
    cub::DeviceScan::ExclusiveSum(nullptr, tb2, vcount, ctx->vseg_ptr, n + 1, st);
    if (tb2 > tmp_bytes) tmp_bytes = tb2;
    HEMO_CHECK_CUDA(ctx, cudaMalloc(&tmp, tmp_bytes));
    HEMO_CHECK_CUDA(ctx, cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, mcount, ctx->mseg_ptr, (int)(nnz_node + 1), st));
    HEMO_CHECK_CUDA(ctx, cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, vcount, ctx->vseg_ptr, n + 1, st));
    ctx->launches += 2;
    HEMO_CHECK_CUDA(ctx, cudaMemsetAsync(mcount, 0, sizeof(int32_t) * (nnz_node + 1), st));
    HEMO_CHECK_CUDA(ctx, cudaMemsetAsync(vcount, 0, sizeof(int32_t) * (n + 1), st));
    k_fill_segments<<<hemo_grid(E, 256), 256, 0, st>>>(E, nv, ctx->cells, ctx->cellpos, ctx->mseg_ptr, ctx->vseg_ptr,
                                                       mcount, vcount, ctx->mseg_src, ctx->vseg_src);
    HEMO_LAUNCH_CHECK(ctx);
    k_sort_segments<<<hemo_grid(nnz_node, 256), 256, 0, st>>>(nnz_node, ctx->mseg_ptr, ctx->mseg_src);
    HEMO_LAUNCH_CHECK(ctx);
    k_sort_segments<<<hemo_grid(n, 256), 256, 0, st>>>(n, ctx->vseg_ptr, ctx->vseg_src);
    HEMO_LAUNCH_CHECK(ctx);
    int bad_h = 0;
    HEMO_CHECK_CUDA(ctx, cudaMemcpyAsync(&bad_h, bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(st));
    cudaFree(tmp); cudaFree(mcount); cudaFree(vcount); cudaFree(bad);
    if (bad_h) HEMO_FAIL(ctx, HEMO_EINVAL, "node graph does not contain every cell edge");
    return 0;
}

extern "C" int hemo_matrix_nnz(hemo_ctx* ctx, int64_t* nnz) {
    if (!ctx || !nnz) return HEMO_EINVAL;
    if (!ctx->nrowptr) HEMO_FAIL(ctx, HEMO_ESTATE, "node graph not set");
    *nnz = (int64_t)(ctx->dim + 1) * (ctx->dim + 1) * ctx->nnz_node;
    return 0;
}

extern "C" int hemo_get_pattern(hemo_ctx* ctx, int64_t* rowptr_dev, int32_t* colind_dev) {
    if (!ctx || !rowptr_dev || !colind_dev) return HEMO_EINVAL;
    if (!ctx->nrowptr) HEMO_FAIL(ctx, HEMO_ESTATE, "node graph not set");
    if (ctx->dim == 3) return hemo_tet_pattern(ctx, rowptr_dev, colind_dev);
    k_pattern<<<hemo_grid(ctx->n + 1, 256), 256, 0, ctx->stream>>>(ctx->n, ctx->nnz_node, ctx->nrowptr, ctx->ncol,
                                                                   rowptr_dev, colind_dev);
    HEMO_LAUNCH_CHECK(ctx);
    return 0;
}

// Quadrilateral rules: points on [0,1]^2 and weights as given.  alias = lowest block id of the
// same group (residual forms F_u, F_p | Jacobian forms J_uu..J_pp) with an identical rule, so a
// rule shared by several block forms is integrated once.
static int set_quadrature_quad(hemo_ctx* ctx, int block, const double* pts, const double* wts, int nq) {
    if (nq > HEMO_MAXQ_QUAD) HEMO_FAIL(ctx, HEMO_EINVAL, "too many quadrature points for a quadrilateral rule");
    if (!ctx->qrules) {
        ctx->qrules = (HemoQuadRule*)calloc(HEMO_NRULES, sizeof(HemoQuadRule));
        if (!ctx->qrules) HEMO_FAIL(ctx, HEMO_EINVAL, "out of host memory");
    }
    HemoQuadRule& r = ctx->qrules[block];
    r.nq = nq;
    for (int q = 0; q < nq; ++q) { r.pt[q][0] = pts[2 * q]; r.pt[q][1] = pts[2 * q + 1]; r.pt[q][2] = wts[q]; }
    ctx->have_rule[block] = true;
    ctx->qrules_dirty = true;
    hemo_quad_rule_aliases(ctx->qrules, ctx->have_rule, HEMO_NRULES);
    return 0;
}

extern "C" int hemo_set_quadrature(hemo_ctx* ctx, int block, const double* pts, const double* wts, int nq) {
    if (!ctx || block < 0 || block >= HEMO_NRULES || !pts || !wts || nq <= 0) return HEMO_EINVAL;
    ctx->rule_version++;
    if (ctx->dim == 3) return hemo_tet_set_quadrature(ctx, block, pts, wts, nq);
    if (ctx->nv == 4) return set_quadrature_quad(ctx, block, pts, wts, nq);
    if (ctx->nv == 6) return hemo_p2_set_quadrature(ctx, block, pts, wts, nq);
    if (nq > HEMO_MAXQ) return HEMO_EINVAL;
    HemoRule& r = ctx->rules[block];
    r.nq = nq;
    r.m0 = 0.0;
    for (int i = 0; i < 3; ++i) r.m1[i] = 0.0;
    for (int i = 0; i < 6; ++i) r.m2[i] = 0.0;
    for (int q = 0; q < nq; ++q) {
        const double xi = pts[2 * q], eta = pts[2 * q + 1];
        const double phi[3] = {1.0 - xi - eta, xi, eta};
        for (int a = 0; a < 3; ++a) r.phi[q][a] = phi[a];
        r.w[q] = wts[q];
        r.m0 += wts[q];
        for (int a = 0; a < 3; ++a) r.m1[a] += wts[q] * phi[a];
        r.m2[0] += wts[q] * phi[0] * phi[0];
        r.m2[1] += wts[q] * phi[1] * phi[1];
        r.m2[2] += wts[q] * phi[2] * phi[2];
        r.m2[3] += wts[q] * phi[0] * phi[1];
        r.m2[4] += wts[q] * phi[0] * phi[2];
        r.m2[5] += wts[q] * phi[1] * phi[2];
    }
    ctx->have_rule[block] = true;
    ctx->rules_dirty = true;
    // alias = lowest-numbered block whose rule is identical
    for (int b = 0; b < HEMO_NRULES; ++b) {
        if (!ctx->have_rule[b]) continue;
        HemoRule& rb = ctx->rules[b];
        rb.alias = b;
        for (int a = 0; a < b; ++a) {
            if (!ctx->have_rule[a] || ctx->rules[a].nq != rb.nq) continue;
            bool same = true;
            for (int q = 0; q < rb.nq && same; ++q)
                same = ctx->rules[a].w[q] == rb.w[q] && ctx->rules[a].phi[q][1] == rb.phi[q][1] &&
                       ctx->rules[a].phi[q][2] == rb.phi[q][2];
            if (same) { rb.alias = a; break; }
        }
    }
    return 0;
}

extern "C" int hemo_set_facet_quadrature(hemo_ctx* ctx, const double* pts, const double* wts, int nq) {
    if (!ctx || !pts || !wts || nq <= 0) return HEMO_EINVAL;
    ctx->rule_version++;
    if (ctx->dim == 3) return hemo_tet_set_facet_quadrature(ctx, pts, wts, nq);   // (s, t) pairs on the reference triangle
    if (nq > HEMO_MAXFQ) return HEMO_EINVAL;
    ctx->frule.nq = nq;
    for (int q = 0; q < nq; ++q) { ctx->frule.s[q] = pts[q]; ctx->frule.w[q] = wts[q]; }
    ctx->rules_dirty = true;
    ctx->qrules_dirty = true;
    return 0;
}

extern "C" int hemo_set_params(hemo_ctx* ctx, const hemo_params* p) {
    if (!ctx || !p || !(p->dt > 0) || !(p->rho > 0) || !(p->mu > 0)) return HEMO_EINVAL;
    ctx->par.dt = p->dt; ctx->par.rho = p->rho; ctx->par.mu = p->mu;
    ctx->par.f[0] = p->f[0]; ctx->par.f[1] = p->f[1];
    ctx->par.eps0 = p->eps0;
    ctx->have_par = true;
    ctx->rules_dirty = true;
    ctx->qrules_dirty = true;
    return 0;
}

extern "C" int hemo_set_time_scheme(hemo_ctx* ctx, double theta, double a0, const double* uh_dev) {
    if (!ctx || !(theta > 0.0) || !(theta <= 1.0) || !(a0 > 0.0)) return HEMO_EINVAL;
    ctx->par.theta = theta;
    ctx->par.a0 = a0;
    ctx->uh = uh_dev;
    ctx->rules_dirty = true;
    ctx->qrules_dirty = true;
    return 0;
}

extern "C" int hemo_set_body_force3(hemo_ctx* ctx, const double* f3_host) {
    if (!ctx || !f3_host) return HEMO_EINVAL;
    ctx->par.f[0] = f3_host[0]; ctx->par.f[1] = f3_host[1]; ctx->fz = f3_host[2];
    ctx->rules_dirty = ctx->qrules_dirty = true;
    return 0;
}

extern "C" int hemo_set_facet_set(hemo_ctx* ctx, int set_id, const int32_t* cells_dev, const int32_t* mask_dev,
                                  int m, const hemo_facet_coef* coef) {
    if (ctx) ctx->fset_version++;
    if (!ctx || set_id < 0 || set_id >= HEMO_MAX_FACET_SETS || m < 0) return HEMO_EINVAL;
    HemoFacetSet& fs = ctx->fsets[set_id];
    if (fs.cells) { cudaFree(fs.cells); fs.cells = nullptr; }
    if (fs.mask) { cudaFree(fs.mask); fs.mask = nullptr; }
    fs.m = 0;
    if (m == 0) return 0;
    if (!cells_dev || !mask_dev || !coef) return HEMO_EINVAL;
    int rc;
    if ((rc = hemo_upload(ctx, &fs.cells, cells_dev, (size_t)m, true))) return rc;
    if ((rc = hemo_upload(ctx, &fs.mask, mask_dev, (size_t)m, true))) return rc;
    fs.m = m;
    fs.coef = *coef;
    if ((rc = hemo_ensure_reduce(ctx, (size_t)m, 8))) return rc;
    return 0;
}

extern "C" int hemo_set_facet_coef(hemo_ctx* ctx, int set_id, const hemo_facet_coef* coef) {
    if (!ctx || set_id < 0 || set_id >= HEMO_MAX_FACET_SETS || !coef) return HEMO_EINVAL;
    ctx->fsets[set_id].coef = *coef;
    return 0;
}

extern "C" int hemo_set_bc(hemo_ctx* ctx, const uint8_t* dofflag_dev, const double* dofmult_dev,
                           const uint8_t* cellflag_dev) {
    if (!ctx) return HEMO_EINVAL;
    if (!ctx->cells) HEMO_FAIL(ctx, HEMO_ESTATE, "hemo_set_mesh must precede hemo_set_bc");
    if (!dofflag_dev) {
        ctx->have_bc = false;
        return 0;
    }
    if (!dofmult_dev || !cellflag_dev) return HEMO_EINVAL;
    int rc;
    const size_t ndof = (size_t)(ctx->dim + 1) * ctx->n;       // [u (dim n) | p (n)]
    if ((rc = hemo_upload(ctx, &ctx->dofflag, dofflag_dev, ndof, true))) return rc;
    if ((rc = hemo_upload(ctx, &ctx->dofmult, dofmult_dev, ndof, true))) return rc;
    if ((rc = hemo_upload(ctx, &ctx->cellflag, cellflag_dev, (size_t)ctx->E, true))) return rc;
    ctx->have_bc = true;
    return 0;
}

// element buffers are allocated on first use (a context that only serves the pressure
// Laplacian never pays for the 81*E Jacobian buffer)
int hemo_ensure_elem(hemo_ctx* ctx, size_t ae_count, size_t fe_count);
static int ensure_elem(hemo_ctx* ctx, size_t ae_count, size_t fe_count) { return hemo_ensure_elem(ctx, ae_count, fe_count); }
int hemo_ensure_elem(hemo_ctx* ctx, size_t ae_count, size_t fe_count) {
    int rc;
    if (ae_count > ctx->Ae_count) {
        if ((rc = hemo_alloc(ctx, &ctx->Ae, ae_count))) return rc;
        ctx->Ae_count = ae_count;
    }
    if (fe_count > ctx->Fe_count) {
        if ((rc = hemo_alloc(ctx, &ctx->Fe, fe_count))) return rc;
        ctx->Fe_count = fe_count;
    }
    return 0;
}

// a set whose coefficients are all zero carries no form term (it only tags facets for the
// post-processing kernels): the assembly loops skip it
static bool facet_set_active(const HemoFacetSet& fs) {
    const hemo_facet_coef& c = fs.coef;
    return fs.m > 0 && (c.a_p != 0.0 || c.pconst != 0.0 || c.a_g != 0.0 || c.a_s != 0.0 || c.a_n != 0.0 || c.a_b != 0.0);
}

static int check_ready(hemo_ctx* ctx) {
    if (!ctx->cells || !ctx->nrowptr) HEMO_FAIL(ctx, HEMO_ESTATE, "mesh / node graph not set");
    return ctx->nv == 3 ? upload_constants(ctx) : 0;   // the quadrilateral kernels upload their own tables
}

extern "C" int hemo_assemble_jacobian(hemo_ctx* ctx, const double* x_dev, const double* un_dev, double* vals_dev) {
    if (!ctx || !x_dev || !un_dev || !vals_dev) return HEMO_EINVAL;
    if (ctx->dim == 3) return hemo_tet_assemble_jacobian(ctx, x_dev, un_dev, vals_dev);
    int rc = check_ready(ctx);
    if (rc) return rc;
    const int E = ctx->E, n = ctx->n, nv = ctx->nv;
    if ((rc = ensure_elem(ctx, (size_t)9 * nv * nv * E, 0))) return rc;
    cudaStream_t st = ctx->stream;
    const double* uh = ctx->uh ? ctx->uh : un_dev;
    if (ctx->formulation == HEMO_FORM_CURLCURL) {
        // stabilized_schur_pressurebc.py: cells + facets of the rotational form, then the standard gather
        if ((rc = ensure_elem(ctx, (size_t)9 * nv * nv * E, (size_t)3 * nv * E))) return rc;
        if ((rc = hemo_cc_cells(ctx, x_dev, un_dev, 0))) return rc;
        k_gather_matrix<<<hemo_grid(ctx->nnz_node, 256), 256, 0, st>>>(
            n, nv * nv, ctx->nnz_node, E, ctx->nrowptr, ctx->ncol, ctx->rowof, ctx->mseg_ptr, ctx->mseg_src, ctx->Ae,
            ctx->have_bc ? ctx->dofflag : nullptr, ctx->dofmult, vals_dev);
        HEMO_LAUNCH_CHECK(ctx);
        return 0;
    }
    HEMO_PROF_BEGIN(ctx, HEMO_PROF_CELL_JAC);
    if (nv == 4) {
        if ((rc = hemo_q1_cell_jacobian(ctx, x_dev, un_dev))) return rc;
    } else if (nv == 6) {
        if ((rc = hemo_p2_cell_jacobian(ctx, x_dev, un_dev))) return rc;
    } else {
        k_cell_jacobian<<<hemo_grid(E, 128), 128, 0, st>>>(E, n, ctx->cells, ctx->x, ctx->h, x_dev, un_dev, uh, ctx->Ae);
        HEMO_LAUNCH_CHECK(ctx);
    }
    HEMO_PROF_END(ctx, HEMO_PROF_CELL_JAC);
    for (int s = 0; s < HEMO_MAX_FACET_SETS; ++s) {
        const HemoFacetSet& fs = ctx->fsets[s];
        if (!facet_set_active(fs)) continue;
        if (nv == 4) {
            if ((rc = hemo_q1_facets(ctx, 1, fs, x_dev, un_dev, nullptr))) return rc;
            continue;
        }
        if (nv == 6) {
            if ((rc = hemo_p2_facets(ctx, 1, fs, x_dev, un_dev, nullptr))) return rc;
            continue;
        }
        k_facets<1><<<hemo_grid(fs.m, 128), 128, 0, st>>>(fs.m, E, n, fs.cells, fs.mask, fs.coef, ctx->cells, ctx->x,
                                                          ctx->h, x_dev, un_dev, uh, nullptr, nullptr, ctx->Ae);
        HEMO_LAUNCH_CHECK(ctx);
    }
    HEMO_PROF_BEGIN(ctx, HEMO_PROF_GATHER_MAT);
    k_gather_matrix<<<hemo_grid(ctx->nnz_node, 256), 256, 0, st>>>(
        n, nv * nv, ctx->nnz_node, E, ctx->nrowptr, ctx->ncol, ctx->rowof, ctx->mseg_ptr, ctx->mseg_src, ctx->Ae,
        ctx->have_bc ? ctx->dofflag : nullptr, ctx->dofmult, vals_dev);
    HEMO_LAUNCH_CHECK(ctx);
    HEMO_PROF_END(ctx, HEMO_PROF_GATHER_MAT);
    return 0;
}

extern "C" int hemo_assemble_residual(hemo_ctx* ctx, const double* x_dev, const double* un_dev,
                                      const double* g_dev, double* b_dev) {
    if (!ctx || !x_dev || !un_dev || !b_dev) return HEMO_EINVAL;
    if (ctx->dim == 3) return hemo_tet_assemble_residual(ctx, x_dev, un_dev, g_dev, b_dev);
    if (ctx->have_bc && !g_dev) return HEMO_EINVAL;
    int rc = check_ready(ctx);
    if (rc) return rc;
    const int E = ctx->E, n = ctx->n, nv = ctx->nv;
    if ((rc = ensure_elem(ctx, 0, (size_t)3 * nv * E))) return rc;
    cudaStream_t st = ctx->stream;
    const double* uh = ctx->uh ? ctx->uh : un_dev;
    const uint8_t* cf = ctx->have_bc ? ctx->cellflag : nullptr;
    if (ctx->have_bc) {
        k_lift_vector<<<hemo_grid(3 * (int64_t)n, 256), 256, 0, st>>>(3 * (int64_t)n, ctx->dofflag, x_dev, g_dev, ctx->dvec);
        HEMO_LAUNCH_CHECK(ctx);
    }
    if (ctx->formulation == HEMO_FORM_CURLCURL) {
        // element Jacobians only on Dirichlet-adjacent cells (lifting), like the tetrahedron path
        if ((rc = ensure_elem(ctx, (size_t)9 * nv * nv * E, (size_t)3 * nv * E))) return rc;
        if ((rc = hemo_cc_cells(ctx, x_dev, un_dev, ctx->have_bc ? 1 : 2))) return rc;
        if (ctx->have_bc && (rc = hemo_cc_lift2d(ctx))) return rc;
        k_gather_vector<<<hemo_grid(n, 256), 256, 0, st>>>(n, nv, E, ctx->vseg_ptr, ctx->vseg_src, ctx->Fe,
                                                           ctx->have_bc ? ctx->dofflag : nullptr, x_dev, g_dev, b_dev);
        HEMO_LAUNCH_CHECK(ctx);
        return 0;
    }
    HEMO_PROF_BEGIN(ctx, HEMO_PROF_CELL_RES);
    if (nv == 4) {
        if ((rc = hemo_q1_cell_residual(ctx, x_dev, un_dev, cf))) return rc;
    } else if (nv == 6) {
        if ((rc = hemo_p2_cell_residual(ctx, x_dev, un_dev, cf))) return rc;
    } else {
        k_cell_residual<<<hemo_grid(E, 128), 128, 0, st>>>(E, n, ctx->cells, ctx->x, ctx->h, x_dev, un_dev, uh, cf, ctx->dvec, ctx->Fe);
        HEMO_LAUNCH_CHECK(ctx);
    }
    HEMO_PROF_END(ctx, HEMO_PROF_CELL_RES);
    for (int s = 0; s < HEMO_MAX_FACET_SETS; ++s) {
        const HemoFacetSet& fs = ctx->fsets[s];
        if (!facet_set_active(fs)) continue;
        if (nv == 4) {
            if ((rc = hemo_q1_facets(ctx, 0, fs, x_dev, un_dev, cf))) return rc;
            continue;
        }
        if (nv == 6) {
            if ((rc = hemo_p2_facets(ctx, 0, fs, x_dev, un_dev, cf))) return rc;
            continue;
        }
        k_facets<0><<<hemo_grid(fs.m, 128), 128, 0, st>>>(fs.m, E, n, fs.cells, fs.mask, fs.coef, ctx->cells, ctx->x,
                                                          ctx->h, x_dev, un_dev, uh, cf, ctx->dvec, ctx->Fe);
        HEMO_LAUNCH_CHECK(ctx);
    }
    k_gather_vector<<<hemo_grid(n, 256), 256, 0, st>>>(n, nv, E, ctx->vseg_ptr, ctx->vseg_src, ctx->Fe,
                                                       ctx->have_bc ? ctx->dofflag : nullptr, x_dev, g_dev, b_dev);
    HEMO_LAUNCH_CHECK(ctx);
    return 0;
}

extern "C" int hemo_outlet_flux(hemo_ctx* ctx, int set_id, const double* un_dev, double* q_host) {
    if (!ctx || set_id < 0 || set_id >= HEMO_MAX_FACET_SETS || !un_dev || !q_host) return HEMO_EINVAL;
    const HemoFacetSet& fs = ctx->fsets[set_id];
    if (fs.m == 0) { *q_host = 0.0; return 0; }
    int rc = hemo_ensure_reduce(ctx, (size_t)fs.m, 8);
    if (rc) return rc;
    cudaStream_t st = ctx->stream;
    if (ctx->dim == 3) {
        if ((rc = hemo_tet_facet_flux(ctx, fs, un_dev, ctx->red_partial))) return rc;
    } else if (ctx->nv == 4) {
        if ((rc = hemo_q1_facet_flux(ctx, fs, un_dev, ctx->red_partial))) return rc;
    } else if (ctx->nv == 6) {
        if ((rc = hemo_p2_facet_flux(ctx, fs, un_dev, ctx->red_partial))) return rc;
    } else {
        k_facet_flux<<<hemo_grid(fs.m, 128), 128, 0, st>>>(fs.m, fs.cells, fs.mask, ctx->cells, ctx->x, un_dev, ctx->red_partial);
        HEMO_LAUNCH_CHECK(ctx);
    }
    k_sum_serial<<<1, 256, 0, st>>>(fs.m, ctx->red_partial, ctx->red_out);
    HEMO_LAUNCH_CHECK(ctx);
    HEMO_CHECK_CUDA(ctx, cudaMemcpyAsync(ctx->red_host, ctx->red_out, sizeof(double), cudaMemcpyDeviceToHost, st));
    HEMO_CHECK_CUDA(ctx, cudaStreamSynchronize(st));
    *q_host = ctx->red_host[0];
    return 0;
}

extern "C" int hemo_assemble_laplace_mass(hemo_ctx* ctx, double* lap_vals_dev, double* mass_dev) {
    if (!ctx || !lap_vals_dev || !mass_dev) return HEMO_EINVAL;
    if (!ctx->cells || !ctx->nrowptr) HEMO_FAIL(ctx, HEMO_ESTATE, "mesh / node graph not set");
    const int E = ctx->E, n = ctx->n, nv = ctx->nv;
    int rc;
    if ((rc = ensure_elem(ctx, (size_t)nv * nv * E, (size_t)nv * E))) return rc;
    cudaStream_t st = ctx->stream;
    // reuse the element buffers: Ke -> Ae[0..nv*nv*E), Me -> Fe[0..nv*E)
    if (ctx->dim == 3) {
        if ((rc = hemo_tet_laplace_mass(ctx))) return rc;
    } else if (nv == 4) {
        if ((rc = hemo_q1_laplace_mass(ctx))) return rc;
    } else if (nv == 6) {
        if ((rc = hemo_p2_laplace_mass(ctx))) return rc;
    } else {
        k_cell_laplace<<<hemo_grid(E, 256), 256, 0, st>>>(E, ctx->cells, ctx->x, ctx->Ae, ctx->Fe);
        HEMO_LAUNCH_CHECK(ctx);
    }
    k_gather_scalar_matrix<<<hemo_grid(ctx->nnz_node, 256), 256, 0, st>>>(nv * nv, ctx->nnz_node, E, ctx->mseg_ptr,
                                                                          ctx->mseg_src, ctx->Ae, lap_vals_dev);
    HEMO_LAUNCH_CHECK(ctx);
    k_gather_scalar_vector<<<hemo_grid(n, 256), 256, 0, st>>>(n, nv, E, ctx->vseg_ptr, ctx->vseg_src, ctx->Fe, mass_dev);
    HEMO_LAUNCH_CHECK(ctx);
    return 0;
}

// SELFP: Sp = A11 - A10 diag(A00)^-1 A01 on the distance-2 node graph, straight from the
// monolithic Jacobian values (PETSc MatSchurComplementGetPmat with SELFP, reference
// src/solvers/stabilized_schur.py:235).  One thread per Sp entry.
__device__ __forceinline__ int find_sorted(const int32_t* __restrict__ col, int lo, int hi, int key) {
    int a = lo, b = hi - 1;
    while (a <= b) {
        const int m = (a + b) >> 1;
        const int c = col[m];
        if (c == key) return m;
        if (c < key) a = m + 1; else b = m - 1;
    }
    return -1;
}

__global__ void __launch_bounds__(256)
k_selfp(int64_t nnz2, int64_t nnz_node, const int32_t* __restrict__ rowof2, const int32_t* __restrict__ col2,
        const int32_t* __restrict__ nrowptr, const int32_t* __restrict__ ncol, const int32_t* __restrict__ diagslot,
        const double* __restrict__ vals, areal* __restrict__ out) {
    const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= nnz2) return;
    const int i = rowof2[s], j = col2[s];
    const int r0i = nrowptr[i];
    const int degi = nrowptr[i + 1] - r0i;
    const int64_t rpi = 6 * nnz_node + 3 * (int64_t)r0i;
    double v = 0.0;
    const int tij = find_sorted(ncol, r0i, r0i + degi, j);
    if (tij >= 0) v = vals[rpi + 2 * degi + (tij - r0i)];             // A11[i, j]
    for (int t = 0; t < degi; ++t) {
        const int k = ncol[r0i + t];
        const int r0k = nrowptr[k];
        const int degk = nrowptr[k + 1] - r0k;
        const int tkj = find_sorted(ncol, r0k, r0k + degk, j);
        if (tkj < 0) continue;
        const int tkk = diagslot[k] - r0k;
        const int64_t ru0 = 6 * (int64_t)r0k, ru1 = ru0 + 3 * degk;
        const double a10x = vals[rpi + 2 * t], a10y = vals[rpi + 2 * t + 1];        // A10[i, (k, x|y)]
        const double a01x = vals[ru0 + 2 * degk + (tkj - r0k)];                     // A01[(k, x), j]
        const double a01y = vals[ru1 + 2 * degk + (tkj - r0k)];
        const double dx = vals[ru0 + 2 * tkk], dy = vals[ru1 + 2 * tkk + 1];        // diag(A00)
        v -= a10x * a01x / dx + a10y * a01y / dy;
    }
    out[s] = (areal)v;
}

extern "C" int hemo_pc_set_schur_selfp(hemo_ctx* ctx, const double* vals_dev, double coarse_shift) {
    if (!ctx || !vals_dev) return HEMO_EINVAL;
    HemoAmg& amg = ctx->amg[1];
    if (!amg.ready || !amg.fine_rowptr) HEMO_FAIL(ctx, HEMO_ESTATE, "pressure hierarchy needs the distance-2 fine pattern");
    if (ctx->dim == 3) {
        int rc = hemo_tet_selfp(ctx, vals_dev);
        if (rc) return rc;
        return hemo_amg_numeric_shift(ctx, &amg, coarse_shift);
    }
    k_selfp<<<hemo_grid(amg.fine_nnz, 256), 256, 0, ctx->stream>>>(amg.fine_nnz, ctx->nnz_node, amg.fine_rowof, amg.fine_col,
                                                                   ctx->nrowptr, ctx->ncol, ctx->diagslot, vals_dev,
                                                                   amg.op[0].val);
    HEMO_LAUNCH_CHECK(ctx);
    return hemo_amg_numeric_shift(ctx, &amg, coarse_shift);
}
