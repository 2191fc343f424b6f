"""Float64 model of the aggregation-AMG V-cycle and of the block preconditioner (amg.cu, solver.cu).

The library runs the cycle on single-precision operators and vectors (DESIGN.md §5); this model keeps every vector
operation in float64 and rounds the operator values to float32 exactly where the library stores them: the fine
operators, the intermediate A*P of each Galerkin product and the coarse operator R*(A*P).  What is left between
the two is the single-precision arithmetic of the cycle, so a tolerance a few times that size separates a correct
kernel from a wrong coefficient, a skipped entry or a skipped row.

numpy / scipy only; the prolongators are the ones `fem.amg_setup.build_hierarchy` returns.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp

# Tolerance of the single-precision hierarchies against this model, on both ||e||_2 / ||x_ref||_2 and
# max|e| / max|x_ref| (tests/test_gpu_amg_reference.py).  Measured on a B200: at most 8.1e-7 and 3.4e-7 over every
# configuration of that file, so 1e-5 leaves a factor 12.  tests/test_amg_oracle.py checks that the defects it must
# catch move the model's output by at least ten times the tolerance.
AMG_TOL = 1e-5

# levels handled by a fused coarse V-cycle kernel that have at most this many nodes pre-smooth with the full
# Chebyshev degree (HEMO_FUSE_MAX_NODES in hemo_internal.cuh: every level of the one-CTA kernel)
STRONG_PRE_NODES = 256


def f32(A: sp.spmatrix) -> sp.csr_matrix:
    """The values of A as the library stores them (float32), held in float64."""
    A = sp.csr_matrix(A, copy=True)
    A.data = A.data.astype(np.float32).astype(np.float64)
    return A


def _identity_rows_cols(A: sp.spmatrix, flag: np.ndarray) -> sp.csr_matrix:
    """Rows and columns of the flagged dofs replaced by those of the identity (the pattern is kept)."""
    A = sp.coo_matrix(A)
    hit = flag[A.row] | flag[A.col]
    data = np.where(hit, (A.row == A.col).astype(np.float64), A.data)
    return sp.csr_matrix((data, (A.row, A.col)), shape=A.shape)


def velocity_level0(J: sp.spmatrix, n: int, node_mask: np.ndarray | None = None) -> sp.csr_matrix:
    """A00 (2x2 node blocks, dofs 2i+k) of the monolithic [u | p] Jacobian, as k_extract_a00 stores it: nodes flagged
    by the preconditioner mask get identity block rows and columns."""
    A = sp.csr_matrix(J)[:2 * n, :2 * n]
    if node_mask is not None:
        A = _identity_rows_cols(A, np.repeat(np.asarray(node_mask, dtype=bool), 2))
    return f32(A)


def a01_block(J: sp.spmatrix, n: int) -> sp.csr_matrix:
    """A01 as the compact single-precision copy k_extract_a00 writes."""
    return f32(sp.csr_matrix(J)[:2 * n, 2 * n:])


def pressure_level0(lap: sp.spmatrix, p_dirichlet: np.ndarray | None = None) -> sp.csr_matrix:
    """Pressure Laplacian with identity rows and columns on Dirichlet pressure dofs (k_lap_with_bc)."""
    if p_dirichlet is not None and np.any(p_dirichlet):
        lap = _identity_rows_cols(lap, np.asarray(p_dirichlet, dtype=bool))
    return f32(lap)


def chebyshev(matvec, dinv: np.ndarray, lmax: float, ratio: float, b: np.ndarray, x: np.ndarray | None,
              degree: int) -> np.ndarray:
    """`degree` Chebyshev steps on D^-1 A x = D^-1 b for the interval [lmax / ratio, lmax] (textbook form);
    x = None starts from zero.  degree 0 returns the start unchanged."""
    x = np.zeros_like(b) if x is None else x.copy()
    if degree <= 0:
        return x
    lmin = lmax / ratio
    theta, delta = 0.5 * (lmax + lmin), 0.5 * (lmax - lmin)
    sigma = theta / delta
    rho = 1.0 / sigma
    r = dinv * (b - matvec(x))
    d = r / theta
    x = x + d
    for _ in range(1, degree):
        rho_new = 1.0 / (2.0 * sigma - rho)
        r = r - dinv * matvec(d)
        d = rho_new * rho * d + (2.0 * rho_new / delta) * r
        x = x + d
        rho = rho_new
    return x


def chebyshev_error_polynomial(lam: np.ndarray, lmax: float, ratio: float, degree: int) -> np.ndarray:
    """p_k(lam) = T_k((theta - lam) / delta) / T_k(theta / delta): the error factor of `degree` steps."""
    lmin = lmax / ratio
    theta, delta = 0.5 * (lmax + lmin), 0.5 * (lmax - lmin)
    T = np.polynomial.chebyshev.Chebyshev.basis(degree)
    return T((theta - lam) / delta) / T(theta / delta)


class Hierarchy:
    """Level operators, transfers, smoother data and the exact coarsest solve of one hierarchy.

    A0: level-0 operator (already rounded as stored); levels: the dicts of `build_hierarchy` (scalar P, R);
    bs: 2 (velocity) or 1 (pressure); coarse_shift: relative diagonal shift of the coarsest dense solve."""

    def __init__(self, A0: sp.spmatrix, levels, bs: int, coarse_shift: float = 0.0):
        self.bs = bs
        I = sp.identity(bs, format="csr")
        self.ops = [sp.csr_matrix(A0)]
        self.P, self.R = [], []
        for lv in levels:
            P = sp.kron(sp.csr_matrix(lv["P"]), I).tocsr() if bs > 1 else sp.csr_matrix(lv["P"])
            R = sp.kron(sp.csr_matrix(lv["R"]), I).tocsr() if bs > 1 else sp.csr_matrix(lv["R"])
            AP = f32(self.ops[-1] @ P)                 # A*P is stored (fp64 accumulation, fp32 values)
            self.ops.append(f32(R @ AP))
            self.P.append(P)
            self.R.append(R)
        self.dinv, self.lmax = [], []
        for A in self.ops[:-1]:
            d = A.diagonal().copy()
            d[d == 0.0] = 1.0
            self.dinv.append(1.0 / d)
            self.lmax.append(float(np.max(np.asarray(abs(A).sum(axis=1)).ravel() / np.abs(d))))
        M = self.ops[-1].toarray()
        M[np.diag_indices_from(M)] *= 1.0 + coarse_shift
        self.coarse = M

    @property
    def nlev(self) -> int:
        return len(self.ops)

    def nodes(self, l: int) -> int:
        return self.ops[l].shape[0] // self.bs

    # the three operator applications of a cycle; a test may override them to model a defective kernel
    def matvec(self, l: int, x: np.ndarray) -> np.ndarray:
        return self.ops[l] @ x

    def restrict(self, l: int, r: np.ndarray) -> np.ndarray:
        return self.R[l] @ r

    def prolong(self, l: int, xc: np.ndarray) -> np.ndarray:
        return self.P[l] @ xc

    def smooth(self, l, b, x, degree, ratio):
        return chebyshev(lambda v: self.matvec(l, v), self.dinv[l], self.lmax[l], ratio, b, x, degree)

    def cycle(self, l: int, b: np.ndarray, x: np.ndarray | None, *, degree: int, degree_pre: int, ratio: float,
              fused=()) -> np.ndarray:
        """One V-cycle from level l on A_l x = b; x = None starts from zero (coarser levels always do)."""
        if l == self.nlev - 1:
            return np.linalg.solve(self.coarse, b)
        strong = l in fused and self.nodes(l) <= STRONG_PRE_NODES
        x = self.smooth(l, b, x, degree if strong else degree_pre, ratio)
        r = b - self.matvec(l, x)
        xc = self.cycle(l + 1, self.restrict(l, r), None, degree=degree, degree_pre=degree_pre, ratio=ratio, fused=fused)
        x = x + self.prolong(l, xc)
        return self.smooth(l, b, x, degree, ratio)

    def apply(self, b: np.ndarray, ncycles: int = 1, *, degree: int = 2, degree_pre: int = 1, ratio: float = 4.0,
              fused=()) -> np.ndarray:
        """hemo_amg_apply: `ncycles` V-cycles from a zero initial guess; cycle c >= 2 starts from the previous
        top-level iterate.  `fused`: levels that run inside a fused coarse V-cycle kernel."""
        ratio = ratio if ratio > 1.0 else 4.0
        x = None
        for _ in range(max(ncycles, 1)):
            x = self.cycle(0, np.asarray(b, dtype=np.float64), x, degree=degree, degree_pre=degree_pre, ratio=ratio,
                           fused=fused)
        return x


def pc_apply_laplace(r: np.ndarray, n: int, Hu: Hierarchy, Hp: Hierarchy, A01: sp.spmatrix, mass: np.ndarray, *,
                     mass_coef: float, lap_coef: float, cycles_u: int = 1, cycles_p: int = 1,
                     project_pressure: bool = False, p_dirichlet: np.ndarray | None = None,
                     node_mask: np.ndarray | None = None, cycle_kw_u=None, cycle_kw_p=None) -> np.ndarray:
    """hemo_pc_apply in laplace mode: upper block-triangular Schur preconditioner with
    S^-1 ~ mass_coef Mp^-1 + lap_coef Lp^-1 (both V-cycle hierarchies)."""
    ru, rp = r[:2 * n], r[2 * n:]
    tp = rp.copy()
    if node_mask is not None:
        tp[node_mask] = 0.0
    if project_pressure:
        tp -= tp.mean()
    q = Hp.apply(tp, cycles_p, **(cycle_kw_p or {}))
    zp = mass_coef * tp / mass + lap_coef * q
    if p_dirichlet is not None:
        zp[p_dirichlet] = rp[p_dirichlet]
    if project_pressure:
        zp -= zp.mean()
    tu = ru - A01 @ zp
    if node_mask is not None:
        tu.reshape(-1, 2)[node_mask] = 0.0
    zu = Hu.apply(tu, cycles_u, **(cycle_kw_u or {}))
    return np.concatenate([zu, zp])


def rel_errors(x: np.ndarray, ref: np.ndarray) -> tuple[float, float]:
    """(||x - ref||_2 / ||ref||_2, max|x - ref| / max|ref|)."""
    e = x - ref
    return float(np.linalg.norm(e) / np.linalg.norm(ref)), float(np.abs(e).max() / np.abs(ref).max())
