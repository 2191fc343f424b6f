"""Host driver for the linear solve of one Newton iteration.

Mirrors the PETSc objects the reference configures in `Solver.setup`
(reference src/solvers/stabilized_schur.py:226-275): an outer FGMRES and a
Schur-complement block preconditioner, rebuilt for every new Jacobian.
All numerics run in libhemo_sm100.so; this file only sequences calls.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp

from .fem import amg_setup


class BlockSchurSolver:
    """KSP(fgmres) + PC(block Schur, AMG) for the monolithic Jacobian."""

    def __init__(self, hemo, nrowptr: np.ndarray, ncol: np.ndarray, u_dirichlet_nodes: np.ndarray,
                 p_dirichlet_nodes: np.ndarray, *, p_open_nodes: np.ndarray | None = None, dt: float, rho: float, mu: float,
                 restart: int = 60, max_it: int = 1000, rtol: float = 1e-5, atol: float = 1e-50,
                 amg_cycles_u: int = 1, amg_cycles_p: int = 1, cheb_degree: int = 2, cheb_ratio: float = 4.0, cheb_degree_pre: int = 1,
                 project_pressure: bool = False, smooth_prolongator: bool = True, strength_theta: float = 0.08,
                 schur_mass_coef: float | None = None, schur_lap_coef: float | None = None,
                 schur_mode: str = "laplace"):
        # "laplace": S^-1 ~ mu Mp^-1 + (2 rho/dt) Lp^-1 (Cahouet–Chabard, constant operators);
        # "selfp": S^-1 ~ Sp^-1 with the reference's Sp = A11 - A10 diag(A00)^-1 A01, re-formed by every setup()
        if schur_mode not in ("laplace", "selfp"):
            raise ValueError(f"schur_mode {schur_mode!r}: 'laplace' and 'selfp' are implemented")
        self.hemo = hemo
        n = nrowptr.shape[0] - 1
        self.n = n
        self.schur_mode = schur_mode
        if schur_mode == "selfp":
            schur_lap_coef = 1.0 if schur_lap_coef is None else schur_lap_coef
            schur_mass_coef = 0.0 if schur_mass_coef is None else schur_mass_coef
        # a pressure operator without any Dirichlet row is singular on the coarsest level
        no_pin = len(p_dirichlet_nodes) == 0 and (schur_mode == "selfp" or p_open_nodes is None or len(p_open_nodes) == 0)
        self.coarse_shift = 1e-8 if (project_pressure or no_pin) else 0.0
        # Schur complement of the mid-point scheme (DESIGN.md §5):
        #   S ~ 1/2 B (rho/dt M + mu/2 K)^-1 B^T  =>  S^-1 ~ mu Mp^-1 + (2 rho/dt) Lp^-1
        self.opts = dict(restart=restart, max_it=max_it, rtol=rtol, atol=atol, amg_cycles_u=amg_cycles_u,
                         amg_cycles_p=amg_cycles_p, cheb_degree=cheb_degree,
                         project_pressure=int(bool(project_pressure)), pc_mode=0,
                         schur_mass_coef=mu if schur_mass_coef is None else schur_mass_coef,
                         schur_lap_coef=2.0 * rho / dt if schur_lap_coef is None else schur_lap_coef,
                         cheb_ratio=cheb_ratio, cheb_degree_pre=cheb_degree_pre)
        hemo.set_solver_opts(**self.opts)
        # constant operators of the Schur approximation, assembled on the device
        self.lap, self.mass = hemo.assemble_laplace_mass()
        lap_host = self.lap.cpu().numpy()
        L = sp.csr_matrix((lap_host, ncol, nrowptr), shape=(n, n))
        umask = np.zeros(n, dtype=bool)
        umask[np.asarray(u_dirichlet_nodes, dtype=np.int64)] = True
        pmask = np.zeros(n, dtype=bool)
        pmask[np.asarray(p_dirichlet_nodes, dtype=np.int64)] = True
        if schur_mode != "selfp" and p_open_nodes is not None and len(p_open_nodes):
            # open (traction) boundary: Dirichlet condition for the Schur-complement Laplacian
            # (identity rows/cols), applied once on the host and uploaded
            omask = np.zeros(n, dtype=bool)
            omask[np.asarray(p_open_nodes, dtype=np.int64)] = True
            rows = np.repeat(np.arange(n), np.diff(nrowptr))
            hit = omask[rows] | omask[ncol]
            lap_host = np.where(hit, (rows == ncol).astype(np.float64), lap_host)
            self.lap = hemo.torch.from_numpy(np.ascontiguousarray(lap_host)).to(hemo.device)
            L = sp.csr_matrix((lap_host, ncol, nrowptr), shape=(n, n))
            pmask |= omask
        self.levels = []
        fine_p = None
        if schur_mode == "selfp":
            # Sp = A11 - A10 D^-1 A01 couples pressure nodes at graph distance 2
            G = sp.csr_matrix((np.ones(ncol.shape[0], dtype=np.float32), ncol, nrowptr), shape=(n, n))
            fine_p = (G @ G).tocsr()
            fine_p.sort_indices()
            hemo.amg_set_fine_pattern(1, fine_p)
            # SELFP carries the boundary conditions algebraically: only true Dirichlet pressure dofs are fixed
            pmask = np.zeros(n, dtype=bool)
            pmask[np.asarray(p_dirichlet_nodes, dtype=np.int64)] = True
        # tetrahedra: the velocity block is handled by block-Jacobi sweeps inside the library
        # (no 3x3-block hierarchy yet, DESIGN.md §5b); only the scalar pressure hierarchy is built
        tet = getattr(hemo, "dim", 2) == 3
        for which, mask, max_coarse in ((0, umask, 80), (1, pmask, 160)):
            if tet and which == 0:
                self.levels.append([])
                continue
            lv = amg_setup.build_hierarchy(L, mask, max_coarse=max_coarse, theta=strength_theta,
                                           smooth=smooth_prolongator, fine_pattern=fine_p if which == 1 else None)
            for l, d in enumerate(lv):
                hemo.amg_set_level(which, l, d["P"], d["R"], d["AP"], d["C"])
            hemo.amg_finalize(which, len(lv) + 1)
            self.levels.append(lv)
        self._first = True

    def set_tolerances(self, rtol=None, max_it=None):
        if rtol is not None:
            self.opts["rtol"] = rtol
        if max_it is not None:
            self.opts["max_it"] = max_it
        self.hemo.set_solver_opts(**self.opts)

    def setup(self, vals):
        """pc.setUp() for a new Jacobian."""
        if self.schur_mode == "selfp":
            self.hemo.pc_set_schur_selfp(vals, self.coarse_shift)
            self.hemo.pc_setup(vals, None, self.mass if self._first else None)
            self._first = False
            return
        if self._first:
            self.hemo.pc_setup(vals, self.lap, self.mass)
            self._first = False
        else:
            self.hemo.pc_setup(vals)

    def solve(self, vals, b, y):
        """KSPSolve with zero initial guess; returns (iterations, relative residual)."""
        return self.hemo.fgmres(vals, b, y)
