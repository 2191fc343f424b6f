"""B200 implementation shared by the three `stabilized_schur*` solver plugins.

What the reference does with UFL/FFCx/DOLFINx/PETSc
(src/solvers/stabilized_schur.py, stabilized_schur_backflow.py,
stabilized_schur_pressure_backflow.py) is done here by libhemo_sm100.so:
this class only sequences C-ABI calls and mirrors the control flow of
`Solver.__init__` / `setup` / `solveStep` and of PETSc's SNES newtonls + bt
line search (SURVEY.md App. B).  P1–P1 triangles and Q1–Q1 quadrilaterals
(`mesh.topology.cell_name()`, stabilized_schur.py:55-58).
"""
from __future__ import annotations

import math
from typing import Callable

import numpy as np

from ..._lib import Hemo, HemoDiverged, Q_FP, Q_FU, Q_PP, Q_PU, Q_UP, Q_UU
from ...fem import discretization as D
from ...fem import quadrature as Q
from ...fem.mesh import exterior_facet_indices
from ...linear_solver import BlockSchurSolver
from ..boundaryCondition import BoundaryCondition
from ..solverBase import SolverBase

# estimated UFL degree of each block form on P1 triangles (SURVEY §7.1; each
# block of extract_blocks() is its own form: stabilized_schur.py:188-189)
BLOCK_DEGREE = {Q_FU: 12, Q_FP: 11, Q_UU: 12, Q_UP: 11, Q_PU: 11, Q_PP: 10}
# Q1 quadrilaterals: Q1 counts as degree 2 and derivatives keep the degree (SURVEY §7.1):
# tau(14) R(4) (u_m.grad v)(4) = 22, PSPG/J_up/J_pu 20, J_pp 18 -> 12x12 / 11x11 / 10x10 Gauss points
BLOCK_DEGREE_QUAD = {Q_FU: 22, Q_FP: 20, Q_UU: 22, Q_UP: 20, Q_PU: 20, Q_PP: 18}
# P2-P2 triangles (p_grade = 2): tau(14) R(3) (u_m.grad v)(3) = 20 (SURVEY §7.1), PSPG / J_up / J_pu 18, J_pp 16; facet terms 6
BLOCK_DEGREE_P2 = {Q_FU: 20, Q_FP: 18, Q_UU: 20, Q_UP: 18, Q_PU: 18, Q_PP: 16}
FACET_POINTS_P2 = 4

# facet-set slots in the library (SET_WSS: all exterior facets with zero coefficients, only tagged
# for the device post-processing kernels)
SET_ALL, SET_INLET, SET_OUTLET = 0, 1, 2
SET_WSS, SET_FORCE = 7, 6

SNES_DIVERGED_LINEAR_SOLVE = -3
SNES_DIVERGED_MAX_IT = -5
SNES_DIVERGED_LINE_SEARCH = -6
SNES_DIVERGED_FNORM_NAN = -4


class StabilizedSchurB200(SolverBase):
    variant = "schur"          # "schur" | "backflow" | "pressure_backflow" | ... | "pressurebc"
    formulation = "standard"   # weak form the library assembles ("curlcurl": stabilized_schur_pressurebc.py)
    _supported_cells = ("triangle", "quadrilateral")

    def __init__(self, mesh, dt, rho, mu, f, initial_velocity: Callable | None = None, **kw):
        super().__init__(mesh, dt, rho, mu, f)
        cell = mesh.topology.cell_name()
        if cell not in self._supported_cells:
            raise NotImplementedError(
                f"cell type {cell}: {', '.join(self._supported_cells)} cells are implemented on the device for this solver")
        self._quad = cell == "quadrilateral"
        # p_grade: Lagrange degree of BOTH spaces (stabilized_schur_pressure_backflow.py:71,102-106;
        # stabilized_schur_backflow.py:63,85-87); 2 = P2-P2 on triangles, "nodes" are then the P2 dof points
        self.p_grade = int(kw.pop("p_grade", 1))
        if self.p_grade not in (1, 2) or (self.p_grade == 2 and cell != "triangle"):
            raise NotImplementedError(f"p_grade = {self.p_grade} on {cell} cells: P1-P1 on every supported cell type and "
                                      "P2-P2 on triangles are implemented on the device")
        self._p2 = self.p_grade == 2
        super().initVelocitySpace("Lagrange", cell, self.p_grade, shape=(mesh.geometry.dim,))
        super().initPressureSpace("Lagrange", cell, self.p_grade)
        if initial_velocity:
            self.u_prev.interpolate(initial_velocity)

        # PETSc option mirrors (stabilized_schur.py:269-273 + PETSc defaults)
        self.snes_rtol = float(kw.pop("snes_rtol", 1e-8))
        self.snes_atol = float(kw.pop("snes_atol", 1e-50))
        self.snes_stol = float(kw.pop("snes_stol", 1e-8))
        self.snes_max_it = int(kw.pop("snes_max_it", 100))
        self.ksp_rtol = float(kw.pop("ksp_rtol", 1e-5))
        self.ksp_atol = float(kw.pop("ksp_atol", 1e-50))      # PETSc: converged when |r| < max(rtol |b|, atol)
        self.ksp_max_it = int(kw.pop("ksp_max_it", 1000))
        self.ksp_restart = int(kw.pop("ksp_restart", 60))
        self.verbose = bool(kw.pop("verbose", False))
        # "newton": PCSetUp for every Jacobian like the reference (SNES lag 1);
        # "step": once per time step, later Newton iterations reuse the hierarchy
        self.pc_rebuild = str(kw.pop("pc_rebuild", "step"))
        # treatment of open (traction) boundary nodes in the pressure operator of the Schur
        # approximation: "dirichlet" (identity rows) or "natural" (regular rows)
        self.schur_open = str(kw.pop("schur_open", "dirichlet"))
        self._pc_kw = {k: kw.pop(k) for k in list(kw) if k in (
            "amg_cycles_u", "amg_cycles_p", "cheb_degree", "cheb_ratio", "cheb_degree_pre", "smooth_prolongator",
            "strength_theta", "schur_mass_coef", "schur_lap_coef", "schur_mode")}
        self._rules = kw.pop("quadrature", None)
        self._device_index = int(kw.pop("device", 0))
        # host_only: build spaces / BC tables / facet tables but create no CUDA context
        # (used by every rank of the multi-GPU driver to derive its partition's tables)
        self._host_only = bool(kw.pop("host_only", False))
        self._facet_tables = {}
        self._setup_count = 0
        self._p_c_frozen: list[float] = []
        self._p_c = 0.0
        self.its_snes = 0
        self.its_ksp = 0
        self.reason = 0
        self.hemo = None
        if self._host_only:
            self._cells_host = np.ascontiguousarray(self.V.dofmap.list, dtype=np.int32)
            self.n = self.V.num_nodes
            self.N = 3 * self.n
            if self.variant == "schur":
                self._register_facets(SET_ALL, exterior_facet_indices(mesh.topology), a_p=1.0, a_g=1.0)
        else:
            self._init_device()

    # ------------------------------------------------------------------
    def _init_device(self):
        import torch
        self._torch = torch
        self.hemo = Hemo(self._device_index)
        dev = self.hemo.device
        mesh = self.mesh
        # nodes = dof points of the (equal-order) spaces: the mesh vertices for P1 / Q1, vertices + edge mid-points for P2
        x = np.ascontiguousarray(self.V.tabulate_dof_coordinates()[:, :2])
        cells = np.ascontiguousarray(self.V.dofmap.list, dtype=np.int32)
        self.n = n = x.shape[0]
        self.N = 3 * n
        E = cells.shape[0]
        h = mesh.h(mesh.topology.dim, np.arange(E))
        self._cells_host = cells
        self.hemo.set_mesh(torch.from_numpy(x).to(dev), torch.from_numpy(cells).to(dev),
                           torch.from_numpy(np.ascontiguousarray(h)).to(dev))
        self.hemo.set_formulation(self.formulation)
        self._nrowptr, self._ncol = D.node_graph(cells, n)
        self.hemo.set_node_graph(torch.from_numpy(self._nrowptr).to(dev), torch.from_numpy(self._ncol).to(dev))
        for block, deg in (BLOCK_DEGREE_QUAD if self._quad else BLOCK_DEGREE_P2 if self._p2 else BLOCK_DEGREE).items():
            if self._rules:
                pts, wts = self._rules[block]
            else:
                pts, wts = Q.quadrilateral_rule(deg) if self._quad else Q.triangle_rule(deg)
            self.hemo.set_quadrature(block, pts, wts)
        self.hemo.set_facet_quadrature(*Q.interval_gauss(Q.FACET_POINTS_QUAD if self._quad else FACET_POINTS_P2 if self._p2 else 2))
        eps0 = float(np.finfo(np.float64).resolution)
        fval = np.asarray(self.f.value, dtype=np.float64).reshape(-1)
        self.hemo.set_params(float(self.dt.value), float(self.rho.value), float(self.mu.value), fval[:2], eps0)

        f64 = torch.float64
        self.d_x = torch.zeros(self.N, dtype=f64, device=dev)        # x_n = [u | p]
        self.d_un = torch.zeros(2 * n, dtype=f64, device=dev)        # u_prev
        self.d_f = torch.zeros(self.N, dtype=f64, device=dev)        # residual b
        self.d_y = torch.zeros(self.N, dtype=f64, device=dev)
        self.d_w = torch.zeros(self.N, dtype=f64, device=dev)
        self.d_g = torch.zeros(self.N, dtype=f64, device=dev)        # trial residual
        self.d_t = torch.zeros(self.N, dtype=f64, device=dev)
        self.d_bcval = torch.zeros(self.N, dtype=f64, device=dev)    # Dirichlet values
        self.d_vals = torch.zeros(self.hemo.nnz, dtype=f64, device=dev)
        # host Functions live in pinned memory so the per-step copies are async DMA
        self._pin = {}
        for name, fn in (("u_sol", self.u_sol), ("p_sol", self.p_sol), ("u_prev", self.u_prev),
                         ("p_prev", self.p_prev), ("u_residual", self.u_residual), ("p_residual", self.p_residual)):
            t = torch.empty(fn.x.array.shape[0], dtype=f64).pin_memory()
            t.numpy()[:] = fn.x.array
            fn.x.array = t.numpy()
            self._pin[name] = t
        # stabilized_schur.py:79 — the all-facet term is part of F in the ctor
        if self.variant == "schur":
            self._register_facets(SET_ALL, exterior_facet_indices(mesh.topology), a_p=1.0, a_g=1.0)
        self.linear = None

    def _register_facets(self, set_id: int, facets, **coef):
        """One tagged ds integral: remembered on the host (export_tables) and, when a
        device context exists, uploaded grouped by cell.  Sets without coefficients only tag
        facets for the post-processing kernels and are not exported as form terms."""
        if coef:
            self._facet_tables[set_id] = (np.asarray(facets, dtype=np.int64), dict(coef))
        if self.hemo is not None:
            torch = self._torch
            dev = self.hemo.device
            fc, fm = D.facet_set_by_cell(self.mesh, facets)
            self.hemo.set_facet_set(set_id, torch.from_numpy(fc).to(dev), torch.from_numpy(fm).to(dev), **coef)

    def export_tables(self) -> dict:
        """Everything the device needs, as host arrays in global numbering: mesh, Dirichlet
        objects in list order, facet sets as (cell, local facet) pairs with coefficients."""
        topo = self.mesh.topology
        return dict(
            x=np.ascontiguousarray(self.V.tabulate_dof_coordinates()[:, :2]), cells=self._cells_host,
            bcs=[("u", bc.block_dofs.copy(), bc.g.x.array.copy()) for bc in self.bcu_d]
                + [("p", bc.block_dofs.copy(), bc.g.x.array.copy()) for bc in self.bcp_d],
            facet_sets={sid: (topo.facet_cell_pairs(f), c) for sid, (f, c) in self._facet_tables.items()},
            params=dict(dt=float(self.dt.value), rho=float(self.rho.value), mu=float(self.mu.value),
                        f=np.asarray(self.f.value, dtype=float).reshape(-1)[:2]),
            variant=self.variant, u_prev=self.u_prev.x.array.copy(), p_prev=self.p_prev.x.array.copy(),
            outlet=dict(R_resistance=getattr(self, "R_resistance", None), alpha_damping=getattr(self, "alpha_damping", None),
                        p_c=self._p_c, p_c_frozen=list(self._p_c_frozen), setup_count=self._setup_count),
            solver_kw=dict(snes_rtol=self.snes_rtol, snes_atol=self.snes_atol, snes_stol=self.snes_stol,
                           snes_max_it=self.snes_max_it, ksp_rtol=self.ksp_rtol, ksp_max_it=self.ksp_max_it,
                           ksp_restart=self.ksp_restart, pc_kw=dict(self._pc_kw)))

    # ------------------------------------------------------------------
    def _facet_setup(self, facet_tags, tags):
        """Boundary terms appended to F by `setup()`; called once per setup()
        call, so a second call doubles them (SURVEY §7.3-1)."""
        return None

    def _update_facet_coefs(self):
        return None

    def _bc_tables(self, bcu, bcp):
        self.bcu_d = [bc.getBC(self.V) for bc in bcu]
        self.bcp_d = [bc.getBC(self.Q) for bc in bcp] if self.variant == "schur" else []
        bcs = [("u", bc.block_dofs, bc.g.x.array) for bc in self.bcu_d]
        bcs += [("p", bc.block_dofs, bc.g.x.array) for bc in self.bcp_d]
        return bcs

    def _upload_bc_values(self):
        """bc.update() for every bc, then refresh the Dirichlet value vector
        (stabilized_schur.py:170).  Only boundary-sized work per step: the
        values are compared on the constrained dofs and uploaded when changed."""
        n = self.n
        parts = []
        for bc in self.bcu_d:
            bc.update()
            d, _ = bc.dof_indices()
            parts.append((d, bc.g.x.array[d]))
        for bc in self.bcp_d:
            bc.update()
            d, _ = bc.dof_indices()
            parts.append((2 * n + d, bc.g.x.array[d]))
        if not parts:
            return
        compact = np.concatenate([v for _, v in parts])
        if self._g_last is None or not np.array_equal(compact, self._g_last):
            g = self._g_host
            for d, v in parts:          # list order: the last BC wins on shared dofs
                g[d] = v
            self.d_bcval.copy_(self._torch.from_numpy(g))
            self._g_last = compact

    def setup(self, bcu: list[BoundaryCondition], bcp: list[BoundaryCondition], facet_tags=None, tags=None) -> None:
        n = self.n
        self._setup_count += 1
        self._facet_setup(facet_tags, tags)

        bcs = self._bc_tables(bcu, bcp)
        if self._host_only:
            return
        torch = self._torch
        dev = self.hemo.device
        flag, mult, cellflag, g = D.dirichlet_arrays(n, self._cells_host, bcs)
        self._g_host = g
        self._g_last = None
        if flag.any():
            self._bc_dev = (torch.from_numpy(flag).to(dev), torch.from_numpy(mult).to(dev), torch.from_numpy(cellflag).to(dev))
            self.hemo.set_bc(*self._bc_dev)
        else:
            self._bc_dev = None
            self.hemo.set_bc(None, None, None)
        self._has_bc = bool(flag.any())
        self._upload_bc_values()

        # x_n <- [u_prev ; p_prev]   (stabilized_schur.py:216-223)
        self.d_x[:2 * n].copy_(self._pin["u_prev"], non_blocking=True)
        self.d_x[2 * n:].copy_(self._pin["p_prev"], non_blocking=True)
        self.d_un.copy_(self._pin["u_prev"], non_blocking=True)
        self._prepare_time_scheme()

        # snes.computeJacobian(x_n, A) + pc.setUp()   (:226-253)
        self.hemo.assemble_jacobian(self.d_x, self.d_un, self.d_vals)
        u_nodes = np.nonzero(flag[0:2 * n:2] | flag[1:2 * n:2])[0]
        p_nodes = np.nonzero(flag[2 * n:])[0]
        p_open = np.zeros(0, dtype=np.int64)
        if self.variant != "schur" and self.schur_open == "dirichlet":
            # without the all-facet term of stabilized_schur.py:79 the Schur complement sees a
            # Dirichlet-like pressure condition wherever the velocity is free on the boundary
            ext = exterior_facet_indices(self.mesh.topology)
            bnodes = np.unique(self.mesh.topology.facet_vertices[ext])
            if self._p2:                     # plus the edge nodes of the boundary facets
                bnodes = np.union1d(bnodes, self.mesh.geometry.x.shape[0] + ext)
            p_open = np.setdiff1d(bnodes, u_nodes)
        self._nullspace = self._test_nullspace()
        self.linear = BlockSchurSolver(
            self.hemo, self._nrowptr, self._ncol, u_nodes, p_nodes, p_open_nodes=p_open,
            dt=float(self.dt.value), rho=float(self.rho.value), mu=float(self.mu.value),
            restart=self.ksp_restart, max_it=self.ksp_max_it, rtol=self.ksp_rtol, atol=self.ksp_atol,
            project_pressure=self._nullspace, **self._pc_kw)
        self.linear.setup(self.d_vals)

    def _test_nullspace(self) -> bool:
        """nullsp.test(A): is the constant-pressure vector in the kernel of A?
        (stabilized_schur.py:283-293,314)."""
        n = self.n
        c = self.d_t
        c.zero_()
        c[2 * n:] = 1.0 / math.sqrt(n)
        self.hemo.spmv(self.d_vals, c, self.d_w)
        r = self.hemo.norm2(self.d_w)
        scale = self.hemo.norm2(self.d_vals) / math.sqrt(self.N)
        return bool(r < 1e-8 * max(scale, 1e-300))

    # ------------------------------------------------------------------
    def _residual(self, x, out):
        self.hemo.assemble_residual(x, self.d_un, self.d_bcval if self._has_bc else None, out)

    def _newton(self):
        """SNESSolve_NEWTONLS with the bt line search (SURVEY.md App. B)."""
        hemo = self.hemo
        x, f, y, w, g = self.d_x, self.d_f, self.d_y, self.d_w, self.d_g
        self._residual(x, f)
        fnorm = hemo.norm2(f)
        if self.verbose:
            print(f"  0 SNES Function norm {fnorm:.12e}")
        if not math.isfinite(fnorm):
            return 0, 0, SNES_DIVERGED_FNORM_NAN
        ttol = self.snes_rtol * fnorm
        lin_its = 0
        if fnorm < self.snes_atol:
            return 0, 0, 2
        for it in range(self.snes_max_it):
            hemo.assemble_jacobian(x, self.d_un, self.d_vals)
            if it == 0 or self.pc_rebuild == "newton":
                self.linear.setup(self.d_vals)
            try:
                kits, _ = self.linear.solve(self.d_vals, f, y)
            except HemoDiverged:
                return it, lin_its, SNES_DIVERGED_LINEAR_SOLVE
            lin_its += kits
            # --- bt line search -------------------------------------------------
            hemo.spmv(self.d_vals, y, self.d_t)
            slope = hemo.dot(f, self.d_t)
            slope = -abs(slope) if slope != 0.0 else -1.0
            alpha = 1e-4
            lam = 1.0
            f2 = 0.5 * fnorm * fnorm
            lam_prev = g_prev = None
            accepted = False
            for _ in range(40):
                w.copy_(x)
                hemo.axpy(-lam, y, w)
                self._residual(w, g)
                gnorm = hemo.norm2(g)
                g2 = 0.5 * gnorm * gnorm
                if math.isfinite(gnorm) and g2 <= f2 + lam * alpha * slope:
                    accepted = True
                    break
                if not math.isfinite(gnorm):
                    lam_new = 0.5 * lam
                elif lam_prev is None:
                    lam_new = -slope / (2.0 * (g2 - f2 - slope))
                else:
                    t1 = g2 - f2 - lam * slope
                    t2 = g_prev - f2 - lam_prev * slope
                    a = (t1 / lam ** 2 - t2 / lam_prev ** 2) / (lam - lam_prev)
                    b = (-lam_prev * t1 / lam ** 2 + lam * t2 / lam_prev ** 2) / (lam - lam_prev)
                    disc = max(b * b - 3.0 * a * slope, 0.0)
                    lam_new = -slope / (2.0 * b) if a == 0.0 else (-b + math.sqrt(disc)) / (3.0 * a)
                lam_new = min(max(lam_new, 0.1 * lam), 0.5 * lam)
                lam_prev, g_prev = lam, g2
                lam = lam_new
            if not accepted:
                return it + 1, lin_its, SNES_DIVERGED_LINE_SEARCH
            ynorm = lam * hemo.norm2(y)
            x.copy_(w)
            f.copy_(g)
            fnorm = gnorm
            if self.verbose:
                print(f"  {it + 1} SNES Function norm {fnorm:.12e}")
            if fnorm < self.snes_atol:
                return it + 1, lin_its, 2
            if fnorm <= ttol:
                return it + 1, lin_its, 3
            if ynorm < self.snes_stol * hemo.norm2(x):
                return it + 1, lin_its, 4
        return self.snes_max_it, lin_its, SNES_DIVERGED_MAX_IT

    def _remove_pressure_mean(self):
        """nullsp.remove(x_n) — unconditional in the reference (:319)."""
        self.hemo.remove_mean(self.d_x[2 * self.n:])

    def _prepare_time_scheme(self):
        """Hook of the variants with another time scheme (stabilized_schur_bdf2)."""
        return None

    def _solve_on_device(self):
        # bc.update() for every bc + refresh of the Dirichlet values (stabilized_schur.py:170): in the
        # host loop and in the device-resident loop alike (boundary-sized, uploads only on change)
        self._upload_bc_values()
        self._remove_pressure_mean()
        self._update_facet_coefs()
        self._prepare_time_scheme()
        self.its_snes, self.its_ksp, self.reason = self._newton()
        if self.verbose:
            print(f"Solver converged in {self.its_snes} nonlinear iterations"
                  f" (with total number of {self.its_ksp} linear iterations)")
        if self.reason < 0:
            raise RuntimeError(f"Did not converge, reason: {self.reason}.")

    def solveStep(self):
        """One time step through the plugin API: host u_prev in, host
        u_sol / p_sol / residuals out (stabilized_schur.py:313-334)."""
        n = self.n
        # the host owns the time-level shift (scenario.py:306-307)
        self.d_un.copy_(self._pin["u_prev"], non_blocking=True)
        self._solve_on_device()
        self._pin["u_sol"].copy_(self.d_x[:2 * n], non_blocking=True)
        self._pin["p_sol"].copy_(self.d_x[2 * n:], non_blocking=True)
        self._pin["u_residual"].copy_(self.d_f[:2 * n], non_blocking=True)
        self._pin["p_residual"].copy_(self.d_f[2 * n:], non_blocking=True)
        self._torch.cuda.current_stream(self.hemo.device).synchronize()
        self._after_step()

    def step_device(self, shift: bool = True):
        """Device-resident time step: same work as solveStep() but nothing crosses PCIe;
        with `shift` the time-level shift u_prev <- u_sol (scenario.py:306) happens on the
        device right away, otherwise the caller does it (`shift_time_level_device`) after its
        own post-processing of (u_sol, u_prev)."""
        self._solve_on_device()
        self._after_step(device=True)
        if shift:
            self.shift_time_level_device()

    def shift_time_level_device(self):
        self.d_un.copy_(self.d_x[:2 * self.n])

    # ---- per-step post-processing on the device (SURVEY §8(f) rank 2) -------------------
    def initStressForm(self):
        """Reference :144-174; additionally tags the exterior facets on the device so that
        `assemble_wss_device` can run without host work."""
        super().initStressForm()
        if self._p2:
            return                            # the device post-processing kernels are P1 / Q1 (include/hemo.h)
        if self.hemo is not None:
            self._register_facets(SET_WSS, exterior_facet_indices(self.mesh.topology))
            self.d_wss = self._torch.zeros(2 * self.n, dtype=self._torch.float64, device=self.hemo.device)

    def assemble_wss_device(self):
        """`assemble_wss()` (src/solverBase.py:184-195) on the device: d_wss <- shear stress of d_x."""
        self.hemo.wall_shear_stress(SET_WSS, self.d_x, self.d_wss)
        return self.d_wss

    def early_stop_norms_device(self):
        """(max|u_sol - u_prev|, max|u_sol|) of scenario.py:268-304 from the device state."""
        return self.hemo.early_stop_norms(self.d_x[:2 * self.n], self.d_un)

    def boundary_force_device(self, facets):
        """Drag / lift integrals of dfg_1.py:189-202 over `facets` (before the factor 500)."""
        key = np.asarray(facets, dtype=np.int64).tobytes()
        if getattr(self, "_force_key", None) != key:
            self._register_facets(SET_FORCE, facets)
            self._force_key = key
        return self.hemo.boundary_force(SET_FORCE, self.d_x)

    def consistent_boundary_force(self, nodes):
        """Force the fluid exerts on the boundary nodes `nodes`, from the momentum residual itself (consistent nodal
        forces): minus the sum of the rows of the raw residual (no Dirichlet treatment, no all-facet boundary term, time
        level u = u_prev) at those nodes.  With v = 1 on the body and the discrete equations satisfied elsewhere this is
        int (sigma n) ds tested with the finite-element extension of v — it converges at twice the rate of the
        boundary-gradient formula the reference's post-processing uses (src/scenarios/dfg_1.py:183-202) and serves as an
        independent anchor on the literature values (tests/test_gpu_literature.py)."""
        torch = self._torch
        hemo = self.hemo
        n = self.n
        saved = {sid: dict(c) for sid, (f, c) in self._facet_tables.items()}
        for sid in saved:
            hemo.set_facet_coef(sid)                       # all coefficients zero: cell integrals only
        hemo.set_bc(None, None, None)
        un_saved = self.d_un.clone()
        self.d_un.copy_(self.d_x[:2 * n])                   # steady state: (u - u_prev)/dt = 0, u_mid = u
        hemo.assemble_residual(self.d_x, self.d_un, None, self.d_t)
        self.d_un.copy_(un_saved)
        for sid, c in saved.items():
            hemo.set_facet_coef(sid, **c)
        if self._bc_dev is not None:
            hemo.set_bc(*self._bc_dev)
        idx = torch.as_tensor(np.asarray(nodes, dtype=np.int64), device=hemo.device)
        r = self.d_t[:2 * n].reshape(-1, 2).index_select(0, idx).sum(dim=0).cpu().numpy()
        return -float(r[0]), -float(r[1])

    def l2_norms_device(self):
        """sqrt(int |u|^2), sqrt(int p^2) of the final state (scenario.py:315-324)."""
        n = self.n
        return (math.sqrt(self.hemo.l2_norm_sq(self.d_x[:2 * n], 2)), math.sqrt(self.hemo.l2_norm_sq(self.d_x[2 * n:], 1)))

    def download_solution(self):
        """Device state -> host Functions (u_sol, p_sol, residuals, u_prev) after a device-resident loop."""
        n = self.n
        self._pin["u_sol"].copy_(self.d_x[:2 * n], non_blocking=True)
        self._pin["p_sol"].copy_(self.d_x[2 * n:], non_blocking=True)
        self._pin["u_residual"].copy_(self.d_f[:2 * n], non_blocking=True)
        self._pin["p_residual"].copy_(self.d_f[2 * n:], non_blocking=True)
        self._pin["u_prev"].copy_(self.d_un, non_blocking=True)
        if getattr(self, "d_wss", None) is not None and getattr(self, "shear_stress", None) is not None:
            self.shear_stress.x.array[:] = self.d_wss.cpu().numpy()
        self._torch.cuda.current_stream(self.hemo.device).synchronize()

    def _after_step(self, device=False):
        return None

    @property
    def h2d_bytes_per_step(self) -> int:
        return 8 * 2 * self.n

    @property
    def d2h_bytes_per_step(self) -> int:
        return 8 * 6 * self.n
