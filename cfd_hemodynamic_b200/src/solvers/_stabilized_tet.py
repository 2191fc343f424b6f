"""P1–P1 tetrahedra behind the same plugin class (reference src/solvers/stabilized_schur.py runs on
whatever `mesh.topology.cell_name()` is, :55-58; src/scenarios/taylor_green.py:34 hands it the unit
cube split into tetrahedra).

`StabilizedSchurTetB200` sits between `StabilizedSchurB200` and the plugin's `Solver`: on triangles
and quadrilaterals every method defers to the 2-D implementation unchanged; on tetrahedra it
sequences the same C-ABI calls with the `[u interleaved (3n) | p (n)]` layout (DESIGN.md §4d, §5b).
Every variant of the family runs in 3-D (the boundary terms of stabilized_schur_pressure_backflow.py:170-217 are
dimension-generic in csrc/simplex_element.cuh; production use: src/experiments/config/arteria_lad.yaml:19).  Both time loops run: `Scenario.solve` (host
post-processing) and `Scenario.solve_device` (wall shear stress, early-stop and L2 norms as kernels).
"""
from __future__ import annotations

import math

import numpy as np

from ..._lib import Hemo
from ...fem import discretization as D
from ...fem import quadrature as Q
from ...fem.mesh import exterior_facet_indices
from ...linear_solver import BlockSchurSolver
from ._stabilized_common import BLOCK_DEGREE, SET_ALL, SET_WSS, StabilizedSchurB200

# UFL's degree estimate of the all-facet term p n.v - mu (grad(u) n).v on P1 (stabilized_schur.py:79)
FACET_DEGREE_TET = 2


class StabilizedSchurTetB200(StabilizedSchurB200):
    _supported_cells = ("triangle", "quadrilateral", "tetrahedron")

    def __init__(self, mesh, dt, rho, mu, f, initial_velocity=None, **kw):
        self._tet = mesh.topology.cell_name() == "tetrahedron"
        super().__init__(mesh, dt, rho, mu, f, initial_velocity, **kw)
        if self._tet:
            self.N = 4 * self.n

    # ------------------------------------------------------------------
    def _init_device(self):
        if not self._tet:
            return super()._init_device()
        import torch
        self._torch = torch
        self.hemo = Hemo(self._device_index)
        dev = self.hemo.device
        mesh = self.mesh
        x = np.ascontiguousarray(mesh.geometry.x[:, :3])
        cells = np.ascontiguousarray(mesh.geometry.dofmap, dtype=np.int32)
        self.n = n = x.shape[0]
        self.N = 4 * n
        E = cells.shape[0]
        h = mesh.h(mesh.topology.dim, np.arange(E))
        self._cells_host = cells
        self.hemo.set_mesh(torch.from_numpy(x).to(dev), torch.from_numpy(cells).to(dev),
                           torch.from_numpy(np.ascontiguousarray(h)).to(dev))
        self.hemo.set_formulation(self.formulation)
        self._nrowptr, self._ncol = D.node_graph(cells, n)
        self.hemo.set_node_graph(torch.from_numpy(self._nrowptr).to(dev), torch.from_numpy(self._ncol).to(dev))
        for block, deg in BLOCK_DEGREE.items():          # affine P1: the same estimated degrees as on triangles
            pts, wts = self._rules[block] if self._rules else Q.tetrahedron_rule(deg)
            self.hemo.set_quadrature(block, pts, wts)
        # all-facet term: degree 2; the backflow term (u_n.n)_- (u_m.v) and the Nitsche penalty of the hemodynamic variants: 4
        self.hemo.set_facet_quadrature(*Q.triangle_rule(FACET_DEGREE_TET if self.variant == "schur" else 4))
        eps0 = float(np.finfo(np.float64).resolution)
        fval = np.zeros(3)
        fv = np.asarray(self.f.value, dtype=np.float64).reshape(-1)
        fval[:min(3, fv.shape[0])] = fv[:3]
        self.hemo.set_params(float(self.dt.value), float(self.rho.value), float(self.mu.value), fval[:2], eps0)
        self.hemo.set_body_force3(fval)

        f64 = torch.float64
        self.d_x = torch.zeros(self.N, dtype=f64, device=dev)        # x_n = [u | p]
        self.d_un = torch.zeros(3 * n, dtype=f64, device=dev)        # u_prev
        self.d_f = torch.zeros(self.N, dtype=f64, device=dev)        # residual b
        self.d_y = torch.zeros(self.N, dtype=f64, device=dev)
        self.d_w = torch.zeros(self.N, dtype=f64, device=dev)
        self.d_g = torch.zeros(self.N, dtype=f64, device=dev)        # trial residual
        self.d_t = torch.zeros(self.N, dtype=f64, device=dev)
        self.d_bcval = torch.zeros(self.N, dtype=f64, device=dev)    # Dirichlet values
        self.d_vals = torch.zeros(self.hemo.nnz, dtype=f64, device=dev)
        self._pin = {}
        for name, fn in (("u_sol", self.u_sol), ("p_sol", self.p_sol), ("u_prev", self.u_prev),
                         ("p_prev", self.p_prev), ("u_residual", self.u_residual), ("p_residual", self.p_residual)):
            t = torch.empty(fn.x.array.shape[0], dtype=f64).pin_memory()
            t.numpy()[:] = fn.x.array
            fn.x.array = t.numpy()
            self._pin[name] = t
        # stabilized_schur.py:79 — the all-facet term is part of F in the ctor (the hemodynamic variants drop it,
        # stabilized_schur_pressure_backflow.py:121-125)
        if self.variant == "schur":
            self._register_facets(SET_ALL, exterior_facet_indices(mesh.topology), a_p=1.0, a_g=1.0)
        self.linear = None

    def export_tables(self) -> dict:
        if not self._tet:
            return super().export_tables()
        raise NotImplementedError("tetrahedra: the multi-GPU partition tables are not implemented yet")

    def _upload_bc_values(self):
        if not self._tet:
            return super()._upload_bc_values()
        n = self.n
        parts = []
        for bc in self.bcu_d:
            bc.update()
            d, _ = bc.dof_indices()
            parts.append((d, bc.g.x.array[d]))
        for bc in self.bcp_d:
            bc.update()
            d, _ = bc.dof_indices()
            parts.append((3 * n + d, bc.g.x.array[d]))
        if not parts:
            return
        compact = np.concatenate([v for _, v in parts])
        if self._g_last is None or not np.array_equal(compact, self._g_last):
            g = self._g_host
            for d, v in parts:          # list order: the last BC wins on shared dofs
                g[d] = v
            self.d_bcval.copy_(self._torch.from_numpy(g))
            self._g_last = compact

    def setup(self, bcu, bcp, facet_tags=None, tags=None) -> None:
        if not self._tet:
            return super().setup(bcu, bcp, facet_tags=facet_tags, tags=tags)
        n = self.n
        self._setup_count += 1
        self._facet_setup(facet_tags, tags)          # boundary terms of the variant (a second call doubles them)
        bcs = self._bc_tables(bcu, bcp)
        if self._host_only:
            return
        torch = self._torch
        dev = self.hemo.device
        flag, mult, cellflag, g = D.dirichlet_arrays(n, self._cells_host, bcs, gdim=3)
        self._g_host = g
        self._g_last = None
        if flag.any():
            self.hemo.set_bc(torch.from_numpy(flag).to(dev), torch.from_numpy(mult).to(dev),
                             torch.from_numpy(cellflag).to(dev))
        else:
            self.hemo.set_bc(None, None, None)
        self._has_bc = bool(flag.any())
        self._upload_bc_values()

        # x_n <- [u_prev ; p_prev]   (stabilized_schur.py:216-223)
        self.d_x[:3 * n].copy_(self._pin["u_prev"], non_blocking=True)
        self.d_x[3 * n:].copy_(self._pin["p_prev"], non_blocking=True)
        self.d_un.copy_(self._pin["u_prev"], non_blocking=True)

        # snes.computeJacobian(x_n, A) + pc.setUp()   (:226-253)
        self.hemo.assemble_jacobian(self.d_x, self.d_un, self.d_vals)
        fu = flag[:3 * n].reshape(n, 3)
        u_nodes = np.nonzero(fu.any(axis=1))[0]
        p_nodes = np.nonzero(flag[3 * n:])[0]
        p_open = None
        if self.variant != "schur" and self.schur_open == "dirichlet":
            # open (traction) boundaries: Dirichlet rows in the pressure operator of the Schur approximation (as in 2-D)
            ext = exterior_facet_indices(self.mesh.topology)
            p_open = np.setdiff1d(np.unique(self.mesh.topology.facet_vertices[ext]), u_nodes)
        self._nullspace = self._test_nullspace()
        self.linear = BlockSchurSolver(
            self.hemo, self._nrowptr, self._ncol, u_nodes, p_nodes, p_open_nodes=p_open,
            dt=float(self.dt.value), rho=float(self.rho.value), mu=float(self.mu.value),
            restart=self.ksp_restart, max_it=self.ksp_max_it, rtol=self.ksp_rtol, atol=self.ksp_atol,
            project_pressure=self._nullspace, **self._pc_kw)
        self.linear.setup(self.d_vals)

    def _test_nullspace(self) -> bool:
        if not self._tet:
            return super()._test_nullspace()
        n = self.n
        c = self.d_t
        c.zero_()
        c[3 * n:] = 1.0 / math.sqrt(n)
        self.hemo.spmv(self.d_vals, c, self.d_w)
        r = self.hemo.norm2(self.d_w)
        scale = self.hemo.norm2(self.d_vals) / math.sqrt(self.N)
        return bool(r < 1e-8 * max(scale, 1e-300))

    def _remove_pressure_mean(self):
        if not self._tet:
            return super()._remove_pressure_mean()
        self.hemo.remove_mean(self.d_x[3 * self.n:])

    def solveStep(self):
        if not self._tet:
            return super().solveStep()
        n = self.n
        self.d_un.copy_(self._pin["u_prev"], non_blocking=True)
        self._solve_on_device()              # refreshes the Dirichlet values first (bc.update(), stabilized_schur.py:170)
        self._pin["u_sol"].copy_(self.d_x[:3 * n], non_blocking=True)
        self._pin["p_sol"].copy_(self.d_x[3 * n:], non_blocking=True)
        self._pin["u_residual"].copy_(self.d_f[:3 * n], non_blocking=True)
        self._pin["p_residual"].copy_(self.d_f[3 * n:], non_blocking=True)
        self._torch.cuda.current_stream(self.hemo.device).synchronize()
        self._after_step()

    def shift_time_level_device(self):
        if not self._tet:
            return super().shift_time_level_device()
        self.d_un.copy_(self.d_x[:3 * self.n])

    def early_stop_norms_device(self):
        if not self._tet:
            return super().early_stop_norms_device()
        return self.hemo.early_stop_norms(self.d_x[:3 * self.n], self.d_un)

    def initStressForm(self):
        if not self._tet:
            return super().initStressForm()
        super(StabilizedSchurB200, self).initStressForm()          # host traction form (SolverBase)
        if self.hemo is not None:
            self._register_facets(SET_WSS, exterior_facet_indices(self.mesh.topology))
            self.d_wss = self._torch.zeros(3 * self.n, dtype=self._torch.float64, device=self.hemo.device)

    def l2_norms_device(self):
        if not self._tet:
            return super().l2_norms_device()
        n = self.n
        return (math.sqrt(self.hemo.l2_norm_sq(self.d_x[:3 * n], 3)), math.sqrt(self.hemo.l2_norm_sq(self.d_x[3 * n:], 1)))

    def boundary_force_device(self, facets):
        if not self._tet:
            return super().boundary_force_device(facets)
        raise NotImplementedError("tetrahedra: the drag / lift integrals are the 2-D forms of dfg_1.py:189-202")

    def download_solution(self):
        if not self._tet:
            return super().download_solution()
        n = self.n
        self._pin["u_sol"].copy_(self.d_x[:3 * n], non_blocking=True)
        self._pin["p_sol"].copy_(self.d_x[3 * n:], non_blocking=True)
        self._pin["u_residual"].copy_(self.d_f[:3 * n], non_blocking=True)
        self._pin["p_residual"].copy_(self.d_f[3 * n:], non_blocking=True)
        self._pin["u_prev"].copy_(self.d_un, non_blocking=True)
        if getattr(self, "d_wss", None) is not None and getattr(self, "shear_stress", None) is not None:
            self.shear_stress.x.array[:] = self.d_wss.cpu().numpy()
        self._torch.cuda.current_stream(self.hemo.device).synchronize()

    @property
    def h2d_bytes_per_step(self) -> int:
        return 8 * 3 * self.n if self._tet else super().h2d_bytes_per_step

    @property
    def d2h_bytes_per_step(self) -> int:
        return 8 * 8 * self.n if self._tet else super().d2h_bytes_per_step
