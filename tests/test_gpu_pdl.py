"""Programmatic dependent launch (PDL) of the FGMRES iteration's kernels: the captured iteration graph chains its
kernels with programmatic edges, and plain launches (HEMO_PDL=0) compute bitwise the same solution."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

# 193^2 nodes: the finest levels get the sliced-ELL kernels and the one-thread-per-row A01 residual
NX, DT, STEPS = 192, 0.01, 2


def _lid(monkeypatch, pdl):
    from cfd_hemodynamic_b200.src.scenarios.lid_driven2D import LidDriven2DSimulation
    monkeypatch.setenv("HEMO_PDL", pdl)        # read when the library context is created
    sc = LidDriven2DSimulation("stabilized_schur", DT, STEPS * DT, rho=1, mu=0.01, nx=NX)
    s = sc.solver
    its = []
    for _ in range(STEPS):
        s.solveStep()
        its.append((s.its_snes, s.its_ksp))
        s.u_prev.x.array[:] = s.u_sol.x.array[:]
        s.p_prev.x.array[:] = s.p_sol.x.array[:]
    return s, its


def test_iteration_graph_has_programmatic_edges(monkeypatch):
    s, _ = _lid(monkeypatch, "1")
    kernels, edges = s.hemo.krylov_graph_info()
    assert kernels > 20, kernels
    # every kernel but the first follows a kernel; the few that follow a non-kernel node launch plainly
    assert edges >= 0.9 * (kernels - 1), (kernels, edges)
    s, _ = _lid(monkeypatch, "0")
    kernels0, edges0 = s.hemo.krylov_graph_info()
    assert kernels0 == kernels and edges0 == 0, (kernels0, edges0)


def test_pdl_results_bitwise_identical(monkeypatch):
    a, its_a = _lid(monkeypatch, "0")
    u0, p0 = a.u_sol.x.array.copy(), a.p_sol.x.array.copy()
    b, its_b = _lid(monkeypatch, "1")
    assert its_a == its_b
    assert np.array_equal(u0, b.u_sol.x.array)
    assert np.array_equal(p0, b.p_sol.x.array)
