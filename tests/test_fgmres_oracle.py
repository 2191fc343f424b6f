"""The float64 FGMRES model of oracle/fgmres_oracle.py (no GPU): against a direct solve, the least-squares property of
flexible GMRES, every exit reason, and its sensitivity to the defects the GPU comparison
(tests/test_gpu_fgmres_reference.py) must catch."""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from oracle import fgmres_oracle as FO


def _small(n=30, seed=0):
    """A nonsymmetric, well-conditioned matrix and a right-hand side."""
    rng = np.random.default_rng(seed)
    A = 3.0 * np.eye(n) + 0.6 * rng.standard_normal((n, n)) / np.sqrt(n) + np.diag(np.linspace(0.0, 2.0, n))
    return A, rng.standard_normal(n)


class _Varying:
    """A preconditioner that changes from call to call (a diagonal scaling drawn afresh); records its outputs Z."""

    def __init__(self, n, seed=1):
        self.rng = np.random.default_rng(seed)
        self.n = n
        self.Z = []

    def __call__(self, v):
        z = v * self.rng.uniform(0.2, 1.8, self.n)
        self.Z.append(z)
        return z


def test_identity_preconditioner_with_full_restart_is_a_direct_solve():
    A, b = _small()
    r = FO.fgmres(lambda x: A @ x, lambda v: v, b, restart=len(b), max_it=1000, rtol=1e-14, atol=0.0)
    assert r.reason == "converged" and r.cycle_ends == []
    x = np.linalg.solve(A, b)
    assert np.linalg.norm(r.y - x) <= 1e-12 * np.linalg.norm(x)


@pytest.mark.parametrize("owned", [False, True], ids=["all", "owned"])
def test_iterates_minimise_the_residual_over_the_flexible_basis(owned):
    """After every k: the estimate is the true residual of y_k, and y_k - y_start is the least-squares minimiser of
    the cycle's residual over span(Z) (over the owned rows only with a mask).  The preconditioner changes from call
    to call, so y = M(V c) of non-flexible GMRES would fail this."""
    A, b = _small(40, seed=2)
    mask = np.ones(len(b), dtype=bool)
    if owned:
        mask[-7:] = False
    P = _Varying(len(b))
    ks = list(range(1, 25))
    r = FO.fgmres(lambda x: A @ x, P, b, restart=9, max_it=24, rtol=1e-30, atol=0.0,
                  owned=mask if owned else None, snapshots=ks)
    assert r.reason == "max_it" and r.its == 24 and r.cycle_ends == [9, 18]
    bn = np.linalg.norm(b[mask])
    starts = [0] + r.cycle_ends
    for k in ks:
        c0 = max(s for s in starts if s < k)                       # iterations before this cycle
        y0 = r.snapshots[c0] if c0 else np.zeros_like(b)
        y = r.snapshots[k]
        res = b - A @ y
        assert abs(r.history[k - 1] - np.linalg.norm(res[mask])) <= 1e-12 * bn, k
        Zk = np.array(P.Z[c0:k]).T
        r0 = b - A @ y0
        c, *_ = np.linalg.lstsq((A @ Zk)[mask], r0[mask], rcond=None)
        assert np.linalg.norm(y - (y0 + Zk @ c)) <= 1e-10 * np.linalg.norm(y), k
    if owned:
        # the unowned rows are not minimised: the full residual is larger than the owned one
        assert np.linalg.norm(b - A @ r.y) > np.linalg.norm((b - A @ r.y)[mask])


def _long(A, b, **kw):
    opts = dict(restart=5, max_it=200, rtol=1e-12, atol=0.0)
    opts.update(kw)
    return FO.fgmres(lambda x: A @ x, lambda v: v / np.diag(A), b, **opts)


def test_exit_reasons():
    A, b = _small()
    bn = np.linalg.norm(b)
    # ||b|| <= atol: nothing to do, rel_resid = ||b|| / ||b||
    r = _long(A, b, atol=2 * bn)
    assert (r.reason, r.its, r.rel_resid, r.history) == ("converged", 0, 1.0, [])
    assert not r.y.any()
    # b = 0
    r = _long(A, np.zeros_like(b))
    assert (r.reason, r.its, r.rel_resid) == ("converged", 0, 0.0) and not r.y.any()
    # a NaN in b: no iteration, y = 0, rel_resid reported as 0 (the norm of b is not > 0)
    bnan = b.copy()
    bnan[3] = np.nan
    r = _long(A, bnan)
    assert (r.reason, r.its, r.rel_resid) == ("nonfinite", 0, 0.0) and not r.y.any()
    # the long solve these truncations are compared with
    full = _long(A, b, snapshots=range(1, 60))
    assert full.reason == "converged" and full.its > 12
    for max_it, restarts in ((7, [5]), (10, [5])):        # mid-cycle; exactly at the end of the second cycle
        r = _long(A, b, max_it=max_it)
        assert (r.reason, r.its, r.cycle_ends) == ("max_it", max_it, restarts)
        assert r.rel_resid == full.history[max_it - 1] / bn
        assert np.array_equal(r.y, full.snapshots[max_it])
    # convergence at the last column of a cycle: no restart follows
    m = 5
    h = np.array(full.history) / bn
    assert h[m - 1] < h[m - 2]
    r = _long(A, b, rtol=np.sqrt(h[m - 1] * h[m - 2]))
    assert (r.reason, r.its, r.cycle_ends) == ("converged", m, [])
    assert np.array_equal(r.y, full.snapshots[m])


def test_breakdown_is_unreachable():
    """An exact solution inside the Krylov space gives hn = 0; the rotation then has s = 0, so res = 0 <= tol is
    tested before the breakdown: the exit is `converged`."""
    A = np.diag([1.0, 2.0, 3.0, 4.0])
    b = np.array([0.0, 4.0, 0.0, 0.0])                  # an eigenvector: w - h v = 0 exactly
    r = FO.fgmres(lambda x: A @ x, lambda v: v, b, restart=10, max_it=10, rtol=0.0, atol=0.0)
    assert (r.reason, r.its, r.history) == ("converged", 1, [0.0])
    assert np.array_equal(r.y, [0.0, 2.0, 0.0, 0.0])


# ---------------------------------------------------------------------------------------------------------------------
# sensitivity: the 41^2 lid-cavity Jacobian of the GPU comparison, restart 5 (row b), a fixed preconditioner
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lid41():
    from cfd_hemodynamic_b200.fem import mesh as M
    from oracle import ns_oracle as O
    from tests import common as T
    nx = 40
    mesh = M.create_unit_square(None, nx, nx, cell_type="triangle")
    prob = T.make_problem(mesh, dt=0.01, rho=1.0, mu=0.05, f=(0.0, 0.0))
    x, n = prob.x, prob.n
    ext = M.exterior_facet_indices(mesh.topology)
    prob.facet_sets = [O.FacetSet(pairs=mesh.topology.facet_cell_pairs(ext), a_p=1.0, a_g=1.0)]
    walls = np.nonzero(np.isclose(x[:, 0], 0) | np.isclose(x[:, 0], 1) | np.isclose(x[:, 1], 0))[0]
    lidf = M.locate_entities_boundary(mesh, 1, lambda X: np.isclose(X[1], 1.0) & (X[0] > 1e-10) & (X[0] < 1 - 1e-10))
    lidn = np.unique(mesh.topology.facet_vertices[lidf])
    g1 = np.zeros(2 * n)
    g1[0::2] = 1.0
    prob.bcs = T.oracle_bcs(prob, [("u", walls, np.zeros(2 * n)), ("u", lidn, g1)])
    u, p, un = T.smooth_fields(x, seed=2, U=0.5)
    J = sp.csr_matrix(O.assemble_J(prob, u, p, un))
    # a preconditioner of the quality of the block preconditioner: an exact solve of a perturbed operator
    d = np.abs(J.diagonal())
    lu = spla.splu(sp.csc_matrix(J + sp.diags(0.5 * d + 0.05 * d.mean())))
    b = J @ np.random.default_rng(4).standard_normal(3 * n)
    opts = dict(restart=5, max_it=300, rtol=1e-8, atol=0.0)
    ref = FO.Fgmres(lambda v: J @ v, lu.solve).solve(b, **opts)
    assert ref.reason == "converged" and len(ref.cycle_ends) >= 2, (ref.its, ref.cycle_ends)
    return dict(J=J, pc=lu.solve, b=b, opts=opts, ref=ref)


class _RestartAyMinusB(FO.Fgmres):
    def restart_residual(self, b, Ay):
        return Ay - b


class _TolFromRestart(FO.Fgmres):
    def restart_tol(self, tol, beta, rtol, atol):
        return max(rtol * beta, atol)


class _DropLastColumn(FO.Fgmres):
    def backsolve(self, R, g, k):
        c = np.zeros(k)
        c[:k - 1] = super().backsolve(R, g, k - 1)
        return c


class _CosineEstimate(FO.Fgmres):
    def estimate(self, c, s, gj):
        return abs(c * gj)


class _SkipEveryFourthCoefficient(FO.Fgmres):
    def gram_schmidt(self, V, w):
        h = super().gram_schmidt(V, w)
        h[3::4] = 0.0
        return h


@pytest.mark.parametrize("defect", [_RestartAyMinusB, _TolFromRestart, _DropLastColumn, _CosineEstimate,
                                    _SkipEveryFourthCoefficient],
                         ids=["restart-Ay-b", "tol-from-restart", "backsolve-drops-last", "estimate-c", "mdot-skip-i+3"])
def test_tolerance_sees_the_defect(lid41, defect):
    """Each defect moves the estimate history (in units of ||b||) by at least ten times the black-box GPU tolerance,
    or changes the iteration count."""
    ref, bn = lid41["ref"], np.linalg.norm(lid41["b"])
    r = defect(lambda v: lid41["J"] @ v, lid41["pc"]).solve(lid41["b"], **lid41["opts"])
    k = min(r.its, ref.its)
    moved = float(np.max(np.abs(np.array(r.history[:k]) - np.array(ref.history[:k])))) / bn
    print(f"{defect.__name__}: its {r.its} vs {ref.its}, history moved {moved:.2e}")
    assert r.its != ref.its or moved >= 10 * FO.BLACKBOX_RESID_TOL, (r.its, ref.its, moved)
