"""The float64 AMG model of oracle/amg_oracle.py (no GPU): its Chebyshev smoother and coarse-grid correction against
closed forms, and its sensitivity to the defects the GPU comparison (tests/test_gpu_amg_reference.py) must catch."""
import numpy as np
import pytest
import scipy.sparse as sp

from oracle import amg_oracle as AO


def test_chebyshev_gives_the_error_polynomial_on_a_diagonal_matrix():
    lam = np.linspace(0.02, 2.0, 57)
    b = np.random.default_rng(0).standard_normal(lam.size)
    for ratio in (4.0, 6.0):
        for k in range(1, 5):
            x = AO.chebyshev(lambda v: lam * v, np.ones_like(lam), 2.0, ratio, b, None, k)
            # e_k = p_k(lam) e_0 with e_0 = x* = b / lam
            expect = (1.0 - AO.chebyshev_error_polynomial(lam, 2.0, ratio, k)) * b / lam
            assert np.allclose(x, expect, rtol=1e-12, atol=1e-12), (ratio, k)
    # from a non-zero start the error polynomial multiplies the initial error
    x0 = np.random.default_rng(1).standard_normal(lam.size)
    x = AO.chebyshev(lambda v: lam * v, np.ones_like(lam), 2.0, 4.0, b, x0, 3)
    e0 = b / lam - x0
    assert np.allclose(b / lam - x, AO.chebyshev_error_polynomial(lam, 2.0, 4.0, 3) * e0, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("bs", [1, 2])
def test_two_level_cycle_without_smoothing_is_the_coarse_grid_correction(bs):
    n = 64
    A = sp.diags([-1.0, 2.05, -1.0], [-1, 0, 1], shape=(n, n)).tocsr()
    if bs == 2:
        A = (sp.kron(A, sp.csr_matrix([[1.0, 0.2], [0.1, 1.5]])) + sp.identity(2 * n)).tocsr()
    T = sp.csr_matrix((np.ones(n), (np.arange(n), np.arange(n) // 2)), shape=(n, n // 2))
    H = AO.Hierarchy(AO.f32(A), [dict(P=T, R=T.T.tocsr())], bs)
    b = np.random.default_rng(2).standard_normal(n * bs)
    x = H.apply(b, 1, degree=0, degree_pre=0)
    P = sp.kron(T, sp.identity(bs)).tocsr()
    Ac = AO.f32(P.T @ AO.f32(AO.f32(A) @ P))
    expect = P @ np.linalg.solve(Ac.toarray(), P.T @ b)
    assert np.allclose(x, expect, rtol=1e-12, atol=1e-12)
    assert np.allclose(H.ops[1].toarray(), Ac.toarray(), rtol=0, atol=0)


# ---------------------------------------------------------------------------------------------------------------------
# sensitivity: the lid-cavity velocity hierarchies of the GPU comparison (41^2 nodes: CSR kernels; 193^2: sliced ELL)
# ---------------------------------------------------------------------------------------------------------------------
def _p1_laplacian(x, cells, n):
    """Stiffness matrix of P1 triangles (the graph the velocity aggregates are built on)."""
    X = x[cells]                                          # (E, 3, 2)
    d1, d2 = X[:, 1] - X[:, 0], X[:, 2] - X[:, 0]
    area = 0.5 * np.abs(d1[:, 0] * d2[:, 1] - d1[:, 1] * d2[:, 0])
    e = np.stack([X[:, 2] - X[:, 1], X[:, 0] - X[:, 2], X[:, 1] - X[:, 0]], axis=1)
    K = np.einsum("eik,ejk->eij", e, e) / (4.0 * area)[:, None, None]
    rows = np.repeat(cells, 3, axis=1).reshape(-1)
    cols = np.tile(cells, (1, 3)).reshape(-1)
    L = sp.csr_matrix((K.reshape(-1), (rows, cols)), shape=(n, n))
    L.sort_indices()
    return L


@pytest.fixture(scope="module", params=[40, 192], ids=["41x41", "193x193"])
def lid(request):
    from cfd_hemodynamic_b200.fem import amg_setup
    from cfd_hemodynamic_b200.fem import mesh as M
    from oracle import ns_oracle as O
    from tests import common as T
    nx = request.param
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
    J = O.assemble_J(prob, u, p, un)
    umask = np.zeros(n, dtype=bool)
    umask[np.concatenate([walls, lidn])] = True
    levels = amg_setup.build_hierarchy(_p1_laplacian(x, prob.cells, n), umask, max_coarse=80)
    H = AO.Hierarchy(AO.velocity_level0(J, n), levels, 2)
    # the default fused range: every level from the first one with at most 256 nodes
    first = next(l for l in range(H.nlev) if H.nodes(l) <= 256)
    b = np.random.default_rng(3).standard_normal(2 * n)
    kw = dict(degree=2, degree_pre=1, ratio=4.0, fused=set(range(first, H.nlev)))
    return dict(n=n, H=H, levels=levels, b=b, kw=kw, ref=H.apply(b, 1, **kw))


def _moved(lid, x):
    return max(AO.rel_errors(x, lid["ref"]))


@pytest.mark.parametrize("change", [dict(ratio=4.4), dict(degree=3), dict(degree=1), dict(degree_pre=2)],
                         ids=["ratio-4.4", "degree-3", "degree-1", "degree_pre-2"])
def test_tolerance_sees_wrong_smoother_coefficients(lid, change):
    x = lid["H"].apply(lid["b"], 1, **dict(lid["kw"], **change))
    assert _moved(lid, x) >= 10 * AO.AMG_TOL, (change, _moved(lid, x))


class _DropProlongEntry(AO.Hierarchy):
    """Top-level prolongation that skips one entry of P (x) I2: one weight of one velocity dof."""
    drop = None

    def prolong(self, l, xc):
        y = super().prolong(l, xc)
        if l == 0:
            i, t = self.drop
            P = self.P[0]
            y[i] -= P.data[t] * xc[P.indices[t]]
        return y


def test_tolerance_sees_a_dropped_prolongator_entry(lid):
    H = lid["H"]
    P = H.P[0]
    nnz_row = np.diff(P.indptr)
    i = int(np.nonzero(nnz_row > 0)[0][len(np.nonzero(nnz_row > 0)[0]) // 2])     # a middle row with entries
    t = int(P.indptr[i] + np.argmax(np.abs(P.data[P.indptr[i]:P.indptr[i + 1]])))
    D = _DropProlongEntry.__new__(_DropProlongEntry)
    D.__dict__.update(H.__dict__)
    D.drop = (i, t)
    x = D.apply(lid["b"], 1, **lid["kw"])
    assert _moved(lid, x) >= 10 * AO.AMG_TOL, _moved(lid, x)


class _DropSliceRow(AO.Hierarchy):
    """One level-0 product (the first one with a non-zero input) leaves out the last row of one 32-row slice."""
    row = None

    def matvec(self, l, v):
        y = super().matvec(l, v)
        if l == 0 and not self.done and np.any(v):
            y[2 * self.row:2 * self.row + 2] = 0.0
            self.done = True
        return y


def test_tolerance_sees_a_skipped_slice_row(lid):
    n = lid["n"]
    D = _DropSliceRow.__new__(_DropSliceRow)
    D.__dict__.update(lid["H"].__dict__)
    D.row = 32 * (n // 64) + 31                # last row of a slice in the middle of the mesh
    D.done = False
    x = D.apply(lid["b"], 1, **lid["kw"])
    assert D.done
    assert _moved(lid, x) >= 10 * AO.AMG_TOL, _moved(lid, x)
