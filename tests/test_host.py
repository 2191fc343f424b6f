"""CPU tests of the host layer: quadrature tables, mesh/topology shim, Dirichlet
tables, node graph vs the oracle's pattern, AMG transfer operators, C-ABI exports."""
import os
import re

import numpy as np
import pytest
import scipy.sparse as sp

from cfd_hemodynamic_b200.fem import discretization as D
from cfd_hemodynamic_b200.fem import mesh as M
from cfd_hemodynamic_b200.fem import quadrature as Q
from cfd_hemodynamic_b200.fem import space as S
from oracle import ns_oracle as O
from tests import common as T

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("degree", [1, 2, 5, 10, 11, 12, 15])
def test_triangle_rules_exact(degree):
    pts, wts = Q.triangle_rule(degree)
    assert abs(wts.sum() - 0.5) < 1e-15
    assert Q.check_triangle_rule(pts, wts, degree) < 1e-15
    assert (pts > 0).all() and (pts.sum(axis=1) < 1).all()


def test_interval_rule():
    x, w = Q.interval_gauss(2)
    assert np.allclose(x, [0.5 - 0.5 / np.sqrt(3), 0.5 + 0.5 / np.sqrt(3)]) and np.allclose(w, [0.5, 0.5])


def test_unit_square_topology():
    m = M.create_unit_square(None, 4, 3)
    assert m.geometry.x.shape == (20, 3) and m.geometry.dofmap.shape == (24, 3)
    ext = M.exterior_facet_indices(m.topology)
    assert ext.shape[0] == 2 * (4 + 3)
    lid = M.locate_entities_boundary(m, 1, lambda X: np.isclose(X[1], 1.0) & (X[0] > 1e-10) & (X[0] < 1 - 1e-10))
    assert lid.shape[0] == 2                      # open interval: corner facets excluded
    pairs = m.topology.facet_cell_pairs(ext)
    cells = m.geometry.dofmap
    for (c, lf), f in zip(pairs, ext):
        fv = set(m.topology.facet_vertices[f])
        assert fv == set(np.delete(cells[c], lf))    # facet lf is opposite vertex lf
    h = m.h(2, np.arange(24))
    assert np.allclose(h, np.hypot(1 / 4, 1 / 3))


def test_function_space_and_bc_shim():
    m = M.create_unit_square(None, 3, 3)
    V = S.functionspace(m, S.element("Lagrange", "triangle", 1, shape=(2,)))
    Qs = S.functionspace(m, ("Lagrange", 1))
    assert V.dofmap.index_map_bs == 2 and V.dofmap.index_map.size_global == 16
    f = S.Function(V)
    f.interpolate(lambda x: np.vstack([x[0] + 1, 2 * x[1]]))
    assert np.allclose(f.x.array[0::2], m.geometry.x[:, 0] + 1) and np.allclose(f.x.array[1::2], 2 * m.geometry.x[:, 1])
    left = M.locate_entities_boundary(m, 1, lambda X: np.isclose(X[0], 0.0))
    dofs = S.locate_dofs_topological(V, 1, left)
    assert np.array_equal(dofs, [0, 4, 8, 12])
    bc = S.dirichletbc(f, dofs)
    d, nown = bc.dof_indices()
    assert np.array_equal(d, [0, 1, 8, 9, 16, 17, 24, 25]) and nown == 8
    assert Qs.dofmap.index_map_bs == 1


def test_node_graph_expands_to_reference_pattern():
    """Sparsity pattern bit-exact vs the oracle's create_matrix_block restatement."""
    mesh = T.perturbed_square(5, 4)
    prob = T.make_problem(mesh)
    nrowptr, ncol = D.node_graph(prob.cells, prob.n)
    n = prob.n
    rowptr = np.zeros(3 * n + 1, dtype=np.int64)
    cols = []
    deg = np.diff(nrowptr)
    for block_rows in (0, 1):
        pass
    rows_cols = []
    for i in range(n):
        nb = ncol[nrowptr[i]:nrowptr[i + 1]]
        rows_cols.append(np.concatenate([np.stack([2 * nb, 2 * nb + 1], axis=1).ravel(), 2 * n + nb]))
    order = [(2 * i + k, rows_cols[i]) for i in range(n) for k in range(2)] + [(2 * n + i, rows_cols[i]) for i in range(n)]
    order.sort(key=lambda t: t[0])
    indices = np.concatenate([c for _, c in order])
    indptr = np.concatenate([[0], np.cumsum([len(c) for _, c in order])])
    ip, idx = O.sparsity_pattern(prob)
    assert np.array_equal(indptr, ip) and np.array_equal(indices, idx)


def test_dirichlet_arrays_and_facet_grouping():
    mesh = M.create_unit_square(None, 3, 3)
    n = 16
    cells = mesh.geometry.dofmap
    g0 = np.arange(2 * n, dtype=float)
    g1 = -np.arange(2 * n, dtype=float)
    flag, mult, cellflag, g = D.dirichlet_arrays(n, cells, [("u", [0, 1], g0), ("u", [1, 2], g1), ("p", [5], np.ones(n))])
    assert flag[:6].tolist() == [1] * 6 and flag[2 * n + 5] == 1
    assert mult[2] == 2.0 and mult[0] == 1.0
    assert g[2] == g1[2] and g[0] == g0[0]
    assert cellflag.sum() == np.isin(cells, [0, 1, 2, 5]).any(axis=1).sum()
    ext = M.exterior_facet_indices(mesh.topology)
    fc, fm = D.facet_set_by_cell(mesh, ext)
    assert len(np.unique(fc)) == len(fc)
    assert sum(bin(int(v)).count("1") for v in fm) == len(ext)      # corner cells carry two facets


def test_c_abi_exports_every_declared_symbol(hemo_lib_built):
    """The shared library loads without a GPU and exports what include/hemo.h declares."""
    from cfd_hemodynamic_b200 import _lib
    lib = _lib.load_library()
    header = open(os.path.join(ROOT, "include", "hemo.h")).read()
    declared = set(re.findall(r"\b(hemo_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    for name in declared:
        assert hasattr(lib, name), name
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)


def test_no_gpu_is_a_loud_failure(hemo_lib_built):
    import torch
    from cfd_hemodynamic_b200 import _lib
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    with pytest.raises(_lib.HemoError):
        _lib.Hemo(0)


def test_block_schur_solver_rejects_unknown_schur_mode():
    """A Schur approximation the library does not implement is refused before the library is touched."""
    from cfd_hemodynamic_b200.linear_solver import BlockSchurSolver

    class NoLibrary:
        def __getattr__(self, name):
            raise AssertionError(f"library call {name} before the schur_mode check")

    nrowptr, ncol = D.node_graph(np.array([[0, 1, 2]]), 3)
    none = np.zeros(0, dtype=np.int64)
    with pytest.raises(ValueError, match="schur_mode"):
        BlockSchurSolver(NoLibrary(), nrowptr, ncol, none, none, dt=0.01, rho=1.0, mu=0.01, schur_mode="assembled")


def test_amg_transfer_operators(hemo_lib_built):
    from cfd_hemodynamic_b200.fem import amg_setup
    m = M.create_unit_square(None, 24, 24)
    x = m.geometry.x[:, :2]
    cells = m.geometry.dofmap
    n = x.shape[0]
    det, dphi = O.cell_geometry(x, cells)
    Ke = (det / 2)[:, None, None] * np.einsum("eai,ebi->eab", dphi, dphi)
    L = sp.coo_matrix((Ke.ravel(), (np.repeat(cells, 3, axis=1).ravel(), np.tile(cells, (1, 3)).ravel())), shape=(n, n)).tocsr()
    L.sort_indices()
    nrowptr, ncol = D.node_graph(cells, n)
    assert np.array_equal(L.indptr, nrowptr) and np.array_equal(L.indices, ncol)
    mask = np.isclose(x[:, 0], 0.0)
    lv = amg_setup.build_hierarchy(L, mask, max_coarse=30)
    assert len(lv) >= 2 and lv[-1]["P"].shape[1] <= 30
    P = lv[0]["P"]
    assert P[mask].nnz == 0                                # Dirichlet nodes are not interpolated
    far = ~mask & (x[:, 0] > 0.2)
    assert np.allclose(np.asarray(P.sum(axis=1)).ravel()[far], 1.0)   # constants reproduced away from the BC
    Ac = (lv[0]["R"] @ L @ P).tocsr()
    assert set(zip(*Ac.nonzero())) <= set(zip(*lv[0]["C"].nonzero()))  # fixed pattern covers the product
    AP = (L @ P).tocsr()
    assert set(zip(*AP.nonzero())) <= set(zip(*lv[0]["AP"].nonzero()))
