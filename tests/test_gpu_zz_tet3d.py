"""GPU parity of the 3-D path beyond the cell integrals, through the generic C-ABI entry points on a
tetrahedral mesh: triangular exterior-facet terms, Dirichlet rows / columns / lifting / set_bc, the
matrix-vector product on the reference's CSR layout and the outlet flux — against
oracle/ns3d_oracle.py (assemble_matrix_block / assemble_vector_block semantics,
src/solvers/stabilized_schur.py:144-175).  Tolerances: pattern bit-exact, matrices and vectors 1e-12.

The per-thread bodies of these kernels are also checked on the host (tests/test_tet_host.py); all of this file runs
green on a B200 (round 2), including the hemodynamic variants on a tetrahedral channel."""
import numpy as np
import pytest
import scipy.sparse as sp

from cfd_hemodynamic_b200.fem import discretization as D
from oracle import ns3d_oracle as O3
from oracle import ns_oracle as O
from oracle import simplex_oracle as S
from tests.test_simplex_oracle import FACET_COEFS
from tests.test_tet_host import _perturbed_cube

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


def _setup(hemo, x, cells, h, rules, frule, par, f):
    dev = hemo.device
    T = lambda a, dt=torch.float64: torch.tensor(np.ascontiguousarray(a), dtype=dt, device=dev)
    keep = dict(x=T(x), cells=T(cells, torch.int32), h=T(h))
    hemo.set_mesh(keep["x"], keep["cells"], keep["h"])
    nrowptr, ncol = D.node_graph(cells, x.shape[0])
    keep["nrowptr"], keep["ncol"] = T(nrowptr, torch.int32), T(ncol, torch.int32)
    hemo.set_node_graph(keep["nrowptr"], keep["ncol"])
    for b, k in enumerate(("Fu", "Fp", "uu", "up", "pu", "pp")):
        hemo.set_quadrature(b, *rules[k])
    hemo.set_facet_quadrature(*frule)
    hemo.set_params(par["dt"], par["rho"], par["mu"], f[:2], O.EPS0)
    hemo.set_body_force3(f)
    return T, keep


@pytest.mark.parametrize("with_bc", [False, True])
@pytest.mark.parametrize("coef", [FACET_COEFS[0], FACET_COEFS[3]])
def test_tet_facets_dirichlet_spmv_match_oracle(coef, with_bc):
    from cfd_hemodynamic_b200._lib import Hemo
    x, cells = _perturbed_cube(3, seed=4)
    E, n = cells.shape[0], x.shape[0]
    h = S.cell_diameter(x, cells)
    rng = np.random.default_rng(11)
    u, p, un = rng.standard_normal((n, 3)), rng.standard_normal(n), rng.standard_normal((n, 3))
    f = np.array([0.3, -0.2, 0.1])
    par = dict(dt=0.01, rho=1.3, mu=0.02)
    rules = {k: S.tet_gauss_jacobi(d) for k, d in dict(Fu=12, Fp=11, uu=12, up=11, pu=11, pp=10).items()}
    frule = S.triangle_facet_rule(4)
    pairs = S.exterior_facets(cells)
    fx = np.array([np.delete(x[cells[c]], lf, axis=0) for c, lf in pairs])
    tagged = np.isclose(fx[:, :, 0], 1.0).all(axis=1) | np.isclose(fx[:, :, 2], 0.0).all(axis=1)
    fpairs = pairs[tagged]
    fcells, fmask = D.pairs_by_cell(fpairs)
    bcs, bc_lists = [], []
    if with_bc:
        gu, gp = rng.standard_normal(3 * n), rng.standard_normal(n)
        n0 = np.nonzero(np.isclose(x[:, 0], 0.0))[0]
        n1 = np.nonzero(np.isclose(x[:, 1], 0.0))[0]
        n2 = np.nonzero(np.isclose(x[:, 0], 1.0))[0]
        bcs = [("u", n0, gu), ("u", n1, 2.0 * gu), ("p", n2, gp)]
        udofs = lambda nodes: (3 * nodes[:, None] + np.arange(3)[None]).reshape(-1)
        bc_lists = [udofs(n0), udofs(n1), 3 * n + n2]
    flag, mult, cellflag, g = D.dirichlet_arrays(n, cells, bcs, gdim=3)
    prob = O3.Problem3D(x=x, cells=cells, f=f, rules=rules, facet_sets=[O.FacetSet(pairs=fpairs, **coef)],
                        facet_rule=frule, **par)
    sol = np.concatenate([u.reshape(-1), p])
    A_ref, b_ref = O3.assemble_system(prob, sol, un.reshape(-1), g, bc_lists=bc_lists)

    hemo = Hemo(0)
    T, keep = _setup(hemo, x, cells, h, rules, frule, par, f)
    keep["fc"], keep["fm"] = T(fcells, torch.int32), T(fmask, torch.int32)
    hemo.set_facet_set(0, keep["fc"], keep["fm"], **coef)
    if with_bc:
        hemo.set_bc(T(flag, torch.uint8), T(mult), T(cellflag, torch.uint8))
    dev = hemo.device
    vals = torch.zeros(hemo.nnz, dtype=torch.float64, device=dev)
    bvec = torch.zeros(4 * n, dtype=torch.float64, device=dev)
    sol_d, un_d, g_d = T(sol), T(un.reshape(-1)), T(g)
    hemo.assemble_jacobian(sol_d, un_d, vals)
    hemo.assemble_residual(sol_d, un_d, g_d if with_bc else None, bvec)
    rowptr, col = hemo.get_pattern()
    xv = rng.standard_normal(4 * n)
    y = torch.zeros(4 * n, dtype=torch.float64, device=dev)
    hemo.spmv(vals, T(xv), y)
    q = hemo.outlet_flux(0, un_d)
    torch.cuda.synchronize()
    A_dev = sp.csr_matrix((vals.cpu().numpy(), col.cpu().numpy(), rowptr.cpu().numpy()), shape=(4 * n, 4 * n))
    assert np.linalg.norm((A_dev - A_ref).tocoo().data) < 1e-12 * np.linalg.norm(A_ref.data)
    assert np.linalg.norm(bvec.cpu().numpy() - b_ref) < 1e-12 * np.linalg.norm(b_ref)
    assert np.linalg.norm(y.cpu().numpy() - A_ref @ xv) < 1e-12 * np.linalg.norm(A_ref @ xv)
    assert abs(q - S.outlet_flux(x, cells, fpairs, un.reshape(-1))) < 1e-12
    if with_bc:
        d = np.nonzero(flag)[0]
        assert np.array_equal(A_dev.diagonal()[d], mult[d])
        assert np.array_equal(bvec.cpu().numpy()[d], sol[d] - g[d])
    # the assembly is atomic-free with a fixed summation order: bitwise reproducible
    vals2 = torch.zeros_like(vals)
    hemo.assemble_jacobian(sol_d, un_d, vals2)
    torch.cuda.synchronize()
    assert torch.equal(vals, vals2)
    hemo.close()


@pytest.mark.parametrize("schur_mode", ["laplace", "selfp"])
def test_tet_newton_step_matches_oracle(schur_mode):
    """First 3-D solve through the C-ABI: Newton iterations on the Ethier-Steinman problem of the
    reference's taylor_green scenario (src/scenarios/taylor_green.py:41-58: Dirichlet velocity and
    pressure on the whole boundary) with hemo_fgmres + the 3-D block preconditioner, against the
    oracle's sparse-LU Newton.  Tolerance 1e-8 relative L2 on velocity and pressure (north_star)."""
    from cfd_hemodynamic_b200._lib import Hemo
    from cfd_hemodynamic_b200.linear_solver import BlockSchurSolver
    from tests.test_ns3d_oracle import exact_pressure, exact_velocity
    nc, dt, rho, mu = 6, 0.005, 1.0, 1.0
    x, cells = O3.unit_cube_tets(nc)
    n = x.shape[0]
    h = S.cell_diameter(x, cells)
    f = np.zeros(3)
    rules = {k: S.tet_gauss_jacobi(d) for k, d in dict(Fu=12, Fp=11, uu=12, up=11, pu=11, pp=10).items()}
    frule = S.triangle_facet_rule(4)
    boundary = np.nonzero((np.abs(x - 0.5) > 0.5 - 1e-12).any(axis=1))[0]
    prob = O3.Problem3D(x=x, cells=cells, dt=dt, rho=rho, mu=mu, f=f, rules=rules)
    prob.bc_dofs = np.concatenate([(3 * boundary[:, None] + np.arange(3)[None, :]).reshape(-1), 3 * n + boundary])

    hemo = Hemo(0)
    T, keep = _setup(hemo, x, cells, h, rules, frule, dict(dt=dt, rho=rho, mu=mu), f)
    dev = hemo.device
    nrowptr, ncol = D.node_graph(cells, n)
    # "selfp": the reference's Schur approximation (stabilized_schur.py:231-235) formed on the device (k_tet_selfp)
    ks = BlockSchurSolver(hemo, nrowptr, ncol, boundary, boundary, dt=dt, rho=rho, mu=mu, rtol=1e-11, amg_cycles_p=2,
                          schur_mode=schur_mode)
    vals = torch.zeros(hemo.nnz, dtype=torch.float64, device=dev)
    bvec = torch.zeros(4 * n, dtype=torch.float64, device=dev)
    y = torch.zeros(4 * n, dtype=torch.float64, device=dev)

    un = exact_velocity(x, 0.0).reshape(-1)
    xk = np.concatenate([un, exact_pressure(x, 0.0)])
    x_d, un_d = T(xk), T(un)
    t = 0.0
    for step in range(2):
        t += dt
        gu, gp = exact_velocity(x, t).reshape(-1), exact_pressure(x, t)
        g = np.concatenate([gu, gp])
        flag, mult, cellflag, g_bc = D.dirichlet_arrays(n, cells, [("u", boundary, gu), ("p", boundary, gp)], gdim=3)
        hemo.set_bc(T(flag, torch.uint8), T(mult), T(cellflag, torch.uint8))
        g_d = T(g_bc)
        xk, its_ref = O3.newton_step(prob, xk, un, g)
        f0 = None
        for it in range(20):
            hemo.assemble_residual(x_d, un_d, g_d, bvec)
            fn = hemo.norm2(bvec)
            f0 = fn if f0 is None else f0
            if fn <= 1e-10 * f0 or fn < 1e-14:
                break
            hemo.assemble_jacobian(x_d, un_d, vals)
            ks.setup(vals)
            lin_its, _ = ks.solve(vals, bvec, y)
            assert lin_its < 200
            hemo.axpy(-1.0, y, x_d)
        assert it <= its_ref + 2
        got = x_d.cpu().numpy()
        eu = np.linalg.norm(got[:3 * n] - xk[:3 * n]) / np.linalg.norm(xk[:3 * n])
        ep = np.linalg.norm(got[3 * n:] - xk[3 * n:]) / np.linalg.norm(xk[3 * n:])
        assert eu < 1e-8 and ep < 1e-8, (step, eu, ep)
        un = xk[:3 * n].copy()
        un_d = T(un)
    ue = exact_velocity(x, t).reshape(-1)
    assert np.linalg.norm(got[:3 * n] - ue) / np.linalg.norm(ue) < 5e-3
    hemo.close()


def test_taylor_green_plugin_matches_oracle(tmp_path):
    """The reference's 3-D scenario through the plugin API (`Scenario` -> `Solver.setup/solveStep` on
    tetrahedra, src/scenarios/taylor_green.py) against the oracle's LU Newton: 1e-8 relative L2 after
    two steps, both sides converged tightly; then the reference time loop itself (`Scenario.solve`,
    boundary data refreshed after every step, error log against the exact solution)."""
    from cfd_hemodynamic_b200.fem import quadrature as Q
    from cfd_hemodynamic_b200.src.scenarios.taylor_green import TaylorGreenSimulation
    nc, dt, steps, mu = 6, 0.005, 2, 1.0
    tight = dict(snes_rtol=1e-12, snes_stol=0.0, ksp_rtol=1e-11, ksp_restart=100, amg_cycles_p=2)
    sc = TaylorGreenSimulation("stabilized_schur", dt, steps * dt, rho=1, mu=mu, n=nc, **tight)
    s = sc.solver
    assert s._tet and not s._nullspace           # Dirichlet pressure on the boundary: no constant-pressure mode
    x = sc.mesh.geometry.x
    cells = sc.mesh.geometry.dofmap
    n = x.shape[0]
    rules = {k: Q.tetrahedron_rule(d) for k, d in dict(Fu=12, Fp=11, uu=12, up=11, pu=11, pp=10).items()}
    ext = S.exterior_facets(cells)
    prob = O3.Problem3D(x=x, cells=cells, dt=dt, rho=1.0, mu=mu, f=np.zeros(3), rules=rules,
                        facet_sets=[O.FacetSet(pairs=ext, a_p=1.0, a_g=1.0)], facet_rule=Q.triangle_rule(2))
    boundary = np.nonzero((np.abs(x - 0.5) > 0.5 - 1e-12).any(axis=1))[0]
    prob.bc_dofs = np.concatenate([(3 * boundary[:, None] + np.arange(3)[None, :]).reshape(-1), 3 * n + boundary])
    un = sc.exact_velocity(0)(x.T).T.reshape(-1)
    xk = np.concatenate([un, np.zeros(n)])       # the reference starts from p = 0 (p_prev is never interpolated)
    t = 0.0
    for _ in range(steps):
        t += dt
        sc.update_boundary_conditions(t)
        s.solveStep()
        s.u_prev.x.array[:] = s.u_sol.x.array[:]
        s.p_prev.x.array[:] = s.p_sol.x.array[:]
        g = np.concatenate([sc.exact_velocity(t)(x.T).T.reshape(-1), sc.exact_pressure(t)(x.T)])
        xk, _ = O3.newton_step(prob, xk, un, g, rtol=1e-12)
        un = xk[:3 * n].copy()
    eu = np.linalg.norm(s.u_sol.x.array - xk[:3 * n]) / np.linalg.norm(xk[:3 * n])
    ep = np.linalg.norm(s.p_sol.x.array - xk[3 * n:]) / np.linalg.norm(xk[3 * n:])
    assert eu < 1e-8 and ep < 1e-8, (eu, ep)
    ue = sc.exact_velocity(t)(x.T).T.reshape(-1)
    assert np.linalg.norm(s.u_sol.x.array - ue) / np.linalg.norm(ue) < 5e-3

    # the reference loop (default tolerances): runs, logs the error against the exact solution
    sc2 = TaylorGreenSimulation("stabilized_schur", dt, 3 * dt, rho=1, mu=mu, n=4)
    sc2.write_output = False
    out = sc2.solve(str(tmp_path / "tg"))
    assert sc2.steps_done == 3
    errs = [float(line.split("error =")[1]) for line in open(f"{out}/err.txt")]
    assert len(errs) == 4 and errs[0] < 1e-12 and max(errs) < 5e-2
    norms = open(f"{out}/norms.txt").read()
    assert "L2 norm of velocity" in norms

    # the device-resident loop (wall shear stress, early-stop and L2 norms as kernels) gives the same fields
    from cfd_hemodynamic_b200.src.scenario import l2_norm_sq
    sc3 = TaylorGreenSimulation("stabilized_schur", dt, 3 * dt, rho=1, mu=mu, n=4)
    nsteps, norm_v, norm_p = sc3.solve_device(None, afterStepCallback=sc3.update_boundary_conditions)
    assert nsteps == 3
    assert np.array_equal(sc3.solver.u_sol.x.array, sc2.solver.u_sol.x.array)
    assert np.array_equal(sc3.solver.p_sol.x.array, sc2.solver.p_sol.x.array)
    assert abs(norm_v - np.sqrt(l2_norm_sq(sc2.mesh, sc2.solver.u_sol))) < 1e-12 * norm_v
    assert abs(norm_p - np.sqrt(l2_norm_sq(sc2.mesh, sc2.solver.p_sol))) < 1e-12 * norm_p
    w_host, w_dev = sc2.solver.shear_stress.x.array, sc3.solver.shear_stress.x.array
    assert np.abs(w_host).max() > 0 and np.abs(w_dev - w_host).max() < 1e-12 * np.abs(w_host).max()


def test_golden_tet_case_on_gpu():
    """The committed 3-D golden vectors (tests/golden/p1tet_small.npz) are reproduced by the CUDA path."""
    import os
    from cfd_hemodynamic_b200._lib import Hemo
    from tests.golden.make_golden_tet import COEF, GOLDEN_TET, bc_values, build_case
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", GOLDEN_TET))
    prob, fpairs, bcs, u, p, un = build_case()
    n = prob.n
    rules = {k: (gold[f"rule_{k}_pts"], gold[f"rule_{k}_wts"]) for k in prob.rules}
    hemo = Hemo(0)
    T, keep = _setup(hemo, prob.x, prob.cells, prob.h, rules, (gold["facet_pts"], gold["facet_wts"]),
                     dict(dt=prob.dt, rho=prob.rho, mu=prob.mu), prob.f)
    fcells, fmask = D.pairs_by_cell(fpairs)
    hemo.set_facet_set(0, T(fcells, torch.int32), T(fmask, torch.int32), **COEF)
    flag, mult, cellflag, g = D.dirichlet_arrays(n, prob.cells, bcs, gdim=3)
    assert np.array_equal(g, bc_values(n, bcs))
    hemo.set_bc(T(flag, torch.uint8), T(mult), T(cellflag, torch.uint8))
    dev = hemo.device
    xd, und = T(np.concatenate([gold["u"], gold["p"]])), T(gold["un"])
    vals = torch.zeros(hemo.nnz, dtype=torch.float64, device=dev)
    b = torch.zeros(4 * n, dtype=torch.float64, device=dev)
    hemo.assemble_jacobian(xd, und, vals)
    hemo.assemble_residual(xd, und, T(g), b)
    rowptr, col = hemo.get_pattern()
    torch.cuda.synchronize()
    A_gold = sp.csr_matrix((gold["data"], gold["indices"], gold["indptr"]), shape=(4 * n, 4 * n))
    A_gpu = sp.csr_matrix((vals.cpu().numpy(), col.cpu().numpy(), rowptr.cpu().numpy()), shape=(4 * n, 4 * n))
    assert np.linalg.norm((A_gpu - A_gold).tocoo().data) < 1e-12 * np.linalg.norm(gold["data"])
    assert np.linalg.norm(b.cpu().numpy() - gold["b"]) < 1e-12 * np.linalg.norm(gold["b"])
    hemo.close()


def test_tet_schur_operators_and_loud_failures():
    """P1 stiffness and lumped mass on tetrahedra (operators of the Schur-complement approximation) against
    numpy; the L2 norm kernel; entry points that do not exist in 3-D fail loudly."""
    from cfd_hemodynamic_b200._lib import Hemo, HemoError
    x, cells = _perturbed_cube(3, seed=2)
    n = x.shape[0]
    h = S.cell_diameter(x, cells)
    rules = {k: S.tet_gauss_jacobi(d) for k, d in dict(Fu=4, Fp=3, uu=4, up=3, pu=3, pp=2).items()}
    hemo = Hemo(0)
    T, keep = _setup(hemo, x, cells, h, rules, S.triangle_facet_rule(2), dict(dt=0.01, rho=1.3, mu=0.02), np.zeros(3))
    nrowptr, ncol = D.node_graph(cells, n)
    lap, mass = hemo.assemble_laplace_mass()
    torch.cuda.synchronize()
    det, dphi = S.simplex_geometry(x, cells)
    Ke = (det / 6.0)[:, None, None] * np.einsum("eai,ebi->eab", dphi, dphi)
    c64 = cells.astype(np.int64)
    L_ref = sp.coo_matrix((Ke.reshape(-1), (np.repeat(c64, 4, axis=1).reshape(-1), np.tile(c64, (1, 4)).reshape(-1))),
                          shape=(n, n)).tocsr()
    L_ref.sort_indices()
    assert np.array_equal(L_ref.indices, ncol) and np.array_equal(L_ref.indptr, nrowptr)
    assert np.linalg.norm(lap.cpu().numpy() - L_ref.data) < 1e-12 * np.linalg.norm(L_ref.data)
    m_ref = np.zeros(n)
    np.add.at(m_ref, cells.reshape(-1), np.repeat(det / 24.0, 4))
    assert np.linalg.norm(mass.cpu().numpy() - m_ref) < 1e-13 * np.linalg.norm(m_ref)
    # L2 norm of a P1 vector field: int |(x + 2y, z, 1)|^2 over the unit cube (exact for the consistent mass matrix)
    u = np.stack([x[:, 0] + 2 * x[:, 1], x[:, 2], np.ones(n)], axis=1).reshape(-1)
    exact = (1 / 3 + 4 / 3 + 1.0) + 1 / 3 + 1.0
    assert abs(hemo.l2_norm_sq(T(u), 3) - exact) < 1e-12
    assert abs(hemo.l2_norm_sq(T(np.full(n, 2.0)), 1) - 4.0) < 1e-12
    # the drag / lift integrals are the 2-D DFG forms
    with pytest.raises(HemoError):
        hemo.boundary_force(0, T(np.zeros(4 * n)))
    with pytest.raises(HemoError):
        hemo.l2_norm_sq(T(u), 2)
    hemo.close()


@pytest.mark.parametrize("double_setup", [False, True])
def test_tet_pressure_backflow_plugin_matches_oracle(double_setup):
    """The hemodynamic variant on tetrahedra (production use of the reference: src/experiments/config/arteria_lad.yaml:19
    runs the stabilized_schur family on P1 tetrahedral artery meshes): weak inlet pressure + Nitsche, resistance outlet,
    backflow stabilisation on a box channel through the plugin API, against the 3-D oracle's LU Newton (1e-8)."""
    from cfd_hemodynamic_b200.fem import mesh as M
    from cfd_hemodynamic_b200.fem import quadrature as Q
    from cfd_hemodynamic_b200.fem.space import Function
    from cfd_hemodynamic_b200.src.boundaryCondition import BoundaryCondition
    from cfd_hemodynamic_b200.src.solvers.stabilized_schur_pressure_backflow import Solver
    dt, rho, mu, p_in, R = 0.01, 1.0, 0.05, 3.0, 4.0
    mesh = M.create_box((0.0, 0.0, 0.0), (2.0, 1.0, 1.0), 6, 3, 3)
    x = mesh.geometry.x
    cells = mesh.geometry.dofmap
    n = x.shape[0]
    ext = M.exterior_facet_indices(mesh.topology)
    xm = x[mesh.topology.facet_vertices[ext]].mean(axis=1)
    vals = np.where(xm[:, 0] < 1e-9, 2, np.where(xm[:, 0] > 2 - 1e-9, 3, 4)).astype(np.int32)
    ft = M.MeshTags(mesh, 2, ext, vals)
    tags = {"inlet": 2, "outlet": 3, "wall": 4, "obstacle": None}
    tight = dict(snes_rtol=1e-12, snes_stol=0.0, ksp_rtol=1e-11, ksp_restart=150, amg_cycles_p=2)
    s = Solver(mesh, dt, rho, mu, [0.0, 0.0, 0.0], None, p_inlet=p_in, R_resistance=R, **tight)
    noslip = Function(s.V)
    bcw = BoundaryCondition(noslip)
    bcw.initTopological(2, ft.find(4))
    s.setup([bcw], [], facet_tags=ft, tags=tags)
    if double_setup:
        s.setup([bcw], [], facet_tags=ft, tags=tags)
    c = float(s._setup_count)
    assert s._tet and s.variant == "pressure_backflow" and c == (2.0 if double_setup else 1.0)
    rules = {k: Q.tetrahedron_rule(d) for k, d in dict(Fu=12, Fp=11, uu=12, up=11, pu=11, pp=10).items()}
    pairs = mesh.topology.facet_cell_pairs
    fs_in = O.FacetSet(pairs=pairs(ft.find(2)), pconst=c * p_in, a_n=c, beta_n=s.beta_nitsche)
    fs_out = O.FacetSet(pairs=pairs(ft.find(3)), pconst=0.0, a_s=c, a_b=c, beta_b=s.beta_backflow)
    prob = O3.Problem3D(x=x, cells=cells, dt=dt, rho=rho, mu=mu, f=np.zeros(3), rules=rules, facet_sets=[fs_in, fs_out],
                        facet_rule=Q.triangle_rule(4))
    wall_nodes = np.unique(mesh.topology.facet_vertices[ft.find(4)])
    prob.bc_dofs = (3 * wall_nodes[:, None] + np.arange(3)[None, :]).reshape(-1)
    xk, un, g = np.zeros(4 * n), np.zeros(3 * n), np.zeros(4 * n)
    frozen, pc = [0.0] * (s._setup_count - 1), 0.0
    for _ in range(3):
        s.solveStep()
        s.u_prev.x.array[:] = s.u_sol.x.array[:]
        s.p_prev.x.array[:] = s.p_sol.x.array[:]
        fs_out.pconst = 0.5 * (sum(frozen) + pc)
        xk, _ = O3.newton_step(prob, xk, un, g, rtol=1e-12)
        q = S.outlet_flux(x, cells, fs_out.pairs, un)                  # Q from the old u_prev (one-step lag)
        pc = s.alpha_damping * R * abs(q) + (1.0 - s.alpha_damping) * pc
        un = xk[:3 * n].copy()
    assert pc > 0.0 and abs(s._p_c - pc) <= 1e-9 * max(1.0, pc)
    eu = np.linalg.norm(s.u_sol.x.array - xk[:3 * n]) / np.linalg.norm(xk[:3 * n])
    ep = np.linalg.norm(s.p_sol.x.array - xk[3 * n:]) / np.linalg.norm(xk[3 * n:])
    assert eu < 1e-8 and ep < 1e-8, (eu, ep)
