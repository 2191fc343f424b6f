"""Shared builders for the parity tests: the same seeded problem is handed to
the numpy oracle (oracle/ns_oracle.py) and to the CUDA library."""
from __future__ import annotations

import numpy as np

from cfd_hemodynamic_b200.fem import mesh as M
from cfd_hemodynamic_b200.fem import quadrature as Q
from cfd_hemodynamic_b200.fem import discretization as D
from oracle import ns_oracle as O

BLOCK_DEGREE = {"Fu": 12, "Fp": 11, "uu": 12, "up": 11, "pu": 11, "pp": 10}
# Q1 quadrilaterals: hand-derived UFL degrees 22 / 20 / 18 (SURVEY.md §7.1) -> m = (deg + 2) // 2
BLOCK_DEGREE_QUAD = {"Fu": 22, "Fp": 20, "uu": 22, "up": 20, "pu": 20, "pp": 18}
BLOCK_ID = {"Fu": 0, "Fp": 1, "uu": 2, "up": 3, "pu": 4, "pp": 5}


def default_rules(cell_type="triangle"):
    if cell_type == "quadrilateral":
        return {k: Q.quadrilateral_rule(d) for k, d in BLOCK_DEGREE_QUAD.items()}
    return {k: Q.triangle_rule(d) for k, d in BLOCK_DEGREE.items()}


def perturbed_square(nx, ny, seed=0, amp=0.25, cell_type="triangle"):
    m = M.create_unit_square(None, nx, ny, cell_type=cell_type)
    x = m.geometry.x[:, :2].copy()
    rng = np.random.default_rng(seed)
    hx = 1.0 / max(nx, ny)
    interior = (np.abs(x - 0.5) < 0.5 - 1e-12).all(axis=1)
    x[interior] += amp * hx * (rng.random((int(interior.sum()), 2)) - 0.5)
    return M.Mesh(x, m.geometry.dofmap.copy(), cell_type=cell_type)


def smooth_fields(x, seed=1, U=1.0):
    """Seeded smooth trigonometric velocity + 1 % noise (SURVEY §8(d)); never zero."""
    rng = np.random.default_rng(seed)
    n = x.shape[0]
    u = np.empty((n, 2))
    u[:, 0] = U * np.sin(2.1 * x[:, 0] + 0.3) * np.cos(1.7 * x[:, 1])
    u[:, 1] = -U * np.cos(1.3 * x[:, 0]) * np.sin(2.3 * x[:, 1] + 0.2)
    un = 0.9 * u + 0.05 * U * np.cos(3.0 * x[:, :1] + x[:, 1:])
    u += 0.01 * U * rng.standard_normal(u.shape)
    un += 0.01 * U * rng.standard_normal(u.shape)
    p = np.sin(1.1 * x[:, 0]) * x[:, 1] + 0.01 * rng.standard_normal(n)
    return u.reshape(-1), p, un.reshape(-1)


def make_problem(mesh, dt=0.01, rho=1.3, mu=0.02, f=(0.3, -0.2), rules=None):
    x = mesh.geometry.x[:, :2].copy()
    cells = mesh.geometry.dofmap
    quad = mesh.topology.cell_name() == "quadrilateral"
    rules = rules or default_rules(mesh.topology.cell_name())
    return O.Problem(x=x, cells=cells, h=mesh.h(2, np.arange(cells.shape[0])), dt=dt, rho=rho, mu=mu,
                     f=np.asarray(f, dtype=float), rules=rules,
                     facet_rule=Q.interval_gauss(Q.FACET_POINTS_QUAD if quad else 2))


def facet_pairs_from_cellmask(cells, mask):
    out = []
    for c, m in zip(cells, mask):
        for lf in range(4):
            if m & (1 << lf):
                out.append((c, lf))
    return np.asarray(out, dtype=np.int32).reshape(-1, 2)


def setup_gpu(hemo, mesh, prob, facet_sets=(), bcs=None):
    """Load a Problem into a Hemo context.  facet_sets: list of (facets, coef dict).
    bcs: list of ('u'|'p', nodes, values)."""
    import torch
    dev = hemo.device
    x2 = torch.tensor(prob.x, dtype=torch.float64, device=dev).contiguous()
    cells = torch.tensor(prob.cells, dtype=torch.int32, device=dev).contiguous()
    h = torch.tensor(prob.h, dtype=torch.float64, device=dev)
    hemo.set_mesh(x2, cells, h)
    nrowptr, ncol = D.node_graph(prob.cells, prob.n)
    hemo.set_node_graph(torch.tensor(nrowptr, device=dev), torch.tensor(ncol, device=dev))
    for k, bid in BLOCK_ID.items():
        pts, wts = prob.rules[k]
        hemo.set_quadrature(bid, pts, wts)
    hemo.set_facet_quadrature(*prob.facet_rule)
    hemo.set_params(prob.dt, prob.rho, prob.mu, prob.f, prob.eps0)
    for sid, (facets, coef) in enumerate(facet_sets):
        fc, fm = D.facet_set_by_cell(mesh, facets)
        hemo.set_facet_set(sid, torch.tensor(fc, device=dev), torch.tensor(fm, device=dev), **coef)
    g = None
    if bcs:
        flag, mult, cellflag, gv = D.dirichlet_arrays(prob.n, prob.cells, bcs)
        hemo.set_bc(torch.tensor(flag, device=dev), torch.tensor(mult, device=dev),
                    torch.tensor(cellflag, device=dev))
        g = torch.tensor(gv, device=dev)
    return g, (nrowptr, ncol)


def oracle_bcs(prob, bcs):
    """Convert ('u', nodes, values) → oracle (block, unrolled dofs, g) tuples."""
    out = []
    for block, nodes, values in bcs:
        nodes = np.asarray(nodes, dtype=np.int64)
        if block == "u":
            d = (2 * nodes[:, None] + np.arange(2)[None, :]).reshape(-1)
        else:
            d = nodes
        out.append((block, d, np.asarray(values, dtype=float)))
    return out


def oracle_problem_from_solver(s, facet_tags=None, tags=None):
    """Build the oracle Problem that mirrors a B200 solver instance after setup():
    same mesh, parameters, quadrature rules, Dirichlet objects (in list order) and the
    boundary terms of its variant with the setup() multiplicity (SURVEY §7.3-1)."""
    from cfd_hemodynamic_b200.fem import mesh as M
    mesh = s.mesh
    fval = np.asarray(s.f.value, dtype=float).reshape(-1)[:2]
    prob = make_problem(mesh, dt=float(s.dt.value), rho=float(s.rho.value), mu=float(s.mu.value), f=fval)
    bcs = [("u", bc.block_dofs, bc.g.x.array.copy()) for bc in s.bcu_d]
    bcs += [("p", bc.block_dofs, bc.g.x.array.copy()) for bc in s.bcp_d]
    prob.bcs = oracle_bcs(prob, bcs)
    c = float(s._setup_count)
    fs = []
    if s.variant == "schur":
        ext = M.exterior_facet_indices(mesh.topology)
        fs.append(O.FacetSet(pairs=mesh.topology.facet_cell_pairs(ext), a_p=1.0, a_g=1.0))
    elif s.variant == "backflow":
        out = facet_tags.find(tags["outlet"])
        fs.append(O.FacetSet(pairs=mesh.topology.facet_cell_pairs(out), a_b=c, beta_b=s.beta_backflow))
    elif s.variant == "velocity_vascular_backflow":
        out = facet_tags.find(tags["outlet"])
        fs.append(O.FacetSet(pairs=mesh.topology.facet_cell_pairs(out), pconst=0.0, a_s=c, a_b=c,
                             beta_b=s.beta_backflow))
    else:
        fin = facet_tags.find(tags["inlet"])
        out = facet_tags.find(tags["outlet"])
        fs.append(O.FacetSet(pairs=mesh.topology.facet_cell_pairs(fin), pconst=c * s.p_inlet, a_n=c,
                             beta_n=s.beta_nitsche))
        fs.append(O.FacetSet(pairs=mesh.topology.facet_cell_pairs(out), pconst=0.0, a_s=c, a_b=c,
                             beta_b=s.beta_backflow))
    prob.facet_sets = fs
    return prob


def lid_case(monkeypatch, nx, cell="triangle", env=None, *, pin=False, smooth=True, degree=2, degree_pre=1, ratio=4.0,
             cycles=1, oracle=True):
    """Fresh context with the lid-cavity Jacobian and a set-up block preconditioner (walls and lid: Dirichlet
    multiplicity 2 at the top corners).  `env` is set before the context is created; `oracle` adds the float64 AMG
    models of both hierarchies (oracle/amg_oracle.py) as "Hu" and "Hp"."""
    import scipy.sparse as sp
    import torch
    from cfd_hemodynamic_b200._lib import Hemo
    from cfd_hemodynamic_b200.linear_solver import BlockSchurSolver
    from oracle import amg_oracle as AO
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    hemo = Hemo(0)
    mesh = M.create_unit_square(None, nx, nx, cell_type=cell)
    prob = make_problem(mesh, dt=0.01, rho=1.0, mu=0.05, f=(0.0, 0.0))
    x, n = prob.x, prob.n
    ext = M.exterior_facet_indices(mesh.topology)
    walls = np.nonzero(np.isclose(x[:, 0], 0) | np.isclose(x[:, 0], 1) | np.isclose(x[:, 1], 0))[0]
    lidf = M.locate_entities_boundary(mesh, 1, lambda X: np.isclose(X[1], 1.0) & (X[0] > 1e-10) & (X[0] < 1 - 1e-10))
    lid = np.unique(mesh.topology.facet_vertices[lidf])
    g1 = np.zeros(2 * n)
    g1[0::2] = 1.0
    bcs = [("u", walls, np.zeros(2 * n)), ("u", lid, g1)]
    pnodes = np.zeros(0, dtype=np.int64)
    if pin:                                   # one pinned pressure dof in the middle of the bottom wall
        pnodes = np.array([int(np.argmin(np.abs(x[:, 0] - 0.5) + np.abs(x[:, 1])))])
        bcs.append(("p", pnodes, np.zeros(n)))
    prob.facet_sets = [O.FacetSet(pairs=mesh.topology.facet_cell_pairs(ext), a_p=1.0, a_g=1.0)]
    _, (nrowptr, ncol) = setup_gpu(hemo, mesh, prob, [(ext, dict(a_p=1.0, a_g=1.0))], bcs)
    u, p, un = smooth_fields(x, seed=2, U=0.5)
    vals = torch.zeros(hemo.nnz, dtype=torch.float64, device=hemo.device)
    hemo.assemble_jacobian(torch.tensor(np.concatenate([u, p]), device=hemo.device),
                           torch.tensor(un, device=hemo.device), vals)
    rowptr, col = hemo.get_pattern()
    J = sp.csr_matrix((vals.cpu().numpy(), col.cpu().numpy(), rowptr.cpu().numpy()), shape=(3 * n, 3 * n))
    s = BlockSchurSolver(hemo, nrowptr, ncol, np.unique(np.concatenate([walls, lid])), pnodes, dt=prob.dt, rho=prob.rho,
                         mu=prob.mu, project_pressure=not pin, smooth_prolongator=smooth, cheb_degree=degree,
                         cheb_degree_pre=degree_pre, cheb_ratio=ratio, amg_cycles_u=cycles, amg_cycles_p=cycles)
    s.setup(vals)
    pflag = np.zeros(n, dtype=bool)
    pflag[pnodes] = True
    lap = sp.csr_matrix((s.lap.cpu().numpy(), ncol, nrowptr), shape=(n, n))
    c = dict(hemo=hemo, s=s, n=n, nx=nx, J=J, vals=vals, nrowptr=nrowptr, ncol=ncol, lap=lap, pflag=pflag, pin=pin,
             project=not pin, cycles=cycles, kw=dict(degree=degree, degree_pre=degree_pre, ratio=ratio))
    if oracle:
        c["Hp"] = AO.Hierarchy(AO.pressure_level0(lap, pflag), s.levels[1], 1, 0.0 if pin else 1e-8)
        c["Hu"] = velocity_oracle(c)
    return c


def velocity_oracle(c, mask=None):
    """The float64 model of the velocity hierarchy of a `lid_case`, with the preconditioner's node mask."""
    from oracle import amg_oracle as AO
    return AO.Hierarchy(AO.velocity_level0(c["J"], c["n"], mask), c["s"].levels[0], 2)


def amg_paths(c, which):
    """amg_level_info of every level of hierarchy `which` of a `lid_case`, and the levels inside the fused coarse
    V-cycle kernel."""
    h = c["hemo"]
    info = [h.amg_level_info(which, l) for l in range(len(c["s"].levels[which]) + 1)]
    return info, {l for l, d in enumerate(info) if d["scope"] == "cta"}
