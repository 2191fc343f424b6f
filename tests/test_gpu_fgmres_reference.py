"""The device-resident FGMRES (csrc/krylov.cu) against the float64 model of oracle/fgmres_oracle.py.

A solve is deterministic, so the same right-hand side solved with max_it = k gives the first k iterations of the long
solve: its iterate and its residual estimate after k iterations.  For every sampled k each row checks
  * the iteration count against the model's,
  * |rel_resid_gpu - rel_resid_model| (the model's estimate after k iterations),
  * ||y_gpu - y_model|| / ||y_model||,
  * the estimate against the true residual of the library's own iterate, ||b - J y_gpu|| / ||b|| (J in float64 from
    `get_pattern`; no model involved),
with the model run twice: on the library's own `hemo_pc_apply` (black box: only the Krylov arithmetic differs) and on
the float64 AMG model `amg_oracle.pc_apply_laplace` (independent).  Each row asserts the exit reason it claims.
"""
import numpy as np
import pytest
import scipy.sparse as sp

from tests import common as T

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import amg_oracle as AO  # noqa: E402
from oracle import fgmres_oracle as FO  # noqa: E402


def _set(c, **kw):
    c["s"].opts.update(kw)
    c["hemo"].set_solver_opts(**c["s"].opts)


def _gpu_solve(c, b, max_it=None, vals=None):
    """(y, its, rel_resid, reason) of one hemo_fgmres from y = 0."""
    from cfd_hemodynamic_b200._lib import HemoDiverged
    h = c["hemo"]
    if max_it is not None:
        _set(c, max_it=max_it)
    bd = torch.tensor(b, device=h.device)
    yd = torch.zeros_like(bd)
    try:
        its, rr = h.fgmres(c["vals"] if vals is None else vals, bd, yd)
        reason = "converged"
    except HemoDiverged as e:
        its, rr = e.its, e.rel_resid
        reason = "nonfinite" if "not finite" in str(e) else "max_it"
    return yd.cpu().numpy(), its, rr, reason


def _blackbox_pc(c):
    h = c["hemo"]

    def pc(v):
        vd = torch.tensor(v, device=h.device)
        zd = torch.zeros_like(vd)
        h.pc_apply(c["vals"], vd, zd)
        return zd.cpu().numpy()
    return pc


def _independent_pc(c):
    n, s = c["n"], c["s"]
    _, fused_u = T.amg_paths(c, 0)
    _, fused_p = T.amg_paths(c, 1)
    A01, mass = AO.a01_block(c["J"], n), s.mass.cpu().numpy()
    kw = dict(mass_coef=s.opts["schur_mass_coef"], lap_coef=s.opts["schur_lap_coef"], cycles_u=c["cycles"],
              cycles_p=c["cycles"], project_pressure=c["project"], p_dirichlet=c["pflag"] if c["pin"] else None,
              cycle_kw_u=dict(fused=fused_u, **c["kw"]), cycle_kw_p=dict(fused=fused_p, **c["kw"]))
    return lambda v: AO.pc_apply_laplace(v, n, c["Hu"], c["Hp"], A01, mass, **kw)


def _report(tag, what, err, at, tol):
    where = "" if at is None else f" (k={at})"
    print(f"FGMREF {tag:<14s} {what:<44s} {err:.2e} tol {tol:.0e}{where}")
    assert err <= tol, (tag, what, err, at)


def _sample(its, m, every):
    if every:
        return list(range(1, its + 1))
    ks = {its}
    for q in range(1, its // m + 1):
        ks |= {q * m - 1, q * m, q * m + 1}
    return sorted(k for k in ks if 1 <= k <= its)


def _run_row(c, tag, b, *, restart, rtol, atol=0.0, max_it=1000, reason, every=True, pcs=("blackbox", "independent"),
             owned=None):
    """The long solve, its truncations at the sampled k and the model on each preconditioner.  Returns the GPU data."""
    _set(c, restart=restart, rtol=rtol, atol=atol)
    J = c["J"]
    mask = np.ones(len(b), dtype=bool) if owned is None else owned
    bn = np.linalg.norm(b[mask])
    yL, itsL, rrL, reasonL = _gpu_solve(c, b, max_it)
    assert reasonL == reason, (tag, reasonL, itsL, rrL)
    ks = _sample(itsL, restart, every)
    gpu = {}
    est = []
    for k in ks:
        y, its, rr, rsn = _gpu_solve(c, b, k)
        assert its == k, (tag, k, its, rsn)
        gpu[k] = (y, rr)
        est.append((abs(rr - np.linalg.norm((b - J @ y)[mask]) / bn), k))
    # a truncation at the long solve's count is the long solve
    assert np.array_equal(gpu[itsL][0], yL), tag
    _report(tag, "estimate vs ||b - J y_gpu|| / ||b||", *max(est), tol=FO.ESTIMATE_TOL)
    for name in pcs:
        pc = _blackbox_pc(c) if name == "blackbox" else _independent_pc(c)
        r = FO.fgmres(lambda z: J @ z, pc, b, restart=restart, max_it=max_it, rtol=rtol, atol=atol, owned=owned,
                      snapshots=ks)
        assert (r.reason, r.its) == (reasonL, itsL), (tag, name, r.reason, r.its, reasonL, itsL)
        assert r.reason != "breakdown"
        rtol_r, ytol = ((FO.BLACKBOX_RESID_TOL, FO.BLACKBOX_Y_TOL) if name == "blackbox" else
                        (FO.INDEP_RESID_TOL, FO.INDEP_Y_TOL))
        er, ey = [], []
        for k in ks:
            y, rr = gpu[k]
            ref = r.history[k - 1] / bn
            er.append((abs(rr - ref), k))
            ym = r.snapshots[k]
            if name == "blackbox" or ref >= FO.INDEP_Y_ABOVE:
                ey.append((np.linalg.norm(y - ym) / np.linalg.norm(ym), k))
        _report(tag, f"{name}: |rel_resid - model|", *max(er), tol=rtol_r)
        if ey:
            _report(tag, f"{name}: ||y - y_model|| / ||y_model||", *max(ey), tol=ytol)
        if reasonL == "converged":
            _report(tag, f"{name}: final rel_resid - model", abs(rrL - r.rel_resid), None, tol=rtol_r)
        print(f"FGMREF {tag:<14s} {name}: its {r.its} ({r.reason}), restarts after {r.cycle_ends}, {len(ks)} k sampled")
    return dict(y=yL, its=itsL, rel_resid=rrL, ks=ks)


def _rhs(c, seed=4):
    """A right-hand side in the range of J (the pressure of an unpinned case is determined up to a constant)."""
    return c["J"] @ np.random.default_rng(seed).standard_normal(c["J"].shape[0])


# (id, nx, cell, env, lid_case options, restart, rtol, atol (x ||b||), max_it, exit reason, every k)
ROWS = [
    ("a-tri41-m60", 40, "triangle", {}, {}, 60, 1e-8, 0.0, 1000, "converged", True),
    ("b-tri41-m5", 40, "triangle", {}, {}, 5, 1e-8, 0.0, 1000, "converged", True),
    ("c-quad41-16", 40, "quadrilateral", {}, dict(pin=True), 8, 1e-14, 0.0, 16, "max_it", True),
    ("c-quad41-13", 40, "quadrilateral", {}, dict(pin=True), 8, 1e-14, 0.0, 13, "max_it", True),
    ("d-tri41-m1", 40, "triangle", {}, {}, 1, 1e-8, 0.0, 20, "max_it", True),
    ("e-quad193-m12", 192, "quadrilateral", {}, {}, 12, 1e-9, 0.0, 1000, "converged", False),
    ("g-tri41-m5-nopdl", 40, "triangle", {"HEMO_PDL": "0"}, {}, 5, 1e-8, 0.0, 1000, "converged", True),
    ("h-tri41-atol", 40, "triangle", {}, {}, 60, 1e-12, 1e-3, 1000, "converged", True),
]


@pytest.mark.parametrize("row", ROWS, ids=[r[0] for r in ROWS])
def test_fgmres_matches_model(monkeypatch, row):
    tag, nx, cell, env, opts, restart, rtol, atol_rel, max_it, reason, every = row
    c = T.lid_case(monkeypatch, nx, cell, env, **opts)
    try:
        b = _rhs(c)
        atol = atol_rel * np.linalg.norm(b)
        out = _run_row(c, tag, b, restart=restart, rtol=rtol, atol=atol, max_it=max_it, reason=reason, every=every)
        if tag.startswith("e"):
            assert out["its"] > restart + 1, out["its"]            # at least one restart
        if tag.startswith("h"):
            # atol ends the solve: the estimate is below atol but far above rtol ||b||
            assert 1e-9 < out["rel_resid"] <= 1e-3, out["rel_resid"]
        if tag.startswith("c"):
            assert out["its"] == max_it and (max_it % restart == 0) == tag.endswith("16")
    finally:
        c["hemo"].close()


def test_long_cycle_through_direct_launches(monkeypatch):
    """Row f: 193^2, no graphs, a weakened preconditioner (Chebyshev degree 1, plain prolongator) and restart 400 (the
    largest the library takes: the largest kpad and shared-memory sizes), so more than 100 columns in one cycle."""
    c = T.lid_case(monkeypatch, 192, "triangle", {"HEMO_NO_GRAPH": "1"}, degree=1, smooth=False)
    try:
        b = _rhs(c)
        out = _run_row(c, "f-tri193-m400", b, restart=400, rtol=1e-12, reason="converged", every=False)
        print(f"FGMREF f-tri193-m400  {out['its']} columns in one cycle")
        assert 100 < out["its"] < 400, out["its"]
    finally:
        c["hemo"].close()


def test_degenerate_right_hand_sides(monkeypatch):
    """Row i: b = 0 and ||b|| <= atol end before the first iteration with y = 0; a NaN in b, and a NaN in the
    operator, end with HemoDiverged ("not finite"); the context then solves a normal b bitwise like a fresh one."""
    c = T.lid_case(monkeypatch, 40, "triangle", oracle=False)
    tag = "i-tri41"
    try:
        b = _rhs(c)
        _set(c, restart=60, rtol=1e-8, atol=0.0, max_it=1000)
        y, its, rr, reason = _gpu_solve(c, np.zeros_like(b))
        assert (its, rr, reason) == (0, 0.0, "converged") and not y.any()
        _set(c, atol=2 * np.linalg.norm(b))
        y, its, rr, reason = _gpu_solve(c, b)
        assert (its, rr, reason) == (0, 1.0, "converged") and not y.any()
        _set(c, atol=0.0)
        bnan = b.copy()
        bnan[len(b) // 2] = np.nan
        y, its, rr, reason = _gpu_solve(c, bnan)
        assert (its, reason) == (0, "nonfinite") and not y.any(), (its, rr, reason)
        # a NaN in the operator reaches the first Hessenberg column
        vnan = c["vals"].clone()
        vnan[vnan.numel() // 2] = float("nan")
        y, its, rr, reason = _gpu_solve(c, b, vals=vnan)
        assert (its, reason) == (1, "nonfinite"), (its, rr, reason)
        for bb, why, jn in ((np.zeros_like(b), "converged", c["J"]), (bnan, "nonfinite", c["J"])):
            r = FO.fgmres(lambda z: jn @ z, lambda v: v, bb, restart=60, max_it=1000, rtol=1e-8, atol=0.0)
            assert (r.reason, r.its) == (why, 0)
        y_after = _gpu_solve(c, b)
    finally:
        c["hemo"].close()
    f = T.lid_case(monkeypatch, 40, "triangle", oracle=False)
    try:
        _set(f, restart=60, rtol=1e-8, atol=0.0, max_it=1000)
        y_fresh = _gpu_solve(f, b)
    finally:
        f["hemo"].close()
    assert np.array_equal(y_after[0], y_fresh[0]) and y_after[1:] == y_fresh[1:]
    print(f"FGMREF {tag:<14s} b = 0, ||b|| <= atol, NaN in b, NaN in J: exits as modelled; "
          f"next solve bitwise equal to a fresh context ({y_after[1]} its)")


def _tet_case(schur_mode):
    from cfd_hemodynamic_b200._lib import Hemo
    from cfd_hemodynamic_b200.fem import discretization as D
    from cfd_hemodynamic_b200.linear_solver import BlockSchurSolver
    from oracle import ns3d_oracle as O3
    from oracle import simplex_oracle as S
    from tests.test_gpu_zz_tet3d import _setup
    from tests.test_ns3d_oracle import exact_pressure, exact_velocity
    dt, rho, mu = 0.005, 1.0, 1.0
    x, cells = O3.unit_cube_tets(6)
    n = x.shape[0]
    rules = {k: S.tet_gauss_jacobi(d) for k, d in dict(Fu=12, Fp=11, uu=12, up=11, pu=11, pp=10).items()}
    boundary = np.nonzero((np.abs(x - 0.5) > 0.5 - 1e-12).any(axis=1))[0]
    hemo = Hemo(0)
    Tt, keep = _setup(hemo, x, cells, S.cell_diameter(x, cells), rules, S.triangle_facet_rule(4),
                      dict(dt=dt, rho=rho, mu=mu), np.zeros(3))
    nrowptr, ncol = D.node_graph(cells, n)
    gu, gp = exact_velocity(x, dt).reshape(-1), exact_pressure(x, dt)
    s = BlockSchurSolver(hemo, nrowptr, ncol, boundary, boundary, dt=dt, rho=rho, mu=mu, amg_cycles_p=2,
                         schur_mode=schur_mode)
    flag, mult, cellflag, _ = D.dirichlet_arrays(n, cells, [("u", boundary, gu), ("p", boundary, gp)], gdim=3)
    hemo.set_bc(Tt(flag, torch.uint8), Tt(mult), Tt(cellflag, torch.uint8))
    un = exact_velocity(x, 0.0).reshape(-1)
    vals = torch.zeros(hemo.nnz, dtype=torch.float64, device=hemo.device)
    hemo.assemble_jacobian(Tt(np.concatenate([un, exact_pressure(x, 0.0)])), Tt(un), vals)
    s.setup(vals)
    rowptr, col = hemo.get_pattern()
    J = sp.csr_matrix((vals.cpu().numpy(), col.cpu().numpy(), rowptr.cpu().numpy()), shape=(4 * n, 4 * n))
    return dict(hemo=hemo, s=s, n=n, J=J, vals=vals, keep=keep)


@pytest.mark.parametrize("schur_mode", ["laplace", "selfp"])
def test_tet_fgmres_matches_model(schur_mode):
    """Row j: tetrahedra (k_fg_store after hemo_tet_spmv, the restart through hemo_tet_spmv); black box only."""
    c = _tet_case(schur_mode)
    try:
        b = np.random.default_rng(8).standard_normal(4 * c["n"])
        out = _run_row(c, f"j-tet-{schur_mode}", b, restart=4, rtol=1e-8, reason="converged", pcs=("blackbox",))
        assert out["its"] > 5, out["its"]                           # at least one restart
    finally:
        c["hemo"].close()


def _single_rank(c, n_owned):
    from cfd_hemodynamic_b200._lib import Hemo, HemoError
    try:
        uid = Hemo.comm_unique_id()
    except HemoError as e:
        pytest.skip(f"NCCL cannot be loaded: {e}")
    h = c["hemo"]
    h.comm_init(uid, 0, 1)
    h.comm_set_partition(n_owned, np.zeros(0, np.int32), np.zeros(1, np.int32), np.zeros(0, np.int32),
                         np.zeros(1, np.int32))


@pytest.mark.parametrize("gap", [False, True], ids=["k-all-owned", "l-last-row-unowned"])
def test_owned_segment_reductions(monkeypatch, gap):
    """Rows k and l: a single-rank communicator without neighbours switches the reductions to the owned-segment
    kernels (k_fg_mdot<true>, the separate k_fg_givens); with the last mesh row left unowned the segments have a real
    gap, and the model takes the owned mask."""
    tag = "l-tri41-gap" if gap else "k-tri41-seg"
    c = T.lid_case(monkeypatch, 40, "triangle")
    n, nx = c["n"], c["nx"]
    n_owned = n - (nx + 1) if gap else n
    owned = None
    if gap:
        node = np.concatenate([np.arange(n).repeat(2), np.arange(n)])
        owned = node < n_owned
    try:
        b = _rhs(c)
        _single_rank(c, n_owned)
        out = _run_row(c, tag, b, restart=5, rtol=1e-8, reason="converged", owned=owned)
    finally:
        c["hemo"].close()
    if not gap:
        f = T.lid_case(monkeypatch, 40, "triangle", oracle=False)
        try:
            _set(f, restart=5, rtol=1e-8, atol=0.0, max_it=1000)
            y, its, rr, _ = _gpu_solve(f, b)
        finally:
            f["hemo"].close()
        same = np.array_equal(y, out["y"]) and (its, rr) == (out["its"], out["rel_resid"])
        print(f"FGMREF {tag:<14s} bitwise equal to row b (no communicator): {same}")


# ---------------------------------------------------------------------------------------------------------------------
POLL_ROWS = [("b-tri41-m5", 40, "triangle", 5), ("e-quad193-m12", 192, "quadrilateral", 12)]
SETTINGS = [("default", {}), ("nopdl", {"HEMO_PDL": "0"}), ("nograph", {"HEMO_NO_GRAPH": "1"})]


@pytest.mark.parametrize("setting", SETTINGS, ids=[s[0] for s in SETTINGS])
@pytest.mark.parametrize("row", POLL_ROWS, ids=[r[0] for r in POLL_ROWS])
def test_iterations_queued_after_convergence_change_nothing(monkeypatch, row, setting):
    """The host queues iterations up to the previous solve's count before it reads the flag.  A solve that converges
    earlier than that must give the bits of a solve that polls after every iteration: the iteration kernels queued
    after convergence return at once, and the preconditioner kernels they bring along write only its scratch."""
    tag, nx, cell, m = row
    name, env = setting
    tight, loose = 1e-10, 1e-4

    def ctx():
        c = T.lid_case(monkeypatch, nx, cell, env, oracle=False)
        _set(c, restart=m, rtol=loose, atol=0.0, max_it=1000)
        return c

    results = {}
    a = ctx()
    try:
        b = _rhs(a)
        _set(a, rtol=tight)
        k1 = _gpu_solve(a, b)[1]
        _set(a, rtol=loose)
        l0 = a["hemo"].launches
        results["A"] = _gpu_solve(a, b)
        da = a["hemo"].launches - l0
    finally:
        a["hemo"].close()
    for every in (1, 7):
        c = ctx()
        try:
            c["hemo"].set_poll_interval(every)
            l0 = c["hemo"].launches
            results[every] = _gpu_solve(c, b)
            d = c["hemo"].launches - l0
            if every == 1:
                db = d
                # launches of one iteration: a solve of two iterations minus a solve of one (one cycle each)
                l1 = c["hemo"].launches
                _gpu_solve(c, b, max_it=1)
                l2 = c["hemo"].launches
                _gpu_solve(c, b, max_it=2)
                per_it = (c["hemo"].launches - l2) - (l2 - l1)
        finally:
            c["hemo"].close()
    k2 = results["A"][1]
    queued = min(k1 - 1, -(-k2 // m) * m)          # up to the prediction, never past the end of the cycle
    print(f"FGMREF poll {tag:<14s} {name:<8s} K1 {k1} K2 {k2} restart {m}: {queued} queued, launches {da} vs {db} "
          f"with poll 1 ({per_it} per iteration)")
    for k in (1, 7):
        assert np.array_equal(results["A"][0], results[k][0]) and results["A"][1:] == results[k][1:], (k, results[k][1:])
    assert results["A"][3] == "converged"
    assert queued >= k2 + 2, (k1, k2, m)
    assert da - db == (queued - k2) * per_it, (da, db, queued, k2, per_it)


def test_restart_changed_on_a_live_context(monkeypatch):
    """Restart 60, 5, 60 on one context (reallocation of the basis, a new iteration graph, the previous solve's
    iteration count from the other restart) gives the bits of fresh contexts."""
    seq = [60, 5, 60]
    c = T.lid_case(monkeypatch, 40, "triangle", oracle=False)
    live = []
    try:
        b = _rhs(c)
        for m in seq:
            _set(c, restart=m, rtol=1e-8, atol=0.0, max_it=1000)
            live.append(_gpu_solve(c, b))
    finally:
        c["hemo"].close()
    for m, got in zip(seq, live):
        f = T.lid_case(monkeypatch, 40, "triangle", oracle=False)
        try:
            _set(f, restart=m, rtol=1e-8, atol=0.0, max_it=1000)
            ref = _gpu_solve(f, b)
        finally:
            f["hemo"].close()
        assert np.array_equal(got[0], ref[0]) and got[1:] == ref[1:], (m, got[1:], ref[1:])
    print(f"FGMREF restart 60/5/60 live context: its {[r[1] for r in live]}, bitwise equal to fresh contexts")
