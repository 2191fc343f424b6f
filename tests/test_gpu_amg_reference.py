"""The AMG V-cycles, their Galerkin products and the block preconditioner against the float64 model of
oracle/amg_oracle.py, on every kernel path of amg.cu.

Each configuration is a fresh library context on a lid-cavity Jacobian (walls and lid: Dirichlet multiplicity 2 at
the top corners, empty prolongator rows on the boundary).  Which kernels run depends on the level size, the row
length, the Chebyshev degrees, the cycle count, the prolongator density and the environment variables HEMO_PDL
(read at context creation), HEMO_NO_GRAPH (read by `Hemo()`) and HEMO_SELL (read by hemo_amg_finalize); every row
asserts the path it claims through `Hemo.amg_level_info`.

The hierarchies are stored and cycled in single precision; the model rounds only the stored operators.  Both
||e||_2 / ||x_ref||_2 and max|e| / max|x_ref| must stay below oracle.amg_oracle.AMG_TOL (the max norm catches one
wrong row).
"""
import numpy as np
import pytest
import scipy.sparse as sp

from tests import common as T

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import amg_oracle as AO  # noqa: E402

TOL = AO.AMG_TOL
GALERKIN_TOL = 1e-6       # level operators: the same float32-rounded products, summed in a different order


def _prolongation_kernel(c, which):
    """Kernel of the top-level prolongation (the rule of vcycle_t)."""
    P, n = c["s"].levels[which][0]["P"], c["n"]
    return "k_prolong_add_row" if P.nnz <= 6 * n and n >= 32768 else "k_transfer"


def _report(tag, what, errs, tol=TOL):
    print(f"AMGREF {tag:<22s} {what:<36s} rel2 {errs[0]:.2e} relmax {errs[1]:.2e} tol {tol:.0e}")
    assert errs[0] <= tol and errs[1] <= tol, (tag, what, errs)


def _check_galerkin(c, tag):
    h, n = c["hemo"], c["n"]
    for which, H in ((0, c["Hu"]), (1, c["Hp"])):
        bs = 2 if which == 0 else 1
        for l in range(H.nlev):
            if l == 0:
                indptr, indices = c["nrowptr"], c["ncol"]
            else:
                C = c["s"].levels[which][l - 1]["C"]
                indptr, indices = C.indptr, C.indices
            nb = len(indptr) - 1
            v = h.amg_level_values(which, l, len(indices) * bs * bs).cpu().numpy()
            G = sp.bsr_matrix((v.reshape(-1, bs, bs), indices, indptr), shape=(nb * bs, nb * bs)).tocsr()
            ref = H.ops[l]
            err = abs(G - ref).max() / abs(ref).max()
            print(f"AMGREF {tag:<22s} galerkin which={which} level={l:<2d} ({nb} nodes)    max-rel {err:.2e} tol {GALERKIN_TOL:.0e}")
            assert err <= GALERKIN_TOL, (tag, which, l, err)


def _check_apply(c, tag, which, seed=0, note=""):
    h, n = c["hemo"], c["n"]
    H = c["Hu"] if which == 0 else c["Hp"]
    info, fused = T.amg_paths(c, which)
    rng = np.random.default_rng(seed + which)
    b = rng.standard_normal(H.ops[0].shape[0])
    singular = which == 1 and c["project"]
    if singular:
        b -= b.mean()
    bd = torch.tensor(b, device=h.device)
    xd = torch.zeros_like(bd)
    h.amg_apply(which, bd, xd, c["cycles"])
    x = xd.cpu().numpy()
    ref = H.apply(b, c["cycles"], fused=fused, **c["kw"])
    if singular:
        x, ref = x - x.mean(), ref - ref.mean()
    path = f"L0 {info[0]['scope']}{' sell' if info[0]['sell'] else ''}, coarsest {info[-1]['scope']}"
    _report(tag, f"amg_apply which={which}{note} ({path})", AO.rel_errors(x, ref))
    return info


def _check_coarse_shift(c, tag, shift=0.25):
    """hemo_amg_setup_scalar with a relative diagonal shift of the coarsest dense solve (the singular pressure
    operators use 1e-8, which only moves the constant mode; a pinned operator shows the shift itself)."""
    c["hemo"].amg_setup_scalar(c["s"].lap, shift)
    c["Hp"] = AO.Hierarchy(AO.pressure_level0(c["lap"], c["pflag"]), c["s"].levels[1], 1, shift)
    _check_apply(c, tag, 1, note=f" shift {shift}")


def _check_pc(c, tag, mask=None, seed=5):
    h, n, s = c["hemo"], c["n"], c["s"]
    _, fused_u = T.amg_paths(c, 0)
    _, fused_p = T.amg_paths(c, 1)
    Hu = c["Hu"]
    if mask is not None:
        h.set_pc_mask(torch.tensor(mask.astype(np.uint8), device=h.device))
        s.setup(c["vals"])
        Hu = T.velocity_oracle(c, mask)
    try:
        rng = np.random.default_rng(seed)
        r = rng.standard_normal(3 * n)
        rd = torch.tensor(r, device=h.device)
        zd = torch.zeros_like(rd)
        h.pc_apply(c["vals"], rd, zd)
        z = zd.cpu().numpy()
        ref = AO.pc_apply_laplace(r, n, Hu, c["Hp"], AO.a01_block(c["J"], n), s.mass.cpu().numpy(),
                                  mass_coef=s.opts["schur_mass_coef"], lap_coef=s.opts["schur_lap_coef"],
                                  cycles_u=c["cycles"], cycles_p=c["cycles"], project_pressure=c["project"],
                                  p_dirichlet=c["pflag"], node_mask=None if mask is None else mask.astype(bool),
                                  cycle_kw_u=dict(fused=fused_u, **c["kw"]), cycle_kw_p=dict(fused=fused_p, **c["kw"]))
        a01 = "k_a01_residual_row" if n >= 32768 and len(c["ncol"]) <= 12 * n else "k_a01_residual"
        what = f"pc_apply {'mask' if mask is not None else 'no mask'} ({a01})"
        _report(tag, what + " u", AO.rel_errors(z[:2 * n], ref[:2 * n]))
        _report(tag, what + " p", AO.rel_errors(z[2 * n:], ref[2 * n:]))
    finally:
        if mask is not None:
            h.set_pc_mask(None)
            s.setup(c["vals"])


# (id, nx, cell, env, options, expected scope of level 0, level 0 on sliced ELL, expected scope of the coarsest level)
CASES = [
    ("csr41-d1", 40, "triangle", {}, dict(degree=2, degree_pre=1, ratio=4.0, cycles=1, smooth=True),
     "level", False, "cta"),
    ("csr41-d2-pin-nopdl", 40, "quadrilateral", {"HEMO_PDL": "0"},
     dict(degree=3, degree_pre=2, ratio=6.0, cycles=3, smooth=False, pin=True), "level", False, "cta"),
    ("sell193-tri", 192, "triangle", {}, dict(degree=2, degree_pre=1, ratio=4.0, cycles=1, smooth=False),
     "level", True, "cta"),
    ("sell193-quad", 192, "quadrilateral", {}, dict(degree=3, degree_pre=2, ratio=6.0, cycles=3, smooth=True),
     "level", True, "cta"),
    ("sell193-tri-nograph", 192, "triangle", {"HEMO_NO_GRAPH": "1"},
     dict(degree=3, degree_pre=1, ratio=6.0, cycles=3, smooth=True, pin=True), "level", True, "cta"),
    ("nosell193-quad", 192, "quadrilateral", {"HEMO_SELL": "0", "HEMO_PDL": "0"},
     dict(degree=2, degree_pre=1, ratio=4.0, cycles=1, smooth=False), "level", False, "cta"),
    ("fused15-nc3", 14, "triangle", {}, dict(degree=2, degree_pre=1, ratio=6.0, cycles=3, smooth=False),
     "cta", False, "cta"),
    ("fused15-nc1-nopdl", 14, "quadrilateral", {"HEMO_PDL": "0", "HEMO_NO_GRAPH": "1"},
     dict(degree=3, degree_pre=2, ratio=4.0, cycles=1, smooth=True, pin=True), "cta", False, "cta"),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_amg_matches_oracle(monkeypatch, case):
    tag, nx, cell, env, opts, scope0, sell0, scope_last = case
    c = T.lid_case(monkeypatch, nx, cell, env, **opts)
    try:
        _check_galerkin(c, tag)
        for which in (0, 1):
            info = _check_apply(c, tag, which)
            assert info[0]["scope"] == scope0, (tag, which, info)
            assert info[-1]["scope"] == scope_last, (tag, which, info)
            if which == 0:
                assert (info[0]["sell"] > 0) == sell0, (tag, info)
                if sell0:
                    assert info[0]["n"] % 32 == 1       # the last slice: one real row, 31 padded ones
        if tag.startswith(("csr41-d1", "sell193-tri", "csr41-d2")):
            _check_pc(c, tag)
            mask = np.zeros(c["n"], dtype=bool)
            mask[-(nx + 1):] = True                     # the last mesh row plays the ghost layer
            _check_pc(c, tag, mask)
        if c["pin"]:
            _check_coarse_shift(c, tag)
        print(f"AMGREF {tag:<22s} prolongation {_prolongation_kernel(c, 0)} (velocity), "
              f"{_prolongation_kernel(c, 1)} (pressure)")
    finally:
        c["hemo"].close()


def test_solver_opts_take_effect_without_new_setup(monkeypatch):
    """Changing options between calls (no new hemo_pc_setup) reaches the captured graphs of hemo_amg_apply,
    hemo_pc_apply and the FGMRES iteration."""
    tag = "stale-opts41"
    c = T.lid_case(monkeypatch, 40, "triangle", {}, degree=2, degree_pre=1, ratio=4.0, cycles=1)
    h, s, n = c["hemo"], c["s"], c["n"]
    try:
        rng = np.random.default_rng(11)
        b = rng.standard_normal(2 * n)
        bd = torch.tensor(b, device=h.device)
        xd = torch.zeros_like(bd)
        r = torch.tensor(rng.standard_normal(3 * n), device=h.device)
        z = torch.zeros_like(r)
        rhs = torch.tensor(c["J"] @ rng.standard_normal(3 * n), device=h.device)
        y = torch.zeros_like(rhs)
        h.amg_apply(0, bd, xd, 1)
        h.pc_apply(c["vals"], r, z)
        its2, _ = s.solve(c["vals"], rhs, y)
        _report(tag, "amg_apply degree 2", AO.rel_errors(xd.cpu().numpy(), c["Hu"].apply(b, 1, **c["kw"])))
        s.opts["cheb_degree"] = 3
        h.set_solver_opts(**s.opts)
        kw = dict(c["kw"], degree=3)
        h.amg_apply(0, bd, xd, 1)
        _report(tag, "amg_apply degree 3, same buffers", AO.rel_errors(xd.cpu().numpy(), c["Hu"].apply(b, 1, **kw)))
        h.pc_apply(c["vals"], r, z)
        _, fused_u = T.amg_paths(c, 0)
        _, fused_p = T.amg_paths(c, 1)
        ref = AO.pc_apply_laplace(r.cpu().numpy(), n, c["Hu"], c["Hp"], AO.a01_block(c["J"], n), s.mass.cpu().numpy(),
                                  mass_coef=s.opts["schur_mass_coef"], lap_coef=s.opts["schur_lap_coef"],
                                  project_pressure=True, cycle_kw_u=dict(fused=fused_u, **kw),
                                  cycle_kw_p=dict(fused=fused_p, **kw))
        _report(tag, "pc_apply degree 3 u", AO.rel_errors(z.cpu().numpy()[:2 * n], ref[:2 * n]))
        y.zero_()
        its3, _ = s.solve(c["vals"], rhs, y)
    finally:
        h.close()
    # the same solve in a context that had degree 3 from the start
    f = T.lid_case(monkeypatch, 40, "triangle", {}, degree=3, degree_pre=1, ratio=4.0, cycles=1)
    try:
        yf = torch.zeros(3 * n, dtype=torch.float64, device=f["hemo"].device)
        its3_fresh, _ = f["s"].solve(f["vals"], rhs, yf)
    finally:
        f["hemo"].close()
    print(f"AMGREF {tag:<22s} fgmres iterations: degree 2 {its2}, degree 3 after set_solver_opts {its3}, "
          f"degree 3 fresh {its3_fresh}")
    assert its3 == its3_fresh, (its2, its3, its3_fresh)
