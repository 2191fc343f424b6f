"""Float64 model of the device-resident FGMRES(restart) of csrc/krylov.cu (`hemo_fgmres`).

Right-preconditioned flexible GMRES with classical Gram-Schmidt (every coefficient from the same w, no
re-orthogonalisation), Givens rotations on the Hessenberg column, restart from the true residual b - A y, and the
library's stopping rules: tol = max(rtol ||b||, atol) fixed by the first cycle, tests in the order non-finite, res <=
tol, happy breakdown.  The preconditioner is any callable, so the same loop runs against the library's own
`hemo_pc_apply` (black box: only the Krylov arithmetic is modelled) or against `amg_oracle.pc_apply_laplace`.

`owned` (boolean mask) models the owned-segment reductions (`FgSeg`): every inner product and norm runs over the
owned entries only, while the operator, the preconditioner and the vector updates act on the whole vector.

numpy only.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

# Tolerances of the library against this model (tests/test_gpu_fgmres_reference.py).  Measured on a B200 (1000 W
# power limit), the largest over every row of that file:
#   black box (the library's own preconditioner applied to the model's vectors):
#     |rel_resid_gpu - rel_resid_model|            1.0e-14   -> 1e-12
#     ||y_gpu - y_model|| / ||y_model||             7.7e-11   -> 1e-9
#   The y difference is above float64 round-off because the preconditioner rounds its input to float32: inputs that
#   differ in their last float64 bits now and then round to neighbouring float32 values.
#   independent (the float64 AMG model, whose preconditioner output differs by up to 8.1e-7):
#     |rel_resid_gpu - rel_resid_model| (absolute)  3.3e-10   -> 1e-8
#     ||y_gpu - y_model|| / ||y_model||, compared while rel_resid >= INDEP_Y_ABOVE   1.8e-7 -> 5e-6
#   the library's estimate against the true residual of its own iterate, |rel_resid - ||b - J y|| / ||b||| (no model):
#                                                   1.2e-16   -> 1e-14
BLACKBOX_RESID_TOL = 1e-12
BLACKBOX_Y_TOL = 1e-9
INDEP_RESID_TOL = 1e-8
INDEP_Y_TOL = 5e-6
INDEP_Y_ABOVE = 1e-3
ESTIMATE_TOL = 1e-14

REASONS = ("converged", "max_it", "nonfinite", "breakdown")


@dataclass
class Result:
    y: np.ndarray
    its: int
    rel_resid: float
    reason: str
    history: list = field(default_factory=list)      # the estimate res after iteration 1, 2, ..., its
    cycle_ends: list = field(default_factory=list)   # iteration counts after which a restart took place
    snapshots: dict = field(default_factory=dict)    # k -> y of the same solve stopped by max_it = k


class Fgmres:
    """The loop of hemo_fgmres.  The kernels' individual steps are methods, so a test can override one of them to
    model a defective kernel."""

    def __init__(self, matvec, precond, owned=None):
        self.matvec, self.precond = matvec, precond
        self.owned = None if owned is None else np.asarray(owned, dtype=bool)

    def own(self, a):
        """a with the entries that are not owned set to zero (sums over it run over the owned entries)."""
        return a if self.owned is None else np.where(self.owned, a, 0.0)

    def norm(self, a):
        a = self.own(a)
        return float(np.sqrt(a @ a))

    # k_fg_residual
    def restart_residual(self, b, Ay):
        return b - Ay

    # k_fg_begin_cycle (first = 0): the restart keeps the tolerance of the first cycle
    def restart_tol(self, tol, beta, rtol, atol):
        return tol

    # k_fg_mdot + k_fg_mdot_final: h_i = <v_i, w>, i <= j, all from the same w (V: the rows v_0 .. v_j)
    def gram_schmidt(self, V, w):
        return V @ self.own(w)

    # fg_givens: the residual estimate after the new rotation (c, s)
    def estimate(self, c, s, gj):
        return abs(s * gj)

    # k_fg_backsolve: coefficients of Z_k from the rotated k x k triangle
    def backsolve(self, R, g, k):
        c = np.zeros(k)
        for i in range(k - 1, -1, -1):
            c[i] = (g[i] - R[i, i + 1:k] @ c[i + 1:k]) / R[i, i]
        return c

    def solve(self, b, *, restart, max_it, rtol, atol, snapshots=()):
        b = np.asarray(b, dtype=np.float64)
        want = set(snapshots)
        y = np.zeros_like(b)
        beta = self.norm(b)
        bnorm = beta
        tol = max(rtol * beta, atol)
        out = Result(y=y, its=0, rel_resid=0.0, reason="")

        def finish(res, reason):
            out.y, out.reason = y, reason
            out.rel_resid = res / bnorm if bnorm > 0.0 else 0.0
            for k in want:
                out.snapshots.setdefault(k, y.copy())
            return out

        if beta == 0.0 or beta <= atol:
            return finish(beta, "converged")
        if not np.isfinite(beta):
            return finish(beta, "nonfinite")
        r = b
        res = beta
        while True:
            m = restart
            V = np.zeros((m + 1, b.size))
            Z = np.zeros((m, b.size))
            V[0] = r * (1.0 / beta)
            k = 0
            R = np.zeros((m + 1, m))
            g = np.zeros(m + 1)
            g[0] = beta
            cs, sn = np.zeros(m), np.zeros(m)
            reason = None
            for j in range(m):
                if out.its >= max_it:
                    break
                Z[j] = self.precond(V[j])
                w = np.asarray(self.matvec(Z[j]), dtype=np.float64)
                h = self.gram_schmidt(V[:j + 1], w)
                w = w - V[:j + 1].T @ h
                hn = self.norm(w)
                col = np.append(h, hn)
                for i in range(j):
                    a, bb = col[i], col[i + 1]
                    col[i], col[i + 1] = cs[i] * a + sn[i] * bb, -sn[i] * a + cs[i] * bb
                a, bb = col[j], col[j + 1]
                d = float(np.hypot(a, bb))
                c, s = (a / d, bb / d) if d > 0.0 else (1.0, 0.0)
                cs[j], sn[j] = c, s
                col[j], col[j + 1] = d, 0.0
                R[:j + 2, j] = col
                gj = g[j]
                g[j + 1], g[j] = -s * gj, c * gj
                res = self.estimate(c, s, gj)
                out.its += 1
                out.history.append(res)
                k = j + 1
                if out.its in want:
                    want.discard(out.its)
                    out.snapshots[out.its] = y + Z[:k].T @ self.backsolve(R, g, k)
                if not (np.isfinite(res) and np.isfinite(d)):
                    reason = "nonfinite"
                elif res <= tol:
                    reason = "converged"
                elif hn == 0.0:
                    reason = "breakdown"      # unreachable: hn = 0 gives s = 0, so res = 0 <= tol is tested first
                if reason:
                    break
                V[j + 1] = w * (1.0 / hn)
            if k:
                y = y + Z[:k].T @ self.backsolve(R, g, k)
            if reason:
                return finish(res, reason)
            if out.its >= max_it:
                return finish(res, "max_it")
            r = self.restart_residual(b, self.matvec(y))
            beta = self.norm(r)
            res = beta
            tol = self.restart_tol(tol, beta, rtol, atol)
            out.cycle_ends.append(out.its)
            if beta <= tol:
                return finish(res, "converged")
            if not np.isfinite(beta):
                return finish(res, "nonfinite")


def fgmres(matvec, precond, b, *, restart, max_it, rtol, atol, owned=None, snapshots=()) -> Result:
    """hemo_fgmres from y = 0.  `snapshots`: iteration counts k whose iterate (the y a solve with max_it = k
    returns) is kept in Result.snapshots."""
    return Fgmres(matvec, precond, owned).solve(b, restart=restart, max_it=max_it, rtol=rtol, atol=atol,
                                                snapshots=snapshots)
