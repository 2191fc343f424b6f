"""ctypes binding of libhemo_sm100.so (the C-ABI declared in include/hemo.h).

PyTorch is used only for device buffers: every array argument is a torch
tensor whose `data_ptr()` is handed to the library.  There is no CPU
fallback: if the shared library is missing, or no CUDA device is present when
a context is created, this module raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhemo_sm100.so")

HEMO_DIVERGED = -100
Q_FU, Q_FP, Q_UU, Q_UP, Q_PU, Q_PP = range(6)
CELL_TRIANGLE, CELL_QUADRILATERAL, CELL_TETRAHEDRON, CELL_TRIANGLE_P2 = 0, 1, 2, 3
# hemo_amg_level_info: what runs an AMG level
AMG_SCOPE_NAMES = ("level", "cta")


class HemoError(RuntimeError):
    pass


class HemoDiverged(HemoError):
    pass


class Params(C.Structure):
    _fields_ = [("dt", C.c_double), ("rho", C.c_double), ("mu", C.c_double),
                ("f", C.c_double * 2), ("eps0", C.c_double)]


class FacetCoef(C.Structure):
    _fields_ = [(k, C.c_double) for k in
                ("a_p", "pconst", "a_g", "a_s", "a_n", "beta_n", "a_b", "beta_b")]


class SolverOpts(C.Structure):
    _fields_ = [("restart", C.c_int), ("max_it", C.c_int), ("rtol", C.c_double),
                ("atol", C.c_double), ("amg_cycles_u", C.c_int), ("amg_cycles_p", C.c_int),
                ("cheb_degree", C.c_int), ("project_pressure", C.c_int), ("pc_mode", C.c_int),
                ("schur_mass_coef", C.c_double), ("schur_lap_coef", C.c_double),
                ("cheb_ratio", C.c_double), ("cheb_degree_pre", C.c_int)]


# name -> (restype, argtypes); every symbol include/hemo.h declares
_VP, _I, _L, _D = C.c_void_p, C.c_int, C.c_int64, C.c_double
SYMBOLS = {
    "hemo_ctx_create": (_I, [_I, C.POINTER(_VP)]),
    "hemo_ctx_destroy": (_I, [_VP]),
    "hemo_last_error": (C.c_char_p, [_VP]),
    "hemo_set_stream": (_I, [_VP, _VP]),
    "hemo_launch_count": (_L, [_VP]),
    "hemo_prof_enable": (_I, [_VP, _I]),
    "hemo_prof_get": (_I, [_VP, _I, C.POINTER(_D), C.POINTER(_L)]),
    "hemo_set_cell_type": (_I, [_VP, _I]),
    "hemo_set_formulation": (_I, [_VP, _I]),
    "hemo_set_mesh": (_I, [_VP, _VP, _I, _VP, _I, _VP]),
    "hemo_set_node_graph": (_I, [_VP, _VP, _VP, _L]),
    "hemo_matrix_nnz": (_I, [_VP, C.POINTER(_L)]),
    "hemo_get_pattern": (_I, [_VP, _VP, _VP]),
    "hemo_set_quadrature": (_I, [_VP, _I, _VP, _VP, _I]),
    "hemo_set_facet_quadrature": (_I, [_VP, _VP, _VP, _I]),
    "hemo_set_params": (_I, [_VP, C.POINTER(Params)]),
    "hemo_set_time_scheme": (_I, [_VP, _D, _D, _VP]),
    "hemo_set_facet_set": (_I, [_VP, _I, _VP, _VP, _I, C.POINTER(FacetCoef)]),
    "hemo_set_facet_coef": (_I, [_VP, _I, C.POINTER(FacetCoef)]),
    "hemo_set_bc": (_I, [_VP, _VP, _VP, _VP]),
    "hemo_assemble_jacobian": (_I, [_VP, _VP, _VP, _VP]),
    "hemo_assemble_residual": (_I, [_VP, _VP, _VP, _VP, _VP]),
    "hemo_outlet_flux": (_I, [_VP, _I, _VP, C.POINTER(_D)]),
    "hemo_assemble_laplace_mass": (_I, [_VP, _VP, _VP]),
    "hemo_set_body_force3": (_I, [_VP, _VP]),
    "hemo_tet_set_quadrature": (_I, [_VP, _I, _VP, _VP, _I]),
    "hemo_tet_element_tensors": (_I, [_VP, _I, _I] + [_VP] * 9),
    "hemo_wall_shear_stress": (_I, [_VP, _I, _VP, _VP]),
    "hemo_boundary_force": (_I, [_VP, _I, _VP, C.POINTER(_D)]),
    "hemo_early_stop_norms": (_I, [_VP, _L, _VP, _VP, C.POINTER(_D)]),
    "hemo_l2_norm_sq": (_I, [_VP, _I, _VP, C.POINTER(_D)]),
    "hemo_spmv": (_I, [_VP, _VP, _VP, _VP]),
    "hemo_axpy": (_I, [_VP, _L, _D, _VP, _VP]),
    "hemo_dot": (_I, [_VP, _L, _VP, _VP, C.POINTER(_D)]),
    "hemo_norm2": (_I, [_VP, _L, _VP, C.POINTER(_D)]),
    "hemo_remove_mean_vec": (_I, [_VP, _L, _VP]),
    "hemo_amg_set_level": (_I, [_VP, _I, _I, _I, _I] + [_VP] * 10),
    "hemo_amg_finalize": (_I, [_VP, _I, _I]),
    "hemo_host_aggregate": (_I, [_I, _VP, _VP, _VP, _VP, C.POINTER(_I)]),
    "hemo_set_solver_opts": (_I, [_VP, C.POINTER(SolverOpts)]),
    "hemo_set_pc_mask": (_I, [_VP, _VP]),
    "hemo_set_external_schur": (_I, [_VP, _I]),
    "hemo_amg_setup_scalar": (_I, [_VP, _VP, _D]),
    "hemo_mask_nodes": (_I, [_VP, _VP, _VP]),
    "hemo_vec_mdot": (_I, [_VP, _L, _I, _VP, _L, _VP, _VP]),
    "hemo_vec_maxpy": (_I, [_VP, _L, _I, _VP, _L, _VP, _D, _VP, C.POINTER(_D)]),
    "hemo_vec_scale": (_I, [_VP, _L, _D, _VP, _VP]),
    "hemo_use_graph": (_I, [_VP, _I]),
    "hemo_amg_set_fine_pattern": (_I, [_VP, _I, _VP, _VP]),
    "hemo_pc_set_schur_selfp": (_I, [_VP, _VP, _D]),
    "hemo_pc_setup": (_I, [_VP, _VP, _VP, _VP]),
    "hemo_amg_apply": (_I, [_VP, _I, _VP, _VP, _I]),
    "hemo_amg_get_level_values": (_I, [_VP, _I, _I, _VP, _L]),
    "hemo_amg_level_info": (_I, [_VP, _I, _I, C.POINTER(_L)]),
    "hemo_pc_apply": (_I, [_VP, _VP, _VP, _VP]),
    "hemo_fgmres": (_I, [_VP, _VP, _VP, _VP, C.POINTER(_I), C.POINTER(_D)]),
    "hemo_comm_unique_id": (_I, [C.c_char_p]),
    "hemo_comm_init": (_I, [_VP, C.c_char_p, _I, _I]),
    "hemo_comm_info": (_I, [_VP, C.POINTER(_I), C.POINTER(_I), C.POINTER(_I), C.POINTER(_L), C.POINTER(_L)]),
    "hemo_comm_set_partition": (_I, [_VP, _I, _I, _VP, _VP, _VP, _VP, _I]),
    "hemo_set_graph": (_I, [_VP, _I, _VP, _VP, _L]),
    "hemo_pc_set_coarse_pressure": (_I, [_VP, _VP, _I] + [_VP] * 6 + [_I]),
    "hemo_comm_halo_update": (_I, [_VP, _VP]),
    "hemo_comm_allreduce": (_I, [_VP, _VP, _I]),
    "hemo_global_dot": (_I, [_VP, _VP, _VP, C.POINTER(_D)]),
    "hemo_set_poll_interval": (_I, [_VP, _I]),
    "hemo_krylov_graph_info": (_I, [_VP, C.POINTER(_L), C.POINTER(_L)]),
}

_lib = None


def load_library(path: str | None = None):
    """dlopen the in-tree shared library and bind every declared symbol."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise HemoError(
            f"{p} not found: build it with `python -m cfd_hemodynamic_b200.build` "
            "(nvcc, sm_100a).  There is no CPU fallback.")
    lib = C.CDLL(p)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if a symbol is missing
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


def _ptr(t):
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def _np_ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


class Hemo:
    """One library context bound to one CUDA device."""

    def __init__(self, device: int = 0):
        import torch
        if not torch.cuda.is_available():
            raise HemoError("no CUDA device: the hot path only exists as sm_100a kernels")
        self.lib = load_library()
        self.torch = torch
        self.device = torch.device("cuda", device)
        self._ctx = C.c_void_p()
        rc = self.lib.hemo_ctx_create(device, C.byref(self._ctx))
        if rc != 0:
            raise HemoError(f"hemo_ctx_create failed ({rc})")
        # all work (library kernels and torch copies) runs on one non-default stream, which
        # the preconditioner's CUDA-graph capture requires; it becomes torch's current stream
        if torch.cuda.current_stream(self.device).cuda_stream == 0:
            self.stream = torch.cuda.Stream(self.device)
            torch.cuda.set_stream(self.stream)
        else:
            self.stream = torch.cuda.current_stream(self.device)
        self.lib.hemo_set_stream(self._ctx, C.c_void_p(self.stream.cuda_stream))
        self._keep = {}     # borrowed tensors must outlive the context
        if os.environ.get("HEMO_NO_GRAPH"):
            self.lib.hemo_use_graph(self._ctx, 0)

    def close(self):
        if self._ctx:
            self.torch.cuda.synchronize(self.device)
            self.lib.hemo_ctx_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int, what: str):
        if rc == 0:
            return
        msg = self.lib.hemo_last_error(self._ctx)
        msg = msg.decode() if msg else ""
        if rc == HEMO_DIVERGED:
            raise HemoDiverged(f"{what}: {msg}")
        raise HemoError(f"{what} failed (code {rc}): {msg}")

    @property
    def launches(self) -> int:
        return int(self.lib.hemo_launch_count(self._ctx))

    def prof_enable(self, on: bool):
        self._check(self.lib.hemo_prof_enable(self._ctx, int(on)), "hemo_prof_enable")

    def prof_get(self, cls: int):
        ms = C.c_double()
        cnt = C.c_int64()
        self._check(self.lib.hemo_prof_get(self._ctx, cls, C.byref(ms), C.byref(cnt)), "hemo_prof_get")
        return ms.value, cnt.value

    # ---- setup ---------------------------------------------------------
    def set_mesh(self, x2, cells, h):
        """cells: (E, 3) P1 triangles or (E, 4) tensor-ordered Q1 quadrilaterals with x2 (n, 2);
        (E, 4) P1 tetrahedra with x2 (n, 3) (what works on tetrahedra: include/hemo.h)."""
        if cells.dim() != 2 or cells.shape[1] not in (3, 4, 6) or not cells.is_contiguous():
            raise HemoError("cells must be a contiguous (E, 3), (E, 4) or (E, 6: P2 triangles) int32 tensor")
        self.nv = int(cells.shape[1])
        self.dim = int(x2.shape[1]) if x2.dim() == 2 else 2
        if self.dim == 3 and self.nv != 4:
            raise HemoError("3-D meshes must be tetrahedral: cells (E, 4)")
        ctype = CELL_TETRAHEDRON if self.dim == 3 else {3: CELL_TRIANGLE, 4: CELL_QUADRILATERAL, 6: CELL_TRIANGLE_P2}[self.nv]
        self._check(self.lib.hemo_set_cell_type(self._ctx, ctype), "hemo_set_cell_type")
        self._keep.update(x=x2, cells=cells, h=h)
        self.n = x2.shape[0]
        self.E = cells.shape[0]
        self._check(self.lib.hemo_set_mesh(self._ctx, _ptr(x2), self.n, _ptr(cells), self.E, _ptr(h)),
                    "hemo_set_mesh")

    def set_formulation(self, name: str):
        """"standard" (stabilized_schur.py:69-121) or "curlcurl" (stabilized_schur_pressurebc.py:85-160)."""
        code = {"standard": 0, "curlcurl": 1}[name]
        self._check(self.lib.hemo_set_formulation(self._ctx, code), "hemo_set_formulation")

    def set_node_graph(self, nrowptr, ncol):
        self._keep.update(nrowptr=nrowptr, ncol=ncol)
        self.nnz_node = int(ncol.shape[0])
        self._check(self.lib.hemo_set_node_graph(self._ctx, _ptr(nrowptr), _ptr(ncol), self.nnz_node),
                    "hemo_set_node_graph")
        self.nnz = (getattr(self, "dim", 2) + 1) ** 2 * self.nnz_node

    def get_pattern(self):
        t = self.torch
        rowptr = t.empty((getattr(self, "dim", 2) + 1) * self.n + 1, dtype=t.int64, device=self.device)
        col = t.empty(self.nnz, dtype=t.int32, device=self.device)
        self._check(self.lib.hemo_get_pattern(self._ctx, _ptr(rowptr), _ptr(col)), "hemo_get_pattern")
        return rowptr, col

    def set_quadrature(self, block: int, pts: np.ndarray, wts: np.ndarray):
        pts = np.ascontiguousarray(pts, dtype=np.float64)
        wts = np.ascontiguousarray(wts, dtype=np.float64)
        self._check(self.lib.hemo_set_quadrature(self._ctx, block, _np_ptr(pts), _np_ptr(wts), len(wts)),
                    "hemo_set_quadrature")

    def set_time_scheme(self, theta: float, a0: float, uh=None):
        """theta = d(u_e)/du, a0 = leading BDF coefficient, uh = history vector (2n, device) or None."""
        self._keep["uh"] = uh
        self._check(self.lib.hemo_set_time_scheme(self._ctx, float(theta), float(a0), _ptr(uh)),
                    "hemo_set_time_scheme")

    def set_body_force3(self, f3):
        f3 = np.ascontiguousarray(f3, dtype=np.float64)
        self._check(self.lib.hemo_set_body_force3(self._ctx, _np_ptr(f3)), "hemo_set_body_force3")

    def set_facet_quadrature(self, pts, wts):
        pts = np.ascontiguousarray(pts, dtype=np.float64)
        wts = np.ascontiguousarray(wts, dtype=np.float64)
        self._check(self.lib.hemo_set_facet_quadrature(self._ctx, _np_ptr(pts), _np_ptr(wts), len(wts)),
                    "hemo_set_facet_quadrature")

    def set_params(self, dt, rho, mu, f, eps0):
        p = Params(dt=dt, rho=rho, mu=mu, eps0=eps0)
        p.f[0], p.f[1] = float(f[0]), float(f[1])
        self._check(self.lib.hemo_set_params(self._ctx, C.byref(p)), "hemo_set_params")

    def set_facet_set(self, set_id: int, cells, mask, **coef):
        c = FacetCoef(**coef)
        m = 0 if cells is None else int(cells.shape[0])
        self._check(self.lib.hemo_set_facet_set(self._ctx, set_id, _ptr(cells), _ptr(mask), m, C.byref(c)),
                    "hemo_set_facet_set")

    def set_facet_coef(self, set_id: int, **coef):
        c = FacetCoef(**coef)
        self._check(self.lib.hemo_set_facet_coef(self._ctx, set_id, C.byref(c)), "hemo_set_facet_coef")

    def set_bc(self, dofflag, dofmult, cellflag):
        self._check(self.lib.hemo_set_bc(self._ctx, _ptr(dofflag), _ptr(dofmult), _ptr(cellflag)), "hemo_set_bc")

    # ---- assembly ------------------------------------------------------
    def assemble_jacobian(self, x, un, vals):
        self._check(self.lib.hemo_assemble_jacobian(self._ctx, _ptr(x), _ptr(un), _ptr(vals)),
                    "hemo_assemble_jacobian")

    def assemble_residual(self, x, un, g, b):
        self._check(self.lib.hemo_assemble_residual(self._ctx, _ptr(x), _ptr(un), _ptr(g), _ptr(b)),
                    "hemo_assemble_residual")

    def outlet_flux(self, set_id, un) -> float:
        q = C.c_double()
        self._check(self.lib.hemo_outlet_flux(self._ctx, set_id, _ptr(un), C.byref(q)), "hemo_outlet_flux")
        return q.value

    def assemble_laplace_mass(self):
        t = self.torch
        lap = t.empty(self.nnz_node, dtype=t.float64, device=self.device)
        mass = t.empty(self.n, dtype=t.float64, device=self.device)
        self._check(self.lib.hemo_assemble_laplace_mass(self._ctx, _ptr(lap), _ptr(mass)),
                    "hemo_assemble_laplace_mass")
        return lap, mass

    # ---- tetrahedra (element tensors only) ------------------------------------
    def tet_set_quadrature(self, block: int, pts: np.ndarray, wts: np.ndarray):
        pts = np.ascontiguousarray(pts, dtype=np.float64)
        wts = np.ascontiguousarray(wts, dtype=np.float64)
        self._check(self.lib.hemo_tet_set_quadrature(self._ctx, block, _np_ptr(pts), _np_ptr(wts), len(wts)),
                    "hemo_tet_set_quadrature")

    def tet_element_tensors(self, x3, cells, h, sol, un, uh, f3):
        """Ae (256, E), Fe (16, E) of P1 tetrahedra; see include/hemo.h."""
        t = self.torch
        E, n = int(cells.shape[0]), int(x3.shape[0])
        Ae = t.empty((256, E), dtype=t.float64, device=self.device)
        Fe = t.empty((16, E), dtype=t.float64, device=self.device)
        f3 = np.ascontiguousarray(f3, dtype=np.float64)
        self._check(self.lib.hemo_tet_element_tensors(self._ctx, n, E, _ptr(x3), _ptr(cells), _ptr(h), _ptr(sol), _ptr(un),
                                                      _ptr(uh), _np_ptr(f3), _ptr(Ae), _ptr(Fe)),
                    "hemo_tet_element_tensors")
        return Ae, Fe

    # ---- post-processing ---------------------------------------------------
    def wall_shear_stress(self, set_id: int, x, out):
        self._check(self.lib.hemo_wall_shear_stress(self._ctx, set_id, _ptr(x), _ptr(out)), "hemo_wall_shear_stress")

    def boundary_force(self, set_id: int, x):
        f = (C.c_double * 2)()
        self._check(self.lib.hemo_boundary_force(self._ctx, set_id, _ptr(x), f), "hemo_boundary_force")
        return f[0], f[1]

    def early_stop_norms(self, u, un):
        f = (C.c_double * 2)()
        self._check(self.lib.hemo_early_stop_norms(self._ctx, u.numel(), _ptr(u), _ptr(un), f), "hemo_early_stop_norms")
        return f[0], f[1]

    def l2_norm_sq(self, f, bs: int) -> float:
        out = C.c_double()
        self._check(self.lib.hemo_l2_norm_sq(self._ctx, bs, _ptr(f), C.byref(out)), "hemo_l2_norm_sq")
        return out.value

    # ---- linear algebra --------------------------------------------------
    def spmv(self, vals, x, y):
        self._check(self.lib.hemo_spmv(self._ctx, _ptr(vals), _ptr(x), _ptr(y)), "hemo_spmv")

    def axpy(self, a, x, y):
        self._check(self.lib.hemo_axpy(self._ctx, x.numel(), float(a), _ptr(x), _ptr(y)), "hemo_axpy")

    def dot(self, x, y) -> float:
        out = C.c_double()
        self._check(self.lib.hemo_dot(self._ctx, x.numel(), _ptr(x), _ptr(y), C.byref(out)), "hemo_dot")
        return out.value

    def norm2(self, x) -> float:
        out = C.c_double()
        self._check(self.lib.hemo_norm2(self._ctx, x.numel(), _ptr(x), C.byref(out)), "hemo_norm2")
        return out.value

    def remove_mean(self, x):
        self._check(self.lib.hemo_remove_mean_vec(self._ctx, x.numel(), _ptr(x)), "hemo_remove_mean_vec")

    # ---- AMG / solve -------------------------------------------------------
    def amg_set_level(self, which, level, P, R, AP_pattern, C_pattern):
        """P, R: scipy CSR (float64); AP_pattern, C_pattern: scipy CSR patterns."""
        def i32(a):
            return np.ascontiguousarray(a, dtype=np.int32)
        p_rp, p_c, p_v = i32(P.indptr), i32(P.indices), np.ascontiguousarray(P.data, dtype=np.float64)
        r_rp, r_c, r_v = i32(R.indptr), i32(R.indices), np.ascontiguousarray(R.data, dtype=np.float64)
        ap_rp, ap_c = i32(AP_pattern.indptr), i32(AP_pattern.indices)
        c_rp, c_c = i32(C_pattern.indptr), i32(C_pattern.indices)
        self._check(self.lib.hemo_amg_set_level(
            self._ctx, which, level, P.shape[0], P.shape[1],
            _np_ptr(p_rp), _np_ptr(p_c), _np_ptr(p_v), _np_ptr(r_rp), _np_ptr(r_c), _np_ptr(r_v),
            _np_ptr(ap_rp), _np_ptr(ap_c), _np_ptr(c_rp), _np_ptr(c_c)), "hemo_amg_set_level")

    def amg_finalize(self, which, n_levels):
        self._check(self.lib.hemo_amg_finalize(self._ctx, which, n_levels), "hemo_amg_finalize")

    def set_solver_opts(self, **kw):
        o = SolverOpts(**kw)
        self._check(self.lib.hemo_set_solver_opts(self._ctx, C.byref(o)), "hemo_set_solver_opts")

    # ---- multi-GPU building blocks ---------------------------------------------
    def set_pc_mask(self, node_mask):
        self._check(self.lib.hemo_set_pc_mask(self._ctx, _ptr(node_mask)), "hemo_set_pc_mask")

    def set_external_schur(self, on: bool):
        self._check(self.lib.hemo_set_external_schur(self._ctx, int(on)), "hemo_set_external_schur")

    def amg_setup_scalar(self, lap, coarse_shift=0.0):
        self._check(self.lib.hemo_amg_setup_scalar(self._ctx, _ptr(lap), float(coarse_shift)), "hemo_amg_setup_scalar")

    def mask_nodes(self, node_mask, x):
        self._check(self.lib.hemo_mask_nodes(self._ctx, _ptr(node_mask), _ptr(x)), "hemo_mask_nodes")

    def vec_mdot(self, V, ldv, k, w) -> np.ndarray:
        h = np.empty(k, dtype=np.float64)
        self._check(self.lib.hemo_vec_mdot(self._ctx, w.numel(), k, _ptr(V), ldv, _ptr(w), _np_ptr(h)), "hemo_vec_mdot")
        return h

    def vec_maxpy(self, V, ldv, coef: np.ndarray, sign, w, want_normsq=False):
        coef = np.ascontiguousarray(coef, dtype=np.float64)
        out = C.c_double()
        self._check(self.lib.hemo_vec_maxpy(self._ctx, w.numel(), len(coef), _ptr(V), ldv, _np_ptr(coef), float(sign),
                                            _ptr(w), C.byref(out) if want_normsq else None), "hemo_vec_maxpy")
        return out.value if want_normsq else None

    def vec_scale(self, a, x, y):
        self._check(self.lib.hemo_vec_scale(self._ctx, x.numel(), float(a), _ptr(x), _ptr(y)), "hemo_vec_scale")

    def use_graph(self, on: bool):
        self._check(self.lib.hemo_use_graph(self._ctx, int(on)), "hemo_use_graph")

    def amg_set_fine_pattern(self, which, pattern):
        """pattern: scipy CSR (values ignored) or None to fall back to the node graph."""
        if pattern is None:
            self._check(self.lib.hemo_amg_set_fine_pattern(self._ctx, which, None, None), "hemo_amg_set_fine_pattern")
            return
        rp = np.ascontiguousarray(pattern.indptr, dtype=np.int32)
        ci = np.ascontiguousarray(pattern.indices, dtype=np.int32)
        self._check(self.lib.hemo_amg_set_fine_pattern(self._ctx, which, _np_ptr(rp), _np_ptr(ci)),
                    "hemo_amg_set_fine_pattern")

    def pc_set_schur_selfp(self, vals, coarse_shift=0.0):
        self._check(self.lib.hemo_pc_set_schur_selfp(self._ctx, _ptr(vals), float(coarse_shift)), "hemo_pc_set_schur_selfp")

    def pc_setup(self, vals, lap=None, mass=None):
        if lap is not None:
            self._keep.update(mass=mass)
        self._check(self.lib.hemo_pc_setup(self._ctx, _ptr(vals), _ptr(lap), _ptr(mass)), "hemo_pc_setup")

    def amg_apply(self, which, b, x, ncycles=1):
        self._check(self.lib.hemo_amg_apply(self._ctx, which, _ptr(b), _ptr(x), ncycles), "hemo_amg_apply")

    def amg_level_values(self, which, level, count):
        t = self.torch
        out = t.empty(count, dtype=t.float64, device=self.device)
        self._check(self.lib.hemo_amg_get_level_values(self._ctx, which, level, _ptr(out), count),
                    "hemo_amg_get_level_values")
        return out

    def amg_level_info(self, which, level):
        """dict(n, nnzb, sell, scope) of level `level` of hierarchy `which`: sell = entries of the sliced-ELL copy
        (0: CSR kernels); scope = "level" (per-level kernels) or "cta" (the one-CTA fused coarse V-cycle kernel)."""
        out = (C.c_int64 * 4)()
        self._check(self.lib.hemo_amg_level_info(self._ctx, which, level, out), "hemo_amg_level_info")
        return dict(n=out[0], nnzb=out[1], sell=out[2], scope=AMG_SCOPE_NAMES[out[3]])

    def pc_apply(self, vals, r, z):
        self._check(self.lib.hemo_pc_apply(self._ctx, _ptr(vals), _ptr(r), _ptr(z)), "hemo_pc_apply")

    def krylov_graph_info(self):
        """(kernel nodes, programmatic-dependent-launch edges) of the last captured FGMRES iteration graph."""
        nodes, edges = C.c_int64(), C.c_int64()
        self._check(self.lib.hemo_krylov_graph_info(self._ctx, C.byref(nodes), C.byref(edges)), "hemo_krylov_graph_info")
        return nodes.value, edges.value

    # ---- multi-GPU: NCCL inside the library ---------------------------------------
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        rc = load_library().hemo_comm_unique_id(buf)
        if rc:
            raise HemoError("hemo_comm_unique_id failed (NCCL not loadable)")
        return buf.raw

    def comm_init(self, uid: bytes, rank: int, nranks: int):
        self._check(self.lib.hemo_comm_init(self._ctx, C.c_char_p(uid), int(rank), int(nranks)), "hemo_comm_init")

    def comm_info(self):
        r, n, v = C.c_int(), C.c_int(), C.c_int()
        h, a = C.c_int64(), C.c_int64()
        self._check(self.lib.hemo_comm_info(self._ctx, C.byref(r), C.byref(n), C.byref(v), C.byref(h), C.byref(a)),
                    "hemo_comm_info")
        return dict(rank=r.value, nranks=n.value, nccl_version=v.value, halo_updates=h.value, allreduces=a.value)

    def comm_set_partition(self, n_owned, peers, send_ptr, send_nodes, recv_ptr, ras_overlap=False):
        peers = np.ascontiguousarray(peers, dtype=np.int32)
        send_ptr = np.ascontiguousarray(send_ptr, dtype=np.int32)
        send_nodes = np.ascontiguousarray(send_nodes, dtype=np.int32)
        recv_ptr = np.ascontiguousarray(recv_ptr, dtype=np.int32)
        hp = lambda a: a.ctypes.data_as(C.c_void_p)
        self._check(self.lib.hemo_comm_set_partition(self._ctx, int(n_owned), int(peers.shape[0]), hp(peers), hp(send_ptr),
                                                     hp(send_nodes), hp(recv_ptr), int(bool(ras_overlap))),
                    "hemo_comm_set_partition")

    def set_graph(self, rowptr, col):
        """Mesh-less context carrying a scalar operator on the graph (rowptr, col) (device int32 tensors, kept alive)."""
        self._keep["graph"] = (rowptr, col)
        self.n = int(rowptr.numel() - 1)
        self.nnz_node = int(col.numel())
        self._check(self.lib.hemo_set_graph(self._ctx, self.n, _ptr(rowptr), _ptr(col), self.nnz_node), "hemo_set_graph")

    def pc_set_coarse_pressure(self, coarse, P0, R0, cycles=1):
        """coarse: Hemo context with the replicated coarse hierarchy (None removes); P0 / R0: scipy CSR."""
        if coarse is None:
            self._check(self.lib.hemo_pc_set_coarse_pressure(self._ctx, None, 0, *([None] * 6), 1), "hemo_pc_set_coarse_pressure")
            return
        arrs = []
        for A in (P0, R0):
            arrs += [np.ascontiguousarray(A.indptr, dtype=np.int32), np.ascontiguousarray(A.indices, dtype=np.int32),
                     np.ascontiguousarray(A.data, dtype=np.float64)]
        hp = lambda a: a.ctypes.data_as(C.c_void_p)
        self._coarse = coarse
        self._check(self.lib.hemo_pc_set_coarse_pressure(self._ctx, coarse._ctx, int(P0.shape[1]), *[hp(a) for a in arrs],
                                                         int(cycles)), "hemo_pc_set_coarse_pressure")

    def halo_update(self, v):
        self._check(self.lib.hemo_comm_halo_update(self._ctx, _ptr(v)), "hemo_comm_halo_update")

    def allreduce(self, buf):
        self._check(self.lib.hemo_comm_allreduce(self._ctx, _ptr(buf), buf.numel()), "hemo_comm_allreduce")

    def global_dot(self, x, y) -> float:
        out = C.c_double()
        self._check(self.lib.hemo_global_dot(self._ctx, _ptr(x), _ptr(y), C.byref(out)), "hemo_global_dot")
        return out.value

    def set_poll_interval(self, every: int):
        self._check(self.lib.hemo_set_poll_interval(self._ctx, int(every)), "hemo_set_poll_interval")

    def fgmres(self, vals, b, y):
        its = C.c_int()
        res = C.c_double()
        rc = self.lib.hemo_fgmres(self._ctx, _ptr(vals), _ptr(b), _ptr(y), C.byref(its), C.byref(res))
        self._check(rc, "hemo_fgmres")
        return its.value, res.value
