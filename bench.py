#!/usr/bin/env python
"""Benchmark of the stabilized_schur per-timestep hot path (BASELINE.json metric:
DOF-timesteps/s; assembly cells/s and nnz/s are reported beside it).

  python bench.py --gpus N --steps K --warmup W            # this repo (CUDA, sm_100a)
  python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the reference's solver configuration
                                                           # restated in C + OpenMP on all host cores
                                                           # (DOLFINx/PETSc cannot be installed)
  python bench.py --gpus 1 ... --dump-outputs DIR          # also writes the solution of the last timed step
                                                           # as DIR/velocity.npy and DIR/pressure.npy

A "step" is one time step (`Solver.solveStep`) of the workload: Newton with Jacobian + residual assemblies and a
preconditioned FGMRES solve per iteration.  `value` is measured with everything resident in HBM
(`Solver.step_device`), `e2e` through the reference-facing plugin API with host buffers (`Solver.solveStep` + the
host-side u_prev <- u_sol shift the reference's time loop performs, src/scenario.py:306-307).

Both arms run the SAME mesh, parameters and time steps (W warm-up steps, then K timed ones): the default workload
is BASELINE config 2 (lid_driven2D, `--solver stabilized_schur`) at the largest size at which the reference's own
algorithm — FGMRES(200) + fieldsplit Schur FULL/SELFP + GMRES(30)/ASM-ILU(0) sub-solves,
src/solvers/stabilized_schur.py:226-275 — finishes W + K steps on the GPU box's host cores within the driver's time
limit (it needs minutes per step at 1 M cells).  The larger configurations (1 M-cell lid cavity, the 16 M-cell
stenosis mesh of the north star) are measured in the same run on the GPU arm and reported under `other_workloads`.
"""
from __future__ import annotations

import argparse
import contextlib
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[1]: lid_driven2D on a refined structured mesh; nx = 707 is the ~1 M-cell size,
    # nx = 512 (0.52 M cells) the largest one the CPU arm finishes W + K = 25 steps of within the driver's time limit:
    # measured on the GPU box's 16 cores 9.7 s per step at nx = 384 and 80 s per step at nx = 707
    "lid_driven2D_nx384": dict(scenario="lid_driven2D", nx=384, mu=0.01, rho=1.0, dt=0.01),
    "lid_driven2D_nx512": dict(scenario="lid_driven2D", nx=512, mu=0.01, rho=1.0, dt=0.01),
    "lid_driven2D_nx707": dict(scenario="lid_driven2D", nx=707, mu=0.01, rho=1.0, dt=0.01),
    "lid_driven2D_nx1414": dict(scenario="lid_driven2D", nx=1414, mu=0.01, rho=1.0, dt=0.01),
    "lid_driven2D_nx2828": dict(scenario="lid_driven2D", nx=2828, mu=0.01, rho=1.0, dt=0.01),
    "lid_driven2D_nx64": dict(scenario="lid_driven2D", nx=64, mu=0.01, rho=1.0, dt=0.01),
    # BASELINE.json configs[2..4] on the mapped split-triangle stenosis channel (SURVEY §7.3-2)
    "stenosis_backflow_1m": dict(scenario="stenosis_mesh_variable", res=0.03, dt=1e-3, v_max=100.0),
    "stenosis_backflow_4m": dict(scenario="stenosis_mesh_variable", res=0.015, dt=1e-3, v_max=100.0),
    "stenosis_pressure_4m": dict(scenario="stenosis_pressure", res=0.015, dt=1e-3, p_inlet=80.0, R_resistance=10.0),
    "stenosis_pressure_structured_250k": dict(scenario="stenosis_pressure_structured", res=0.06, dt=1e-3,
                                              p_inlet=80.0, R_resistance=10.0),
    "stenosis_pressure_structured_1m": dict(scenario="stenosis_pressure_structured", res=0.03, dt=1e-3,
                                            p_inlet=80.0, R_resistance=10.0),
    "stenosis_pressure_structured_16m": dict(scenario="stenosis_pressure_structured", res=0.0075, dt=1e-3,
                                             p_inlet=80.0, R_resistance=10.0),
    # the same transfinite grid with the reference's recombined Q1 cells (SURVEY §8(f) rank 1)
    "stenosis_pressure_structured_q1_1m": dict(scenario="stenosis_pressure_structured", res=0.0212, dt=1e-3,
                                               p_inlet=80.0, R_resistance=10.0, cell_type="quadrilateral"),
    "stenosis_pressure_structured_q1_4m": dict(scenario="stenosis_pressure_structured", res=0.0106, dt=1e-3,
                                               p_inlet=80.0, R_resistance=10.0, cell_type="quadrilateral"),
    "stenosis_pressure_structured_q1_8m": dict(scenario="stenosis_pressure_structured", res=0.0075, dt=1e-3,
                                               p_inlet=80.0, R_resistance=10.0, cell_type="quadrilateral"),
}
DEFAULT_WORKLOAD = "lid_driven2D_nx512"
# measured on the GPU arm in the same run (N = 1, default workload only): (name, warm-up, steps)
EXTRA_WORKLOADS = [("lid_driven2D_nx707", 3, 10), ("stenosis_pressure_structured_16m", 2, 4)]
CPU_BUDGET_S = 1500.0        # the CPU arm stops taking new steps beyond this (driver limit: 1800 s per arm)
CPU_BUDGET_WEAK_S = 420.0    # the same for the weak-scaled meshes of the N > 1 lines (minutes per time step)
DUMP_BYTES = 64_000_000      # --dump-outputs writes at most this many bytes of array data

PROF_CLASSES = {0: "spmv_node(J)", 1: "cell_jacobian", 2: "gather_matrix", 3: "cell_residual",
                4: "cheb_step<2>(A00,l0)", 5: "cheb_step<1>(Lp,l0)", 6: "mdot", 7: "maxpy_norm",
                8: "numeric_rap<2>(l0)"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi sampling during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) < 8:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dump_outputs(dirname, arrays):
    """Write each array as dirname/<name>.npy in float64.  When they hold more than DUMP_BYTES in all, each is cut to
    a fixed, seeded sample of its entries (in index order), the same from run to run for the same workload."""
    os.makedirs(dirname, exist_ok=True)
    total = sum(8 * a.size for a in arrays.values())
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64).reshape(-1)
        if total > DUMP_BYTES:
            keep = np.random.default_rng(0).choice(a.size, a.size * DUMP_BYTES // total, replace=False)
            a = a[np.sort(keep)]
        np.save(os.path.join(dirname, name + ".npy"), a)


def build_scenario(w, **solver_kw):
    if w["scenario"] == "lid_driven2D":
        from cfd_hemodynamic_b200.src.scenarios.lid_driven2D import LidDriven2DSimulation
        return LidDriven2DSimulation("stabilized_schur", w["dt"], 1.0, rho=w["rho"], mu=w["mu"], nx=w["nx"], **solver_kw)
    if w["scenario"] == "stenosis_mesh_variable":
        from cfd_hemodynamic_b200.src.scenarios.stenosis_mesh_variable import StenosisMeshVariableSimulation
        return StenosisMeshVariableSimulation("stabilized_schur_backflow", w["dt"], 1.0, grade="severe",
                                              v_max=w["v_max"], res=w["res"], **solver_kw)
    from cfd_hemodynamic_b200.src.scenarios.stenosis_pressure_structured import StenosisPressureStructuredSimulation
    return StenosisPressureStructuredSimulation("stabilized_schur_pressure_backflow", w["dt"], 1.0, grade="severe",
                                                p_inlet=w["p_inlet"], R_resistance=w["R_resistance"], res=w["res"],
                                                cell_type=w.get("cell_type", "triangle"), **solver_kw)


def workload_config(name, sc):
    """The part of the JSON line both arms must agree on: what was solved."""
    s = sc.solver
    cells = s._cells_host
    n = s.n
    nv = int(cells.shape[1])
    return {"workload": name, "solver": sc.solver_name, "cell_type": s.mesh.topology.cell_name(),
            "cells": int(cells.shape[0]), "dofs": int(3 * n), "dt": float(s.dt.value), "mu": float(s.mu.value),
            "rho": float(s.rho.value),
            "tolerances": {"snes_rtol": s.snes_rtol, "snes_stol": s.snes_stol, "ksp_rtol": s.ksp_rtol},
            "l2": "inputs larger than L2: Jacobian values + element buffer %.0f MB vs 126 MB L2"
                  % ((8 * 9 * 7.0 * n + 72 * nv * nv * cells.shape[0]) / 1e6)}


# ------------------------------------------------------------------------------------------------------
# CPU arm
# ------------------------------------------------------------------------------------------------------
def cpu_sub_pc(name):
    """Sub-solvers of the reference for this workload's solver module: asm/ilu(0) for stabilized_schur
    (stabilized_schur.py:256-267), lu for the pressure variants (stabilized_schur_pressure_backflow.py:284-288)."""
    return "ilu" if WORKLOADS[name]["scenario"] == "lid_driven2D" else "lu"


def cpu_steps(name, n_warm, n_steps, budget_s, nranks=None, nx=None):
    """The reference's solver configuration restated on host cores (oracle/cpu_reference.CReferenceSolver:
    C + OpenMP, one thread per `mpirun` rank) marching the same scenario.  `nx` overrides the cavity resolution (the
    weak-scaled mesh of an N-GPU run).  Returns a dict."""
    from oracle.workload import CpuMarcher
    w = dict(WORKLOADS[name])
    if nx is not None:
        w["nx"] = int(nx)
    with contextlib.redirect_stdout(sys.stderr):
        sc = build_scenario(w, host_only=True)
    cores = int(nranks or os.cpu_count() or 1)
    t_setup = time.perf_counter()
    m = CpuMarcher(sc, solver="reference", nranks=cores, sub_pc=cpu_sub_pc(name))
    t_setup = time.perf_counter() - t_setup
    t_begin = time.perf_counter()
    for _ in range(n_warm):
        m.step()
    done = 0
    t0 = time.perf_counter()
    for _ in range(n_steps):
        m.step()
        done += 1
        if time.perf_counter() - t_begin > budget_s:
            break
    secs = time.perf_counter() - t0
    st = m.ref.stats()
    return dict(config=workload_config(name, sc), ndof=3 * m.n, steps=done, seconds=secs, cores=cores,
                newton_its=m.ref.newton_its, outer_its=st["outer_its"], inner_its=st["inner_its"],
                timers=dict(m.ref.timers), setup_s=t_setup, total_steps=n_warm + done)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = args.workload
    w = WORKLOADS[name]
    if w["scenario"] == "stenosis_mesh_variable" or w.get("cell_type", "triangle") != "triangle":
        raise SystemExit("bench.py --impl reference: the CPU arm is written for P1 triangles and for the lid_driven2D "
                         "(asm/ilu(0) sub-solves, stabilized_schur.py:256-267) and stenosis_pressure_structured (lu sub-solves, "
                         "stabilized_schur_pressure_backflow.py:284-288) workloads")
    W = max(0, args.warmup)
    K = args.steps
    N = max(int(args.gpus), 1)
    nx = None
    budget = CPU_BUDGET_S
    if N > 1:
        # the GPU arm at N > 1 solves ONE lid cavity of nx * sqrt(N) squared (run_distributed, weak scaling): the same mesh
        # here, on the same host cores whatever N is — one time step of it costs minutes, so at most one warm-up step and
        # a tighter budget (the number of timed steps is reported)
        if w["scenario"] != "lid_driven2D":
            name = "lid_driven2D_nx707"
            w = WORKLOADS[name]
        nx = int(round(w["nx"] * math.sqrt(N)))
        W = min(W, 1)
        budget = CPU_BUDGET_WEAK_S
    r = cpu_steps(name, W, K, budget, nx=nx)
    if nx is not None:
        r["config"]["global_nx"] = nx
        r["config"]["cells_per_gpu"] = r["config"]["cells"] // N
    val = r["ndof"] * r["steps"] / r["seconds"]
    if cpu_sub_pc(name) == "lu":
        how = (f"FGMRES(200) + fieldsplit Schur FULL/SELFP + gmres/lu + preonly/lu (stabilized_schur_pressure_backflow.py:255-297): "
               f"cell kernels in C + OpenMP on {r['cores']} threads, A00 and Sp factorised by SciPy's SuperLU for every Jacobian "
               f"(sequential, like PETSc's own lu); ")
    else:
        how = (f"FGMRES(200) + fieldsplit Schur FULL/SELFP + GMRES(30)/ASM-ILU(0) (stabilized_schur.py:226-275) restated in "
               f"C + OpenMP, {r['cores']} threads = {r['cores']} ASM blocks; ")
    sample = (f"{r['steps']} timed time step(s) after {W} warm-up step(s) of {name} ({r['ndof']} DOFs), the same mesh and "
              f"steps as the GPU arm; " + how + 
              f"{r['newton_its']} Newton, {r['outer_its']} outer and {r['inner_its']} inner Krylov iterations in "
              f"{r['total_steps']} steps; assembly {r['timers']['assembly']:.1f} s, PCSetUp {r['timers']['pc_setup']:.1f} s, "
              f"KSPSolve {r['timers']['ksp']:.1f} s")
    line = {
        "impl": "reference", "metric": "DOF-timesteps/s", "value": val, "unit": "DOF-timesteps/s",
        "n_gpus": args.gpus, "steps": r["steps"], "warmup": W, "ms_per_step": 1e3 * r["seconds"] / r["steps"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": r["config"],
        "note": "DOLFINx/PETSc are not installable in this image (no wheels, no MPI): the CPU arm is the reference's "
                "solver configuration restated in C + OpenMP on all host cores (oracle/c/ref_ksp.c, "
                "oracle/c/p1tri_cells.c), parity unpinned against PETSc itself",
        "cpu_baseline": {"value": val, "unit": "DOF-timesteps/s", "cores": r["cores"], "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "DOF-timesteps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# ------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------
def hierarchy_bytes(s):
    """Algorithmic bytes of one preconditioner application from the level sizes (fp32 hierarchy storage):
    per level and cycle, the operator is read by 1 (pre, from zero) + 1 (residual) + 2 (post) sweeps and the
    transfer operators once each."""
    lin = s.linear
    out = 0.0
    n0 = s.n
    for which, bs in ((0, 2), (1, 1)):
        lv = lin.levels[which] if which < len(lin.levels) else []
        if not lv:
            continue
        nn = n0
        nnz = s.hemo.nnz_node if not (which == 1 and lin.schur_mode == "selfp") else lv[0]["AP"].shape[0] * 19
        cyc = lin.opts["amg_cycles_u"] if which == 0 else lin.opts["amg_cycles_p"]
        for d in lv:
            op = nnz * (4 * bs * bs + 4) + nn * (4 + 4 * bs * 7)
            tr = 2 * d["P"].nnz * (8 + 4) + 2 * nn * 4 * bs
            out += cyc * (3 * op + tr)
            nnz = d["C"].nnz
            nn = d["P"].shape[1]
    return out


def measure_workload(name, W, K, local_rank, want_e2e=True, want_prof=True, solver_kw=None, dump_dir=None):
    import torch
    w = WORKLOADS[name]
    t_build = time.perf_counter()
    with contextlib.redirect_stdout(sys.stderr):       # stdout carries exactly one JSON line
        sc = build_scenario(w, device=local_rank, **(solver_kw or {}))
    t_build = time.perf_counter() - t_build
    s = sc.solver
    hemo = s.hemo
    ndof = s.N
    E = s._cells_host.shape[0]
    nnz = hemo.nnz
    dev = hemo.device
    n = s.n
    nnz_node = hemo.nnz_node
    nv = int(s._cells_host.shape[1])

    # ---- device-resident timed region --------------------------------------
    for _ in range(W):
        s.step_device()
    torch.cuda.synchronize(dev)
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = hemo.launches
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    newton = ksp = 0
    e0.record()
    for _ in range(K):
        s.step_device()
        newton += s.its_snes
        ksp += s.its_ksp
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    launches = hemo.launches - launches0
    clocks = sampler.stop()
    if dump_dir:
        # the solution of the last timed step, as step_device() leaves it for its caller (the steps below march on)
        dump_outputs(dump_dir, {"velocity": s.d_x[:2 * n].cpu().numpy(), "pressure": s.d_x[2 * n:].cpu().numpy()})
    out = dict(config=workload_config(name, sc), value=ndof * K / (ms * 1e-3), ms_per_step=ms / K, steps=K, warmup=W,
               newton_its_per_step=newton / K, fgmres_its_per_step=ksp / K, gpu_launches=launches, clocks=clocks,
               nnz=nnz, build_s=t_build)

    # ---- per-kernel-class CUDA-event times: the timed region above replays whole FGMRES iterations as CUDA graphs,
    # whose kernels carry no event pairs; two extra steps with direct launches (same kernels, same data) time the
    # classes with the library's event pairs and their shares are scaled to the timed region -------------------
    prof = None
    if want_prof:
        hemo.use_graph(False)
        s.step_device()
        hemo.prof_enable(True)
        g0 = torch.cuda.Event(enable_timing=True)
        g1 = torch.cuda.Event(enable_timing=True)
        g0.record()
        kp = 0
        for _ in range(2):
            s.step_device()
            kp += s.its_ksp
        g1.record()
        torch.cuda.synchronize(dev)
        ms_nograph = g0.elapsed_time(g1)
        prof = {c: hemo.prof_get(c) for c in PROF_CLASSES}
        hemo.prof_enable(False)
        hemo.use_graph(True)
        s.step_device()          # re-captures the graphs
        out["ms_per_step_direct_launches"] = ms_nograph / 2

    # ---- isolated assembly timings (cells/s, nnz/s) ------------------------------
    def time_fn(fn, reps=5):
        fn()
        torch.cuda.synchronize(dev)
        a = torch.cuda.Event(enable_timing=True)
        b = torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize(dev)
        return a.elapsed_time(b) / reps

    jac_ms = time_fn(lambda: hemo.assemble_jacobian(s.d_x, s.d_un, s.d_vals))
    res_ms = time_fn(lambda: hemo.assemble_residual(s.d_x, s.d_un, s.d_bcval, s.d_g))
    out["assembly"] = {"jacobian_cells_per_s": E / (jac_ms * 1e-3), "jacobian_nnz_per_s": nnz / (jac_ms * 1e-3),
                       "residual_cells_per_s": E / (res_ms * 1e-3), "jacobian_ms": jac_ms, "residual_ms": res_ms}

    # ---- end to end through the plugin API (host buffers) ------------------------
    if want_e2e:
        for _ in range(2):
            s.solveStep()
            s.u_prev.x.array[:] = s.u_sol.x.array[:]
            s.p_prev.x.array[:] = s.p_sol.x.array[:]
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(K):
            s.solveStep()
            s.u_prev.x.array[:] = s.u_sol.x.array[:]
            s.p_prev.x.array[:] = s.p_sol.x.array[:]
        torch.cuda.synchronize(dev)
        out["e2e"] = {"value": ndof * K / (time.perf_counter() - t0), "unit": "DOF-timesteps/s",
                      "h2d_bytes_per_step": s.h2d_bytes_per_step, "d2h_bytes_per_step": s.d2h_bytes_per_step}

    # ---- roofline ---------------------------------------------------------------------
    peak, peak_kind = measured_peaks()
    ae_bytes = 72 * nv * nv * E
    its_per_solve = max(ksp / max(newton, 1), 1.0)
    # average number of basis vectors per Gram-Schmidt pass: iteration i of a solve works on (i mod restart) + 1
    restart = max(int(getattr(s, "ksp_restart", 60)), 1)
    L = max(int(round(its_per_solve)), 1)
    kavg = sum((i % restart) + 1 for i in range(L)) / L
    alg_bytes = {
        0: 76 * nnz_node + 52 * n + 24 * n,               # J values + node cols + rowptr + x + y (+ the Z_j copy)
        1: 4 * nv * E + 8 * E + 56 * n + ae_bytes,        # cells, h, nodal gathers, element matrices out
        2: ae_bytes + 4 * nv * nv * E + 12 * nnz_node + 72 * nnz_node,
        3: 4 * nv * E + 8 * E + 56 * n + 24 * nv * E,
        4: 20 * nnz_node + 4 * n + 56 * n,                # A00 BSR2 fp32 values + cols + rowptr + 7 fp32 vectors of 2n
        5: 8 * nnz_node + 4 * n + 28 * n,
        6: 8 * ndof * (kavg + 1),                          # V_0..V_j and w read once
        7: 8 * ndof * (kavg + 2),                          # V_0..V_j read, w read + written
        8: None,
    }
    if prof is not None:
        scale = (ms / K) / (ms_nograph / 2) if ms_nograph > 0 else 1.0
        classes = {}
        for c, (t, cnt) in prof.items():
            if cnt == 0:
                continue
            avg_us = 1e3 * t / cnt
            gbps = alg_bytes[c] / (avg_us * 1e-6) / 1e9 if alg_bytes.get(c) else None
            classes[PROF_CLASSES[c]] = {"avg_us": avg_us, "launches_per_step": cnt / 2, "share_of_step": t / ms_nograph,
                                        "GBps": gbps, "frac_of_hbm_peak": gbps / peak if gbps else None}
        hbm = [c for c in (0, 2, 4, 5, 6, 7) if prof[c][1] > 0]
        dom = max(hbm, key=lambda c: prof[c][0], default=0)
        dms, dcnt = prof[dom]
        achieved = alg_bytes[dom] / (dms / dcnt * 1e-3) / 1e9 if dcnt else 0.0
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            traffic = tj.get("workloads", {}).get(name, {}).get("dram_bytes_per_launch", {}).get(PROF_CLASSES[dom])
        # whole step: algorithmic bytes of everything executed / step time
        step_bytes = (ksp / K) * (alg_bytes[0] + alg_bytes[6] + alg_bytes[7] + hierarchy_bytes(s) + 16 * ndof) \
            + (newton / K) * (alg_bytes[1] + alg_bytes[2]) + (newton / K + 1) * alg_bytes[3]
        out["roofline"] = {
            "bound": "hbm", "kernel": PROF_CLASSES[dom], "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "traffic": traffic, "peak_source": peak_kind, "launches_timed": dcnt,
            "avg_us": 1e3 * dms / max(dcnt, 1), "share_of_step": dms / ms_nograph,
            "how": "CUDA-event pairs around every launch of the class (library side, on the solver's stream) during two "
                   "extra time steps with direct launches; the timed region itself replays CUDA graphs",
            "whole_step": {"algorithmic_bytes": step_bytes, "GBps": step_bytes / (ms / K * 1e-3) / 1e9,
                           "frac": step_bytes / (ms / K * 1e-3) / 1e9 / peak},
            "fp64_bound": {"kernels": ["cell_jacobian", "cell_residual"],
                           "cell_jacobian_Gcells_per_s": E / max(prof[1][0] / max(prof[1][1], 1), 1e-9) / 1e6,
                           "cell_residual_Gcells_per_s": E / max(prof[3][0] / max(prof[3][1], 1), 1e-9) / 1e6},
            "classes": classes, "graph_vs_direct_scale": scale}
    out["precision"] = ("outer FGMRES, Jacobian, residuals, reductions: fp64; multigrid hierarchy storage (operators, "
                        "smoother vectors, A01 copy): fp32 with fp64 accumulation (preconditioner only)")
    # free the device before the next workload
    sc.solver.hemo.close()
    del sc, s
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    return out


def run_distributed(args, name, W, K, world, rank, local_rank):
    """N > 1: ONE mesh partitioned over the GPUs (vertex-owned x-slabs), halo exchange and Krylov allreduces with
    NCCL inside the library.  Weak scaling: the per-GPU cell count is held at the single-GPU workload's, so the
    global mesh is nx*sqrt(N) squared."""
    import torch
    import torch.distributed as dist
    from cfd_hemodynamic_b200.distributed_solver import DistributedStabilizedSchur
    from cfd_hemodynamic_b200.parallel import slab_partition
    from cfd_hemodynamic_b200.src.scenarios.lid_driven2D import LidDriven2DSimulation
    w = WORKLOADS[name]
    nx = int(round(w["nx"] * math.sqrt(world)))
    with contextlib.redirect_stdout(sys.stderr):
        sc = LidDriven2DSimulation("stabilized_schur", w["dt"], 1.0, rho=w["rho"], mu=w["mu"], nx=nx, host_only=True)
    tables = sc.solver.export_tables()
    owner = slab_partition(tables["x"][:, 0], world)
    ds = DistributedStabilizedSchur(tables, owner, local_rank)
    dev = ds.hemo.device
    ndof = 3 * ds.n_global
    E = tables["cells"].shape[0]

    def barrier():
        torch.cuda.synchronize(dev)
        dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(W):
        ds.step_device()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = ds.launches()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    newton = ksp = 0
    e0.record()
    for _ in range(K):
        ds.step_device()
        newton += ds.its_snes
        ksp += ds.its_ksp
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    launches = torch.tensor([float(ds.launches() - l0)], dtype=torch.float64, device=dev)
    dist.all_reduce(launches)
    clocks = sampler.stop()
    # e2e: owned values are pulled to pinned host memory and u_prev pushed back every step
    nl = ds.n
    host = torch.empty(3 * nl, dtype=torch.float64).pin_memory()
    hun = torch.empty(2 * nl, dtype=torch.float64).pin_memory()
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        ds.d_un.copy_(hun.copy_(ds.d_un, non_blocking=True), non_blocking=True)   # host-owned time-level shift
        ds.step_device()
        host.copy_(ds.d_x, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
    barrier()
    te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    dist.all_reduce(te, op=dist.ReduceOp.MAX)
    info = ds.comm_summary()
    # per-phase CUDA-event times (library side) from two extra steps with direct launches: the timed region replays
    # CUDA graphs; a rank's halo / allreduce time includes waiting for its peers
    ds.hemo.use_graph(False)
    ds.step_device()
    ds.hemo.prof_enable(True)
    g0 = torch.cuda.Event(enable_timing=True)
    g1 = torch.cuda.Event(enable_timing=True)
    g0.record()
    kp = 0
    for _ in range(2):
        ds.step_device()
        kp += ds.its_ksp
    g1.record()
    torch.cuda.synchronize(dev)
    names = {0: "spmv", 6: "mdot", 7: "maxpy_norm", 9: "halo", 10: "allreduce", 11: "pressure_coarse_space", 12: "preconditioner"}
    phases = {}
    for c, nm in names.items():
        t_c, cnt = ds.hemo.prof_get(c)
        phases[nm] = {"ms_per_iteration": t_c / max(kp, 1), "launches_per_iteration": cnt / max(kp, 1)}
    phases["direct_launch_ms_per_iteration"] = g0.elapsed_time(g1) / max(kp, 1)
    phases["graph_ms_per_iteration"] = ms / max(ksp, 1)
    ds.hemo.prof_enable(False)
    ds.hemo.use_graph(True)
    info["phases_rank0"] = phases
    if rank == 0:
        peak, peak_kind = measured_peaks()
        # roofline of the dominant HBM-bound kernel on rank 0's partition (library-side CUDA events of the direct-launch steps)
        roof = {"bound": "hbm", "kernel": "see the N=1 line (same kernels per partition)", "achieved": None, "peak": peak,
                "unit": "GB/s", "frac": None, "traffic": None, "peak_source": peak_kind}
        try:
            per_launch_ms = phases["spmv"]["ms_per_iteration"] / max(phases["spmv"]["launches_per_iteration"], 1e-12)
            alg = 76.0 * float(ds.hemo.nnz_node) + 76.0 * float(ds.n)      # J values + node columns + x, y, Z_j of the partition
            if per_launch_ms > 0.0:
                ach = alg / (per_launch_ms * 1e-3) / 1e9
                roof.update({"kernel": "spmv_node(J) on rank 0's partition (owned + overlap nodes)", "achieved": ach,
                             "frac": ach / peak, "avg_us": 1e3 * per_launch_ms, "algorithmic_bytes": alg})
        except Exception as exc:                                  # never lose the line over a derived figure
            roof["note"] = f"{type(exc).__name__}: {exc}"
        line = {
            "metric": "DOF-timesteps/s", "value": ndof * K / (ms * 1e-3), "unit": "DOF-timesteps/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": name, "solver": "stabilized_schur", "cell_type": "triangle", "cells": E, "dofs": ndof,
                       "global_nx": nx, "cells_per_gpu": E // world, "dt": w["dt"], "mu": w["mu"], "rho": w["rho"],
                       "l2": "inputs larger than L2 (per-GPU matrix %.0f MB vs 126 MB L2)" % (8 * ds.hemo.nnz / 1e6)},
            "solve": {"newton_its_per_step": newton / K, "fgmres_its_per_step": ksp / K},
            "parallelism": info,
            "e2e": {"value": ndof * K / float(te.item()), "unit": "DOF-timesteps/s",
                    "h2d_bytes_per_step": world * 8 * 2 * nl, "d2h_bytes_per_step": world * 8 * 3 * nl},
            "gpu_launches": int(launches.item()), "clocks": clocks,
            "roofline": roof,
            "cpu_baseline": None,
        }
        emit(line)
    dist.destroy_process_group()


_REAL_STDOUT = None


def _guard_stdout():
    """stdout must carry exactly one JSON line: C-level writers (the NCCL version banner, library diagnostics) and
    stray prints are sent to stderr for the whole run; emit() writes the line to the real stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the larger GPU-only workloads")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the velocity and pressure of the last timed step as DIR/<name>.npy (float64, at most "
                         "64 MB in all; a fixed, seeded sample of larger solutions); single-GPU arm only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs is implemented for the single-GPU arm only")
    _guard_stdout()
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the hot path exists only as sm_100a kernels (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    W = max(3, args.warmup)
    K = args.steps
    name = args.workload

    if world > 1:
        run_distributed(args, name if WORKLOADS[name]["scenario"] == "lid_driven2D" else "lid_driven2D_nx707", W, K,
                        world, rank, local_rank)
        return

    r = measure_workload(name, W, K, local_rank, want_e2e=not args.no_e2e, dump_dir=args.dump_outputs)
    others = {}
    if name == DEFAULT_WORKLOAD and not args.no_extra:
        for ename, ew, ek in EXTRA_WORKLOADS:
            t0 = time.perf_counter()
            try:
                o = measure_workload(ename, ew, ek, local_rank, want_e2e=True, want_prof=True)
                o["wall_s"] = time.perf_counter() - t0
                o["cpu_arm"] = ("not run in this line: the reference's algorithm needs 80 s per time step of lid_driven2D_nx707 on the GPU box's "
                                "16 host cores (profiles/r02_cpu_arm_lid707.json), i.e. more than the driver's time limit for W + K steps")
                others[ename] = o
            except Exception as exc:                        # a failed extra workload must not void the main line
                others[ename] = {"error": f"{type(exc).__name__}: {exc}"}

    # ---- CPU baseline: the reference's algorithm on the host cores, one time step of the SAME mesh ----------
    cpu = None
    if not args.no_cpu_baseline and WORKLOADS[name]["scenario"] == "lid_driven2D":
        c = cpu_steps(name, 0, 1, 120.0)
        cpu = {"value": c["ndof"] * c["steps"] / c["seconds"], "unit": "DOF-timesteps/s", "cores": c["cores"], "kind": "port",
               "sample": f"the first time step of {name} ({c['ndof']} DOFs, the same mesh) with the reference's solver "
                         f"configuration restated in C + OpenMP (FGMRES(200) + fieldsplit Schur FULL/SELFP + "
                         f"GMRES(30)/ASM-ILU(0), {c['cores']} threads): {c['seconds']:.1f} s, {c['newton_its']} Newton / "
                         f"{c['outer_its']} outer / {c['inner_its']} inner iterations; DOLFINx/PETSc not installable here"}

    line = {
        "metric": "DOF-timesteps/s", "value": r["value"], "unit": "DOF-timesteps/s", "n_gpus": 1, "steps": K,
        "warmup": W, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": r["config"],
        "solve": {"newton_its_per_step": r["newton_its_per_step"], "fgmres_its_per_step": r["fgmres_its_per_step"],
                  "nnz": r["nnz"], "ms_per_step_direct_launches": r.get("ms_per_step_direct_launches")},
        "parallelism": "1 GPU", "precision": r["precision"],
        "assembly": r["assembly"], "e2e": r.get("e2e"), "gpu_launches": r["gpu_launches"], "clocks": r["clocks"],
        "roofline": r.get("roofline"), "cpu_baseline": cpu, "other_workloads": others,
    }
    emit(line)


if __name__ == "__main__":
    main()
