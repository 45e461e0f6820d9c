#!/usr/bin/env python3
"""bench.py -- IPCS time steps per second, 3D Taylor-Green P2-P1 on an N^3 box (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--mesh 96] [--workload cavity]
                   [--dump-outputs DIR]

One "step" = one ``FractionalStep_AB_CN.solve(dt, nu, max_iter=1)`` (fracstep.py:660-696) on the
z-extruded Taylor-Green problem of SURVEY.md 8(d): box [-1,1]^3, N^3 x 6 Kuhn tetrahedra, P2-P1,
nu = 0.01, dt = 0.005, BiCGStab+Jacobi (tentative velocity), CG+multigrid (pressure, null space projected),
CG+Jacobi (mass), rtol 1e-10, initial guesses extrapolated from the solution histories (KRYLOV below; the CPU arm uses
the same options except a Jacobi-preconditioned pressure CG).  Default: the reference demo's 100 steps after 3 warm-up
steps; the first ~30 steps carry the start-up transient (more Krylov iterations), so short runs report fewer steps/s.

  value   device-timed steps/s with every input (state, BC values of all timed steps) resident in HBM;
  e2e     the same steps through the public Python API (host evaluation of the callable BCs, H2D of
          the BC values, D2H of the step result), wall clock between two device synchronisations;
  roofline  the dominant kernel (CSR SpMM of the P2xP2 operator on gdim right-hand sides) timed live
          with CUDA events on the context's stream, algorithmic bytes / time vs MEASURED_PEAKS.json;
  cpu_baseline  the CPU restatement (oracle/) on the box's host cores on a bounded sample.

``--impl reference`` times the CPU restatement only (the DOLFINx/PETSc reference cannot be installed
here: DESIGN.md).  No torch: ranks are launched by torchrun but only RANK/WORLD_SIZE are read.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "IPCS steps/s, 3D Taylor-Green P2-P1 box"
DT, NU = 0.005, 0.01
PARITY_TOL = 1e-8  # GPU fields against the CPU port after the same steps (north_star: 1e-8 relative at rtol 1e-10)
KRYLOV = {
    "tentative": {"ksp_type": "bcgs", "pc_type": "jacobi", "ksp_rtol": 1e-10, "ksp_initial_guess_nonzero": True,
                  "b200_guess": "extrapolate2", "b200_block_rtol": True},
    "pressure": {"ksp_type": "cg", "pc_type": "mg", "ksp_rtol": 1e-10, "ksp_initial_guess_nonzero": True,
                 "b200_guess": "extrapolate"},
    "scalar": {"ksp_type": "cg", "pc_type": "jacobi", "ksp_rtol": 1e-10, "ksp_initial_guess_nonzero": True,
               "b200_guess": "extrapolate2", "b200_block_rtol": True},
}


def ncu_traffic(mesh: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of one k_spmm launch from the committed `ncu --set full`
    capture (profiles/r02_ncu_spmm_96cube.txt, first kernel of the file); only valid for the mesh it was taken on."""
    if mesh != 96:
        return None
    try:
        tot, seen = 0.0, set()
        for line in open(os.path.join(ROOT, "profiles", "r02_ncu_spmm_96cube.txt")):
            f = line.split()
            if len(f) >= 3 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and f[0] not in seen:
                seen.add(f[0])
                tot += float(f[1]) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[f[2]]
        return tot or None
    except Exception:
        return None


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def step_algorithmic_bytes(n2, n1, nnz22, nnz21, nnz11, gdim, its, bytes_assemble, bytes_spmm, bytes_spmv_q):
    """Algorithmic bytes of ONE IPCS step with the measured Krylov iteration counts its = (k_u, k_p, k_m): the
    per-kernel figures of SURVEY.md 8(d) (k-RHS SpMM, CSR-value passes, 8 bytes per vector entry read or written)
    summed over the kernels a step launches (DESIGN.md section 4).  An accounting aid for `step_roofline`, not a
    measurement."""
    k_u, k_p, k_m = its
    vec = 8.0 * gdim * n2  # one pass over a velocity-space vector (all components)
    q = 8.0 * n1           # one pass over a pressure-space vector
    rect = nnz21 * (8.0 * gdim + 4.0)  # one pass over a rectangular operator family ([nnz][gdim] values + columns)
    tentative = (rect + 2 * vec + q) + 4 * vec + (bytes_spmm + 5 * vec) + k_u * (2 * bytes_spmm + 14 * vec) + 6 * vec
    pressure = (rect + vec + q) + 6 * q + k_p * (1.15 * (3 * bytes_spmv_q + 10 * q) + 6 * q) + 4 * q
    update = (bytes_spmm) + (rect + 2 * vec + q) + 7 * vec + (bytes_spmm + 5 * vec) + k_m * (bytes_spmm + 10 * vec) + 5 * vec
    state = 2 * vec + 2 * q  # u1 <- u, p <- ps
    return {"assemble_first": bytes_assemble, "tentative": tentative, "pressure": pressure, "update": update,
            "total": bytes_assemble + tentative + pressure + update + state}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.proc, self.path = device, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        try:
            rows = [r.strip().split(", ") for r in open(self.path) if r.strip()]
            os.unlink(self.path)
            sm = [float(r[0]) for r in rows if len(r) >= 7]
            if sm:
                out["sm_mhz"] = float(np.median(sm))
                out["sm_max_mhz"] = float(rows[0][1])
                out["power_w_max"] = max(float(r[2]) for r in rows if len(r) >= 7)
                out["samples"] = len(sm)
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                for k, nm in enumerate(names):
                    if any(r[3 + k].strip() == "Active" for r in rows if len(r) >= 7):
                        out["reasons"].append(nm)
        except Exception:
            pass
        return out


DUMP_MAX_ENTRIES = 1 << 20  # per array (8 MiB in float64): at most 4 arrays, 32 MiB per run


def dump_outputs(out_dir: str, arrays: dict):
    """Write each array as <out_dir>/<name>.npy in float64, so that two builds run with the same arguments can be
    compared output for output.  An array longer than DUMP_MAX_ENTRIES is replaced by the entries at a fixed, seeded
    sample of sorted indices (the same indices for the same array length).  The device reductions do not sum in a
    fixed order: two runs of one build differ by about 1e-14 relative (B200, 48^3, 10 steps)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64).ravel()
        if a.size > DUMP_MAX_ENTRIES:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ENTRIES, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def bc_series(solver, tg, t_first: float, n_steps: int):
    """g_i at the merged BC dofs for n_steps consecutive steps, evaluated on the host ahead of time."""
    out = []
    for i, bcl in enumerate(solver._bcs_u):
        bc = bcl[0]
        own = bc._dofs < solver._nV_owned  # the device list holds the owned BC dofs only
        xT = np.ascontiguousarray(bc._xT[:, own])
        vals = np.empty((n_steps, int(own.sum())))
        for s in range(n_steps):
            tg.t_u = t_first + s * DT
            vals[s] = bc._value(xT)
        out.append(vals)
    return out


# ---- second workload: lid-driven cavity (BASELINE.json configs[4]), unit cube, Re = 1000 ---------------------
CAVITY_NU, CAVITY_DT = 1.0e-3, 0.005


def _cavity_markers():
    lid = lambda x: np.isclose(x[2], 1.0)
    walls = lambda x: (np.isclose(x[0], 0) | np.isclose(x[0], 1) | np.isclose(x[1], 0) | np.isclose(x[1], 1) | np.isclose(x[2], 0)) & ~lid(x)
    return lid, walls


def make_cavity_solver(N: int, comm, device: int, nz_factor: int = 1):
    """Unit cube, u = (1, 0, 0) on the lid z = top, no slip on the other walls, no pressure BC, start from rest
    (the set-up of tests/test_gpu_parity.py::test_lid_driven_cavity_matches_oracle at Re = 1000).  nz_factor > 1
    (weak scaling): the box [0,1]^2 x [0, nz_factor] with N x N x (N nz_factor) cubes -- one N^3 block per rank."""
    import oasisx_b200 as oasisx
    from oasisx_b200 import mesh as bmesh

    top = float(nz_factor)
    msh = bmesh.create_box(comm, [[0.0, 0.0, 0.0], [1.0, 1.0, top]], [N, N, N * nz_factor])
    lid = lambda x: np.isclose(x[2], top)
    walls = lambda x: (np.isclose(x[0], 0) | np.isclose(x[0], 1) | np.isclose(x[1], 0) | np.isclose(x[1], 1) | np.isclose(x[2], 0)) & ~lid(x)
    G = oasisx.LocatorMethod.GEOMETRICAL
    bcs_u = [[oasisx.DirichletBC(0.0, G, walls), oasisx.DirichletBC(1.0 if k == 0 else 0.0, G, lid)] for k in range(3)]
    s = oasisx.FractionalStep_AB_CN(msh, ("Lagrange", 2), ("Lagrange", 1), bcs_u=bcs_u, bcs_p=[], solver_options=KRYLOV,
                                    options={"low_memory_version": False}, device=device)
    return msh, s


def cpu_sample_cavity(n_cpu: int, n_steps: int, n_warm: int = 1):
    from oasisx_b200 import fem, mesh as bmesh
    from oracle import ipcs_cpu as cpu

    cpu.use_all_cores()
    msh = bmesh.create_unit_cube(None, n_cpu, n_cpu, n_cpu)
    V, Q = fem.functionspace(msh, ("Lagrange", 2)), fem.functionspace(msh, ("Lagrange", 1))
    lid, walls = _cavity_markers()
    bd = fem.locate_dofs_geometrical(V, lambda x: lid(x) | walls(x))
    vals = [lambda x: np.where(lid(x), 1.0, 0.0), lambda x: np.zeros_like(x[0]), lambda x: np.zeros_like(x[0])]
    c = cpu.CpuIPCS(msh.geometry.x, msh.geometry.dofmap, 3, V.dofmap.list, Q.dofmap.list, V.tabulate_dof_coordinates(),
                    Q.tabulate_dof_coordinates(), 2, bcs_u=[[(bd, f)] for f in vals],
                    rtol=KRYLOV["tentative"]["ksp_rtol"], nonzero_guess=True, block_rtol=True,
                    extrapolate={"extrapolate": 1, "extrapolate2": 2}.get(KRYLOV["tentative"].get("b200_guess"), 0))
    if KRYLOV["pressure"].get("pc_type") == "mg":
        c.attach_pressure_multigrid(msh)
    for _ in range(n_warm):
        c.solve(CAVITY_DT, CAVITY_NU)
    t0 = time.perf_counter()
    for _ in range(n_steps):
        c.solve(CAVITY_DT, CAVITY_NU)
    return (time.perf_counter() - t0) / n_steps, getattr(msh, "num_cells_global", msh.num_cells), cpu.lib().ipcs_cpu_threads(), c.its.tolist()


def run_cavity(args):
    """Lid-driven cavity at Re = 1000 on an N^3 unit cube (default 128^3 = 53 M dofs on ONE GPU; with several ranks
    the same global mesh is split in z-slabs: strong scaling).  --weak: BASELINE.json configs[4], one N^3 block of cubes
    per GPU, box [0,1]^2 x [0, n_gpus]; every rank builds only its own slab (oasisx_b200/slab.py), so the set-up time
    does not grow with the job.  Same JSON contract as the Taylor-Green line; constant boundary values, so the
    end-to-end path moves no boundary data after the first step."""
    from oasisx_b200.comm import HostComm

    comm = HostComm.from_env()
    rank, world = comm.rank, comm.size
    device = int(os.environ.get("LOCAL_RANK", "0"))
    N, K, W = args.mesh, args.steps, max(args.warmup, 3)
    weak = bool(args.weak)
    t_setup = time.perf_counter()
    msh, solver = make_cavity_solver(N, comm if world > 1 else None, device, world if weak else 1)
    ctx = solver._ctx
    t_setup = time.perf_counter() - t_setup
    t_setup_max = comm.allreduce(t_setup, "max")
    dt, nu = CAVITY_DT, CAVITY_NU
    for s in range(W):
        solver.solve(dt, nu, max_iter=1)
    st0 = ctx.stats()
    sampler = ClockSampler(device)
    sampler.start()
    ctx.synchronize()
    comm.Barrier()
    ctx.event_record(0)
    t0 = time.perf_counter()
    its, stage_ms = [], np.zeros(4)
    for s in range(K):
        solver.solve(dt, nu, max_iter=1)  # constant BCs: after the first step this is the device path plus one scalar D2H
        st = ctx.stats()
        its.append((max(st.its_tentative), st.its_pressure, max(st.its_update)))
        stage_ms += [st.ms_assemble_first, st.ms_tentative, st.ms_pressure, st.ms_update]
    ctx.event_record(1)
    ctx.synchronize()
    e2e_s = comm.allreduce((time.perf_counter() - t0) / K, "max")
    ms_total = comm.allreduce(ctx.event_elapsed_ms(0, 1), "max")
    comm.Barrier()
    clocks = sampler.stop()
    st1 = ctx.stats()
    launches = comm.allreduce(int(st1.kernel_launches - st0.kernel_launches))
    umax = comm.allreduce(float(np.abs(solver._u[0].x.array_ro()).max()), "max")
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {**{f"u{i}": solver._u[i].x.array_ro()[:solver._nV_owned] for i in range(3)},
                                         "p": solver._p.x.array_ro()[:solver._nQ_owned]})
    peak, peak_kind = measured_peaks()
    ms_k, bytes_k = ctx.bench_kernel(3, 20)
    if rank != 0:
        comm.Barrier()
        return
    cpu = None
    if not args.no_cpu and world == 1:
        n_cpu = args.cpu_mesh if args.cpu_mesh > 0 else min(N, 64)
        sec, cells, threads, cits = cpu_sample_cavity(n_cpu, 2, 1)
        sps = (1.0 / sec) * cells / getattr(msh, "num_cells_global", msh.num_cells)
        cpu = {"value": sps, "unit": "steps/s", "cores": threads, "kind": "port",
               "sample": f"C++/OpenMP restatement, 2 cavity steps after 1 warm-up on a {n_cpu}^3 cube ({sec:.2f} s/step, its u/p/m {cits})"
                         + ("" if n_cpu == N else f", scaled by cell count to {N}^3 (optimistic for the CPU: its Jacobi-PCG pressure iterations grow with N)"),
               "host_cpus": os.cpu_count()}
    nV = solver._lp.V.n_global if world > 1 else solver._nV_owned
    nQ = solver._lp.Q.n_global if world > 1 else solver._nQ_owned
    line = {
        "metric": "IPCS steps/s, 3D lid-driven cavity P2-P1 box", "value": 1000.0 * K / ms_total, "unit": "steps/s", "n_gpus": world,
        "steps": K, "warmup": W, "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak" if weak else "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": (f"3D lid-driven cavity P2-P1, WEAK scaling: one {N}^3 block of cubes per GPU, box [0,1]^2 x [0,{world}] "
                                f"({N}x{N}x{N * world} cubes)" if weak else f"3D lid-driven cavity P2-P1 {N}^3 unit cube")
                               + f", Re=1000 (nu={nu}, lid speed 1), dt={dt}, from rest, max_iter=1, rtol=1e-10",
                   "mesh": N, "cells": getattr(msh, "num_cells_global", msh.num_cells), "dofs": 3 * nV + nQ, "krylov": KRYLOV, "setup_s": t_setup,
                   "setup_s_max_over_ranks": t_setup_max,
                   "mesh_provider": "slab-local (each rank builds its own slab)" if hasattr(msh, "is_global_boundary") else
                                    ("replicated global mesh, partitioned" if world > 1 else "single rank"),
                   "l2": "working set per step >> 126 MB L2; no flush needed"},
        "iterations": {"tentative": int(np.median([i[0] for i in its])), "pressure": int(np.median([i[1] for i in its])),
                       "update": int(np.median([i[2] for i in its]))},
        "stage_ms": dict(zip(["assemble_first", "tentative", "pressure", "update"], (stage_ms / K).round(3).tolist())),
        "max_abs_u_x": umax,
        "roofline": {"bound": "hbm", "kernel": "k_spmm<K=3> (P2xP2 SELL-32 operator, 3 right-hand sides)", "achieved": bytes_k / (ms_k * 1e-3) / 1e9,
                     "peak": peak, "peak_kind": peak_kind, "unit": "GB/s", "frac": bytes_k / (ms_k * 1e-3) / 1e9 / peak, "traffic": None,
                     "ms_per_launch": ms_k, "algorithmic_bytes": bytes_k},
        "cpu_baseline": cpu,
        "e2e": {"value": 1.0 / e2e_s, "unit": "steps/s", "h2d_bytes_per_step": int(st1.bytes_h2d - st0.bytes_h2d) // K,
                "d2h_bytes_per_step": int(st1.bytes_d2h - st0.bytes_d2h) // K,
                "note": "the timed loop IS the public-API loop (constant boundary values: nothing to prefetch); value = device events, e2e = wall clock"},
        "gpu_launches": int(launches), "clocks": clocks,
    }
    print(json.dumps(line), flush=True)
    comm.Barrier()


def run_assembly_strategies(args):
    """BASELINE.json configs[1] = demo/assembly_strategies.py:56-152,221,230 on the device: P2 on the unit cube
    30 x 25 x 23 and 50 x 40 x 45, u_1 = sin(x) cos(y), u_ab,i = x, dt = 0.5, nu = 0.3; the tentative-velocity
    right-hand side b = (M/dt - nu/2 K - 1/2 C(u_ab)) u_1 by the matvec strategy (fused pass over the assembled value
    arrays) and by the action strategy (matrix-free element kernel), `assert np.allclose(b, b_d)` as the reference
    (:142), and the CPU port's timings of the reference's two blocks beside them.  One JSON line per mesh."""
    import oasisx_b200 as oasisx
    from oasisx_b200 import _lib as L, fem, mesh as bmesh

    dt, nu, reps = 0.5, 0.3, max(args.steps, 10)
    peak, peak_kind = measured_peaks()
    sizes = [(30, 25, 23), (50, 40, 45)] if args.mesh <= 0 or args.mesh == 96 else [(args.mesh,) * 3]
    u1f = lambda x: np.sin(x[0]) * np.cos(x[1])
    uabf = lambda x: x[0].copy()
    for shape in sizes:
        msh = bmesh.create_unit_cube(None, *shape)
        s = oasisx.FractionalStep_AB_CN(msh, ("Lagrange", 2), ("Lagrange", 1), bcs_u=[[], [], []], bcs_p=[],
                                        options={"low_memory_version": True}, device=int(os.environ.get("LOCAL_RANK", "0")))
        ctx = s._ctx
        for i in range(3):
            s._u1[i].interpolate(u1f)
            s._uab[i].interpolate(uabf)
        s._flush()
        sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
        sampler.start()
        r = ctx.bench_assembly_strategies(dt, nu, reps)
        clocks = sampler.stop()
        s._written(s._rhs1, s._b_first)
        b = s._rhs1[0].x.array_ro().copy()
        b_d = s._b_first[0].x.array_ro().copy()
        ok = bool(np.allclose(b, b_d))  # the reference's own assertion (rtol 1e-5, atol 1e-8)
        rel = float(np.abs(b - b_d).max() / np.abs(b).max())
        cpu = None
        if not args.no_cpu:
            from oracle import ipcs_cpu as cpum

            hi = host_info(stream=True)
            V, Q = fem.functionspace(msh, ("Lagrange", 2)), fem.functionspace(msh, ("Lagrange", 1))
            c = cpum.CpuIPCS(msh.geometry.x, msh.geometry.dofmap, 3, V.dofmap.list, Q.dofmap.list, V.tabulate_dof_coordinates(),
                             Q.tabulate_dof_coordinates(), 2, bcs_u=[[(np.zeros(0, np.int32), u1f)]] * 3)
            xV = V.tabulate_dof_coordinates().T
            for i in range(3):
                c.set(cpum.U1, i, u1f(xV))
                c.set(cpum.UAB, i, uabf(xV))
            sec, bm, ba = c.bench_strategies(0, dt, nu, 3)
            cpu = {"kind": "port", "cores": hi["threads"], "host": hi, "unit": "ms",
                   "ms_convection_assembly": sec[0] * 1e3, "ms_matvec": sec[1] * 1e3, "ms_action": sec[2] * 1e3,
                   "value": sec[1] * 1e3,
                   "sample": "oracle/ipcs_cpu.cpp: the reference's timed blocks (4 CSR passes / one cell loop), ONE scalar field, best of 3",
                   "allclose": bool(np.allclose(bm, ba)),
                   "gpu_vs_cpu_rel_diff": float(np.abs(b - bm).max() / np.abs(bm).max())}
        nnz = ctx.pattern_nnz(L.PAT_VV)
        line = {
            "metric": "tentative-velocity RHS assembly time, P2 unit cube (demo/assembly_strategies.py)", "unit": "ms",
            "value": r["ms_action"], "higher_is_better": False, "n_gpus": 1, "steps": reps, "warmup": 1, "ms_per_step": r["ms_action"],
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"assembly-strategies: unit cube {shape[0]}x{shape[1]}x{shape[2]}, P2, dt={dt}, nu={nu}, "
                                   "u_1 = sin(x)cos(y), u_ab,i = x; 3 right-hand sides (the reference times one scalar field)",
                       "cells": getattr(msh, "num_cells_global", msh.num_cells), "dofs_P2": s._nV_owned, "nnz": nnz, "first_plan": ctx.first_plan_info(),
                       "l2": "flush not needed at 50x40x45 (value arrays 3 x 0.3 GB); 30x25x23 (3 x 57 MB) partly fits the 126 MB L2: "
                             "back-to-back launches see warm lines there"},
            "strategies": {
                "matvec": {"ms": r["ms_matvec"], "algorithmic_bytes": r["bytes_matvec"], "GBs": r["bytes_matvec"] / r["ms_matvec"] / 1e6,
                           "frac_of_peak": r["bytes_matvec"] / r["ms_matvec"] / 1e6 / peak},
                "action": {"ms": r["ms_action"], "algorithmic_bytes": r["bytes_action"], "GBs": r["bytes_action"] / r["ms_action"] / 1e6,
                           "frac_of_peak": r["bytes_action"] / r["ms_action"] / 1e6 / peak,
                           "note": "FP64-compute-bound (about 2.6 kflop per cell against 56 B): the HBM fraction is not its roofline"},
                "convection_assembly": {"ms": r["ms_convection_assembly"], "algorithmic_bytes": r["bytes_convection_assembly"],
                                        "GBs": r["bytes_convection_assembly"] / r["ms_convection_assembly"] / 1e6},
                "allclose_b_matvec_b_action": ok, "max_rel_diff": rel},
            "roofline": {"bound": "hbm", "kernel": "k_matvec_rhs<3> (fused matvec strategy)", "achieved": r["bytes_matvec"] / r["ms_matvec"] / 1e6,
                         "peak": peak, "peak_kind": peak_kind, "unit": "GB/s", "frac": r["bytes_matvec"] / r["ms_matvec"] / 1e6 / peak, "traffic": None},
            "cpu_baseline": cpu, "gpu_launches": 3 * (reps + 1), "clocks": clocks,
            "e2e": None,
        }
        print(json.dumps(line), flush=True)
        if not ok:
            raise SystemExit("assembly-strategies: matvec and action right-hand sides differ")


def make_field(workload: str):
    """The exact solution a Taylor-Green workload runs on: `taylor-green-rot` = the 2D vortex rotated out of the x-y
    plane (three live velocity components, PETSc-standard per-component rtol), `taylor-green-z` = the z-extruded field
    (w = 0) with the block-relative tolerance of round 1."""
    from problems import TaylorGreen, TaylorGreenRot

    if workload == "taylor-green-2d":
        return TaylorGreen(NU, 2)
    return TaylorGreenRot(NU) if workload == "taylor-green-rot" else TaylorGreen(NU, 3)


def gdim_of(workload: str) -> int:
    return 2 if workload == "taylor-green-2d" else 3


def krylov_for(workload: str) -> dict:
    import copy

    k = copy.deepcopy(KRYLOV)
    if workload in ("taylor-green-rot", "taylor-green-2d"):  # PETSc's convergence test: every component against its own right-hand side
        for o in k.values():
            o.pop("b200_block_rtol", None)
    return k


def host_info(stream: bool = True) -> dict:
    """CPU model, affinity, the OpenMP team the CPU port runs with, and a STREAM-triad figure of the host memory."""
    from oracle import ipcs_cpu as cpu

    info = cpu.use_all_cores()
    try:
        with open("/proc/cpuinfo") as f:
            models = [ln.split(":", 1)[1].strip() for ln in f if ln.startswith("model name")]
        info["cpu_model"] = models[0] if models else None
    except Exception:
        info["cpu_model"] = None
    if stream:
        info["stream_triad_GBs"] = round(cpu.stream_triad_gbs(), 1)
    return info


def cpu_step_bytes(n2, n1, nnz22, nnz21, nnz11, gdim, its, mg: bool) -> float:
    """Algorithmic bytes of one step of the CPU port's OWN algorithm (oracle/ipcs_cpu.cpp: unfused CSR passes of
    fracstep.py:435-469, one component at a time): what its achieved bandwidth is computed from."""
    k_u, k_p, k_m = its
    v2, v1 = 8.0 * n2, 8.0 * n1
    spmv22 = 12.0 * nnz22 + 4.0 * n2 + 2 * v2
    spmv21 = 12.0 * nnz21 + 4.0 * n2 + v2 + v1
    spmv11 = 12.0 * nnz11 + 4.0 * n1 + 2 * v1
    assemble = 8.0 * nnz22 * (1 + 2) + 3 * 8.0 * nnz22 + 3 * 8.0 * nnz22 + gdim * (spmv22 + 3 * v2)  # zero+RMW, 2 value passes, d SpMV
    tent = gdim * (spmv21 + 3 * v2) + gdim * (spmv22 + 5 * v2 + k_u * (2 * spmv22 + 12 * v2))
    pres = gdim * (spmv21 + 2 * v1) + 6 * v1 + k_p * ((3.3 if mg else 1.0) * spmv11 + 10 * v1)
    upd = gdim * (spmv22 + spmv21 + 3 * v2) + gdim * (spmv22 + 4 * v2 + k_m * (spmv22 + 10 * v2))
    return assemble + tent + pres + upd


def cpu_sample(n_cpu: int, n_steps: int, n_warm: int = 1, workload: str = "taylor-green-z", want_fields: bool = False,
               krylov: dict | None = None):
    """Time the CPU restatement (oracle/ipcs_cpu.cpp: C++/OpenMP, CSR, BiCGStab+Jacobi / CG+multigrid / CG+Jacobi: the
    same Krylov options, preconditioners and initial guesses as the GPU arm) on an n_cpu^3 box with all host threads
    (set explicitly: host_info()).  Returns a dict: seconds per step, cells, threads, iterations, sizes, and -- when
    asked -- the fields after the last step (the parity check of bench.py compares the GPU state with them)."""
    from oasisx_b200 import fem
    from oracle import ipcs_cpu as cpu
    from problems import boundary_facets, make_mesh

    cpu.use_all_cores()
    krylov = krylov or krylov_for(workload)
    tg = make_field(workload)
    gd = gdim_of(workload)
    msh = make_mesh(gd, n_cpu)
    V, Q = fem.functionspace(msh, ("Lagrange", 2)), fem.functionspace(msh, ("Lagrange", 1))
    bd = fem.locate_dofs_topological(V, gd - 1, boundary_facets(msh))
    c = cpu.CpuIPCS(msh.geometry.x, msh.geometry.dofmap, gd, V.dofmap.list, Q.dofmap.list, V.tabulate_dof_coordinates(),
                    Q.tabulate_dof_coordinates(), 2, bcs_u=[[(bd, f)] for f in tg.components],
                    rtol=krylov["tentative"]["ksp_rtol"], nonzero_guess=krylov["tentative"]["ksp_initial_guess_nonzero"],
                    block_rtol=bool(krylov["tentative"].get("b200_block_rtol", False)),
                    extrapolate={"extrapolate": 1, "extrapolate2": 2}.get(krylov["tentative"].get("b200_guess"), 0))
    mg = krylov["pressure"].get("pc_type") == "mg"
    if mg:  # the GPU arm's pressure preconditioner on the CPU arm too
        c.attach_pressure_multigrid(msh)
    xV, xQ = V.tabulate_dof_coordinates().T, Q.tabulate_dof_coordinates().T
    tg.t_u = -DT
    for i, f in enumerate(tg.components):
        c.set(cpu.U2, i, f(xV))
    tg.t_u = 0.0
    for i, f in enumerate(tg.components):
        c.set(cpu.U1, i, f(xV))
    tg.t_p = -DT / 2
    c.set(cpu.P, 0, tg.eval_p(xQ))
    for _ in range(n_warm):  # first-touch page faults and cold caches are not part of a step
        tg.t_u += DT
        c.solve(DT, NU)
    t0 = time.perf_counter()
    all_its = []
    for _ in range(n_steps):
        tg.t_u += DT
        c.solve(DT, NU)
        all_its.append(c.its.tolist())
    sec = (time.perf_counter() - t0) / max(n_steps, 1)
    nnz = [int(cpu.lib().ipcs_cpu_nnz(c.h, k)) for k in range(4)]
    med = [int(np.median([i[j] for i in all_its])) for j in range(3)] if all_its else [0, 0, 0]
    out = {"sec_per_step": sec, "cells": getattr(msh, "num_cells_global", msh.num_cells), "threads": int(cpu.lib().ipcs_cpu_threads()), "its": c.its.tolist(),
           "its_median": med, "bytes_per_step": cpu_step_bytes(c.nV, c.nQ, nnz[0], nnz[1], nnz[3], gd, med, mg),
           "steps_done": n_warm + n_steps}
    if want_fields:
        out["u"] = [c.get(cpu.U, i) for i in range(gd)]
        out["p"] = c.get(cpu.P, 0)
    return out


def cpu_mesh_for(args) -> int:
    """Bounded CPU sample: full IPCS steps on the benchmark mesh itself up to 96^3 (about 9 s per step on 16
    cores); larger meshes are sampled at 96^3 and scaled by the cell count (conservative: pressure
    iterations grow with N)."""
    return args.cpu_mesh if args.cpu_mesh > 0 else min(args.mesh, 96)


def run_reference(args):
    """The reference arm: the CPU restatement of the path (the DOLFINx/PETSc reference cannot be installed here) on ALL
    host cores of the box -- the OpenMP team is set from the CPU affinity mask, not from OMP_NUM_THREADS, which
    torch.distributed.run forces to 1 -- on rank 0 only.  The line declares the steps it EXECUTED."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    hi = host_info()
    n_cpu = cpu_mesh_for(args)
    W, K = max(args.warmup, 0), max(args.steps, 1)
    # keep the whole run within a few minutes (3-7 s per step at 96^3 during the start-up transient): the GPU arm's
    # minimum of 3 warm-up steps, then at most 12 timed steps; the EXECUTED counts are what the line declares
    K_run, W_run = (K, W) if n_cpu < 96 else (min(K, 12), min(W, 3))
    wl = args.workload
    r = cpu_sample(n_cpu, K_run, W_run, wl)
    sec = r["sec_per_step"]
    target_cells = 6 * args.mesh**3 if gdim_of(wl) == 3 else 2 * args.mesh**2
    sps = (1.0 / sec) * r["cells"] / target_cells
    gbs = r["bytes_per_step"] / sec / 1e9
    line = {
        "impl": "reference", "metric": METRIC, "value": sps, "unit": "steps/s", "n_gpus": args.gpus, "steps": K_run,
        "warmup": W_run, "requested": {"steps": K, "warmup": W}, "ms_per_step": 1000.0 / sps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(wl, args.mesh), "mesh": args.mesh, "krylov": krylov_for(wl)},
        "cpu_baseline": {"value": sps, "unit": "steps/s", "cores": r["threads"], "kind": "port",
                         "sample": f"C++/OpenMP restatement (oracle/ipcs_cpu.cpp, same Krylov methods, preconditioners incl. the pressure multigrid, and "
                                   f"initial guesses as the GPU arm), {K_run} full IPCS steps after {W_run} warm-up on a "
                                   f"{n_cpu}^3 box ({sec:.2f} s/step, Krylov its u/p/m median {r['its_median']})"
                                   + ("" if n_cpu == args.mesh else f", scaled by cell count to {args.mesh}^3"),
                         "host": hi, "achieved_GBs": round(gbs, 1),
                         "frac_of_stream_triad": round(gbs / hi["stream_triad_GBs"], 3) if hi.get("stream_triad_GBs") else None},
        "e2e": {"value": sps, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "CPU restatement of the reference algorithm on the host cores; the DOLFINx/PETSc/MUMPS reference itself "
                "cannot be installed in this image (DESIGN.md)",
    }
    print(json.dumps(line))


def workload_name(wl: str, N: int) -> str:
    if wl == "taylor-green-2d":
        return (f"2D Taylor-Green P2-P1 {N}x{N} rectangle [-1,1]^2 (demo/taylor_green.py, BASELINE configs[0]), dt={DT}, nu={NU}, "
                "max_iter=1, rtol=1e-10")
    field = {"taylor-green-rot": "exact 2D vortex rotated out of the x-y plane: 3 live components, per-component rtol",
             "taylor-green-z": "z-extruded exact solution, w = 0, block-relative rtol"}[wl]
    return f"3D Taylor-Green P2-P1 {N}^3 box ({field}), dt={DT}, nu={NU}, max_iter=1, rtol=1e-10"


def reinit_state(solver, tg):
    """ICs of demo/taylor_green.py:167-182 again (u2 = u(-dt), u1 = u(0), p = p(-dt/2)), solution histories forgotten."""
    solver._written(solver._u, solver._u1, solver._u2, solver._p, solver._ps, solver._dp)
    tg.t_u = -DT
    for i, f in enumerate(tg.components):
        solver._u2[i].interpolate(f)
    tg.t_u = 0.0
    for i, f in enumerate(tg.components):
        solver._u1[i].interpolate(f)
        solver._u[i].x.array[:] = 0.0
    tg.t_p = -DT / 2
    solver._p.interpolate(tg.eval_p)
    solver._dp.x.array[:] = 0.0
    solver._flush()
    solver._ctx.reset_time_history()
    solver._ctx.select_bc_step(-1)


def parity_vs_cpu_port(solver, tg, cpu_fields: dict) -> dict:
    """The GPU path against the CPU port at FULL size: same mesh, same ICs, same Krylov options, the same number of
    steps; max-norm difference of every velocity component (relative to the largest component) and of the pressure."""
    n = int(cpu_fields["steps_done"])
    reinit_state(solver, tg)
    for _ in range(n):
        tg.t_u += DT
        tg.t_p += DT
        solver.solve(DT, NU, max_iter=1)
    gd = len(cpu_fields["u"])
    u = [solver._u[i].x.array_ro() for i in range(gd)]
    scale = max(float(np.abs(v).max()) for v in cpu_fields["u"])
    du = max(float(np.abs(u[i] - cpu_fields["u"][i]).max()) for i in range(gd)) / scale
    pg, pc = solver._p.x.array_ro(), cpu_fields["p"]
    dpp = float(np.abs(pg - pc).max()) / float(np.abs(pc).max())
    return {"steps": n, "rel_diff_u_vs_cpu_port": du, "rel_diff_p_vs_cpu_port": dpp}


def parity_small(workload: str, N: int, n_steps: int, device: int) -> dict:
    """The same check on a second, smaller box (48^3) with its own solver and CPU port."""
    from problems import make_mesh, make_solver

    tg = make_field(workload)
    solver = make_solver(make_mesh(gdim_of(workload), N), 2, tg, DT, solver_options=krylov_for(workload), device=device)
    r = cpu_sample(N, n_steps, 0, workload, want_fields=True)
    out = parity_vs_cpu_port(solver, tg, r)
    out["mesh"] = N
    return out


def run_ours(args):
    from oasisx_b200.comm import HostComm
    from problems import make_mesh, make_solver

    comm = HostComm.from_env()
    rank, world = comm.rank, comm.size
    if world != args.gpus and rank == 0:
        print(f"# note: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE", file=sys.stderr)
    device = int(os.environ.get("LOCAL_RANK", "0"))
    wl = args.workload
    krylov = krylov_for(wl)

    N, K, W = args.mesh, args.steps, max(args.warmup, 3)
    t_setup = time.perf_counter()
    tg = make_field(wl)
    gd = gdim_of(wl)
    msh = make_mesh(gd, N, comm if world > 1 else None)
    if args.dof_order != "class":  # coordinate-sorted dofs and slices, as for a mesh without lattice information
        msh._dof_order = args.dof_order  # "sigma": plus SELL-C-sigma's window sort by row length
    solver = make_solver(msh, 2, tg, DT, solver_options=krylov, device=device, low_memory=args.low_memory)
    ctx = solver._ctx
    t_setup = time.perf_counter() - t_setup
    nbc = comm.allreduce(sum(len(d) for d in solver._bc_dofs))
    from oasisx_b200 import _lib as L
    sell = ctx.pattern_sell(L.PAT_VV)

    # ---- device-timed region: state and the BC values of every step already in HBM -------------
    series = bc_series(solver, tg, DT, W + K)
    for i, v in enumerate(series):
        ctx.set_velocity_bc_series(i, v)
    solver._flush()
    for s in range(W):
        ctx.select_bc_step(s)
        ctx.step(DT, NU, 1e-12, 1)
    st0 = ctx.stats()
    sampler = ClockSampler(device)
    sampler.start()
    ctx.synchronize()
    comm.Barrier()
    profile_range = os.environ.get("B200_PROFILE_RANGE") == "1"  # ncu --profile-from-start off: the timed steps only
    if profile_range:
        ctx.profiler_range(True)
    ctx.event_record(0)
    its = []
    stage_ms = np.zeros(4)
    for s in range(K):
        ctx.select_bc_step(W + s)
        ctx.step(DT, NU, 1e-12, 1)
        st = ctx.stats()
        its.append((max(st.its_tentative), st.its_pressure, max(st.its_update)))
        res0 = (st.res0_tentative, st.res0_pressure, st.res0_update)
        stage_ms += [st.ms_assemble_first, st.ms_tentative, st.ms_pressure, st.ms_update]
    ctx.event_record(1)
    ctx.synchronize()
    if profile_range:
        ctx.profiler_range(False)
    ms_total = comm.allreduce(ctx.event_elapsed_ms(0, 1), "max")  # max over ranks of the device time
    comm.Barrier()
    clocks = sampler.stop()
    st1 = ctx.stats()
    launches = comm.allreduce(int(st1.kernel_launches - st0.kernel_launches))
    ms_per_step = ms_total / K
    value = 1000.0 / ms_per_step

    # ---- full-size sanity of the state the timed steps produced (not part of any timing) --------
    # the discrete solution against the analytic Taylor-Green field (nodal interpolant, mass-matrix norm), and the
    # Euclidean norms of the owned entries to 15 digits: equal across 1/2/4/8 ranks up to the summation order
    tg.t_u = (W + K) * DT
    solver._written(solver._u, solver._u1, solver._u2, solver._p, solver._ps, solver._dp)  # ctx.step bypassed the host mirrors
    xV = solver._Vi[0][0].tabulate_dof_coordinates().T
    exact = np.stack([f(xV) for f in tg.components], axis=1)  # blocked [n][gdim] at the time of the last step
    err2 = ctx.l2_diff_sq(L.VEC_U, exact)
    nrm2 = ctx.l2_diff_sq(L.VEC_U, exact * 0.0)
    nVo, nQo = solver._nV_owned, solver._nQ_owned
    su = comm.allreduce(float(sum(np.dot(solver._u[i].x.array_ro()[:nVo], solver._u[i].x.array_ro()[:nVo]) for i in range(gd))))
    sp = comm.allreduce(float(np.dot(solver._p.x.array_ro()[:nQo], solver._p.x.array_ro()[:nQo])))
    checks = {"t_end": tg.t_u, "rel_l2_error_u_vs_exact": float(np.sqrt(err2 / nrm2)),
              "norm_u": float(f"{np.sqrt(su):.15e}"), "norm_p": float(f"{np.sqrt(sp):.15e}")}
    if wl == "taylor-green-z":
        checks["max_abs_w"] = comm.allreduce(float(np.abs(solver._u[2].x.array_ro()).max()), "max")
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {**{f"u{i}": solver._u[i].x.array_ro()[:nVo] for i in range(gd)},
                                         "p": solver._p.x.array_ro()[:nQo]})

    # ---- end to end through the public API: callable BCs on the host, H2D, D2H ------------------
    # the SAME K steps again (state re-initialised, solution histories forgotten, W untimed steps first), so that
    # `e2e` and `value` see the same Krylov iteration counts
    reinit_state(solver, tg)
    for s in range(W):
        tg.t_u += DT
        tg.t_p += DT
        solver.solve(DT, NU, max_iter=1)
    stA = ctx.stats()
    ctx.synchronize()
    comm.Barrier()
    t0 = time.perf_counter()
    e2e_its = []
    for s in range(K):
        tg.t_u += DT
        tg.t_p += DT
        solver.solve(DT, NU, max_iter=1)
        st = ctx.stats()
        e2e_its.append((max(st.its_tentative), st.its_pressure, max(st.its_update)))
    ctx.synchronize()
    e2e_s = comm.allreduce((time.perf_counter() - t0) / K, "max")
    stB = ctx.stats()
    e2e = {"value": 1.0 / e2e_s, "unit": "steps/s",
           "h2d_bytes_per_step": comm.allreduce(int(stB.bytes_h2d - stA.bytes_h2d)) // K,
           "d2h_bytes_per_step": comm.allreduce(int(stB.bytes_d2h - stA.bytes_d2h)) // K,
           "iterations": [int(np.median([i[j] for i in e2e_its])) for j in range(3)]}

    # ---- roofline of the dominant kernel, measured live (rank 0's share of the rows) ------------
    peak, peak_kind = measured_peaks()
    comm.Barrier()
    ms_k, bytes_k = ctx.bench_kernel(3, 20)   # SpMM on the P2xP2 pattern (mass operator), gdim RHS: the kernel the steps ran
    achieved = bytes_k / (ms_k * 1e-3) / 1e9
    ms_a, bytes_a = ctx.bench_kernel(1, 5)
    ms_q, bytes_q = ctx.bench_kernel(2, 50)
    ms_d1, ms_d2 = ctx.bench_kernel(4, 20)[0], ctx.bench_kernel(5, 20)[0]  # the same SpMM with its fused epilogues
    collectives = None
    if world > 1:  # latency of the cross-GPU building blocks, 200 back-to-back launches each (every rank takes part)
        collectives = {"path": "peer memory (CUDA IPC over NVLink)" if ctx.peer_enabled() else "NCCL"}
        for name, kid in (("halo_Q_us", 10), ("halo_V3_us", 11), ("allreduce_3_doubles_us", 12), ("mg_level1_vector_sum_us", 13)):
            try:
                collectives[name] = round(1e3 * ctx.bench_kernel(kid, 200)[0], 2)
            except Exception:
                collectives[name] = None
    comm.Barrier()
    roofline = {"bound": "hbm", "kernel": f"k_spmm<K={gd}> (P2xP2 SELL-32 operator, {gd} right-hand sides)",
                "achieved": achieved, "peak": peak, "peak_kind": peak_kind, "unit": "GB/s", "frac": achieved / peak,
                "traffic": ncu_traffic(N) if world == 1 else None, "ms_per_launch": ms_k, "algorithmic_bytes": bytes_k,
                "other_kernels": {
                    "assemble_first_ms": ms_a, "assemble_first_GBs": bytes_a / (ms_a * 1e-3) / 1e9,
                    "assemble_first_algorithmic_bytes": bytes_a,
                    "spmv_Ap_GBs": bytes_q / (ms_q * 1e-3) / 1e9, "spmv_Ap_ms": ms_q,
                    "spmm_row_scale_1_dot_ms": ms_d1, "spmm_row_scale_2_dots_ms": ms_d2}}
    step_roofline = None
    try:
        if world == 1:
            med = (int(np.median([i[0] for i in its])), int(np.median([i[1] for i in its])), int(np.median([i[2] for i in its])))
            sb = step_algorithmic_bytes(solver._nV_owned, solver._nQ_owned, ctx.pattern_nnz(L.PAT_VV), ctx.pattern_nnz(L.PAT_VQ),
                                        ctx.pattern_nnz(L.PAT_QQ), gd, med, bytes_a, bytes_k, bytes_q)
            gbs = sb["total"] / (ms_per_step * 1e-3) / 1e9
            step_roofline = {"algorithmic_bytes_per_step": sb["total"], "iterations_assumed": list(med), "achieved": gbs, "peak": peak,
                             "unit": "GB/s", "frac": gbs / peak,
                             "stage_frac": {k: sb[k] / (v * 1e-3) / 1e9 / peak for k, v in
                                            zip(["assemble_first", "tentative", "pressure", "update"], (stage_ms / K).tolist()) if v > 0},
                             "note": "whole step and stages against the HBM roofline: algorithmic bytes (SURVEY.md 8d formulas, median "
                                     "iteration counts) / measured time / peak; the pressure stage is latency-bound by construction"}
    except Exception as exc:  # an accounting aid must never cost the bench line
        step_roofline = {"error": repr(exc)}
    halos = int(st1.halo_exchanges - st0.halo_exchanges) // K
    allred = int(st1.allreduces - st0.allreduces) // K
    if rank != 0:
        comm.Barrier()
        return

    # ---- CPU restatement on the host cores, bounded sample (rank 0, N = 1 only), and the parity of the two --------
    cpu = None
    parity_failed = False
    if not args.no_cpu and world == 1:
        try:
            hi = host_info()
            n_cpu = cpu_mesh_for(args)
            n_cpu_steps, n_cpu_warm = (2, 1) if n_cpu < 96 else (3, 3)  # 96^3: steps 4-6 after the GPU arm's 3 warm-up steps
            r = cpu_sample(n_cpu, n_cpu_steps, n_cpu_warm, wl, want_fields=(n_cpu == N))
            sec = r["sec_per_step"]
            sps = (1.0 / sec) * r["cells"] / getattr(msh, "num_cells_global", msh.num_cells)
            gbs = r["bytes_per_step"] / sec / 1e9
            cpu = {"value": sps, "unit": "steps/s", "cores": r["threads"], "kind": "port",
                   "sample": f"C++/OpenMP restatement (oracle/ipcs_cpu.cpp, same Krylov methods, preconditioners incl. the pressure "
                             f"multigrid, and initial guesses as the GPU arm), {n_cpu_steps} full IPCS step(s) after {n_cpu_warm} warm-up on "
                             f"a {n_cpu}^3 box ({sec:.2f} s/step, Krylov its u/p/m {r['its']})"
                             + ("" if n_cpu == N else f", scaled by cell count to {N}^3"),
                   "note": "bounded sample: the CPU steps are the first steps after the warm-up (start-up transient, more Krylov iterations per "
                           "step: see its u/p/m) while `value` averages all timed steps of the GPU run (`iterations`); at equal "
                           "iteration counts the CPU step would be shorter by about the ratio of the velocity iteration counts",
                   "host": hi, "achieved_GBs": round(gbs, 1),
                   "frac_of_stream_triad": round(gbs / hi["stream_triad_GBs"], 3) if hi.get("stream_triad_GBs") else None}
            if n_cpu == N:  # GPU fields against the CPU port's after the same steps, at the benchmark size itself
                checks["parity"] = [dict(parity_vs_cpu_port(solver, tg, r), mesh=N)]
                if N > 48 and not args.no_parity48:
                    checks["parity"].append(parity_small(wl, 48, 6, device))
                worst = max(max(c["rel_diff_u_vs_cpu_port"], c["rel_diff_p_vs_cpu_port"]) for c in checks["parity"])
                checks["rel_diff_u_vs_cpu_port"] = max(c["rel_diff_u_vs_cpu_port"] for c in checks["parity"])
                checks["rel_diff_p_vs_cpu_port"] = max(c["rel_diff_p_vs_cpu_port"] for c in checks["parity"])
                checks["parity_tolerance"] = PARITY_TOL
                parity_failed = not (worst <= PARITY_TOL)
        except Exception as exc:  # the GPU measurements above must not be lost to a failure of the CPU leg
            cpu = {"value": None, "unit": "steps/s", "kind": "port", "error": repr(exc)}

    nV = solver._lp.V.n_global if world > 1 else solver._nV_owned
    nQ = solver._lp.Q.n_global if world > 1 else solver._nQ_owned
    line = {
        "metric": METRIC if gd == 3 else "IPCS steps/s, 2D Taylor-Green P2-P1 rectangle", "value": value, "unit": "steps/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(wl, N), "mesh": N, "cells": getattr(msh, "num_cells_global", msh.num_cells),
                   "dofs": 3 * nV + nQ, "partition": (f"{world} z-slab(s), " + ("peer-memory halo + in-kernel all-reduce (no NCCL call on the data path)"
                                                           if ctx.peer_enabled() else "NCCL halo + all-reduce")) if world > 1 else "single GPU",
                   "l2": "working set per step >> 126 MB L2 (P2xP2 operators alone "
                         f"{3 * 12 * (230 * N**3) / 1e9:.2f} GB over all ranks); no flush needed",
                   "krylov": krylov, "low_memory_version": bool(args.low_memory), "dof_order": args.dof_order,
                   "multigrid": "V(1,1) damped Jacobi 0.85, exact dense solve on the first level <= 5000 dofs",
                   "sell_P2xP2": {"slots": sell, "slice_columns": sell // 32},
                   "setup_s": t_setup},
        "iterations": {"tentative": int(np.median([i[0] for i in its])), "pressure": int(np.median([i[1] for i in its])),
                       "update": int(np.median([i[2] for i in its]))},
        "initial_rel_residual": dict(zip(["tentative", "pressure", "update"], [float(f"{r:.3e}") for r in res0])),
        "stage_ms": dict(zip(["assemble_first", "tentative", "pressure", "update"], (stage_ms / K).round(3).tolist())),
        "nccl_per_step": {"halo_exchanges": halos, "allreduces": allred}, "collectives": collectives,
        "roofline": roofline, "step_roofline": step_roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        "bc_dofs": nbc, "checks": checks,
    }
    print(json.dumps(line), flush=True)
    comm.Barrier()
    if parity_failed:
        raise SystemExit(f"PARITY FAILURE: GPU fields differ from the CPU port by more than {PARITY_TOL} ({checks['parity']})")


HEADLINE = "taylor-green-rot"  # what `--workload taylor-green` (the default) runs: see DESIGN.md section 6


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100, help="timed steps (the reference demo's T/dt = 100, SURVEY.md 8d)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mesh", type=int, default=0, help="cubes per direction (default 96 = BASELINE's metric, 48 = configs[2]; cavity: 128)")
    ap.add_argument("--workload", default="taylor-green",
                    choices=["taylor-green", "taylor-green-rot", "taylor-green-z", "taylor-green-2d", "cavity", "assembly-strategies"],
                    help="taylor-green = BASELINE.json's metric (the line the driver reads) = taylor-green-rot: the exact vortex "
                         "rotated out of the x-y plane, three live components, per-component rtol; taylor-green-z = round 1's "
                         "z-extruded field (w = 0) with the block-relative tolerance; cavity = configs[4]; assembly-strategies = "
                         "configs[1] (demo/assembly_strategies.py)")
    ap.add_argument("--cpu-mesh", type=int, default=0, help="box size of the bounded CPU sample (0: min(mesh, 96))")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity48", action="store_true", help="skip the second (48^3) GPU-vs-CPU-port field comparison")
    ap.add_argument("--weak", action="store_true", help="cavity workload: weak scaling, one mesh^3 block of cubes per GPU (BASELINE configs[4])")
    ap.add_argument("--dof-order", default="class", choices=["class", "generic", "sigma"],
                    help="class: stencil-class dof order of the box provider (32 consecutive rows share a stencil); generic: the "
                         "coordinate sort every other mesh gets (DOLFINx, unstructured): how much of the SpMM roofline fraction is the lattice")
    ap.add_argument("--low-memory", action="store_true", help="options={'low_memory_version': True}: matrix-free element vectors "
                                                               "instead of the 9 rectangular operators (fracstep.py:259)")
    ap.add_argument("--pressure-pc", default="mg", choices=["mg", "jacobi"], help="pressure preconditioner of the GPU arm")
    ap.add_argument("--scalar-ksp", default="auto", choices=["auto", "cg", "chebyshev"],
                    help="mass-solve method (auto = cg; chebyshev is reduction-free but needs ~3x the iterations once the "
                         "initial guesses are good)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the velocity components and the pressure of the last timed step as "
                         "DIR/<name>.npy (float64; a fixed seeded sample of arrays longer than 2^20 entries); one GPU only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload == "assembly-strategies"):
        ap.error("--dump-outputs applies to the time-stepping workloads of --impl ours")
    if args.dump_outputs and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        ap.error("--dump-outputs writes the state of one GPU: run it on a single rank")
    KRYLOV["pressure"]["pc_type"] = args.pressure_pc
    KRYLOV["scalar"]["ksp_type"] = args.scalar_ksp if args.scalar_ksp != "auto" else "cg"
    if args.workload == "taylor-green":
        args.workload = HEADLINE
    if args.mesh <= 0:
        args.mesh = 128 if args.workload == "cavity" else (64 if args.workload == "taylor-green-2d" else 96)
    if args.workload == "cavity":
        if args.impl == "reference":
            raise SystemExit("--impl reference times the Taylor-Green metric; the cavity line carries its own cpu_baseline")
        run_cavity(args)
    elif args.workload == "assembly-strategies":
        run_assembly_strategies(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
