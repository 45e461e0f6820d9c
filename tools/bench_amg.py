#!/usr/bin/env python3
"""Pressure solve with the smoothed-aggregation multigrid against Jacobi-PCG and the geometric multigrid.

    python tools/bench_amg.py [--sizes 32 64 96] [--steps 20] [--warmup 3] [--box 96] [--out FILE]

One JSON line per case, 3D Taylor-Green P2-P1 with the benchmark's solver settings (bench.KRYLOV):
  jittered N^3 meshes (no geometric hierarchy), pressure on the algebraic hierarchy ("gamg") and on Jacobi;
  the N^3 provider box with the algebraic hierarchy forced through the Context API against the geometric one.
The algebraic hierarchy is built on a solver set up with Jacobi (b2_pressure_amg_build, host clock around it ending
in a device synchronise), then the pressure slot is switched to it.  Reported: set-up time, levels (n, nnz), operator
complexity sum nnz(A_l) / nnz(A_0), mean pressure iterations and stage_ms.pressure over the timed steps, steps/s from
device events, and the card's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bench  # noqa: E402
from problems import TaylorGreen, jittered_mesh, make_mesh, make_solver  # noqa: E402


def card() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.splitlines()[0]
    name, power = (v.strip() for v in out.split(","))
    return {"gpu": name, "power_limit": power}


def run_case(msh, label: str, pc: str, steps: int, warmup: int) -> dict:
    """pc: 'jacobi', 'mg' (geometric), or 'amg' (algebraic, built through the Context API)."""
    dt, nu = bench.DT, bench.NU
    tg = TaylorGreen(nu, 3)
    opts = copy.deepcopy(bench.KRYLOV)
    opts["pressure"]["pc_type"] = "mg" if pc == "mg" else "jacobi"
    t0 = time.perf_counter()
    s = make_solver(msh, 2, tg, dt, solver_options=opts)
    ctx = s._ctx
    ctx.synchronize()
    t_solver = time.perf_counter() - t0
    rec = {"case": label, "pc": pc, "dofs": 3 * s._Vi[0][0].num_dofs + s._Q.num_dofs, "solver_setup_s": round(t_solver, 3)}
    if pc == "amg":
        ctx.synchronize()
        t0 = time.perf_counter()
        ctx.pressure_amg_build()
        ctx.synchronize()
        rec["amg_setup_s"] = round(time.perf_counter() - t0, 4)
        s._solver_p.updateOptions({"pc_type": "gamg"})
    if pc != "jacobi":
        levels, l = [], 0
        while True:
            try:
                info = ctx.pressure_mg_level_info(l)
            except Exception:
                break
            levels.append({k: info[k] for k in ("n", "nnz_A", "dense", "omega", "rho_hat")})
            l += 1
        rec["levels"] = levels
        rec["operator_complexity"] = round(sum(v["nnz_A"] for v in levels) / levels[0]["nnz_A"], 4)
    tg.t_u, tg.t_p = 0.0, -dt / 2
    for _ in range(warmup):
        tg.t_u += dt
        tg.t_p += dt
        s.solve(dt, nu, max_iter=1)
    ctx.synchronize()
    ctx.event_record(0)
    its, ms_p = [], []
    for _ in range(steps):
        tg.t_u += dt
        tg.t_p += dt
        s.solve(dt, nu, max_iter=1)
        st = ctx.stats()
        its.append(st.its_pressure)
        ms_p.append(st.ms_pressure)
    ctx.event_record(1)
    ctx.synchronize()
    ms = ctx.event_elapsed_ms(0, 1)
    rec.update({"its_pressure_mean": round(float(np.mean(its)), 2), "its_pressure": its,
                "stage_ms_pressure": round(float(np.mean(ms_p)), 3), "steps_per_s": round(1000.0 * steps / ms, 3),
                "steps": steps, "warmup": warmup})
    ctx.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="*", default=[32, 64, 96])
    ap.add_argument("--box", type=int, default=96, help="provider box for geometric vs algebraic (0: skip)")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file too")
    args = ap.parse_args()
    info = card()
    cases = []
    for N in args.sizes:
        msh = jittered_mesh(3, N, seed=1)
        cases += [(msh, f"jittered{N}", pc) for pc in ("amg", "jacobi")]
    if args.box:
        msh = make_mesh(3, args.box)
        cases += [(msh, f"box{args.box}", pc) for pc in ("amg", "mg")]
    for msh, label, pc in cases:
        rec = dict(info, **run_case(msh, label, pc, args.steps, args.warmup))
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
