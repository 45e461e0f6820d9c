#!/usr/bin/env python3
"""Pressure solve with the smoothed-aggregation multigrid against Jacobi-PCG and the geometric multigrid.

    python tools/bench_amg.py [--sizes 32 64 96] [--steps 20] [--warmup 3] [--box 96] [--out FILE]
    python -m torch.distributed.run --nproc-per-node=G tools/bench_amg.py --sizes 64 --box 0 [...]   (G ranks)

One JSON line per case, 3D Taylor-Green P2-P1 with the benchmark's solver settings (bench.KRYLOV):
  jittered N^3 meshes (no geometric hierarchy), pressure on the algebraic hierarchy ("gamg") and on Jacobi;
  the N^3 provider box with the algebraic hierarchy forced through the Context API against the geometric one.
The algebraic hierarchy is built on a solver set up with Jacobi (b2_pressure_amg_build, host clock around it ending
in a device synchronise), then the pressure slot is switched to it.  Reported: set-up time, levels (n, nnz), operator
complexity sum nnz(A_l) / nnz(A_0), mean pressure iterations and stage_ms.pressure over the timed steps, steps/s from
device events, and the card's name and power limit read in the same run.

Under torch.distributed.run every rank takes one GPU and its slab of the replicated mesh (oasisx_b200.partition); the
algebraic set-up then passes the global pressure dof ids first and gathers the global Ap on every rank.  Reported:
set-up time, stage_ms.pressure and step time as the maximum over the ranks, operator complexity from the global nnz
of Ap; rank 0 prints.
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
from oasisx_b200 import mesh as bmesh  # noqa: E402
from oasisx_b200.comm import HostComm  # noqa: E402
from problems import TaylorGreen, jittered_mesh, make_mesh, make_solver  # noqa: E402

COMM = HostComm.from_env()


def card() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.splitlines()[0]
    name, power = (v.strip() for v in out.split(","))
    return {"gpu": name, "power_limit": power}


def run_case(msh, label: str, pc: str, steps: int, warmup: int) -> dict:
    """pc: 'jacobi', 'mg' (geometric), or 'amg' (algebraic, built through the Context API)."""
    dt, nu = bench.DT, bench.NU
    comm = COMM
    if comm.size > 1:
        msh = bmesh.Mesh(msh.geometry.x, msh.geometry.dofmap, msh.geometry.dim, comm)
    tg = TaylorGreen(nu, 3)
    opts = copy.deepcopy(bench.KRYLOV)
    opts["pressure"]["pc_type"] = "mg" if pc == "mg" else "jacobi"
    t0 = time.perf_counter()
    s = make_solver(msh, 2, tg, dt, solver_options=opts, device=int(os.environ.get("LOCAL_RANK", "0")))
    ctx = s._ctx
    ctx.synchronize()
    t_solver = comm.allreduce(time.perf_counter() - t0, "max")
    lp = s._lp
    dofs = 3 * s._Vi[0][0].num_dofs + s._Q.num_dofs if lp is None else 3 * lp.V.n_global + lp.Q.n_global
    rec = {"case": label, "pc": pc, "ranks": comm.size, "dofs": dofs, "solver_setup_s": round(t_solver, 3)}
    if pc == "amg":
        comm.Barrier()
        ctx.synchronize()
        t0 = time.perf_counter()
        if comm.size > 1:
            ctx.set_pressure_global_ids(lp.Q.l2g)
        ctx.pressure_amg_build()
        ctx.synchronize()
        rec["amg_setup_s"] = round(comm.allreduce(time.perf_counter() - t0, "max"), 4)
        if comm.size > 1 and ctx.peer_enabled():
            ctx.peer_setup(comm, 1)
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
        levels[0]["n"] = comm.allreduce(levels[0]["n"])  # level 0 is distributed, the coarse levels are replicated
        levels[0]["nnz_A"] = comm.allreduce(levels[0]["nnz_A"])
        rec["levels"] = levels
        rec["operator_complexity"] = round(sum(v["nnz_A"] for v in levels) / levels[0]["nnz_A"], 4)
    tg.t_u, tg.t_p = 0.0, -dt / 2
    for _ in range(warmup):
        tg.t_u += dt
        tg.t_p += dt
        s.solve(dt, nu, max_iter=1)
    ctx.synchronize()
    comm.Barrier()
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
    ms = comm.allreduce(ctx.event_elapsed_ms(0, 1), "max")
    ms_p = comm.allreduce(float(np.mean(ms_p)), "max")
    rec.update({"its_pressure_mean": round(float(np.mean(its)), 2), "its_pressure": its,
                "stage_ms_pressure": round(ms_p, 3), "steps_per_s": round(1000.0 * steps / ms, 3),
                "steps": steps, "warmup": warmup})
    if comm.size > 1:
        rec["peer_path"] = ctx.peer_enabled()
    comm.Barrier()
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
    info = card() if COMM.rank == 0 else {}
    cases = []
    for N in args.sizes:
        msh = jittered_mesh(3, N, seed=1)
        cases += [(msh, f"jittered{N}", pc) for pc in ("amg", "jacobi")]
    if args.box:
        msh = make_mesh(3, args.box)
        cases += [(msh, f"box{args.box}", pc) for pc in ("amg", "mg")]
    for msh, label, pc in cases:
        rec = dict(info, **run_case(msh, label, pc, args.steps, args.warmup))
        if COMM.rank != 0:
            continue
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
