#!/usr/bin/env python3
"""GMRES(m) against the default Krylov methods in the time step.

    python tools/bench_gmres.py [--mesh 96] [--steps 20] [--warmup 5] [--rounds 2] [--out FILE]

3D Taylor-Green P2-P1 box with the rotated field (three live velocity components) and the benchmark's solver settings
(bench.krylov_for("taylor-green-rot")).  Three solvers, timed alternately in one run (`rounds` times each, state
re-initialised before every round):
  base          the benchmark's settings: tentative BiCGStab, mass solve CG;
  tent_gmres    tentative ksp_type gmres (everything else as base);
  scalar_gmres  mass solve ksp_type gmres (everything else as base).
One JSON line per variant: steps/s from device events over the timed steps, per-stage ms (the context's event
timers), per-component iterations per step, norm_u / norm_p after the same number of steps and their difference
from base.  Then one line of kernel times: k_gmres_dots and k_gmres_orth (K = 3) at several Arnoldi indices j, from
torch.profiler over one tentative solve forced to 30 steps (rtol 1e-30, ksp_max_it 30), with their algorithmic bytes
and the share of the HBM bandwidth a device-to-device copy reaches in the same run.  The card's name and power limit
are read in the same run.
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bench  # noqa: E402
from problems import make_mesh, make_solver  # noqa: E402

WL = "taylor-green-rot"
CH = 8  # basis vectors per pass of k_gmres_dots (gmres_solve in b200ipcs.cu)


def card() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.splitlines()[0]
    name, power = (v.strip() for v in out.split(","))
    return {"gpu": name, "power_limit": power}


def copy_bandwidth_gbs() -> float:
    """Device-to-device copy of 4 GiB (read + write), CUDA events, best of 5: the HBM rate a streaming kernel reaches."""
    import torch

    a = torch.empty(1 << 29, dtype=torch.float64, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    best = 1e30
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    return 2 * 8 * (1 << 29) / (best * 1e-3) / 1e9


def variants() -> dict:
    base = bench.krylov_for(WL)
    tent = copy.deepcopy(base)
    tent["tentative"]["ksp_type"] = "gmres"
    scal = copy.deepcopy(base)
    scal["scalar"]["ksp_type"] = "gmres"
    return {"base": base, "tent_gmres": tent, "scalar_gmres": scal}


def run_round(s, tg, steps: int, warmup: int):
    bench.reinit_state(s, tg)
    ctx = s._ctx
    for _ in range(warmup):
        tg.t_u += bench.DT
        tg.t_p += bench.DT
        s.solve(bench.DT, bench.NU, max_iter=1)
    ctx.synchronize()
    ctx.event_record(0)
    its_t, its_m, stage = [], [], np.zeros(4)
    for _ in range(steps):
        tg.t_u += bench.DT
        tg.t_p += bench.DT
        s.solve(bench.DT, bench.NU, max_iter=1)
        st = s.stats()
        its_t.append(list(st.its_tentative))
        its_m.append(list(st.its_update))
        stage += [st.ms_assemble_first, st.ms_tentative, st.ms_pressure, st.ms_update]
    ctx.event_record(1)
    ctx.synchronize()
    ms = ctx.event_elapsed_ms(0, 1)
    u = [s._u[i].x.array_ro() for i in range(3)]
    norm_u = float(np.sqrt(sum(float(v @ v) for v in u)))
    p = s._p.x.array_ro()
    return {"steps_per_s": 1000.0 * steps / ms, "stage_ms": stage / steps, "its_t": its_t, "its_m": its_m,
            "norm_u": norm_u, "norm_p": float(np.sqrt(p @ p))}


def kernel_times(s, n: int, bw_gbs: float, peak_gbs: float) -> dict:
    """One tentative solve forced to 30 Arnoldi steps, traced; the i-th k_gmres_dots / k_gmres_orth launch is step j = i."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    s._solver_u.updateOptions({"ksp_type": "gmres", "ksp_rtol": 1e-30, "ksp_max_it": 30, "ksp_gmres_restart": 30,
                               "b200_guess": "none", "ksp_initial_guess_nonzero": False})
    tg_dt = bench.DT
    s.assemble_first(tg_dt, bench.NU)
    s.velocity_tentative_assemble()
    s.velocity_tentative_solve()  # warm-up of the same shapes
    s._ctx.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _, reasons = s.velocity_tentative_solve()
        s._ctx.synchronize()
    torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if e.device_type.name == "CUDA"), key=lambda e: e.time_range.start)
    dots = [e.time_range.elapsed_us() for e in ev if "k_gmres_dots" in e.name]
    orth = [e.time_range.elapsed_us() for e in ev if "k_gmres_orth" in e.name]
    spmm = [e.time_range.elapsed_us() for e in ev if "k_spmm" in e.name]
    K, vec = 3, 8.0 * 3 * n
    rows = []
    for j in (0, 4, 9, 19, 29):
        if j >= len(dots) or j >= len(orth):
            continue
        bd = vec * ((j + 1) + -(-(j + 1) // CH))  # v_0..v_j once, w once per chunk of CH basis vectors
        bo = vec * ((j + 1) + 2)                  # v_0..v_j, w read and written
        rows.append({"j": j, "dots_us": round(dots[j], 1), "orth_us": round(orth[j], 1),
                     "dots_GBs": round(bd / dots[j] / 1e3, 1), "orth_GBs": round(bo / orth[j] / 1e3, 1),
                     "dots_frac_copy_bw": round(bd / dots[j] / 1e3 / bw_gbs, 3),
                     "orth_frac_copy_bw": round(bo / orth[j] / 1e3 / bw_gbs, 3),
                     "dots_frac_datasheet": round(bd / dots[j] / 1e3 / peak_gbs, 3),
                     "orth_frac_datasheet": round(bo / orth[j] / 1e3 / peak_gbs, 3)})
    return {"kernel_times": rows, "K": K, "arnoldi_steps_traced": len(dots), "reasons": [int(r) for r in reasons],
            "spmm_us_median": round(float(np.median(spmm)), 1) if spmm else None,
            "bytes": "dots 8 K n ((j+1) + ceil((j+1)/8)), orth 8 K n ((j+1) + 2), scale 8 K n 2"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mesh", type=int, default=96)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = card()
    bw = copy_bandwidth_gbs()
    peak = 7700.0
    solvers = {}
    for name, opts in variants().items():
        tg = bench.make_field(WL)
        solvers[name] = (make_solver(make_mesh(3, args.mesh), 2, tg, bench.DT, solver_options=opts), tg)
    res = {name: [] for name in solvers}
    for _ in range(args.rounds):
        for name, (s, tg) in solvers.items():
            res[name].append(run_round(s, tg, args.steps, args.warmup))
    lines = []
    base = res["base"][-1]
    for name, rs in res.items():
        last = rs[-1]
        rec = {"variant": name, "mesh": args.mesh, "workload": bench.workload_name(WL, args.mesh),
               "krylov": {k: variants()[name][k] for k in ("tentative", "scalar")},
               "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds,
               "steps_per_s": round(float(np.mean([r["steps_per_s"] for r in rs])), 3),
               "steps_per_s_rounds": [round(r["steps_per_s"], 3) for r in rs],
               "stage_ms": dict(zip(["assemble_first", "tentative", "pressure", "update"],
                                    np.mean([r["stage_ms"] for r in rs], axis=0).round(3).tolist())),
               "its_tentative_per_step": np.mean(last["its_t"], axis=0).round(2).tolist(),
               "its_update_per_step": np.mean(last["its_m"], axis=0).round(2).tolist(),
               "norm_u": float(f"{last['norm_u']:.15e}"), "norm_p": float(f"{last['norm_p']:.15e}"),
               "rel_diff_norm_u_vs_base": abs(last["norm_u"] - base["norm_u"]) / base["norm_u"],
               "rel_diff_norm_p_vs_base": abs(last["norm_p"] - base["norm_p"]) / base["norm_p"], **info}
        lines.append(rec)
    s, _ = solvers["tent_gmres"]
    kt = kernel_times(s, s._Vi[0][0].num_dofs, bw, peak)
    lines.append({"variant": "kernels", "mesh": args.mesh, "copy_bw_GBs": round(bw, 1), "datasheet_GBs": peak, **kt, **info})
    text = "\n".join(json.dumps(r) for r in lines)
    print(text, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
