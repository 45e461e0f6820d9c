#!/usr/bin/env python3
"""Sweep the tile size of the SpMM slice schedule on the GPU.  Usage: python tools/sweep_spmm.py [mesh]"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
from problems import TaylorGreen, make_mesh, make_solver  # noqa: E402
from oasisx_b200 import _lib as L, fem  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 96
dt, nu = 0.005, 0.01
tg = TaylorGreen(nu, 3)
opts = {k: {"ksp_type": t, "pc_type": "jacobi", "ksp_rtol": 1e-10}
        for k, t in (("tentative", "bcgs"), ("pressure", "cg"), ("scalar", "cg"))}
msh = make_mesh(3, N)
s = make_solver(msh, 2, tg, dt, solver_options=opts)
ctx = s._ctx
tg.t_u, tg.t_p = dt, dt / 2
s.solve(dt, nu, max_iter=1)
Vs = s._Vi[0][0]
n_slices = (Vs.num_dofs + 31) // 32
for tile in ((8, 8), (4, 4), (2, 2), (16, 16)):
    ctx.set_slice_order(L.PAT_VV, fem.slice_order(Vs.tabulate_dof_coordinates(), Vs.num_dofs, msh._lattice, tile=tile))
    for kern in (3, 0):
        ms, nbytes = ctx.bench_kernel(kern, 10)
        print(f"tile {tile} kernel {kern}: {ms:.4f} ms  {nbytes / ms / 1e6:7.1f} GB/s", flush=True)
