"""Worker of the multi-rank GMRES test (tests/test_gpu_gmres.py): launched with torch.distributed.run, one rank per GPU.
Each rank advances the 3D Taylor-Green problem on its slab with GMRES for the tentative and the mass solves, compares
its local fields with the single-process LU oracle at the same global dofs, and checks that every rank took the same
number of iterations (all ranks must take the same decisions from bitwise equal all-reduced sums)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oasisx_b200.comm import HostComm  # noqa: E402
from problems import TaylorGreen, make_mesh, make_oracle, make_solver, relerr, vscale  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 8
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
comm = HostComm.from_env()
dt, nu = 0.005, 0.01
gm = {"ksp_type": "gmres", "pc_type": "jacobi", "ksp_rtol": 1e-11, "ksp_gmres_restart": 6}
opts = {"tentative": gm, "pressure": {"ksp_type": "cg", "pc_type": "jacobi", "ksp_rtol": 1e-11}, "scalar": gm}
tg, tg2 = TaylorGreen(nu, 3), TaylorGreen(nu, 3)
s = make_solver(make_mesh(3, N, comm), 2, tg, dt, solver_options=opts, device=int(os.environ.get("LOCAL_RANK", "0")))
o = make_oracle(make_mesh(3, N), 2, tg2, dt)
lp = s._lp
tg.t_u = tg2.t_u = 0.0
tg.t_p = tg2.t_p = -dt / 2
worst = 0.0
its = []
for n in range(steps):
    for t in (tg, tg2):
        t.t_u += dt
        t.t_p += dt
    s.solve(dt, nu, max_iter=1)
    o.solve(dt, nu, max_iter=1)
    st = s.stats()
    its.append((list(st.its_tentative), list(st.its_update)))
    for i in range(3):
        worst = max(worst, relerr(s._u[i].x.array_ro(), o.u[i][lp.V.l2g], vscale(o.u)))
    worst = max(worst, relerr(s._p.x.array_ro(), o.p[lp.Q.l2g]))
worst = comm.allreduce(worst, "max")
all_its = comm.allgather(its)
print(f"rank {comm.rank}/{comm.size}: max rel err {worst:.2e} peer path {'on' if s._ctx.peer_enabled() else 'off'} "
      f"its (tentative, update) per step {its}", flush=True)
assert worst <= 1e-7, worst
assert all(a == all_its[0] for a in all_its), all_its
assert all(max(t) > 0 for t, _ in its)  # the tentative solves iterated
comm.Barrier()
print("MR_OK", comm.rank, flush=True)
