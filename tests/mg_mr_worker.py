"""Worker of the multi-rank V-cycle test (tests/test_gpu_mg_vcycle.py): launched with torch.distributed.run, one rank
per GPU.  For every case, the first two PCG iterates of the partitioned pressure solve (pc_type mg / gamg, zero guess,
ksp_max_it 1 and 2) against the host restatement (tests/mg_reference.py) of the single-rank hierarchy of the same
global mesh, owned entries mapped through the partition's l2g:

  partition-16 / partition-36  the replicated provider box (B200_GLOBAL_MESH=1) cut by oasisx_b200.partition;
  slab-16                      the slab-local provider box;
  algebraic-8                  jittered_mesh(3, 8) rebuilt as Mesh(x, cells, gdim, comm), pc_type gamg.

The single-rank solver of the same mesh on the same device supplies the reference hierarchy; its Ap must equal the
partitioned owned rows (to rounding: the slabs sum the element contributions in another order)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import scipy.sparse as sp  # noqa: E402

import mg_reference as ref  # noqa: E402
from oasisx_b200 import _lib as L  # noqa: E402
from oasisx_b200 import mesh as bmesh  # noqa: E402
from oasisx_b200.comm import HostComm  # noqa: E402
from problems import TaylorGreen, jittered_mesh, make_mesh, make_solver  # noqa: E402

comm = HostComm.from_env()
device = int(os.environ.get("LOCAL_RANK", "0"))
LU = {"ksp_type": "preonly", "pc_type": "lu"}
MG = {"ksp_type": "cg", "pc_type": "mg", "ksp_rtol": 1e-12}
CASES = {"partition-16": ("partition", 16), "partition-36": ("partition", 36), "slab-16": ("slab", 16),
         "algebraic-8": ("algebraic", 8)}


def csr(mat):
    ip, ix, v = mat.getValuesCSR()
    return sp.csr_matrix((v, ix, ip), shape=mat.getSize())


def solver(msh, pc):
    return make_solver(msh, 1, TaylorGreen(0.01, 3), 0.005, device=device,
                       solver_options={"tentative": LU, "scalar": LU, "pressure": dict(MG, pc_type=pc)})


def iterate(s, b, k):
    s._solver_p.updateOptions({"ksp_max_it": k, "ksp_rtol": 1e-30, "ksp_initial_guess_nonzero": False})
    x = np.zeros(b.size)
    reason = s._ctx.ksp_solve(L.SOLVER_PRESSURE, L.MAT_AP, b, x)
    assert reason == -3, (k, reason)
    return x


def run(name):
    route, N = CASES[name]
    pc = "gamg" if route == "algebraic" else "mg"
    if route == "algebraic":
        g = jittered_mesh(3, N)
        msh = bmesh.Mesh(g.geometry.x, g.geometry.dofmap, 3, comm)
        glob = jittered_mesh(3, N)
    else:
        os.environ["B200_GLOBAL_MESH"] = "1" if route == "partition" else "0"
        msh = make_mesh(3, N, comm)
        glob = make_mesh(3, N)
    assert hasattr(msh, "is_global_boundary") == (route == "slab"), route
    s = solver(msh, pc)
    assert s._lp is not None and s._mg_kind == ("algebraic" if route == "algebraic" else "geometric"), (name, s._mg_kind)
    # the single-rank hierarchy of the global problem on this rank's device
    s1 = solver(glob, pc)
    assert s1._mg_kind == s._mg_kind and s1._mg_levels == s._mg_levels
    A0 = csr(s1._Ap)
    V = ref.VCycle.from_context(s1._ctx, A0, s1._mg_levels, 1, 1, 16)
    l2g = np.asarray(s._lp.Q.l2g)
    n_owned = s._nQ_owned
    A_loc = csr(s._Ap)  # owned rows, local columns
    A_glob_rows = sp.csr_matrix(A_loc @ sp.csr_matrix((np.ones(l2g.size), (np.arange(l2g.size), l2g)),
                                                     shape=(l2g.size, A0.shape[0])))
    assert abs(A_glob_rows - A0[l2g[:n_owned]]).max() <= 1e-12 * abs(A0).max(), name
    b = np.random.default_rng(N).uniform(-1.0, 1.0, A0.shape[0])
    b -= b.mean()
    host = ref.pcg(A0, b, V, k=2)[0]
    worst = 0.0
    for k in (1, 2):
        x = iterate(s, b[l2g], k)
        xr = host[k - 1]
        worst = max(worst, abs(x[:n_owned] - xr[l2g[:n_owned]]).max() / abs(xr).max())
    x1_other = ref.pcg(A0, b, V.with_(post=0), k=1)[0][0]  # the tolerance tells one post-sweep fewer apart
    far = abs(iterate(s, b[l2g], 1)[:n_owned] - x1_other[l2g[:n_owned]]).max() / abs(x1_other).max()
    worst, far = comm.allreduce(worst, "max"), comm.allreduce(far, "max")
    print(f"rank {comm.rank}/{comm.size} {name}: levels {s._mg_levels} owned {n_owned} x1, x2 max rel err {worst:.2e}, "
          f"one post-sweep fewer {far:.2e}", flush=True)
    assert worst <= 1e-10, (name, worst)
    assert far > 1e-6, (name, far)


for case in sys.argv[1:] or list(CASES):
    run(case)
comm.Barrier()
print("MR_OK", comm.rank, flush=True)
