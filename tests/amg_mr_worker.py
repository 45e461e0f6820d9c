"""Worker of the multi-rank algebraic multigrid test (tests/test_gpu_amg_multirank.py): launched with
torch.distributed.run, one rank per GPU, with the cases to run as arguments:

  partition-jittered / partition-lshape  jittered_mesh(3, 8) / l_shaped_mesh(2, 16) rebuilt as Mesh(x, cells, gdim, comm):
      global ids are the replicated mesh's own dof numbers, so rank 0 builds the single-rank gamg solver of the same
      mesh as the reference: aggregates bit for bit, A_l to 1e-13, rho_l to 1e-12, owned rows of P_1 to 1e-14, pressure
      iterations within 1 of the single-rank run;
  adapter  the jittered mesh through tests/fake_dolfinx.py (DOLFINx numbering): level 1 against tests/amg_reference.py
      on the global Ap gathered on the host from every rank's owned rows;
  iters  jittered_mesh(3, 24): AMG-PCG needs at most a fifth of Jacobi-PCG's iterations on the same ranks.

Every case checks that the hierarchy is algebraic and that no rank fell back to Jacobi, and that every rank holds the
same coarse hierarchy bit for bit; the time-step cases run 3 steps against the LU oracle at the same global dofs."""
import hashlib
import logging
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import scipy.sparse as sp  # noqa: E402

import amg_reference as ref  # noqa: E402
from oasisx_b200 import _lib as L  # noqa: E402
from oasisx_b200 import mesh as bmesh  # noqa: E402
from oasisx_b200.comm import HostComm  # noqa: E402
from problems import (TaylorGreen, boundary_facets, jittered_mesh, l_shaped_mesh, make_oracle, make_solver, relerr,  # noqa: E402
                      vscale)

cases = sys.argv[1:]
comm = HostComm.from_env()
device = int(os.environ.get("LOCAL_RANK", "0"))
dt, nu = 0.005, 0.01
LU = {"ksp_type": "preonly", "pc_type": "lu"}
GAMG = {"ksp_type": "cg", "pc_type": "gamg", "ksp_rtol": 1e-12}
OPTS = {"tentative": LU, "scalar": LU, "pressure": GAMG}

warnings = []


class _Catch(logging.Handler):
    def emit(self, record):
        warnings.append(record.getMessage())


logging.getLogger("oasisx").addHandler(_Catch(level=logging.WARNING))


def on_comm(msh):
    return bmesh.Mesh(msh.geometry.x, msh.geometry.dofmap, msh.geometry.dim, comm)


def csr(mat):
    ip, ix, v = mat.getValuesCSR()
    return sp.csr_matrix((v, ix, ip), shape=mat.getSize())


def rel(a, b):
    return abs(a - b).max() / abs(b).max()


def check_replicated(s):
    """Every rank: the same level info (this rank's own sizes of level 0 and nnz(P_1) left out), the same A_l, P_l, R_l
    and aggregates of the replicated levels, the same omega and rho_hat, bit for bit (sha256 of the bytes)."""
    ctx = s._ctx
    h = hashlib.sha256()
    info0 = ctx.pressure_mg_level_info(0)
    h.update(np.array([info0["omega"], info0["rho_hat"]]).tobytes())
    for l in range(1, s._mg_levels + 1):
        info = ctx.pressure_mg_level_info(l)
        h.update(repr(sorted((k, v) for k, v in info.items() if not (l == 1 and k == "nnz_P"))).encode())
        for w in ((0,) if l == 1 else (0, 1, 2)):
            m = ctx.pressure_mg_get_level(l, w)
            for a in (m.indptr, m.indices, m.data):
                h.update(np.ascontiguousarray(a).tobytes())
        if l >= 2:
            h.update(ctx.pressure_mg_get_level(l, 3).tobytes())
    digests = comm.allgather(h.hexdigest())
    assert all(d == digests[0] for d in digests), digests


def check_level1_local(s):
    """P_1 holds this rank's owned rows, R_1 = P_1^T with local columns, the aggregates of the owned dofs."""
    ctx = s._ctx
    n_owned = s._nQ_owned
    P = ctx.pressure_mg_get_level(1, 1)
    R = ctx.pressure_mg_get_level(1, 2)
    assert P.shape[0] == n_owned and ctx.pressure_mg_get_level(1, 3).shape == (n_owned,)
    Rt = sp.csr_matrix(P.T)
    Rt.sort_indices()
    assert np.array_equal(R.indptr, Rt.indptr) and np.array_equal(R.indices, Rt.indices) and np.array_equal(R.data, Rt.data)


def run_steps(s, msh, owned_map=None, collective=True):
    """3 time steps against the LU oracle.  The solver's local dofs are compared at their global oracle dofs: the
    partition's l2g, all of them when the solver has one rank; owned_map = (V, Q) oracle dofs of the owned dofs when the
    solver's numbering is not the provider's (adapter route)."""
    gd = msh.geometry.dim
    tg2 = TaylorGreen(nu, gd)
    o = make_oracle(msh, 2, tg2, dt)
    tg2.t_u, tg2.t_p = 0.0, -dt / 2
    if owned_map is None:
        everything = np.arange(len(o.p)), np.arange(len(o.u[0]))
        gv, gq = (everything[1], everything[0]) if s._lp is None else (s._lp.V.l2g, s._lp.Q.l2g)
    else:
        gv, gq = owned_map
    worst, its = 0.0, []
    for _ in range(3):
        for t in (s._tg, tg2):
            t.t_u += dt
            t.t_p += dt
        s.solve(dt, nu, max_iter=1)
        o.solve(dt, nu, max_iter=1)
        its.append(s.stats().its_pressure)
        for i in range(gd):
            worst = max(worst, relerr(s._u[i].x.array_ro()[: len(gv)], o.u[i][gv], vscale(o.u)))
        worst = max(worst, relerr(s._p.x.array_ro()[: len(gq)], o.p[gq]))
    return (comm.allreduce(worst, "max") if collective else worst), its


def solver(msh, opts=OPTS, deg=2):
    tg = TaylorGreen(nu, msh.geometry.dim)
    s = make_solver(msh, deg, tg, dt, solver_options=opts, device=device)
    s._tg = tg
    return s


def check_kind(s):
    assert s._mg_kind == "algebraic" and s._mg_levels >= 1, (s._mg_kind, s._mg_levels)
    assert not any("Jacobi" in w for w in warnings), warnings


def ref_hierarchy(msh):
    """Rank 0: the single-rank gamg solver of the same mesh (same device, same process), its hierarchy and its pressure
    iterations over the same 3 steps; broadcast to every rank."""
    out = None
    if comm.rank == 0:
        r = solver(msh)
        ctx = r._ctx
        levels = []
        for l in range(0, r._mg_levels + 1):
            info = ctx.pressure_mg_level_info(l)
            lev = {"rho": info["rho_hat"], "omega": info["omega"]}
            if l >= 1:
                A = ctx.pressure_mg_get_level(l, 0)
                lev["A"] = (A.indptr, A.indices, A.data, A.shape[0])
            if l == 1:
                P = ctx.pressure_mg_get_level(1, 1)
                lev["P"] = (P.indptr, P.indices, P.data, P.shape[1])
                lev["agg"] = ctx.pressure_mg_get_level(1, 3)
            levels.append(lev)
        worst, its = run_steps(r, msh, collective=False)
        assert worst <= 1e-8, worst
        out = {"levels": levels, "its": its}
        ctx.close()
    return comm.bcast(out)


def partition_case(msh):
    s = solver(on_comm(msh))
    check_kind(s)
    check_replicated(s)
    check_level1_local(s)
    R = ref_hierarchy(msh)
    ctx = s._ctx
    rl = R["levels"]
    assert len(rl) == s._mg_levels + 1, (len(rl), s._mg_levels)
    owned = s._lp.Q.l2g[: s._nQ_owned]
    for l, lev in enumerate(rl):
        info = ctx.pressure_mg_level_info(l)
        assert abs(info["rho_hat"] - lev["rho"]) <= 1e-12 * lev["rho"], (l, info["rho_hat"], lev["rho"])
        if l >= 1:
            ip, ix, v, n = lev["A"]
            Aref = sp.csr_matrix((np.asarray(v), np.asarray(ix), np.asarray(ip)), shape=(n, n))
            A = ctx.pressure_mg_get_level(l, 0)
            assert A.shape == Aref.shape and rel(A, Aref) <= 1e-13, l
    ip, ix, v, nc = rl[1]["P"]
    Pref = sp.csr_matrix((np.asarray(v), np.asarray(ix), np.asarray(ip)), shape=(len(ip) - 1, nc))
    np.testing.assert_array_equal(ctx.pressure_mg_get_level(1, 3), np.asarray(rl[1]["agg"])[owned])
    P = ctx.pressure_mg_get_level(1, 1)
    assert abs(P - Pref[owned]).max() <= 1e-14 * abs(Pref).max()
    worst, its = run_steps(s, msh)
    all_its = comm.allgather(its)
    assert all(a == all_its[0] for a in all_its), all_its
    assert all(abs(a - b) <= 1 for a, b in zip(its, R["its"])), (its, R["its"])
    return worst, its, R["its"], s


def adapter_case():
    from fake_dolfinx import make_fake

    import oasisx_b200 as oasisx

    msh = jittered_mesh(3, 8)
    mod, fmesh, plp = make_fake(msh, 2, 1, comm.size, comm.rank)
    fmesh.comm = comm
    sys.modules["dolfinx"] = mod
    tg = TaylorGreen(nu, 3)
    facets = boundary_facets(msh)
    tags = bmesh.meshtags(msh, 2, facets, np.full_like(facets, 3, dtype=np.int32))
    bcs_u = [[oasisx.DirichletBC(f, oasisx.LocatorMethod.TOPOLOGICAL, (tags, np.int32(3)))] for f in tg.components]
    s = oasisx.FractionalStep_AB_CN(fmesh, ("Lagrange", 2), ("Lagrange", 1), bcs_u=bcs_u, bcs_p=[], solver_options=OPTS,
                                    options={"low_memory_version": False}, device=device)
    assert s._foreign
    check_kind(s)
    check_replicated(s)
    check_level1_local(s)
    # the global Ap on the host, from every rank's owned rows in DOLFINx numbering
    lp = s._lp
    no = s._nQ_owned
    A = csr(s._Ap).tocoo()
    parts = comm.allgather((lp.Q.l2g[:no][A.row], lp.Q.l2g[A.col], A.data))
    ng = lp.Q.n_global
    Ag = sp.csr_matrix((np.concatenate([p[2] for p in parts]), (np.concatenate([p[0] for p in parts]),
                                                                 np.concatenate([p[1] for p in parts]))), shape=(ng, ng))
    Ag.sort_indices()
    ctx = s._ctx
    ragg, _ = ref.mis2_aggregate(Ag)
    owned = lp.Q.l2g[:no]
    np.testing.assert_array_equal(ctx.pressure_mg_get_level(1, 3), ragg[owned])
    Pref = ref.smoothed_prolongator(Ag, ragg, ctx.pressure_mg_level_info(0)["omega"])
    P = ctx.pressure_mg_get_level(1, 1)
    assert abs(P - Pref[owned]).max() <= 1e-14 * abs(Pref).max()
    assert rel(ctx.pressure_mg_get_level(1, 0), ref.galerkin(Ag, Pref)) <= 1e-13
    # initial state at the fake local dofs, then 3 steps against the oracle on the owned dofs (provider global ids)
    tg.t_u = -dt
    for i, f in enumerate(tg.components):
        s._u2[i].interpolate(f)
    tg.t_u = 0.0
    for i, f in enumerate(tg.components):
        s._u1[i].interpolate(f)
    tg.t_p = -dt / 2
    s._p.interpolate(tg.eval_p)
    s._tg = tg
    tg.t_u, tg.t_p = 0.0, -dt / 2
    worst, its = run_steps(s, msh, owned_map=(plp.V.l2g[: plp.V.n_owned], plp.Q.l2g[: plp.Q.n_owned]))
    all_its = comm.allgather(its)
    assert all(a == all_its[0] for a in all_its), all_its
    return worst, its, None, s


def iters_case():
    msh = jittered_mesh(3, 24, seed=1)
    pressure = {"ksp_type": "cg", "pc_type": "gamg", "ksp_rtol": 1e-10}
    s = solver(on_comm(msh), {"tentative": LU, "scalar": LU, "pressure": pressure}, deg=1)
    check_kind(s)
    check_replicated(s)
    lp = s._lp
    ng = lp.Q.n_global
    b = np.random.default_rng(24).uniform(-1.0, 1.0, ng)
    b -= b.mean()
    its = {}
    for pc in ("gamg", "jacobi"):
        s._solver_p.updateOptions({"pc_type": pc, "ksp_rtol": 1e-10, "ksp_initial_guess_nonzero": False})
        x = np.zeros(lp.Q.n_local)
        assert s._ctx.ksp_solve(L.SOLVER_PRESSURE, L.MAT_AP, b[lp.Q.l2g], x) > 0
        its[pc] = s.stats().its_pressure
    all_its = comm.allgather(its)
    assert all(a == all_its[0] for a in all_its), all_its
    single = None
    if comm.rank == 0:
        r = solver(msh, {"tentative": LU, "scalar": LU, "pressure": pressure}, deg=1)
        x = np.zeros(ng)
        assert r._ctx.ksp_solve(L.SOLVER_PRESSURE, L.MAT_AP, b, x) > 0
        single = r.stats().its_pressure
        r._ctx.close()
    single = comm.bcast(single)
    print(f"rank {comm.rank}: iterations {its}, single-rank gamg {single}", flush=True)
    assert 5 * its["gamg"] <= its["jacobi"], its
    assert abs(its["gamg"] - single) <= 1, (its, single)
    return 0.0, its, single, s


CASES = {"partition-jittered": lambda: partition_case(jittered_mesh(3, 8)),
         "partition-lshape": lambda: partition_case(l_shaped_mesh(2, 16)),
         "adapter": adapter_case, "iters": iters_case}
for case in cases:
    worst, its, ref_its, s = CASES[case]()
    print(f"rank {comm.rank}/{comm.size} {case}: max rel err {worst:.2e}, pressure its {its} (single rank {ref_its}), "
          f"levels {s._mg_levels}, peer path {'on' if s._ctx.peer_enabled() else 'off'}", flush=True)
    assert worst <= 1e-8, worst
    if os.environ.get("B200_PEER") == "0":
        assert not s._ctx.peer_enabled()
    comm.Barrier()  # no rank still reads a peer's memory
    s._ctx.close()
comm.Barrier()
print("MR_OK", comm.rank, flush=True)
