"""Worker of the multi-rank test of the algebraic multigrid with PressureBCs (tests/test_gpu_amg_pressure_bc_multirank.py):
launched with torch.distributed.run, one rank per GPU, with the routes to run as arguments.  The open channel of
tests/channel_problem.py flows along the last axis, so the outlet lies in the last slab and the other ranks hold no
outlet facet.

  partition  jittered_mesh(3, 8) rebuilt as Mesh(x, cells, gdim, comm);
  slab       the slab-local provider box make_mesh(3, 8, comm);
  adapter    the jittered mesh through tests/fake_dolfinx.py (DOLFINx numbering).

partition and slab: rank 0 builds the single-rank gamg solver of the whole mesh; the owned aggregates (-1 on the
Dirichlet dofs) must match bit for bit, the owned rows of P_1 to 1e-14, A_l to 1e-13.  adapter: level 1 against
tests/amg_mask_reference.py on the global Ap and Dirichlet mask gathered on the host.  Every route: every rank holds the
same replicated levels bit for bit, and two inner-iterated steps stay within 1e-7 of the LU oracle."""
import hashlib
import logging
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import scipy.sparse as sp  # noqa: E402

import amg_mask_reference as ref  # noqa: E402
from channel_problem import GAMG, LU, channel  # noqa: E402
from oasisx_b200 import mesh as bmesh  # noqa: E402
from oasisx_b200.comm import HostComm  # noqa: E402
from problems import jittered_mesh, make_mesh, relerr, vscale  # noqa: E402

comm = HostComm.from_env()
device = int(os.environ.get("LOCAL_RANK", "0"))
OPTS = {"tentative": LU, "pressure": GAMG, "scalar": LU}
warnings = []


class _Catch(logging.Handler):
    def emit(self, record):
        warnings.append(record.getMessage())


logging.getLogger("oasisx").addHandler(_Catch(level=logging.WARNING))


def csr(mat):
    ip, ix, v = mat.getValuesCSR()
    return sp.csr_matrix((v, ix, ip), shape=mat.getSize())


def rel(a, b):
    return abs(a - b).max() / abs(b).max()


def mask_of(s):
    """Dirichlet flags of the owned pressure dofs."""
    m = np.zeros(s._nQ_owned, dtype=bool)
    d = np.unique(np.concatenate([b.bc.dofs for b in s._bcs_p]))
    m[d[d < s._nQ_owned]] = True
    return m


def check_common(s):
    """Algebraic hierarchy, no Jacobi fallback, the same replicated levels on every rank bit for bit, P_1 zero on the
    owned Dirichlet rows and -1 their aggregates, and a rank without outlet dofs."""
    assert s._mg_kind == "algebraic" and s._mg_levels >= 1, (s._mg_kind, s._mg_levels)
    assert not any("Jacobi" in w for w in warnings), warnings
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
    mask = mask_of(s)
    agg = ctx.pressure_mg_get_level(1, 3)
    P = ctx.pressure_mg_get_level(1, 1)
    assert agg.shape == (s._nQ_owned,) and (agg[mask] == -1).all() and (agg[~mask] >= 0).all()
    assert not P[mask].toarray().any()
    R = ctx.pressure_mg_get_level(1, 2)
    Rt = sp.csr_matrix(P.T)
    Rt.sort_indices()
    assert np.array_equal(R.indptr, Rt.indptr) and np.array_equal(R.indices, Rt.indices) and np.array_equal(R.data, Rt.data)
    counts = comm.allgather(int(mask.sum()))
    assert sum(counts) > 0 and (comm.size == 1 or min(counts) == 0), counts
    return mask


def run_steps(s, o, inlet, gv, gq):
    dt, nu = 0.01, 0.5
    worst = 0.0
    mask = mask_of(s)
    for _ in range(2):
        inlet.t += dt
        s.solve(dt, nu, max_iter=2, max_error=1e-30)
        o.solve(dt, nu, max_iter=2, max_error=1e-30)
        assert not s._dp.x.array_ro()[: s._nQ_owned][mask].any()
        for i in range(3):
            worst = max(worst, relerr(s._u[i].x.array_ro()[: len(gv)], o.u[i][gv], vscale(o.u)))
        worst = max(worst, relerr(s._p.x.array_ro()[: len(gq)], o.p[gq]))
    return comm.allreduce(worst, "max")


def single_rank_levels(msh):
    """Rank 0: the hierarchy of the single-rank gamg solver of the whole mesh, broadcast."""
    out = None
    if comm.rank == 0:
        r, _, _ = channel(msh, deg=2, solver_options=OPTS, device=device, axis=2)
        ctx = r._ctx
        out = {"agg": ctx.pressure_mg_get_level(1, 3), "mask": mask_of(r), "A": [], "P": None}
        P = ctx.pressure_mg_get_level(1, 1)
        out["P"] = (P.indptr, P.indices, P.data, P.shape)
        for l in range(1, r._mg_levels + 1):
            A = ctx.pressure_mg_get_level(l, 0)
            out["A"].append((A.indptr, A.indices, A.data, A.shape))
        ctx.close()
    return comm.bcast(out)


def global_route(msh, smsh):
    s, o, inlet = channel(smsh, deg=2, solver_options=OPTS, device=device, axis=2, oracle=msh)
    mask = check_common(s)
    R = single_rank_levels(msh)
    ctx = s._ctx
    owned = s._lp.Q.l2g[: s._nQ_owned]
    assert np.array_equal(mask, R["mask"][owned])
    np.testing.assert_array_equal(ctx.pressure_mg_get_level(1, 3), R["agg"][owned])
    ip, ix, v, shape = R["P"]
    Pref = sp.csr_matrix((v, ix, ip), shape=shape)
    assert abs(ctx.pressure_mg_get_level(1, 1) - Pref[owned]).max() <= 1e-14 * abs(Pref).max()
    assert len(R["A"]) == s._mg_levels
    for l, (ip, ix, v, shape) in enumerate(R["A"], start=1):
        assert rel(ctx.pressure_mg_get_level(l, 0), sp.csr_matrix((v, ix, ip), shape=shape)) <= 1e-13, l
    return s, run_steps(s, o, inlet, s._lp.V.l2g, s._lp.Q.l2g)


def adapter_route():
    from fake_dolfinx import make_fake

    msh = jittered_mesh(3, 8)
    s, o, inlet = channel(msh, deg=2, solver_options=OPTS, device=device, axis=2, oracle=True, foreign=True, comm=comm)
    assert s._foreign
    check_common(s)
    lp, no = s._lp, s._nQ_owned
    A = csr(s._Ap).tocoo()
    parts = comm.allgather((lp.Q.l2g[:no][A.row], lp.Q.l2g[A.col], A.data, lp.Q.l2g[:no][mask_of(s)]))
    ng = lp.Q.n_global
    Ag = sp.csr_matrix((np.concatenate([p[2] for p in parts]), (np.concatenate([p[0] for p in parts]),
                                                                 np.concatenate([p[1] for p in parts]))), shape=(ng, ng))
    Ag.sort_indices()
    gmask = np.zeros(ng, dtype=bool)
    gmask[np.concatenate([p[3] for p in parts])] = True
    ctx = s._ctx
    ragg, _ = ref.mis2_aggregate(Ag, gmask)
    owned = lp.Q.l2g[:no]
    np.testing.assert_array_equal(ctx.pressure_mg_get_level(1, 3), ragg[owned])
    Pref = ref.smoothed_prolongator(Ag, ragg, ctx.pressure_mg_level_info(0)["omega"])
    assert abs(ctx.pressure_mg_get_level(1, 1) - Pref[owned]).max() <= 1e-14 * abs(Pref).max()
    assert rel(ctx.pressure_mg_get_level(1, 0), ref.galerkin(Ag, Pref)) <= 1e-13
    plp = make_fake(msh, 2, 1, comm.size, comm.rank)[2]
    return s, run_steps(s, o, inlet, plp.V.l2g[: plp.V.n_owned], plp.Q.l2g[: plp.Q.n_owned])


def partition():
    msh = jittered_mesh(3, 8)
    return global_route(msh, bmesh.Mesh(msh.geometry.x, msh.geometry.dofmap, 3, comm))


ROUTES = {"partition": partition, "slab": lambda: global_route(make_mesh(3, 8), make_mesh(3, 8, comm)),
          "adapter": adapter_route}
for route in sys.argv[1:]:
    s, worst = ROUTES[route]()
    print(f"rank {comm.rank}/{comm.size} {route}: max rel err {worst:.2e}, levels {s._mg_levels}, outlet dofs "
          f"{int(mask_of(s).sum())}, pressure its {s.stats().its_pressure}, "
          f"peer path {'on' if s._ctx.peer_enabled() else 'off'}", flush=True)
    assert worst <= 1e-7, worst
    if os.environ.get("B200_PEER") == "0":
        assert not s._ctx.peer_enabled()
    comm.Barrier()
    s._ctx.close()
comm.Barrier()
print("MR_OK", comm.rank, flush=True)
