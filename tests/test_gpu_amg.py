"""The smoothed-aggregation multigrid of the pressure (pc_type gamg / hypre on meshes without a geometric hierarchy):
the device hierarchy against the host reference (tests/amg_reference.py), its smoother damping against scipy's
spectral radius, time steps against the LU oracle and the C++ port, iteration counts against Jacobi-PCG, and the
geometric path unchanged."""
import copy
import sys

import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.linalg import eigsh

import amg_reference as ref
import oasisx_b200 as oasisx
from oasisx_b200 import _lib as L
from problems import (TaylorGreen, boundary_facets, jittered_mesh, l_shaped_mesh, make_cpu_port, make_mesh, make_oracle,
                      make_solver, relerr, vscale)

pytestmark = pytest.mark.gpu

LU = {"ksp_type": "preonly", "pc_type": "lu"}
GAMG = {"ksp_type": "cg", "pc_type": "gamg", "ksp_rtol": 1e-12}
REF_MESHES = {"jittered3d_8": lambda: jittered_mesh(3, 8), "jittered3d_16": lambda: jittered_mesh(3, 16),
              "lshape2d_16": lambda: l_shaped_mesh(2, 16)}


def _csr(mat):
    ip, ix, v = mat.getValuesCSR()
    return sp.csr_matrix((v, ix, ip), shape=mat.getSize())


def _gamg_solver(msh, deg=1, pressure=GAMG):
    tg = TaylorGreen(0.01, msh.geometry.dim)
    return make_solver(msh, deg, tg, 0.005, solver_options={"tentative": LU, "scalar": LU, "pressure": pressure})


def _hierarchy(s):
    ctx = s._ctx
    out = []
    for l in range(1, s._mg_levels + 1):
        out.append((ctx.pressure_mg_level_info(l - 1), ctx.pressure_mg_level_info(l), ctx.pressure_mg_get_level(l, 3),
                    *(ctx.pressure_mg_get_level(l, w) for w in (0, 1, 2))))
    return out


def _rel(a, b):
    return abs(a - b).max() / abs(b).max()


@pytest.mark.parametrize("name", list(REF_MESHES))
def test_hierarchy_equals_the_reference(name):
    s = _gamg_solver(REF_MESHES[name]())
    assert s._mg_kind == "algebraic" and s._mg_levels >= 1
    A = _csr(s._Ap)
    levels = _hierarchy(s)
    for l, (info_f, info, agg, Ac, P, R) in enumerate(levels, start=1):
        assert info["algebraic"] == 1 and info["n"] == Ac.shape[0] == P.shape[1]
        ragg, roots = ref.mis2_aggregate(A)
        np.testing.assert_array_equal(agg, ragg, err_msg=f"aggregates of level {l}")
        assert _rel(P, ref.smoothed_prolongator(A, ragg, info_f["omega"])) <= 1e-14, l
        Rt = sp.csr_matrix(P.T)
        Rt.sort_indices()
        assert np.array_equal(R.indptr, Rt.indptr) and np.array_equal(R.indices, Rt.indices) and np.array_equal(R.data, Rt.data)
        assert all(np.all(np.diff(Ac.indices[Ac.indptr[i]:Ac.indptr[i + 1]]) > 0) for i in range(Ac.shape[0]))
        assert _rel(Ac, sp.csr_matrix(P.T @ (A @ P))) <= 1e-13, l
        A = Ac
    assert levels[-1][1]["dense"] == 1 or s._mg_levels == 15 or 2 * levels[-1][1]["n"] > levels[-1][0]["n"]
    # a second context on the same mesh assembles the same Ap and builds the same hierarchy, bit for bit
    s2 = _gamg_solver(REF_MESHES[name]())
    A0, A0b = _csr(s._Ap), _csr(s2._Ap)
    assert np.array_equal(A0.indices, A0b.indices) and np.array_equal(A0.data.view(np.uint64), A0b.data.view(np.uint64))
    again = _hierarchy(s2)
    for a, b in zip(levels, again):
        assert a[0] == b[0] and a[1] == b[1] and np.array_equal(a[2], b[2])
        for m, n in zip(a[3:], b[3:]):
            assert np.array_equal(m.indptr, n.indptr) and np.array_equal(m.indices, n.indices)
            assert np.array_equal(m.data.view(np.uint64), n.data.view(np.uint64))


@pytest.mark.parametrize("name", list(REF_MESHES))
def test_smoother_damping_is_safe(name):
    """rho_hat (20 power iterations) within [0.9, 1.05] of scipy's largest eigenvalue of D^-1 A on every level, so
    omega_l rho_l = 4 rho_l / (3 rho_hat_l) < 2 with margin."""
    s = _gamg_solver(REF_MESHES[name]())
    A = _csr(s._Ap)
    for l in range(0, s._mg_levels + 1):
        if l:
            A = s._ctx.pressure_mg_get_level(l, 0)
        info = s._ctx.pressure_mg_level_info(l)
        d = 1.0 / np.sqrt(A.diagonal())
        As = sp.diags(d) @ A @ sp.diags(d)
        rho = eigsh(As, k=1, which="LA", return_eigenvectors=False)[0] if A.shape[0] > 50 else np.linalg.eigvalsh(As.toarray())[-1]
        assert 0.9 * rho <= info["rho_hat"] <= 1.05 * rho, (l, info, rho)
        assert info["omega"] * rho < 1.5 and info["omega"] == pytest.approx(4.0 / (3.0 * info["rho_hat"]), rel=1e-15)


@pytest.mark.parametrize("kind,gdim", [("jittered", 3), ("jittered", 2), ("lshape", 3), ("lshape", 2)])
def test_time_steps_match_oracle(kind, gdim):
    dt, nu = 0.005, 0.01
    N = 8 if gdim == 3 else 16
    msh = (jittered_mesh if kind == "jittered" else l_shaped_mesh)(gdim, N, seed=5)
    tg = TaylorGreen(nu, gdim)
    s = make_solver(msh, 2, tg, dt, solver_options={"tentative": LU, "scalar": LU, "pressure": GAMG})
    assert s._mg_kind == "algebraic" and s._mg_levels >= 1
    o = make_oracle(msh, 2, tg, dt)
    tg.t_u, tg.t_p = 0.0, -dt / 2
    for n in range(3):
        tg.t_u += dt
        tg.t_p += dt
        s.solve(dt, nu, max_iter=1)
        o.solve(dt, nu, max_iter=1)
        for i in range(gdim):
            assert relerr(s._u[i].x.array_ro(), o.u[i], vscale(o.u)) <= 1e-8, (n, i)
        assert relerr(s._p.x.array_ro(), o.p) <= 1e-8, n


def test_iterations_are_few_and_mesh_independent():
    """KSPSolver.solve on Ap, seeded mean-free right-hand side, zero guess, rtol 1e-10: AMG-PCG needs at most a fifth
    of Jacobi-PCG's iterations and grows by at most 1.5x from N = 16 to 48.  Measured on one NVIDIA B200 (1000 W
    limit): AMG-PCG 28 / 30 / 30 iterations at N = 16 / 32 / 48, Jacobi-PCG 149 / 261 / 385."""
    its = {}
    for N in (16, 32, 48):
        s = _gamg_solver(jittered_mesh(3, N, seed=1), pressure={"ksp_type": "cg", "pc_type": "gamg", "ksp_rtol": 1e-10})
        assert s._mg_kind == "algebraic"
        n = s._Q.num_dofs
        b = np.random.default_rng(N).uniform(-1.0, 1.0, n)
        b -= b.mean()
        row = {}
        for pc in ("gamg", "jacobi"):
            s._solver_p.updateOptions({"pc_type": pc, "ksp_rtol": 1e-10, "ksp_initial_guess_nonzero": False})
            x = np.zeros(n)
            assert s._ctx.ksp_solve(L.SOLVER_PRESSURE, L.MAT_AP, b, x) > 0
            row[pc] = s.stats().its_pressure
            assert np.linalg.norm(_csr(s._Ap) @ x - b) <= 1e-9 * np.linalg.norm(b)
        its[N] = row
    print("iterations", its)
    for N, row in its.items():
        assert 5 * row["gamg"] <= row["jacobi"], its
    assert its[48]["gamg"] <= 1.5 * its[16]["gamg"], its


def test_graph_replay_at_benchmark_settings():
    """The 17^3 jittered box with the benchmark's solver settings and the pressure on gamg: the captured PCG body
    replays the algebraic V-cycle; 8 steps against the C++ port at rtol 1e-12."""
    import bench
    from oracle import ipcs_cpu as cpu

    dt, nu = 0.005, 0.01
    msh = jittered_mesh(3, 17, seed=7)
    tg, tg2 = TaylorGreen(nu, 3), TaylorGreen(nu, 3)
    opts = copy.deepcopy(bench.KRYLOV)
    opts["pressure"]["pc_type"] = "gamg"
    for o_ in opts.values():
        o_["ksp_rtol"] = 1e-12
    s = make_solver(msh, 2, tg, dt, solver_options=opts)
    assert s._mg_kind == "algebraic" and s._mg_levels >= 1
    c = make_cpu_port(msh, 2, tg2, dt, rtol=1e-12, nonzero_guess=True, block_rtol=True, extrapolate=2)
    for t in (tg, tg2):
        t.t_u, t.t_p = 0.0, -dt / 2
    for n in range(8):
        for t in (tg, tg2):
            t.t_u += dt
            t.t_p += dt
        s.solve(dt, nu, max_iter=1)
        c.solve(dt, nu)
        cu = [c.get(cpu.U, i) for i in range(3)]
        for i in range(3):
            assert relerr(s._u[i].x.array_ro(), cu[i], vscale(cu)) <= 1e-8, (n, i)
        assert relerr(s._p.x.array_ro(), c.get(cpu.P)) <= 1e-8, n
    assert s.stats().its_pressure <= 40


def test_geometric_path_is_untouched():
    """On a provider box gamg takes the geometric hierarchy of pc_type=mg: the same levels, the same P and R bit for bit,
    every level damped with the configured omega, the same pressure iterations, the same fields.  The fields are
    compared to 1e-12, not bitwise: two contexts assemble the velocity operators and assemble_first with atomicAdd,
    so even two pc_type=mg runs differ in the last bits."""
    dt, nu = 0.005, 0.01
    out = {}
    for pc in ("mg", "gamg"):
        tg = TaylorGreen(nu, 3)
        s = make_solver(make_mesh(3, 8), 2, tg, dt, solver_options={"tentative": LU, "scalar": LU,
                                                                     "pressure": dict(GAMG, pc_type=pc)})
        assert s._mg_kind == "geometric" and s._mg_levels >= 2
        ctx = s._ctx
        levels = []
        for l in range(s._mg_levels + 1):
            info = ctx.pressure_mg_level_info(l)
            assert info["algebraic"] == 0 and info["rho_hat"] == 0.0 and info["omega"] == 0.85, (l, info)
            levels.append((info["n"], info["nnz_A"], info["nnz_P"]) if l == 0 else
                          (info["n"], info["nnz_A"], *(ctx.pressure_mg_get_level(l, w) for w in (1, 2))))
        tg.t_u, tg.t_p = 0.0, -dt / 2
        its = []
        for n in range(3):
            tg.t_u += dt
            tg.t_p += dt
            s.solve(dt, nu, max_iter=1)
            its.append(s.stats().its_pressure)
        out[pc] = (levels, its, [s._u[i].x.array_ro().copy() for i in range(3)] + [s._p.x.array_ro().copy()])
    (lm, im, fm), (lg, ig, fg) = out["mg"], out["gamg"]
    assert lm[0] == lg[0] and im == ig
    for a, b in zip(lm[1:], lg[1:]):
        assert a[:2] == b[:2]
        for m, n in zip(a[2:], b[2:]):
            assert np.array_equal(m.indptr, n.indptr) and np.array_equal(m.indices, n.indices)
            assert np.array_equal(m.data.view(np.uint64), n.data.view(np.uint64))
    for a, b in zip(fm, fg):
        assert relerr(b, a, vscale(fm)) <= 1e-12


def test_foreign_mesh_takes_the_algebraic_hierarchy(monkeypatch):
    """A DOLFINx mesh (duck-typed, tests/fake_dolfinx.py) through the adapter with gamg: algebraic hierarchy, oracle
    fields."""
    from fake_dolfinx import make_fake
    from oasisx_b200 import mesh as bmesh

    dt, nu, gdim = 0.005, 0.01, 3
    msh = make_mesh(gdim, 4)
    mod, fmesh, _ = make_fake(msh, 2, 1, 1, 0)
    monkeypatch.setitem(sys.modules, "dolfinx", mod)
    tg, tg2 = TaylorGreen(nu, gdim), TaylorGreen(nu, gdim)
    facets = boundary_facets(msh)
    tags = bmesh.meshtags(msh, gdim - 1, facets, np.full_like(facets, 3, dtype=np.int32))
    bcs_u = [[oasisx.DirichletBC(f, oasisx.LocatorMethod.TOPOLOGICAL, (tags, np.int32(3)))] for f in tg.components]
    s = oasisx.FractionalStep_AB_CN(fmesh, ("Lagrange", 2), ("Lagrange", 1), bcs_u=bcs_u, bcs_p=[],
                                    solver_options={"tentative": LU, "pressure": GAMG, "scalar": LU},
                                    options={"low_memory_version": False})
    assert s._foreign and s._mg_kind == "algebraic" and s._mg_levels >= 1
    o = make_oracle(msh, 2, tg2, dt)
    tg.t_u = -dt
    for i, f in enumerate(tg.components):
        s._u2[i].interpolate(f)
    tg.t_u = 0.0
    for i, f in enumerate(tg.components):
        s._u1[i].interpolate(f)
    tg.t_p = -dt / 2
    s._p.interpolate(tg.eval_p)
    for t in (tg, tg2):
        t.t_u, t.t_p = 0.0, -dt / 2
    for n in range(2):
        for t in (tg, tg2):
            t.t_u += dt
            t.t_p += dt
        s.solve(dt, nu, max_iter=1)
        o.solve(dt, nu, max_iter=1)
    for i in range(gdim):
        assert relerr(s._u[i].x.array_ro(), o.u[i], vscale(o.u)) <= 1e-8
    assert relerr(s._p.x.array_ro(), o.p) <= 1e-8


def test_build_errors_leave_the_context_usable():
    ctx = L.Context()
    with pytest.raises(L.B200Error, match="after b2_preassemble"):
        ctx.pressure_amg_build()
    with pytest.raises(L.B200Error, match="after b2_preassemble"):
        ctx.pressure_mg_level_info(0)
    ctx.close()
    s = _gamg_solver(jittered_mesh(3, 6, seed=4))
    levels = s._mg_levels
    with pytest.raises(L.B200Error, match="already has a multigrid hierarchy"):
        s._ctx.pressure_amg_build()
    assert s._mg_levels == levels and s._ctx.pressure_mg_level_info(levels)["n"] > 0
    s.solve(0.005, 0.01, max_iter=1)
    assert s.stats().its_pressure > 0
