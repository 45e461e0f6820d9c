"""ksp_type gmres on the device (oasisx_b200/csrc/gmres.cuh) against the host restatement tests/gmres_reference.py and
the LU oracle: KSPSolver.solve on the assembled tentative operator, the three-component tentative and mass solves of
the time step, reasons, CGS2, extrapolated guesses, determinism, Projector, and several ranks.

Iteration counts must equal the restatement's.  Rounding in the device's reductions may move the step at which the
estimate crosses the tolerance by one where the restatement's estimate lies within 1e-8 (relative) of it; the tests
allow that difference only after checking the condition."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

import gmres_reference as ref
from oasisx_b200 import _lib as L
from oasisx_b200 import fem
from oasisx_b200.ksp import KSPSolver
from problems import TaylorGreen, make_mesh, make_oracle, make_solver, relerr, vscale

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
CASES = [(2, 8, 2), (3, 4, 2), (2, 8, 1), (3, 3, 1)]
GM = {"ksp_type": "gmres", "pc_type": "jacobi", "ksp_rtol": 1e-12}
LU = {"ksp_type": "preonly", "pc_type": "lu"}


def _csr(mat):
    ip, ix, v = mat.getValuesCSR()
    return sp.csr_matrix((v, ix, ip), shape=mat.getSize())


def _first_operator(gdim, N):
    """A solver after assemble_first of the first Taylor-Green step, its A as scipy CSR and a seeded right-hand side."""
    dt, nu = 0.005, 0.01
    tg = TaylorGreen(nu, gdim)
    s = make_solver(make_mesh(gdim, N), 2, tg, dt)
    tg.t_u = dt
    s.assemble_first(dt, nu)
    A = _csr(s._A)
    b = np.random.default_rng(7).uniform(-1, 1, A.shape[0])
    return s, A, b


# options stay set on a device solver slot: every solve restates the ones a test varies
DEFAULTS = {"pc_type": "jacobi", "ksp_atol": 1e-50, "ksp_max_it": 10000, "ksp_gmres_restart": 30,
            "ksp_gmres_cgs_refinement_type": "refine_never", "ksp_initial_guess_nonzero": False}


def _ksp_solve(s, opts, b, slot=L.SOLVER_TENTATIVE, mat=None, x0=None):
    ksp = KSPSolver(None, {**DEFAULTS, **opts})
    ksp.bind(s._ctx, slot)
    ksp.setOperators(s._A if mat is None else mat)
    V = s._Vi[0][0]
    bf, xf = fem.Function(V), fem.Function(V)
    bf.x.array[:] = b
    if x0 is not None:
        xf.x.array[:] = x0
    reason = ksp.solve(bf.x, xf)
    return reason, xf.x.array.copy()


def _device_its(s, opts, b, guess):
    """The device's iteration count, read through ksp_max_it: the solve converges with the cap at `guess` and not below.
    Returns guess when that holds, guess +- 1 when the count is one off, None otherwise."""
    def ok(cap):
        return cap >= 1 and _ksp_solve(s, dict(opts, ksp_max_it=cap), b)[0] > 0

    for its in (guess, guess + 1, guess - 1):
        if ok(its) and not ok(its - 1):
            return its
    return None


def _check_its(dev, r, k=0):
    assert dev is not None
    if dev != r["its"][k]:
        assert abs(dev - r["its"][k]) == 1 and ref.near_threshold(r, k), (dev, r["its"][k], r["est"][k][-2:], r["tol2"][k])


@pytest.mark.parametrize("gdim,N", [(2, 8), (3, 4)])
def test_kspsolver_gmres_on_the_tentative_operator(gdim, N):
    s, A, b = _first_operator(gdim, N)
    dinv = 1.0 / A.diagonal()
    exact = spla.spsolve(A.tocsc(), b)
    its = {}
    for m in (30, 5):
        opts = dict(GM, ksp_gmres_restart=m)
        reason, x = _ksp_solve(s, opts, b)
        assert reason == 2
        assert np.abs(x - exact).max() <= 1e-9 * np.abs(exact).max()
        r = ref.gmres(A, b, dinv=dinv, rtol=1e-12, restart=m)
        assert r["reasons"] == [2]
        dev = _device_its(s, opts, b, r["its"][0])
        _check_its(dev, r)
        its[m] = r["its"][0]
    assert its[5] != its[30]  # the restart is real


def test_reasons_refinement_and_guess_on_the_tentative_operator():
    s, A, b = _first_operator(2, 8)
    dinv = 1.0 / A.diagonal()
    reason, x = _ksp_solve(s, GM, b)
    assert reason == 2
    bnorm = np.linalg.norm(dinv * b)
    assert _ksp_solve(s, dict(GM, ksp_rtol=1e-30, ksp_atol=1e-6 * bnorm), b)[0] == 3
    reason, x2 = _ksp_solve(s, dict(GM, ksp_max_it=2), b)
    r2 = ref.gmres(A, b, dinv=dinv, rtol=1e-12, maxit=2)
    assert reason == -3 == r2["reasons"][0]
    assert np.abs(x2 - r2["x"]).max() <= 1e-10 * np.abs(r2["x"]).max()  # the capped iterate is the restatement's
    for refine in ("refine_always", "refine_ifneeded"):
        reason, xr = _ksp_solve(s, dict(GM, ksp_gmres_cgs_refinement_type=refine), b)
        assert reason == 2
        assert np.abs(xr - x).max() <= 1e-10 * np.abs(x).max()
    # a nonzero initial guess: started from x0, same solution
    x0 = np.random.default_rng(2).uniform(-1, 1, len(b))
    reason, xg = _ksp_solve(s, dict(GM, ksp_initial_guess_nonzero=True), b, x0=x0)
    rg = ref.gmres(A, b, dinv=dinv, x0=x0, rtol=1e-12)
    assert reason == 2 and np.abs(xg - rg["x"]).max() <= 1e-9 * np.abs(rg["x"]).max()
    # pc_type none
    reason, xn = _ksp_solve(s, dict(GM, pc_type="none"), b)
    assert reason == 2 and np.abs(xn - x).max() <= 1e-9 * np.abs(x).max()


def test_bad_gmres_options_raise():
    s, _, _ = _first_operator(2, 4)
    for opts in ({"ksp_type": "gmres", "ksp_gmres_restart": 0}, {"ksp_type": "gmres", "ksp_gmres_restart": 101},
                 {"ksp_type": "gmres", "ksp_gmres_cgs_refinement_type": "sometimes"}):
        with pytest.raises(Exception):
            KSPSolver(None, opts).bind(s._ctx, L.SOLVER_TENTATIVE)
    with pytest.raises(Exception, match="gmres"):
        KSPSolver(None, {"ksp_type": "gmres"}).bind(s._ctx, L.SOLVER_PRESSURE)


@pytest.mark.parametrize("gdim,N,deg", CASES + [(2, 8, -2)])
def test_time_steps_with_gmres_match_oracle(gdim, N, deg):
    """tentative and scalar solves with GMRES at rtol 1e-12: fields to 1e-8 as tests/test_gpu_parity.py; the first
    tentative solve's per-component iteration counts equal the restatement's.  deg < 0: low_memory_version."""
    low_memory = deg < 0
    deg = abs(deg)
    dt, nu = 0.005, 0.01
    msh = make_mesh(gdim, N)
    tg = TaylorGreen(nu, gdim)
    s = make_solver(msh, deg, tg, dt, solver_options={"tentative": GM, "pressure": LU, "scalar": GM}, low_memory=low_memory)
    o = make_oracle(msh, deg, tg, dt)
    tg.t_u, tg.t_p = 0.0, -dt / 2
    for n in range(3):
        tg.t_u += dt
        tg.t_p += dt
        s.solve(dt, nu, max_iter=1)
        o.solve(dt, nu, max_iter=1)
        if n == 0:
            its = list(s.stats().its_tentative)[:gdim]
            dinv = 1.0 / o.A.diagonal()
            r = ref.gmres(o.A, np.stack(o.rhs1), dinv=dinv, rtol=1e-12)
            bb = [float(np.sum((dinv * v) ** 2)) for v in o.rhs1]
            for k in range(gdim):
                if bb[k] > 1e-20 * max(bb):  # w = 0 of the 3D field: its right-hand side is rounding noise
                    _check_its(its[k], r, k)
        for i in range(gdim):
            assert relerr(s._u[i].x.array_ro(), o.u[i], vscale(o.u)) <= 1e-8, (n, i)
        assert relerr(s._p.x.array_ro(), o.p) <= 1e-8, n


def test_extrapolated_guess_with_gmres_gives_the_zero_guess_fields():
    dt, nu = 0.005, 0.01
    out = []
    for guess in ("none", "extrapolate2"):
        tg = TaylorGreen(nu, 2)
        g = dict(GM, b200_guess=guess)
        s = make_solver(make_mesh(2, 8), 2, tg, dt, solver_options={"tentative": g, "pressure": LU, "scalar": g})
        tg.t_u, tg.t_p = 0.0, -dt / 2
        for _ in range(5):
            tg.t_u += dt
            tg.t_p += dt
            s.solve(dt, nu, max_iter=1)
        out.append(([s._u[i].x.array_ro().copy() for i in range(2)], s._p.x.array_ro().copy()))
    (u0, p0), (u1, p1) = out
    for i in range(2):
        assert relerr(u1[i], u0[i], vscale(u0)) <= 1e-8
    assert relerr(p1, p0) <= 1e-8


def test_gmres_is_deterministic():
    """Two contexts, the same mass matrix (assembled in a fixed order) and right-hand side: bitwise equal solutions."""
    xs = []
    for _ in range(2):
        s = make_solver(make_mesh(3, 4), 2, TaylorGreen(0.01, 3), 0.005)
        b = np.random.default_rng(5).uniform(-1, 1, s._Vi[0][0].num_dofs)
        for _ in range(2):
            reason, x = _ksp_solve(s, dict(GM, ksp_gmres_restart=4), b, slot=L.SOLVER_SCALAR, mat=s._M)
            assert reason == 2
            xs.append(x)
    for x in xs[1:]:
        np.testing.assert_array_equal(x, xs[0])


def test_projector_with_gmres_matches_cg():
    import oasisx_b200 as oasisx
    from oasisx_b200 import mesh as bmesh
    from oasisx_b200.function import grad

    msh = bmesh.create_unit_cube(None, 4, 4, 4)
    V = fem.functionspace(msh, ("Lagrange", 2))
    u = fem.Function(V)
    u.interpolate(lambda x: np.sin(x[0]) * x[1] + x[2] ** 3)
    W = fem.functionspace(msh, ("Lagrange", 1, (3,)))
    Q = fem.functionspace(msh, ("Lagrange", 1))
    for target, src in ((W, grad(u)), (Q, u)):
        res = []
        for opts in (dict(GM, ksp_gmres_restart=10), {"ksp_type": "cg", "pc_type": "jacobi", "ksp_rtol": 1e-12}):
            p = oasisx.Projector(src, target, petsc_options=opts)
            assert p.solve() > 0
            res.append(p.x.x.array.copy())
        assert np.abs(res[0] - res[1]).max() <= 1e-10 * np.abs(res[1]).max()


def _ngpu():
    return L.load_library().b2_device_count()


@pytest.mark.parametrize("nranks,peer", [(2, "1"), (2, "0"), (4, "1")])
def test_gmres_on_several_ranks(nranks, peer):
    if _ngpu() < nranks:
        pytest.skip(f"needs {nranks} GPUs")
    port = 29900 + 10 * nranks + int(peer)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nranks}", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(HERE, "gmres_mr_worker.py"), "8", "3"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, B200_PEER=peer))
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert res.stdout.count("MR_OK") == nranks
