"""The host restatement of the device GMRES (tests/gmres_reference.py): after j steps without a restart its iterate
minimises the preconditioned residual over x0 + K_j, it converges to the sparse direct solution with and without
restarts, ksp_max_it ends it with KSP_DIVERGED_ITS; and the Python layer forwards the GMRES options to the device
context.  tests/test_gpu_gmres.py holds the device to this restatement."""
import logging

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

import gmres_reference as ref
from problems import TaylorGreen, make_mesh, make_oracle


def _random_system(n=80, seed=0):
    rng = np.random.default_rng(seed)
    A = sp.random(n, n, density=0.08, random_state=rng, format="csr")
    A = A + sp.diags(np.abs(A).sum(axis=1).A1 + 1.0 + rng.uniform(0, 2, n))  # nonsymmetric, diagonally dominant
    return A.tocsr(), rng.uniform(-1, 1, n)


def _tg_system():
    """A of the first 2D P2 Taylor-Green step (8 x 8), Dirichlet rows -> identity, and its right-hand side."""
    dt, nu = 0.005, 0.01
    msh = make_mesh(2, 8)
    tg = TaylorGreen(nu, 2)
    o = make_oracle(msh, 2, tg, dt)
    tg.t_u = dt
    o.update_bcs()
    o.assemble_first(dt, nu)
    o.velocity_tentative_assemble()
    return o.A.tocsr(), np.asarray(o.rhs1[0])


SYSTEMS = {"random": _random_system, "taylor_green_p2": _tg_system}


@pytest.fixture(scope="module", params=list(SYSTEMS))
def system(request):
    A, b = SYSTEMS[request.param]()
    assert abs(A - A.T).max() > 1e-3 * abs(A).max()  # the methods are meant for nonsymmetric matrices
    return A, b, 1.0 / A.diagonal()


@pytest.mark.parametrize("j", [1, 3, 8])
@pytest.mark.parametrize("guess", [False, True])
def test_iterate_minimises_the_preconditioned_residual(system, j, guess):
    A, b, dinv = system
    n = len(b)
    x0 = np.random.default_rng(1).uniform(-1, 1, n) if guess else np.zeros(n)
    out = ref.gmres(A, b, dinv=dinv, x0=x0 if guess else None, rtol=1e-30, maxit=j, restart=30)
    assert out["reasons"] == [-3] and out["its"] == [j]
    # dense least squares over the Krylov space of D^-1 A with r0 = D^-1 (b - A x0)
    DA = (sp.diags(dinv) @ A).toarray()
    r0 = dinv * (b - A @ x0)
    Kry = [r0]
    for _ in range(j - 1):
        Kry.append(DA @ Kry[-1])
    Q, _ = np.linalg.qr(np.stack(Kry, axis=1))
    c, *_ = np.linalg.lstsq(DA @ Q, r0, rcond=None)
    best = np.linalg.norm(r0 - DA @ Q @ c)
    mine = np.linalg.norm(dinv * (b - A @ out["x"]))
    assert abs(mine - best) <= 1e-9 * np.linalg.norm(r0)
    # the estimate |g_{j+1}| is the true preconditioned residual norm
    assert abs(np.sqrt(out["est"][0][-1]) - mine) <= 1e-9 * np.linalg.norm(r0)


@pytest.mark.parametrize("m", [5, 30])
@pytest.mark.parametrize("cgs2", [False, True])
def test_converges_to_the_direct_solution(system, m, cgs2):
    A, b, dinv = system
    exact = spla.spsolve(A.tocsc(), b)
    out = ref.gmres(A, b, dinv=dinv, rtol=1e-12, restart=m, cgs2=cgs2)
    assert out["reasons"] == [2]
    assert np.abs(out["x"] - exact).max() <= 1e-9 * np.abs(exact).max()


def test_restarts_change_the_iteration_count(system):
    A, b, dinv = system
    its = {m: ref.gmres(A, b, dinv=dinv, rtol=1e-12, restart=m)["its"][0] for m in (5, 30)}
    assert its[5] > its[30]


def test_several_right_hand_sides_and_reasons():
    A, b = _random_system()
    dinv = 1.0 / A.diagonal()
    B = np.stack([b, 2 * b[::-1], 1e-3 * b])
    out = ref.gmres(A, B, dinv=dinv, rtol=1e-10, restart=7)
    for k in range(3):
        one = ref.gmres(A, B[k], dinv=dinv, rtol=1e-10, restart=7)
        assert out["its"][k] == one["its"][0]
        np.testing.assert_array_equal(out["x"][k], one["x"])
    # block tolerance: relative to the largest right-hand side, the small one converges earlier
    blk = ref.gmres(A, B, dinv=dinv, rtol=1e-10, restart=7, block_rtol=True)
    assert blk["its"][2] < out["its"][2]
    # a dominant atol gives KSP_CONVERGED_ATOL, ksp_max_it KSP_DIVERGED_ITS
    assert ref.gmres(A, b, dinv=dinv, rtol=1e-30, atol=1e-3)["reasons"] == [3]
    capped = ref.gmres(A, b, dinv=dinv, rtol=1e-14, maxit=2, restart=30)
    assert capped["reasons"] == [-3] and capped["its"] == [2]
    capped = ref.gmres(A, b, dinv=dinv, rtol=1e-14, maxit=7, restart=3)  # the cap inside the third cycle
    assert capped["reasons"] == [-3] and capped["its"] == [7]


class _Recorder:
    def __init__(self):
        self.calls = []

    def set_solver_option(self, slot, key, value):
        self.calls.append((slot, key, value))


GMRES_OPTS = {"ksp_type": "gmres", "pc_type": "jacobi", "ksp_rtol": 1e-9, "ksp_gmres_restart": 12,
              "ksp_gmres_cgs_refinement_type": "refine_always", "ksp_gmres_modifiedgramschmidt": True}


def test_kspsolver_forwards_the_gmres_options_without_a_warning(caplog):
    from oasisx_b200 import _lib as L
    from oasisx_b200.ksp import KSPSolver

    ctx = _Recorder()
    with caplog.at_level(logging.DEBUG, logger="oasisx"):
        KSPSolver(None, GMRES_OPTS, prefix="tentative_velocity").bind(ctx, L.SOLVER_TENTATIVE)
    assert not [r for r in caplog.records if r.levelno >= logging.WARNING]
    got = {k: v for _, k, v in ctx.calls}
    assert got == {k: v for k, v in GMRES_OPTS.items() if k != "ksp_gmres_modifiedgramschmidt"}  # MGS: not built
    assert {s for s, _, _ in ctx.calls} == {L.SOLVER_TENTATIVE}


def test_projector_forwards_the_gmres_options(monkeypatch):
    from oasisx_b200 import _lib as L
    from oasisx_b200 import fem, function
    from oasisx_b200 import mesh as bmesh

    class _Stop(Exception):
        pass

    class _Ctx(_Recorder):
        def space_size(self, s):
            return V.num_dofs if s == L.SPACE_V else -1

        def space_degree(self, s):
            return 2

    def _stop(*a, **k):  # the options are forwarded before the quadrature rule is built: stop there
        raise _Stop

    msh = bmesh.create_unit_square(None, 2, 2)
    V = fem.functionspace(msh, ("Lagrange", 2))
    ctx = _Ctx()
    monkeypatch.setattr(function, "_projection_context", lambda space, device: ctx)
    monkeypatch.setattr(function, "simplex_rule", _stop)
    with pytest.raises(_Stop):
        function.Projector(lambda x: x[0], V, petsc_options=GMRES_OPTS)
    got = {k: v for _, k, v in ctx.calls}
    for k in ("ksp_type", "pc_type", "ksp_rtol", "ksp_gmres_restart", "ksp_gmres_cgs_refinement_type"):
        assert got[k] == GMRES_OPTS[k]
    assert {s for s, _, _ in ctx.calls} == {L.SOLVER_PROJECTOR}
