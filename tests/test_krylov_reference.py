"""The host restatements of the device CG, BiCGStab and Chebyshev methods (tests/krylov_reference.py) checked against
properties independent of them: CG's iterate minimises the A-norm error over the Krylov space, Chebyshev's error is
the closed-form Chebyshev polynomial of the preconditioned operator applied to the initial error, BiCGStab's recursive
residual is the true one and its first step is the textbook formula, small hand-built matrices drive the BiCGStab
restart and breakdown branches; and all converge to the sparse direct solution.  tests/test_gpu_krylov.py holds the
device to these restatements."""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla
from numpy.polynomial import chebyshev as npcheb

import krylov_reference as ref
from oasisx_b200 import fem as bfem
from problems import TaylorGreen, make_mesh, make_oracle


def _random_spd(n=60, seed=0):
    rng = np.random.default_rng(seed)
    R = rng.uniform(-1, 1, (n, n))
    A = R @ R.T + np.diag(rng.uniform(0.5, 3.0, n))
    return sp.csr_matrix(A), rng.uniform(-1, 1, n)


def _oracle(gdim=2, N=6, deg=2):
    dt, nu = 0.005, 0.01
    tg = TaylorGreen(nu, gdim)
    o = make_oracle(make_mesh(gdim, N), deg, tg, dt)
    tg.t_u = dt
    o.update_bcs()
    o.assemble_first(dt, nu)
    o.velocity_tentative_assemble()
    return o


@pytest.fixture(scope="module")
def oracle():
    return _oracle()


def _mass(o):
    M = o.M.tocsr()
    return M, np.random.default_rng(3).uniform(-1, 1, M.shape[0])


def _nonsym(o):
    A = o.A.tocsr()
    return A, np.asarray(o.rhs1[0])


def _krylov_basis(DA, z0, j):
    V = [z0]
    for _ in range(j - 1):
        V.append(DA @ V[-1])
    return np.linalg.qr(np.stack(V, axis=1))[0]


@pytest.mark.parametrize("which", ["random", "mass"])
@pytest.mark.parametrize("pc", ["jacobi", "none"])
@pytest.mark.parametrize("j", [1, 2, 3, 6])
def test_cg_iterate_minimises_the_energy_error(oracle, which, pc, j):
    A, b = _random_spd() if which == "random" else _mass(oracle)
    n = len(b)
    dinv = 1.0 / A.diagonal() if pc == "jacobi" else None
    x0 = np.random.default_rng(1).uniform(-1, 1, n)
    out = ref.cg(A, b, dinv=dinv, x0=x0, rtol=1e-30, maxit=j)
    assert out["reasons"] == [-3] and out["its"] == [j]
    d = np.ones(n) if dinv is None else dinv
    Ad = A.toarray()
    exact = np.linalg.solve(Ad, b)
    r0 = b - Ad @ x0
    Q = _krylov_basis(d[:, None] * Ad, d * r0, j)
    best = x0 + Q @ np.linalg.solve(Q.T @ Ad @ Q, Q.T @ r0)

    def energy(x):
        e = x - exact
        return np.sqrt(e @ Ad @ e)

    assert abs(energy(out["x"]) - energy(best)) <= 1e-9 * energy(x0)
    assert np.linalg.norm(out["x"] - best) <= 1e-8 * np.linalg.norm(exact)
    # the recursive residual is the true one
    assert abs(np.sqrt(out["est"][0][-1]) - np.linalg.norm(b - Ad @ out["x"])) <= 1e-10 * np.linalg.norm(r0)


@pytest.mark.parametrize("gdim,deg", [(2, 1), (2, 2), (3, 1), (3, 2)])
def test_chebyshev_error_is_the_chebyshev_polynomial(gdim, deg):
    o = _oracle(gdim, 6 if gdim == 2 else 3, deg)
    M, b = _mass(o)
    lo, hi = bfem.mass_jacobi_bounds(gdim, deg)
    dinv = 1.0 / M.diagonal()
    Md = M.toarray()
    s = np.sqrt(dinv)
    lam, U = np.linalg.eigh(s[:, None] * Md * s[None, :])
    assert lam[0] >= lo * (1 - 1e-12) and lam[-1] <= hi * (1 + 1e-12)  # the element-level bounds hold
    exact = np.linalg.solve(Md, b)
    x0 = np.random.default_rng(4).uniform(-1, 1, len(b))
    theta, delta = 0.5 * (hi + lo), 0.5 * (hi - lo)
    for j in (1, 2, 5, 17, 30):
        out = ref.chebyshev(M, b, lo, hi, dinv=dinv, x0=x0, rtol=1e-30, maxit=j)
        assert out["reasons"] == [-3] and out["its"] == [j]
        c = np.zeros(j + 1)
        c[j] = 1.0
        poly = npcheb.chebval((theta - lam) / delta, c) / npcheb.chebval(theta / delta, c)
        # D^-1 M = D^-1/2 S D^1/2: in the variable D^1/2 e the error is S's polynomial applied to D^1/2 e0
        e0 = (x0 - exact) / s
        ej = s * (U @ (poly * (U.T @ e0)))
        assert np.linalg.norm(out["x"] - exact - ej) <= 1e-11 * np.linalg.norm(x0 - exact), j
    # the check schedule: first at the smallest j with 2 rate^j |r0| <= tol (the Chebyshev bound), then every 4
    out = ref.chebyshev(M, b, lo, hi, dinv=dinv, rtol=1e-10)
    assert out["reasons"] == [2]
    kappa = hi / lo
    rate = (np.sqrt(kappa) - 1) / (np.sqrt(kappa) + 1)
    r0, tol = np.linalg.norm(b), 1e-10 * np.linalg.norm(b)
    j = 1
    while 2 * rate ** j * r0 > tol * (1 + 1e-12):
        j += 1
    assert out["first_check"] == j
    fc = out["checks"][0]
    assert fc == j and out["checks"] == list(range(fc, out["its"][0] + 1, 4))
    assert np.sqrt(out["est"][0][-1]) <= tol
    assert len(out["checks"]) == 1 or out["est"][0][out["checks"][-2] - 1] > tol ** 2


def test_bcgs_residual_and_first_step(oracle):
    A, b = _nonsym(oracle)
    dinv = 1.0 / A.diagonal()
    x0 = np.random.default_rng(5).uniform(-1, 1, len(b))
    for j in (1, 2, 5):
        out = ref.bcgs(A, b, dinv=dinv, x0=x0, rtol=1e-30, maxit=j)
        assert out["reasons"] == [-3] and out["its"] == [j]
        true = dinv * (b - A @ out["x"])
        assert abs(np.sqrt(out["est"][0][-1]) - np.linalg.norm(true)) <= 1e-10 * np.linalg.norm(dinv * b)
        assert np.linalg.norm(out["r"][0] - true) <= 1e-10 * np.linalg.norm(dinv * b)
    # iterate 1 from a zero guess: the textbook step with rhat = r0 = D^-1 b
    r0 = dinv * b
    v = dinv * (A @ r0)
    alpha = (r0 @ r0) / (r0 @ v)
    s = r0 - alpha * v
    t = dinv * (A @ s)
    omega = (t @ s) / (t @ t)
    out = ref.bcgs(A, b, dinv=dinv, rtol=1e-30, maxit=1)
    assert np.linalg.norm(out["x"] - (alpha * r0 + omega * s)) <= 1e-13 * np.linalg.norm(out["x"])
    assert out["alpha"][0][0] == pytest.approx(alpha, rel=1e-13) and out["omega"][0][0] == pytest.approx(omega, rel=1e-13)


def test_bcgs_restart_and_breakdown_branches():
    # rhat . r1 = 0 exactly after the first step (integer data): the restart takes rhat = p = r1 and then converges
    A = sp.csr_matrix(np.array([[-1.0, 2, -1], [-1, -2, -2], [1, -1, 2]]))
    b = np.array([0.0, 2, 0])
    v = A @ b
    alpha = (b @ b) / (b @ v)
    s = b - alpha * v
    t = A @ s
    r1 = s - (t @ s) / (t @ t) * t
    assert abs(b @ r1) <= 1e-15 * (b @ b)
    out = ref.bcgs(A, b, rtol=1e-12)
    assert out["restart"][0][0] and not any(out["restart"][0][1:])
    assert out["beta"][0][0] == 0.0 and out["reasons"] == [2]
    assert np.abs(out["x"] - np.linalg.solve(A.toarray(), b)).max() <= 1e-12
    # t . s = 0 (a zero diagonal entry where s lives): omega = 0 restarts too
    A = sp.csr_matrix(np.array([[1.0, 1], [1, 0]]))
    out = ref.bcgs(A, np.array([1.0, 0]), rtol=1e-12)
    assert out["omega"][0][0] == 0.0 and out["restart"][0][0]
    # skew-symmetric: rhat . v = r0 . A r0 = 0 at once -> KSP_DIVERGED_BREAKDOWN before any step
    A = sp.csr_matrix(np.array([[0.0, 1], [-1, 0]]))
    out = ref.bcgs(A, np.array([1.0, 2]), rtol=1e-12)
    assert out["reasons"] == [-5] and out["its"] == [0]
    # CG: an indefinite matrix gives KSP_DIVERGED_INDEFINITE_PC, p . A p = 0 breakdown
    assert ref.cg(sp.csr_matrix(np.diag([1.0, -3.0])), np.array([1.0, 1.0]))["reasons"] == [-8]
    assert ref.cg(sp.csr_matrix(np.array([[1.0, 0], [0, -1]])), np.array([1.0, 1.0]))["reasons"] == [-5]


METHODS = {
    "cg": lambda A, B, **kw: ref.cg(A, B, **kw),
    "bcgs": lambda A, B, **kw: ref.bcgs(A, B, **kw),
    "chebyshev": lambda A, B, **kw: ref.chebyshev(A, B, *kw.pop("bounds"), **kw),
}


def _system(o, method):
    if method == "bcgs":
        return _nonsym(o)
    return _mass(o)


@pytest.mark.parametrize("method", list(METHODS))
def test_converges_to_the_direct_solution(oracle, method):
    A, b = _system(oracle, method)
    dinv = 1.0 / A.diagonal()
    kw = {"bounds": bfem.mass_jacobi_bounds(2, 2)} if method == "chebyshev" else {}
    exact = spla.spsolve(A.tocsc(), b)
    for guess in (None, np.random.default_rng(6).uniform(-1, 1, len(b))):
        out = METHODS[method](A, b, dinv=dinv, x0=guess, rtol=1e-12, **dict(kw))
        assert out["reasons"] == [2]
        assert np.abs(out["x"] - exact).max() <= 1e-9 * np.abs(exact).max()
    if method != "chebyshev":  # pc_type none
        out = METHODS[method](A, b, rtol=1e-12)
        assert out["reasons"] == [2] and np.abs(out["x"] - exact).max() <= 1e-9 * np.abs(exact).max()


@pytest.mark.parametrize("method", list(METHODS))
def test_several_right_hand_sides_block_tolerance_and_reasons(oracle, method):
    A, b = _system(oracle, method)
    dinv = 1.0 / A.diagonal()
    kw = {"bounds": bfem.mass_jacobi_bounds(2, 2)} if method == "chebyshev" else {}
    run = lambda B, **k: METHODS[method](A, B, dinv=dinv, **dict(kw), **k)  # noqa: E731
    B = np.stack([b, 2 * b[::-1], 1e-4 * np.roll(b, 7)])
    out = run(B, rtol=1e-10)
    for k in range(3):
        if method == "chebyshev":  # one step count for all: component k is the single run capped there
            one = run(B[k], rtol=1e-30, maxit=out["its"][k])
        else:
            one = run(B[k], rtol=1e-10)
        assert out["its"][k] == one["its"][0]
        np.testing.assert_array_equal(out["x"][k], one["x"])
    # block tolerance: relative to the largest right-hand side; the small one needs fewer steps
    blk = run(B, rtol=1e-10, block_rtol=True)
    bb = np.array([np.sum(((dinv if method == "bcgs" else 1.0) * v) ** 2) for v in B])
    np.testing.assert_allclose(blk["tol2"], np.full(3, 1e-20 * bb.max()), rtol=1e-14)
    np.testing.assert_allclose(out["tol2"], 1e-20 * bb, rtol=1e-14)
    if method == "chebyshev":
        assert blk["its"][2] < out["its"][2] or blk["its"][0] == out["its"][0]
    else:
        assert blk["its"][2] < out["its"][2]
    # a dominant atol: KSP_CONVERGED_ATOL (Chebyshev reports 2 for either tolerance); ksp_max_it: KSP_DIVERGED_ITS
    bn = np.linalg.norm((dinv if method == "bcgs" else 1.0) * b)
    assert run(b, rtol=1e-30, atol=1e-3 * bn)["reasons"] == [2 if method == "chebyshev" else 3]
    capped = run(b, rtol=1e-14, maxit=3)
    assert capped["reasons"] == [-3] and capped["its"] == [3]
    if method == "chebyshev":
        # a lower bound 2x too high: the first check comes too early and fails, the next ones follow every 4 steps;
        # ksp_max_it between two checks ends it with -3
        lo, hi = kw["bounds"]
        full = ref.chebyshev(A, b, 2 * lo, hi, dinv=dinv, rtol=1e-10)
        fc = full["checks"][0]
        assert full["reasons"] == [2] and len(full["checks"]) > 2 and full["checks"] == list(range(fc, full["its"][0] + 1, 4))
        capped = ref.chebyshev(A, b, 2 * lo, hi, dinv=dinv, rtol=1e-10, maxit=fc + 2)
        assert capped["reasons"] == [-3] and capped["its"] == [fc + 2]


def test_nan_component_is_masked(oracle):
    A, b = _mass(oracle)
    dinv = 1.0 / A.diagonal()
    B = np.stack([b, b[::-1]])
    B[1, 5] = np.nan
    for f in (ref.cg, ref.bcgs):
        out = f(A, B, dinv=dinv, rtol=1e-10)
        assert out["reasons"][1] == -9 and out["its"][1] == 0
        one = f(A, B[0], dinv=dinv, rtol=1e-10)
        assert out["its"][0] == one["its"][0] and out["reasons"][0] == 2


class _Recorder:
    def __init__(self, n):
        self.calls, self.n = [], n

    def set_solver_option(self, slot, key, value):
        self.calls.append((slot, key, value))

    def space_size(self, s):
        return self.n

    def space_degree(self, s):
        return 2


@pytest.mark.parametrize("deg", [1, 2])
def test_projector_passes_chebyshev_bounds(monkeypatch, deg):
    from oasisx_b200 import _lib as L
    from oasisx_b200 import fem, function
    from oasisx_b200 import mesh as bmesh

    class _Stop(Exception):
        pass

    def _stop(*a, **k):  # the options are forwarded before the quadrature rule is built: stop there
        raise _Stop

    monkeypatch.setattr(function, "simplex_rule", _stop)
    msh = bmesh.create_unit_square(None, 2, 2)
    V = fem.functionspace(msh, ("Lagrange", deg))
    for given in (None, "0.3,2.5"):
        ctx = _Recorder(V.num_dofs)
        monkeypatch.setattr(function, "_projection_context", lambda space, device: ctx)
        opts = {"ksp_type": "chebyshev", "pc_type": "jacobi"}
        if given:
            opts["ksp_chebyshev_eigenvalues"] = given
        with pytest.raises(_Stop):
            function.Projector(lambda x: x[0], V, petsc_options=opts)
        got = {k: v for _, k, v in ctx.calls}
        lo, hi = bfem.mass_jacobi_bounds(2, deg)
        assert got["ksp_chebyshev_eigenvalues"] == (given or f"{lo!r},{hi!r}")
        assert {s for s, _, _ in ctx.calls} == {L.SOLVER_PROJECTOR}
