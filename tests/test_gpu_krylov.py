"""The device CG, BiCGStab and Chebyshev solves against their host restatements (tests/krylov_reference.py), iterate by
iterate: KSPSolver.solve on M, MQ and the tentative A; the K-component velocity update, tentative solve and Projector;
iteration counts and reasons per component; masking of a NaN component; and, for each method, a plausibly wrong
recurrence that the tolerances reject.  Operators and right-hand sides are read back from the device, so only the
solver is under test.

Iteration counts must equal the restatement's.  Rounding in the device's reductions may move the step at which the
residual crosses the tolerance by one where the restatement's residual lies within 1e-8 (relative) of it; the tests
allow that difference only after checking the condition."""
import numpy as np
import pytest
import scipy.sparse as sp

import krylov_reference as ref
from oasisx_b200 import _lib as L
from oasisx_b200 import fem
from oasisx_b200.ksp import KSPSolver
from problems import TaylorGreen, make_mesh, make_oracle, make_solver, relerr, vscale

pytestmark = pytest.mark.gpu
CASES = [(2, 8, 2), (3, 4, 2), (2, 16, 1), (3, 6, 1)]
LU = {"ksp_type": "preonly", "pc_type": "lu"}
DT, NU = 0.005, 0.01
# options stay set on a device solver slot: every solve restates the ones a test varies
DEFAULTS = {"pc_type": "jacobi", "ksp_rtol": 1e-10, "ksp_atol": 1e-50, "ksp_max_it": 10000,
            "ksp_initial_guess_nonzero": False, "b200_block_rtol": False}


def _csr(mat):
    ip, ix, v = mat.getValuesCSR()
    return sp.csr_matrix((v, ix, ip), shape=mat.getSize())


def _solver(gdim, N, deg, tentative=LU, scalar=LU):
    """A rotational solver (so that MQ is assembled) after assemble_first of the first Taylor-Green step."""
    tg = TaylorGreen(NU, gdim)
    s = make_solver(make_mesh(gdim, N), deg, tg, DT, rotational=True,
                    solver_options={"tentative": tentative, "pressure": LU, "scalar": scalar})
    tg.t_u, tg.t_p = DT, DT / 2
    [[bc.update_bc() for bc in b] for b in s._bcs_u]
    s.assemble_first(DT, NU)
    return s


def _operators(s):
    ctx = s._ctx
    nQ = s._Q.num_dofs
    mq = fem.Function(s._Q)
    ctx.ksp_solve(L.SOLVER_SCALAR, L.MAT_MQ, np.ones(nQ), mq.x.array.copy())  # MQ exists before it is read
    ip, ix = ctx.pattern(L.PAT_QQ, nQ)
    MQ = sp.csr_matrix((ctx.matrix_values(L.MAT_MQ, 0, len(ix)), ix, ip), shape=(nQ, nQ))
    return {"M": (_csr(s._M), L.MAT_M, s._Vi[0][0]), "MQ": (MQ, L.MAT_MQ, s._Q), "A": (_csr(s._A), L.MAT_A, s._Vi[0][0])}


class _Dev:
    """KSPSolver.solve on one device slot and operator."""

    def __init__(self, s, slot, mat, space):
        self.s, self.slot, self.mat, self.space = s, slot, mat, space

    def solve(self, opts, b, x0=None):
        ksp = KSPSolver(None, {**DEFAULTS, **opts})
        ksp.bind(self.s._ctx, self.slot)
        ksp.setOperators(type("Op", (), {"_mat": self.mat})())
        bf, xf = fem.Function(self.space), fem.Function(self.space)
        bf.x.array[:] = b
        if x0 is not None:
            xf.x.array[:] = x0
        return ksp.solve(bf.x, xf), xf.x.array.copy()

    def its(self, opts, b, x0, guess):
        """The device's iteration count through ksp_max_it: converged with the cap at `its` and not below."""
        def ok(cap):
            return cap >= 1 and self.solve(dict(opts, ksp_max_it=cap), b, x0)[0] > 0

        for its in (guess, guess + 1, guess - 1):
            if ok(its) and not ok(its - 1):
                return its
        return None


def _host(method, A, B, dinv, x0, opts, bounds=None):
    kw = dict(dinv=dinv, x0=x0, rtol=opts.get("ksp_rtol", 1e-10), atol=opts.get("ksp_atol", 1e-50),
              maxit=opts.get("ksp_max_it", 10000), block_rtol=bool(opts.get("b200_block_rtol", False)))
    if method == "chebyshev":
        return ref.chebyshev(A, B, *bounds, **kw)
    return getattr(ref, method)(A, B, **kw)


def _rel(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / max(np.abs(np.asarray(b)).max(), 1e-300))


def _check_its(dev, r, k=0, method="cg"):
    assert dev is not None
    if dev != r["its"][k]:
        # Chebyshev reads its residual only at scheduled checks: no rounding allowance
        assert method != "chebyshev" and abs(dev - r["its"][k]) == 1 and ref.near_threshold(r, k), \
            (method, dev, r["its"][k], r["est"][k][-3:], r["tol2"][k])
        print("+-1 allowance used:", method, "component", k, "device", dev, "host", r["its"][k])


def _cg_beta_rr(A, b, dinv, j):
    """CG with beta = r.r / r.r (a plausible slip for r.z / r.z)."""
    x, r = np.zeros_like(b), b.copy()
    p, rr = dinv * r, r @ r
    rz = r @ p
    for _ in range(j):
        q = A @ p
        alpha = rz / (p @ q)
        x, r = x + alpha * p, r - alpha * q
        rr_new = r @ r
        rz = r @ (dinv * r)
        p = dinv * r + rr_new / rr * p
        rr = rr_new
    return x


def _bcgs_no_omega_s(A, b, dinv, j):
    """BiCGStab whose x update forgets the omega s term."""
    r = dinv * b
    x, rhat, p, rho = np.zeros_like(b), r.copy(), r.copy(), r @ r
    for _ in range(j):
        v = dinv * (A @ p)
        alpha = rho / (rhat @ v)
        s = r - alpha * v
        t = dinv * (A @ s)
        omega = (t @ s) / (t @ t)
        x = x + alpha * p
        r = s - omega * t
        rn = rhat @ r
        p = r + (rn / rho) * (alpha / omega) * (p - omega * v)
        rho = rn
    return x


@pytest.mark.parametrize("gdim,N,deg", CASES)
def test_single_solves_match_the_restatement(gdim, N, deg):
    s = _solver(gdim, N, deg)
    ops = _operators(s)
    lo_hi = {"M": fem.mass_jacobi_bounds(gdim, deg), "MQ": fem.mass_jacobi_bounds(gdim, 1)}
    routes = [("cg", "M", L.SOLVER_SCALAR), ("cg", "MQ", L.SOLVER_SCALAR), ("bcgs", "A", L.SOLVER_TENTATIVE),
              ("bcgs", "M", L.SOLVER_SCALAR), ("chebyshev", "M", L.SOLVER_SCALAR), ("chebyshev", "MQ", L.SOLVER_SCALAR)]
    rng = np.random.default_rng(gdim * 100 + N)
    for method, name, slot in routes:
        A, mat, space = ops[name]
        dev = _Dev(s, slot, mat, space)
        n = A.shape[0]
        b = rng.uniform(-1, 1, n)
        for pc in (("jacobi",) if method == "chebyshev" else ("jacobi", "none")):
            dinv = 1.0 / A.diagonal() if pc == "jacobi" else None
            for guess in (None, rng.uniform(-1, 1, n)):
                opts = {"ksp_type": method, "pc_type": pc, "ksp_initial_guess_nonzero": guess is not None}
                bounds = None
                if method == "chebyshev":
                    bounds = lo_hi[name]
                    opts["ksp_chebyshev_eigenvalues"] = f"{bounds[0]!r},{bounds[1]!r}"
                steps, tol = ((1, 2, 3, 8, 17, 30), 1e-12) if method == "chebyshev" else ((1, 2, 3, 8), 1e-10)
                for j in steps:
                    o = dict(opts, ksp_rtol=1e-30, ksp_max_it=j)
                    reason, x = dev.solve(o, b, guess)
                    r = _host(method, A, b, dinv, guess, o, bounds)
                    assert reason == -3 == r["reasons"][0], (method, name, j)
                    assert _rel(x, r["x"]) <= tol, (method, name, pc, j, _rel(x, r["x"]))
                # converged: reason and iteration count.  Without a preconditioner the mass matrices need long runs, over
                # which the rounding of the two implementations drifts apart: those are held to a shorter run
                opts["ksp_rtol"] = 1e-10 if pc == "jacobi" else 1e-6
                reason, x = dev.solve(opts, b, guess)
                r = _host(method, A, b, dinv, guess, opts, bounds)
                assert reason == r["reasons"][0] == 2, (method, name, reason)
                assert _rel(x, r["x"]) <= (1e-8 if pc == "jacobi" else 1e-6), (method, name, pc, _rel(x, r["x"]))
                d_its = dev.its(opts, b, guess, r["its"][0])
                _check_its(d_its, r, 0, method)
                print("single", (gdim, N, deg), method, name, pc, "x0" if guess is not None else "zero", "device", d_its,
                      "host", r["its"][0])
                if method == "bcgs":
                    assert not any(r["restart"][0])  # assembled operators did not reach the restart
        # non-vacuity: the device's third iterate is far from a plausibly wrong recurrence
        dinv = 1.0 / A.diagonal()
        if method == "cg":
            _, x = dev.solve({"ksp_type": "cg", "ksp_rtol": 1e-30, "ksp_max_it": 3}, b)
            assert _rel(x, _cg_beta_rr(A, b, dinv, 3)) > 1e-6
        elif method == "bcgs":
            _, x = dev.solve({"ksp_type": "bcgs", "ksp_rtol": 1e-30, "ksp_max_it": 3}, b)
            assert _rel(x, _bcgs_no_omega_s(A, b, dinv, 3)) > 1e-6
        else:
            lo, hi = lo_hi[name]
            o = {"ksp_type": "chebyshev", "ksp_rtol": 1e-30, "ksp_max_it": 3, "ksp_chebyshev_eigenvalues": f"{lo!r},{hi!r}"}
            _, x = dev.solve(o, b)
            off = ref.chebyshev(A, b, 0.99 * lo, 1.01 * hi, dinv=dinv, rtol=1e-30, maxit=3)
            assert _rel(x, off["x"]) > 1e-6


def _velocity_update(s, U, opts):
    """K = gdim solves with M through the velocity update: b3 = M u (dp = 0), zero guess."""
    ctx = s._ctx
    s._solver_c.updateOptions({**DEFAULTS, **opts})
    for k, u in enumerate(U):
        ctx.set_vector(L.VEC_U, k, u)
    ctx.set_vector(L.VEC_DP, 0, np.zeros(s._Q.num_dofs))
    reasons = ctx.velocity_update(DT)
    n = len(U[0])
    B = np.stack([ctx.get_vector(L.VEC_B3, k, np.empty(n)) for k in range(len(U))])
    X = np.stack([ctx.get_vector(L.VEC_U, k, np.empty(n)) for k in range(len(U))])
    return list(reasons), list(ctx.stats().its_update)[: len(U)], B, X


@pytest.mark.parametrize("gdim,N,deg", CASES[:2])
@pytest.mark.parametrize("method", ["cg", "chebyshev"])
def test_velocity_update_components_match_the_restatement(gdim, N, deg, method):
    s = _solver(gdim, N, deg)
    M = _csr(s._M)
    dinv = 1.0 / M.diagonal()
    n = M.shape[0]
    rng = np.random.default_rng(11)
    scales = [1.0, 1e-4, 0.0][:gdim]
    U = [c * rng.uniform(-1, 1, n) for c in scales]
    bounds = fem.mass_jacobi_bounds(gdim, deg)
    base = {"ksp_type": method}
    if method == "chebyshev":
        base["ksp_chebyshev_eigenvalues"] = f"{bounds[0]!r},{bounds[1]!r}"
    for block in (False, True):
        opts = dict(base, b200_block_rtol=block)
        reasons, its, B, X = _velocity_update(s, U, opts)
        r = _host(method, M, B, dinv, None, opts, bounds)
        assert reasons == list(r["reasons"]), (reasons, r["reasons"])
        for k in range(gdim):
            _check_its(its[k], r, k, method)
            assert _rel(X[k], r["x"][k]) <= 1e-8, (block, k)
        if method == "cg" and block:
            assert its[0] > its[1]  # relative to the largest right-hand side, the small one stops earlier
    # iterates of every component at j steps
    for j in (1, 3, 8):
        opts = dict(base, ksp_rtol=1e-30, ksp_max_it=j)
        reasons, its, B, X = _velocity_update(s, U, opts)
        r = _host(method, M, B, dinv, None, opts, bounds)
        for k in range(gdim):
            assert _rel(X[k], r["x"][k]) <= (1e-12 if method == "chebyshev" else 1e-10), (j, k)


def _tentative(s, B, opts):
    ctx = s._ctx
    s._solver_u.updateOptions({**DEFAULTS, **opts})
    n = B.shape[1]
    for k in range(len(B)):
        ctx.set_vector(L.VEC_RHS1, k, B[k])
    _, reasons = ctx.tentative_solve()
    Bd = np.stack([ctx.get_vector(L.VEC_RHS1, k, np.empty(n)) for k in range(len(B))])  # Dirichlet values applied
    X = np.stack([ctx.get_vector(L.VEC_U, k, np.empty(n)) for k in range(len(B))])
    return list(reasons), list(ctx.stats().its_tentative)[: len(B)], Bd, X


@pytest.mark.parametrize("gdim,N,deg", CASES)
def test_tentative_bcgs_components_match_the_restatement(gdim, N, deg):
    s = _solver(gdim, N, deg)
    A = _csr(s._A)
    dinv = 1.0 / A.diagonal()
    n = A.shape[0]
    rng = np.random.default_rng(13)
    scales = [1.0, 1e-4, 0.0][:gdim]
    B = np.stack([c * rng.uniform(-1, 1, n) for c in scales])
    for block in (False, True):
        opts = {"ksp_type": "bcgs", "b200_block_rtol": block}
        reasons, its, Bd, X = _tentative(s, B, opts)
        r = ref.bcgs(A, Bd, dinv=dinv, rtol=1e-10, block_rtol=block)
        assert reasons == list(r["reasons"])
        for k in range(gdim):
            _check_its(its[k], r, k, "bcgs")
            assert _rel(X[k], r["x"][k]) <= 1e-8
        assert not any(any(x) for x in r["restart"])
        print("tentative bcgs", (gdim, N, deg), "block" if block else "", "device", its, "host", r["its"])
    for j in (1, 2, 3, 8):
        reasons, its, Bd, X = _tentative(s, B, {"ksp_type": "bcgs", "ksp_rtol": 1e-30, "ksp_max_it": j})
        r = ref.bcgs(A, Bd, dinv=dinv, rtol=1e-30, maxit=j)
        assert reasons == list(r["reasons"]) and its == list(r["its"])  # 3D: w's right-hand side is zero (reason 3)
        for k in range(gdim):
            assert _rel(X[k], r["x"][k]) <= 1e-10, (j, k)


def _project(ctx, slot, rhs, opts):
    for k, v in {**DEFAULTS, **opts}.items():
        ctx.set_solver_option(L.SOLVER_PROJECTOR, k, v)
    K, n = rhs.shape
    ctx.project_set_bcs(slot, np.zeros(0, np.int32), np.zeros((K, 0)))
    ctx.project_load_rhs(slot, rhs)
    X, reasons = ctx.project_solve(n, K)
    return list(reasons), ctx.stats().its_projector, X


@pytest.mark.parametrize("method", ["cg", "bcgs"])
def test_nan_component_is_masked(method):
    """A NaN in component 1 gives it reason -9; components 0 and 2 are bitwise those of the solve with b_1 = 0."""
    s = _solver(3, 4, 2)
    n = s._Vi[0][0].num_dofs
    rng = np.random.default_rng(17)
    B = rng.uniform(-1, 1, (3, n))
    Bz = B.copy()
    Bz[1] = 0.0
    Bn = B.copy()
    Bn[1, n // 2] = np.nan
    out = []
    for rhs in (Bn, Bz):
        if method == "cg":
            reasons, _, X = _project(s._ctx, L.SPACE_V, rhs, {"ksp_type": "cg"})
            its = None
        else:
            reasons, its, _, X = _tentative(s, rhs, {"ksp_type": "bcgs"})
        out.append((reasons, its, X))
    (rn, itn, Xn), (rz, itz, Xz) = out
    assert rn[1] == -9 and rn[0] == rz[0] == 2 and rn[2] == rz[2] == 2
    for k in (0, 2):
        np.testing.assert_array_equal(Xn[k], Xz[k])
    if method == "bcgs":
        assert itn[1] == 0 and itn[0] == itz[0] and itn[2] == itz[2]


def _projector_cases():
    import oasisx_b200 as oasisx
    from oasisx_b200 import mesh as bmesh
    from oasisx_b200.function import grad

    msh = bmesh.create_unit_cube(None, 4, 4, 4)
    V = fem.functionspace(msh, ("Lagrange", 2))
    u = fem.Function(V)
    u.interpolate(lambda x: np.sin(x[0]) * x[1] + x[2] ** 3)
    Q = fem.functionspace(msh, ("Lagrange", 1))
    W1 = fem.functionspace(msh, ("Lagrange", 1, (3,)))  # three P1 components in the P2-P1 context: the Q work space
    W2 = fem.functionspace(msh, ("Lagrange", 2, (3,)))
    return oasisx, [("V scalar", V, u), ("Q scalar", Q, u), ("Q x3", W1, grad(u)), ("V x3", W2, grad(u)),
                    ("Q x2", None, [grad(u)[0], grad(u)[1]])], Q


@pytest.mark.parametrize("method", ["cg", "chebyshev"])
def test_projector_matches_the_restatement(method):
    """Projector onto V and Q targets, K = 1..3; for Chebyshev the bounds come from the target's degree."""
    oasisx, cases, Q = _projector_cases()
    from oasisx_b200 import mesh as bmesh

    report = []
    for name, target, src in cases:
        if target is None:  # K = 2: a blocked P1 space of a 2D mesh
            msh2 = bmesh.create_unit_square(None, 8, 8)
            u2 = fem.Function(fem.functionspace(msh2, ("Lagrange", 2)))
            u2.interpolate(lambda x: np.cos(x[0]) * x[1] ** 2)
            from oasisx_b200.function import grad
            target, src = fem.functionspace(msh2, ("Lagrange", 1, (2,))), grad(u2)
        opts = {"ksp_type": method, "pc_type": "jacobi", "ksp_rtol": 1e-10}
        p = oasisx.Projector(src, target, petsc_options=opts)
        ctx, slot = p._ctx, p._slot
        ctx.set_solver_option(L.SOLVER_PROJECTOR, "ksp_atol", 1e-50)
        ctx.set_solver_option(L.SOLVER_PROJECTOR, "ksp_max_it", 10000)
        ctx.set_solver_option(L.SOLVER_PROJECTOR, "b200_block_rtol", False)
        ctx.set_solver_option(L.SOLVER_PROJECTOR, "ksp_initial_guess_nonzero", False)
        reason = p.solve()
        its = ctx.stats().its_projector
        n = target._scalar.num_dofs
        ip, ix = ctx.pattern(L.PAT_VV if slot == L.SPACE_V else L.PAT_QQ, n)
        Mt = sp.csr_matrix((ctx.matrix_values(L.MAT_M if slot == L.SPACE_V else L.MAT_MQ, 0, len(ix)), ix, ip), shape=(n, n))
        bounds = fem.mass_jacobi_bounds(target.mesh.geometry.dim, target.degree)
        r = _host(method, Mt, p._rhs, 1.0 / Mt.diagonal(), None, opts, bounds)
        K = p._rhs.shape[0]
        X = p.x.x.array.reshape(-1, K).T if K > 1 else p.x.x.array[None, :]
        assert reason == min(r["reasons"]) == 2, name
        assert max(_rel(X[k], r["x"][k]) for k in range(K)) <= 1e-8, name
        k_max = int(np.argmax(r["its"]))
        _check_its(its, r, k_max, method)
        report.append((name, its, r["its"]))
        # iterates at j steps, every component
        for j in ((1, 3, 8, 30) if method == "chebyshev" else (1, 3, 8)):
            o = dict(opts, ksp_rtol=1e-30, ksp_max_it=j)
            reasons, _, Xj = _project(ctx, slot, p._rhs, o)
            rj = _host(method, Mt, p._rhs, 1.0 / Mt.diagonal(), None, o, bounds)
            assert reasons == [-3] * K
            assert max(_rel(Xj[k], rj["x"][k]) for k in range(K)) <= (1e-12 if method == "chebyshev" else 1e-10), (name, j)
    print(method, "projector its (device max, host per component):", report)


def test_kspsolver_chebyshev_on_the_projector_slot_and_scalar_slot():
    """ksp_type chebyshev through KSPSolver.solve (caller-supplied work vectors) on the projector and scalar slots."""
    gdim, N, deg = 3, 4, 2
    s = _solver(gdim, N, deg)
    ops = _operators(s)
    rng = np.random.default_rng(19)
    for slot in (L.SOLVER_PROJECTOR, L.SOLVER_SCALAR):
        for name, bdeg in (("M", deg), ("MQ", 1)):
            A, mat, space = ops[name]
            b = rng.uniform(-1, 1, A.shape[0])
            lo, hi = fem.mass_jacobi_bounds(gdim, bdeg)
            opts = {"ksp_type": "chebyshev", "ksp_chebyshev_eigenvalues": f"{lo!r},{hi!r}"}
            reason, x = _Dev(s, slot, mat, space).solve(opts, b)
            r = ref.chebyshev(A, b, lo, hi, dinv=1.0 / A.diagonal(), rtol=1e-10)
            assert reason == 2 and _rel(x, r["x"]) <= 1e-10, (slot, name)


def test_rotational_with_chebyshev_matches_oracle():
    dt, nu = DT, NU
    msh = make_mesh(2, 8)
    tg = TaylorGreen(nu, 2)
    cheb = {"ksp_type": "chebyshev", "pc_type": "jacobi", "ksp_rtol": 1e-12}
    s = make_solver(msh, 2, tg, dt, rotational=True, solver_options={"tentative": LU, "pressure": LU, "scalar": cheb})
    o = make_oracle(msh, 2, tg, dt, rotational=True)
    tg.t_u, tg.t_p = 0.0, -dt / 2
    for n in range(3):
        tg.t_u += dt
        tg.t_p += dt
        s.solve(dt, nu, max_iter=1)
        o.solve(dt, nu, max_iter=1)
        assert relerr(s._p.x.array_ro(), o.p) <= 1e-8
        for i in range(2):
            assert relerr(s._u[i].x.array_ro(), o.u[i], vscale(o.u)) <= 1e-8
        assert s.stats().its_projector > 0
