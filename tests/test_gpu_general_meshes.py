"""The CUDA path on meshes that are not uniform boxes (tests/problems.py: `jittered_mesh`, `l_shaped_mesh`,
`mapped_box`): no lattice information, scrambled numbering, both tetrahedron orientations, a re-entrant corner, a box
deformed in place.  None of the lattice fast paths (closed-form P2 space on the jittered meshes, stencil-class dof
order, congruence-class cell schedule, lattice slice order, multigrid hierarchy) can carry them.

Two kinds of checks: parity with the CPU oracle on identical inputs (test_gpu_parity.py's tolerances), and exact
identities that do not go through the host's dof coordinates twice -- those catch a host-side error that device and
oracle would share."""
import copy
import json
import os

import numpy as np
import pytest
import scipy.sparse as sp

import oasisx_b200 as oasisx
from oasisx_b200 import _lib as L
from oasisx_b200 import fem, mesh as bmesh
from problems import (TaylorGreen, TaylorGreenRot, jittered_mesh, l_shaped_mesh, make_cpu_port, make_mesh, make_oracle,
                      make_solver, mapped_box, relerr, vscale)

pytestmark = pytest.mark.gpu

MESHES = {
    "jittered": lambda gdim, N: jittered_mesh(gdim, N, seed=2),
    "lshape": lambda gdim, N: l_shaped_mesh(gdim, N, seed=3),
    "mapped": mapped_box,
}
VOLUME = {("jittered", 3): 8.0, ("jittered", 2): 4.0, ("lshape", 3): 7.0, ("lshape", 2): 3.0, ("mapped", 3): 8.0,
          ("mapped", 2): 4.0}
SIZE = {3: 4, 2: 8}
CASES = [(k, g, deg) for k in MESHES for g in (3, 2) for deg in (2, 1)]
LU = {"ksp_type": "preonly", "pc_type": "lu"}
KRY = {"tentative": {"ksp_type": "bcgs", "pc_type": "jacobi", "ksp_rtol": 1e-12},
       "pressure": {"ksp_type": "cg", "pc_type": "jacobi", "ksp_rtol": 1e-12},
       "scalar": {"ksp_type": "cg", "pc_type": "jacobi", "ksp_rtol": 1e-12}}

# largest relative error per group of checks, written as JSON to $B200_GENERAL_MESH_ERRORS if set
_WORST = {}


def _seen(group, value):
    _WORST[group] = max(_WORST.get(group, 0.0), float(value))
    return value


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    path = os.environ.get("B200_GENERAL_MESH_ERRORS")
    if path:
        with open(path, "w") as f:
            json.dump(_WORST, f, indent=1, sort_keys=True)


def _csr(mat):
    ip, ix, v = mat.getValuesCSR()
    return sp.csr_matrix((v, ix, ip), shape=mat.getSize())


def _mesh(kind, gdim, N=None):
    return MESHES[kind](gdim, SIZE[gdim] if N is None else N)


def mult(mat, x):
    y = np.zeros(mat.getSize()[0])
    mat.mult(np.ascontiguousarray(x), y)
    return y


def _advance(tgs, dt):
    for t in tgs:
        t.t_u += dt
        t.t_p += dt


@pytest.mark.parametrize("kind,gdim,deg", CASES)
def test_patterns_and_preassembled_matrices(kind, gdim, deg):
    msh = _mesh(kind, gdim)
    tg = TaylorGreen(0.01, gdim)
    s = make_solver(msh, deg, tg, 0.01)
    o = make_oracle(msh, deg, tg, 0.01)
    V, Q = fem.functionspace(msh, ("Lagrange", deg)), fem.functionspace(msh, ("Lagrange", 1))
    for pat, (R, C) in {L.PAT_VV: (V, V), L.PAT_VQ: (V, Q), L.PAT_QV: (Q, V), L.PAT_QQ: (Q, Q)}.items():
        ip, ix = fem.build_csr_pattern(R.dofmap.list, C.dofmap.list, R.num_dofs, C.num_dofs)
        dip, dix = s._ctx.pattern(pat, R.num_dofs)
        np.testing.assert_array_equal(dip, ip)
        np.testing.assert_array_equal(dix, ix)
    pairs = [(s._M, o.M), (s._K, o.K), (s._Ap, o.Ap)]
    for i in range(gdim):
        pairs += [(s._p_vdxi_Mat[i], o.P[i]), (s._grad_p_Mat[i], o.G[i]), (s._divu_Mat[i], o.D[i])]
    for dev, ref in pairs:
        assert _seen("matrices", abs(_csr(dev) - ref).max() / abs(ref).max()) <= 1e-12


@pytest.mark.parametrize("kind,gdim,deg", CASES)
@pytest.mark.parametrize("rows", [1, 0])
def test_assemble_first_and_tentative_rhs(kind, gdim, deg, rows):
    dt, nu = 0.1, 0.5
    f = [0.3, -0.1, 0.2][:gdim]
    msh = _mesh(kind, gdim)
    tg = TaylorGreen(nu, gdim)
    s = make_solver(msh, deg, tg, dt, body_force=f)
    s._ctx.set_tuning("first_order", rows)
    info = s._ctx.first_plan_info()
    if rows and kind != "mapped":  # no two cells are translates of each other (vertex order scrambled, jitter)
        assert info["congruence_classes"] >= 0.9 * msh.num_cells, info
    o = make_oracle(msh, deg, tg, dt, body_force=f)
    ps = lambda x: x[1] + 0.5 * x[0] ** 2
    s._ps.interpolate(ps)
    o.ps = ps(o.xQ.T)
    tg.t_u = dt
    [[bc.update_bc() for bc in b] for b in s._bcs_u]
    o.update_bcs()
    s.assemble_first(dt, nu)
    o.assemble_first(dt, nu)
    assert _seen("assemble_first", abs(_csr(s._A) - o.A).max() / abs(o.A).max()) <= 1e-12
    for i in range(gdim):
        assert _seen("assemble_first", relerr(s._b_first[i].x.array_ro(), o.b_first[i], vscale(o.b_first))) <= 1e-12
    s.velocity_tentative_assemble()
    o.velocity_tentative_assemble()
    for i in range(gdim):
        assert _seen("assemble_first", relerr(s._rhs1[i].x.array_ro(), o.rhs1[i], vscale(o.rhs1))) <= 1e-12


@pytest.mark.parametrize("kind,gdim,deg", CASES)
def test_mat_mult_matches_oracle(kind, gdim, deg):
    msh = _mesh(kind, gdim)
    tg = TaylorGreen(0.01, gdim)
    s = make_solver(msh, deg, tg, 0.01)
    o = make_oracle(msh, deg, tg, 0.01)
    rng = np.random.default_rng(0)
    xv, xq = rng.uniform(-1, 1, o.nV), rng.uniform(-1, 1, o.nQ)
    cases = [(s._M, o.M, xv), (s._K, o.K, xv), (s._Ap, o.Ap, xq)]
    for i in range(gdim):
        cases += [(s._p_vdxi_Mat[i], o.P[i], xq), (s._grad_p_Mat[i], o.G[i], xq), (s._divu_Mat[i], o.D[i], xv)]
    for dev, ref, x in cases:
        y = np.zeros(ref.shape[0])
        dev.mult(x, y)
        assert _seen("mat_mult", relerr(y, ref @ x)) <= 1e-13


@pytest.mark.parametrize("kind,gdim,deg", CASES)
@pytest.mark.parametrize("solver", ["lu", "krylov"])
@pytest.mark.parametrize("low_memory", [False, True])
def test_time_steps_match_oracle(kind, gdim, deg, solver, low_memory):
    dt, nu = 0.005, 0.01
    msh = _mesh(kind, gdim)
    tg = TaylorGreen(nu, gdim)
    s = make_solver(msh, deg, tg, dt, solver_options=KRY if solver == "krylov" else None, low_memory=low_memory)
    o = make_oracle(msh, deg, tg, dt)
    tg.t_u, tg.t_p = 0.0, -dt / 2
    for n in range(3):
        _advance([tg], dt)
        s.solve(dt, nu, max_iter=1)
        o.solve(dt, nu, max_iter=1)
        for i in range(gdim):
            for dev, ref in ((s._u, o.u), (s._u1, o.u1), (s._u2, o.u2)):
                assert _seen("time_steps", relerr(dev[i].x.array_ro(), ref[i], vscale(ref))) <= 1e-8, (n, i)
        assert _seen("time_steps", relerr(s._p.x.array_ro(), o.p)) <= 1e-8, n


@pytest.mark.parametrize("kind,gdim", [("jittered", 3), ("lshape", 2)])
def test_rotational_steps_match_oracle(kind, gdim):
    dt, nu = 0.005, 0.01
    msh = _mesh(kind, gdim)
    tg = TaylorGreenRot(nu) if gdim == 3 else TaylorGreen(nu, gdim)
    s = make_solver(msh, 2, tg, dt, rotational=True)
    o = make_oracle(msh, 2, tg, dt, rotational=True)
    tg.t_u, tg.t_p = 0.0, -dt / 2
    for n in range(3):
        _advance([tg], dt)
        s.solve(dt, nu, max_iter=1)
        o.solve(dt, nu, max_iter=1)
        for i in range(gdim):
            assert _seen("time_steps", relerr(s._u[i].x.array_ro(), o.u[i], vscale(o.u))) <= 1e-8
        assert _seen("time_steps", relerr(s._p.x.array_ro(), o.p)) <= 1e-8


@pytest.mark.parametrize("kind", ["jittered", "mapped"])
def test_pressure_multigrid(kind):
    """pc_type=mg: the jittered mesh has no hierarchy (Jacobi fallback), the deformed box keeps its own; the fields
    are the oracle's either way."""
    dt, nu, gdim = 0.005, 0.01, 3
    msh = _mesh(kind, gdim, 8)
    tg = TaylorGreen(nu, gdim)
    opts = {"tentative": LU, "scalar": LU, "pressure": {"ksp_type": "cg", "pc_type": "mg", "ksp_rtol": 1e-12}}
    s = make_solver(msh, 2, tg, dt, solver_options=opts)
    assert (s._mg_levels == 0) if kind == "jittered" else (s._mg_levels >= 2)
    o = make_oracle(msh, 2, tg, dt)
    tg.t_u, tg.t_p = 0.0, -dt / 2
    its = []
    for n in range(3):
        _advance([tg], dt)
        s.solve(dt, nu, max_iter=1)
        o.solve(dt, nu, max_iter=1)
        its.append(s.stats().its_pressure)
        for i in range(gdim):
            assert _seen("multigrid", relerr(s._u[i].x.array_ro(), o.u[i], vscale(o.u))) <= 1e-8
        assert _seen("multigrid", relerr(s._p.x.array_ro(), o.p)) <= 1e-8
    if kind == "mapped":
        _WORST["its_pressure_mapped_box_8"] = its
        assert max(its) <= 40, its


class Inlet:
    def __init__(self, t):
        self.t = t

    def eval(self, x):
        return (1 + self.t) * (1 - x[1] ** 2) * (1 - x[2] ** 2)


@pytest.mark.parametrize("deg", [2, 1])
def test_channel_with_pressure_bc_on_a_jittered_box(deg):
    """3D open channel on an unstructured box: inlet callable at x = -1, no-slip walls, PressureBC on the outlet x = 1
    (k_pressure_surface with the 3-point triangle rule), two inner-iterated steps against the oracle."""
    from oracle.ipcs_oracle import OracleIPCS
    from test_gpu_tentative import _global_pressure_facets

    msh = jittered_mesh(3, 4, seed=5)
    dim = 2
    left = bmesh.locate_entities_boundary(msh, dim, lambda x: np.isclose(x[0], -1))
    walls = np.unique(np.hstack([bmesh.locate_entities_boundary(msh, dim, lambda x, k=k, v=v: np.isclose(x[k], v))
                                 for k in (1, 2) for v in (-1.0, 1.0)]))
    right = bmesh.locate_entities_boundary(msh, dim, lambda x: np.isclose(x[0], 1))
    assert len(left) == len(right) == 32 and len(walls) == 128
    facets = np.hstack([left, walls, right])
    values = np.hstack([np.full_like(left, 1), np.full_like(walls, 2), np.full_like(right, 3)])
    order = np.argsort(facets)
    tags = bmesh.meshtags(msh, dim, facets[order], values[order])
    inlet = Inlet(0.0)
    T = oasisx.LocatorMethod.TOPOLOGICAL
    bc_w = oasisx.DirichletBC(0.0, T, (tags, 2))
    bcs_u = [[oasisx.DirichletBC(inlet.eval, T, (tags, 1)), bc_w], [oasisx.DirichletBC(0.0, T, (tags, 1)), bc_w],
             [oasisx.DirichletBC(0.0, T, (tags, 1)), bc_w]]
    s = oasisx.FractionalStep_AB_CN(msh, ("Lagrange", deg), ("Lagrange", 1), bcs_u=bcs_u,
                                    bcs_p=[oasisx.PressureBC(4.0, (tags, 3))],
                                    solver_options={"tentative": LU, "pressure": LU, "scalar": LU},
                                    options={"low_memory_version": False})
    V, Q = fem.functionspace(msh, ("Lagrange", deg)), fem.functionspace(msh, ("Lagrange", 1))
    dl, dw = fem.locate_dofs_topological(V, dim, left), fem.locate_dofs_topological(V, dim, walls)
    o = OracleIPCS(msh.geometry.x, msh.geometry.dofmap, 3, V.dofmap.list, Q.dofmap.list, V.tabulate_dof_coordinates(),
                   Q.tabulate_dof_coordinates(), deg,
                   bcs_u=[[(dl, inlet.eval), (dw, 0.0)], [(dl, 0.0), (dw, 0.0)], [(dl, 0.0), (dw, 0.0)]],
                   bcs_p=[fem.locate_dofs_topological(Q, dim, right)],
                   pressure_facets=[_global_pressure_facets(msh, right) + (4.0,)])
    dt, nu = 0.01, 0.5
    for n in range(2):
        inlet.t += dt
        s.solve(dt, nu, max_iter=2, max_error=1e-30)
        o.solve(dt, nu, max_iter=2, max_error=1e-30)
        for i in range(3):
            assert _seen("channel_pressure_bc", relerr(s._u[i].x.array_ro(), o.u[i], vscale(o.u))) <= 1e-8, (n, i)
        assert _seen("channel_pressure_bc", relerr(s._p.x.array_ro(), o.p)) <= 1e-8, n
    assert max(np.abs(p).max() for p in o.p_surf) > 1e-3  # the natural pressure term is there and matters


@pytest.mark.parametrize("gdim", [3, 2])
def test_l2_error_functionals(gdim):
    dt, nu = 0.005, 0.01
    msh = _mesh("jittered", gdim)
    tg = TaylorGreen(nu, gdim)
    s = make_solver(msh, 2, tg, dt)
    o = make_oracle(msh, 2, tg, dt)
    tg.t_u, tg.t_p = dt, dt / 2
    s.solve(dt, nu, max_iter=1)
    o.solve(dt, nu, max_iter=1)
    ou = o.F.l2_error_sq(o.u, o.vdofs, tg.components, degree=10)
    op = o.F.l2_error_sq([o.p], o.qdofs, [tg.eval_p], degree=10, space="Q")
    for e_u, e_p in ((s.assemble_l2_error_sq("u", tg.components, degree=10), s.assemble_l2_error_sq("p", tg.eval_p, degree=10)),
                     (s.assemble_l2_error_sq("u", tg, degree=10), s.assemble_l2_error_sq("p", tg, degree=10))):
        assert _seen("l2_error", abs(e_u - ou) / ou) <= 1e-10
        assert _seen("l2_error", abs(e_p - op) / op) <= 1e-10


# ---- exact identities: independent of the host's dof coordinates being handed to both sides ----------------------

def _quadratics(gdim):
    return [lambda x: x[0] ** 2 + 3.0 * x[1] * x[2] - x[1], lambda x: x[1] ** 2 - 2.0 * x[0] * x[1] + 0.5,
            lambda x: x[2] ** 2 + x[0] * x[2] + x[0]][:gdim]


@pytest.mark.parametrize("kind", list(MESHES))
@pytest.mark.parametrize("gdim", [3, 2])
def test_exact_identities(kind, gdim):
    """1^T M 1 = |Omega| = sum(mQ); G_i I1(x_i) = M 1 and D_i I2(x_i) = mQ; on rows off the boundary, with u_ab = c and
    u_1 = l linear, A l = M l / dt + 1/2 (c . grad l) M 1 and b_first = M l / dt - 1/2 (c . grad l) M 1 (K l vanishes
    there); the P2 interpolant of a quadratic and the P1 interpolant of a linear function have zero L2 error."""
    dt, nu = 0.1, 0.3
    msh = _mesh(kind, gdim)
    vol = VOLUME[(kind, gdim)]
    tg = TaylorGreen(nu, gdim)
    s = make_solver(msh, 2, tg, dt)
    o = make_oracle(msh, 2, tg, dt)
    nV, nQ = o.nV, o.nQ
    xV, xQ = s._Vi[0][0].tabulate_dof_coordinates(), s._Q.tabulate_dof_coordinates()
    M1 = mult(s._M, np.ones(nV))
    assert _seen("identities", abs(M1.sum() - vol) / vol) <= 1e-13
    assert _seen("identities", abs(o.mQ.sum() - vol) / vol) <= 1e-13
    for i in range(gdim):
        assert _seen("identities", relerr(mult(s._grad_p_Mat[i], xQ[:, i]), M1)) <= 1e-13
        assert _seen("identities", relerr(mult(s._divu_Mat[i], xV[:, i]), o.mQ)) <= 1e-13
    # assemble_first on a linear field advected by a constant one
    c = [0.7, -0.4, 0.25][:gdim]
    grad = np.array([0.5, -1.0, 2.0])[:gdim]
    lin = lambda x: 1.0 + grad @ x[:gdim]
    lv = lin(xV.T)
    for i in range(gdim):
        s._u1[i].x.array[:] = lv
        s._u2[i].x.array[:] = 3.0 * lv - 2.0 * c[i]  # u_ab = 1.5 u1 - 0.5 u2 = c
    s.assemble_first(dt, nu)
    interior = np.setdiff1d(np.arange(nV), s._bc_dofs[0])
    assert len(interior) > 0
    Ml = mult(s._M, lv)
    adv = 0.5 * float(np.dot(c, grad)) * M1
    Al = mult(s._A, lv)
    scale = np.abs(Ml / dt).max()
    assert _seen("identities", np.abs(Al - (Ml / dt + adv))[interior].max() / scale) <= 1e-12
    for i in range(gdim):
        b = s._b_first[i].x.array_ro()
        assert _seen("identities", np.abs(b - (Ml / dt - adv))[interior].max() / scale) <= 1e-12
    # interpolation is exact for the space's own polynomials, measured against the callables
    qs = _quadratics(gdim)
    for i, q in enumerate(qs):
        s._u[i].interpolate(q)
    s._p.interpolate(lin)
    assert _seen("interpolation_l2_sq", s.assemble_l2_error_sq("u", qs, degree=4)) <= 1e-24
    assert _seen("interpolation_l2_sq", s.assemble_l2_error_sq("p", lin, degree=4)) <= 1e-24
    s1 = make_solver(_mesh(kind, gdim), 1, TaylorGreen(nu, gdim), dt)
    lins = [lambda x, k=k: 0.5 - x[k] + 2.0 * x[(k + 1) % gdim] for k in range(gdim)]
    for i, f in enumerate(lins):
        s1._u[i].interpolate(f)
    assert _seen("interpolation_l2_sq", s1.assemble_l2_error_sq("u", lins, degree=4)) <= 1e-24


# ---- medium size ----------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def medium():
    import bench

    dt, nu, N = 0.005, 0.01, 17
    msh = jittered_mesh(3, N, seed=7)
    tg = TaylorGreen(nu, 3)
    opts = copy.deepcopy(bench.KRYLOV)
    for o_ in opts.values():
        o_["ksp_rtol"] = 1e-12
    s = make_solver(msh, 2, tg, dt, solver_options=opts)
    return msh, tg, s, dt, nu


def test_medium_jittered_box_matches_the_cpu_port(medium):
    """17^3 cubes (0.13 M dofs), 8 steps with the benchmark's solver settings (the multigrid falls back to Jacobi) against the
    C++/OpenMP port at rtol 1e-12."""
    from oracle import ipcs_cpu as cpu

    msh, tg, s, dt, nu = medium
    assert s._mg_levels == 0 and 3 * s._Vi[0][0].num_dofs + s._Q.num_dofs > 130000
    tg2 = TaylorGreen(nu, 3)
    c = make_cpu_port(msh, 2, tg2, dt, rtol=1e-12, nonzero_guess=True, block_rtol=True, extrapolate=2)
    for t in (tg, tg2):
        t.t_u, t.t_p = 0.0, -dt / 2
    for n in range(8):
        _advance([tg, tg2], dt)
        s.solve(dt, nu, max_iter=1)
        c.solve(dt, nu)
        cu = [c.get(cpu.U, i) for i in range(3)]
        for i in range(3):
            assert _seen("medium_cpu_port", relerr(s._u[i].x.array_ro(), cu[i], vscale(cu))) <= 1e-8, (n, i)
        assert _seen("medium_cpu_port", relerr(s._p.x.array_ro(), c.get(cpu.P))) <= 1e-8, n


def test_spmm_matches_scipy_on_the_medium_jittered_box(medium):
    """M x, K x and A x (after assemble_first) through the device SpMM against the scipy product to 1e-13."""
    msh, tg, s, dt, nu = medium
    s.assemble_first(dt, nu)
    x = np.random.default_rng(3).uniform(-1, 1, s._Vi[0][0].num_dofs)
    for k, m in {"M": s._M, "K": s._K, "A": s._A}.items():
        assert _seen("spmm", relerr(mult(m, x), _csr(m) @ x)) <= 1e-13, k


def test_dof_orders_give_the_same_fields():
    """The stencil-class, window-sorted ("sigma") and plain coordinate ("generic") dof orders of a box: the same
    fields after 3 steps once matched by dof coordinates."""
    dt, nu = 0.005, 0.01
    out = {}
    for kind in ("class", "sigma", "generic"):
        msh = make_mesh(3, 8)
        msh._dof_order = kind
        tg = TaylorGreen(nu, 3)
        s = make_solver(msh, 2, tg, dt, solver_options=KRY)
        tg.t_u, tg.t_p = 0.0, -dt / 2
        for n in range(3):
            _advance([tg], dt)
            s.solve(dt, nu, max_iter=1)
        xv, xq = s._Vi[0][0].tabulate_dof_coordinates(), s._Q.tabulate_dof_coordinates()
        ov, oq = np.lexsort(xv.T[::-1]), np.lexsort(xq.T[::-1])
        out[kind] = (xv[ov], [s._u[i].x.array_ro()[ov] for i in range(3)], s._p.x.array_ro()[oq])
    xr, ur, pr = out["class"]
    for kind in ("sigma", "generic"):
        x, u, p = out[kind]
        np.testing.assert_array_equal(x, xr)
        for i in range(3):
            assert _seen("dof_orders", relerr(u[i], ur[i], vscale(ur))) <= 1e-10, (kind, i)
        assert _seen("dof_orders", relerr(p, pr)) <= 1e-10, kind
