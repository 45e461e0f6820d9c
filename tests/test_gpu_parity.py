"""Parity of the CUDA path (through the C ABI) with the CPU oracle on identical inputs.

Tolerances are north_star's: CSR sparsity bit-exact; assembled FP64 entries <= 1e-12 relative
(measured against the row/matrix max, SURVEY.md Appendix C tolerance note); per-step fields <= 1e-8
relative with the solvers run to rtol 1e-12 ("preonly+lu" equivalent)."""
import numpy as np
import pytest
import scipy.sparse as sp

from oasisx_b200 import _lib as L
from oasisx_b200 import fem
from problems import TaylorGreen, boundary_facets, make_mesh, make_oracle, make_solver, relerr, vscale

pytestmark = pytest.mark.gpu

CASES = [(2, 8, 2), (3, 4, 2), (2, 8, 1), (3, 3, 1)]


def _csr(mat):
    ip, ix, v = mat.getValuesCSR()
    return sp.csr_matrix((v, ix, ip), shape=mat.getSize())


@pytest.mark.parametrize("gdim,N,deg", CASES)
def test_patterns_bit_exact(gdim, N, deg):
    msh = make_mesh(gdim, N)
    s = make_solver(msh, deg, TaylorGreen(0.01, gdim), 0.01)
    V, Q = fem.functionspace(msh, ("Lagrange", deg)), fem.functionspace(msh, ("Lagrange", 1))
    for pat, (R, C) in {L.PAT_VV: (V, V), L.PAT_VQ: (V, Q), L.PAT_QV: (Q, V), L.PAT_QQ: (Q, Q)}.items():
        ip, ix = fem.build_csr_pattern(R.dofmap.list, C.dofmap.list, R.num_dofs, C.num_dofs)
        dip, dix = s._ctx.pattern(pat, R.num_dofs)
        assert dip.dtype == np.int32 and dix.dtype == np.int32
        np.testing.assert_array_equal(dip, ip)
        np.testing.assert_array_equal(dix, ix)


@pytest.mark.parametrize("gdim,N,deg", CASES)
def test_preassembled_matrices(gdim, N, deg):
    msh = make_mesh(gdim, N)
    tg = TaylorGreen(0.01, gdim)
    s = make_solver(msh, deg, tg, 0.01)
    o = make_oracle(msh, deg, tg, 0.01)
    pairs = [(s._M, o.M), (s._K, o.K), (s._Ap, o.Ap)]
    for i in range(gdim):
        pairs += [(s._p_vdxi_Mat[i], o.P[i]), (s._grad_p_Mat[i], o.G[i]), (s._divu_Mat[i], o.D[i])]
    for dev, ref in pairs:
        A = _csr(dev)
        assert abs(A - ref).max() <= 1e-12 * abs(ref).max()
    b0 = s._b0[0].x.array_ro()
    np.testing.assert_allclose(b0, 0.0, atol=0)


@pytest.mark.parametrize("gdim,N,deg", CASES)
@pytest.mark.parametrize("body_force", [False, True])
@pytest.mark.parametrize("rows", [1, 0])
def test_assemble_first_and_tentative_rhs(gdim, N, deg, body_force, rows):
    """A, b_first and rhs1 after assemble_first + velocity_tentative_assemble
    (test/test_tentative_velocity.py:172-173,235), with the congruence-class cell schedule (rows=1, the default:
    coalesced scatter) and in mesh order (rows=0)."""
    dt, nu = 0.1, 0.5
    f = [0.3, -0.1, 0.2][:gdim] if body_force else None
    msh = make_mesh(gdim, N)
    tg = TaylorGreen(nu, gdim)
    s = make_solver(msh, deg, tg, dt, body_force=f)
    s._ctx.set_tuning("first_order", rows)
    o = make_oracle(msh, deg, tg, dt, body_force=f)
    ps = lambda x: x[1] + 0.5 * x[0] ** 2
    s._ps.interpolate(ps)
    o.ps = ps(o.xQ.T)
    tg.t_u = dt
    [[bc.update_bc() for bc in b] for b in s._bcs_u]
    o.update_bcs()
    s.assemble_first(dt, nu)
    o.assemble_first(dt, nu)
    A = _csr(s._A)
    assert abs(A - o.A).max() <= 1e-12 * abs(o.A).max()
    for i in range(gdim):
        assert relerr(s._b_first[i].x.array_ro(), o.b_first[i], vscale(o.b_first)) <= 1e-12
    s.velocity_tentative_assemble()
    o.velocity_tentative_assemble()
    for i in range(gdim):
        assert relerr(s._rhs1[i].x.array_ro(), o.rhs1[i], vscale(o.rhs1)) <= 1e-12
    diff, reasons = s.velocity_tentative_solve()
    odiff, _ = o.velocity_tentative_solve()
    assert (reasons > 0).all()
    for i in range(gdim):
        assert relerr(s._rhs1[i].x.array_ro(), o.rhs1[i], vscale(o.rhs1)) <= 1e-12  # now with BC values applied
        assert relerr(s._u[i].x.array_ro(), o.u[i], vscale(o.u)) <= 1e-9
    assert abs(diff - odiff) <= 1e-8 * odiff


@pytest.mark.parametrize("gdim,N", [(3, 20), (2, 96)])
def test_rowwise_and_scatter_assembly_agree_on_larger_meshes(gdim, N):
    """Beyond the sizes the LU oracle reaches: the fused row-wise assemble_first and the scatter + combine pair give
    the same A (<= 1e-13 of its largest entry), b_first and Jacobi scaling on meshes with thousands of slices."""
    dt, nu = 0.005, 0.01
    msh = make_mesh(gdim, N)
    tg = TaylorGreen(nu, gdim)
    kry = {"ksp_type": "bcgs", "pc_type": "jacobi", "ksp_rtol": 1e-10}
    cg = {"ksp_type": "cg", "pc_type": "jacobi", "ksp_rtol": 1e-10}
    s = make_solver(msh, 2, tg, dt, solver_options={"tentative": kry, "pressure": cg, "scalar": cg})
    tg.t_u = dt
    out = []
    for rows in (1, 0):
        s._ctx.set_tuning("first_order", rows)
        s.assemble_first(dt, nu)
        out.append((_csr(s._A), [s._b_first[i].x.array_ro().copy() for i in range(gdim)]))
    (A1, b1), (A0, b0) = out
    assert abs(A1 - A0).max() <= 1e-13 * abs(A0).max()
    for i in range(gdim):
        assert relerr(b1[i], b0[i], vscale(b0)) <= 1e-13


@pytest.mark.parametrize("gdim,N,steps", [(3, 24, 8), (2, 128, 8)])
def test_medium_meshes_match_the_cpu_port(gdim, N, steps):
    """Sizes between the LU oracle's reach and the benchmark (3D 24^3: 0.37 M dofs, 2D 128^2): the CUDA path with the
    benchmark's settings (multigrid, history-extrapolated guesses, block tolerance) against the C++/OpenMP restatement
    with Jacobi-PCG, both at rtol 1e-12: per-step fields <= 1e-8, long enough for the three-deep histories to fill."""
    import copy

    import bench
    from oracle import ipcs_cpu as cpu
    from problems import make_cpu_port

    dt, nu = 0.005, 0.01
    msh = make_mesh(gdim, N)
    tg, tg2 = TaylorGreen(nu, gdim), TaylorGreen(nu, gdim)
    opts = copy.deepcopy(bench.KRYLOV)
    for o_ in opts.values():
        o_["ksp_rtol"] = 1e-12
    s = make_solver(msh, 2, tg, dt, solver_options=opts)
    c = make_cpu_port(msh, 2, tg2, dt, rtol=1e-12, nonzero_guess=True, block_rtol=True, extrapolate=2)
    for t in (tg, tg2):
        t.t_u, t.t_p = 0.0, -dt / 2
    for n in range(steps):
        for t in (tg, tg2):
            t.t_u += dt
            t.t_p += dt
        s.solve(dt, nu, max_iter=1)
        c.solve(dt, nu)
        cu = [c.get(cpu.U, i) for i in range(gdim)]
        for i in range(gdim):
            assert relerr(s._u[i].x.array_ro(), cu[i], vscale(cu)) <= 1e-8, (n, i)
        assert relerr(s._p.x.array_ro(), c.get(cpu.P)) <= 1e-8, n


@pytest.mark.parametrize("gdim,N,deg", [(2, 8, 2), (3, 4, 2), (2, 8, 1)])
def test_spmv_matches_oracle(gdim, N, deg):
    msh = make_mesh(gdim, N)
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
        assert relerr(y, ref @ x) <= 1e-13


@pytest.mark.parametrize("gdim,N,deg,steps", [(2, 8, 2, 5), (3, 4, 2, 3), (2, 16, 2, 3), (2, 8, 1, 3)])
def test_time_steps_match_oracle(gdim, N, deg, steps):
    """Per-step velocity and pressure fields (demo/taylor_green.py:199-213 loop), <= 1e-8 relative."""
    dt, nu = 0.005, 0.01
    msh = make_mesh(gdim, N)
    tg = TaylorGreen(nu, gdim)
    s = make_solver(msh, deg, tg, dt)
    o = make_oracle(msh, deg, tg, dt)
    tg.t_u, tg.t_p = 0.0, -dt / 2
    for n in range(steps):
        tg.t_u += dt
        tg.t_p += dt
        d1 = s.solve(dt, nu, max_iter=1)
        d2 = o.solve(dt, nu, max_iter=1)
        for i in range(gdim):
            assert relerr(s._u[i].x.array_ro(), o.u[i], vscale(o.u)) <= 1e-8, (n, i)
            assert relerr(s._u1[i].x.array_ro(), o.u1[i], vscale(o.u1)) <= 1e-8
            assert relerr(s._u2[i].x.array_ro(), o.u2[i], vscale(o.u2)) <= 1e-8
        assert relerr(s._p.x.array_ro(), o.p) <= 1e-8, n
        assert abs(d1 - d2) <= 1e-7 * max(d2, 1e-300)
    # blocked output vector == interleaved components (fracstep.py:698-705)
    u = s.u.x.array
    for i in range(gdim):
        np.testing.assert_array_equal(u[i::gdim], s._u[i].x.array_ro())
    st = s.stats()
    assert st.kernel_launches > 0 and st.its_pressure > 0


def test_inner_iterations_and_staged_calls_equal_fused_step():
    """solve() == the staged sequence of fracstep.py:673-693 with max_iter=2."""
    dt, nu = 0.01, 0.01
    msh = make_mesh(2, 8)
    tg = TaylorGreen(nu, 2)
    s = make_solver(msh, 2, tg, dt)
    o = make_oracle(msh, 2, tg, dt)
    tg.t_u, tg.t_p = dt, dt / 2
    s.solve(dt, nu, max_error=1e-30, max_iter=2)
    o.solve(dt, nu, max_error=1e-30, max_iter=2)
    for i in range(2):
        assert relerr(s._u[i].x.array_ro(), o.u[i], vscale(o.u)) <= 1e-8
    assert relerr(s._p.x.array_ro(), o.p) <= 1e-8


def test_rotational_pressure_update():
    dt, nu = 0.005, 0.01
    msh = make_mesh(2, 8)
    tg = TaylorGreen(nu, 2)
    s = make_solver(msh, 2, tg, dt, rotational=True)
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


def test_krylov_options_and_reasons():
    """Explicit Krylov options (Appendix G) reach the device; reasons are PETSc codes."""
    dt, nu = 0.005, 0.01
    msh = make_mesh(3, 4)
    tg = TaylorGreen(nu, 3)
    opts = {
        "tentative": {"ksp_type": "bcgs", "pc_type": "jacobi", "ksp_rtol": 1e-10},
        "pressure": {"ksp_type": "cg", "pc_type": "jacobi", "ksp_rtol": 1e-10},
        "scalar": {"ksp_type": "cg", "pc_type": "jacobi", "ksp_rtol": 1e-10},
    }
    s = make_solver(msh, 2, tg, dt, solver_options=opts)
    o = make_oracle(msh, 2, tg, dt)
    tg.t_u, tg.t_p = dt, dt / 2
    [[bc.update_bc() for bc in b] for b in s._bcs_u]
    s._ps.x.array[:] = s._p.x.array
    s.assemble_first(dt, nu)
    s.velocity_tentative_assemble()
    _, r = s.velocity_tentative_solve()
    assert set(r.tolist()) <= {2, 3}
    s.pressure_assemble(dt)
    assert s.pressure_solve(nu) in (2, 3)
    assert set(s.velocity_update(dt).tolist()) <= {2, 3}
    o.solve(dt, nu, max_iter=1)
    for i in range(3):
        assert relerr(s._u[i].x.array_ro(), o.u[i], vscale(o.u)) <= 1e-7
    # an impossible iteration budget reports KSP_DIVERGED_ITS
    s._solver_p.updateOptions({"ksp_max_it": 2, "ksp_rtol": 1e-14})
    s.pressure_assemble(dt)
    assert s.pressure_solve(nu) == -3


@pytest.mark.parametrize("gdim,N,dense", [(3, 8, 1), (3, 8, 0), (2, 16, 1), (3, 48, 1)])
def test_pressure_multigrid_matches_oracle(gdim, N, dense):
    """pc_type=mg on the pressure: same converged fields as the oracle's direct solve (<= 1e-8), with the exact
    (dense-inverse) coarse-level solve and with smoothing all the way down; 48^3 puts the dense level (13^3 dofs)
    two levels below the fine one (49^3, 25^3, 13^3)."""
    dt, nu = 0.005, 0.01
    msh = make_mesh(gdim, N)
    tg = TaylorGreen(nu, gdim)
    lu = {"ksp_type": "preonly", "pc_type": "lu"}
    opts = {"tentative": lu, "scalar": lu, "pressure": {"ksp_type": "cg", "pc_type": "mg", "ksp_rtol": 1e-12}}
    if N >= 32:  # the LU oracle cannot follow: compare with Jacobi-PCG on the same device path instead
        _multigrid_vs_jacobi(msh, tg, dt, nu)
        return
    s = make_solver(msh, 2, tg, dt, solver_options=opts)
    s._ctx.set_tuning("mg_dense", dense)
    assert s._mg_levels >= 2
    o = make_oracle(msh, 2, tg, dt)
    tg.t_u, tg.t_p = 0.0, -dt / 2
    its = []
    for n in range(3):
        tg.t_u += dt
        tg.t_p += dt
        s.solve(dt, nu, max_iter=1)
        o.solve(dt, nu, max_iter=1)
        its.append(s.stats().its_pressure)
        for i in range(gdim):
            assert relerr(s._u[i].x.array_ro(), o.u[i], vscale(o.u)) <= 1e-8
        assert relerr(s._p.x.array_ro(), o.p) <= 1e-8
    assert max(its) <= 40, its  # mesh-independent convergence (Jacobi-PCG needs hundreds at scale)


def _multigrid_vs_jacobi(msh, tg, dt, nu):
    kry = {"ksp_type": "bcgs", "pc_type": "jacobi", "ksp_rtol": 1e-12}
    cg = {"ksp_type": "cg", "pc_type": "jacobi", "ksp_rtol": 1e-12}
    sols = []
    for pc in ("mg", "jacobi"):
        tg.t_u, tg.t_p = 0.0, -dt / 2
        s = make_solver(msh, 2, tg, dt, solver_options={"tentative": kry, "scalar": cg, "pressure": {**cg, "pc_type": pc}})
        tg.t_u, tg.t_p = 0.0, -dt / 2
        for n in range(2):
            tg.t_u += dt
            tg.t_p += dt
            s.solve(dt, nu, max_iter=1)
        sols.append(([s._u[i].x.array_ro().copy() for i in range(3)], s._p.x.array_ro().copy(), s.stats().its_pressure))
    (u_mg, p_mg, its_mg), (u_j, p_j, its_j) = sols
    for i in range(3):
        assert relerr(u_mg[i], u_j[i], vscale(u_j)) <= 1e-8
    assert relerr(p_mg, p_j) <= 1e-8
    assert its_mg <= 20 < its_j, (its_mg, its_j)


@pytest.mark.parametrize("guess,max_iter", [("extrapolate", 1), ("extrapolate2", 1), ("extrapolate2", 2)])
def test_extrapolated_initial_guesses_do_not_change_the_solution(guess, max_iter):
    """b200_guess=extrapolate / extrapolate2 only change the Krylov starting point and b200_block_rtol only stops
    the solver from polishing a component whose right-hand side is round-off (w = 0 in the z-extruded field):
    fields still match the oracle (also with repeated inner passes, which must not enter the time history twice),
    and the zero component needs no more iterations than the others."""
    dt, nu = 0.005, 0.01
    msh = make_mesh(3, 6)
    tg = TaylorGreen(nu, 3)
    opts = {
        "tentative": {"ksp_type": "bcgs", "pc_type": "jacobi", "ksp_rtol": 1e-12, "b200_guess": guess,
                      "b200_block_rtol": True},
        "pressure": {"ksp_type": "cg", "pc_type": "mg", "ksp_rtol": 1e-12, "b200_guess": "extrapolate"},
        "scalar": {"ksp_type": "cg", "pc_type": "jacobi", "ksp_rtol": 1e-12, "b200_guess": guess,
                   "b200_block_rtol": True},
    }
    s = make_solver(msh, 2, tg, dt, solver_options=opts)
    o = make_oracle(msh, 2, tg, dt)
    tg.t_u, tg.t_p = 0.0, -dt / 2
    for n in range(6):
        tg.t_u += dt
        tg.t_p += dt
        s.solve(dt, nu, max_iter=max_iter)
        o.solve(dt, nu, max_iter=max_iter)
        for i in range(3):
            assert relerr(s._u[i].x.array_ro(), o.u[i], vscale(o.u)) <= 1e-8, n
        assert relerr(s._p.x.array_ro(), o.p) <= 1e-8, n
    st = s.stats()
    assert st.its_update[2] <= max(st.its_update[0], st.its_update[1])


@pytest.mark.parametrize("gdim,N", [(2, 8), (3, 4)])
def test_l2_error_functional_matches_oracle(gdim, N):
    """assemble_scalar of |u_h - u_ex|^2 and |p_h - p_ex|^2 (demo/taylor_green.py:186-207) <= 1e-10 rel."""
    dt, nu = 0.005, 0.01
    msh = make_mesh(gdim, N)
    tg = TaylorGreen(nu, gdim)
    s = make_solver(msh, 2, tg, dt)
    o = make_oracle(msh, 2, tg, dt)
    tg.t_u, tg.t_p = dt, dt / 2
    s.solve(dt, nu, max_iter=1)
    o.solve(dt, nu, max_iter=1)
    eu = s.assemble_l2_error_sq("u", tg.components, degree=10)
    ep = s.assemble_l2_error_sq("p", tg.eval_p, degree=10)
    ou = o.F.l2_error_sq(o.u, o.vdofs, tg.components, degree=10)
    op = o.F.l2_error_sq([o.p], o.qdofs, [tg.eval_p], degree=10, space="Q")
    assert abs(eu - ou) <= 1e-8 * ou and abs(ep - op) <= 1e-8 * op


@pytest.mark.parametrize("field", ["z", "rot", "2d"])
def test_l2_error_functional_device_evaluator(field):
    """The analytic field evaluated ON THE DEVICE (trigonometric product terms, b2_l2_error_trig) gives the same
    functional as the host-sampled path: the demo loop's error norms without moving the field over the bus."""
    from problems import TaylorGreenRot

    dt, nu = 0.005, 0.01
    gdim = 2 if field == "2d" else 3
    msh = make_mesh(gdim, 8 if gdim == 2 else 4)
    tg = TaylorGreenRot(nu) if field == "rot" else TaylorGreen(nu, gdim)
    s = make_solver(msh, 2, tg, dt)
    tg.t_u, tg.t_p = dt, dt / 2
    s.solve(dt, nu, max_iter=1)
    eu_h = s.assemble_l2_error_sq("u", tg.components, degree=10)
    ep_h = s.assemble_l2_error_sq("p", tg.eval_p, degree=10)
    h2d = s.stats().bytes_h2d
    eu_d = s.assemble_l2_error_sq("u", tg, degree=10)
    ep_d = s.assemble_l2_error_sq("p", tg, degree=10)
    assert s.stats().bytes_h2d - h2d < 20000  # a term list and a quadrature rule, not the sampled field
    assert abs(eu_d - eu_h) <= 1e-10 * eu_h and abs(ep_d - ep_h) <= 1e-10 * ep_h


@pytest.mark.parametrize("gdim,N,deg", [(2, 8, 2), (3, 4, 2), (2, 8, 1)])
@pytest.mark.parametrize("rotational", [False, True])
def test_low_memory_version_matches_oracle(gdim, N, deg, rotational):
    """options={"low_memory_version": True} (the reference's class default, fracstep.py:259): the
    matrix-free element-vector kernels give the same steps as the oracle (and as the matrix strategy)."""
    dt, nu = 0.005, 0.01
    msh = make_mesh(gdim, N)
    tg = TaylorGreen(nu, gdim)
    s = make_solver(msh, deg, tg, dt, low_memory=True, rotational=rotational)
    assert not hasattr(s, "_p_vdxi_Mat")
    o = make_oracle(msh, deg, tg, dt, rotational=rotational)
    tg.t_u, tg.t_p = 0.0, -dt / 2
    for n in range(3):
        tg.t_u += dt
        tg.t_p += dt
        s.solve(dt, nu, max_iter=1)
        o.solve(dt, nu, max_iter=1)
        for i in range(gdim):
            assert relerr(s._rhs1[i].x.array_ro(), o.rhs1[i], vscale(o.rhs1)) <= 1e-11
            assert relerr(s._u[i].x.array_ro(), o.u[i], vscale(o.u)) <= 1e-8
        assert relerr(s._p.x.array_ro(), o.p) <= 1e-8


def test_lid_driven_cavity_matches_oracle():
    """BASELINE config 5 in miniature: 3D lid-driven cavity (u = (1,0,0) on the lid z = 1, no-slip elsewhere,
    no pressure BC), constant-value DirichletBCs, Re = 100, a few steps against the oracle."""
    import oasisx_b200 as oasisx
    from oasisx_b200 import fem, mesh as bmesh
    from oracle.ipcs_oracle import OracleIPCS

    N, dt, nu = 6, 0.01, 0.01
    msh = bmesh.create_unit_cube(None, N, N, N)
    lid = lambda x: np.isclose(x[2], 1.0)
    walls = lambda x: np.isclose(x[0], 0) | np.isclose(x[0], 1) | np.isclose(x[1], 0) | np.isclose(x[1], 1) | np.isclose(x[2], 0)
    G = oasisx.LocatorMethod.GEOMETRICAL
    bcs_u = [[oasisx.DirichletBC(0.0, G, walls), oasisx.DirichletBC(1.0, G, lid)],
             [oasisx.DirichletBC(0.0, G, walls), oasisx.DirichletBC(0.0, G, lid)],
             [oasisx.DirichletBC(0.0, G, walls), oasisx.DirichletBC(0.0, G, lid)]]
    lu = {"ksp_type": "preonly", "pc_type": "lu"}
    s = oasisx.FractionalStep_AB_CN(msh, ("Lagrange", 2), ("Lagrange", 1), bcs_u=bcs_u, bcs_p=[],
                                    solver_options={"tentative": lu, "pressure": lu, "scalar": lu})
    V, Q = fem.functionspace(msh, ("Lagrange", 2)), fem.functionspace(msh, ("Lagrange", 1))
    dw, dl = fem.locate_dofs_geometrical(V, walls), fem.locate_dofs_geometrical(V, lid)
    o = OracleIPCS(msh.geometry.x, msh.geometry.dofmap, 3, V.dofmap.list, Q.dofmap.list, V.tabulate_dof_coordinates(),
                   Q.tabulate_dof_coordinates(), 2,
                   bcs_u=[[(dw, 0.0), (dl, 1.0)], [(dw, 0.0), (dl, 0.0)], [(dw, 0.0), (dl, 0.0)]])
    for n in range(4):
        s.solve(dt, nu, max_iter=1)
        o.solve(dt, nu, max_iter=1)
        for i in range(3):
            assert relerr(s._u[i].x.array_ro(), o.u[i], vscale(o.u)) <= 1e-8, (n, i)
        assert relerr(s._p.x.array_ro(), o.p) <= 1e-8, n
    assert np.abs(s._u[0].x.array_ro()).max() > 0.5  # the lid drives the flow


@pytest.mark.parametrize("gdim,N,deg", [(3, 6, 2), (2, 12, 2), (2, 10, 1)])
def test_chebyshev_mass_solve_matches_oracle(gdim, N, deg):
    """ksp_type=chebyshev on the velocity update (reduction-free, element-level eigenvalue bounds)."""
    dt, nu = 0.005, 0.01
    msh = make_mesh(gdim, N)
    tg = TaylorGreen(nu, gdim)
    lu = {"ksp_type": "preonly", "pc_type": "lu"}
    opts = {"tentative": lu, "pressure": lu, "scalar": {"ksp_type": "chebyshev", "pc_type": "jacobi", "ksp_rtol": 1e-12}}
    s = make_solver(msh, deg, tg, dt, solver_options=opts)
    o = make_oracle(msh, deg, tg, dt)
    tg.t_u, tg.t_p = 0.0, -dt / 2
    for n in range(3):
        tg.t_u += dt
        tg.t_p += dt
        s.solve(dt, nu, max_iter=1)
        o.solve(dt, nu, max_iter=1)
        for i in range(gdim):
            assert relerr(s._u[i].x.array_ro(), o.u[i], vscale(o.u)) <= 1e-8
    assert 0 < max(s.stats().its_update) < 80


def test_checkpoint_restart_reproduces_the_run(tmp_path):
    """u1, u2, p and t (fracstep.py:689-693) are all a restart needs: 3 steps + checkpoint + 2 steps equals
    5 steps; the VTU export of the final state is written and well-formed."""
    from oasisx_b200.io import load_checkpoint, save_checkpoint, write_vtu

    dt, nu = 0.005, 0.01
    msh = make_mesh(3, 4)
    tg = TaylorGreen(nu, 3)
    s = make_solver(msh, 2, tg, dt)
    tg.t_u, tg.t_p = 0.0, -dt / 2
    for n in range(3):
        tg.t_u += dt
        tg.t_p += dt
        s.solve(dt, nu, max_iter=1)
    save_checkpoint(str(tmp_path / "chk"), s, tg.t_u)
    for n in range(2):
        tg.t_u += dt
        tg.t_p += dt
        s.solve(dt, nu, max_iter=1)
    ref_u = [s._u[i].x.array_ro().copy() for i in range(3)]
    ref_p = s._p.x.array_ro().copy()
    tg2 = TaylorGreen(nu, 3)
    s2 = make_solver(make_mesh(3, 4), 2, tg2, dt)
    t = load_checkpoint(str(tmp_path / "chk"), s2)
    assert abs(t - 3 * dt) < 1e-15
    tg2.t_u, tg2.t_p = t, t - dt / 2
    for n in range(2):
        tg2.t_u += dt
        tg2.t_p += dt
        s2.solve(dt, nu, max_iter=1)
    for i in range(3):
        assert relerr(s2._u[i].x.array_ro(), ref_u[i], vscale(ref_u)) <= 1e-10
    assert relerr(s2._p.x.array_ro(), ref_p) <= 1e-9
    out = tmp_path / "state.vtu"
    write_vtu(str(out), s2._Vi[0][0], {"u": s2.u.x.array.reshape(-1, 3)})
    txt = out.read_text()
    assert txt.count("<DataArray") == 5 and 'Name="u"' in txt and txt.rstrip().endswith("</VTKFile>")


def test_foreign_mesh_goes_through_the_dolfinx_adapter(monkeypatch):
    """``FractionalStep_AB_CN(mesh=<DOLFINx mesh>)`` (fracstep.py:187-190,212): a mesh that is not the provider's is
    consumed through ``oasisx_b200.adapter`` -- here duck-typed DOLFINx objects (tests/fake_dolfinx.py) -- and the step
    gives the oracle's fields."""
    import sys

    import oasisx_b200 as oasisx
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
    lu = {"ksp_type": "preonly", "pc_type": "lu"}
    s = oasisx.FractionalStep_AB_CN(fmesh, ("Lagrange", 2), ("Lagrange", 1), bcs_u=bcs_u, bcs_p=[],
                                    solver_options={"tentative": lu, "pressure": lu, "scalar": lu}, options={"low_memory_version": False})
    assert s._foreign and s._lp is not None
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
