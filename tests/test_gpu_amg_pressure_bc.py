"""The algebraic pressure multigrid (pc_type gamg / hypre) on problems with PressureBC outlets: the pressure Dirichlet
dofs stay out of every aggregate and the dense level is solved without the null-space shift.

- The device hierarchy against tests/amg_mask_reference.py with the Dirichlet mask (jittered channel, provider-box channel,
  DOLFINx adapter): aggregates bit for bit, P, R = P^T, A_l = P_l^T A_{l-1} P_l, two contexts bitwise equal.
- PCG iterates 1..3 against tests/mg_reference.py with the unshifted dense factor (amg_mask_reference.unshifted); the tolerance tells it apart from the
  shifted factor and from the hierarchy that keeps every Dirichlet dof as a singleton aggregate.
- An outlet face of more than 5000 dofs, which the singleton hierarchy can never coarsen to the dense level.
- Time steps of the open channel against the LU oracle; dp stays exactly 0 on the Dirichlet dofs.
- KSPSolver.solve with a right-hand side that is nonzero on Dirichlet rows; iterations against Jacobi; dispatch."""
import logging

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

import amg_mask_reference as ref
import amg_reference
import mg_reference as mgref
from channel_problem import GAMG, LU, channel
from oasisx_b200 import _lib as L
from oasisx_b200 import mesh as bmesh
from problems import jittered_mesh, l_shaped_mesh, make_mesh, relerr, vscale

pytestmark = pytest.mark.gpu

CFG = (1, 1, 16)


def _csr(mat):
    ip, ix, v = mat.getValuesCSR()
    return sp.csr_matrix((v, ix, ip), shape=mat.getSize())


def _mask(s):
    pdofs = np.unique(np.concatenate([b.bc.dofs for b in s._bcs_p]))
    mask = np.zeros(s._nQ_owned, dtype=bool)
    mask[pdofs[pdofs < s._nQ_owned]] = True
    return mask


def _rel(a, b):
    return abs(a - b).max() / abs(b).max()


def _hierarchy(s):
    ctx = s._ctx
    return [(ctx.pressure_mg_level_info(l - 1), ctx.pressure_mg_level_info(l), ctx.pressure_mg_get_level(l, 3),
             *(ctx.pressure_mg_get_level(l, w) for w in (0, 1, 2))) for l in range(1, s._mg_levels + 1)]


def _same_bits(m, n):
    return (np.array_equal(m.indptr, n.indptr) and np.array_equal(m.indices, n.indices)
            and np.array_equal(m.data.view(np.uint64), n.data.view(np.uint64)))


REF_CASES = {"jittered3d_4": lambda mp: channel(jittered_mesh(3, 4, seed=5)),
             "jittered3d_12": lambda mp: channel(jittered_mesh(3, 12, seed=5)),
             "box3d_12": lambda mp: channel(make_mesh(3, 12)),
             "adapter_jittered3d_10": lambda mp: channel(jittered_mesh(3, 10, seed=2), foreign=mp)}


@pytest.mark.parametrize("name", list(REF_CASES))
def test_hierarchy_equals_the_reference(name, monkeypatch):
    s, _, _ = REF_CASES[name](monkeypatch)
    assert s._mg_kind == "algebraic" and s._mg_levels >= 1
    A = _csr(s._Ap)
    mask = _mask(s)
    assert mask.sum() > 0 and np.array_equal(A.diagonal()[mask], np.ones(mask.sum()))
    levels = _hierarchy(s)
    for l, (info_f, info, agg, Ac, P, R) in enumerate(levels, start=1):
        assert info["algebraic"] == 1 and info["n"] == Ac.shape[0] == P.shape[1]
        ragg, _ = ref.mis2_aggregate(A, mask if l == 1 else None)
        np.testing.assert_array_equal(agg, ragg, err_msg=f"aggregates of level {l}")
        if l == 1:
            assert (agg[mask] == -1).all() and (agg[~mask] >= 0).all()
            assert not P[mask].toarray().any()  # zero rows of P at the Dirichlet dofs
        assert _rel(P, ref.smoothed_prolongator(A, ragg, info_f["omega"])) <= 1e-14, l
        Rt = sp.csr_matrix(P.T)
        Rt.sort_indices()
        assert np.array_equal(R.indptr, Rt.indptr) and np.array_equal(R.indices, Rt.indices) and np.array_equal(R.data, Rt.data)
        assert _rel(Ac, sp.csr_matrix(P.T @ (A @ P))) <= 1e-13, l
        if Ac.shape[0] <= 3000:
            assert np.linalg.eigvalsh(Ac.toarray()).min() > 0, l  # no null space left
        A = Ac
    assert levels[-1][1]["dense"] == 1
    s2, _, _ = REF_CASES[name](monkeypatch)
    assert _same_bits(_csr(s._Ap), _csr(s2._Ap))
    for a, b in zip(levels, _hierarchy(s2)):
        assert a[0] == b[0] and a[1] == b[1] and np.array_equal(a[2], b[2])
        assert all(_same_bits(m, n) for m, n in zip(a[3:], b[3:]))


def _iterate(s, b, k):
    s._solver_p.updateOptions({"ksp_max_it": k, "ksp_rtol": 1e-30, "ksp_initial_guess_nonzero": False})
    x = np.zeros(b.size)
    assert s._ctx.ksp_solve(L.SOLVER_PRESSURE, L.MAT_AP, b, x) == -3
    return x


def _check_iterates(s, seed=0):
    """Device iterates 1..3 against the unshifted reference; the shifted dense factor and the singleton-aggregate
    hierarchy are both far from the device's first iterate."""
    A0 = _csr(s._Ap)
    mask = _mask(s)
    shifted = mgref.VCycle.from_context(s._ctx, A0, s._mg_levels, *CFG)
    V = ref.unshifted(shifted)
    assert V.dense is not None
    b = np.random.default_rng(seed).uniform(-1.0, 1.0, A0.shape[0])
    b[mask] = 0.0  # as b2 in a time step
    dev = [_iterate(s, b, k) for k in (1, 2, 3)]
    for k, (xd, xr) in enumerate(zip(dev, mgref.pcg(A0, b, V, k=3)[0]), start=1):
        assert _rel(xd, xr) <= (1e-11 if k == 1 else 1e-10), (k, _rel(xd, xr))
        assert not xd[mask].any()
    As, Ps, _, om = ref.hierarchy(A0, None)
    dense = mgref.first_dense_level([a.shape[0] for a in As])
    singleton = ref.unshifted(mgref.VCycle(As, Ps, [None] + [sp.csr_matrix(p.T) for p in Ps[1:]], om, *CFG, dense))
    for name, W in (("shifted dense solve", shifted), ("singleton aggregates", singleton)):
        assert _rel(dev[0], mgref.pcg(A0, b, W, k=1)[0][0]) > 1e-6, name
    return V


VCYCLE_CASES = {"jittered3d_16": lambda: jittered_mesh(3, 16, seed=3), "box3d_16": lambda: make_mesh(3, 16),
                "lshape2d_48": lambda: l_shaped_mesh(2, 48, seed=1)}


@pytest.mark.parametrize("name", list(VCYCLE_CASES))
def test_vcycle_iterates(name):
    s, _, _ = channel(VCYCLE_CASES[name]())
    assert s._mg_kind == "algebraic" and s._ctx.pressure_mg_level_info(s._mg_levels)["dense"] == 1
    _check_iterates(s)


def test_outlet_face_above_the_dense_threshold():
    """A 6 x 72 x 72 box with the outlet on its 73 x 73 face: 5329 Dirichlet dofs.  With them excluded the hierarchy
    reaches a dense level; kept as singleton aggregates, no level ever gets below 5000 dofs."""
    msh = bmesh.create_box(None, [[-1.0, -1.0, -1.0], [1.0, 1.0, 1.0]], [6, 72, 72])
    s, _, _ = channel(msh)
    assert s._mg_kind == "algebraic" and _mask(s).sum() == 73 * 73
    sizes = [s._ctx.pressure_mg_level_info(l)["n"] for l in range(s._mg_levels + 1)]
    assert min(sizes[1:]) <= 5000 and s._ctx.pressure_mg_level_info(s._mg_levels)["dense"] == 1, sizes
    A0 = _csr(s._Ap)
    As, _, _, _ = ref.hierarchy(A0, None, omega=lambda a: 4.0 / 3.0 / 2.0)
    assert min(a.shape[0] for a in As[1:]) > 5000, [a.shape[0] for a in As]
    _check_iterates(s, seed=1)


STEP_CASES = {"3d": dict(gdim=3), "3d_low_memory": dict(gdim=3, low_memory=True),
              "3d_rotational": dict(gdim=3, rotational=True), "2d": dict(gdim=2)}


@pytest.mark.parametrize("name", list(STEP_CASES))
def test_time_steps_match_oracle(name):
    kw = dict(STEP_CASES[name])
    gdim = kw.pop("gdim")
    msh = jittered_mesh(3, 6, seed=5) if gdim == 3 else jittered_mesh(2, 16, seed=5)
    s, o, inlet = channel(msh, deg=2, oracle=True, **kw)
    assert s._mg_kind == "algebraic" and s._mg_levels >= 1
    mask = _mask(s)
    dt, nu = 0.01, 0.5
    for n in range(2):
        inlet.t += dt
        s.solve(dt, nu, max_iter=2, max_error=1e-30)
        o.solve(dt, nu, max_iter=2, max_error=1e-30)
        assert s.stats().its_pressure > 0
        assert not s._dp.x.array_ro()[: s._nQ_owned][mask].any()
        for i in range(gdim):
            assert relerr(s._u[i].x.array_ro(), o.u[i], vscale(o.u)) <= 1e-8, (n, i)
        assert relerr(s._p.x.array_ro(), o.p) <= 1e-8, n
    assert max(np.abs(p).max() for p in o.p_surf) > 1e-3


def test_ksp_solve_with_a_nonzero_dirichlet_right_hand_side():
    """On Dirichlet rows the V-cycle acts as omega (2 - omega) times the identity: still SPD, so PCG converges through
    the multigrid path to the solution of Ap x = b."""
    s, _, _ = channel(jittered_mesh(3, 16, seed=3))
    A = _csr(s._Ap)
    mask = _mask(s)
    b = np.random.default_rng(7).uniform(-1.0, 1.0, A.shape[0])
    assert np.abs(b[mask]).min() > 0
    its = {}
    for pc in ("gamg", "jacobi"):
        s._solver_p.updateOptions({"pc_type": pc, "ksp_rtol": 1e-10, "ksp_max_it": 1000, "ksp_initial_guess_nonzero": False})
        x = np.zeros(b.size)
        assert s._ctx.ksp_solve(L.SOLVER_PRESSURE, L.MAT_AP, b, x) > 0
        its[pc] = s.stats().its_pressure
        xs = spla.spsolve(A.tocsc(), b)
        assert np.abs(x - xs).max() <= 1e-8 * np.abs(xs).max(), pc
    assert 5 * its["gamg"] <= its["jacobi"], its


def test_iterations_against_jacobi():
    """24^3 jittered channel, seeded right-hand side zero on the outlet, rtol 1e-10: gamg needs at most a fifth of
    Jacobi's pressure iterations."""
    s, _, _ = channel(jittered_mesh(3, 24, seed=1))
    A = _csr(s._Ap)
    b = np.random.default_rng(24).uniform(-1.0, 1.0, A.shape[0])
    b[_mask(s)] = 0.0
    its = {}
    for pc in ("gamg", "jacobi"):
        s._solver_p.updateOptions({"pc_type": pc, "ksp_rtol": 1e-10, "ksp_max_it": 2000, "ksp_initial_guess_nonzero": False})
        x = np.zeros(b.size)
        assert s._ctx.ksp_solve(L.SOLVER_PRESSURE, L.MAT_AP, b, x) > 0
        its[pc] = s.stats().its_pressure
        assert np.linalg.norm(A @ x - b) <= 1e-9 * np.linalg.norm(b)
    print("iterations", its)
    assert 5 * its["gamg"] <= its["jacobi"], its


def test_dispatch(caplog):
    """Provider box with a PressureBC: gamg and hypre take the algebraic hierarchy, mg keeps Jacobi and says so.
    Without PressureBCs the algebraic hierarchy is the unmasked one."""
    for pc in ("gamg", "hypre"):
        s, _, _ = channel(make_mesh(3, 8), pressure=dict(GAMG, pc_type=pc))
        assert s._mg_kind == "algebraic" and s._mg_levels >= 1, pc
    with caplog.at_level(logging.WARNING, logger="oasisx"):
        s, _, _ = channel(make_mesh(3, 8), pressure=dict(GAMG, pc_type="mg"))
    assert s._mg_levels == 0 and s._mg_kind is None
    assert any("PressureBC" in r.getMessage() and "Jacobi" in r.getMessage() for r in caplog.records)
    s.solve(0.01, 0.5, max_iter=1)
    assert s.stats().its_pressure > 0
    from test_gpu_amg import _gamg_solver

    s = _gamg_solver(jittered_mesh(3, 8))
    A = _csr(s._Ap)
    agg = s._ctx.pressure_mg_get_level(1, 3)
    np.testing.assert_array_equal(agg, amg_reference.mis2_aggregate(A)[0])
    np.testing.assert_array_equal(agg, ref.mis2_aggregate(A, np.zeros(A.shape[0], dtype=bool))[0])
