"""The pressure V-cycle on the device against its host restatement (tests/mg_reference.py), iterate by iterate.

``KSPSolver.solve`` on Ap with pc_type mg / gamg, a zero guess and ksp_max_it k returns the k-th PCG iterate; the first
is alpha V(b), so it pins the V-cycle itself: the fused first sweeps (k_cgz_init_x0, k_cgz_update_x0, k_mg_restrict),
the fused last sweep with r.z (k_mg_sweep_rz) or k_cgz_rz after it (no post-sweep), the single-block sub-cycle
(k_mg_small_cycle) and the buffer its result is taken from, and the exact solve of the dense level.  Iterates 2 and 3
replay the captured PCG body.  Ap and every coarse level are read back from the device, so only the cycle is under
test.  Each case also shows that the tolerance can tell a cycle with one sweep fewer, and one with the other coarse
treatment (dense solve against coarse sweeps), from the device's.

Also: the geometric coarse operators against the host P1 stiffness of the coarse meshes and the Galerkin product,
the dense flag, and recovery of the pressure solver after a solve with a NaN in its right-hand side."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

import mg_reference as ref
from oasisx_b200 import _lib as L
from oasisx_b200 import mesh as bmesh
from oasisx_b200 import multigrid as _mg
from problems import TaylorGreen, jittered_mesh, l_shaped_mesh, make_mesh, make_solver, relerr, vscale

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
LU = {"ksp_type": "preonly", "pc_type": "lu"}
MG = {"ksp_type": "cg", "pc_type": "mg", "ksp_rtol": 1e-12}
DEFAULT = (1, 1, 16, 0.85)


def _csr(mat):
    ip, ix, v = mat.getValuesCSR()
    return sp.csr_matrix((v, ix, ip), shape=mat.getSize())


def _deformed_box(N):
    """The unit box graded toward x = 0 in place (x -> x^2): lattice numbering kept, coordinates moved."""
    msh = bmesh.create_box(None, [[0.0, 0.0, 0.0], [1.0, 1.0, 1.0]], [N, N, N])
    msh.geometry.x[:, 0] **= 2
    return msh


def _solver(msh, pc="mg", cfg=DEFAULT):
    tg = TaylorGreen(0.01, msh.geometry.dim)
    mgopt = dict(zip(("nu_pre", "nu_post", "coarse_sweeps", "omega"), cfg))
    return make_solver(msh, 1, tg, 0.005, solver_options={"tentative": LU, "scalar": LU, "pressure": dict(MG, pc_type=pc)},
                       options={"multigrid": mgopt})


def _mean_free(n, seed):
    b = np.random.default_rng(seed).uniform(-1.0, 1.0, n)
    return b - b.mean()


def _iterate(s, b, k):
    """x_k of the device PCG from a zero guess (ksp_max_it k, a tolerance it cannot reach)."""
    s._solver_p.updateOptions({"ksp_max_it": k, "ksp_rtol": 1e-30, "ksp_initial_guess_nonzero": False})
    x = np.zeros(b.size)
    reason = s._ctx.ksp_solve(L.SOLVER_PRESSURE, L.MAT_AP, b, x)
    assert reason == -3, (k, reason)
    return x


def _rel(a, b):
    return abs(a - b).max() / abs(b).max()


def _check_iterates(s, V, A0, b, what):
    dev = [_iterate(s, b, k) for k in (1, 2, 3)]
    host = ref.pcg(A0, b, V, k=3)[0]
    for k, (xd, xr) in enumerate(zip(dev, host), start=1):
        err = _rel(xd, xr)
        assert err <= (1e-11 if k == 1 else 1e-10), (what, k, err)
    # the tolerance is not vacuous: one sweep fewer (post, or pre where there is no post-sweep), and the other coarse
    # treatment, are far from the device
    others = {"one post-sweep fewer": V.with_(post=V.post - 1)} if V.post else {"one pre-sweep fewer": V.with_(pre=V.pre - 1)}
    if V.dense is not None:
        others["coarse sweeps instead of the dense solve"] = V.with_(mg_dense=False)
    for name, W in others.items():
        x1 = ref.pcg(A0, b, W, k=1)[0][0]
        assert _rel(dev[0], x1) > 1e-6, (what, name)


def _check_cycle(s, pc_dense=(1, 0), cfg=DEFAULT, seed=0):
    """Iterates 1..3 against the restatement with mg_dense on and off."""
    ctx = s._ctx
    ctx.set_tuning("mg_dense", 1)
    A0 = _csr(s._Ap)
    V = ref.VCycle.from_context(ctx, A0, s._mg_levels, *cfg[:3])
    assert V.dense is not None
    b = _mean_free(A0.shape[0], seed)
    for on in pc_dense:
        ctx.set_tuning("mg_dense", on)
        _check_iterates(s, V.with_(mg_dense=bool(on)), A0, b, (cfg, on))
    ctx.set_tuning("mg_dense", 1)


BOXES = {"2d_16": lambda: make_mesh(2, 16), "2d_160": lambda: make_mesh(2, 160), "3d_8": lambda: make_mesh(3, 8),
         "3d_36": lambda: make_mesh(3, 36), "3d_48": lambda: make_mesh(3, 48), "deformed_16": lambda: _deformed_box(16)}


@pytest.mark.parametrize("name", list(BOXES))
def test_geometric_vcycle_and_coarse_operators(name):
    """Coarse operators against the P1 stiffness of box_hierarchy's coarse meshes (and, undeformed, against P^T A P),
    the dense flag on the first level with at most 5000 dofs only, then the iterates with mg_dense 1 and 0.  2D 160
    and 3D 36 have a level of 5000 < n <= 8192 dofs above the dense one."""
    msh = BOXES[name]()
    s = _solver(msh)
    assert s._mg_kind == "geometric"
    ctx = s._ctx
    from oasisx_b200 import fem as _fem

    deformed = _fem.is_deformed(msh)
    assert deformed == name.startswith("deformed")
    levels = _mg.box_hierarchy(msh, fine_x=msh.geometry.x if deformed else None)
    assert len(levels) == s._mg_levels
    A_prev = _csr(s._Ap)
    sizes = [A_prev.shape[0]]
    dense = []
    for l, (cm, _) in enumerate(levels, start=1):
        info = ctx.pressure_mg_level_info(l)
        A = ctx.pressure_mg_get_level(l, 0)
        H = ref.p1_stiffness(cm.geometry.x, cm.geometry.dofmap)
        assert abs(A - H).max() <= 1e-12 * abs(H).max(), (name, l)
        if not deformed:
            P = ctx.pressure_mg_get_level(l, 1)
            G = sp.csr_matrix(P.T @ A_prev @ P)
            assert abs(A - G).max() <= 1e-12 * abs(H).max(), (name, l)
        sizes.append(info["n"])
        if info["dense"]:
            dense.append(l)
        A_prev = A
    assert dense == [ref.first_dense_level(sizes)], (sizes, dense)
    _check_cycle(s)


CONFIGS = [DEFAULT, (2, 0, 3, 0.7), (1, 3, 1, 1.0), (3, 2, 2, 0.6)]


@pytest.mark.parametrize("cfg", CONFIGS, ids=lambda c: "-".join(map(str, c)))
def test_multigrid_settings(cfg):
    """3D 16 (levels 9^3, 5^3, 3^3; the sub-cycle runs with mg_dense 0): no post-sweep (k_cgz_rz), and sweep counts
    of both parities for the sub-cycle's result buffer."""
    s = _solver(make_mesh(3, 16), cfg=cfg)
    assert s._mg_kind == "geometric" and s._mg_levels == 3
    for l in range(s._mg_levels + 1):
        assert s._ctx.pressure_mg_level_info(l)["omega"] == cfg[3]
    _check_cycle(s, cfg=cfg, seed=1)


ALGEBRAIC = {"jittered3d_16": lambda: jittered_mesh(3, 16), "jittered3d_24": lambda: jittered_mesh(3, 24),
             "lshape2d_16": lambda: l_shaped_mesh(2, 16)}


@pytest.mark.parametrize("name", list(ALGEBRAIC))
def test_algebraic_vcycle(name):
    """Every level damped with its own 4 / (3 rho_hat), the hierarchy ends at its dense level."""
    s = _solver(ALGEBRAIC[name](), pc="gamg")
    assert s._mg_kind == "algebraic" and s._mg_levels >= 1
    assert s._ctx.pressure_mg_level_info(s._mg_levels)["dense"] == 1
    _check_cycle(s, seed=2)


def test_recovery_after_a_nan_right_hand_side():
    """A solve whose right-hand side holds a NaN stops with reason -9; the next solve on the same context is not
    affected by it: its first iterate is the restatement's and it converges."""
    s = _solver(make_mesh(3, 16))
    ctx = s._ctx
    A0 = _csr(s._Ap)
    V = ref.VCycle.from_context(ctx, A0, s._mg_levels, *DEFAULT[:3])
    b = _mean_free(A0.shape[0], 3)
    bad = b.copy()
    bad[7] = np.nan
    full = {"ksp_max_it": 200, "ksp_rtol": 1e-10, "ksp_initial_guess_nonzero": False}
    x1 = ref.pcg(A0, b, V, k=1)[0][0]
    for _ in range(2):
        s._solver_p.updateOptions(full)
        x = np.zeros(b.size)
        assert ctx.ksp_solve(L.SOLVER_PRESSURE, L.MAT_AP, b, x) == 2  # a few iterations: bodies run unpolled next time
        assert ctx.ksp_solve(L.SOLVER_PRESSURE, L.MAT_AP, bad, np.zeros(b.size)) == -9
        assert _rel(_iterate(s, b, 1), x1) <= 1e-11
        assert ctx.ksp_solve(L.SOLVER_PRESSURE, L.MAT_AP, bad, np.zeros(b.size)) == -9
        s._solver_p.updateOptions(full)
        x = np.zeros(b.size)
        assert ctx.ksp_solve(L.SOLVER_PRESSURE, L.MAT_AP, b, x) == 2
        assert np.linalg.norm(b - A0 @ x) <= 1e-10 * np.linalg.norm(b)


def test_time_step_after_a_nan_right_hand_side():
    """The same through a time step: a pressure solve with a NaN between two steps leaves the second step equal to
    that of a context that never saw it."""
    dt, nu = 0.005, 0.01
    tgs = [TaylorGreen(nu, 3), TaylorGreen(nu, 3)]
    ss = [make_solver(make_mesh(3, 8), 1, tg, dt, solver_options={"tentative": LU, "scalar": LU, "pressure": MG})
          for tg in tgs]
    n = ss[0]._Q.num_dofs
    bad = np.full(n, np.nan)
    for tg in tgs:
        tg.t_u, tg.t_p = 0.0, -dt / 2
    for step in range(3):
        if step:
            assert ss[0]._ctx.ksp_solve(L.SOLVER_PRESSURE, L.MAT_AP, bad, np.zeros(n)) == -9
        for s, tg in zip(ss, tgs):
            tg.t_u += dt
            tg.t_p += dt
            s.solve(dt, nu, max_iter=1)
        assert ss[0].stats().its_pressure > 0
        u = [[s._u[i].x.array_ro().copy() for i in range(3)] for s in ss]
        for i in range(3):
            assert relerr(u[0][i], u[1][i], vscale(u[1])) <= 1e-10, (step, i)
        assert relerr(ss[0]._p.x.array_ro(), ss[1]._p.x.array_ro()) <= 1e-10, step


def _ngpu():
    return L.load_library().b2_device_count()


@pytest.mark.parametrize("nranks,peer", [(2, "1"), (2, "0"), (4, "1"), (4, "0")])
def test_vcycle_on_several_ranks(nranks, peer):
    """tests/mg_mr_worker.py: x_1, x_2 of the partitioned problem against the single-rank restatement of the global
    one (geometric partition route at 16^3 and 36^3, slab-local provider at 16^3, algebraic route on jittered 8^3)."""
    if _ngpu() < nranks:
        pytest.skip(f"needs {nranks} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nranks}", "--master-addr",
           "127.0.0.1", "--master-port", str(29850 + 10 * nranks + int(peer)), os.path.join(HERE, "mg_mr_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=1500, env=dict(os.environ, B200_PEER=peer))
    assert res.returncode == 0, res.stdout[-4000:] + res.stderr[-4000:]
    assert res.stdout.count("MR_OK") == nranks
    print(res.stdout[-3000:])
