"""The smoothed-aggregation pressure multigrid on several ranks (pc_type gamg / hypre on meshes without a geometric
hierarchy): the global Ap gathered by global dof index, the same hierarchy on every rank, level 1 cut back to each
rank's owned rows.  The multi-rank cases run tests/amg_mr_worker.py under torch.distributed.run and are skipped on boxes
with fewer GPUs; the checks of the global dof ids run in one process."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

import amg_reference as ref

from oasisx_b200 import _lib as L
from problems import TaylorGreen, jittered_mesh, make_solver

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
GAMG = {"ksp_type": "cg", "pc_type": "gamg", "ksp_rtol": 1e-12}
LU = {"ksp_type": "preonly", "pc_type": "lu"}


def _ngpu():
    return L.load_library().b2_device_count()


def _launch(nranks, peer, port, *cases):
    if _ngpu() < nranks:
        pytest.skip(f"needs {nranks} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nranks}", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(HERE, "amg_mr_worker.py"), *cases]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=1500, env=dict(os.environ, B200_PEER=peer))
    assert res.returncode == 0, res.stdout[-4000:] + res.stderr[-4000:]
    assert res.stdout.count("MR_OK") == nranks
    print(res.stdout[-3000:])


@pytest.mark.parametrize("nranks,peer", [(2, "1"), (2, "0"), (4, "1"), (4, "0")])
def test_amg_on_several_ranks(nranks, peer):
    """Partition route (jittered 8^3, L-shape 16^2) against the single-rank hierarchy and iterations, adapter route
    against tests/amg_reference.py, replicated levels bitwise equal on every rank, 3 steps against the LU oracle."""
    _launch(nranks, peer, 29950 + 10 * nranks + int(peer), "partition-jittered", "partition-lshape", "adapter")


def test_amg_iterations_on_two_ranks():
    """Jittered 24^3 on 2 ranks: AMG-PCG needs at most a fifth of Jacobi-PCG's iterations, and within one of the
    single-rank AMG-PCG."""
    _launch(2, "1", 29995, "iters")


def _hierarchy_with_ids(msh, ids):
    """A solver set up with Jacobi, then the algebraic hierarchy built through the gathered path with global ids `ids`
    (None: the single-rank path)."""
    s = make_solver(msh, 1, TaylorGreen(0.01, msh.geometry.dim), 0.005,
                    solver_options={"tentative": LU, "scalar": LU, "pressure": dict(GAMG, pc_type="jacobi")})
    if ids is not None:
        s._ctx.set_pressure_global_ids(ids)
    s._ctx.pressure_amg_build()
    s._solver_p.updateOptions({"pc_type": "gamg"})
    levels, l = [], 1
    while True:
        try:
            info = s._ctx.pressure_mg_level_info(l)
        except L.B200Error:
            break
        levels.append((info, *(s._ctx.pressure_mg_get_level(l, w) for w in range(4))))
        l += 1
    return s, levels


def _bitwise(a, b):
    if sp.issparse(a):
        return all(np.array_equal(x, y) for x, y in ((a.indptr, b.indptr), (a.indices, b.indices))) and \
            np.array_equal(a.data.view(np.uint64), b.data.view(np.uint64))
    return np.array_equal(a, b)


def test_gathered_setup_on_one_rank():
    """The gathered set-up (global pairs, global CSR, row gather of level 1) on one GPU: with the identity as global ids
    it gives the single-rank hierarchy bit for bit; with a random permutation it is the reference hierarchy of the
    permuted matrix, with P_1 and the aggregates back in local order, and the V-cycle converges with it."""
    msh = jittered_mesh(3, 12, seed=6)
    s0, plain = _hierarchy_with_ids(msh, None)
    n = s0._Q.num_dofs
    s1, same = _hierarchy_with_ids(msh, np.arange(n))
    assert len(plain) == len(same) >= 1
    for a, b in zip(plain, same):
        assert a[0] == b[0] and all(_bitwise(x, y) for x, y in zip(a[1:], b[1:]))
    for l in (0, 1):
        assert s0._ctx.pressure_mg_level_info(l) == s1._ctx.pressure_mg_level_info(l)
    perm = np.random.default_rng(8).permutation(n)
    s2, levels = _hierarchy_with_ids(msh, perm)
    A = _csr(s2._Ap)
    Pm = sp.csr_matrix((np.ones(n), (perm, np.arange(n))), shape=(n, n))  # global row perm[i] = local row i
    Ag = sp.csr_matrix(Pm @ A @ Pm.T)
    Ag.sort_indices()
    ragg, _ = ref.mis2_aggregate(Ag)
    info0 = s2._ctx.pressure_mg_level_info(0)
    info1, A1, P1, R1, agg1 = levels[0]
    np.testing.assert_array_equal(agg1, ragg[perm])
    Pref = ref.smoothed_prolongator(Ag, ragg, info0["omega"])
    assert abs(P1 - Pref[perm]).max() <= 1e-14 * abs(Pref).max()
    Rt = sp.csr_matrix(P1.T)
    Rt.sort_indices()
    assert _bitwise(R1, Rt)
    assert abs(A1 - ref.galerkin(Ag, Pref)).max() <= 1e-13 * abs(A1).max()
    b = np.random.default_rng(9).uniform(-1.0, 1.0, n)
    b -= b.mean()
    its = {}
    for s in (s0, s2):
        s._solver_p.updateOptions({"ksp_rtol": 1e-10, "ksp_initial_guess_nonzero": False})
        x = np.zeros(n)
        assert s._ctx.ksp_solve(L.SOLVER_PRESSURE, L.MAT_AP, b, x) > 0
        assert np.linalg.norm(A @ x - b) <= 1e-9 * np.linalg.norm(b)
        its[s is s0] = s.stats().its_pressure
    assert its[False] <= 1.5 * its[True], its


def _csr(mat):
    ip, ix, v = mat.getValuesCSR()
    return sp.csr_matrix((v, ix, ip), shape=mat.getSize())


def test_global_ids_are_checked():
    s = make_solver(jittered_mesh(3, 4, seed=2), 1, TaylorGreen(0.01, 3), 0.005,
                    solver_options={"tentative": LU, "scalar": LU, "pressure": GAMG})
    assert s._mg_kind == "algebraic"
    ctx = s._ctx
    n = s._Q.num_dofs
    ids = np.random.default_rng(3).permutation(n)
    ctx.set_pressure_global_ids(ids)  # a permutation of 0 .. n-1 covers the global range once
    dup = ids.copy()
    dup[5] = dup[7]
    for bad, what in ((dup, "same global index twice"), (np.where(ids == 0, n, ids), "outside"),
                      (np.where(ids == 0, -1, ids), "outside"), (np.where(ids == 0, 1 << 31, ids), "outside")):
        with pytest.raises(L.B200Error, match=what):
            ctx.set_pressure_global_ids(bad)
    with pytest.raises(L.B200Error, match="one global index per local pressure dof"):
        ctx.set_pressure_global_ids(ids[:-1])
    # the context stays usable
    s.solve(0.005, 0.01, max_iter=1)
    assert s.stats().its_pressure > 0
