"""The host reference of the smoothed-aggregation multigrid with a Dirichlet mask (tests/amg_mask_reference.py, built
on tests/amg_reference.py) on a pressure operator with
Dirichlet dofs (identity rows and columns, as Ap is assembled with PressureBCs): the Dirichlet dofs stay out of every
aggregate, P is zero on their rows, the coarse operators are SPD with no isolated row, an empty mask changes nothing,
and PCG with the V-cycle (tests/mg_reference.py) needs the iterations the design was chosen on.
tests/test_gpu_amg_pressure_bc.py holds the device to this reference."""
import numpy as np
import pytest
import scipy.sparse as sp

import amg_mask_reference as ref
import amg_reference
import mg_reference as mgref
from problems import jittered_mesh, l_shaped_mesh, make_mesh


def _outlet(msh):
    """Ap with Dirichlet dofs on the x = 1 face (x = -1 for the L-shape, whose x = 1 side is partly missing)."""
    x = msh.geometry.x
    side = -1.0 if msh.geometry.dim == 2 else 1.0
    bc = np.flatnonzero(np.isclose(x[:, 0], side))
    A = ref.with_dirichlet(ref.p1_stiffness(x, msh.geometry.dofmap, msh.geometry.dim), bc)
    mask = np.zeros(A.shape[0], dtype=bool)
    mask[bc] = True
    return A, mask


MESHES = {"box3d_12": lambda: make_mesh(3, 12), "jittered3d_10": lambda: jittered_mesh(3, 10, seed=5),
          "lshape2d_24": lambda: l_shaped_mesh(2, 24)}


@pytest.fixture(scope="module", params=list(MESHES))
def problem(request):
    A, mask = _outlet(MESHES[request.param]())
    return A, mask, ref.hierarchy(A, mask)


def test_operator_has_identity_dirichlet_rows_and_columns(problem):
    A, mask, _ = problem
    D = A.toarray()
    assert mask.sum() > 0
    assert np.array_equal(D[mask][:, mask], np.eye(mask.sum()))
    assert not D[mask][:, ~mask].any() and not D[~mask][:, mask].any()
    assert (np.diff(A.indptr)[mask] > 1).all()  # the zeroed entries stay stored, as on the device


def test_empty_mask_is_the_unmasked_aggregation(problem):
    A, mask, _ = problem
    agg, roots = amg_reference.mis2_aggregate(A)
    for empty in (None, np.zeros(A.shape[0], dtype=bool)):
        agg2, roots2 = ref.mis2_aggregate(A, empty)
        assert np.array_equal(agg, agg2) and np.array_equal(roots, roots2)
    # unmasked, every Dirichlet dof is an isolated node and so a singleton aggregate of its own
    assert all((agg == agg[i]).sum() == 1 for i in np.flatnonzero(mask))


def test_dirichlet_dofs_join_no_aggregate(problem):
    A, mask, (As, Ps, aggs, om) = problem
    agg = aggs[1]
    assert (agg[mask] == -1).all() and (agg[~mask] >= 0).all()
    assert np.array_equal(np.unique(agg[~mask]), np.arange(As[1].shape[0]))
    T = ref.tentative(agg)
    assert np.array_equal(np.diff(T.indptr), (~mask).astype(int))


def test_prolongator_is_zero_on_dirichlet_rows(problem):
    A, mask, (As, Ps, aggs, om) = problem
    P = Ps[1]
    assert not P[mask].toarray().any()
    assert np.abs(P[~mask] @ np.ones(P.shape[1])).min() > 0  # interior rows still interpolate


def test_coarse_operators_are_spd_without_isolated_rows(problem):
    A, mask, (As, Ps, aggs, om) = problem
    assert len(As) >= 2
    for l, Ac in enumerate(As[1:], start=1):
        D = Ac.toarray()
        assert np.abs(D - D.T).max() <= 1e-14 * np.abs(D).max(), l
        assert np.linalg.eigvalsh(D).min() > 0, l
        off = D - np.diag(np.diag(D))
        assert (np.abs(off).max(axis=1) > 0).all(), l  # no Dirichlet singleton is carried to a coarse level
        assert np.allclose(D, (Ps[l].T @ As[l - 1] @ Ps[l]).toarray(), rtol=0, atol=1e-13 * np.abs(D).max())


# Kuhn box [-1,1]^3, Dirichlet dofs on x = 1, seeded right-hand side zero there, rtol 1e-10, V(1,1), exact solve of the
# first level of at most 5000 dofs: (Jacobi-PCG, level sizes with the mask, its unshifted, its shifted, level sizes
# without the mask)
TABLE = {16: (151, [4913, 446], 18, 21, [4913, 735]), 24: (223, [15625, 883], 24, 26, [15625, 1508])}


@pytest.mark.parametrize("N", list(TABLE))
def test_host_iteration_counts(N):
    """Excluding the Dirichlet dofs gives a smaller dense level than keeping them as singletons; the unshifted exact
    solve beats the null-space shift, which is wrong once Ap is nonsingular."""
    jac, sizes, its, its_shift, sizes_singleton = TABLE[N]
    msh = make_mesh(3, N)
    A, mask = _outlet(msh)
    b = np.random.default_rng(0).standard_normal(A.shape[0])
    b[mask] = 0.0
    assert mgref.pcg(A, b, lambda r: r / A.diagonal(), rtol=1e-10)[1] == jac
    got = {}
    for name, m in (("excluded", mask), ("singleton", None)):
        As, Ps, aggs, om = ref.hierarchy(A, m)
        n = [a.shape[0] for a in As]
        dense = mgref.first_dense_level(n)
        Rs = [None] + [sp.csr_matrix(p.T) for p in Ps[1:]]
        V = mgref.VCycle(As, Ps, Rs, om, 1, 1, 16, dense)
        got[name] = (n, {s: mgref.pcg(A, b, V if s else ref.unshifted(V), rtol=1e-10)[1] for s in (False, True)})
    (n, it), (n_s, _) = got["excluded"], got["singleton"]
    assert n == sizes and n_s == sizes_singleton, got
    assert abs(it[False] - its) <= 1 and abs(it[True] - its_shift) <= 1, got
    assert it[False] < it[True], got
    assert 5 * it[False] <= jac
