"""The host reference of the smoothed-aggregation multigrid (tests/amg_reference.py) on meshes without a geometric
hierarchy: the aggregation is a valid MIS(2) aggregation, and the smoothed prolongator and the Galerkin product keep
the constant null space of the pressure operator.  tests/test_gpu_amg.py holds the device to this reference."""
import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.csgraph import connected_components

import amg_reference as ref
from problems import jittered_mesh, l_shaped_mesh

MESHES = {"jittered3d_8": lambda: jittered_mesh(3, 8), "jittered3d_16": lambda: jittered_mesh(3, 16),
          "lshape2d_16": lambda: l_shaped_mesh(2, 16)}


@pytest.fixture(scope="module", params=list(MESHES))
def level(request):
    msh = MESHES[request.param]()
    A = ref.p1_stiffness(msh.geometry.x, msh.geometry.dofmap, msh.geometry.dim)
    agg, roots = ref.mis2_aggregate(A)
    P = ref.smoothed_prolongator(A, agg, 4.0 / 3.0 / 1.9)
    return A, agg, roots, P, ref.galerkin(A, P)


def test_fmix32_is_the_murmur3_finaliser():
    def py(h):
        h ^= h >> 16
        h = (h * 0x85EBCA6B) & 0xFFFFFFFF
        h ^= h >> 13
        h = (h * 0xC2B2AE35) & 0xFFFFFFFF
        return h ^ (h >> 16)

    xs = np.array([0, 1, 2, 12345, 0x9E3779B9, 0xFFFFFFFF], dtype=np.uint32)
    assert ref.fmix32(xs).tolist() == [py(int(v)) for v in xs]


def test_aggregates_partition_the_nodes(level):
    A, agg, roots, P, Ac = level
    assert agg.min() == 0 and (agg >= 0).all()
    assert np.array_equal(np.unique(agg), np.arange(roots.size))
    assert 2 * roots.size < A.shape[0]  # it does coarsen


def test_roots_are_at_least_three_apart(level):
    A, agg, roots, P, Ac = level
    S = ref.strength(A)
    S1 = (S + sp.identity(S.shape[0], format="csr")).tocsr()
    reach2 = (S1 @ S1).tocsr()
    within = reach2[roots][:, roots]
    assert within.nnz == roots.size  # every root reaches only itself within two hops


def test_aggregates_are_connected_and_hold_their_root(level):
    A, agg, roots, P, Ac = level
    assert np.array_equal(agg[roots], np.arange(roots.size))
    S = ref.strength(A).tocoo()
    inside = agg[S.row] == agg[S.col]
    G = sp.csr_matrix((np.ones(inside.sum()), (S.row[inside], S.col[inside])), shape=S.shape)
    n_comp, _ = connected_components(G, directed=False)
    assert n_comp == roots.size


def test_prolongator_and_galerkin_keep_the_constant(level):
    A, agg, roots, P, Ac = level
    assert np.abs(P @ np.ones(P.shape[1]) - 1.0).max() <= 1e-14
    assert np.abs(Ac @ np.ones(Ac.shape[0])).max() <= 1e-12 * np.abs(Ac.data).max()
    assert abs(Ac - Ac.T).max() <= 1e-14 * np.abs(Ac.data).max()


def test_second_level_aggregates_too(level):
    """The coarse operator is again a valid input: the reference coarsens it once more."""
    A, agg, roots, P, Ac = level
    agg2, roots2 = ref.mis2_aggregate(Ac)
    assert np.array_equal(np.unique(agg2), np.arange(roots2.size)) and roots2.size < Ac.shape[0]
