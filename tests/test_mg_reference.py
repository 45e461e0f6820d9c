"""The host restatement of the pressure V-cycle (tests/mg_reference.py) on its own: a symmetric positive definite
preconditioner on mean-free vectors, the Galerkin coarse correction when the first coarse level is solved exactly,
few PCG iterations, and the coarse P1 stiffness of a box equal to the Galerkin product.  CPU only."""
import numpy as np
import pytest
import scipy.sparse as sp

import mg_reference as ref
from problems import make_mesh

DEFAULT = dict(pre=1, post=1, coarse=16)
OMEGA = 0.85


def _vcycle(msh, mg_dense=True, **cfg):
    A, P, R = ref.box_levels(msh)
    c = dict(DEFAULT, **cfg)
    dense = ref.first_dense_level([a.shape[0] for a in A])
    return ref.VCycle(A, P, R, [OMEGA] * len(A), c["pre"], c["post"], c["coarse"], dense, mg_dense)


def _mean_free(n, seed):
    b = np.random.default_rng(seed).uniform(-1.0, 1.0, n)
    return b - b.mean()


@pytest.mark.parametrize("mg_dense", [True, False])
@pytest.mark.parametrize("nu", [1, 2])
def test_vcycle_is_spd_on_mean_free_vectors(nu, mg_dense):
    V = _vcycle(make_mesh(3, 8), mg_dense, pre=nu, post=nu)
    assert V.dense == (1 if mg_dense else None)
    n = V.A[0].shape[0]
    # orthonormal basis of the mean-free vectors: the columns of Q
    Q = np.linalg.qr(np.eye(n)[:, 1:] - 1.0 / n)[0]
    M = np.column_stack([V(Q[:, j]) for j in range(n - 1)])
    S = Q.T @ M
    assert abs(S - S.T).max() <= 1e-12 * abs(S).max()
    ev = np.linalg.eigvalsh(0.5 * (S + S.T))
    assert ev[0] > 1e-3 * ev[-1], (ev[0], ev[-1])


def test_exact_first_level_gives_the_galerkin_correction():
    """pre = post = 0 with level 1 solved exactly: V(b) = P_1 A_1^+ R_1 b, so the coarse residual R_1 (b - A V(b))
    vanishes and V(b) has no component outside the range of P_1."""
    V = _vcycle(make_mesh(3, 8), pre=0, post=0)
    assert V.dense == 1
    b = _mean_free(V.A[0].shape[0], 3)
    x = V(b)
    P, A1 = V.P[1], V.A[1].toarray()
    y = np.linalg.lstsq(A1, V.R[1] @ b, rcond=None)[0]
    y -= y.mean()  # A_1^+ g: the minimum-norm solution is mean free
    assert abs(x - P @ y).max() <= 1e-12 * abs(x).max()
    assert abs(V.R[1] @ (b - V.A[0] @ x)).max() <= 1e-12 * abs(b).max()


@pytest.mark.parametrize("mg_dense", [True, False])
def test_pcg_converges_in_few_iterations(mg_dense):
    V = _vcycle(make_mesh(3, 16), mg_dense)
    b = _mean_free(V.A[0].shape[0], 16)
    xs, its = ref.pcg(V.A[0], b, V, rtol=1e-10, maxit=100)
    assert its <= 20, its
    assert np.linalg.norm(b - V.A[0] @ xs[-1]) <= 1e-10 * np.linalg.norm(b)


@pytest.mark.parametrize("gdim,N", [(2, 16), (3, 8), (3, 16)])
def test_coarse_stiffness_is_the_galerkin_product(gdim, N):
    A, P, R = ref.box_levels(make_mesh(gdim, N))
    assert len(A) >= 3
    for l in range(1, len(A)):
        G = sp.csr_matrix(R[l] @ A[l - 1] @ P[l])
        assert abs(A[l] - G).max() <= 1e-13 * abs(A[l]).max(), l
        assert (R[l] != P[l].T).nnz == 0


def test_exact_coarse_solve_iterations_at_36():
    """3D N = 36 (levels 37^3, 19^3, 10^3; 10^3 = 1000 dofs is the first level with at most 5000): PCG iterations to
    rtol 1e-10 from a seeded mean-free right-hand side with the exact solve of the 10^3 level, and with 16 Jacobi
    sweeps there instead (what a sub-cycle that starts at the 19^3 level computes).  Computed on the host: 16 against
    18 iterations."""
    V = _vcycle(make_mesh(3, 36))
    assert [a.shape[0] for a in V.A] == [37**3, 19**3, 10**3] and V.dense == 2
    b = _mean_free(V.A[0].shape[0], 36)
    its = {}
    for dense in (True, False):
        xs, its[dense] = ref.pcg(V.A[0], b, V.with_(mg_dense=dense), rtol=1e-10, maxit=100)
        assert np.linalg.norm(b - V.A[0] @ xs[-1]) <= 1e-10 * np.linalg.norm(b)
    print("N = 36 PCG iterations: exact coarse solve", its[True], ", 16 coarse sweeps", its[False])
    assert its == {True: 16, False: 18}, its
