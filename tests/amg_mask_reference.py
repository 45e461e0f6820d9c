"""Host restatement of the smoothed-aggregation set-up of ``b2_pressure_amg_build`` on a pressure operator with
Dirichlet dofs, built on tests/amg_reference.py: an exclusion mask of the fine level keeps nodes out of every
aggregate (they start out of the MIS, are never roots, keep aggregate -1, and get an empty row of T), and the dense
level of such a hierarchy is factored without the null-space shift.  Without a mask every function here gives what
tests/amg_reference.py and tests/mg_reference.py give."""
from __future__ import annotations

import numpy as np
import scipy.linalg as sla
import scipy.sparse as sp

from amg_reference import OUT, ROOT, UNDECIDED, _hop_max, galerkin, keys, p1_stiffness, strength  # noqa: F401


def mis2_aggregate(A, exclude=None) -> tuple[np.ndarray, np.ndarray]:
    """`amg_reference.mis2_aggregate` with `exclude`, a boolean mask of nodes that start out of the MIS, are never
    roots and keep aggregate -1 (None: none).  Returns (aggregate of every node, root nodes in increasing order)."""
    S = strength(A)
    n = S.shape[0]
    k = keys(n)
    excl = np.zeros(n, dtype=bool) if exclude is None else np.asarray(exclude, dtype=bool)
    state = np.where(excl, OUT, UNDECIDED).astype(np.uint64)
    while (state == UNDECIDED).any():  # synchronous rounds on the values at the start of the round
        t0 = (state << np.uint64(62)) | k
        m2 = _hop_max(S, _hop_max(S, t0))
        und = state == UNDECIDED
        root = und & (m2 == t0)
        out = und & ~root & ((m2 >> np.uint64(62)) == ROOT)
        state[root] = ROOT
        state[out] = OUT
    roots = np.flatnonzero(state == ROOT)
    rid = np.full(n, -1, dtype=np.int64)
    rid[roots] = np.arange(roots.size)
    # pass 1: roots and their neighbours (a neighbour sees exactly one root)
    agg1 = rid.copy()
    Sr = S[:, roots].tocsr()
    has = np.diff(Sr.indptr) > 0
    sel = has & (agg1 < 0)
    agg1[sel] = rid[roots[Sr.indices[Sr.indptr[:-1][sel]]]]
    # pass 2: the pass-1 neighbour with the largest key; excluded nodes keep -1
    rows = np.repeat(np.arange(n), np.diff(S.indptr))
    cand = np.where(agg1[S.indices] >= 0, k[S.indices] + np.uint64(1), np.uint64(0))
    best = np.zeros(n, dtype=np.uint64)
    np.maximum.at(best, rows, cand)
    agg = agg1.copy()
    left = (agg < 0) & ~excl
    assert (best[left] > 0).all(), "MIS(2) left a node unassigned"
    j = (best[left] - np.uint64(1)) & np.uint64((1 << 30) - 1)
    agg[left] = agg1[j.astype(np.int64)]
    return agg, roots


def tentative(agg: np.ndarray) -> sp.csr_matrix:
    """T[i, agg_i] = 1; the row of a node with aggregate -1 is empty."""
    n, nc = agg.size, int(agg.max()) + 1
    kept = np.flatnonzero(agg >= 0)
    return sp.csr_matrix((np.ones(kept.size), (kept, agg[kept])), shape=(n, nc))


def smoothed_prolongator(A, agg: np.ndarray, omega: float) -> sp.csr_matrix:
    """P = (I - omega D^-1 A) T, zero on the rows of excluded nodes."""
    A = sp.csr_matrix(A)
    Dinv = sp.diags(1.0 / A.diagonal())
    P = sp.csr_matrix((sp.identity(A.shape[0], format="csr") - omega * (Dinv @ A)) @ tentative(agg))
    P.sort_indices()
    return P


def with_dirichlet(A, dofs) -> sp.csr_matrix:
    """`A` with the rows and columns of `dofs` zeroed and a unit diagonal there, the stored pattern kept: the pressure
    operator Ap as assembled with pressure Dirichlet dofs."""
    A = sp.csr_matrix(A, dtype=np.float64, copy=True)
    A.sort_indices()
    bc = np.zeros(A.shape[0], dtype=bool)
    bc[np.asarray(dofs)] = True
    rows = np.repeat(np.arange(A.shape[0]), np.diff(A.indptr))
    hit = bc[rows] | bc[A.indices]
    A.data[hit] = np.where(rows[hit] == A.indices[hit], 1.0, 0.0)
    return A


def damping(A) -> float:
    """4 / (3 rho(D^-1 A)) with rho from scipy (the device estimates it by a power iteration)."""
    from scipy.sparse.linalg import eigsh

    d = 1.0 / np.sqrt(sp.csr_matrix(A).diagonal())
    As = sp.diags(d) @ A @ sp.diags(d)
    rho = eigsh(As, k=1, which="LA", return_eigenvectors=False)[0] if A.shape[0] > 50 else np.linalg.eigvalsh(As.toarray())[-1]
    return 4.0 / (3.0 * rho)


def hierarchy(A, exclude=None, dense_max: int = 5000, max_levels: int = 15, omega=damping):
    """The levels ``b2_pressure_amg_build`` builds from `A`: (A_l, P_l, agg_l, omega_l) with A[0] = A and P[0], agg[0]
    None, coarsened until a level has at most `dense_max` dofs, the coarsening ratio drops below 2, or `max_levels`
    coarse levels.  `exclude` masks the fine level only."""
    A = [sp.csr_matrix(A)]
    P, agg, om = [None], [None], [omega(A[0])]
    while len(A) <= max_levels:
        n = A[-1].shape[0]
        a, _ = mis2_aggregate(A[-1], exclude if len(A) == 1 else None)
        nc = int(a.max()) + 1
        if nc <= 0 or nc >= n:
            break
        p = smoothed_prolongator(A[-1], a, om[-1])
        A.append(galerkin(A[-1], p))
        P.append(p)
        agg.append(a)
        om.append(omega(A[-1]))
        if nc <= dense_max or 2 * nc > n:
            break
    return A, P, agg, om


def unshifted(V):
    """A copy of the host V-cycle `V` (tests/mg_reference.VCycle) whose dense level is factored as A itself instead of
    A + alpha e e^T: the device's exact solve on an algebraic hierarchy of a pressure with Dirichlet dofs."""
    W = V.with_()
    if W.dense is not None:
        W._chol = sla.cho_factor(W.A[W.dense].toarray())
    return W
