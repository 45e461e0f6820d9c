"""Host restatement of the smoothed-aggregation set-up of ``b2_pressure_amg_build`` (oasisx_b200/csrc/amg.cuh):
strength graph, MIS(2) aggregation, smoothed prolongator and Galerkin product, with the same key function and the same
synchronous rounds, so that it reproduces the device aggregates exactly.  The damping omega is an argument: the device
estimates rho(D^-1 A) by a power iteration this file does not repeat."""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp

OUT, UNDECIDED, ROOT = 0, 1, 2


def fmix32(h):
    """murmur3 finaliser on uint32."""
    h = np.asarray(h, dtype=np.uint32).copy()
    with np.errstate(over="ignore"):
        h ^= h >> np.uint32(16)
        h *= np.uint32(0x85EBCA6B)
        h ^= h >> np.uint32(13)
        h *= np.uint32(0xC2B2AE35)
        h ^= h >> np.uint32(16)
    return h


def keys(n: int) -> np.ndarray:
    """(fmix32(i ^ 0x9E3779B9), i) packed into one uint64 whose order is the lexicographic one (i < 2^30)."""
    i = np.arange(n, dtype=np.uint64)
    h = fmix32(np.arange(n, dtype=np.uint32) ^ np.uint32(0x9E3779B9)).astype(np.uint64)
    return (h << np.uint64(30)) | i


def strength(A: sp.csr_matrix) -> sp.csr_matrix:
    """j != i is a strong neighbour of i when a_ij != 0 (every stored nonzero coupling, threshold 0)."""
    A = sp.csr_matrix(A)
    rows = np.repeat(np.arange(A.shape[0]), np.diff(A.indptr))
    keep = (A.indices != rows) & (A.data != 0)
    S = sp.csr_matrix((np.ones(keep.sum()), (rows[keep], A.indices[keep])), shape=A.shape)
    S.sort_indices()
    return S


def _hop_max(S: sp.csr_matrix, v: np.ndarray) -> np.ndarray:
    """out_i = max(v_i, v_j over the strong neighbours j of i)."""
    out = v.copy()
    nz = np.flatnonzero(np.diff(S.indptr))
    if nz.size:
        m = np.maximum.reduceat(v[S.indices], S.indptr[nz])
        out[nz] = np.maximum(out[nz], m)
    return out


def mis2_aggregate(A) -> tuple[np.ndarray, np.ndarray]:
    """(aggregate of every node, root nodes in increasing order)."""
    S = strength(A)
    n = S.shape[0]
    k = keys(n)
    state = np.full(n, UNDECIDED, dtype=np.uint64)
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
    # pass 2: the pass-1 neighbour with the largest key
    rows = np.repeat(np.arange(n), np.diff(S.indptr))
    cand = np.where(agg1[S.indices] >= 0, k[S.indices] + np.uint64(1), np.uint64(0))
    best = np.zeros(n, dtype=np.uint64)
    np.maximum.at(best, rows, cand)
    agg = agg1.copy()
    left = agg < 0
    assert (best[left] > 0).all(), "MIS(2) left a node unassigned"
    j = (best[left] - np.uint64(1)) & np.uint64((1 << 30) - 1)
    agg[left] = agg1[j.astype(np.int64)]
    return agg, roots


def tentative(agg: np.ndarray) -> sp.csr_matrix:
    n, nc = agg.size, int(agg.max()) + 1
    return sp.csr_matrix((np.ones(n), (np.arange(n), agg)), shape=(n, nc))


def smoothed_prolongator(A, agg: np.ndarray, omega: float) -> sp.csr_matrix:
    """P = (I - omega D^-1 A) T."""
    A = sp.csr_matrix(A)
    Dinv = sp.diags(1.0 / A.diagonal())
    P = (sp.identity(A.shape[0], format="csr") - omega * (Dinv @ A)) @ tentative(agg)
    P = sp.csr_matrix(P)
    P.sort_indices()
    return P


def galerkin(A, P) -> sp.csr_matrix:
    Ac = sp.csr_matrix(P.T @ (A @ P))
    Ac.sort_indices()
    return Ac


def p1_stiffness(x: np.ndarray, cells: np.ndarray, gdim: int) -> sp.csr_matrix:
    """The P1 stiffness matrix (the pressure operator Ap without boundary conditions) of a simplex mesh."""
    X = x[cells][:, :, :gdim]
    J = np.transpose(X[:, 1:] - X[:, :1], (0, 2, 1))  # (cells, gdim, gdim), columns = edge vectors
    ref = np.vstack([-np.ones(gdim), np.eye(gdim)])  # reference gradients of the barycentric functions
    G = ref @ np.linalg.inv(J)  # (cells, gdim + 1, gdim): physical gradients as rows
    vol = np.abs(np.linalg.det(J)) / np.prod(np.arange(1, gdim + 1))
    Ke = vol[:, None, None] * (G @ np.transpose(G, (0, 2, 1)))
    nd = gdim + 1
    r = np.repeat(cells, nd, axis=1).ravel()
    c = np.tile(cells, (1, nd)).ravel()
    A = sp.csr_matrix((Ke.ravel(), (r, c)), shape=(x.shape[0],) * 2)
    A.sort_indices()
    return A
