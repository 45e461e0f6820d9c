"""Host restatement of the pressure multigrid preconditioner (oasisx_b200/csrc/mg.cuh, ``mg_vcycle`` and
``pcg_mg_solve`` in b200ipcs.cu) in float64: damped-Jacobi V-cycle over a given hierarchy, the exact solve of the dense
level, and the PCG recurrence of the ``k_cgz_*`` kernels with z = V(r).

The device fuses and reorders these steps (first sweeps written by the kernel that produced the right-hand side, r.z
fused into the last post-sweep, the small end of the hierarchy in one single-block kernel whose result buffer depends
on the parity of the sweep counts); none of that changes the arithmetic beyond rounding, so the device iterates must
agree with these to a few ulps times the conditioning.  The GPU tests hold the device to this file."""
from __future__ import annotations

import numpy as np
import scipy.linalg as sla
import scipy.sparse as sp

import amg_reference as _amg
from oasisx_b200 import multigrid as _mg

DENSE_MAX = 5000  # b2_ctx::mg_dense_max: the first coarse level with at most this many dofs is solved exactly


def p1_stiffness(x: np.ndarray, cells: np.ndarray) -> sp.csr_matrix:
    """The P1 stiffness matrix of a simplex mesh in its node numbering (gradients of the barycentric coordinates)."""
    cells = np.asarray(cells)
    return _amg.p1_stiffness(np.asarray(x), cells, cells.shape[1] - 1)


def first_dense_level(sizes, dense_max: int = DENSE_MAX):
    """Index (>= 1) of the first coarse level with at most `dense_max` dofs; `sizes[l]` is the size of level l (level
    0 the fine level, which is never solved exactly).  None: no such level."""
    for l, n in enumerate(sizes):
        if l >= 1 and n <= dense_max:
            return l
    return None


class VCycle:
    """V(l, b) on the hierarchy ``A[0..L]`` with ``P[l]`` (level l-1 x level l) and ``R[l]`` (level l x level l-1) for
    l >= 1 (``P[0]``, ``R[0]`` unused).  ``omega[l]``: damping of level l.  ``dense``: index of the exactly solved level
    (None: none), used while ``mg_dense`` is true; otherwise the coarsest level gets ``coarse`` sweeps from zero."""

    def __init__(self, A, P, R, omega, pre: int, post: int, coarse: int, dense=None, mg_dense: bool = True):
        self.A = [sp.csr_matrix(a, dtype=np.float64) for a in A]
        self.P, self.R = list(P), list(R)
        self.omega = [float(w) for w in omega]
        self.pre, self.post, self.coarse = int(pre), int(post), int(coarse)
        self.dense = dense if mg_dense else None
        self.dinv = [1.0 / a.diagonal() for a in self.A]
        self._chol = None
        if self.dense is not None:
            Ad = self.A[self.dense].toarray()
            alpha = Ad[0, 0] / Ad.shape[0]  # the device's 1 / (dinv_0 n)
            self._chol = sla.cho_factor(Ad + alpha)

    @classmethod
    def from_context(cls, ctx, A0, n_levels: int, pre: int, post: int, coarse: int, mg_dense: bool = True):
        """The hierarchy a context holds: fine operator `A0` (read back by the caller), coarse A_l, P_l, R_l, the damping
        and the dense flag of every level from ``pressure_mg_level_info`` (dense as reported with mg_dense on)."""
        A, P, R, omega, dense = [A0], [None], [None], [ctx.pressure_mg_level_info(0)["omega"]], None
        for l in range(1, n_levels + 1):
            info = ctx.pressure_mg_level_info(l)
            A.append(ctx.pressure_mg_get_level(l, 0))
            P.append(ctx.pressure_mg_get_level(l, 1))
            R.append(ctx.pressure_mg_get_level(l, 2))
            omega.append(info["omega"])
            if info["dense"]:
                dense = l
        return cls(A, P, R, omega, pre, post, coarse, dense, mg_dense)

    def with_(self, **kw):
        """A copy with some of (pre, post, coarse, mg_dense) changed; the operators are shared."""
        args = dict(pre=self.pre, post=self.post, coarse=self.coarse, mg_dense=self.dense is not None)
        args.update(kw)
        v = VCycle.__new__(VCycle)
        v.__dict__.update(self.__dict__)
        v.pre, v.post, v.coarse = args["pre"], args["post"], args["coarse"]
        if not args["mg_dense"]:
            v.dense, v._chol = None, None
        return v

    def sweeps(self, l: int, b: np.ndarray, x: np.ndarray | None, k: int) -> np.ndarray:
        """k damped-Jacobi sweeps x <- x + omega_l D_l^-1 (b - A_l x); x None: from zero."""
        A, wd = self.A[l], self.omega[l] * self.dinv[l]
        for _ in range(k):
            x = wd * b if x is None else x + wd * (b - A @ x)
        return np.zeros_like(b) if x is None else x

    def __call__(self, b: np.ndarray, l: int = 0) -> np.ndarray:
        b = np.asarray(b, dtype=np.float64)
        if l >= 1 and l == self.dense:
            return sla.cho_solve(self._chol, b)
        if l == len(self.A) - 1:
            return self.sweeps(l, b, None, self.coarse)
        x = self.sweeps(l, b, None, self.pre)
        r = b - self.A[l] @ x
        x = x + self.P[l + 1] @ self(self.R[l + 1] @ r, l + 1)
        return self.sweeps(l, b, x, self.post)


def pcg(A, b, M, k: int | None = None, rtol: float = 0.0, atol: float = 0.0, maxit: int = 10000):
    """The ``k_cgz_*`` recurrence from a zero guess with z = M(r): returns (iterates x_1 .. x_its, its), stopping after
    `k` iterations or when |r|^2 <= max(rtol^2 |b|^2, atol^2), as the device's convergence test does."""
    A = sp.csr_matrix(A)
    b = np.asarray(b, dtype=np.float64)
    x, r = np.zeros_like(b), b.copy()
    tol2 = max(rtol * rtol * float(b @ b), atol * atol)
    out, p, rz_old = [], None, None
    limit = maxit if k is None else min(k, maxit)
    while len(out) < limit and float(r @ r) > tol2:
        z = M(r)
        rz = float(r @ z)
        p = z if p is None else z + (rz / rz_old) * p
        rz_old = rz
        q = A @ p
        alpha = rz / float(p @ q)
        x = x + alpha * p
        r = r - alpha * q
        out.append(x.copy())
    return out, len(out)


def box_levels(msh):
    """The geometric hierarchy of a provider box/rectangle (deformed in place or not) on the host, in node numbering:
    (A, P, R) with A[0] the fine P1 stiffness, A[l] that of the coarse mesh `multigrid.box_hierarchy` returns, P[l] its
    prolongation and R[l] = P[l]^T."""
    from oasisx_b200 import fem as _fem

    fine_x = msh.geometry.x if _fem.is_deformed(msh) else None
    A, P, R = [p1_stiffness(msh.geometry.x, msh.geometry.dofmap)], [None], [None]
    for cm, Pl in _mg.box_hierarchy(msh, fine_x=fine_x):
        A.append(p1_stiffness(cm.geometry.x, cm.geometry.dofmap))
        P.append(sp.csr_matrix(Pl))
        R.append(sp.csr_matrix(Pl.T))
    return A, P, R
