"""Host restatement of the device GMRES (oasisx_b200/csrc/gmres.cuh): restarted GMRES(m) with left Jacobi
preconditioning, classical Gram-Schmidt (one pass, or two with ``cgs2``), Givens rotations, PETSc's happy-breakdown
test and the tolerance rule of the other device Krylov methods, on K right-hand sides that share the matrix.

The components advance in lockstep on the device, but each has its own Hessenberg matrix, rotations and stop index,
and all start a cycle at the same step: running them one after the other here gives the same iterates.  Only the
tolerance couples them (``block_rtol``).  The GPU tests hold the device to this function: same solution, same
iteration counts, same reasons."""
from __future__ import annotations

import numpy as np

HAPTOL = 1e-30  # PETSc's gmres->haptol


def _reason(rr, tol2, its, maxit, rtol, atol, bb):
    if not np.isfinite(rr):
        return -9  # KSP_DIVERGED_NANORINF
    if rr <= tol2:
        return 3 if (rr <= atol * atol and atol * atol >= rtol * rtol * bb) else 2
    if its >= maxit:
        return -3  # KSP_DIVERGED_ITS
    return 0


def gmres(A, B, dinv=None, x0=None, rtol=1e-5, atol=1e-50, maxit=10000, restart=30, cgs2=False, block_rtol=False):
    """Solve A x_k = b_k for the rows b_k of B (shape (K, n), or (n,) for one system).

    dinv: the left preconditioner D^-1 as a vector (None: pc_type none); x0: initial guess (None: zero guess).
    Returns a dict: ``x`` (shape of B), ``its`` and ``reasons`` per component, ``tol2`` per component and ``est``:
    per component the squared residual estimate after every Arnoldi step (the quantity compared with tol2)."""
    one = np.ndim(B) == 1
    B = np.atleast_2d(np.asarray(B, dtype=np.float64))
    K, n = B.shape
    d = np.ones(n) if dinv is None else np.asarray(dinv, dtype=np.float64)
    X = np.zeros((K, n)) if x0 is None else np.atleast_2d(np.array(x0, dtype=np.float64))
    DB = d * B
    bb = (DB * DB).sum(axis=1)
    bref = np.full(K, bb.max()) if block_rtol else bb
    tol2 = np.maximum(rtol * rtol * bref, atol * atol)
    out = {"its": [], "reasons": [], "tol2": tol2, "est": []}
    m = restart
    passes = 2 if cgs2 else 1
    for k in range(K):
        x = X[k]
        its, est = 0, []
        r = DB[k] - (d * (A @ x) if x0 is not None else 0.0)
        rr = float(r @ r)
        reason = _reason(rr, tol2[k], its, maxit, rtol, atol, bb[k])
        while reason == 0:
            beta = np.sqrt(rr)
            V = np.zeros((m + 1, n))
            V[0] = r / beta
            H = np.zeros((m + 1, m))
            cs, sn = np.zeros(m), np.zeros(m)
            g = np.zeros(m + 1)
            g[0] = beta
            steps = 0
            for j in range(m):
                w = d * (A @ V[j])
                for _ in range(passes):
                    h = V[: j + 1] @ w
                    w = w - V[: j + 1].T @ h
                    H[: j + 1, j] += h
                tt = float(np.sqrt(w @ w))
                happy = tt < min(abs(tt / g[j]), HAPTOL)
                for i in range(j):
                    a, b = H[i, j], H[i + 1, j]
                    H[i, j] = cs[i] * a + sn[i] * b
                    H[i + 1, j] = cs[i] * b - sn[i] * a
                hjj = H[j, j]
                dd = np.sqrt(hjj * hjj + tt * tt)
                its += 1
                if dd == 0.0:
                    reason = -5
                    break
                steps = j + 1
                cs[j], sn[j] = hjj / dd, tt / dd
                H[j, j] = dd
                g[j + 1] = -sn[j] * g[j]
                g[j] = cs[j] * g[j]
                rr = g[j + 1] * g[j + 1]
                est.append(rr)
                reason = _reason(rr, tol2[k], its, maxit, rtol, atol, bb[k])
                if reason == 0 and happy:
                    reason = -5  # KSP_DIVERGED_BREAKDOWN
                if reason != 0:
                    break
                V[j + 1] = w / tt
            y = np.zeros(steps)
            for i in range(steps - 1, -1, -1):
                y[i] = (g[i] - H[i, i + 1: steps] @ y[i + 1:]) / H[i, i]
            x = x + V[:steps].T @ y
            if reason != 0:
                break
            r = DB[k] - d * (A @ x)
            rr = float(r @ r)
            reason = _reason(rr, tol2[k], its, maxit, rtol, atol, bb[k])
        X[k] = x
        out["its"].append(its)
        out["reasons"].append(reason)
        out["est"].append(est)
    out["x"] = X[0] if one else X
    return out


def near_threshold(ref: dict, k: int, rel: float = 1e-8) -> bool:
    """True when component k's estimate at its last step, or at the step before, lies within `rel` (relative) of the
    tolerance: rounding in the device's reductions may then move the crossing by one step."""
    t = ref["tol2"][k]
    return any(abs(e - t) <= rel * t for e in ref["est"][k][-2:])
