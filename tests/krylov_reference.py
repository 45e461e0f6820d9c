"""Host restatements of the device Krylov methods of oasisx_b200/csrc/linalg.cuh and b200ipcs.cu other than GMRES
(tests/gmres_reference.py) and the multigrid PCG (tests/mg_reference.py):

* ``cg``: Jacobi-preconditioned CG (k_cg_init / k_cg_update / k_cg_p, FIN_CG_*);
* ``bcgs``: BiCGStab with left Jacobi preconditioning and the restart rule of FIN_BCGS_UPDATE (k_bcgs_*);
* ``chebyshev``: the reduction-free Chebyshev iteration of chebyshev_solve with its host check schedule.

All run on K right-hand sides that share the matrix.  The device advances them in lockstep, but only the tolerance
couples them (``block_rtol``), so they run one after the other here.  Each returns a dict with the keys of
``gmres_reference.gmres`` (``x``, ``its``, ``reasons``, ``tol2``, ``est``: per component the squared residual norm
after every step, the quantity compared with tol2) and the recurrence scalars per component and step."""
from __future__ import annotations

import numpy as np

from gmres_reference import _reason, near_threshold  # noqa: F401  (near_threshold: shared with the GPU tests)

RESTART_TOL = 1e-24  # FIN_BCGS_UPDATE: restart when (rhat . r)^2 <= 1e-24 |r|^2 |rhat|^2


def _setup(A, B, dinv, x0):
    one = np.ndim(B) == 1
    B = np.atleast_2d(np.asarray(B, dtype=np.float64))
    K, n = B.shape
    d = np.ones(n) if dinv is None else np.asarray(dinv, dtype=np.float64)
    X = np.zeros((K, n)) if x0 is None else np.atleast_2d(np.array(x0, dtype=np.float64))
    return one, B, K, d, X


def _tol2(bb, rtol, atol, block_rtol):
    bref = np.full(len(bb), bb.max()) if block_rtol else bb
    return np.maximum(rtol * rtol * bref, atol * atol)


def _finish(out, one, X):
    out["x"] = X[0] if one else X
    return out


def cg(A, B, dinv=None, x0=None, rtol=1e-5, atol=1e-50, maxit=10000, block_rtol=False):
    """Jacobi PCG.  The tolerance is on the unpreconditioned residual: r.r against max(rtol^2 b.b, atol^2).
    dinv: D^-1 as a vector (None: pc_type none); x0: initial guess (None: zero guess)."""
    one, B, K, d, X = _setup(A, B, dinv, x0)
    bb = (B * B).sum(axis=1)
    tol2 = _tol2(bb, rtol, atol, block_rtol)
    out = {"its": [], "reasons": [], "tol2": tol2, "est": [], "alpha": [], "beta": []}
    for k in range(K):
        x = X[k]
        r = B[k] - (A @ x if x0 is not None else 0.0)
        p = d * r
        rz, rr = float(r @ p), float(r @ r)
        its, est, al, be = 0, [], [], []
        reason = _reason(rr, tol2[k], its, maxit, rtol, atol, bb[k])
        while reason == 0:
            q = A @ p
            pq = float(p @ q)
            if not np.isfinite(pq):
                reason = -9
            elif pq == 0.0:
                reason = -5  # KSP_DIVERGED_BREAKDOWN
            elif pq < 0.0:
                reason = -8  # KSP_DIVERGED_INDEFINITE_PC
            if reason != 0:
                break
            alpha = rz / pq
            x = x + alpha * p
            r = r - alpha * q
            rz_new, rr = float(r @ (d * r)), float(r @ r)
            beta = rz_new / rz
            rz = rz_new
            its += 1
            est.append(rr)
            al.append(alpha)
            be.append(beta)
            reason = _reason(rr, tol2[k], its, maxit, rtol, atol, bb[k])
            if reason == 0:
                p = d * r + beta * p
        X[k] = x
        for key, v in (("its", its), ("reasons", reason), ("est", est), ("alpha", al), ("beta", be)):
            out[key].append(v)
    return _finish(out, one, X)


def bcgs(A, B, dinv=None, x0=None, rtol=1e-5, atol=1e-50, maxit=10000, block_rtol=False):
    """BiCGStab on D^-1 A x = D^-1 b: r0 = D^-1 b - D^-1 A x0, rhat = p = r0.  Convergence is tested after the full
    step only (not at s), omega = 0 when t.t = 0, and a vanishing omega or rho, or (rhat.r)^2 <= 1e-24 |r|^2 |rhat|^2,
    restarts with rhat = p = r instead of failing.  ``restart`` records per step whether it did; ``r`` is the last
    recursive residual per component."""
    one, B, K, d, X = _setup(A, B, dinv, x0)
    DB = d * B
    bb = (DB * DB).sum(axis=1)
    tol2 = _tol2(bb, rtol, atol, block_rtol)
    out = {"its": [], "reasons": [], "tol2": tol2, "est": [], "alpha": [], "omega": [], "beta": [], "restart": [], "r": []}
    for k in range(K):
        x = X[k]
        r = DB[k] - (d * (A @ x) if x0 is not None else 0.0)
        rhat, p = r.copy(), r.copy()
        rr = float(r @ r)
        rho, rh2 = rr, rr
        its, est, al, om, be, rs = 0, [], [], [], [], []
        reason = _reason(rr, tol2[k], its, maxit, rtol, atol, bb[k])
        while reason == 0:
            v = d * (A @ p)
            dv = float(rhat @ v)
            if not np.isfinite(dv):
                reason = -9
            elif dv == 0.0:
                reason = -5
            if reason != 0:
                break
            alpha = rho / dv
            s = r - alpha * v
            t = d * (A @ s)
            tt = float(t @ t)
            omega = float(t @ s) / tt if tt > 0.0 else 0.0
            x = x + alpha * p + omega * s
            r = s - omega * t
            rr, rn = float(r @ r), float(rhat @ r)
            its += 1
            est.append(rr)
            al.append(alpha)
            om.append(omega)
            reason = _reason(rr, tol2[k], its, maxit, rtol, atol, bb[k])
            if reason == 0 and not np.isfinite(rn):
                reason = -9
            if reason != 0:
                break
            if omega == 0.0 or rho == 0.0 or rn * rn <= RESTART_TOL * rr * rh2:
                rho, rh2, beta = rr, rr, 0.0
                rhat, p = r.copy(), r.copy()
                rs.append(True)
            else:
                beta = (rn / rho) * (alpha / omega)
                rho = rn
                p = r + beta * (p - omega * v)
                rs.append(False)
            be.append(beta)
        X[k] = x
        for key, val in (("its", its), ("reasons", reason), ("est", est), ("alpha", al), ("omega", om), ("beta", be),
                         ("restart", rs), ("r", r)):
            out[key].append(val)
    return _finish(out, one, X)


def chebyshev_first_check(rr0, tol2, lo, hi):
    """The step of the first residual check: enough steps for the worst component's |r0| / tol under the rate
    (sqrt(kappa) - 1) / (sqrt(kappa) + 1), plus ln 2 for the constant of the Chebyshev bound."""
    need = max(0.5 * np.log(r / t) for r, t in zip(rr0, tol2) if r > t)
    kappa = hi / lo
    rate = (np.sqrt(kappa) - 1.0) / (np.sqrt(kappa) + 1.0)
    return max(1, int(np.ceil((need + np.log(2.0)) / -np.log(rate))))


def chebyshev(A, B, lo, hi, dinv=None, x0=None, rtol=1e-5, atol=1e-50, maxit=10000, block_rtol=False):
    """Chebyshev iteration on the spectrum [lo, hi] of D^-1 A.  The scalars are data independent: theta, delta,
    sigma1 = theta / delta, rho_0 = 1 / sigma1, rho_new = 1 / (2 sigma1 - rho), c1 = rho_new rho, c2 = 2 rho_new / delta.
    The residual norms are read at ``first_check`` and then every 4 steps; all components take the same number of
    steps, and stop when all are below tolerance (reason 2; -3 when maxit comes first, also between checks).
    Unlike the other methods the components are not independent: they share the step count."""
    one, B, K, d, X = _setup(A, B, dinv, x0)
    bb = (B * B).sum(axis=1)
    tol2 = _tol2(bb, rtol, atol, block_rtol)
    theta, delta = 0.5 * (hi + lo), 0.5 * (hi - lo)
    sigma1 = theta / delta
    R = B - ((A @ X.T).T if x0 is not None else 0.0)
    Dd = d * R / theta
    rr0 = (R * R).sum(axis=1)
    out = {"tol2": tol2, "est": [[] for _ in range(K)], "c1": [], "c2": [], "checks": [], "first_check": None}
    conv = bool(np.all(~(rr0 > tol2)))  # the device tests rr > tol2 (a NaN counts as converged here)
    it = 0
    if not conv:
        nxt = out["first_check"] = chebyshev_first_check(rr0, tol2, lo, hi)
        rho = 1.0 / sigma1
        while it < maxit:
            Q = (A @ Dd.T).T
            rho_new = 1.0 / (2.0 * sigma1 - rho)
            c1, c2 = rho_new * rho, 2.0 * rho_new / delta
            X = X + Dd
            R = R - Q
            Dd = c1 * Dd + c2 * d * R
            rho = rho_new
            it += 1
            out["c1"].append(c1)
            out["c2"].append(c2)
            rr = (R * R).sum(axis=1)
            for k in range(K):
                out["est"][k].append(float(rr[k]))
            if it >= nxt:
                out["checks"].append(it)
                conv = bool(np.all(rr <= tol2))
                if conv:
                    break
                nxt = it + 4
    out["its"] = [it] * K
    out["reasons"] = [2 if conv else -3] * K
    return _finish(out, one, X)
