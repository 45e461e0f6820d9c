"""``KSPSolver`` with the surface of ``/root/reference/src/oasisx/ksp.py:14-91``.

It carries a PETSc-style options dict under a prefix and forwards the options the GPU Krylov
stack understands (SURVEY.md Appendix G) to one of the context's solver slots.  ``preonly`` +
``lu`` (the reference demo's choice, ``demo/taylor_green.py:117-121``) has no sparse-LU
counterpart on the device and is mapped to "Krylov to rtol 1e-12".
"""
from __future__ import annotations

import logging

logger = logging.getLogger("oasisx")

_UNDERSTOOD = {"ksp_type", "pc_type", "ksp_rtol", "ksp_atol", "ksp_max_it", "ksp_initial_guess_nonzero", "b200_guess",
               "ksp_chebyshev_eigenvalues", "b200_block_rtol", "ksp_gmres_restart", "ksp_gmres_cgs_refinement_type"}


class KSPSolver:
    def __init__(self, comm, petsc_options: dict | None = None, prefix: str = "oasis_solver"):
        self._prefix = prefix
        self._options: dict = {}
        self._ctx = None
        self._slot = None
        self._operator = None
        self.updateOptions({} if petsc_options is None else petsc_options)

    def bind(self, ctx, slot: int):
        self._ctx, self._slot = ctx, slot
        self._push(self._options)

    def _push(self, options: dict):
        if self._ctx is None:
            return
        for k, v in options.items():
            if k in _UNDERSTOOD:
                self._ctx.set_solver_option(self._slot, k, v)
            else:
                logger.debug("option %s%s=%s ignored by the B200 Krylov stack", self._prefix, k, v)

    def updateOptions(self, options: dict):
        """``ksp.py:38-53``."""
        self._options.update(options)
        self._push(options)

    def setOptions(self, op):
        """``ksp.py:55-59``: matrix/vector options are a no-op for device CSR storage."""

    def setOperators(self, A, P=None):
        self._operator = A

    def solve(self, b, x):
        """``ksp.py:71-78``: solve ``A x = b`` with this solver's options, refresh the ghosts of ``x`` and return the
        KSP converged reason.  ``b``: a vector (``Function.x``, its ``petsc_vec`` stand-in or a numpy array) of the
        operator's row space; ``x``: a Function (initial guess if ``ksp_initial_guess_nonzero``)."""
        import numpy as np

        if self._ctx is None or self._operator is None:
            raise RuntimeError("KSPSolver.solve needs bind(ctx, slot) and setOperators(A) first")
        bv = b
        for attr in ("x", "petsc_vec"):
            bv = getattr(bv, attr, bv)
        barr = np.ascontiguousarray(bv.array_ro() if hasattr(bv, "array_ro") else getattr(bv, "array", bv), dtype=np.float64)
        xv = x.x
        xarr = np.ascontiguousarray(xv.array_ro(), dtype=np.float64).copy()
        reason = self._ctx.ksp_solve(self._slot, self._operator._mat, barr, xarr)
        xv.array[:] = xarr
        return reason

    @property
    def options(self) -> dict:
        return dict(self._options)
