"""``Projector`` with the surface of ``/root/reference/src/oasisx/function.py:13-143``: L2 projection of a function
into a Lagrange space -- mass matrix once, right-hand side re-assembled on demand, Krylov solve -- on the device.

The reference takes a UFL expression; there is no form compiler here (SURVEY.md N14), so ``function`` is one of

* a :class:`oasisx_b200.fem.Function` on the same mesh (any of the P1 / P2 spaces, scalar or blocked),
* ``grad(u)`` of a scalar Function (:func:`grad`; the expression of ``test/test_projector.py:33``),
  or one component ``grad(u)[i]``,
* a Python callable ``f(x)`` (``x`` of shape (3, n)), sampled at the quadrature points by the host,
* a list of the scalar kinds above, one per component of a blocked target space.

``bcs`` is a list of :class:`oasisx_b200.DirichletBC` (``function.py:70,114-118``: identity rows and columns in the
mass matrix, lifting of the right-hand side, ``set_bc``; on a blocked space a condition applies to every component
unless it carries ``component = k``).  ``space`` is a scalar or blocked Lagrange P1/P2 space of the mesh (the reference's test uses DG1; the continuous
space reproduces its known-answer check because the projected gradient is globally linear).  The right-hand side
``(f, v)`` is integrated by a device element kernel (``b2_project_assemble``), the mass solve runs with the
options of the ``oasis_projector`` prefix (``b2_project_solve``).  On the IPCS hot path the projector appears only
in the rotational pressure update, which the step kernel sequence does itself (``fracstep.py:237-247,593-602``).
"""
from __future__ import annotations

import numpy as np

from . import _lib as L
from . import fem as _fem
from .quadrature import simplex_rule

__all__ = ["Projector", "grad", "Grad"]


class Grad:
    """``ufl.grad(u)`` of a scalar Lagrange Function; ``grad(u)[i]`` is one component."""

    def __init__(self, u: _fem.Function, component: int | None = None):
        if u.function_space.bs != 1:
            raise NotImplementedError("grad of a scalar Function only")
        self.u, self.component = u, component

    def __getitem__(self, i: int) -> "Grad":
        return Grad(self.u, int(i))


def grad(u: _fem.Function) -> Grad:
    return Grad(u)


def _projection_context(space: _fem.FunctionSpace, device: int):
    """One device context per (mesh, P2-or-P1 velocity degree): mesh, both scalar spaces, patterns, mass matrices.
    A space that belongs to a FractionalStep_AB_CN keeps using that solver's context (``space._b2_ctx``)."""
    ctx = getattr(space._scalar, "_b2_ctx", None)
    if ctx is not None:
        return ctx
    mesh = space.mesh
    cache = mesh.__dict__.setdefault("_b2_projection_ctx", {})
    if device not in cache:
        V2 = _fem.functionspace(mesh, ("Lagrange", 2))
        Q1 = _fem.functionspace(mesh, ("Lagrange", 1))
        ctx = L.Context(device=device)
        ctx.set_mesh(mesh.geometry.dim, mesh.geometry.x, mesh.geometry.dofmap)
        ctx.set_space(L.SPACE_V, 2, V2.num_dofs, 0, V2.dofmap.list)
        ctx.set_space(L.SPACE_Q, 1, Q1.num_dofs, 0, Q1.dofmap.list)
        ctx.set_global_sizes(V2.num_dofs, Q1.num_dofs)
        ctx.build_patterns()
        for i in range(mesh.geometry.dim):
            ctx.set_velocity_bc_dofs(i, np.zeros(0, np.int32))
        ctx.declare_pressure_bcs(False)
        ctx.set_pressure_bc_dofs(np.zeros(0, np.int32))
        ctx.preassemble([0.0] * mesh.geometry.dim, True, True)
        cache[device] = ctx
    return cache[device]


class Projector:
    """``Projector(function, space, bcs, petsc_options, jit_options, form_compiler_options, metadata)``
    (``function.py:48-106``).  ``jit_options`` / ``form_compiler_options`` are accepted and unused (kernels are
    precompiled); ``metadata={"quadrature_degree": q}`` overrides the rule (default: exact for P2 x P2 products)."""

    def __init__(self, function, space: _fem.FunctionSpace, bcs=None, petsc_options: dict | None = None,
                 jit_options: dict | None = None, form_compiler_options: dict | None = None,
                 metadata: dict | None = None, device: int = 0):
        if space.degree not in (1, 2):
            raise NotImplementedError("Lagrange P1 / P2 targets")
        self._function, self._space = function, space
        self._ctx: L.Context = _projection_context(space, device)
        # which device space carries this degree in that context (a solver's context may be P1-P1)
        self._slot = self._space_slot(space)
        self._options = {k: v for k, v in (petsc_options or {}).items()
                         if k in ("ksp_type", "pc_type", "ksp_rtol", "ksp_atol", "ksp_max_it", "ksp_gmres_restart",
                                  "ksp_gmres_cgs_refinement_type", "ksp_chebyshev_eigenvalues")}
        if self._options.get("ksp_type") == "chebyshev" and "ksp_chebyshev_eigenvalues" not in self._options:
            # bounds of spec(D^-1 M) for the target's degree (fracstep.py does the same for the velocity update).  Dirichlet
            # rows turn M into an identity-bordered principal submatrix: its Jacobi-scaled spectrum interlaces with the
            # full one, and the identity's eigenvalue 1 lies inside the bounds, so they still hold.
            lo, hi = _fem.mass_jacobi_bounds(space.mesh.geometry.dim, space.degree)
            self._options["ksp_chebyshev_eigenvalues"] = f"{lo!r},{hi!r}"
        self._push_options()
        degree = int((metadata or {}).get("quadrature_degree", 4))
        self._pts, self._w = simplex_rule(space.mesh.geometry.dim, degree)
        self._x = _fem.Function(space)
        self._b = _fem.Function(space)
        self._sources = self._parse(function)
        self._bcs = list(bcs) if bcs else []
        for bc in self._bcs:  # our DirichletBC objects, one list entry per condition; blocked targets: one per component
            if not hasattr(bc, "_values"):
                bc.create_bc(space._scalar)
        self.assemble_rhs()

    # ---- helpers ---------------------------------------------------------------------------
    def _push_options(self):
        """The context's projector solver slot is shared by every Projector on it: each solve restates its options."""
        for k, v in self._options.items():
            self._ctx.set_solver_option(L.SOLVER_PROJECTOR, k, v)

    def _space_slot(self, sp: _fem.FunctionSpace) -> int:
        n = sp._scalar.num_dofs
        if self._ctx.space_size(L.SPACE_V) == n and self._ctx.space_degree(L.SPACE_V) == sp.degree:
            return L.SPACE_V
        if self._ctx.space_size(L.SPACE_Q) == n and sp.degree == 1:
            return L.SPACE_Q
        raise NotImplementedError("the space is not one of the two Lagrange spaces of the device context")

    def _parse(self, function):
        bs = self._space.bs
        if isinstance(function, Grad) and function.component is None:
            if bs != self._space.mesh.geometry.dim:
                raise ValueError("grad(u) needs a blocked target space with gdim components")
            return [("grad", function.u)]
        items = list(function) if isinstance(function, (list, tuple)) else None
        if items is None:
            if isinstance(function, _fem.Function) and function.function_space.bs == bs and bs > 1:
                return [("blocked", function)]
            items = [function]
        if len(items) != bs:
            raise ValueError(f"{len(items)} source component(s) for a space with block size {bs}")
        out = []
        for f in items:
            if isinstance(f, Grad):
                out.append(("deriv", f.u, f.component))
            elif isinstance(f, _fem.Function):
                if f.function_space.bs != 1:
                    raise ValueError("list entries must be scalar")
                out.append(("nodal", f))
            elif callable(f):
                out.append(("callable", f))
            else:
                raise TypeError(f"cannot project {type(f)!r}")
        return out

    def _quad_points(self):
        mesh = self._space.mesh
        X = mesh.geometry.x[mesh.geometry.dofmap]
        lam = np.hstack([1.0 - self._pts.sum(axis=1, keepdims=True), self._pts])
        return np.einsum("qa,cak->kcq", lam, X).reshape(3, -1), X.shape[0]

    def assemble_rhs(self):
        """``function.py:108-119``: b = (f, v), re-evaluating the source."""
        ctx, bs, n = self._ctx, self._space.bs, self._space._scalar.num_dofs
        rhs = np.zeros((bs, n))
        kind0 = self._sources[0][0]
        if kind0 == "grad":
            u = self._sources[0][1]
            ctx.project_assemble(self._slot, bs, self._pts, self._w, src_space=self._space_slot(u.function_space),
                                 src_nodal=u.x.array_ro(), grad=True)
            rhs[:] = ctx.project_rhs(bs * n).reshape(bs, n)
        elif kind0 == "blocked":
            f = self._sources[0][1]
            nodal = np.ascontiguousarray(f.x.array_ro().reshape(-1, bs).T)
            ctx.project_assemble(self._slot, bs, self._pts, self._w, src_space=self._space_slot(f.function_space), src_nodal=nodal)
            rhs[:] = ctx.project_rhs(bs * n).reshape(bs, n)
        else:
            for k, src in enumerate(self._sources):
                if src[0] == "nodal":
                    ctx.project_assemble(self._slot, 1, self._pts, self._w, src_space=self._space_slot(src[1].function_space),
                                         src_nodal=src[1].x.array_ro())
                elif src[0] == "deriv":
                    ctx.project_assemble(self._slot, 1, self._pts, self._w, src_space=self._space_slot(src[1].function_space),
                                         src_nodal=src[1].x.array_ro(), deriv=src[2])
                else:
                    xq, nc = self._quad_points()
                    fq = np.asarray(src[1](xq), dtype=np.float64).reshape(nc, len(self._w), 1)
                    ctx.project_assemble(self._slot, 1, self._pts, self._w, f_quad=np.ascontiguousarray(fq))
                rhs[k] = ctx.project_rhs(n)
        self._rhs = rhs
        self._b.x.array[:] = np.ascontiguousarray(rhs.T).reshape(-1) if bs > 1 else rhs[0]

    def solve(self, assemble_rhs: bool = True):
        """``function.py:121-133``; returns the KSP converged reason (the smallest over the components)."""
        if assemble_rhs:
            self.assemble_rhs()
        ctx, bs, n = self._ctx, self._space.bs, self._space._scalar.num_dofs
        self._push_options()
        self._push_bcs()
        ctx.project_load_rhs(self._slot, self._rhs)  # the right-hand side this object assembled last, all components
        out, reasons = ctx.project_solve(n, bs)      # one Krylov run on bs systems sharing the mass matrix
        self._x.x.array[:] = np.ascontiguousarray(out.T).reshape(-1) if bs > 1 else out[0]
        return int(min(reasons))

    def _push_bcs(self):
        """``function.py:70,114-118``: Dirichlet rows/columns of the mass matrix -> identity, lifting, set_bc.  The
        conditions (``oasisx_b200.DirichletBC``; for a blocked space a condition may carry ``component = k``, default
        all components) are merged into one dof list per projector, later conditions winning on shared dofs."""
        ctx, bs = self._ctx, self._space.bs
        if not self._bcs:
            ctx.project_set_bcs(self._slot, np.zeros(0, np.int32), np.zeros((bs, 0)))
            return
        dofs = np.unique(np.concatenate([bc._dofs for bc in self._bcs])).astype(np.int32)
        vals = np.zeros((bs, len(dofs)))
        for bc in self._bcs:
            bc.update_bc()
            pos = np.searchsorted(dofs, bc._dofs)
            comp = getattr(bc, "component", None)
            for k in (range(bs) if comp is None else [int(comp)]):
                vals[k, pos] = bc.current_values()
        ctx.project_set_bcs(self._slot, dofs, vals)

    @property
    def x(self):
        return self._x
