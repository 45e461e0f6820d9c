"""``FractionalStep_AB_CN`` -- the IPCS fractional step (Adams-Bashforth convection,
Crank-Nicolson diffusion) with the Python surface of
``/root/reference/src/oasisx/fracstep.py:29-705`` on top of ``libb200ipcs.so``.

Host side (this file): spaces, dof maps, boundary dof lists, evaluation of Python-callable
boundary values on the boundary dofs, option plumbing.  Device side (the C ABI): sparsity,
element kernels, CSR algebra, Krylov solves -- every ``dolfinx.fem.petsc`` / ``PETSc`` call of the
reference.  There is no CPU path: without the library or a GPU the constructor raises.
"""
from __future__ import annotations

import logging

import numpy as np

from . import _lib as L
from . import fem as _fem
from .bcs import DirichletBC, PressureBC
from .ksp import KSPSolver

__all__ = ["FractionalStep_AB_CN", "DeviceMatrix"]

logger = logging.getLogger("oasisx")


class _Binding:
    def __init__(self, ctx: L.Context, vec: int, comp: int):
        self.ctx, self.vec, self.comp = ctx, vec, comp

    def pull(self, host: np.ndarray):
        self.ctx.get_vector(self.vec, self.comp, host)

    def push(self, host: np.ndarray):
        self.ctx.set_vector(self.vec, self.comp, host)


class DeviceMatrix:
    """Handle to a device CSR matrix with the few ``PETSc.Mat`` calls the reference's callers use
    (``test/test_tentative_velocity.py:28,39``)."""

    def __init__(self, ctx: L.Context, mat: int, pattern: int, shape: tuple[int, int], comp: int = 0):
        self._ctx, self._mat, self._pattern, self._shape, self._comp = ctx, mat, pattern, shape, comp

    def getSize(self):
        return self._shape

    def getValuesCSR(self):
        indptr, indices = self._ctx.pattern(self._pattern, self._shape[0])
        return indptr, indices, self._ctx.matrix_values(self._mat, self._comp, len(indices))

    def mult(self, x, y):
        xa = x.array if hasattr(x, "array") else x
        ya = y.array if hasattr(y, "array") else y
        ya[: self._shape[0]] = self._ctx.mat_mult(self._mat, self._comp, xa, self._shape[0])


def _element_degree(el) -> int:
    if isinstance(el, (tuple, list)):
        if el[0] not in ("Lagrange", "CG", "P"):
            raise NotImplementedError(f"element family {el[0]!r}")
        return int(el[1])
    raise TypeError("element must be a (family, degree) tuple")


class FractionalStep_AB_CN:
    """
    Create the fractional step solver with Adam-Bashforth linearization of the convective term,
    and Crank-Nicholson time discretization (``fracstep.py:29-54``).

    Args:
        mesh: The computational domain (:class:`oasisx_b200.mesh.Mesh`, or a DOLFINx mesh through
            :mod:`oasisx_b200.adapter`)
        u_element: ``("Lagrange", degree)`` of one velocity component (degree 1 or 2)
        p_element: ``("Lagrange", 1)``
        bcs_u: list of Dirichlet BCs for each component of the velocity
        bcs_p: list of pressure BCs
        rotational: If True, use rotational form of pressure update
        solver_options: Dictionary with keys ``'tentative'``, ``'pressure'`` and ``'scalar'``,
            each a dictionary of PETSc-style options (SURVEY.md Appendix G)
        jit_options: accepted for API compatibility (there is no JIT: kernels are precompiled)
        body_force: constant force per direction
        options: ``"low_memory_version"`` True/False (``fracstep.py:47-50``)
        device: CUDA device ordinal (extension; default 0)
    """

    def __init__(
        self,
        mesh,
        u_element,
        p_element,
        bcs_u: list[list[DirichletBC]],
        bcs_p: list[PressureBC],
        rotational: bool = False,
        solver_options: dict | None = None,
        jit_options: dict | None = None,
        body_force=None,
        options: dict | None = None,
        device: int = 0,
    ):
        self._mesh = mesh
        gdim = mesh.geometry.dim
        deg_u, deg_p = _element_degree(u_element), _element_degree(p_element)
        if deg_p != 1:
            raise NotImplementedError("pressure element must be P1 on the B200 hot path")

        # spaces (fracstep.py:187-190,212); with more than one rank every rank keeps the slab of the
        # mesh it owns plus a ghost layer (oasisx_b200.partition)
        comm = mesh.comm
        self._nranks, self._rank = int(getattr(comm, "size", 1)), int(getattr(comm, "rank", 0))
        from . import adapter as _adapter

        self._foreign = _adapter.is_foreign_mesh(mesh)
        if self._foreign:
            # a DOLFINx mesh: its partition, dof maps and index maps are consumed as they are (north_star: "reuses
            # DOLFINx's mesh partition"); also on one rank, where the ghost blocks are simply empty
            self._lp, self._V, self._Q, self._geom_x = _adapter.problem_from_dolfinx(mesh, deg_u, deg_p)
        elif hasattr(mesh, "is_global_boundary"):
            # slab-local box mesh (oasisx_b200.slab): this rank built only its own slab; same LocalProblem as the
            # partition of a replicated mesh below
            from . import slab as _slab

            self._lp, _, self._Q = _slab.local_problem(mesh, deg_u, deg_p)
            self._V = _fem.functionspace(mesh, ("Lagrange", deg_u, (gdim,)))
        elif self._nranks > 1:
            gV = _fem.functionspace(mesh, ("Lagrange", deg_u))
            gQ = _fem.functionspace(mesh, ("Lagrange", deg_p))
            from . import partition as _part

            self._lp = lp = _part.partition(mesh, gV, gQ, self._nranks, self._rank)
            self._V = _fem.LocalFunctionSpace(gV, lp.V, gdim)
            self._Q = _fem.LocalFunctionSpace(gQ, lp.Q, 1)
            for sp_ in (self._V, self._V._scalar, self._Q):
                sp_._local_cells = lp.cells  # global ids of the cells this rank holds (owned first, then ghost cells)
        else:
            self._lp = None
            self._V = _fem.functionspace(mesh, ("Lagrange", deg_u, (gdim,)))
            self._Q = _fem.functionspace(mesh, ("Lagrange", deg_p))
        self._sol_u = _fem.Function(self._V, name="u")
        self._Vi = [self._V.sub(i).collapse() for i in range(self._V.num_sub_spaces)]
        Vs = self._Vi[0][0]
        mk = lambda space, name: _fem.Function(space, name=name)
        self._u = [mk(Vs, f"u{i}") for i in range(gdim)]
        self._u1 = [mk(Vs, f"u_{i}1") for i in range(gdim)]
        self._u2 = [mk(Vs, f"u_{i}2") for i in range(gdim)]
        self._uab = [mk(Vs, f"u_{i}ab") for i in range(gdim)]
        self._rhs1 = [mk(Vs, f"rhs1_{i}") for i in range(gdim)]
        self._b0 = [mk(Vs, f"b0_{i}") for i in range(gdim)]
        self._b_first = [mk(Vs, f"b_first_{i}") for i in range(gdim)]
        self._ps, self._p = mk(self._Q, "ps"), mk(self._Q, "p")
        self._dp, self._b2 = mk(self._Q, "dp"), mk(self._Q, "b2")

        # boundary conditions (fracstep.py:196-200,218-227)
        self._bcs_u = bcs_u
        for bc_i, Vi in zip(self._bcs_u, self._Vi):
            for bc in bc_i:
                bc.create_bc(Vi[0])
        self._bcs_p = bcs_p
        for bcp in self._bcs_p:
            bcp.create_bcs(Vs, self._Q)

        options = {} if options is None else options
        self._low_memory = bool(options.get("low_memory_version", True))
        self._rotational = bool(rotational)
        if body_force is None:
            body_force = (0.0,) * gdim
        body_force = [float(f.value) if isinstance(f, _fem.Constant) else float(f) for f in body_force]

        # ---- device context: upload mesh + dof maps, build patterns, preassemble (:265-268) ----
        if self._lp is not None:
            if self._nranks > 1:
                uid = comm.bcast(L.nccl_unique_id() if self._rank == 0 else None)
                self._ctx = ctx = L.Context(device=device, nranks=self._nranks, rank=self._rank, nccl_uid=uid)
            else:
                self._ctx = ctx = L.Context(device=device)
            lp = self._lp
            ctx.set_mesh(gdim, self._geom_x if self._foreign else mesh.geometry.x, lp.cell_nodes)
            ctx.set_space(L.SPACE_V, deg_u, lp.V.n_owned, lp.V.n_ghost, lp.V.cell_dofs)
            ctx.set_space(L.SPACE_Q, deg_p, lp.Q.n_owned, lp.Q.n_ghost, lp.Q.cell_dofs)
            ctx.set_global_sizes(lp.V.n_global, lp.Q.n_global)
            if self._nranks > 1:
                from . import partition as _part

                _part.check_halo_counts(comm, lp.V.halo, "V")
                _part.check_halo_counts(comm, lp.Q.halo, "Q")
                ctx.set_halo(L.SPACE_V, lp.V.halo)
                ctx.set_halo(L.SPACE_Q, lp.Q.halo)
                # halo + dot-product all-reduce through peer-mapped memory (NVLink) instead of NCCL calls, if every
                # rank can map every other rank's arena; otherwise all of them keep the NCCL path
                self._peer = ctx.peer_setup(comm, 0)
            self._nV_owned, self._nQ_owned = lp.V.n_owned, lp.Q.n_owned
        else:
            self._ctx = ctx = L.Context(device=device)
            ctx.set_mesh(gdim, mesh.geometry.x, mesh.geometry.dofmap)
            ctx.set_space(L.SPACE_V, deg_u, Vs.num_dofs, 0, Vs.dofmap.list)
            ctx.set_space(L.SPACE_Q, deg_p, self._Q.num_dofs, 0, self._Q.dofmap.list)
            ctx.set_global_sizes(Vs.num_dofs, self._Q.num_dofs)
            self._nV_owned, self._nQ_owned = Vs.num_dofs, self._Q.num_dofs
        Vs._b2_ctx = ctx  # a Projector on one of the solver's spaces shares its device context
        self._Q._scalar._b2_ctx = ctx
        ctx.build_patterns()
        if deg_u == 2:  # tile-major schedule of the SELL slices (L1 reuse of the gathered vector); any schedule is a
            # permutation of the slices, so a lattice that no longer fits the coordinates (a deformed box) costs speed only
            lat = getattr(mesh, "_lattice", None) if getattr(mesh, "_dof_order", "class") == "class" else None
            ctx.set_slice_order(L.PAT_VV, _fem.slice_order(Vs.tabulate_dof_coordinates()[: self._nV_owned], self._nV_owned, lat))
        self._bc_dofs: list[np.ndarray] = []
        self._bc_versions: list[tuple] = [() for _ in range(gdim)]
        self._bc_merge_maps: dict = {}
        self._bc_sorted: dict = {}
        for i in range(gdim):
            dofs = self._merged_bc_dofs(i)
            self._bc_dofs.append(dofs)
            ctx.set_velocity_bc_dofs(i, dofs)
        pdofs = (
            np.unique(np.concatenate([b.bc.dofs for b in self._bcs_p])) if self._bcs_p else np.zeros(0, np.int32)
        )
        ctx.declare_pressure_bcs(len(self._bcs_p) > 0)  # the same on every rank, also on one whose slab has no such dof
        ctx.set_pressure_bc_dofs(pdofs)  # local dofs, owned and ghost (columns of ghost BC dofs are zeroed too)
        ctx.preassemble(body_force, self._low_memory, self._rotational)

        # solvers (fracstep.py:230-255)
        solver_options = {} if solver_options is None else solver_options
        self._solver_u = KSPSolver(comm, solver_options.get("tentative"), prefix="tentative_velocity")
        self._solver_p = KSPSolver(comm, solver_options.get("pressure"), prefix="pressure_correction")
        self._solver_c = KSPSolver(comm, solver_options.get("scalar"), prefix="velocity_update")
        if (solver_options.get("scalar") or {}).get("ksp_type") == "chebyshev" and "ksp_chebyshev_eigenvalues" not in solver_options["scalar"]:
            # rigorous bounds of spec(D^-1 M): extreme generalised eigenvalues of the reference element mass
            # matrix against its own diagonal (Wathen 1987) -- mesh independent for affine simplices
            lo, hi = _fem.mass_jacobi_bounds(gdim, deg_u)
            self._solver_c.updateOptions({"ksp_chebyshev_eigenvalues": f"{lo!r},{hi!r}"})
        self._solver_u.bind(ctx, L.SOLVER_TENTATIVE)
        self._solver_p.bind(ctx, L.SOLVER_PRESSURE)
        self._solver_c.bind(ctx, L.SOLVER_SCALAR)
        if self._rotational:
            self._solver_proj = KSPSolver(comm, solver_options.get("scalar"), prefix="oasis_projector")
            self._solver_proj.bind(ctx, L.SOLVER_PROJECTOR)
        if len(self._bcs_p) == 0 and "ksp_type" not in (solver_options.get("pressure") or {}):
            # fracstep.py:562-576 forces a direct solve of the singular system; the device
            # equivalent is the null-space-projected CG run to the "exact" tolerance
            self._solver_p.updateOptions({"ksp_type": "preonly", "pc_type": "lu"})

        # optional multigrid for the pressure: "mg" takes the geometric hierarchy of a provider box; "gamg" / "hypre"
        # take it too where it exists and otherwise the algebraic hierarchy built from Ap (several ranks: from the
        # global Ap gathered by global dof index)
        self._mg_levels = 0
        self._mg_kind = None  # "geometric" | "algebraic" | None
        pc_p = (solver_options.get("pressure") or {}).get("pc_type")
        if pc_p in ("mg", "gamg", "hypre") and not self._bcs_p:
            from . import multigrid as _mg

            dof_nodes = getattr(self._Q, "_dof_nodes", None)
            if dof_nodes is None:  # P1: every local dof sits on the node its cells put it on
                cell_nodes, cell_dofs = (self._lp.cell_nodes, self._lp.Q.cell_dofs) if self._lp is not None else (
                    mesh.geometry.dofmap, self._Q.dofmap.list)
                dof_nodes = np.empty(self._Q.num_dofs, dtype=np.int64)
                dof_nodes[cell_dofs.ravel()] = cell_nodes.ravel()
            mg_config = options.get("multigrid") or {}
            self._mg_levels = _mg.attach_pressure_multigrid(ctx, mesh, dof_nodes, self._nQ_owned, **mg_config)
            if self._mg_levels:
                self._mg_kind = "geometric"
            elif pc_p != "mg":
                gids = self._lp.Q.l2g if self._nranks > 1 else None
                self._mg_levels = _mg.attach_pressure_amg(ctx, gids, **mg_config)
                self._mg_kind = "algebraic" if self._mg_levels else None
            if self._mg_levels == 0:
                logger.warning("pc_type=mg requested but the mesh carries no nested hierarchy: using Jacobi")
            elif self._nranks > 1 and ctx.peer_enabled():
                ctx.peer_setup(comm, 1)  # staging of the replicated level-1 right-hand side

        # matrices visible to callers (test/test_tentative_velocity.py:175)
        # (owned rows, local columns = owned + ghosts), like the local part of a PETSc MPIAIJ matrix
        nV, nQ, cV, cQ = self._nV_owned, self._nQ_owned, Vs.num_dofs, self._Q.num_dofs
        self._A = DeviceMatrix(ctx, L.MAT_A, L.PAT_VV, (nV, cV))
        self._M = DeviceMatrix(ctx, L.MAT_M, L.PAT_VV, (nV, cV))
        self._K = DeviceMatrix(ctx, L.MAT_K, L.PAT_VV, (nV, cV))
        self._Ap = DeviceMatrix(ctx, L.MAT_AP, L.PAT_QQ, (nQ, cQ))
        if not self._low_memory:  # fracstep.py:315,336,352: these exist only in the matrix-vector strategy
            self._p_vdxi_Mat = [DeviceMatrix(ctx, L.MAT_P, L.PAT_VQ, (nV, cQ), i) for i in range(gdim)]
            self._grad_p_Mat = [DeviceMatrix(ctx, L.MAT_G, L.PAT_VQ, (nV, cQ), i) for i in range(gdim)]
            self._divu_Mat = [DeviceMatrix(ctx, L.MAT_D, L.PAT_QV, (nQ, cV), i) for i in range(gdim)]
        self._solver_p.setOperators(self._Ap)
        self._solver_c.setOperators(self._M)
        self._solver_u.setOperators(self._A)

        # bind host mirrors to device vectors
        self._bound: list[_fem.Vector] = []
        for vec, fs in (
            (L.VEC_U, self._u), (L.VEC_U1, self._u1), (L.VEC_U2, self._u2), (L.VEC_UAB, self._uab),
            (L.VEC_RHS1, self._rhs1), (L.VEC_B0, self._b0), (L.VEC_BFIRST, self._b_first),
        ):
            for i, f in enumerate(fs):
                self._bind(f, vec, i)
        for vec, f in ((L.VEC_PS, self._ps), (L.VEC_P, self._p), (L.VEC_DP, self._dp), (L.VEC_B2, self._b2)):
            self._bind(f, vec, 0)
        self._bind(self._sol_u, L.VEC_U, -1)
        for f in self._b0:  # assembled on the device by b2_preassemble
            f.x.mark_device_written()
        self._bound.remove(self._sol_u.x)  # output-only view of VEC_U: never pushed
        self._upload_bcs()

    # ---- plumbing ------------------------------------------------------------------------
    def _bind(self, f: _fem.Function, vec: int, comp: int):
        f.x._binding = _Binding(self._ctx, vec, comp)
        self._bound.append(f.x)

    def _flush(self):
        for v in self._bound:
            v.flush()

    def _written(self, *groups):
        for g in groups:
            for f in g if isinstance(g, (list, tuple)) else (g,):
                f.x.mark_device_written()

    def _merged_bc_dofs(self, i: int) -> np.ndarray:
        """Sorted union of the OWNED dofs of all BCs of component i (ghost copies follow by halo)."""
        if not self._bcs_u[i]:
            return np.zeros(0, dtype=np.int32)
        d = np.unique(np.concatenate([bc._dofs for bc in self._bcs_u[i]]))
        return d[d < self._nV_owned].astype(np.int32)

    def _upload_bcs(self):
        """Send g_i on the merged BC dof list of each component; later BCs in the list win on shared
        dofs, as successive ``bc.apply`` calls do (``fracstep.py:517-518``)."""
        for i, bcl in enumerate(self._bcs_u):
            if not bcl:
                continue
            vals = [bc.current_values() for bc in bcl]
            version = tuple(bc._version for bc in bcl)
            if version == self._bc_versions[i]:
                continue
            if len(bcl) == 1 and len(vals[0]) == len(self._bc_dofs[i]) and self._bc_is_sorted(i, bcl[0]):
                merged = vals[0]  # the device list is the sorted unique dof list: identical order only if bc._dofs is
            else:
                # positions of every BC's owned dofs in the merged list: located once, not every time step
                maps = self._bc_merge_maps.setdefault(i, {})
                merged = np.zeros(len(self._bc_dofs[i]))
                for k, (bc, v) in enumerate(zip(bcl, vals)):
                    m = maps.get(k)
                    if m is None or m[0] is not bc._dofs:
                        own = np.flatnonzero(bc._dofs < self._nV_owned)
                        m = (bc._dofs, own, np.searchsorted(self._bc_dofs[i], bc._dofs[own]))
                        maps[k] = m
                    merged[m[2]] = v[m[1]]
            self._ctx.set_velocity_bc_values(i, merged)
            self._bc_versions[i] = version

    def _bc_is_sorted(self, i: int, bc) -> bool:
        """bc._dofs strictly increasing (checked once per dof array: `set_dofs` may inject any order)."""
        hit = self._bc_sorted.get(i)
        if hit is None or hit[0] is not bc._dofs:
            d = bc._dofs
            hit = (d, bool(len(d) < 2 or np.all(d[1:] > d[:-1])))
            self._bc_sorted[i] = hit
        return hit[1]

    def _assemble_pressure_surface(self):
        """``fracstep.py:445-446,461-465``: refresh the PressureBC values and assemble their ds-terms."""
        for k, bcp in enumerate(self._bcs_p):
            bcp.update_bc()
            self._ctx.assemble_pressure_surface(bcp._facet_cells, bcp._facet_local, bcp._h, accumulate=k > 0)

    # ---- stages (same names and meaning as the reference) ---------------------------------
    def assemble_first(self, dt: float, nu: float):
        """``fracstep.py:411-472``: A = M/dt + C/2 + nu K/2 (Dirichlet rows -> identity) and
        b_k = (M/dt - C/2 - nu K/2) u_k^{n-1} + f_k."""
        self._flush()
        self._assemble_pressure_surface()
        self._ctx.assemble_first(float(dt), float(nu))
        self._written(self._uab, self._b_first)

    def velocity_tentative_assemble(self):
        """``fracstep.py:474-506``: rhs1_k = b_k + int p* dv/dx_k."""
        self._flush()
        self._ctx.tentative_assemble()
        self._written(self._rhs1)

    def velocity_tentative_solve(self):
        """``fracstep.py:508-525``: apply Dirichlet values to the RHS and solve each component.
        Returns (sum_k ||u_k^old - u_k||_2, KSP converged reasons)."""
        self._upload_bcs()
        self._flush()
        diff, errors = self._ctx.tentative_solve()
        self._written(self._rhs1, self._u)
        return diff, errors

    def pressure_assemble(self, dt: float):
        """``fracstep.py:527-551``: b2 = -(1/dt) int div(u) q."""
        self._flush()
        self._ctx.pressure_assemble(float(dt))
        self._written(self._b2)

    def pressure_solve(self, nu: float | None = None, rotational: bool = False):
        """``fracstep.py:553-605`` (the ``rotational`` argument is ignored there too)."""
        if self._rotational and nu is None:
            raise RuntimeWarning("Kinematic viscosity not set for rotational pressure correction")
        self._flush()
        reason = self._ctx.pressure_solve(0.0 if nu is None else float(nu))
        self._written(self._b2, self._dp, self._ps)
        return reason

    def velocity_update(self, dt) -> np.ndarray:
        """``fracstep.py:607-658``: M u_k = M u_k - dt int d(dp)/dx_k v."""
        self._flush()
        errors = self._ctx.velocity_update(float(dt))
        self._written(self._u)
        return errors

    def solve(self, dt: float, nu: float, max_error: float = 1e-12, max_iter: int = 10):
        """Propagate the splitting scheme one time step (``fracstep.py:660-696``)."""
        # enqueue p* <- p and assemble_first first: they do not read the velocity Dirichlet values, so the host
        # evaluates the boundary callables (the reference does it up front, :675) while the GPU assembles
        self._flush()
        self._assemble_pressure_surface()
        self._ctx.step_begin(float(dt), float(nu))
        [[bc.update_bc() for bc in bcu] for bcu in self._bcs_u]
        self._upload_bcs()
        diff = self._ctx.step(float(dt), float(nu), float(max_error), int(max_iter))
        self._written(self._u, self._u1, self._u2, self._uab, self._rhs1, self._b_first, self._ps, self._p,
                      self._dp, self._b2)
        return diff

    @property
    def u(self):
        """The velocity as a blocked vector function (``fracstep.py:698-705``); the device layout is
        already interleaved, so this is one contiguous copy."""
        self._flush()
        self._sol_u.x._dev_newer = True
        self._sol_u.x._host_touched = False
        return self._sol_u

    def assemble_l2_error_sq(self, which: str, exact, degree: int = 8) -> float:
        """``assemble_scalar(inner(u_h - u_ex, u_h - u_ex) * dx)`` summed over ranks
        (``demo/taylor_green.py:186-207``).  which: "u" (the velocity, `exact` = one callable per
        component) or "p" (the pressure `_p`, `exact` = one callable).  The exact field is sampled by the
        host at the quadrature points of a degree-`degree` rule; the integration runs on the device.  An `exact` object
        with a ``trig_terms(which)`` method (the Taylor-Green fields of tests/problems.py and demo/taylor_green.py) is
        evaluated on the device instead: usable at 96^3, where the sampled field would be 27 GB per call."""
        from .quadrature import simplex_rule

        mesh, d = self._mesh, self._mesh.geometry.dim
        pts, w = simplex_rule(d, degree)
        if self._lp is not None:
            cells = self._lp.cell_nodes[: self._lp.n_cells_owned]
        else:
            cells = mesh.geometry.dofmap
        vec = L.VEC_U if which == "u" else L.VEC_P
        terms = getattr(exact, "trig_terms", None)
        if terms is not None:
            # analytic field given as trigonometric product terms (see b2_l2_error_trig): evaluated on the device at
            # the quadrature points, nothing but the term list crosses the bus
            self._flush()
            return self._ctx.l2_error_trig(vec, len(cells), pts, w, terms(which))
        X = mesh.geometry.x[cells]  # (nc, d+1, 3)
        lam = np.hstack([1.0 - pts.sum(axis=1, keepdims=True), pts])  # (nq, d+1)
        xq = np.einsum("qa,cak->kcq", lam, X)  # (3, nc, nq)
        flat = xq.reshape(3, -1)
        fs = list(exact) if which == "u" else [exact]
        ex = np.stack([np.asarray(f(flat), dtype=np.float64).reshape(len(cells), len(w)) for f in fs], axis=2)
        self._flush()
        return self._ctx.l2_error_quadrature(vec, len(cells), pts, w, np.ascontiguousarray(ex))

    def stats(self):
        return self._ctx.stats()
