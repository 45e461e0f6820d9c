"""Host side of the pressure multigrid: nested box/rectangle meshes and P1 prolongations.

The Kuhn (Freudenthal) subdivision the provider uses is self-similar under 2x refinement: every
edge of the fine mesh lies along a direction with components in {0, 1}, so a fine vertex with lattice
index (i, j, k) and parity (a, b, c) = (i%2, j%2, k%2) is either a coarse vertex (parity 0) or the
midpoint of the coarse edge between (i-a, j-b, k-c)/2 and (i+a, j+b, k+c)/2.  The P1 spaces are
nested, hence the coarse stiffness matrix equals the Galerkin product R A P and is simply assembled
on the coarse mesh by the library (``b2_pressure_mg_add_level``).

For meshes that come from DOLFINx the same C entry point accepts any nested hierarchy (e.g. from
``dolfinx.mesh.refine`` [ext]) as long as P/R are supplied.

Meshes without such a hierarchy get a smoothed-aggregation algebraic multigrid built on the device from the assembled
pressure matrix instead (:func:`attach_pressure_amg`), on one rank or several; the V-cycle is the same.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp

from . import _lib
from . import fem as _fem
from . import mesh as _mesh


def _node_ids(idx: np.ndarray, shape) -> np.ndarray:
    n = [s + 1 for s in shape]
    out = idx[:, 0].copy()
    stride = n[0]
    for k in range(1, len(shape)):
        out += idx[:, k] * stride
        stride *= n[k]
    return out


def lattice_prolongation(fine_shape, coarse_shape, rows: np.ndarray | None = None) -> sp.csr_matrix:
    """(fine nodes) x (coarse nodes) P1 interpolation, both in lexicographic node numbering.  `rows`: lattice indices
    (n, d) of the fine nodes wanted, in that order (a rank's owned pressure dofs) instead of all fine nodes."""
    d = len(fine_shape)
    if rows is None:
        grids = np.meshgrid(*[np.arange(s + 1) for s in fine_shape[::-1]], indexing="ij")
        idx = np.stack([g.ravel() for g in grids[::-1]], axis=1).astype(np.int64)  # (nf, d): (i, j[, k]), i fastest
    else:
        idx = np.asarray(rows, dtype=np.int64)
    par = idx & 1
    lo, hi = (idx - par) // 2, (idx + par) // 2
    nf = idx.shape[0]
    nc = int(np.prod([s + 1 for s in coarse_shape]))
    rows = np.concatenate([np.arange(nf), np.arange(nf)])
    cols = np.concatenate([_node_ids(lo, coarse_shape), _node_ids(hi, coarse_shape)])
    vals = np.full(2 * nf, 0.5)
    P = sp.coo_matrix((vals, (rows, cols)), shape=(nf, nc)).tocsr()
    P.sum_duplicates()
    return P


def box_hierarchy(msh, min_cells: int = 2, max_levels: int = 16, first_rows: np.ndarray | None = None,
                  fine_x: np.ndarray | None = None):
    """[(coarse mesh, P from the previous level)] for a provider-built box/rectangle mesh.  `first_rows`: lattice
    indices of the fine nodes the FIRST prolongation is wanted for (its rows, in that order).  `fine_x`: coordinates of
    all fine nodes in the provider's (lexicographic) numbering, for a box deformed in place: every coarse node then
    takes the coordinates of the fine node it coincides with (lattice index doubled) instead of the uniform box's."""
    shape = getattr(msh, "_shape", None)
    if shape is None:
        return []
    p0, p1 = msh._box
    d = len(shape)
    out = []
    fine = tuple(shape)
    while len(out) < max_levels and all(n % 2 == 0 for n in fine) and min(fine) // 2 >= min_cells:
        coarse = tuple(n // 2 for n in fine)
        cm = (_mesh.create_rectangle if d == 2 else _mesh.create_box)(None, [list(p0), list(p1)], list(coarse))
        if fine_x is not None:
            cm.geometry.x[:] = fine_x[_node_ids(2 * _fem.lattice_node_index(cm), fine)]
            fine_x = cm.geometry.x
        out.append((cm, lattice_prolongation(fine, coarse, first_rows if not out else None)))
        fine = coarse
    return out


def attach_pressure_multigrid(ctx, msh, dof_nodes: np.ndarray, n_owned: int, **config) -> int:
    """Build the hierarchy for the pressure space whose LOCAL dofs (owned first) sit on the geometry nodes
    `dof_nodes` and register it with the context.  Returns the number of coarse levels (0: the mesh carries no
    hierarchy).

    The lattice index of a dof comes from the provider's node numbering, not from its coordinates, so a box deformed
    in place keeps its hierarchy.  Its coarse levels take their coordinates from the deformed fine geometry (one rank,
    or several with the replicated mesh; a slab-local mesh cannot be deformed, see `slab.SlabFunctionSpace`)."""
    if getattr(msh, "_shape", None) is None:
        return 0
    slab = hasattr(msh, "is_global_boundary")
    if not (slab or getattr(msh, "_canonical", False)):
        return 0  # nodes renumbered: the lattice index of a node is unknown
    idx = _fem.lattice_node_index(msh)[dof_nodes]  # fine lattice node of each local dof
    fine_x = msh.geometry.x if not slab and _fem.is_deformed(msh) else None
    levels = box_hierarchy(msh, first_rows=idx[:n_owned], fine_x=fine_x)  # rows of the owned dofs only
    if not levels:
        return 0
    n_local = len(dof_nodes)
    for lvl, (cm, P) in enumerate(levels):
        if lvl == 0:
            Pl = P.tocsr()
            R = sp.csr_matrix(Pl.T)
            R = sp.csr_matrix((R.data, R.indices, R.indptr), shape=(P.shape[1], n_local))
        else:
            Pl, R = P, sp.csr_matrix(P.T)
        Pl.sort_indices()
        R.sort_indices()
        ctx.pressure_mg_add_level(cm.geometry.x, cm.geometry.dofmap, Pl, R)
    if config:
        ctx.pressure_mg_configure(**config)
    return len(levels)


def attach_pressure_amg(ctx, global_ids: np.ndarray | None = None, **config) -> int:
    """Build the smoothed-aggregation hierarchy of the assembled pressure matrix on the device
    (``b2_pressure_amg_build``, no pressure Dirichlet dofs) and apply `config` as :func:`attach_pressure_multigrid` does
    (its ``omega`` only damps geometric levels).  Returns the number of coarse levels.

    On several ranks `global_ids` is the global index of every local pressure dof (``LocalSpace.l2g``), and every rank
    must call this: the owned rows of all ranks are gathered into the global matrix, every rank builds the same
    hierarchy from it, and level 1 keeps this rank's owned rows, as the geometric path does."""
    if global_ids is not None:
        ctx.set_pressure_global_ids(global_ids)
    ctx.pressure_amg_build()
    if config:
        ctx.pressure_mg_configure(**config)
    n = 0
    while True:  # level_info fails past the coarsest level
        try:
            ctx.pressure_mg_level_info(n + 1)
        except _lib.B200Error:
            return n
        n += 1
