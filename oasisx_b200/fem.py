"""Host-side function spaces, dof maps, CSR patterns and (device-mirrored) functions.

Stands in for the slice of ``dolfinx.fem`` / ``dolfinx.la`` that the reference's IPCS loop touches
(SURVEY.md N3, N12, N15): ``functionspace``, ``Function`` (``.x.array``, ``.interpolate``),
``Constant``, ``locate_dofs_topological`` / ``locate_dofs_geometrical`` and the sparsity pattern
behind ``dolfinx.fem.petsc.create_matrix`` (``/root/reference/src/oasisx/fracstep.py:293-352``).

A :class:`Function` owns a host numpy array.  Once the solver binds it to a device vector the host
array becomes a *mirror*: reading ``.x.array`` pulls from the GPU if the GPU copy is newer and marks
the host copy as possibly edited, so that it is pushed back before the next device stage.  Inside
``FractionalStep_AB_CN.solve`` nothing touches the host mirrors.
"""
from __future__ import annotations

from typing import Callable

import numpy as np

from .mesh import _BOX_CELLS, _EDGE_VERTS, Mesh

__all__ = [
    "Constant",
    "DofMap",
    "Function",
    "FunctionSpace",
    "Vector",
    "build_csr_pattern",
    "functionspace",
    "locate_dofs_geometrical",
    "locate_dofs_topological",
]


class IndexMap:
    """Owned-first / ghosts-last index map (``dolfinx.common.IndexMap`` look-alike)."""

    def __init__(self, size_local: int, ghosts=None, owners=None, size_global=None, offset=0):
        self.size_local = int(size_local)
        self.ghosts = np.zeros(0, np.int64) if ghosts is None else np.asarray(ghosts, np.int64)
        self.owners = np.zeros(0, np.int32) if owners is None else np.asarray(owners, np.int32)
        self.num_ghosts = len(self.ghosts)
        self.size_global = self.size_local if size_global is None else int(size_global)
        self.local_range = (int(offset), int(offset) + self.size_local)


class DofMap:
    def __init__(self, cell_dofs: np.ndarray, index_map: IndexMap, bs: int = 1):
        self.list = np.ascontiguousarray(cell_dofs, dtype=np.int32)
        self.index_map = index_map
        self.index_map_bs = bs

    def cell_dofs(self, c: int) -> np.ndarray:
        return self.list[c]


class _Element:
    def __init__(self, cell: str, degree: int):
        d = 2 if cell == "triangle" else 3
        pts = [np.zeros(d)] + [np.eye(d)[i] for i in range(d)]
        if degree == 2:
            pts += [0.5 * (pts[a] + pts[b]) for a, b in _EDGE_VERTS[d]]
        self.interpolation_points = np.array(pts)
        self.degree = degree


def _class_order(x: np.ndarray, lattice) -> np.ndarray:
    """Dof order for lattice (box/rectangle) meshes: group the P2 dofs by the parity class of their
    half-step lattice index (vertices, and one class per edge direction), lexicographic inside a
    class.  Consecutive dofs then have the same stencil, which is what lets a 32-row slice of the
    sliced-ELL operator gather 32 CONSECUTIVE vector entries per step (DESIGN.md, SpMM).  A permutation for any `x`:
    on coordinates off the lattice (a deformed box) the classes mix, which costs SpMM speed, not correctness."""
    p0, h = lattice
    idx = np.rint((x - p0) / (0.5 * h)).astype(np.int64)
    cls = (idx[:, 0] & 1) + 2 * (idx[:, 1] & 1) + 4 * (idx[:, 2] & 1)
    return np.lexsort((idx[:, 0], idx[:, 1], idx[:, 2], cls))


def lattice_node_index(mesh) -> np.ndarray:
    """(n_nodes, gdim) lattice indices of the geometry nodes of a provider-built box/rectangle mesh (lexicographic node
    numbering, x fastest); a slab-local mesh carries its own table."""
    idx = getattr(mesh, "_node_index", None)
    if idx is None:
        shape = mesh._shape
        v = np.arange(mesh.geometry.x.shape[0], dtype=np.int64)
        cols = []
        for a in range(len(shape)):
            cols.append(v % (shape[a] + 1))
            v = v // (shape[a] + 1)
        idx = mesh._node_index = np.stack(cols, axis=1)
    return idx


def lattice_dof_ids(hidx: np.ndarray, shape, degree: int, order: str) -> np.ndarray:
    """Dof number of the lattice points `hidx` (half-step indices for degree 2, node indices for degree 1) on a box of
    `shape` cubes: the closed form of `_class_order` ("class", degree 2: parity class of the half-step index, then
    lexicographic z, y, x inside the class) or of `_lex_order` (everything else)."""
    d = len(shape)
    h = [hidx[:, a] for a in range(d)]
    if degree == 1 or order != "class":
        n = [(s + 1) if degree == 1 else (2 * s + 1) for s in shape]
        g = h[d - 1].copy()
        for a in range(d - 2, -1, -1):
            g = g * n[a] + h[a]
        return g
    par = [h[a] & 1 for a in range(d)]
    cls = par[0] + 2 * par[1] + (4 * par[2] if d == 3 else 0)
    sizes = np.zeros(8 if d == 3 else 4, dtype=np.int64)
    for c in range(len(sizes)):  # N + 1 lattice points of even parity along an axis, N of odd parity
        sizes[c] = int(np.prod([shape[a] + 1 - ((c >> a) & 1) for a in range(d)]))
    offset = np.concatenate([[0], np.cumsum(sizes)[:-1]])
    j = [h[a] >> 1 for a in range(d)]
    g = j[d - 1].copy()
    for a in range(d - 2, -1, -1):
        g = g * np.where(par[a] == 0, shape[a] + 1, shape[a]) + j[a]
    return offset[cls] + g


def lattice_node_coordinates(mesh) -> np.ndarray:
    """(n_nodes, 3) coordinates the box/rectangle provider gives the geometry nodes: per axis, ``np.linspace`` over the
    box evaluated at the node's lattice index -- bitwise what `mesh.create_box` / `create_rectangle` (and a slab of
    either) store."""
    idx, shape = lattice_node_index(mesh), mesh._shape
    p0, p1 = mesh._box
    x = np.zeros((len(idx), 3))
    for a in range(len(shape)):
        x[:, a] = np.linspace(p0[a], p1[a], shape[a] + 1)[idx[:, a]]
    return x


def is_deformed(mesh) -> bool:
    """True if the nodes of a provider-built box/rectangle mesh are no longer where the provider put them: the mesh
    was moved in place (``mesh.geometry.x[:, 0] = ...``, e.g. graded toward the walls).  Its topology, node numbering
    and lattice attributes are still the box's, its coordinates are not.  O(n_nodes)."""
    return not np.array_equal(mesh.geometry.x, lattice_node_coordinates(mesh))


def _p2_coordinates_from_geometry(mesh, cell_dofs: np.ndarray, n_dofs: int) -> np.ndarray:
    """P2 dof coordinates from the actual geometry: vertex dofs at their nodes, edge dofs at 0.5 * (x_a + x_b) of the
    edge's end points (`_EDGE_VERTS` order) -- what the general route computes, for any numbering of the dofs."""
    gx, cells, d = mesh.geometry.x, mesh.geometry.dofmap, mesh.geometry.dim
    x = np.empty((n_dofs, 3))
    x[cell_dofs[:, : d + 1]] = gx[cells]
    for e, (a, b) in enumerate(_EDGE_VERTS[d]):
        x[cell_dofs[:, d + 1 + e]] = 0.5 * (gx[cells[:, a]] + gx[cells[:, b]])
    return x


def _lattice_p2(mesh):
    """(dof coordinates, cell dofs) of the P2 space on a provider-built box/rectangle mesh in the stencil-class order,
    from closed forms: the 3^d lattice points of every cube get their dof numbers by `lattice_dof_ids`, a cell's ten
    (six) dofs are a fixed selection of them, and the coordinates of a class are a tensor product of per-axis tables.
    No edge table, no sort -- the general route spends most of the host set-up of a 96^3 box in np.unique over 37 M cell
    edges and a four-key lexsort of 7 M points.  Same numbers and bitwise the same coordinates as the general route
    (tests/test_host.py).

    The numbering depends on the topology alone, the closed-form coordinates on the box.  A box deformed in place
    keeps the first and not the second: there the coordinates are taken from the geometry instead."""
    d, shape = mesh.geometry.dim, mesh._shape
    p0, p1 = mesh._box
    # per-axis coordinate of a half-step index: a node's own coordinate, or the midpoint of its two neighbours --
    # exactly what 0.5 * (x_a + x_b) gives for an edge whose end points differ by at most one step along the axis
    tabs = []
    for a in range(d):
        ax = np.linspace(p0[a], p1[a], shape[a] + 1)
        t = np.empty(2 * shape[a] + 1)
        t[0::2] = ax
        t[1::2] = 0.5 * (ax[:-1] + ax[1:])
        tabs.append(t)
    n = int(np.prod([2 * s_ + 1 for s_ in shape]))
    x = np.zeros((n, 3))
    off = 0
    for cls in range(2**d):  # classes in order, lexicographic (z, y, x) inside: a tensor product per class
        sel = [tabs[a][(cls >> a) & 1::2] for a in range(d)]
        grids = np.meshgrid(*sel[::-1], indexing="ij")  # slowest axis first
        m = grids[0].size
        for a in range(d):
            x[off:off + m, a] = grids[d - 1 - a].ravel()
        off += m
    # dof numbers of the 3^d lattice points of every cube, cube index lexicographic with x fastest (the cell order)
    cube = np.stack([g.ravel() for g in np.meshgrid(*[np.arange(s_) for s_ in shape[::-1]], indexing="ij")][::-1], axis=1)
    pts = {}
    for o in np.ndindex(*(3,) * d):
        pts[o] = lattice_dof_ids(2 * cube + np.array(o), shape, 2, "class")
    corner = lambda c: tuple((c >> a) & 1 for a in range(d))
    cols = []
    for cell in _BOX_CELLS[d]:
        cv = [corner(c) for c in cell]
        verts = [pts[tuple(2 * o for o in v)] for v in cv]
        edges = [pts[tuple(cv[a][k] + cv[b][k] for k in range(d))] for a, b in _EDGE_VERTS[d]]
        cols.append(np.stack(verts + edges, axis=1))
    cell_dofs = np.stack(cols, axis=1).reshape(-1, cols[0].shape[1])  # (cube, cell in cube) -> rows
    if is_deformed(mesh):
        x = _p2_coordinates_from_geometry(mesh, cell_dofs, n)
    return x, cell_dofs


def _lex_order(x: np.ndarray) -> np.ndarray:
    """Permutation sorting points by (z, y, x): spatial locality for SpMV gathers."""
    span = max(float(np.ptp(x)), 1e-300)
    q = np.round(x / span * 2**40).astype(np.int64)
    return np.lexsort((q[:, 0], q[:, 1], q[:, 2]))


def _sigma_order(x: np.ndarray, cell_dofs: np.ndarray, sigma: int = 2048) -> np.ndarray:
    """Dof order for meshes without lattice information ("sigma"): the coordinate sort, then inside every window of
    `sigma` consecutive dofs a stable sort by the number of adjacent cells (SELL-C-sigma's window sort, Kreutzer et al.
    2014 [ext]).  Dofs with equally many adjacent cells have (nearly) equally long matrix rows, so the 32-row slices
    of the sliced-ELL operator are padded far less than under the plain coordinate sort, where vertex rows (long) and
    edge rows (short) share slices; the window keeps the rows of a slice spatially close."""
    lex = _lex_order(x)
    adj = np.bincount(cell_dofs.ravel(), minlength=len(x))[lex]
    window = np.arange(len(lex)) // sigma
    return lex[np.lexsort((np.arange(len(lex)), -adj, window))]


class FunctionSpace:
    """Scalar Lagrange P1/P2 space (``bs == 1``) or its blocked vector version (``bs == gdim``)."""

    def __init__(self, mesh: Mesh, degree: int, bs: int = 1, _scalar: "FunctionSpace | None" = None):
        if degree not in (1, 2):
            raise NotImplementedError("only Lagrange degree 1 and 2 are on the B200 hot path")
        self.mesh = mesh
        self.degree = degree
        self.bs = bs
        self.element = _Element(mesh.cell_name(), degree)
        if _scalar is not None:
            self._x = _scalar._x
            self.dofmap = DofMap(_scalar.dofmap.list, _scalar.dofmap.index_map, bs)
            self._scalar = _scalar
            return
        self._scalar = self
        if (degree == 2 and getattr(mesh, "_canonical", False) and getattr(mesh, "_lattice", None) is not None
                and getattr(mesh, "_dof_order", "class") == "class"):
            self._x, cell_dofs = _lattice_p2(mesh)
            self.dofmap = DofMap(cell_dofs, IndexMap(self._x.shape[0]), 1)
            self._lattice_ids = True
            return
        cells = mesh.geometry.dofmap.astype(np.int64)
        nv = mesh.geometry.x.shape[0]
        if degree == 1:
            x = mesh.geometry.x
            cell_dofs = cells
        else:
            edges = mesh.topology.entities(1)
            ce = mesh.topology.cell_entities(1)
            x = np.vstack([mesh.geometry.x, 0.5 * (mesh.geometry.x[edges[:, 0]] + mesh.geometry.x[edges[:, 1]])])
            cell_dofs = np.hstack([cells, nv + ce])
        # renumber for locality (DOLFINx applies a graph reordering here [ext]); vertex-first
        # numbering would scatter every P2 row's columns over the whole vector
        lattice = getattr(mesh, "_lattice", None)
        kind = getattr(mesh, "_dof_order", "class")
        if kind != "class":
            lattice = None  # "generic" / "sigma": what a mesh without lattice information (unstructured) can get
        if lattice is not None and degree == 2:
            order = _class_order(x, lattice)
        elif degree == 2 and kind != "generic":  # no lattice information: window-sorted coordinate order (measured
            order = _sigma_order(x, cell_dofs)   # 0.76 of the HBM peak in the SpMM against 0.62 for the plain sort)
        else:
            order = _lex_order(x)
        new_of_old = np.empty(len(order), dtype=np.int64)
        new_of_old[order] = np.arange(len(order))
        self._x = np.ascontiguousarray(x[order])
        self.dofmap = DofMap(new_of_old[cell_dofs], IndexMap(len(order)), 1)
        if degree == 1:
            self._dof_nodes = order  # geometry node of every dof (the pressure multigrid's lattice indices)

    # -- dolfinx.fem.FunctionSpace surface -------------------------------------------------
    @property
    def num_sub_spaces(self) -> int:
        return self.bs if self.bs > 1 else 0

    def sub(self, i: int) -> "_SubSpace":
        assert 0 <= i < self.bs and self.bs > 1
        return _SubSpace(self, i)

    def tabulate_dof_coordinates(self) -> np.ndarray:
        return self._x

    @property
    def num_dofs(self) -> int:
        return self._x.shape[0]

    def entity_closure_dofs(self, edim: int, entities: np.ndarray) -> np.ndarray:
        """Sorted unique dofs on the closure of the given mesh entities."""
        top = self.mesh.topology
        ents = top.entities(edim)[np.asarray(entities, dtype=np.int64)]
        verts = np.unique(ents.ravel())
        cells = self.mesh.geometry.dofmap
        # vertex dof lookup: geometry vertex v -> dof, via any cell containing it
        vdof = np.empty(self.mesh.geometry.x.shape[0], dtype=np.int64)
        nvloc = cells.shape[1]
        vdof[cells.ravel()] = self.dofmap.list[:, :nvloc].ravel()
        dofs = [vdof[verts]]
        if self.degree == 2 and edim >= 1 and getattr(self, "_lattice_ids", False):
            # closed form: the midpoint of the edge between two vertices of an entity is the lattice point at the sum of
            # their lattice indices (no edge table)
            nidx, shape = lattice_node_index(self.mesh), self.mesh._shape
            k = ents.shape[1]
            for a in range(k):
                for b in range(a + 1, k):
                    dofs.append(lattice_dof_ids(nidx[ents[:, a]] + nidx[ents[:, b]], shape, 2, "class"))
        elif self.degree == 2 and edim >= 1:
            nv = self.mesh.geometry.x.shape[0]
            edges = top.entities(1)
            ekey = edges[:, 0] * nv + edges[:, 1]  # sorted by construction (np.unique)
            ce = top.cell_entities(1)
            edof = np.empty(len(edges), dtype=np.int64)
            edof[ce.ravel()] = self.dofmap.list[:, nvloc:].ravel()
            k = ents.shape[1]
            for a in range(k):
                for b in range(a + 1, k):
                    key = np.minimum(ents[:, a], ents[:, b]) * nv + np.maximum(ents[:, a], ents[:, b])
                    dofs.append(edof[np.searchsorted(ekey, key)])
        return np.unique(np.concatenate(dofs)).astype(np.int32)


class LocalFunctionSpace(FunctionSpace):
    """The part of a scalar space one rank holds in a multi-GPU run: owned dofs first, then ghosts
    (``oasisx_b200.partition.LocalSpace``); same surface as :class:`FunctionSpace`."""

    def __init__(self, gspace: FunctionSpace, lsp, bs: int = 1):
        self.mesh = gspace.mesh
        self.degree = gspace.degree
        self.bs = bs
        self.element = gspace.element
        self._g, self._l = gspace._scalar, lsp
        self._x = lsp.x
        self._scalar = self if bs == 1 else LocalFunctionSpace(gspace, lsp, 1)
        self.dofmap = DofMap(lsp.cell_dofs, IndexMap(lsp.n_owned, ghosts=lsp.l2g[lsp.n_owned:], size_global=lsp.n_global), bs)

    def entity_closure_dofs(self, edim: int, entities: np.ndarray) -> np.ndarray:
        loc = self._l.g2l[self._g.entity_closure_dofs(edim, entities)]
        return np.sort(loc[loc >= 0]).astype(np.int32)


class _SubSpace:
    def __init__(self, parent: FunctionSpace, i: int):
        self.parent, self.i = parent, i

    def collapse(self):
        """(component space, map into the blocked parent): ``map[j] = bs*j + i`` (Appendix D)."""
        Vi = self.parent._scalar
        n = Vi.num_dofs
        return Vi, np.arange(n, dtype=np.int32) * self.parent.bs + self.i


def slice_order(x: np.ndarray, n_rows: int, lattice=None, tile=(8, 8), rows_per_slice: int = 32) -> np.ndarray:
    """Schedule of the 32-row slices of the sliced-ELL operators: slices sorted by the spatial tile of
    their first row, so that all slices of one tile (every stencil class) are adjacent.  A tile spans
    one slice (32 dofs) in x and `tile` x-lines in y and z; on meshes without lattice information the
    tile edge is taken from the bounding box and the dof count."""
    n_slices = (n_rows + rows_per_slice - 1) // rows_per_slice
    first = x[np.arange(n_slices) * rows_per_slice]
    if lattice is not None:
        p0, h = lattice
    else:
        p0 = x.min(axis=0)
        ext = np.maximum(x.max(axis=0) - p0, 1e-300)
        dim = int(np.count_nonzero(ext > 1e-12 * ext.max()))
        h = np.where(ext > 1e-12 * ext.max(), ext / max(n_rows ** (1.0 / max(dim, 1)) / 2.0, 1.0), 1.0)
    q = np.floor((first - p0) / h + 1e-9).astype(np.int64)
    key = (q[:, 2] // tile[1], q[:, 1] // tile[0], q[:, 0] // rows_per_slice)
    return np.lexsort((np.arange(n_slices), key[2], key[1], key[0])).astype(np.int32)


def mass_jacobi_bounds(gdim: int, degree: int) -> tuple[float, float]:
    """[lambda_min, lambda_max] of diag(M_e)^-1 M_e on the reference simplex: bounds of the spectrum of the
    Jacobi-scaled assembled mass matrix on any affine mesh (element-by-element bound)."""
    import os

    t = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref_tables.npz"))
    M = t[f"D{gdim}P{degree}_MV"]
    d = np.sqrt(np.diag(M))
    w = np.linalg.eigvalsh(M / np.outer(d, d))
    return float(w[0]), float(w[-1])


def functionspace(mesh: Mesh, element) -> FunctionSpace:
    """``functionspace(mesh, ("Lagrange", k))`` or ``("Lagrange", k, (gdim,))``.  Scalar spaces of
    equal degree on one mesh share a dof map (one ``A`` serves every velocity component)."""
    family, degree = element[0], int(element[1])
    if family not in ("Lagrange", "CG", "P"):
        raise NotImplementedError(family)
    if hasattr(mesh, "is_global_boundary"):  # slab-local mesh of a multi-rank run: local space, owned dofs first
        from .slab import slab_functionspace

        return slab_functionspace(mesh, degree, int(element[2][0]) if len(element) > 2 and element[2] else 1)
    cache = mesh.__dict__.setdefault("_spaces", {})
    if degree not in cache:
        cache[degree] = FunctionSpace(mesh, degree)
    scalar = cache[degree]
    if len(element) > 2 and element[2]:
        return FunctionSpace(mesh, degree, bs=int(element[2][0]), _scalar=scalar)
    return scalar


class Constant:
    def __init__(self, mesh, value):
        self.value = np.asarray(value, dtype=np.float64)

    def __float__(self):
        return float(self.value)


class Vector:
    """Host mirror of a (possibly device-resident) vector; ``dolfinx.la.Vector`` look-alike."""

    def __init__(self, n: int):
        self._host = np.zeros(n, dtype=np.float64)
        self._binding = None  # object with pull(host) / push(host)
        self._dev_newer = False
        self._host_touched = False

    @property
    def array(self) -> np.ndarray:
        if self._binding is not None:
            if self._dev_newer:
                self._binding.pull(self._host)
                self._dev_newer = False
            self._host_touched = True
        return self._host

    def array_ro(self) -> np.ndarray:
        """Up-to-date host copy that the caller promises not to modify (no push-back)."""
        if self._binding is not None and self._dev_newer:
            self._binding.pull(self._host)
            self._dev_newer = False
        return self._host

    def flush(self):
        if self._binding is not None and self._host_touched:
            self._binding.push(self._host)
            self._host_touched = False

    def mark_device_written(self):
        self._dev_newer = True
        self._host_touched = False

    # serial: owner->ghost / ghost->owner exchanges are no-ops (multi-GPU halos live on the device)
    def scatter_forward(self):
        pass

    def scatter_reverse(self, mode=None):
        pass

    @property
    def petsc_vec(self):
        return self


class Function:
    def __init__(self, V: FunctionSpace, name: str = "f"):
        self.function_space = V
        self.name = name
        self.x = Vector(V.num_dofs * V.bs)

    def interpolate(self, f: Callable[[np.ndarray], np.ndarray]):
        """Nodal interpolation of ``f(x)``, ``x`` of shape (3, n) (``Function.interpolate`` for
        Lagrange, Appendix D)."""
        V = self.function_space
        vals = np.asarray(f(V.tabulate_dof_coordinates().T), dtype=np.float64)
        if V.bs == 1:
            self.x.array[:] = vals.reshape(-1)
        else:
            self.x.array[:] = np.ascontiguousarray(vals.reshape(V.bs, -1).T).reshape(-1)


def locate_dofs_topological(V: FunctionSpace, entity_dim: int, entities) -> np.ndarray:
    return V.entity_closure_dofs(entity_dim, np.asarray(entities))


def locate_dofs_geometrical(V: FunctionSpace, marker) -> np.ndarray:
    return np.flatnonzero(np.asarray(marker(V.tabulate_dof_coordinates().T), dtype=bool)).astype(np.int32)


def build_csr_pattern(row_dofs: np.ndarray, col_dofs: np.ndarray, n_rows: int, n_cols: int):
    """CSR sparsity of a cell-integral bilinear form: row r couples to every column dof of every
    cell containing r; columns sorted per row (``create_matrix`` semantics, Appendix D).
    Host/numpy builder used for small meshes and as the bit-exact check of the device builder."""
    nr, nc = row_dofs.shape[1], col_dofs.shape[1]
    rows = np.repeat(row_dofs.astype(np.int64), nc, axis=1).ravel()
    cols = np.tile(col_dofs.astype(np.int64), (1, nr)).ravel()
    key = np.unique(rows * n_cols + cols)
    r = key // n_cols
    indices = (key % n_cols).astype(np.int32)
    indptr = np.zeros(n_rows + 1, dtype=np.int64)
    np.add.at(indptr, r + 1, 1)
    indptr = np.cumsum(indptr)
    return indptr.astype(np.int32 if indptr[-1] < 2**31 else np.int64), indices
