"""Slab-local box/rectangle provider for one-rank-per-GPU runs.

``oasisx_b200.partition.partition`` cuts a GLOBAL mesh that every rank has built: simple, but the host set-up then
grows with the job (every rank numbers all dofs of the whole box) and a 8 x 128^3 weak-scaling box cannot be set up at
all.  A box mesh, its dof numbering (``fem._class_order`` / ``fem._lex_order``) and the slab partition are all closed
forms of the lattice indices, so a rank can build ONLY its slab: the cube layers it owns plus the one layer above
(whose cells touch the owned dofs of the slab's top plane).  ``create_slab_mesh`` does that, ``SlabFunctionSpace``
numbers the local dofs owned-first / ghosts-by-owner with their global ids from the closed forms, and ``local_problem``
returns exactly the ``partition.LocalProblem`` the global route produces -- array for array, which is what
``tests/test_slab.py`` asserts -- so nothing downstream (halo plans, device set-up, checkpoints) can tell the routes
apart.  DOLFINx plays this role in the reference: ``create_box(MPI.COMM_WORLD, ...)`` is distributed from the start
(``/root/reference/demo/taylor_green.py:126-131``).
"""
from __future__ import annotations

import numpy as np

from . import fem
from .mesh import Mesh
from .partition import HaloPlan, LocalProblem, LocalSpace

from .mesh import _BOX_CELLS  # noqa: E402

_TETS = _BOX_CELLS[3]


def layer_ranks(n_layers: int, nranks: int) -> np.ndarray:
    """Rank of each cube layer along the last axis: ``partition.cell_ranks`` for layers of equal cell count."""
    counts = np.ones(n_layers)
    cum = np.cumsum(counts)
    mid = cum - counts / 2.0
    lrank = np.minimum((mid * nranks / cum[-1]).astype(np.int64), nranks - 1)
    if n_layers >= nranks:
        for r in range(nranks):
            if not np.any(lrank == r):
                lrank = np.minimum(np.arange(n_layers) * nranks // n_layers, nranks - 1)
                break
    return lrank


class _SearchMap:
    """global id -> local index (or -1) without a table of the global size."""

    def __init__(self, l2g: np.ndarray):
        self._order = np.argsort(l2g, kind="stable")
        self._sorted = l2g[self._order]

    def __getitem__(self, g):
        g = np.asarray(g, dtype=np.int64)
        pos = np.searchsorted(self._sorted, g)
        pos = np.minimum(pos, len(self._sorted) - 1) if len(self._sorted) else pos
        hit = (self._sorted[pos] == g) if len(self._sorted) else np.zeros(g.shape, dtype=bool)
        return np.where(hit, self._order[pos], -1)


class SlabMesh(Mesh):
    """The cells one rank holds of a box (3D) or rectangle (2D) mesh cut into slabs along the last axis: owned layers
    ``[l0, l1)`` first, then the ghost layer ``l1`` (absent on the last rank).  ``geometry`` / ``topology`` are local;
    ``_shape``, ``_lattice``, ``_box`` describe the GLOBAL box (multigrid hierarchy, dof classes)."""

    @property
    def num_cells_global(self) -> int:
        return int(np.prod(self._shape)) * (6 if self.geometry.dim == 3 else 2)

    def is_global_boundary(self, verts: np.ndarray) -> np.ndarray:
        """Facets (rows of local vertex ids) lying on the boundary of the global box; the cut planes between slabs and
        the top of the ghost layer are not."""
        d = self.geometry.dim
        idx = self._node_index[verts]  # (n, k, d) global lattice indices
        on = np.zeros(len(verts), dtype=bool)
        for a in range(d):
            on |= (idx[:, :, a] == 0).all(axis=1) | (idx[:, :, a] == self._shape[a]).all(axis=1)
        return on


def create_slab_mesh(comm, points, n, gdim: int) -> SlabMesh:
    rank, nranks = int(comm.rank), int(comm.size)
    p0, p1 = (np.asarray(p, dtype=np.float64)[:gdim] for p in points)
    shape = tuple(int(v) for v in n)[:gdim]
    nl = shape[-1]
    if nl < nranks:
        raise ValueError(f"{nranks} ranks need at least {nranks} cube layers along the last axis, the mesh has {nl}")
    lrank = layer_ranks(nl, nranks)
    mine = np.flatnonzero(lrank == rank)
    l0, l1 = int(mine[0]), int(mine[-1]) + 1
    lg = min(l1 + 1, nl)  # one ghost layer above
    axes = [np.linspace(p0[a], p1[a], shape[a] + 1) for a in range(gdim)]  # the global provider's coordinates, bitwise
    planes = np.arange(l0, lg + 1)
    if gdim == 3:
        nx, ny, _ = shape
        Z, Y, X = np.meshgrid(axes[2][planes], axes[1], axes[0], indexing="ij")
        x = np.stack([X.ravel(), Y.ravel(), Z.ravel()], axis=1)
        KZ, KY, KX = np.meshgrid(planes, np.arange(ny + 1), np.arange(nx + 1), indexing="ij")
        node_index = np.stack([KX.ravel(), KY.ravel(), KZ.ravel()], axis=1)
        iz, iy, ix = np.meshgrid(np.arange(l0, lg), np.arange(ny), np.arange(nx), indexing="ij")
        sx, sy, sz = 1, nx + 1, (nx + 1) * (ny + 1)
        v0 = ((iz - l0) * sz + iy * sy + ix).ravel()
        v = [v0, v0 + sx, v0 + sy, v0 + sx + sy, v0 + sz, v0 + sx + sz, v0 + sy + sz, v0 + sx + sy + sz]
        cells = np.empty((len(v0), 6, 4), dtype=np.int64)
        for t, tet in enumerate(_TETS):
            cells[:, t] = np.stack([v[a] for a in tet], axis=1)
        cells = cells.reshape(-1, 4)
        cube = ((iz * ny + iy) * nx + ix).ravel()
        per = 6
    else:
        nx, _ = shape
        Y, X = np.meshgrid(axes[1][planes], axes[0], indexing="ij")
        x = np.stack([X.ravel(), Y.ravel()], axis=1)
        KY, KX = np.meshgrid(planes, np.arange(nx + 1), indexing="ij")
        node_index = np.stack([KX.ravel(), KY.ravel()], axis=1)
        iy, ix = np.meshgrid(np.arange(l0, lg), np.arange(nx), indexing="ij")
        v0 = ((iy - l0) * (nx + 1) + ix).ravel()
        v1, v2, v3 = v0 + 1, v0 + nx + 1, v0 + nx + 2
        cells = np.empty((len(v0), 2, 3), dtype=np.int64)
        cells[:, 0] = np.stack([v0, v1, v3], axis=1)
        cells[:, 1] = np.stack([v0, v2, v3], axis=1)
        cells = cells.reshape(-1, 3)
        cube = (iy * nx + ix).ravel()
        per = 2
    msh = SlabMesh(x, cells, gdim, comm)
    h = (p1 - p0) / np.array(shape, dtype=np.float64)
    pad = lambda a, fill: np.concatenate([a, np.full(3 - gdim, fill)])
    msh._lattice = (pad(p0, 0.0), pad(h, 1.0))
    msh._shape = shape
    msh._box = (p0.copy(), p1.copy())
    msh._layers = (l0, l1, lg)
    msh._layer_ranks = lrank
    msh._node_index = node_index
    msh._cells_global = (np.repeat(cube * per, per) + np.tile(np.arange(per), len(cube))).astype(np.int64)
    msh._n_cells_owned = (l1 - l0) * int(np.prod(shape[:-1])) * per
    return msh


def _owner_of(h_last: np.ndarray, lrank: np.ndarray, degree: int) -> np.ndarray:
    """Lowest rank whose cells touch the lattice plane/point with last-axis (half-)index `h_last`."""
    hh = h_last * 2 if degree == 1 else h_last
    layer = np.where(hh % 2 == 1, (hh - 1) // 2, np.maximum(hh // 2 - 1, 0))
    return lrank[layer].astype(np.int32)


def _slab_p2_block(mesh: SlabMesh):
    """(coordinates, cell dofs, half-step lattice indices) of the P2 dofs of a slab mesh, numbered along the slab's own
    block of the half-step lattice (x fastest) -- a preliminary local numbering the caller reorders owned-first.  Closed
    forms as in ``fem._lattice_p2``: no edge table, no sort over cell edges (which took most of the per-rank set-up)."""
    from .mesh import _BOX_CELLS, _EDGE_VERTS

    d, shape = mesh.geometry.dim, mesh._shape
    p0, p1 = mesh._box
    l0, _, lg = mesh._layers
    lo = [0] * (d - 1) + [2 * l0]                                   # first half-step index of the block per axis
    dims = [2 * shape[a] + 1 for a in range(d - 1)] + [2 * (lg - l0) + 1]
    tabs = []
    for a in range(d):
        ax = np.linspace(p0[a], p1[a], shape[a] + 1)                # the global provider's node coordinates, bitwise
        t = np.empty(2 * shape[a] + 1)
        t[0::2] = ax
        t[1::2] = 0.5 * (ax[:-1] + ax[1:])
        tabs.append(t[lo[a]:lo[a] + dims[a]])
    grids = np.meshgrid(*[np.arange(n) for n in dims[::-1]], indexing="ij")  # slowest axis first
    loc = [grids[d - 1 - a].ravel() for a in range(d)]             # block-local half-step indices, x fastest
    hidx = np.stack([loc[a] + lo[a] for a in range(d)], axis=1)
    x = np.zeros((len(hidx), 3))
    for a in range(d):
        x[:, a] = tabs[a][loc[a]]
    # cells: cube by cube in the slab mesh's order (layers l0 .. lg - 1, lexicographic, x fastest)
    ncube = [shape[a] for a in range(d - 1)] + [lg - l0]
    cg = np.meshgrid(*[np.arange(n) for n in ncube[::-1]], indexing="ij")
    cube = [cg[d - 1 - a].ravel() for a in range(d)]
    stride = [1]
    for a in range(1, d):
        stride.append(stride[-1] * dims[a - 1])
    flat = lambda off: sum((2 * cube[a] + off[a]) * stride[a] for a in range(d))
    corner = lambda c: tuple((c >> a) & 1 for a in range(d))
    cols = []
    for cell in _BOX_CELLS[d]:
        cv = [corner(c) for c in cell]
        verts = [flat(tuple(2 * o for o in v)) for v in cv]
        edges = [flat(tuple(cv[a][k] + cv[b][k] for k in range(d))) for a, b in _EDGE_VERTS[d]]
        cols.append(np.stack(verts + edges, axis=1))
    cell_dofs = np.stack(cols, axis=1).reshape(-1, cols[0].shape[1])
    return x, cell_dofs, hidx


def slab_functionspace(mesh: SlabMesh, degree: int, bs: int = 1):
    """Scalar (or blocked) Lagrange space on a slab mesh: ``fem.LocalFunctionSpace`` surface, local numbering
    owned-first then ghosts grouped by owner (each group in global order)."""
    cache = mesh.__dict__.setdefault("_spaces", {})
    if degree not in cache:
        cache[degree] = SlabFunctionSpace(mesh, degree)
    scalar = cache[degree]
    if bs > 1:
        return fem.FunctionSpace(mesh, degree, bs=bs, _scalar=scalar)
    return scalar


class SlabFunctionSpace(fem.FunctionSpace):
    def __init__(self, mesh: SlabMesh, degree: int):
        if degree not in (1, 2):
            raise NotImplementedError("only Lagrange degree 1 and 2 are on the B200 hot path")
        if fem.is_deformed(mesh):
            # the P2 coordinates and the halo plans below come from the box's closed forms and from coordinates
            raise NotImplementedError("a slab-local mesh moved in place is not supported: deform the replicated mesh "
                                      "(B200_GLOBAL_MESH=1), which oasisx_b200.partition cuts from the actual geometry")
        self.mesh, self.degree, self.bs = mesh, degree, 1
        self.element = fem._Element(mesh.cell_name(), degree)
        self._scalar = self
        d = mesh.geometry.dim
        cells = mesh.geometry.dofmap.astype(np.int64)
        nidx = mesh._node_index
        if degree == 1:
            x, cell_dofs, hidx = mesh.geometry.x, cells, nidx
        else:
            x, cell_dofs, hidx = _slab_p2_block(mesh)  # closed form on the slab's block of the half-step lattice
        order_kind = getattr(mesh, "_dof_order", "class")
        if order_kind == "sigma":
            raise NotImplementedError("the window-sorted dof order has no closed form: use 'class' or 'generic' on several ranks")
        gid = fem.lattice_dof_ids(hidx, mesh._shape, degree, order_kind)
        owner = _owner_of(hidx[:, d - 1], mesh._layer_ranks, degree)
        rank = int(mesh.comm.rank)
        mine = owner == rank
        # owned dofs in global order, then ghosts by (owner, global id): partition._local_space
        key_owner = np.where(mine, -1, owner)
        perm = np.lexsort((gid, key_owner))
        new_of_old = np.empty(len(perm), dtype=np.int64)
        new_of_old[perm] = np.arange(len(perm))
        n_owned = int(np.count_nonzero(mine))
        self._x = np.ascontiguousarray(x[perm])
        self._gid = gid[perm]
        self._owner = owner[perm]
        n_global = int(np.prod([(s + 1) if degree == 1 else (2 * s + 1) for s in mesh._shape]))
        self.dofmap = fem.DofMap(new_of_old[cell_dofs], fem.IndexMap(n_owned, ghosts=self._gid[n_owned:], owners=self._owner[n_owned:],
                                                                     size_global=n_global), 1)
        self._local = self._build_local(n_owned, n_global)

    def entity_closure_dofs(self, edim: int, entities: np.ndarray) -> np.ndarray:
        """Sorted unique local dofs on the closure of the given (local) mesh entities; for P2 from the lattice in closed
        form (vertex dofs at twice the node index, edge-midpoint dofs at the sum of the end points' indices)."""
        if self.degree == 1:
            return super().entity_closure_dofs(edim, entities)
        mesh = self.mesh
        ents = mesh.topology.entities(edim)[np.asarray(entities, dtype=np.int64)]
        nidx = mesh._node_index
        pts = [2 * nidx[np.unique(ents.ravel())]]
        k = ents.shape[1]
        for a in range(k):
            for b in range(a + 1, k):
                pts.append(nidx[ents[:, a]] + nidx[ents[:, b]])
        gids = np.unique(fem.lattice_dof_ids(np.vstack(pts), mesh._shape, 2, getattr(mesh, "_dof_order", "class")))
        return np.sort(self._local.g2l[gids]).astype(np.int32)

    def _build_local(self, n_owned: int, n_global: int) -> LocalSpace:
        mesh = self.mesh
        rank, nranks = int(mesh.comm.rank), int(mesh.comm.size)
        d = mesh.geometry.dim
        gid, owner = self._gid, self._owner
        gown = owner[n_owned:]
        # send side.  Rank q = rank - 1 holds my first layer as its ghost layer: it needs every dof of that layer I
        # own (all but the layer's bottom plane).  Rank q = rank + 1 owns the cells of my ghost layer: of my dofs
        # only the top plane of my slab is on them.  (partition.cell_holders, evaluated for slabs.)
        l0, l1, lg = mesh._layers
        hl = self._half_last()[:n_owned]
        send = {}
        if l0 > 0:
            m = hl <= 2 * l0 + 2
            if m.any():
                send[int(mesh._layer_ranks[l0 - 1])] = np.flatnonzero(m)
        if lg > l1:
            up = int(mesh._layer_ranks[l1])
            m = hl == 2 * l1
            if m.any():
                send[up] = np.flatnonzero(m)
        neighbors = np.array(sorted(set(np.unique(gown).tolist()) | set(send.keys())), dtype=np.int32)
        send_off, recv_off, send_idx = [0], [0], []
        for q in neighbors:
            s = send.get(int(q), np.zeros(0, dtype=np.int64))  # owned dofs are already in global order
            send_idx.append(s)
            send_off.append(send_off[-1] + len(s))
            recv_off.append(recv_off[-1] + int(np.count_nonzero(gown == q)))
        halo = HaloPlan(neighbors=neighbors, send_off=np.asarray(send_off, dtype=np.int64),
                        send_idx=(np.concatenate(send_idx) if send_idx else np.zeros(0, np.int64)).astype(np.int32),
                        recv_off=np.asarray(recv_off, dtype=np.int64))
        return LocalSpace(n_owned=n_owned, n_ghost=len(gid) - n_owned, n_global=n_global, l2g=gid.astype(np.int64),
                          g2l=_SearchMap(gid), cell_dofs=self.dofmap.list, halo=halo, x=self._x)

    def _half_last(self) -> np.ndarray:
        """Half-step lattice index along the slab axis of every local dof."""
        mesh = self.mesh
        d = mesh.geometry.dim
        p0, h = mesh._lattice
        return np.rint((self._x[:, d - 1] - p0[d - 1]) / (0.5 * h[d - 1])).astype(np.int64)


def local_problem(mesh: SlabMesh, deg_u: int, deg_p: int):
    """(LocalProblem, scalar velocity space, pressure space) of this rank: what ``partition.partition`` + two
    ``fem.LocalFunctionSpace`` give on a replicated mesh."""
    V = slab_functionspace(mesh, deg_u)
    Q = slab_functionspace(mesh, deg_p)
    lp = LocalProblem(rank=int(mesh.comm.rank), nranks=int(mesh.comm.size), cells=mesh._cells_global,
                      n_cells_owned=mesh._n_cells_owned, cell_nodes=mesh.geometry.dofmap)
    lp.V, lp.Q = V._local, Q._local
    return lp, V, Q
