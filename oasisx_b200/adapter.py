"""DOLFINx adapter: feed a real ``dolfinx.mesh.Mesh`` / ``dolfinx.fem.FunctionSpace`` to the B200 library.

DOLFINx cannot be installed in the build environment (SURVEY.md F3), so this module is exercised only
where it exists; it contains no numerics, only array extraction (SURVEY.md Appendix D list):

* ``mesh.geometry.x``, ``mesh.geometry.dofmap``                       -> ``b2_set_mesh``
* ``V.dofmap.list``, ``index_map.size_local / num_ghosts``            -> ``b2_set_space``
* ``index_map.ghosts / owners`` + the owners' send lists              -> ``b2_set_halo``
* ``bc._cpp_object.dof_indices()``                                    -> ``b2_set_velocity_bc_dofs``

With these arrays coming from DOLFINx, the CSR patterns built by ``b2_build_patterns`` are DOLFINx's
own (same cells, same dof numbers): compare ``Context.pattern`` with
``dolfinx.la.matrix_csr(dolfinx.fem.create_sparsity_pattern(form))`` for the bit-exact check.
One requirement beyond DOLFINx's defaults: the mesh must be created with
``ghost_mode=GhostMode.shared_vertex`` so that every rank holds the ghost cells touching its owned dofs
(owned matrix rows are then assembled without any exchange of matrix entries).
"""
from __future__ import annotations

import numpy as np

from . import fem as _fem
from .partition import HaloPlan, LocalProblem, LocalSpace


def is_foreign_mesh(mesh) -> bool:
    """True for a mesh that is not the built-in provider's (a ``dolfinx.mesh.Mesh``): it is consumed through this
    module -- geometry, dof maps and index maps are taken as they are (``fracstep.py:187-190,212``)."""
    from .mesh import Mesh

    return not isinstance(mesh, Mesh)


def _ghost_permutation(index_map):
    """DOLFINx keeps ghosts in discovery order; the library wants them grouped by owner, sorted by global index inside
    a group (one contiguous receive block per neighbour).  Returns new_of_old for the whole local range."""
    n_owned = index_map.size_local
    ghosts = np.asarray(index_map.ghosts, dtype=np.int64)
    owners = np.asarray(index_map.owners, dtype=np.int32)
    order = np.lexsort((ghosts, owners))  # old ghost position of the k-th ghost in the new order
    new_of_old = np.arange(n_owned + len(ghosts), dtype=np.int64)
    new_of_old[n_owned + order] = n_owned + np.arange(len(order))
    return new_of_old, ghosts[order], owners[order]


def halo_plan_from_index_map(index_map, comm, ghosts=None, owners=None) -> HaloPlan:
    """Pack/unpack lists of a ``dolfinx.common.IndexMap``: ghosts are received from their owners; what
    this rank must send is learnt from the other ranks' ghost lists (one all-to-all of global indices)."""
    n_owned = index_map.size_local
    ghosts = np.asarray(index_map.ghosts if ghosts is None else ghosts, dtype=np.int64)
    owners = np.asarray(index_map.owners if owners is None else owners, dtype=np.int32)
    lo, _ = index_map.local_range
    order = np.lexsort((ghosts, owners))
    if not np.array_equal(order, np.arange(len(order))):
        raise ValueError("ghosts must be grouped by owner (and sorted by global index inside a group); "
                         "permute the ghost block of the local numbering accordingly before calling the library")
    wanted = {int(q): ghosts[owners == q] for q in np.unique(owners)}  # what I need from rank q
    all_wanted = comm.allgather(wanted)  # all_wanted[r][q] = globals rank r needs from q
    me = comm.rank
    # np.asarray: oasisx_b200.comm.HostComm carries the arrays as plain lists
    send = {r: np.asarray(w[me], dtype=np.int64) for r, w in enumerate(all_wanted) if me in w and len(w[me])}
    neighbors = np.array(sorted(set(wanted) | set(send)), dtype=np.int32)
    send_off, recv_off, send_idx = [0], [0], []
    for q in neighbors:
        s = send.get(int(q), np.zeros(0, dtype=np.int64))
        send_idx.append((s - lo).astype(np.int32))  # owned entries: global - local_range[0]
        send_off.append(send_off[-1] + len(s))
        recv_off.append(recv_off[-1] + int(np.count_nonzero(owners == q)))
    assert recv_off[-1] == len(ghosts) and all((i >= 0).all() and (i < n_owned).all() for i in send_idx)
    return HaloPlan(neighbors, np.asarray(send_off, np.int64),
                    np.concatenate(send_idx).astype(np.int32) if send_idx else np.zeros(0, np.int32),
                    np.asarray(recv_off, np.int64))


def local_space_from_dolfinx(V, comm) -> LocalSpace:
    im = V.dofmap.index_map
    n_owned, n_ghost = im.size_local, im.num_ghosts
    lo, _ = im.local_range
    new_of_old, ghosts, owners = _ghost_permutation(im)
    l2g = np.concatenate([np.arange(lo, lo + n_owned, dtype=np.int64), ghosts])
    g2l = np.full(im.size_global, -1, dtype=np.int64)
    g2l[l2g] = np.arange(len(l2g))
    nd = V.dofmap.cell_dofs(0).shape[0]
    cell_dofs = np.ascontiguousarray(new_of_old[np.asarray(V.dofmap.list).reshape(-1, nd)], dtype=np.int32)
    x = np.empty((n_owned + n_ghost, 3))
    x[new_of_old] = np.asarray(V.tabulate_dof_coordinates())[: n_owned + n_ghost]
    sp = LocalSpace(n_owned=n_owned, n_ghost=n_ghost, n_global=im.size_global, l2g=l2g, g2l=g2l, cell_dofs=cell_dofs,
                    halo=halo_plan_from_index_map(im, comm, ghosts, owners), x=np.ascontiguousarray(x))
    sp.new_of_old = new_of_old
    sp.owners = owners
    return sp


def local_problem_from_dolfinx(mesh, Vi, Q) -> LocalProblem:
    """``Vi = V.sub(0).collapse()[0]`` (fracstep.py:190) and ``Q`` (fracstep.py:212) of a DOLFINx mesh."""
    comm = mesh.comm
    tdim = mesh.topology.dim
    cmap = mesh.topology.index_map(tdim)
    n_cells = cmap.size_local + cmap.num_ghosts
    cells = np.ascontiguousarray(np.asarray(mesh.geometry.dofmap).reshape(n_cells, -1)[:, : tdim + 1], dtype=np.int32)
    lp = LocalProblem(rank=comm.rank, nranks=comm.size, cells=np.arange(n_cells), n_cells_owned=cmap.size_local, cell_nodes=cells)
    lp.V = local_space_from_dolfinx(Vi, comm)
    lp.Q = local_space_from_dolfinx(Q, comm)
    return lp


class AdapterSpace(_fem.FunctionSpace):
    """A DOLFINx scalar Lagrange space seen through the surface the host layer uses (``oasisx_b200.fem.FunctionSpace``):
    local dofs owned-first with the ghost block regrouped by owner; dof LOCATION (boundary conditions) is delegated to
    DOLFINx and mapped through that regrouping."""

    def __init__(self, Vd, lsp: LocalSpace, bs: int = 1, _scalar=None):
        self.mesh = Vd.mesh
        self.degree = int(getattr(getattr(Vd, "element", None), "degree", None) or getattr(Vd.ufl_element(), "degree"))
        self.bs = bs
        self.element = Vd.element
        self._dolfinx, self._l = Vd, lsp
        self._x = lsp.x
        self._scalar = self if bs == 1 else (_scalar or AdapterSpace(Vd, lsp, 1))
        self.dofmap = _fem.DofMap(lsp.cell_dofs, _fem.IndexMap(lsp.n_owned, ghosts=lsp.l2g[lsp.n_owned:], owners=lsp.owners,
                                                             size_global=lsp.n_global, offset=int(lsp.l2g[0]) if lsp.n_owned else 0), bs)

    def entity_closure_dofs(self, edim: int, entities: np.ndarray) -> np.ndarray:
        import dolfinx

        d = np.asarray(dolfinx.fem.locate_dofs_topological(self._dolfinx, edim, np.asarray(entities, dtype=np.int32)), dtype=np.int64)
        return np.sort(self._l.new_of_old[d]).astype(np.int32)


def problem_from_dolfinx(mesh, deg_u: int, deg_p: int):
    """Spaces, local problem and geometry of a DOLFINx mesh for ``FractionalStep_AB_CN`` (``fracstep.py:187-190,212``):
    returns (LocalProblem, V blocked adapter space, Q adapter space, local geometry x)."""
    import dolfinx

    gdim = mesh.geometry.dim
    Vd = dolfinx.fem.functionspace(mesh, ("Lagrange", int(deg_u)))  # the collapsed component space: all Vi share its dof map
    Qd = dolfinx.fem.functionspace(mesh, ("Lagrange", int(deg_p)))
    lp = local_problem_from_dolfinx(mesh, Vd, Qd)
    Vs = AdapterSpace(Vd, lp.V, 1)
    V = AdapterSpace(Vd, lp.V, gdim, _scalar=Vs)
    Q = AdapterSpace(Qd, lp.Q, 1)
    x = np.zeros((np.asarray(mesh.geometry.x).shape[0], 3))
    x[:, : np.asarray(mesh.geometry.x).shape[1]] = np.asarray(mesh.geometry.x)
    return lp, V, Q, x
