"""Domain decomposition for one-rank-per-GPU runs (SURVEY.md 8e).

With DOLFINx the partition, the owned-first/ghosts-last index maps and the scatter plans come from
``mesh.topology.index_map`` / ``V.dofmap.index_map`` [ext]; this module produces the same *kind* of
data for the built-in provider: contiguous slabs of cells along the last axis, a dof owned by the
lowest rank whose cells touch it (the DOLFINx convention [ext]), local numbering = owned dofs (in
global order) followed by ghosts grouped by owner.  Every rank additionally holds the ghost cells
that touch one of its owned dofs, so that matrix rows of owned dofs are assembled completely
locally -- no matrix-entry communication (``Mat.assemble()`` stash exchange, fracstep.py:374-404,437)
is ever needed; only vectors are exchanged:

* forward halo (owner -> ghost)  == ``Vector.scatter_forward`` / the implicit ``MatMult`` gather,
* all-reduce of dot products     == ``KSP`` reductions / ``comm.allreduce`` (fracstep.py:581-589).
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np


@dataclass
class HaloPlan:
    """For neighbour k: send owned entries ``send_idx[send_off[k]:send_off[k+1]]`` (local indices),
    receive into ghost slots ``n_owned + recv_off[k] : n_owned + recv_off[k+1]``."""

    neighbors: np.ndarray
    send_off: np.ndarray
    send_idx: np.ndarray
    recv_off: np.ndarray


@dataclass
class LocalSpace:
    n_owned: int
    n_ghost: int
    n_global: int
    l2g: np.ndarray  # (n_owned + n_ghost,) global dof of each local dof
    g2l: np.ndarray  # (n_global,) local index or -1
    cell_dofs: np.ndarray  # (n_local_cells, nd) local dof ids
    halo: HaloPlan
    x: np.ndarray  # coordinates of the local dofs

    @property
    def n_local(self) -> int:
        return self.n_owned + self.n_ghost


@dataclass
class LocalProblem:
    rank: int
    nranks: int
    cells: np.ndarray  # global ids of the local cells: owned first, then ghost cells
    n_cells_owned: int
    cell_nodes: np.ndarray  # geometry dofmap of the local cells (global node ids: x is replicated)
    V: LocalSpace = field(default=None)
    Q: LocalSpace = field(default=None)


def cell_ranks(mesh, nranks: int) -> np.ndarray:
    """Slab partition of the cells along the last geometric axis, balanced by cell count."""
    d = mesh.geometry.dim
    cells = mesh.geometry.dofmap
    zc = mesh.geometry.x[cells][:, :, d - 1].mean(axis=1)
    lattice = getattr(mesh, "_lattice", None)
    if lattice is not None:  # any layer assignment is a valid partition: on a box deformed in place only the balance suffers
        p0, h = lattice
        layer = np.floor((zc - p0[d - 1]) / h[d - 1] + 1e-9).astype(np.int64)
    else:  # no lattice: rank the cells by centroid height and cut into equal chunks
        order = np.argsort(zc, kind="stable")
        layer = np.empty(len(zc), dtype=np.int64)
        layer[order] = np.arange(len(zc)) * max(nranks * 16, 1) // len(zc)
    nl = int(layer.max()) + 1
    counts = np.bincount(layer, minlength=nl)
    cum = np.cumsum(counts)
    total = cum[-1]
    # layer l goes to the rank whose quota its midpoint falls into
    mid = cum - counts / 2.0
    lrank = np.minimum((mid * nranks / total).astype(np.int64), nranks - 1)
    # guarantee every rank gets at least one layer when there are enough layers
    if nl >= nranks:
        for r in range(nranks):
            if not np.any(lrank == r):
                lrank = np.minimum(np.arange(nl) * nranks // nl, nranks - 1)
                break
    return lrank[layer].astype(np.int32)


def _owners(cell_dofs: np.ndarray, crank: np.ndarray, n_dofs: int, nranks: int) -> np.ndarray:
    owner = np.full(n_dofs, nranks, dtype=np.int32)
    np.minimum.at(owner, cell_dofs.ravel(), np.repeat(crank, cell_dofs.shape[1]))
    return owner


def cell_holders(crank: np.ndarray, owners_and_dofmaps, nranks: int) -> np.ndarray:
    """holders[c, q] = rank q keeps cell c in its local mesh: q is the cell's own rank, or q owns a dof of ANY of the
    spaces on the cell (the ghost-cell rule of `partition`: every cell touching an owned dof).  The send lists are
    derived from this -- the rule that builds each rank's ghost block -- and not from a per-space shortcut: a rank may
    hold a cell only through its cell rank or through the other space's ownership, and its ghosts include all dofs of
    that cell."""
    H = np.zeros((len(crank), nranks), dtype=bool)
    rows = np.arange(len(crank))
    H[rows, crank] = True
    for owner, dofmap in owners_and_dofmaps:
        O = owner[dofmap]
        for j in range(O.shape[1]):
            H[rows, O[:, j]] = True
    return H


def _local_space(space, cells_local: np.ndarray, owner: np.ndarray, rank: int, nranks: int,
                 holders: np.ndarray | None = None) -> LocalSpace:
    gd = space.dofmap.list.astype(np.int64)
    n_global = space.num_dofs
    owned = np.flatnonzero(owner == rank)
    touched = np.unique(gd[cells_local].ravel())
    ghosts = touched[owner[touched] != rank]
    ghosts = ghosts[np.lexsort((ghosts, owner[ghosts]))]
    l2g = np.concatenate([owned, ghosts]).astype(np.int64)
    g2l = np.full(n_global, -1, dtype=np.int64)
    g2l[l2g] = np.arange(len(l2g))
    # receive side: ghosts grouped by owner
    gown = owner[ghosts]
    neigh_recv = np.unique(gown)
    # send side: my owned dofs on every cell rank q holds  <=> q has them in its ghost block (same rule as q's own
    # `touched` set above, evaluated here without communication because the mesh is replicated)
    O = owner[gd]  # (n_cells, nd)
    send = {}
    mine_in_cell = (O == rank)
    has_mine = mine_in_cell.any(axis=1)
    for q in range(nranks):
        if q == rank:
            continue
        m = has_mine & (holders[:, q] if holders is not None else (O == q).any(axis=1))
        if not m.any():
            continue
        d = np.unique(gd[m][mine_in_cell[m]])
        if len(d):
            send[q] = d
    neighbors = np.array(sorted(set(neigh_recv.tolist()) | set(send.keys())), dtype=np.int32)
    send_off, recv_off, send_idx = [0], [0], []
    for q in neighbors:
        s = send.get(int(q), np.zeros(0, dtype=np.int64))
        send_idx.append(g2l[s])
        send_off.append(send_off[-1] + len(s))
        recv_off.append(recv_off[-1] + int(np.count_nonzero(gown == q)))
    halo = HaloPlan(
        neighbors=neighbors,
        send_off=np.asarray(send_off, dtype=np.int64),
        send_idx=(np.concatenate(send_idx) if send_idx else np.zeros(0, np.int64)).astype(np.int32),
        recv_off=np.asarray(recv_off, dtype=np.int64),
    )
    return LocalSpace(
        n_owned=len(owned), n_ghost=len(ghosts), n_global=n_global, l2g=l2g, g2l=g2l,
        cell_dofs=g2l[gd[cells_local]].astype(np.int32), halo=halo,
        x=np.ascontiguousarray(space.tabulate_dof_coordinates()[l2g]),
    )


def partition(mesh, V, Q, nranks: int, rank: int) -> LocalProblem:
    """Local view of rank `rank`: owned + ghost cells, owned-first dof numbering and halo plans for the
    velocity-component space V and the pressure space Q."""
    crank = cell_ranks(mesh, nranks)
    ownV = _owners(V.dofmap.list, crank, V.num_dofs, nranks)
    ownQ = _owners(Q.dofmap.list, crank, Q.num_dofs, nranks)
    mine = crank == rank
    touches = (ownV[V.dofmap.list] == rank).any(axis=1) | (ownQ[Q.dofmap.list] == rank).any(axis=1)
    owned_cells = np.flatnonzero(mine)
    ghost_cells = np.flatnonzero(touches & ~mine)
    cells_local = np.concatenate([owned_cells, ghost_cells])
    lp = LocalProblem(rank=rank, nranks=nranks, cells=cells_local, n_cells_owned=len(owned_cells),
                      cell_nodes=np.ascontiguousarray(mesh.geometry.dofmap[cells_local]))
    holders = cell_holders(crank, [(ownV, V.dofmap.list), (ownQ, Q.dofmap.list)], nranks)
    lp.V = _local_space(V, cells_local, ownV, rank, nranks, holders)
    lp.Q = _local_space(Q, cells_local, ownQ, rank, nranks, holders)
    return lp


def check_halo_counts(comm, halo: HaloPlan, name: str = ""):
    """Cross-check over the ranks, before the first exchange: what rank r sends to q is what q expects from r
    (a mismatch would hang or corrupt the grouped ncclSend/ncclRecv)."""
    me = {"n": halo.neighbors.tolist(), "s": np.diff(halo.send_off).tolist(), "r": np.diff(halo.recv_off).tolist()}
    plans = comm.allgather(me)
    r = comm.rank
    for k, q in enumerate(me["n"]):
        other = plans[int(q)]
        if r not in other["n"]:
            raise RuntimeError(f"halo plan {name}: rank {r} lists {q} as neighbour but not vice versa")
        kq = other["n"].index(r)
        if other["r"][kq] != me["s"][k] or other["s"][kq] != me["r"][k]:
            raise RuntimeError(f"halo plan {name}: rank {r} <-> {q} counts disagree: send {me['s'][k]} vs recv "
                               f"{other['r'][kq]}, recv {me['r'][k]} vs send {other['s'][kq]}")


def halo_forward_numpy(plans: list[HaloPlan], n_owned: list[int], vectors: list[np.ndarray]):
    """Reference (single-process) execution of the forward halo on all ranks at once: used by the CPU
    tests and as the statement of what the NCCL path must do."""
    for r, plan in enumerate(plans):
        for k, q in enumerate(plan.neighbors):
            qplan = plans[int(q)]
            kq = int(np.flatnonzero(qplan.neighbors == r)[0])
            sent = vectors[int(q)][qplan.send_idx[qplan.send_off[kq]:qplan.send_off[kq + 1]]]
            lo, hi = n_owned[r] + plan.recv_off[k], n_owned[r] + plan.recv_off[k + 1]
            assert hi - lo == len(sent), (r, q, hi - lo, len(sent))
            vectors[r][lo:hi] = sent
