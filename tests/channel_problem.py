"""The open channel of the reference's test/test_tentative_velocity.py on a box or rectangle [-1, 1]^d: inlet
callable at x_a = -1, no-slip walls, PressureBC outlet at x_a = 1 (a = `axis`, x by default) -- for the solver and for
the LU oracle.  Shared by the
tests of the pressure multigrid with PressureBCs and by tools/bench_amg.py."""
import sys

import numpy as np

import oasisx_b200 as oasisx
from oasisx_b200 import fem, mesh as bmesh

LU = {"ksp_type": "preonly", "pc_type": "lu"}
GAMG = {"ksp_type": "cg", "pc_type": "gamg", "ksp_rtol": 1e-12}


class Inlet:
    """(1 + t)(1 - y^2), y the first coordinate across the channel."""

    def __init__(self, t, across=1):
        self.t, self.across = t, across

    def eval(self, x):
        return (1 + self.t) * (1 - x[self.across] ** 2)


def _tags(msh, axis=0):
    """inlet x_axis = -1 (1), walls (2), outlet x_axis = 1 (3) of a box or rectangle [-1, 1]^d."""
    d = msh.topology.dim
    dim = d - 1
    left = bmesh.locate_entities_boundary(msh, dim, lambda x: np.isclose(x[axis], -1))
    right = bmesh.locate_entities_boundary(msh, dim, lambda x: np.isclose(x[axis], 1))
    walls = np.unique(np.hstack([bmesh.locate_entities_boundary(msh, dim, lambda x, k=k, v=v: np.isclose(x[k], v))
                                 for k in range(d) if k != axis for v in (-1.0, 1.0)]))
    walls = np.setdiff1d(walls, np.union1d(left, right))
    facets = np.hstack([left, walls, right])
    values = np.hstack([np.full_like(left, 1), np.full_like(walls, 2), np.full_like(right, 3)])
    order = np.argsort(facets)
    return left, walls, right, bmesh.meshtags(msh, dim, facets[order], values[order])


def channel(msh, deg=1, pressure=GAMG, low_memory=False, rotational=False, oracle=False, foreign=None,
            solver_options=None, device=0, axis=0, comm=None, p_out=4.0):
    """The open channel: inlet callable, no-slip walls, PressureBC(p_out) on the outlet.  Returns (solver, oracle or
    None, inlet).  solver_options: all three solvers (default: LU, `pressure`, LU).  oracle: True or the whole mesh
    (several ranks; `msh` is then this rank's mesh): the LU oracle of the same problem.  foreign: pytest's
    monkeypatch (or True: sys.modules itself) to take `msh` through the DOLFINx adapter (tests/fake_dolfinx.py), this
    rank's part of a partition over `comm` when given."""
    d = msh.geometry.dim
    left, walls, right, tags = _tags(msh, axis)
    smsh, stags = msh, tags
    if foreign is not None:
        from fake_dolfinx import make_fake

        mod, fmesh, _ = make_fake(msh, deg, 1, 1 if comm is None else comm.size, 0 if comm is None else comm.rank)
        if comm is not None:
            fmesh.comm = comm
        if foreign is True:
            sys.modules["dolfinx"] = mod
        else:
            foreign.setitem(sys.modules, "dolfinx", mod)
        smsh, stags = fmesh, fmesh.fake_tags(tags)
    inlet = Inlet(0.0, 1 if axis == 0 else 0)
    T = oasisx.LocatorMethod.TOPOLOGICAL
    bc_w = oasisx.DirichletBC(0.0, T, (stags, 2))
    bcs_u = [[oasisx.DirichletBC(inlet.eval if i == axis else 0.0, T, (stags, 1)), bc_w] for i in range(d)]
    s = oasisx.FractionalStep_AB_CN(smsh, ("Lagrange", deg), ("Lagrange", 1), bcs_u=bcs_u,
                                    bcs_p=[oasisx.PressureBC(p_out, (stags, 3))], rotational=rotational,
                                    solver_options=solver_options or {"tentative": LU, "pressure": pressure, "scalar": LU},
                                    options={"low_memory_version": low_memory}, device=device)
    o = None
    if oracle is not False:
        from oracle.ipcs_oracle import OracleIPCS
        from test_gpu_tentative import _global_pressure_facets

        if oracle is not True:
            msh = oracle
            left, walls, right, _ = _tags(msh, axis)
        dim = d - 1
        V, Q = fem.functionspace(msh, ("Lagrange", deg)), fem.functionspace(msh, ("Lagrange", 1))
        dl, dw = fem.locate_dofs_topological(V, dim, left), fem.locate_dofs_topological(V, dim, walls)
        o = OracleIPCS(msh.geometry.x, msh.geometry.dofmap, d, V.dofmap.list, Q.dofmap.list, V.tabulate_dof_coordinates(),
                       Q.tabulate_dof_coordinates(), deg,
                       bcs_u=[[(dl, inlet.eval if i == axis else 0.0), (dw, 0.0)] for i in range(d)],
                       bcs_p=[fem.locate_dofs_topological(Q, dim, right)], low_memory=low_memory, rotational=rotational,
                       pressure_facets=[_global_pressure_facets(msh, right) + (p_out,)])
    return s, o, inlet
