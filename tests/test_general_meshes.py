"""Host side on meshes that are not uniform boxes (tests/problems.py: `jittered_mesh`, `l_shaped_mesh`, `mapped_box`).

A box deformed in place keeps its lattice attributes, and with them the closed-form P2 space of `fem._lattice_p2`: its
dof coordinates must follow the geometry, not the undeformed box.  The parity tests cannot see such an error (device and
oracle are handed the same coordinates), the interpolation identity below can.  The CPU port is checked against the
LU oracle on the unstructured meshes because the medium-size GPU tests use it as their reference."""
import numpy as np
import pytest

from oasisx_b200 import fem
from oasisx_b200 import multigrid as mg
from oracle import ipcs_cpu as cpu
from problems import (TaylorGreen, jittered_mesh, l_shaped_mesh, make_cpu_port, make_mesh, make_oracle, mapped_box,
                      relerr, vscale)


def quadratic(x):
    return x[0] ** 2 + 3.0 * x[1] * x[2] - 0.5 * x[0] * x[1] + x[1]


@pytest.mark.parametrize("gdim,N", [(3, 4), (2, 8)])
def test_p2_dof_coordinates_follow_a_box_deformed_in_place(gdim, N):
    msh = mapped_box(gdim, N)
    assert fem.is_deformed(msh) and not fem.is_deformed(make_mesh(gdim, N))
    V = fem.functionspace(msh, ("Lagrange", 2))
    assert getattr(V, "_lattice_ids", False)  # still the closed-form numbering
    x, gx = V.tabulate_dof_coordinates(), msh.geometry.x
    cells, dofs = msh.geometry.dofmap, V.dofmap.list
    np.testing.assert_array_equal(x[dofs[:, : gdim + 1]], gx[cells])  # vertex dofs: exactly the nodes
    for e, (a, b) in enumerate(fem._EDGE_VERTS[gdim]):  # edge dofs: midpoints of the actual edges
        np.testing.assert_array_equal(x[dofs[:, gdim + 1 + e]], 0.5 * (gx[cells[:, a]] + gx[cells[:, b]]))
    # P2 reproduces a quadratic exactly, on any affine mesh: the interpolant's L2 error vanishes
    o = make_oracle(msh, 2, TaylorGreen(0.01, gdim), 0.01)
    err = o.F.l2_error_sq([quadratic(o.xV.T)], o.vdofs, [quadratic], degree=4)
    assert err <= 1e-24, err


@pytest.mark.parametrize("kind", ["box", "rectangle"])
def test_geometry_route_is_the_closed_form_on_an_undeformed_box(kind):
    """The deformed-box route of `_lattice_p2` gives bitwise the closed-form coordinates when nothing moved."""
    msh = make_mesh(3 if kind == "box" else 2, 5)
    x, dofs = fem._lattice_p2(msh)
    np.testing.assert_array_equal(fem._p2_coordinates_from_geometry(msh, dofs, len(x)), x)


def test_multigrid_hierarchy_of_a_deformed_box_follows_the_node_numbering():
    """Lattice indices of the pressure dofs from the node numbering (not from rounded coordinates, which a deformed box
    breaks); coarse levels on the deformed fine geometry at the even lattice nodes."""
    msh = mapped_box(3, 8)
    Q = fem.functionspace(msh, ("Lagrange", 1))
    idx = fem.lattice_node_index(msh)[Q._dof_nodes]
    np.testing.assert_array_equal(fem.lattice_node_coordinates(msh)[Q._dof_nodes], make_mesh(3, 8).geometry.x[Q._dof_nodes])
    assert len(np.unique(mg._node_ids(idx, msh._shape))) == Q.num_dofs
    levels = mg.box_hierarchy(msh, first_rows=idx, fine_x=msh.geometry.x)
    assert [lv[0]._shape for lv in levels] == [(4, 4, 4), (2, 2, 2)]
    cm = levels[0][0]
    even = mg._node_ids(2 * fem.lattice_node_index(cm), msh._shape)
    np.testing.assert_array_equal(cm.geometry.x, msh.geometry.x[even])
    # the first prolongation maps the coarse interpolant of a linear function in lattice index space onto the fine one
    P = levels[0][1]
    lin = lambda i: 1.0 + i[:, 0] - 2.0 * i[:, 1] + 0.5 * i[:, 2]
    np.testing.assert_allclose(P @ lin(2.0 * fem.lattice_node_index(cm)), lin(idx.astype(float)), rtol=0, atol=1e-12)


def test_slab_mesh_moved_in_place_is_refused():
    from oasisx_b200 import mesh as bmesh
    from test_slab import FakeComm

    m = bmesh.create_box(FakeComm(0, 2), [[0, 0, 0], [1, 1, 1]], [2, 2, 4])
    m.geometry.x[:, 0] = m.geometry.x[:, 0] ** 2
    with pytest.raises(NotImplementedError, match="moved in place"):
        fem.functionspace(m, ("Lagrange", 2))


@pytest.mark.parametrize("factory,gdim,N,deg", [(jittered_mesh, 3, 4, 2), (l_shaped_mesh, 3, 4, 2), (jittered_mesh, 2, 8, 2),
                                                (l_shaped_mesh, 2, 8, 2), (jittered_mesh, 3, 4, 1), (l_shaped_mesh, 2, 8, 1)])
def test_cpu_port_matches_the_oracle_on_unstructured_meshes(factory, gdim, N, deg):
    dt, nu = 0.005, 0.01
    msh = factory(gdim, N, seed=1)
    assert not hasattr(msh, "_lattice")
    tg, tg2 = TaylorGreen(nu, gdim), TaylorGreen(nu, gdim)
    c = make_cpu_port(msh, deg, tg, dt, rtol=1e-13)
    o = make_oracle(msh, deg, tg2, dt)
    for t in (tg, tg2):
        t.t_u, t.t_p = 0.0, -dt / 2
    for n in range(3):
        for t in (tg, tg2):
            t.t_u += dt
            t.t_p += dt
        c.solve(dt, nu)
        o.solve(dt, nu, max_iter=1)
        for i in range(gdim):
            assert relerr(c.get(cpu.U, i), o.u[i], vscale(o.u)) <= 1e-9, (n, i)
        assert relerr(c.get(cpu.P), o.p) <= 1e-9, n
