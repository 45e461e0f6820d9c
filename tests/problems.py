"""Shared problem set-ups for the parity tests: the Taylor-Green vortex of
``/root/reference/demo/taylor_green.py:36-53,126-182`` (2D, and its z-extruded 3D version,
SURVEY.md F5) built both for the CUDA path (``oasisx_b200``) and for the oracle."""
from __future__ import annotations

import numpy as np

from oasisx_b200 import fem, mesh as bmesh


class TaylorGreen:
    """The exact solution is separable, f(x) * g(t).  A caller that passes the SAME coordinate array again (the
    boundary conditions do, every time step) gets the spatial factor from a one-entry cache and only the scalar time
    factor is re-evaluated -- bitwise the same values as evaluating the full expression (same operation order), the
    way the reference's compiled ``Expression`` with a time ``Constant`` avoids re-deriving anything per step."""

    def __init__(self, nu: float, gdim: int):
        self.nu, self.gdim = nu, gdim
        self.t_u = 0.0
        self.t_p = 0.0
        self._cache = {}

    def _spatial(self, key, x, f):
        hit = self._cache.get(key)
        if hit is None or hit[0] is not x:
            hit = (x, f(x))
            self._cache[key] = hit
        return hit[1]

    def eval_x(self, x):
        return self._spatial("x", x, lambda x: -np.cos(np.pi * x[0]) * np.sin(np.pi * x[1])) * np.exp(-2.0 * self.nu * np.pi**2 * self.t_u)

    def eval_y(self, x):
        return self._spatial("y", x, lambda x: np.cos(np.pi * x[1]) * np.sin(np.pi * x[0])) * np.exp(-2.0 * self.nu * np.pi**2 * self.t_u)

    def eval_z(self, x):
        return np.zeros_like(x[0])

    def eval_p(self, x):
        return self._spatial("p", x, lambda x: -0.25 * (np.cos(2 * np.pi * x[0]) + np.cos(2 * np.pi * x[1]))) * np.exp(-4 * self.nu * np.pi**2 * self.t_p)

    @property
    def components(self):
        return [self.eval_x, self.eval_y, self.eval_z][: self.gdim]

    def trig_terms(self, which: str):
        """The field at the current time as trigonometric product terms (c, a[3], a0, b[3], b0, f1, f2, component) for
        the device-side evaluator of ``FractionalStep_AB_CN.assemble_l2_error_sq`` (1 = sin, 2 = cos, 0 = one)."""
        pi = np.pi
        if which == "p":
            g = -0.25 * np.exp(-4 * self.nu * pi**2 * self.t_p)
            return [[g, 2 * pi, 0, 0, 0, 0, 0, 0, 0, 2, 0, 0], [g, 0, 2 * pi, 0, 0, 0, 0, 0, 0, 2, 0, 0]]
        g = np.exp(-2.0 * self.nu * pi**2 * self.t_u)
        return [[-g, pi, 0, 0, 0, 0, pi, 0, 0, 2, 1, 0], [g, pi, 0, 0, 0, 0, pi, 0, 0, 1, 2, 1]]


class TaylorGreenRot(TaylorGreen):
    """The 2D Taylor-Green vortex of ``demo/taylor_green.py:36-53`` ROTATED out of the x-y plane: with an orthogonal
    R and in-plane coordinates (xi, eta) = (R^T x)[:2],

        u(x, t) = R[:, 0] u_xi(xi, eta, t) + R[:, 1] u_eta(xi, eta, t),   p(x, t) = p_2d(xi, eta, t).

    The Navier-Stokes equations are invariant under rotations, so this is still an exact solution on the box with
    Dirichlet data from the formula -- but all three velocity components are live and of the same size, unlike the
    z-extruded field (w = 0) whose z-systems are solved for free by a block-relative tolerance.  Same caching of the
    spatial factors as the parent class (one time factor per evaluation, bitwise reproducible)."""

    def __init__(self, nu: float, gdim: int = 3, axis=(1.0, 2.0, 3.0), angle_deg: float = 50.0):
        super().__init__(nu, 3)
        a = np.asarray(axis, dtype=np.float64)
        a /= np.linalg.norm(a)
        th = np.deg2rad(angle_deg)
        Kx = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
        self.R = np.eye(3) + np.sin(th) * Kx + (1 - np.cos(th)) * (Kx @ Kx)  # Rodrigues

    def _plane(self, x):
        R = self.R
        xi = R[0, 0] * x[0] + R[1, 0] * x[1] + R[2, 0] * x[2]
        eta = R[0, 1] * x[0] + R[1, 1] * x[1] + R[2, 1] * x[2]
        return xi, eta

    def _comp(self, k):
        def spatial(x):
            xi, eta = self._plane(x)
            return (self.R[k, 0] * (-np.cos(np.pi * xi) * np.sin(np.pi * eta))
                    + self.R[k, 1] * (np.cos(np.pi * eta) * np.sin(np.pi * xi)))

        def f(x):
            return self._spatial(("u", k), x, spatial) * np.exp(-2.0 * self.nu * np.pi**2 * self.t_u)

        return f

    def eval_p(self, x):
        def spatial(x):
            xi, eta = self._plane(x)
            return -0.25 * (np.cos(2 * np.pi * xi) + np.cos(2 * np.pi * eta))

        return self._spatial("p", x, spatial) * np.exp(-4 * self.nu * np.pi**2 * self.t_p)

    def trig_terms(self, which: str):
        pi, R = np.pi, self.R
        a, b = (pi * R[:, 0]).tolist(), (pi * R[:, 1]).tolist()
        if which == "p":
            g = -0.25 * np.exp(-4 * self.nu * pi**2 * self.t_p)
            return [[g, *(2 * pi * R[:, 0]), 0, 0, 0, 0, 0, 2, 0, 0], [g, *(2 * pi * R[:, 1]), 0, 0, 0, 0, 0, 2, 0, 0]]
        g = np.exp(-2.0 * self.nu * pi**2 * self.t_u)
        out = []
        for k in range(3):  # u_k = R[k,0] (-cos(pi xi) sin(pi eta)) g + R[k,1] (sin(pi xi) cos(pi eta)) g
            out.append([-g * R[k, 0], *a, 0, *b, 0, 2, 1, k])
            out.append([g * R[k, 1], *a, 0, *b, 0, 1, 2, k])
        return out

    @property
    def components(self):
        if not hasattr(self, "_comps"):
            self._comps = [self._comp(k) for k in range(3)]
        return self._comps


def make_mesh(gdim: int, N: int, comm=None):
    if gdim == 2:
        return bmesh.create_rectangle(comm, [[-1.0, -1.0], [1.0, 1.0]], [N, N])
    return bmesh.create_box(comm, [[-1.0, -1.0, -1.0], [1.0, 1.0, 1.0]], [N, N, N])


def _signed_dets(x, cells, gdim):
    X = x[cells][:, :, :gdim]
    return np.linalg.det(np.transpose(X[:, 1:] - X[:, :1], (0, 2, 1)))


def _scramble(msh, N, seed, keep=None):
    """`msh` rebuilt through ``Mesh(x, cells, gdim)``, so without lattice information: only the cells `keep` (all if
    None), the interior vertices moved by up to 0.2 h (boundary vertices, found from the exterior facets, stay put:
    Dirichlet data from a formula stays exact), node numbering, cell order and the vertex order inside every cell
    permuted at random.  Both orientations occur; min |det J| > 0.1 of the undeformed cells'."""
    gdim = msh.geometry.dim
    rng = np.random.default_rng(seed)
    cells = msh.geometry.dofmap.astype(np.int64)
    if keep is not None:
        cells = cells[keep]
    used, cells = np.unique(cells, return_inverse=True)
    cells = cells.reshape(-1, gdim + 1)
    x = msh.geometry.x[used].copy()
    tmp = bmesh.Mesh(x, cells, gdim)
    onb = np.zeros(len(x), dtype=bool)
    onb[np.unique(tmp.topology.entities(gdim - 1)[boundary_facets(tmp)])] = True
    h = 2.0 / N
    dirs = rng.normal(size=(len(x), gdim))
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    x[:, :gdim] += np.where(onb, 0.0, 0.2 * h * rng.uniform(0.0, 1.0, len(x)))[:, None] * dirs
    new_of_old = rng.permutation(len(x))
    xn = np.empty_like(x)
    xn[new_of_old] = x
    cells = new_of_old[cells][rng.permutation(len(cells))]
    cells = np.take_along_axis(cells, np.argsort(rng.uniform(size=cells.shape), axis=1), axis=1)
    det = _signed_dets(xn, cells, gdim)
    assert (det > 0).any() and (det < 0).any()
    assert np.abs(det).min() > 0.1 * h**gdim
    return bmesh.Mesh(xn[:, :gdim], cells, gdim)


def jittered_mesh(gdim: int, N: int, seed: int = 0):
    """The box/rectangle of `make_mesh` as an unstructured mesh: jittered interior, scrambled numbering, no lattice."""
    return _scramble(make_mesh(gdim, N), N, seed)


def l_shaped_mesh(gdim: int, N: int, seed: int = 0):
    """`jittered_mesh` with the cells of the quadrant (octant) x, y (, z) > 0 removed: a re-entrant corner, and a
    bounding box with an empty region.  Area 3 (volume 7)."""
    msh = make_mesh(gdim, N)
    cen = msh.geometry.x[msh.geometry.dofmap].mean(axis=1)[:, :gdim]
    return _scramble(msh, N, seed, keep=np.flatnonzero(~(cen > 0).all(axis=1)))


def mapped_box(gdim: int, N: int):
    """The provider mesh graded toward its centre planes IN PLACE (x_a -> sign(x_a) |x_a|^1.5, the usual DOLFINx
    idiom of moving ``mesh.geometry.x``): boundary planes fixed, volume unchanged, lattice attributes kept."""
    msh = make_mesh(gdim, N)
    x = msh.geometry.x
    for a in range(gdim):
        x[:, a] = np.sign(x[:, a]) * np.abs(x[:, a]) ** 1.5
    return msh


def boundary_facets(msh):
    d = msh.topology.dim
    msh.topology.create_connectivity(d - 1, d)
    return bmesh.exterior_facet_indices(msh.topology)


def make_oracle(msh, deg_u, tg: TaylorGreen, dt, **kw):
    from oracle.ipcs_oracle import OracleIPCS

    d = msh.geometry.dim
    V = fem.functionspace(msh, ("Lagrange", deg_u))
    Q = fem.functionspace(msh, ("Lagrange", 1))
    bd = fem.locate_dofs_topological(V, d - 1, boundary_facets(msh))
    o = OracleIPCS(msh.geometry.x, msh.geometry.dofmap, d, V.dofmap.list, Q.dofmap.list,
                   V.tabulate_dof_coordinates(), Q.tabulate_dof_coordinates(), deg_u,
                   bcs_u=[[(bd, f)] for f in tg.components], **kw)
    xV, xQ = V.tabulate_dof_coordinates().T, Q.tabulate_dof_coordinates().T
    tg.t_u = -dt
    o.u2 = [f(xV) for f in tg.components]
    tg.t_u = 0.0
    o.u1 = [f(xV) for f in tg.components]
    tg.t_p = -dt / 2
    o.p = tg.eval_p(xQ)
    return o


def make_solver(msh, deg_u, tg: TaylorGreen, dt, solver_options=None, low_memory=False, options=None, **kw):
    """The set-up of ``demo/taylor_green.py:135-182`` against oasisx_b200; `options` adds to the solver's options
    (e.g. ``{"multigrid": {...}}``)."""
    import oasisx_b200 as oasisx

    d = msh.geometry.dim
    facets = boundary_facets(msh)
    value = np.int32(3)
    tags = bmesh.meshtags(msh, d - 1, facets, np.full_like(facets, value, dtype=np.int32))
    bcs_u = [[oasisx.DirichletBC(f, oasisx.LocatorMethod.TOPOLOGICAL, (tags, value))] for f in tg.components]
    if solver_options is None:
        lu = {"ksp_type": "preonly", "pc_type": "lu"}
        solver_options = {"tentative": lu, "pressure": lu, "scalar": lu}
    s = oasisx.FractionalStep_AB_CN(msh, ("Lagrange", deg_u), ("Lagrange", 1), bcs_u=bcs_u, bcs_p=[],
                                    solver_options=solver_options, options={"low_memory_version": low_memory, **(options or {})}, **kw)
    tg.t_u = -dt
    for i, f in enumerate(tg.components):
        s._u2[i].interpolate(f)
    tg.t_u = 0.0
    for i, f in enumerate(tg.components):
        s._u1[i].interpolate(f)
    tg.t_p = -dt / 2
    s._p.interpolate(tg.eval_p)
    return s


def relerr(a, b, scale=None):
    """max|a-b| / scale, scale = max|b| unless given (pass the max over all components when one
    component is identically zero, e.g. w in the z-extruded Taylor-Green field)."""
    a, b = np.asarray(a), np.asarray(b)
    if scale is None:
        scale = np.max(np.abs(b))
    return float(np.max(np.abs(a - b)) / max(scale, 1e-300))


def vscale(vs):
    return max(float(np.max(np.abs(v))) for v in vs)


def make_cpu_port(msh, deg_u, tg: TaylorGreen, dt, **kw):
    """The same set-up for the C++/OpenMP CPU restatement (oracle/ipcs_cpu.cpp), which reaches meshes the LU oracle
    cannot and is itself pinned against that oracle in tests/test_cpu_port.py."""
    from oracle import ipcs_cpu as cpu

    d = msh.geometry.dim
    V, Q = fem.functionspace(msh, ("Lagrange", deg_u)), fem.functionspace(msh, ("Lagrange", 1))
    bd = fem.locate_dofs_topological(V, d - 1, boundary_facets(msh))
    c = cpu.CpuIPCS(msh.geometry.x, msh.geometry.dofmap, d, V.dofmap.list, Q.dofmap.list, V.tabulate_dof_coordinates(),
                    Q.tabulate_dof_coordinates(), deg_u, bcs_u=[[(bd, f)] for f in tg.components], **kw)
    xV, xQ = V.tabulate_dof_coordinates().T, Q.tabulate_dof_coordinates().T
    tg.t_u = -dt
    for i, f in enumerate(tg.components):
        c.set(cpu.U2, i, f(xV))
    tg.t_u = 0.0
    for i, f in enumerate(tg.components):
        c.set(cpu.U1, i, f(xV))
    tg.t_p = -dt / 2
    c.set(cpu.P, 0, tg.eval_p(xQ))
    return c
