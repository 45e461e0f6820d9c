"""ctypes wrapper of oracle/libipcs_cpu.so (C++/OpenMP CPU restatement; test + baseline infrastructure,
never imported by the product path)."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from .build_cpu import LIB, build

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB):
            build()
        L = C.CDLL(LIB)
        vp, i32, i64, dbl = C.c_void_p, C.c_int, C.c_int64, C.c_double
        L.ipcs_cpu_threads.restype = i32
        L.ipcs_cpu_set_threads.argtypes = [i32]
        L.ipcs_cpu_numa_interleave.restype = i32
        L.ipcs_cpu_stream_triad.restype = dbl
        L.ipcs_cpu_stream_triad.argtypes = [i64, i32]
        L.ipcs_cpu_create.restype = vp
        L.ipcs_cpu_create.argtypes = [i32, i32, i64, vp, i64, vp, i64, vp, i64, vp]
        L.ipcs_cpu_destroy.argtypes = [vp]
        L.ipcs_cpu_nnz.restype = i64
        L.ipcs_cpu_nnz.argtypes = [vp, i32]
        L.ipcs_cpu_get_pattern.argtypes = [vp, i32, vp, vp]
        L.ipcs_cpu_set_bc.argtypes = [vp, i32, i64, vp]
        L.ipcs_cpu_set_bc_values.argtypes = [vp, i32, vp]
        L.ipcs_cpu_set_options.argtypes = [vp, dbl, i32, i32]
        L.ipcs_cpu_set_block_rtol.argtypes = [vp, i32]
        L.ipcs_cpu_set_extrapolate.argtypes = [vp, i32]
        L.ipcs_cpu_preassemble.argtypes = [vp, vp]
        L.ipcs_cpu_set_vec.argtypes = [vp, i32, i32, vp]
        L.ipcs_cpu_get_vec.argtypes = [vp, i32, i32, vp]
        L.ipcs_cpu_get_matrix.argtypes = [vp, i32, i32, vp]
        L.ipcs_cpu_mg_add_level.argtypes = [vp, i32, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp]
        L.ipcs_cpu_mg_set_dense.argtypes = [vp, i32, vp]
        L.ipcs_cpu_set_pressure_mg.argtypes = [vp, i32, dbl]
        L.ipcs_cpu_bench_strategies.argtypes = [vp, i32, dbl, dbl, i32, vp, vp, vp]
        L.ipcs_cpu_step.restype = i32
        L.ipcs_cpu_step.argtypes = [vp, dbl, dbl, vp]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def use_all_cores() -> dict:
    """Pin the OpenMP team of the CPU port to every core this process may run on (the CPU affinity mask), whatever
    OMP_NUM_THREADS says (torch.distributed.run exports OMP_NUM_THREADS=1), and interleave its pages over the NUMA
    nodes.  Call before the first CpuIPCS is built.  Returns what was set, for the bench line."""
    L = lib()
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    L.ipcs_cpu_set_threads(int(n))
    nodes = L.ipcs_cpu_numa_interleave()
    return {"threads": int(L.ipcs_cpu_threads()), "affinity_cpus": int(n), "host_cpus": os.cpu_count(),
            "omp_num_threads_env": os.environ.get("OMP_NUM_THREADS"), "numa_nodes_interleaved": int(nodes)}


def stream_triad_gbs(n: int = 1 << 26, reps: int = 5) -> float:
    """STREAM triad on the host with the port's thread team (GB/s, 24 B per element, best of reps)."""
    return float(lib().ipcs_cpu_stream_triad(int(n), int(reps)))


U, U1, U2, P, PS, DP, RHS1, BFIRST, B2, UAB = range(10)


class CpuIPCS:
    """Same problem description as ``OracleIPCS`` (one BC per component: (dofs, callable))."""

    def __init__(self, x, cells, d, vdofs, qdofs, xV, xQ, deg_v, bcs_u, rtol=1e-10, nonzero_guess=False, body_force=None,
                 block_rtol=False, extrapolate=False):
        L = lib()
        self.L, self.d = L, d
        x = np.ascontiguousarray(x, np.float64)
        cells = np.ascontiguousarray(cells, np.int32)
        vdofs = np.ascontiguousarray(vdofs, np.int32)
        qdofs = np.ascontiguousarray(qdofs, np.int32)
        self.nV, self.nQ, self.xV, self.xQ = xV.shape[0], xQ.shape[0], xV, xQ
        self._dof_nodes = np.empty(self.nQ, dtype=np.int64)  # P1: geometry node of every pressure dof
        self._dof_nodes[qdofs.ravel()] = cells.ravel()
        self.h = C.c_void_p(L.ipcs_cpu_create(d, deg_v, x.shape[0], _p(x), cells.shape[0], _p(cells), self.nV, _p(vdofs),
                                              self.nQ, _p(qdofs)))
        self.bcs_u = bcs_u
        for i, bcl in enumerate(bcs_u):
            dofs = np.ascontiguousarray(bcl[0][0], np.int32)
            L.ipcs_cpu_set_bc(self.h, i, len(dofs), _p(dofs))
        L.ipcs_cpu_set_options(self.h, rtol, 10000, int(nonzero_guess))
        L.ipcs_cpu_set_block_rtol(self.h, int(block_rtol))
        L.ipcs_cpu_set_extrapolate(self.h, int(extrapolate))
        f = np.ascontiguousarray(list(body_force or [0.0] * d) + [0.0] * (3 - d), np.float64)
        L.ipcs_cpu_preassemble(self.h, _p(f))
        self.its = np.zeros(3, np.int32)

    def __del__(self):
        try:
            self.L.ipcs_cpu_destroy(self.h)
        except Exception:
            pass

    def update_bcs(self):
        for i, bcl in enumerate(self.bcs_u):
            dofs, val = bcl[0]
            v = np.ascontiguousarray(val(self.xV[dofs].T), np.float64)
            self.L.ipcs_cpu_set_bc_values(self.h, i, _p(v))

    def set(self, which, comp, v):
        v = np.ascontiguousarray(v, np.float64)
        self.L.ipcs_cpu_set_vec(self.h, which, comp, _p(v))

    def get(self, which, comp=0):
        out = np.empty(self.nQ if which in (P, PS, DP, B2) else self.nV)
        self.L.ipcs_cpu_get_vec(self.h, which, comp, _p(out))
        return out

    def pattern(self, which, n_rows):
        nnz = self.L.ipcs_cpu_nnz(self.h, which)
        ip, ix = np.empty(n_rows + 1, np.int32), np.empty(nnz, np.int32)
        self.L.ipcs_cpu_get_pattern(self.h, which, _p(ip), _p(ix))
        return ip, ix

    def matrix(self, which, comp, nnz):
        out = np.empty(nnz)
        self.L.ipcs_cpu_get_matrix(self.h, which, comp, _p(out))
        return out

    def attach_pressure_multigrid(self, msh, dense_max: int = 5000, omega: float = 0.85) -> int:
        """The GPU arm's pressure preconditioner on the CPU (pc_type=mg): nested box/rectangle hierarchy from the mesh
        provider, Galerkin coarse operators (= the stiffness matrices of the coarse meshes: the P1 spaces are nested),
        V(1,1) damped-Jacobi cycle, exact dense solve on the first level with at most `dense_max` dofs.  Returns the
        number of coarse levels (0: the mesh carries no hierarchy, Jacobi stays)."""
        import scipy.sparse as sp

        from oasisx_b200 import multigrid as mg

        levels = mg.box_hierarchy(msh)
        if not levels:
            return 0
        nnz = self.L.ipcs_cpu_nnz(self.h, 3)
        ip, ix = self.pattern(3, self.nQ)
        A = sp.csr_matrix((self.matrix(3, 0, nnz), ix, ip), shape=(self.nQ, self.nQ))
        from oasisx_b200 import fem

        node_of_dof = mg._node_ids(fem.lattice_node_index(msh)[self._dof_nodes], msh._shape)  # also on a deformed box
        n_levels = 0
        for lvl, (cm, P) in enumerate(levels):
            Pl = sp.csr_matrix(P)[node_of_dof, :].tocsr() if lvl == 0 else sp.csr_matrix(P)
            Pl.sort_indices()
            R = sp.csr_matrix(Pl.T)
            R.sort_indices()
            A = sp.csr_matrix(R @ A @ Pl)
            A.sort_indices()
            n = A.shape[0]
            i32 = lambda a: np.ascontiguousarray(a, np.int32)
            f64 = lambda a: np.ascontiguousarray(a, np.float64)
            arrs = [i32(A.indptr), i32(A.indices), f64(A.data), i32(Pl.indptr), i32(Pl.indices), f64(Pl.data),
                    i32(R.indptr), i32(R.indices), f64(R.data)]
            self.L.ipcs_cpu_mg_add_level(self.h, n, _p(arrs[0]), _p(arrs[1]), _p(arrs[2]), Pl.shape[0], _p(arrs[3]), _p(arrs[4]),
                                         _p(arrs[5]), _p(arrs[6]), _p(arrs[7]), _p(arrs[8]))
            n_levels += 1
            if n <= dense_max:
                alpha = A[0, 0] / n
                inv = f64(np.linalg.inv(A.toarray() + alpha))
                self.L.ipcs_cpu_mg_set_dense(self.h, n, _p(inv))
                break
        else:  # no level small enough for the exact coarse solve: keep Jacobi
            self.L.ipcs_cpu_set_pressure_mg(self.h, 0, float(omega))
            return 0
        self.L.ipcs_cpu_set_pressure_mg(self.h, 1, float(omega))
        return n_levels

    def bench_strategies(self, comp: int, dt: float, nu: float, reps: int = 3):
        """demo/assembly_strategies.py:121-142 on the host: (seconds {assembly, matvec, action}, b_matvec, b_action)."""
        out, bm, ba = np.zeros(3), np.empty(self.nV), np.empty(self.nV)
        self.L.ipcs_cpu_bench_strategies(self.h, comp, dt, nu, reps, _p(out), _p(bm), _p(ba))
        return out, bm, ba

    def solve(self, dt, nu):
        self.update_bcs()
        rc = self.L.ipcs_cpu_step(self.h, dt, nu, _p(self.its))
        if rc != 0:
            raise RuntimeError(f"CPU restatement: Krylov solve diverged in stage {rc}")
        return rc
