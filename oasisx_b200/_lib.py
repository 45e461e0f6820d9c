"""ctypes binding of ``libb200ipcs.so`` (``include/b200ipcs.h``).

There is no CPU fallback: if the shared library is missing or no B200 is visible, constructing a
:class:`Context` raises.  The library is built in-tree by ``oasisx_b200/build.py``
(``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libb200ipcs.so")

# ids of include/b200ipcs.h
SPACE_V, SPACE_Q = 0, 1
PAT_VV, PAT_VQ, PAT_QV, PAT_QQ = 0, 1, 2, 3
MAT_M, MAT_K, MAT_A, MAT_AP, MAT_P, MAT_G, MAT_D, MAT_MQ = range(8)
VEC_U, VEC_U1, VEC_U2, VEC_UAB, VEC_RHS1, VEC_BFIRST, VEC_B0, VEC_PSURF, VEC_B3, VEC_WRK = range(10)
VEC_PS, VEC_P, VEC_DP, VEC_B2, VEC_MQ = 16, 17, 18, 19, 20
SOLVER_TENTATIVE, SOLVER_PRESSURE, SOLVER_SCALAR, SOLVER_PROJECTOR = range(4)

# every symbol include/b200ipcs.h declares (tests/test_host.py::test_abi_exports_every_declared_symbol checks the .so exports them all)
SYMBOLS = [
    "b2_abi_version", "b2_device_count", "b2_nccl_unique_id", "b2_create", "b2_destroy", "b2_last_error",
    "b2_host_alloc", "b2_host_free", "b2_set_mesh", "b2_set_space", "b2_set_halo", "b2_set_global_sizes",
    "b2_first_plan_info", "b2_bench_assembly_strategies", "b2_peer_export", "b2_peer_import", "b2_peer_disable", "b2_peer_enabled",
    "b2_build_patterns", "b2_pattern_nnz", "b2_pattern_sell_slots", "b2_set_slice_order", "b2_pressure_mg_add_level", "b2_pressure_mg_configure", "b2_pressure_amg_build",
    "b2_set_pressure_global_ids",
    "b2_pressure_mg_level_info", "b2_pressure_mg_get_level", "b2_get_pattern", "b2_set_velocity_bc_dofs",
    "b2_set_velocity_bc_values", "b2_set_velocity_bc_series", "b2_select_bc_step", "b2_reset_time_history", "b2_profiler_range", "b2_set_pressure_bc_dofs", "b2_declare_pressure_bcs", "b2_preassemble", "b2_set_vector", "b2_get_vector",
    "b2_get_matrix_values", "b2_mat_mult", "b2_set_solver_option", "b2_assemble_first", "b2_tentative_assemble",
    "b2_tentative_solve", "b2_pressure_assemble", "b2_pressure_solve", "b2_velocity_update", "b2_step_begin", "b2_step",
    "b2_assemble_pressure_surface", "b2_project_assemble", "b2_project_get_rhs", "b2_project_set_rhs", "b2_project_set_bcs", "b2_project_solve", "b2_ksp_solve", "b2_l2_diff_sq", "b2_l2_error_quadrature", "b2_l2_error_trig", "b2_get_stats", "b2_bench_kernel", "b2_synchronize",
    "b2_event_record", "b2_event_elapsed_ms", "b2_set_tuning",
]


class Stats(C.Structure):
    _fields_ = [
        ("its_tentative", C.c_int32 * 3),
        ("its_pressure", C.c_int32),
        ("its_update", C.c_int32 * 3),
        ("its_projector", C.c_int32),
        ("kernel_launches", C.c_int64),
        ("ms_assemble_first", C.c_double),
        ("ms_tentative", C.c_double),
        ("ms_pressure", C.c_double),
        ("ms_update", C.c_double),
        ("ms_step", C.c_double),
        ("bytes_h2d", C.c_int64),
        ("bytes_d2h", C.c_int64),
        ("halo_exchanges", C.c_int64),
        ("allreduces", C.c_int64),
        ("res0_tentative", C.c_double),
        ("res0_pressure", C.c_double),
        ("res0_update", C.c_double),
        ("peer_kernels", C.c_int64),
    ]


class B200Error(RuntimeError):
    pass


_lib = None


def load_library() -> C.CDLL:
    """dlopen the in-tree library; raise loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200Error(
            f"{LIB_PATH} not found: build it with `python -m oasisx_b200.build` "
            "(oasisx_b200 has no CPU fallback)"
        )
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, dbl = C.c_void_p, C.c_int, C.c_int64, C.c_double
    sig = {
        "b2_abi_version": (i32, []),
        "b2_device_count": (i32, []),
        "b2_nccl_unique_id": (i32, [vp]),
        "b2_create": (i32, [C.POINTER(vp), i32, i32, i32, vp]),
        "b2_destroy": (None, [vp]),
        "b2_last_error": (C.c_char_p, [vp]),
        "b2_host_alloc": (vp, [i64]),
        "b2_host_free": (None, [vp]),
        "b2_set_mesh": (i32, [vp, i32, i64, vp, i64, vp]),
        "b2_set_space": (i32, [vp, i32, i32, i64, i64, vp]),
        "b2_set_halo": (i32, [vp, i32, i32, vp, vp, vp, vp]),
        "b2_first_plan_info": (i32, [vp, vp]),
        "b2_bench_assembly_strategies": (i32, [vp, C.c_double, C.c_double, i32, vp]),
        "b2_peer_export": (i32, [vp, i32, vp]),
        "b2_peer_import": (i32, [vp, i32, vp]),
        "b2_peer_disable": (i32, [vp]),
        "b2_peer_enabled": (i32, [vp]),
        "b2_set_global_sizes": (i32, [vp, i64, i64]),
        "b2_build_patterns": (i32, [vp]),
        "b2_pattern_nnz": (i64, [vp, i32]),
        "b2_pattern_sell_slots": (i64, [vp, i32]),
        "b2_set_slice_order": (i32, [vp, i32, i64, vp]),
        "b2_pressure_mg_add_level": (i32, [vp, i64, vp, i64, vp, i64, vp, vp, vp, vp, vp, vp]),
        "b2_pressure_mg_configure": (i32, [vp, i32, i32, i32, dbl]),
        "b2_pressure_amg_build": (i32, [vp]),
        "b2_set_pressure_global_ids": (i32, [vp, i64, vp]),
        "b2_pressure_mg_level_info": (i32, [vp, i32, vp]),
        "b2_pressure_mg_get_level": (i32, [vp, i32, i32, vp, vp, vp]),
        "b2_get_pattern": (i32, [vp, i32, vp, vp]),
        "b2_set_velocity_bc_dofs": (i32, [vp, i32, i64, vp]),
        "b2_set_velocity_bc_values": (i32, [vp, i32, i64, vp]),
        "b2_set_velocity_bc_series": (i32, [vp, i32, i32, i64, vp]),
        "b2_select_bc_step": (i32, [vp, i32]),
        "b2_reset_time_history": (i32, [vp]),
        "b2_declare_pressure_bcs": (i32, [vp, i32]),
        "b2_profiler_range": (i32, [vp, i32]),
        "b2_set_pressure_bc_dofs": (i32, [vp, i64, vp]),
        "b2_preassemble": (i32, [vp, vp, i32, i32]),
        "b2_set_vector": (i32, [vp, i32, i32, vp, i64]),
        "b2_get_vector": (i32, [vp, i32, i32, vp, i64]),
        "b2_get_matrix_values": (i32, [vp, i32, i32, vp]),
        "b2_mat_mult": (i32, [vp, i32, i32, vp, vp]),
        "b2_set_solver_option": (i32, [vp, i32, C.c_char_p, C.c_char_p]),
        "b2_assemble_first": (i32, [vp, dbl, dbl]),
        "b2_tentative_assemble": (i32, [vp]),
        "b2_tentative_solve": (i32, [vp, vp, vp]),
        "b2_pressure_assemble": (i32, [vp, dbl]),
        "b2_pressure_solve": (i32, [vp, dbl, vp]),
        "b2_velocity_update": (i32, [vp, dbl, vp]),
        "b2_step_begin": (i32, [vp, dbl, dbl]),
        "b2_step": (i32, [vp, dbl, dbl, dbl, i32, vp]),
        "b2_assemble_pressure_surface": (i32, [vp, i64, vp, vp, vp, i32]),
        "b2_project_assemble": (i32, [vp, i32, i32, i32, vp, i32, i32, i32, vp, vp, vp]),
        "b2_project_get_rhs": (i32, [vp, vp]),
        "b2_project_set_rhs": (i32, [vp, i32, i32, vp]),
        "b2_project_set_bcs": (i32, [vp, i32, i32, i64, vp, vp]),
        "b2_project_solve": (i32, [vp, vp, vp]),
        "b2_ksp_solve": (i32, [vp, i32, i32, vp, vp, vp]),
        "b2_l2_diff_sq": (i32, [vp, i32, vp, i64, vp]),
        "b2_l2_error_quadrature": (i32, [vp, i32, i64, i32, vp, vp, vp, vp]),
        "b2_l2_error_trig": (i32, [vp, i32, i64, i32, vp, vp, i32, vp, vp]),
        "b2_get_stats": (i32, [vp, vp]),
        "b2_bench_kernel": (i32, [vp, i32, i32, vp, vp]),
        "b2_synchronize": (i32, [vp]),
        "b2_set_tuning": (i32, [vp, C.c_char_p, i32]),
        "b2_event_record": (i32, [vp, i32]),
        "b2_event_elapsed_ms": (i32, [vp, i32, i32, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _f64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float64)


def _i32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.int32)


def nccl_unique_id() -> bytes:
    lib = load_library()
    buf = C.create_string_buffer(128)
    rc = lib.b2_nccl_unique_id(buf)
    if rc != 0:
        raise B200Error(f"b2_nccl_unique_id failed ({rc}): {lib.b2_last_error(None).decode()}")
    return buf.raw


class Context:
    """One ``b2_ctx`` (one rank / one GPU)."""

    def __init__(self, device: int = 0, nranks: int = 1, rank: int = 0, nccl_uid: bytes | None = None):
        self.lib = load_library()
        self._h = C.c_void_p()
        uid = C.create_string_buffer(nccl_uid, 128) if nccl_uid is not None else None
        rc = self.lib.b2_create(C.byref(self._h), device, nranks, rank, uid)
        if rc != 0:
            msg = self.lib.b2_last_error(None).decode()
            raise B200Error(f"b2_create failed ({rc}): {msg}")
        self.gdim = 0
        self.n = {SPACE_V: 0, SPACE_Q: 0}

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.b2_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int, what: str):
        if rc != 0:
            raise B200Error(f"{what} failed ({rc}): {self.lib.b2_last_error(self._h).decode()}")

    # ---- setup ---------------------------------------------------------------------------
    def set_mesh(self, gdim: int, x: np.ndarray, cell_nodes: np.ndarray):
        x, cn = _f64(x), _i32(cell_nodes)
        assert x.shape[1] == 3 and cn.shape[1] == gdim + 1
        self.gdim = gdim
        self._check(self.lib.b2_set_mesh(self._h, gdim, x.shape[0], _ptr(x), cn.shape[0], _ptr(cn)), "b2_set_mesh")

    def set_space(self, space: int, degree: int, n_owned: int, n_ghost: int, cell_dofs: np.ndarray):
        cd = _i32(cell_dofs)
        self.n[space] = n_owned + n_ghost
        if not hasattr(self, "_space_info"):
            self._space_info = {}
        self._space_info[space] = (n_owned + n_ghost, int(degree))
        self._check(self.lib.b2_set_space(self._h, space, degree, n_owned, n_ghost, _ptr(cd)), "b2_set_space")

    def set_halo(self, space: int, plan):
        nb = _i32(plan.neighbors)
        so = np.ascontiguousarray(plan.send_off, dtype=np.int64)
        si = _i32(plan.send_idx)
        ro = np.ascontiguousarray(plan.recv_off, dtype=np.int64)
        self._check(self.lib.b2_set_halo(self._h, space, len(nb), _ptr(nb), _ptr(so), _ptr(si), _ptr(ro)), "b2_set_halo")

    def set_global_sizes(self, nv: int, nq: int):
        self._check(self.lib.b2_set_global_sizes(self._h, nv, nq), "b2_set_global_sizes")

    def build_patterns(self):
        self._check(self.lib.b2_build_patterns(self._h), "b2_build_patterns")

    def set_slice_order(self, which: int, order):
        o = _i32(order)
        self._check(self.lib.b2_set_slice_order(self._h, which, o.size, _ptr(o)), "b2_set_slice_order")

    def pressure_mg_add_level(self, x, cell_nodes, P, R):
        """P, R: scipy CSR (fine-owned x coarse, coarse x fine-local)."""
        x, cn = _f64(x), _i32(cell_nodes)
        Pi, Px, Pv = _i32(P.indptr), _i32(P.indices), _f64(P.data)
        Ri, Rx, Rv = _i32(R.indptr), _i32(R.indices), _f64(R.data)
        self._check(self.lib.b2_pressure_mg_add_level(self._h, x.shape[0], _ptr(x), cn.shape[0], _ptr(cn), P.shape[0],
                                                      _ptr(Pi), _ptr(Px), _ptr(Pv), _ptr(Ri), _ptr(Rx), _ptr(Rv)),
                    "b2_pressure_mg_add_level")

    def pressure_mg_configure(self, nu_pre=1, nu_post=1, coarse_sweeps=16, omega=0.85):
        self._check(self.lib.b2_pressure_mg_configure(self._h, nu_pre, nu_post, coarse_sweeps, omega), "b2_pressure_mg_configure")

    def pressure_amg_build(self):
        """Smoothed-aggregation hierarchy from the assembled pressure matrix (after preassemble; on several ranks
        after :meth:`set_pressure_global_ids`, collectively)."""
        self._check(self.lib.b2_pressure_amg_build(self._h), "b2_pressure_amg_build")

    def set_pressure_global_ids(self, l2g):
        """Global index of every local pressure dof, owned then ghost (``LocalSpace.l2g``); collective on several
        ranks.  Raises B200Error on every rank unless the owned indices of all ranks cover 0 .. n_global-1 once."""
        g = np.ascontiguousarray(l2g, dtype=np.int64)
        self._check(self.lib.b2_set_pressure_global_ids(self._h, g.size, _ptr(g)), "b2_set_pressure_global_ids")

    MG_LEVEL_INFO = ("n", "nnz_A", "nnz_P", "algebraic", "dense", "omega", "rho_hat")

    def pressure_mg_level_info(self, level: int) -> dict:
        out = np.zeros(7, dtype=np.float64)
        self._check(self.lib.b2_pressure_mg_level_info(self._h, level, _ptr(out)), "b2_pressure_mg_level_info")
        d = dict(zip(self.MG_LEVEL_INFO, out.tolist()))
        for k in ("n", "nnz_A", "nnz_P", "algebraic", "dense"):
            d[k] = int(d[k])
        return d

    def pressure_mg_get_level(self, level: int, what: int):
        """what = 0: A_l, 1: P_l, 2: R_l as scipy CSR; 3: the aggregate of every dof of level - 1 (int32 array)."""
        import scipy.sparse as sp

        info = self.pressure_mg_level_info(level)
        n, nf = info["n"], self.pressure_mg_level_info(level - 1)["n"]
        if what == 3:
            agg = np.empty(nf, dtype=np.int32)
            self._check(self.lib.b2_pressure_mg_get_level(self._h, level, 3, None, _ptr(agg), None), "b2_pressure_mg_get_level")
            return agg
        shape = {0: (n, n), 1: (nf, n), 2: (n, nf)}[what]
        nnz = info["nnz_A"] if what == 0 else info["nnz_P"]
        indptr = np.empty(shape[0] + 1, dtype=np.int32)
        indices = np.empty(nnz, dtype=np.int32)
        vals = np.empty(nnz, dtype=np.float64)
        self._check(self.lib.b2_pressure_mg_get_level(self._h, level, what, _ptr(indptr), _ptr(indices), _ptr(vals)),
                    "b2_pressure_mg_get_level")
        return sp.csr_matrix((vals, indices, indptr), shape=shape)

    def pattern(self, which: int, n_rows: int):
        nnz = self.lib.b2_pattern_nnz(self._h, which)
        if nnz < 0:
            raise B200Error("pattern not built")
        indptr = np.empty(n_rows + 1, dtype=np.int32)
        indices = np.empty(nnz, dtype=np.int32)
        self._check(self.lib.b2_get_pattern(self._h, which, _ptr(indptr), _ptr(indices)), "b2_get_pattern")
        return indptr, indices

    PEER_BLOB_BYTES = 256

    def peer_setup(self, comm, segment: int) -> bool:
        """Export this rank's arena, all-gather the blobs over `comm`, import the peers' arenas.  Every rank must
        call it; if ANY rank fails to map a peer, all ranks fall back to the NCCL path.  Returns the agreed state."""
        blob = C.create_string_buffer(self.PEER_BLOB_BYTES)
        ok = self.lib.b2_peer_export(self._h, segment, blob) == 0
        blobs = comm.allgather(bytes(blob.raw) if ok else b"")
        ok = ok and all(len(b) == self.PEER_BLOB_BYTES for b in blobs)
        if ok:
            ok = self.lib.b2_peer_import(self._h, segment, C.create_string_buffer(b"".join(blobs), len(blobs) * self.PEER_BLOB_BYTES)) == 0
        agreed = bool(comm.allreduce(int(ok), "min"))
        if not agreed:
            self.lib.b2_peer_disable(self._h)
        comm.Barrier()
        return agreed

    def bench_assembly_strategies(self, dt: float, nu: float, reps: int = 10) -> dict:
        out = np.zeros(6, dtype=np.float64)
        self._check(self.lib.b2_bench_assembly_strategies(self._h, float(dt), float(nu), int(reps), _ptr(out)), "b2_bench_assembly_strategies")
        return {"ms_convection_assembly": out[0], "ms_matvec": out[1], "ms_action": out[2],
                "bytes_convection_assembly": out[3], "bytes_matvec": out[4], "bytes_action": out[5]}

    def first_plan_info(self) -> dict:
        out = np.zeros(4, dtype=np.int64)
        self._check(self.lib.b2_first_plan_info(self._h, _ptr(out)), "b2_first_plan_info")
        return dict(zip(("cell_schedule", "congruence_classes", "slab", "cells"), (int(v) for v in out)))

    def peer_enabled(self) -> bool:
        return bool(self.lib.b2_peer_enabled(self._h))

    def pattern_nnz(self, which: int) -> int:
        return int(self.lib.b2_pattern_nnz(self._h, which))

    def pattern_sell(self, which: int) -> int:
        """(slots, run slice columns) of the sliced-ELL form of a square pattern."""
        return int(self.lib.b2_pattern_sell_slots(self._h, which))

    def set_velocity_bc_dofs(self, comp: int, dofs):
        d = _i32(dofs)
        self._check(self.lib.b2_set_velocity_bc_dofs(self._h, comp, d.size, _ptr(d)), "b2_set_velocity_bc_dofs")

    def set_velocity_bc_values(self, comp: int, values):
        v = _f64(values)
        self._check(self.lib.b2_set_velocity_bc_values(self._h, comp, v.size, _ptr(v)), "b2_set_velocity_bc_values")

    def set_velocity_bc_series(self, comp: int, values: np.ndarray):
        v = _f64(values)
        assert v.ndim == 2
        self._check(self.lib.b2_set_velocity_bc_series(self._h, comp, v.shape[0], v.shape[1], _ptr(v)),
                    "b2_set_velocity_bc_series")

    def select_bc_step(self, step: int):
        self._check(self.lib.b2_select_bc_step(self._h, step), "b2_select_bc_step")

    def profiler_range(self, on: bool):
        self._check(self.lib.b2_profiler_range(self._h, int(bool(on))), "b2_profiler_range")

    def reset_time_history(self):
        self._check(self.lib.b2_reset_time_history(self._h), "b2_reset_time_history")

    def declare_pressure_bcs(self, any_bc: bool):
        self._check(self.lib.b2_declare_pressure_bcs(self._h, int(bool(any_bc))), "b2_declare_pressure_bcs")

    def set_pressure_bc_dofs(self, dofs):
        d = _i32(dofs)
        self._check(self.lib.b2_set_pressure_bc_dofs(self._h, d.size, _ptr(d)), "b2_set_pressure_bc_dofs")

    def preassemble(self, body_force, low_memory: bool, rotational: bool):
        f = _f64(list(body_force) + [0.0] * (3 - len(body_force)))
        self._check(self.lib.b2_preassemble(self._h, _ptr(f), int(low_memory), int(rotational)), "b2_preassemble")

    # ---- state ---------------------------------------------------------------------------
    def set_vector(self, vec: int, comp: int, host: np.ndarray):
        h = _f64(host)
        self._check(self.lib.b2_set_vector(self._h, vec, comp, _ptr(h), h.size), "b2_set_vector")

    def get_vector(self, vec: int, comp: int, out: np.ndarray) -> np.ndarray:
        assert out.dtype == np.float64 and out.flags.c_contiguous
        self._check(self.lib.b2_get_vector(self._h, vec, comp, _ptr(out), out.size), "b2_get_vector")
        return out

    def matrix_values(self, mat: int, comp: int, nnz: int) -> np.ndarray:
        out = np.empty(nnz, dtype=np.float64)
        self._check(self.lib.b2_get_matrix_values(self._h, mat, comp, _ptr(out)), "b2_get_matrix_values")
        return out

    def mat_mult(self, mat: int, comp: int, x: np.ndarray, n_rows: int) -> np.ndarray:
        x = _f64(x)
        y = np.empty(n_rows, dtype=np.float64)
        self._check(self.lib.b2_mat_mult(self._h, mat, comp, _ptr(x), _ptr(y)), "b2_mat_mult")
        return y

    def set_solver_option(self, solver: int, key: str, value):
        self._check(
            self.lib.b2_set_solver_option(self._h, solver, str(key).encode(), str(value).encode()),
            "b2_set_solver_option",
        )

    # ---- stages --------------------------------------------------------------------------
    def assemble_first(self, dt: float, nu: float):
        self._check(self.lib.b2_assemble_first(self._h, dt, nu), "b2_assemble_first")

    def tentative_assemble(self):
        self._check(self.lib.b2_tentative_assemble(self._h), "b2_tentative_assemble")

    def tentative_solve(self):
        diff = C.c_double(0.0)
        reasons = np.zeros(3, dtype=np.int32)
        self._check(self.lib.b2_tentative_solve(self._h, C.byref(diff), _ptr(reasons)), "b2_tentative_solve")
        return diff.value, reasons[: self.gdim].copy()

    def pressure_assemble(self, dt: float):
        self._check(self.lib.b2_pressure_assemble(self._h, dt), "b2_pressure_assemble")

    def pressure_solve(self, nu: float) -> int:
        reason = C.c_int32(0)
        self._check(self.lib.b2_pressure_solve(self._h, float(nu), C.byref(reason)), "b2_pressure_solve")
        return reason.value

    def velocity_update(self, dt: float):
        reasons = np.zeros(3, dtype=np.int32)
        self._check(self.lib.b2_velocity_update(self._h, dt, _ptr(reasons)), "b2_velocity_update")
        return reasons[: self.gdim].copy()

    def step_begin(self, dt: float, nu: float):
        self._check(self.lib.b2_step_begin(self._h, dt, nu), "b2_step_begin")

    def step(self, dt: float, nu: float, max_error: float, max_iter: int) -> float:
        diff = C.c_double(0.0)
        self._check(self.lib.b2_step(self._h, dt, nu, max_error, max_iter, C.byref(diff)), "b2_step")
        return diff.value

    def assemble_pressure_surface(self, facet_cells, facet_local, h_nodal, accumulate: bool):
        fc, fl, h = _i32(facet_cells), _i32(facet_local), _f64(h_nodal)
        self._check(self.lib.b2_assemble_pressure_surface(self._h, fc.size, _ptr(fc), _ptr(fl), _ptr(h), int(accumulate)),
                    "b2_assemble_pressure_surface")

    def l2_error_trig(self, vec: int, n_cells: int, pts, w, terms) -> float:
        pts, w = _f64(pts), _f64(w)
        terms = _f64(np.asarray(terms, dtype=np.float64).reshape(-1, 12))
        out = C.c_double(0.0)
        self._check(self.lib.b2_l2_error_trig(self._h, vec, n_cells, len(w), _ptr(pts), _ptr(w), terms.shape[0], _ptr(terms), C.byref(out)),
                    "b2_l2_error_trig")
        return out.value

    def project_assemble(self, target_space: int, n_comp: int, pts, w, src_space: int = 0, src_nodal=None, deriv: int = -1,
                         grad: bool = False, f_quad=None):
        pts, w = _f64(pts), _f64(w)
        sn = _f64(src_nodal) if src_nodal is not None else None
        fq = _f64(f_quad) if f_quad is not None else None
        self._check(self.lib.b2_project_assemble(self._h, target_space, n_comp, src_space, _ptr(sn) if sn is not None else None,
                                                 deriv, int(grad), len(w), _ptr(pts), _ptr(w), _ptr(fq) if fq is not None else None),
                    "b2_project_assemble")

    def project_rhs(self, n: int) -> np.ndarray:
        out = np.empty(n, dtype=np.float64)
        self._check(self.lib.b2_project_get_rhs(self._h, _ptr(out)), "b2_project_get_rhs")
        return out

    def project_set_bcs(self, target_space: int, dofs, values):
        d = _i32(dofs)
        v = _f64(np.atleast_2d(values))
        assert v.shape[1] == d.size
        self._check(self.lib.b2_project_set_bcs(self._h, target_space, v.shape[0], d.size, _ptr(d), _ptr(v)), "b2_project_set_bcs")

    def project_load_rhs(self, target_space: int, rhs: np.ndarray):
        rhs = _f64(np.atleast_2d(rhs))
        self._check(self.lib.b2_project_set_rhs(self._h, target_space, rhs.shape[0], _ptr(rhs)), "b2_project_set_rhs")

    def space_size(self, space: int) -> int:
        return self._space_info[space][0]

    def space_degree(self, space: int) -> int:
        return self._space_info[space][1]

    def project_solve(self, n_local: int, n_comp: int):
        x = np.empty(n_local * n_comp, dtype=np.float64)
        reasons = np.zeros(3, dtype=np.int32)
        self._check(self.lib.b2_project_solve(self._h, _ptr(x), _ptr(reasons)), "b2_project_solve")
        return x.reshape(n_comp, n_local), reasons[:n_comp]

    def ksp_solve(self, solver: int, mat: int, b: np.ndarray, x: np.ndarray) -> int:
        b = _f64(b)
        assert x.dtype == np.float64 and x.flags.c_contiguous and x.shape == b.shape
        reason = C.c_int32(0)
        self._check(self.lib.b2_ksp_solve(self._h, solver, mat, _ptr(b), _ptr(x), C.byref(reason)), "b2_ksp_solve")
        return int(reason.value)

    def l2_diff_sq(self, vec: int, exact: np.ndarray) -> float:
        e = _f64(exact)
        out = C.c_double(0.0)
        self._check(self.lib.b2_l2_diff_sq(self._h, vec, _ptr(e), e.size, C.byref(out)), "b2_l2_diff_sq")
        return out.value

    def l2_error_quadrature(self, vec: int, n_cells: int, ref_points, weights, exact) -> float:
        p, w, e = _f64(ref_points), _f64(weights), _f64(exact)
        out = C.c_double(0.0)
        self._check(self.lib.b2_l2_error_quadrature(self._h, vec, n_cells, len(w), _ptr(p), _ptr(w), _ptr(e), C.byref(out)),
                    "b2_l2_error_quadrature")
        return out.value

    def stats(self) -> Stats:
        s = Stats()
        self._check(self.lib.b2_get_stats(self._h, C.byref(s)), "b2_get_stats")
        return s

    def bench_kernel(self, kernel: int, reps: int):
        ms, nbytes = C.c_double(0.0), C.c_double(0.0)
        self._check(self.lib.b2_bench_kernel(self._h, kernel, reps, C.byref(ms), C.byref(nbytes)), "b2_bench_kernel")
        return ms.value, nbytes.value

    def set_tuning(self, key: str, value: int):
        self._check(self.lib.b2_set_tuning(self._h, key.encode(), int(value)), "b2_set_tuning")

    def event_record(self, slot: int):
        self._check(self.lib.b2_event_record(self._h, slot), "b2_event_record")

    def event_elapsed_ms(self, a: int, b: int) -> float:
        ms = C.c_double(0.0)
        self._check(self.lib.b2_event_elapsed_ms(self._h, a, b, C.byref(ms)), "b2_event_elapsed_ms")
        return ms.value

    def synchronize(self):
        self._check(self.lib.b2_synchronize(self._h), "b2_synchronize")
