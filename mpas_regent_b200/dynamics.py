"""Host-side mirror of the reference's task interface for the RK3 dynamics hot path.

``Dynamics`` owns one ``mpasb200_t`` handle of libmpas_b200.so and exposes the hot-path
leaf tasks under the reference's own names and argument meaning (reference:
dynamics/dynamics_tasks.rg signatures at :328-337, 460-466, 513-520, 747-752, 1484-1496,
1530-1535, 1707-1715, 1726-1732, 1875-1883, 1951-1959), and the driver ``atm_srk3`` /
``atm_timestep`` (dynamics/rk_timestep.rg:361-519).  Regions are replaced by the device-
resident mirror behind the handle; ``upload_field`` / ``download_field`` are the only
calls that touch host memory.

There is no CPU fallback: if libmpas_b200.so is missing, or no CUDA device is usable,
construction raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Iterable, Optional, Sequence

import numpy as np

from . import _abi
from ._abi import (CELL, EDGE, FIELD_ENTITY, FIELD_ID, FIELD_SLOTS, FIELDS, VERTEX, VERTICAL, MpasConfig, MpasDims,
                   MpasMeshPtrs)

_LIB_PATH = os.environ.get("MPAS_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "libmpas_b200.so")   # the override selects a laboratory build (profiles/ scripts only)
_lib = None


class MpasB200Error(RuntimeError):
    pass


def load_library(path: Optional[str] = None):
    """dlopen libmpas_b200.so (built in-tree by __graft_entry__.build / csrc/Makefile)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or _LIB_PATH
    if not os.path.exists(p):
        raise MpasB200Error(f"{p} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                            f"(there is no CPU fallback)")
    lib = C.CDLL(p, mode=C.RTLD_GLOBAL)
    _declare(lib, "mpasb200_")
    if path is None:
        _lib = lib
    return lib


def _declare(lib, prefix: str, handle_t=C.c_void_p):
    H, I, D = handle_t, C.c_int, C.c_double
    sig = {
        "create": ([C.POINTER(MpasDims), C.POINTER(MpasConfig), C.POINTER(H)], I),
        "destroy": ([H], I),
        "upload_mesh": ([H, C.POINTER(MpasMeshPtrs)], I),
        "rk_integration_setup": ([H], I),
        "compute_moist_coefficients": ([H], I),
        "compute_vert_imp_coefs": ([H, D], I),
        "compute_dyn_tend": ([H, I, D, I, D, I, I], I),
        "set_smlstep_pert_variables": ([H], I),
        "advance_acoustic_step": ([H, D, I], I),
        "divergence_damping_3d": ([H, D], I),
        "recover_large_step_variables": ([H, I, I, D], I),
        "compute_solve_diagnostics": ([H, I, I], I),
        "rk_dynamics_substep_finish": ([H, I, I], I),
        "advance_scalars": ([H, D, I], I),
        "init_coupled_diagnostics": ([H], I),
        "reconstruct_2d": ([H, I, I], I),
        "srk3": ([H, D], I),
        "timestep": ([H, D], I),
        "compute_signs": ([H, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p], I),
        "compute_zb_cell": ([H], I),
        "adv_coef_compression": ([H, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p], I),
        "couple_coef_3rd_order": ([H, D, C.c_void_p], I),
        "compute_mesh_scaling": ([H, C.c_void_p, C.c_void_p, I, C.c_void_p, C.c_void_p], I),
        "compute_damping_coefs": ([H, C.c_void_p, D, D], I),
    }
    if prefix == "mpasb200_":
        sig["init_atm_case_jw"] = ([H, C.c_void_p], I)
    for name, (args, res) in sig.items():
        fn = getattr(lib, prefix + name)
        fn.argtypes, fn.restype = args, res
    if prefix == "mpasb200_":
        lib.mpasb200_default_config.argtypes, lib.mpasb200_default_config.restype = [C.POINTER(MpasConfig)], None
        lib.mpasb200_last_error.argtypes, lib.mpasb200_last_error.restype = [H], C.c_char_p
        lib.mpasb200_mesh_member.argtypes, lib.mpasb200_mesh_member.restype = [H, C.c_char_p, C.c_void_p, C.c_int64], I
        lib.mpasb200_upload_mesh_staged.argtypes, lib.mpasb200_upload_mesh_staged.restype = [H], I
        lib.mpasb200_upload_field.argtypes = [H, I, C.c_void_p, C.c_int64, C.c_int64]
        lib.mpasb200_download_field.argtypes = [H, I, C.c_void_p, C.c_int64, C.c_int64]
        lib.mpasb200_zero_field.argtypes = [H, I]
        lib.mpasb200_upload_field_async.argtypes = [H, I, C.c_void_p]
        lib.mpasb200_download_field_async.argtypes = [H, I, C.c_void_p]
        lib.mpasb200_transfer_wait.argtypes = [H]
        lib.mpasb200_sync.argtypes = [H]
        lib.mpasb200_register_list.argtypes = [H, I, C.c_void_p, C.c_int32, C.POINTER(C.c_int32)]
        lib.mpasb200_pack.argtypes = [H, I, C.c_void_p, C.c_int32, C.c_void_p]
        lib.mpasb200_unpack.argtypes = [H, I, C.c_void_p, C.c_int32, C.c_void_p]
        lib.mpasb200_set_stream.argtypes = [H, C.c_void_p]
        lib.mpasb200_set_use_graph.argtypes, lib.mpasb200_set_use_graph.restype = [H, I], I
        lib.mpasb200_class_range.argtypes = [H, I, I, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        lib.mpasb200_set_range.argtypes = [H, I, C.c_int32, C.c_int32]
        lib.mpasb200_class_range.restype = lib.mpasb200_set_range.restype = I
        lib.mpasb200_set_global_ids.argtypes, lib.mpasb200_set_global_ids.restype = [H, I, C.c_void_p, C.c_int32], I
        lib.mpasb200_summarize_field.argtypes = [H, I, C.c_int32, C.c_int32, C.POINTER(_abi.MpasFieldSummary)]
        lib.mpasb200_summarize_field.restype = I
        lib.mpasb200_register_weights.argtypes = [H, I, C.c_void_p, C.c_int32, C.POINTER(C.c_int32)]
        lib.mpasb200_integrate.argtypes = [H, I, I, I, I, I, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(_abi.MpasIntegral)]
        lib.mpasb200_integral_merge.argtypes = [C.POINTER(_abi.MpasIntegral), C.POINTER(_abi.MpasIntegral)]
        lib.mpasb200_integral_value.argtypes, lib.mpasb200_integral_value.restype = [C.POINTER(_abi.MpasIntegral)], D
        lib.mpasb200_register_weights.restype = lib.mpasb200_integrate.restype = lib.mpasb200_integral_merge.restype = I
        lib.mpasb200_dist_unique_id.argtypes, lib.mpasb200_dist_unique_id.restype = [C.c_void_p], I
        lib.mpasb200_dist_init.argtypes, lib.mpasb200_dist_init.restype = [H, I, I, C.c_void_p], I
        lib.mpasb200_dist_set_halo.argtypes = [H, I, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.mpasb200_dist_set_halo.restype = I
        lib.mpasb200_dist_exchange.argtypes, lib.mpasb200_dist_exchange.restype = [H, I], I
        lib.mpasb200_dist_flush.argtypes, lib.mpasb200_dist_flush.restype = [H], I
        lib.mpasb200_srk3_dist.argtypes, lib.mpasb200_srk3_dist.restype = [H, D], I
        lib.mpasb200_launch_count.argtypes, lib.mpasb200_launch_count.restype = [H], C.c_int64
        lib.mpasb200_device_bytes.argtypes, lib.mpasb200_device_bytes.restype = [H], C.c_int64
        lib.mpasb200_field_info.argtypes = [I, C.POINTER(I), C.POINTER(I), C.POINTER(C.c_char_p)]
        lib.mpasb200_field_by_name.argtypes, lib.mpasb200_field_by_name.restype = [C.c_char_p], I
        lib.mpasb200_enable_timing.argtypes = [H, I]
        lib.mpasb200_task_time.argtypes = [H, I, C.POINTER(D), C.POINTER(C.c_int64), C.POINTER(C.c_char_p)]
        lib.mpasb200_reset_timing.argtypes = [H]
        lib.mpasb200_enable_kernel_timing.argtypes = [H, I]
        lib.mpasb200_reset_kernel_timing.argtypes = [H]
        lib.mpasb200_kernel_time.argtypes = [H, I, C.POINTER(C.c_char_p), C.POINTER(D), C.POINTER(C.c_int64)]
        lib.mpasb200_timeline_entry.argtypes = [H, I, C.POINTER(C.c_char_p), C.POINTER(D), C.POINTER(D), C.POINTER(I)]
        lib.mpasb200_timeline_entry.restype = I
        for n in ("enable_kernel_timing", "reset_kernel_timing", "kernel_time"):
            getattr(lib, "mpasb200_" + n).restype = I
        for n in ("upload_field_async", "download_field_async", "transfer_wait"):
            getattr(lib, "mpasb200_" + n).restype = I
        for n in ("upload_field", "download_field", "zero_field", "sync", "register_list", "pack", "unpack", "set_stream",
                  "field_info", "enable_timing", "task_time", "reset_timing"):
            getattr(lib, "mpasb200_" + n).restype = I


class TaskAPI:
    """The task-level interface shared by the CUDA library wrapper and the CPU oracle wrapper
    (so parity tests drive both with the same code).  Subclasses provide _call and the field I/O."""

    dims: MpasDims
    cfg: MpasConfig

    # ---- shape helpers -----------------------------------------------------------------------
    def entity_count(self, ent: int) -> int:
        return {CELL: self.dims.nCells, EDGE: self.dims.nEdges, VERTEX: self.dims.nVertices, VERTICAL: 1}[ent]

    def field_shape(self, name: str):
        ent, s, L1 = FIELD_ENTITY[name], FIELD_SLOTS[name], self.dims.nVertLevels + 1
        if ent == VERTICAL:
            return (L1,)
        n = self.entity_count(ent)
        return (n, L1) if s == 1 else (n, L1, s)

    # ---- bulk helpers ------------------------------------------------------------------------
    def upload_state(self, fields: Dict[str, np.ndarray], vert: Optional[Dict[str, np.ndarray]] = None):
        for k, a in fields.items():
            if k in FIELD_ID:
                self.upload_field(k, a)
        for k, a in (vert or {}).items():
            if k in FIELD_ID:
                self.upload_field(k, a)

    def download_all(self, names: Optional[Iterable[str]] = None) -> Dict[str, np.ndarray]:
        names = list(names) if names is not None else [n for (n, _, _) in FIELDS]
        return {n: self.download_field(n) for n in names}

    # ---- the reference's task names -----------------------------------------------------------
    def atm_rk_integration_setup(self):
        self._call("rk_integration_setup")

    def atm_compute_moist_coefficients(self):
        self._call("compute_moist_coefficients")

    def atm_compute_vert_imp_coefs(self, dts: float):
        self._call("compute_vert_imp_coefs", float(dts))

    def atm_compute_dyn_tend(self, rk_step: int, dt: float, config_horiz_mixing: Optional[int] = None,
                             config_mpas_cam_coef: Optional[float] = None, config_mix_full: Optional[bool] = None,
                             config_rayleigh_damp_u: Optional[bool] = None):
        c = self.cfg
        self._call("compute_dyn_tend", int(rk_step), float(dt),
                   int(c.config_horiz_mixing if config_horiz_mixing is None else config_horiz_mixing),
                   float(c.config_mpas_cam_coef if config_mpas_cam_coef is None else config_mpas_cam_coef),
                   int(c.config_mix_full if config_mix_full is None else config_mix_full),
                   int(c.config_rayleigh_damp_u if config_rayleigh_damp_u is None else config_rayleigh_damp_u))

    def atm_set_smlstep_pert_variables(self):
        self._call("set_smlstep_pert_variables")

    def atm_advance_acoustic_step(self, dts: float, small_step: int):
        self._call("advance_acoustic_step", float(dts), int(small_step))

    def atm_divergence_damping_3d(self, dts: float):
        self._call("divergence_damping_3d", float(dts))

    def atm_recover_large_step_variables(self, ns: int, rk_step: int, dt: float):
        self._call("recover_large_step_variables", int(ns), int(rk_step), float(dt))

    def atm_compute_solve_diagnostics(self, hollingsworth: bool, rk_step: int):
        self._call("compute_solve_diagnostics", int(bool(hollingsworth)), int(rk_step))

    def atm_advance_scalars(self, dt: float, rk_step: int):
        """not in the reference (rk_timestep.rg:465 skips it): atm_advance_scalars_work of MPAS-A v7 (mpas_b200.h)"""
        self._call("advance_scalars", float(dt), int(rk_step))

    def atm_init_coupled_diagnostics(self):
        """dynamics_tasks.rg:651-725 (one-time task of atm_core_init) on the device"""
        self._call("init_coupled_diagnostics")

    def mpas_reconstruct_2d(self, includeHalos: bool = False, on_a_sphere: bool = True):
        """dynamics_tasks.rg:1894-1948"""
        self._call("reconstruct_2d", int(bool(includeHalos)), int(bool(on_a_sphere)))

    # ---- the mesh-only producers of atm_core_init (SURVEY.md 8f rank 3); `mesh` holds RAW ids in the caller's numbering ----
    def atm_compute_signs(self, mesh: Dict[str, np.ndarray]) -> Dict[str, np.ndarray]:
        """dynamics_tasks.rg:60-86, 113-129: edgesOnVertexSign, edgesOnCellSign, kiteForCell (the 3-D part is atm_compute_zb_cell)"""
        d = self.dims
        m, keep = _abi.init_mesh_ptrs(mesh, d)
        out = dict(edgesOnVertexSign=np.zeros((d.nVertices, d.vertexDegree)), edgesOnCellSign=np.zeros((d.nCells, d.maxEdges)),
                   kiteForCell=np.zeros((d.nCells, d.maxEdges), dtype=np.int32))
        self._call("compute_signs", C.addressof(m), out["edgesOnVertexSign"].ctypes.data, out["edgesOnCellSign"].ctypes.data,
                   out["kiteForCell"].ctypes.data)
        del keep
        return out

    def atm_compute_zb_cell(self):
        """dynamics_tasks.rg:88-110: fields zb, zb3 -> zb_cell, zb3_cell (after upload_mesh)"""
        self._call("compute_zb_cell")

    def atm_adv_coef_compression(self, mesh: Dict[str, np.ndarray]) -> Dict[str, np.ndarray]:
        """dynamics_tasks.rg:133-269"""
        d = self.dims
        m, keep = _abi.init_mesh_ptrs(mesh, d)
        out = dict(nAdvCellsForEdge=np.zeros(d.nEdges, dtype=np.int32), advCellsForEdge=np.zeros((d.nEdges, d.nAdvCells), dtype=np.int32),
                   adv_coefs=np.zeros((d.nEdges, d.nAdvCells)), adv_coefs_3rd=np.zeros((d.nEdges, d.nAdvCells)))
        self._call("adv_coef_compression", C.addressof(m), out["nAdvCellsForEdge"].ctypes.data, out["advCellsForEdge"].ctypes.data,
                   out["adv_coefs"].ctypes.data, out["adv_coefs_3rd"].ctypes.data)
        del keep
        return out

    def atm_couple_coef_3rd_order(self, config_coef_3rd_order: float, adv_coefs_3rd: Optional[np.ndarray] = None):
        """dynamics_tasks.rg:303-325: adv_coefs_3rd (in place, C-contiguous float64) and zb3_cell at level 0"""
        if adv_coefs_3rd is not None:
            assert adv_coefs_3rd.dtype == np.float64 and adv_coefs_3rd.flags.c_contiguous
        self._call("couple_coef_3rd_order", float(config_coef_3rd_order), None if adv_coefs_3rd is None else adv_coefs_3rd.ctypes.data)

    def atm_compute_mesh_scaling(self, mesh: Dict[str, np.ndarray], meshDensity: np.ndarray, config_h_ScaleWithMesh: bool = True):
        """dynamics_tasks.rg:595-646 -> {meshScalingDel2, meshScalingDel4}"""
        d = self.dims
        m, keep = _abi.init_mesh_ptrs({"cellsOnEdge": mesh["cellsOnEdge"]}, d)
        md = np.ascontiguousarray(meshDensity, dtype=np.float64)
        out = dict(meshScalingDel2=np.zeros(d.nEdges), meshScalingDel4=np.zeros(d.nEdges))
        self._call("compute_mesh_scaling", C.addressof(m), md.ctypes.data, int(bool(config_h_ScaleWithMesh)),
                   out["meshScalingDel2"].ctypes.data, out["meshScalingDel4"].ctypes.data)
        del keep
        return out

    def atm_compute_damping_coefs(self, meshDensity: np.ndarray, config_zd: float = 22000.0, config_xnutr: float = 0.2):
        """dynamics_tasks.rg:274-300: zgrid -> dss (after upload_mesh)"""
        md = np.ascontiguousarray(meshDensity, dtype=np.float64)
        assert md.shape == (self.dims.nCells,)
        self._call("compute_damping_coefs", md.ctypes.data, float(config_zd), float(config_xnutr))

    def init_atm_case_jw(self, latCell: np.ndarray, areaCell: np.ndarray, latVertex: np.ndarray, n_lat_table: int = 0):
        """vertical_init/init_atm_cases.rg:24-743 on the device (corrected reading = init_jw.py); geometry scaled to the sphere"""
        a = [np.ascontiguousarray(x, dtype=np.float64) for x in (latCell, areaCell, latVertex)]
        assert a[0].shape == (self.dims.nCells,) and a[1].shape == (self.dims.nCells,) and a[2].shape == (self.dims.nVertices,)
        geo = _abi.MpasJwGeometry(a[0].ctypes.data, a[1].ctypes.data, a[2].ctypes.data, int(n_lat_table))
        self._call("init_atm_case_jw", C.addressof(geo))

    def atm_rk_dynamics_substep_finish(self, dynamics_substep: int, dynamics_split: int):
        self._call("rk_dynamics_substep_finish", int(dynamics_substep), int(dynamics_split))

    def atm_srk3(self, dt: float):
        """The library's own replay of rk_timestep.rg:361-500 (one call, optionally a CUDA graph)."""
        self._call("srk3", float(dt))

    def atm_timestep(self, dt: float):
        self._call("timestep", float(dt))

    def atm_srk3_by_tasks(self, dt: float, hook=None, acoustic_pair=None):
        """atm_srk3 replayed task by task from the host, exactly in the reference's order
        (rk_timestep.rg:378-481).  ``hook(name, *args)`` is called after every task (halo exchange point).
        ``acoustic_pair(dts, small_step)``, if given, runs one iteration of the acoustic loop (:450-457) in place of
        the two task calls and their hooks (the multi-GPU driver splits them to overlap the halo exchange)."""
        c = self.cfg
        number_of_sub_steps = c.number_of_sub_steps
        dynamics_split = c.config_dynamics_split_steps
        rk_timestep = [dt / 3, dt / 2, dt]                                        # rk_timestep.rg:386-389
        rk_sub_timestep = [dt / 3, dt / number_of_sub_steps, dt / number_of_sub_steps]
        number_sub_steps = [max(1, number_of_sub_steps // 2), max(1, number_of_sub_steps // 2), number_of_sub_steps]
        h = hook or (lambda name, *args: None)
        self.atm_rk_integration_setup(); h("rk_integration_setup")
        self.atm_compute_moist_coefficients(); h("compute_moist_coefficients")
        self.atm_compute_vert_imp_coefs(rk_sub_timestep[0]); h("compute_vert_imp_coefs")
        for rk_step in range(3):
            if rk_step == 1:
                self.atm_compute_vert_imp_coefs(rk_sub_timestep[rk_step]); h("compute_vert_imp_coefs")
            rk_arg = int(rk_sub_timestep[rk_step]) if c.rkarg_policy == _abi.RKARG_SUBSTEP_TRUNC else rk_step
            self.atm_compute_dyn_tend(rk_arg, dt); h("compute_dyn_tend")
            self.atm_set_smlstep_pert_variables(); h("set_smlstep_pert_variables")
            for small_step in range(number_sub_steps[rk_step] + 1):
                if acoustic_pair is not None:
                    acoustic_pair(rk_sub_timestep[rk_step], small_step)
                    continue
                self.atm_advance_acoustic_step(rk_sub_timestep[rk_step], small_step); h("advance_acoustic_step", rk_sub_timestep[rk_step], small_step)
                self.atm_divergence_damping_3d(rk_sub_timestep[rk_step]); h("divergence_damping_3d")
            if c.physics_mode == _abi.PHYSICS_CORRECTED:      # rk_timestep.rg:459-460, commented out in the reference
                self.atm_recover_large_step_variables(number_sub_steps[rk_step], rk_step, dt); h("recover_large_step_variables")
            if c.config_scalar_advection:                     # rk_timestep.rg:465 (skipped by the reference), :469 = the halo update
                self.atm_advance_scalars(rk_timestep[rk_step], rk_step); h("advance_scalars")
            self.atm_compute_solve_diagnostics(False, rk_step); h("compute_solve_diagnostics", False, rk_step)
        self.atm_rk_dynamics_substep_finish(1, dynamics_split); h("rk_dynamics_substep_finish")


class Dynamics(TaskAPI):
    """One device-resident mirror (one GPU).  See module docstring."""

    def __init__(self, dims: MpasDims, cfg: Optional[MpasConfig] = None, lib_path: Optional[str] = None):
        self._lib = load_library(lib_path)
        self.dims = dims
        self.cfg = cfg if cfg is not None else _abi.default_config()
        self._h = C.c_void_p()
        rc = self._lib.mpasb200_create(C.byref(self.dims), C.byref(self.cfg), C.byref(self._h))
        if rc != 0:
            msg = self._lib.mpasb200_last_error(None)
            raise MpasB200Error(f"mpasb200_create failed ({rc}): {msg.decode() if msg else ''}")
        self._keep = []
        self._ids_cache = {}
        self._class_cache = {}

    # ---- plumbing ------------------------------------------------------------------------------
    def _check(self, rc: int, what: str):
        if rc != 0:
            msg = self._lib.mpasb200_last_error(self._h)
            raise MpasB200Error(f"mpasb200_{what} failed ({rc}): {msg.decode() if msg else ''}")

    def _call(self, name: str, *args):
        self._check(getattr(self._lib, "mpasb200_" + name)(self._h, *args), name)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.mpasb200_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- mesh + fields ---------------------------------------------------------------------------
    def upload_mesh(self, static: Dict[str, np.ndarray]):
        m, keep = _abi.mesh_ptrs(static, self.dims)
        self._check(self._lib.mpasb200_upload_mesh(self._h, C.byref(m)), "upload_mesh")
        self._class_cache = {}
        del keep

    def upload_field(self, name: str, a: np.ndarray):
        a = np.ascontiguousarray(a, dtype=np.float64)
        shp = self.field_shape(name)
        if a.shape != shp:
            raise ValueError(f"{name}: shape {a.shape}, expected {shp}")
        s = FIELD_SLOTS[name]
        L1 = self.dims.nVertLevels + 1
        self._check(self._lib.mpasb200_upload_field(self._h, FIELD_ID[name], a.ctypes.data, 8 * L1 * s, 8 * s), "upload_field")

    def download_field(self, name: str, out: Optional[np.ndarray] = None) -> np.ndarray:
        shp = self.field_shape(name)
        a = out if out is not None else np.empty(shp, dtype=np.float64)
        assert a.shape == shp and a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
        s = FIELD_SLOTS[name]
        L1 = self.dims.nVertLevels + 1
        self._check(self._lib.mpasb200_download_field(self._h, FIELD_ID[name], a.ctypes.data, 8 * L1 * s, 8 * s), "download_field")
        return a

    def upload_field_async(self, name: str, a: np.ndarray):
        """pipelined upload of a page-locked, C-contiguous array (mpas_b200.h); reuse ``a`` only after transfer_wait()."""
        assert a.shape == self.field_shape(name) and a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
        self._check(self._lib.mpasb200_upload_field_async(self._h, FIELD_ID[name], a.ctypes.data), "upload_field_async")

    def download_field_async(self, name: str, out: np.ndarray):
        """pipelined download into a page-locked, C-contiguous array; read ``out`` only after transfer_wait()."""
        assert out.shape == self.field_shape(name) and out.dtype == np.float64 and out.flags["C_CONTIGUOUS"]
        self._check(self._lib.mpasb200_download_field_async(self._h, FIELD_ID[name], out.ctypes.data), "download_field_async")

    def transfer_wait(self):
        self._check(self._lib.mpasb200_transfer_wait(self._h), "transfer_wait")

    def zero_field(self, name: str):
        self._check(self._lib.mpasb200_zero_field(self._h, FIELD_ID[name]), "zero_field")

    def sync(self):
        self._check(self._lib.mpasb200_sync(self._h), "sync")

    def set_stream(self, cuda_stream: int):
        self._check(self._lib.mpasb200_set_stream(self._h, C.c_void_p(cuda_stream)), "set_stream")

    def set_use_graph(self, on: bool):
        self._check(self._lib.mpasb200_set_use_graph(self._h, int(bool(on))), "set_use_graph")
        self.cfg.use_graph = int(bool(on))

    def class_range(self, entity: int, cls: int):
        """[begin, end) of a launch class (MpasMeshPtrs.cellClass / edgeClass) in the library's internal order."""
        b, e = C.c_int32(0), C.c_int32(0)
        self._check(self._lib.mpasb200_class_range(self._h, entity, cls, C.byref(b), C.byref(e)), "class_range")
        return int(b.value), int(e.value)

    def restrict(self, entity: int, cls=None):
        """run atm_advance_acoustic_step (cells) / atm_divergence_damping_3d (edges) on one launch class of
        MpasMeshPtrs.cellClass / edgeClass only; None = everything."""
        if cls is None:
            self.set_range(entity)
            return
        r = self._class_cache.get((entity, cls))
        if r is None:
            r = self._class_cache[(entity, cls)] = self.class_range(entity, cls)
        self.set_range(entity, r[0], r[1])

    def set_range(self, entity: int, begin: int = -1, end: int = -1):
        """restrict atm_advance_acoustic_step (cells) / atm_divergence_damping_3d (edges) to [begin, end); no arguments = everything."""
        self._check(self._lib.mpasb200_set_range(self._h, entity, begin, end), "set_range")

    # ---- summarize_timestep (rk_timestep.rg:29-359) as a device scan ------------------------------------
    def set_global_ids(self, entity: int, gid: Optional[np.ndarray]):
        """global id of every local entity (partitions): summaries then report places / checksums in global numbering."""
        if gid is None:
            self._check(self._lib.mpasb200_set_global_ids(self._h, entity, None, 0), "set_global_ids")
            return
        gid = np.ascontiguousarray(gid, dtype=np.int32)
        self._check(self._lib.mpasb200_set_global_ids(self._h, entity, gid.ctypes.data, gid.shape[0]), "set_global_ids")

    def summarize_field(self, name: str, n_first: Optional[int] = None, nlevels: Optional[int] = None) -> dict:
        """min / max (+ place), NaN / Inf counts and the order-independent bit checksum of the first ``n_first``
        entities (default all) and levels [0, nlevels) (default all nVertLevels+1) of a scalar 3-D field."""
        out = _abi.MpasFieldSummary()
        n = self.entity_count(FIELD_ENTITY[name]) if n_first is None else int(n_first)
        nl = self.dims.nVertLevels + 1 if nlevels is None else int(nlevels)
        self._check(self._lib.mpasb200_summarize_field(self._h, FIELD_ID[name], n, nl, C.byref(out)), "summarize_field")
        return out.as_dict()

    # ---- exact global integrals (mpasb200_integrate) ------------------------------------------------------------
    def register_weights(self, entity: int, w: np.ndarray) -> int:
        """upload a per-entity weight (caller's numbering, one value per local entity) once; returns its id"""
        w = np.ascontiguousarray(w, dtype=np.float64)
        wid = C.c_int32(-1)
        self._check(self._lib.mpasb200_register_weights(self._h, entity, w.ctypes.data, w.shape[0], C.byref(wid)), "register_weights")
        return int(wid.value)

    def integrate(self, a: str, slot_a: int = 0, b: Optional[str] = None, slot_b: int = 0, weight_id: Optional[int] = None,
                  wv: Optional[np.ndarray] = None, n_first: Optional[int] = None, nlevels: Optional[int] = None) -> dict:
        """the exact sum of ((a * b) * wh[i]) * wv[k] over the first ``n_first`` entities (default all) and levels
        [0, nlevels) (default all nVertLevels+1), non-finite products counted and left out (mpas_b200.h); see integral_result"""
        n = self.entity_count(FIELD_ENTITY[a]) if n_first is None else int(n_first)
        nl = self.dims.nVertLevels + 1 if nlevels is None else int(nlevels)
        if wv is not None:
            wv = np.ascontiguousarray(wv, dtype=np.float64)
            if wv.shape != (nl,):
                raise ValueError(f"wv: shape {wv.shape}, expected ({nl},)")
        out = _abi.MpasIntegral()
        self._check(self._lib.mpasb200_integrate(self._h, FIELD_ID[a], int(slot_a), -1 if b is None else FIELD_ID[b], int(slot_b),
                                                 -1 if weight_id is None else int(weight_id), None if wv is None else wv.ctypes.data,
                                                 n, nl, C.byref(out)), "integrate")
        return integral_result(out)

    # ---- the distributed step inside the library (mpasb200_dist_*) --------------------------------------------
    @staticmethod
    def dist_unique_id() -> bytes:
        """128 bytes (ncclGetUniqueId) made on ONE rank; the host's own channel carries them to the others"""
        buf = C.create_string_buffer(128)
        rc = load_library().mpasb200_dist_unique_id(buf)
        if rc != 0:
            raise MpasB200Error(f"mpasb200_dist_unique_id failed ({rc}): {load_library().mpasb200_last_error(None).decode()}")
        return buf.raw

    def dist_init(self, rank: int, world: int, unique_id: bytes):
        assert len(unique_id) == 128
        self._check(self._lib.mpasb200_dist_init(self._h, rank, world, C.c_char_p(unique_id)), "dist_init")

    def dist_set_halo(self, entity: int, send: Dict[int, np.ndarray], recv: Dict[int, np.ndarray]):
        """send / recv: peer rank -> local indices (partition.LocalMesh.send[ent] / .recv[ent])"""
        def flat(d):
            peers = sorted(d)
            off = np.cumsum([0] + [len(d[p]) for p in peers]).astype(np.int32)
            idx = np.concatenate([np.asarray(d[p], dtype=np.int32) for p in peers]) if peers else np.zeros(0, np.int32)
            return np.asarray(peers, dtype=np.int32), off, np.ascontiguousarray(idx, dtype=np.int32)
        sp, so, si = flat(send)
        rp, ro, ri = flat(recv)
        self._check(self._lib.mpasb200_dist_set_halo(self._h, entity, len(sp), sp.ctypes.data, so.ctypes.data, si.ctypes.data,
                                                     len(rp), rp.ctypes.data, ro.ctypes.data, ri.ctypes.data), "dist_set_halo")

    def dist_exchange(self, kind: int):
        self._check(self._lib.mpasb200_dist_exchange(self._h, int(kind)), "dist_exchange")

    def dist_flush(self):
        self._check(self._lib.mpasb200_dist_flush(self._h), "dist_flush")

    def atm_srk3_dist(self, dt: float):
        """atm_srk3 on one rank of an N-rank run, exchanges issued by the library (mpasb200_srk3_dist)"""
        self._check(self._lib.mpasb200_srk3_dist(self._h, float(dt)), "srk3_dist")

    # ---- halo building blocks ------------------------------------------------------------------------
    def register_list(self, entity: int, idx: np.ndarray) -> int:
        idx = np.ascontiguousarray(idx, dtype=np.int32)
        lid = C.c_int32(-1)
        self._check(self._lib.mpasb200_register_list(self._h, entity, idx.ctypes.data, idx.shape[0], C.byref(lid)), "register_list")
        return int(lid.value)

    def _field_ids(self, fields: Sequence[str]) -> np.ndarray:
        key = tuple(fields)
        ids = self._ids_cache.get(key)
        if ids is None:
            ids = self._ids_cache[key] = np.asarray([FIELD_ID[f] for f in fields], dtype=np.int32)
        return ids

    def pack(self, list_id: int, fields: Sequence[str], d_buf_ptr: int):
        ids = self._field_ids(fields)
        self._check(self._lib.mpasb200_pack(self._h, list_id, ids.ctypes.data, len(ids), C.c_void_p(d_buf_ptr)), "pack")

    def unpack(self, list_id: int, fields: Sequence[str], d_buf_ptr: int):
        ids = self._field_ids(fields)
        self._check(self._lib.mpasb200_unpack(self._h, list_id, ids.ctypes.data, len(ids), C.c_void_p(d_buf_ptr)), "unpack")

    # ---- introspection ------------------------------------------------------------------------------------
    @property
    def launch_count(self) -> int:
        return int(self._lib.mpasb200_launch_count(self._h))

    @property
    def device_bytes(self) -> int:
        return int(self._lib.mpasb200_device_bytes(self._h))

    def enable_timing(self, on: bool = True):
        self._check(self._lib.mpasb200_enable_timing(self._h, int(on)), "enable_timing")

    def reset_timing(self):
        self._check(self._lib.mpasb200_reset_timing(self._h), "reset_timing")

    def enable_kernel_timing(self, on=True):
        """on = 2 also keeps a timeline (see timeline())"""
        self._check(self._lib.mpasb200_enable_kernel_timing(self._h, int(on)), "enable_kernel_timing")

    def timeline(self):
        """[(kernel, start ms, end ms, stream)] since enable_kernel_timing(2); stream 0 = compute, 1 = communication"""
        out, i = [], 0
        while True:
            nm, t0, t1, st = C.c_char_p(), C.c_double(), C.c_double(), C.c_int()
            if self._lib.mpasb200_timeline_entry(self._h, i, C.byref(nm), C.byref(t0), C.byref(t1), C.byref(st)) != 0:
                return out
            out.append((nm.value.decode(), t0.value, t1.value, st.value))
            i += 1

    def reset_kernel_timing(self):
        self._check(self._lib.mpasb200_reset_kernel_timing(self._h), "reset_kernel_timing")

    def kernel_times(self) -> Dict[str, tuple]:
        """{kernel name: (total ms, launches)} measured with CUDA events on the launching stream."""
        out, i = {}, 0
        while True:
            nm, ms, n = C.c_char_p(), C.c_double(), C.c_int64()
            if self._lib.mpasb200_kernel_time(self._h, i, C.byref(nm), C.byref(ms), C.byref(n)) != 0:
                return out
            out[nm.value.decode()] = (ms.value, n.value)
            i += 1

    def task_times(self) -> Dict[str, tuple]:
        out = {}
        for t in range(len(_abi.TASK_NAMES)):
            ms, calls, nm = C.c_double(), C.c_int64(), C.c_char_p()
            self._check(self._lib.mpasb200_task_time(self._h, t, C.byref(ms), C.byref(calls), C.byref(nm)), "task_time")
            out[nm.value.decode()] = (ms.value, calls.value)
        return out


def integral_result(acc: _abi.MpasIntegral) -> dict:
    """an MpasIntegral as {value (rounded once), bits (of value, 16 hex digits), count, n_nan, n_pinf, n_ninf, limbs (int64[68])}"""
    v = float(load_library().mpasb200_integral_value(C.byref(acc)))
    return {"value": v, "bits": f"{int(np.float64(v).view(np.uint64)):016x}", "count": int(acc.count), "n_nan": int(acc.n_nan),
            "n_pinf": int(acc.n_pinf), "n_ninf": int(acc.n_ninf), "limbs": np.array(acc.limb[:], dtype=np.int64)}


def as_integral(r: dict) -> _abi.MpasIntegral:
    """the MpasIntegral of an integral_result dict (limbs and counts; the value is derived)"""
    acc = _abi.MpasIntegral()
    acc.limb[:] = [int(x) for x in r["limbs"]]
    acc.count, acc.n_nan, acc.n_pinf, acc.n_ninf = (int(r[k]) for k in ("count", "n_nan", "n_pinf", "n_ninf"))
    return acc


def merge_integrals(parts: Iterable[dict]) -> dict:
    """exact merge of integral_result dicts (mpasb200_integral_merge: the order of ``parts`` does not matter)"""
    lib, acc = load_library(), _abi.MpasIntegral()
    for r in parts:
        if lib.mpasb200_integral_merge(C.byref(acc), C.byref(as_integral(r))) != 0:
            raise MpasB200Error("mpasb200_integral_merge: the sum leaves the accumulator's range")
    return integral_result(acc)


def dims_of(mesh, nVertLevels: int) -> MpasDims:
    return _abi.make_dims(mesh.nCells, mesh.nEdges, mesh.nVertices, nVertLevels)
