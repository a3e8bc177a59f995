"""ctypes image of include/mpas_b200.h (POD structs, enums, the field table).

The field table is parsed from include/mpas_b200_fields.def so that there is exactly one
list of fields in the repository.
"""
from __future__ import annotations

import ctypes as C
import os
import re
from typing import Dict, List, Tuple

import numpy as np

REPO_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INCLUDE_DIR = os.path.join(REPO_ROOT, "include")

CELL, EDGE, VERTEX, VERTICAL = 0, 1, 2, 3
_ENT = {"CELL": CELL, "EDGE": EDGE, "VERTEX": VERTEX}

INDEX_LITERAL, INDEX_CORRECTED = 0, 1
MIX_2D_SMAGORINSKY, MIX_2D_FIXED, MIX_OTHER = 0, 1, 2
RKARG_SUBSTEP_TRUNC, RKARG_STAGE_INDEX = 0, 1
PHYSICS_LITERAL, PHYSICS_CORRECTED = 0, 1

X_ACOUSTIC_FIRST, X_ACOUSTIC, X_DIAG, X_RECOVER, X_SCALARS = range(5)     # mpasb200_dist_exchange kinds

E_OK, E_INVAL, E_CUDA, E_NODEVICE, E_STATE, E_NOMEM = 0, -1, -2, -3, -4, -5

TASK_NAMES = ("rk_integration_setup", "compute_moist_coefficients", "compute_vert_imp_coefs", "compute_dyn_tend",
              "set_smlstep_pert_variables", "advance_acoustic_step", "divergence_damping_3d",
              "recover_large_step_variables", "compute_solve_diagnostics", "rk_dynamics_substep_finish", "advance_scalars")


def _parse_fields() -> List[Tuple[str, int, int]]:
    out = []
    with open(os.path.join(INCLUDE_DIR, "mpas_b200_fields.def")) as fh:
        for line in fh:
            m = re.match(r"\s*MPASB200_FIELD\(\s*(\w+)\s*,\s*(\w+)\s*,\s*(\d+)\s*\)", line)
            if m:
                out.append((m.group(1), _ENT[m.group(2)], int(m.group(3))))
                continue
            m = re.match(r"\s*MPASB200_VFIELD\(\s*(\w+)\s*\)", line)
            if m and m.group(1) != "name":
                out.append((m.group(1), VERTICAL, 1))
    return out


FIELDS: List[Tuple[str, int, int]] = _parse_fields()
FIELD_ID: Dict[str, int] = {n: i for i, (n, _, _) in enumerate(FIELDS)}
FIELD_ENTITY: Dict[str, int] = {n: e for (n, e, _) in FIELDS}
FIELD_SLOTS: Dict[str, int] = {n: s for (n, _, s) in FIELDS}
N_FIELDS = len(FIELDS)


RESTART_WHEN = ("ALWAYS", "CORRECTED", "SCALARS")


def _parse_restart() -> List[Tuple[str, str]]:
    out = []
    with open(os.path.join(INCLUDE_DIR, "mpas_b200_restart.def")) as fh:
        for line in fh:
            m = re.match(r"\s*MPASB200_RESTART\(\s*(\w+)\s*,\s*(\w+)\s*\)", line)
            if m:
                if m.group(1) not in FIELD_ID or m.group(2) not in RESTART_WHEN:
                    raise ValueError(f"mpas_b200_restart.def: bad line {line.strip()}")
                out.append((m.group(1), m.group(2)))
    return out


#: include/mpas_b200_restart.def: (field, when) in file order
RESTART: List[Tuple[str, str]] = _parse_restart()


def restart_fields(cfg: "MpasConfig") -> List[str]:
    """the restart set under ``cfg``, in the order of mpasb200_restart_fields"""
    on = {"ALWAYS": True, "CORRECTED": cfg.physics_mode == PHYSICS_CORRECTED, "SCALARS": cfg.config_scalar_advection != 0}
    return [n for n, when in RESTART if on[when]]


class MpasDims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in
                ("nCells", "nEdges", "nVertices", "nVertLevels", "maxEdges", "maxEdges2", "vertexDegree", "nAdvCells")]


_CFG_D = ("gravity", "rgas", "cp", "cv", "omega", "sphere_radius", "prandtl", "config_epssm", "config_smdiv",
          "config_len_disp", "config_smagorinsky_coef", "config_visc4_2dsmag", "config_del4u_div_factor",
          "config_v_mom_eddy_visc2", "config_v_theta_eddy_visc2", "config_h_mom_eddy_visc4",
          "config_h_theta_eddy_visc4", "config_rayleigh_damp_u_timescale_days", "config_mpas_cam_coef")
_CFG_I = ("config_number_rayleigh_damp_u_levels", "config_horiz_mixing", "config_mix_full", "config_rayleigh_damp_u",
          "nRelaxZone", "number_of_sub_steps", "config_dynamics_split_steps", "index_policy", "rkarg_policy",
          "sfc_renumber", "device", "use_graph", "acoustic_exact", "acoustic_tma", "physics_mode", "gather_stage", "config_scalar_advection", "edge_tiles", "kernel_forms", "reserved0")


class MpasConfig(C.Structure):
    _fields_ = [(n, C.c_double) for n in _CFG_D] + [(n, C.c_int32) for n in _CFG_I] + [("config_coef_3rd_order", C.c_double)]


# (member, ctype, entity, width-key)   width-key: 1 | "maxEdges" | "maxEdges2" | "vertexDegree" | "nAdvCells" | 2
MESH_MEMBERS = (
    ("nEdgesOnCell", np.int32, CELL, 1), ("edgesOnCell", np.int32, CELL, "maxEdges"),
    ("verticesOnCell", np.int32, CELL, "maxEdges"), ("kiteForCell", np.int32, CELL, "maxEdges"),
    ("edgesOnCellSign", np.float64, CELL, "maxEdges"), ("edgesOnCell_sign", np.float64, CELL, "maxEdges"),
    ("invAreaCell", np.float64, CELL, 1), ("latCell", np.float64, CELL, 1),
    ("defc_a", np.float64, CELL, "maxEdges"), ("defc_b", np.float64, CELL, "maxEdges"),
    ("bdyMaskCell", np.int32, CELL, 1), ("specZoneMaskCell", np.float64, CELL, 1),
    ("isShared", np.uint8, CELL, 1), ("inCpr", np.uint8, CELL, 1),
    ("cellsOnEdge", np.int32, EDGE, 2), ("verticesOnEdge", np.int32, EDGE, 2),
    ("nEdgesOnEdge", np.int32, EDGE, 1), ("edgesOnEdge_ECP", np.int32, EDGE, "maxEdges2"),
    ("edgesOnEdge", np.int32, EDGE, "maxEdges2"), ("weightsOnEdge", np.float64, EDGE, "maxEdges2"),
    ("dcEdge", np.float64, EDGE, 1), ("dvEdge", np.float64, EDGE, 1),
    ("invDcEdge", np.float64, EDGE, 1), ("invDvEdge", np.float64, EDGE, 1),
    ("angleEdge", np.float64, EDGE, 1), ("latEdge", np.float64, EDGE, 1),
    ("nAdvCellsForEdge", np.int32, EDGE, 1), ("advCellsForEdge", np.int32, EDGE, "nAdvCells"),
    ("adv_coefs", np.float64, EDGE, "nAdvCells"), ("adv_coefs_3rd", np.float64, EDGE, "nAdvCells"),
    ("meshScalingDel2", np.float64, EDGE, 1), ("meshScalingDel4", np.float64, EDGE, 1),
    ("specZoneMaskEdge", np.float64, EDGE, 1),
    ("edgesOnVertex", np.int32, VERTEX, "vertexDegree"), ("edgesOnVertexSign", np.float64, VERTEX, "vertexDegree"),
    ("edgesOnVertex_sign", np.float64, VERTEX, "vertexDegree"), ("kiteAreasOnVertex", np.float64, VERTEX, "vertexDegree"),
    ("fVertex", np.float64, VERTEX, 1), ("invAreaTriangle", np.float64, VERTEX, 1),
    ("xCell", np.float64, CELL, 1), ("yCell", np.float64, CELL, 1), ("zCell", np.float64, CELL, 1),
    ("cellClass", np.uint8, CELL, 1), ("edgeClass", np.uint8, EDGE, 1),
    ("lonCell", np.float64, CELL, 1), ("coeffs_reconstruct", np.float64, CELL, "maxEdges3"),
)


class MpasFieldSummary(C.Structure):
    """image of MpasFieldSummary (mpas_b200.h): the device form of summarize_timestep, rk_timestep.rg:29-359"""
    _fields_ = [("min", C.c_double), ("max", C.c_double), ("min_index", C.c_int64), ("max_index", C.c_int64),
                ("min_level", C.c_int32), ("max_level", C.c_int32), ("n_nan", C.c_int64), ("n_inf", C.c_int64),
                ("count", C.c_int64), ("checksum", C.c_uint64)]

    def as_dict(self):
        return {"min": self.min, "max": self.max, "min_at": [int(self.min_index), int(self.min_level)],
                "max_at": [int(self.max_index), int(self.max_level)], "n_nan": int(self.n_nan), "n_inf": int(self.n_inf),
                "count": int(self.count), "checksum": f"{int(self.checksum):016x}"}


INTEGRAL_LIMBS, INTEGRAL_BIAS = 68, 1088     # MpasIntegral: sum = sum_j limb[j] * 2^(32 j - INTEGRAL_BIAS), exactly


class MpasIntegral(C.Structure):
    """image of MpasIntegral (mpas_b200.h): an exact global integral as a fixed-point accumulator, plus its counts"""
    _fields_ = [("limb", C.c_int64 * INTEGRAL_LIMBS), ("count", C.c_int64), ("n_nan", C.c_int64), ("n_pinf", C.c_int64),
                ("n_ninf", C.c_int64)]


#: mpasb200_isobaric_diagnostics: at most this many pressure levels per call; each output row is surface pressure, then per
#: level these six values in this order
ISOBARIC_MAX_LEVELS = 32
ISOBARIC_FIELDS = ("temperature", "height", "uzonal", "umeridional", "w", "vorticity")


INIT_MESH_MEMBERS = (
    ("nEdgesOnCell", np.int32, CELL, 1), ("edgesOnCell", np.int32, CELL, "maxEdges"), ("verticesOnCell", np.int32, CELL, "maxEdges"),
    ("cellsOnCell", np.int32, CELL, "maxEdges"), ("cellsOnEdge", np.int32, EDGE, 2), ("verticesOnEdge", np.int32, EDGE, 2),
    ("cellsOnVertex", np.int32, VERTEX, "vertexDegree"), ("edgesOnVertex", np.int32, VERTEX, "vertexDegree"),
    ("dcEdge", np.float64, EDGE, 1), ("dvEdge", np.float64, EDGE, 1), ("deriv_two", np.float64, EDGE, "twoFifteen"),
)


class MpasInitMesh(C.Structure):
    """image of MpasInitMesh (mpas_b200.h): raw connectivity for the mesh-only producers of atm_core_init"""
    _fields_ = [(n, C.c_void_p) for (n, _, _, _) in INIT_MESH_MEMBERS]


def init_mesh_ptrs(arrays: Dict[str, np.ndarray], dims: "MpasDims"):
    """MpasInitMesh over numpy arrays (missing members stay null); the keep-alive list must outlive the call"""
    m, keep = MpasInitMesh(), []
    counts = {CELL: dims.nCells, EDGE: dims.nEdges, VERTEX: dims.nVertices}
    for name, dt, ent, wkey in INIT_MESH_MEMBERS:
        a = arrays.get(name)
        if a is None:
            setattr(m, name, None)
            continue
        w = wkey if isinstance(wkey, int) else (2 * dims.nAdvCells if wkey == "twoFifteen" else getattr(dims, wkey))
        a = np.ascontiguousarray(a, dtype=dt)
        want = (counts[ent],) if w == 1 else (counts[ent], w)
        if a.shape != want:
            raise ValueError(f"{name}: shape {a.shape}, expected {want}")
        keep.append(a)
        setattr(m, name, a.ctypes.data)
    return m, keep


class MpasJwGeometry(C.Structure):
    """image of MpasJwGeometry (mpas_b200.h)"""
    _fields_ = [("latCell", C.c_void_p), ("areaCell", C.c_void_p), ("latVertex", C.c_void_p), ("n_lat_table", C.c_int32)]


class MpasMeshPtrs(C.Structure):
    _fields_ = [(n, C.c_void_p) for (n, _, _, _) in MESH_MEMBERS]


def make_dims(nCells, nEdges, nVertices, nVertLevels, maxEdges=10, maxEdges2=20, vertexDegree=3, nAdvCells=15) -> MpasDims:
    return MpasDims(nCells, nEdges, nVertices, nVertLevels, maxEdges, maxEdges2, vertexDegree, nAdvCells)


EDGE_TILES_DEFAULT = 0
KERNEL_FORMS_DEFAULT = 0
KF_SPLIT_CELLC = 1


def default_config(**over) -> MpasConfig:
    """The values of constants.rg (reference: constants.rg:27-69,99-104; rk_timestep.rg:378-382).
    Mirrors mpasb200_default_config; tests check the two agree."""
    rgas = 287.0
    cp = 7.0 * rgas / 2.0
    c = MpasConfig()
    c.gravity, c.rgas, c.cp, c.cv = 9.80616, rgas, cp, cp - rgas
    c.omega, c.sphere_radius, c.prandtl = 7.29212e-5, 6371229.0, 1.0
    c.config_epssm, c.config_smdiv, c.config_len_disp = 0.1, 0.1, 120000.0
    c.config_smagorinsky_coef, c.config_visc4_2dsmag, c.config_del4u_div_factor = 0.125, 0.05, 10.0
    c.config_v_mom_eddy_visc2 = c.config_v_theta_eddy_visc2 = 0.0
    c.config_h_mom_eddy_visc4 = c.config_h_theta_eddy_visc4 = 0.0
    c.config_rayleigh_damp_u_timescale_days, c.config_mpas_cam_coef = 5.0, 0.0
    c.config_number_rayleigh_damp_u_levels = 6
    c.config_horiz_mixing = MIX_2D_SMAGORINSKY
    c.config_mix_full = c.config_rayleigh_damp_u = 0
    c.nRelaxZone, c.number_of_sub_steps, c.config_dynamics_split_steps = 5, 2, 1
    c.index_policy, c.rkarg_policy = INDEX_CORRECTED, RKARG_SUBSTEP_TRUNC
    c.sfc_renumber, c.device, c.use_graph, c.acoustic_exact, c.acoustic_tma = 1, -1, 0, 0, 3
    c.physics_mode = PHYSICS_LITERAL
    c.gather_stage = 0
    c.config_scalar_advection = 0
    c.edge_tiles = EDGE_TILES_DEFAULT
    c.kernel_forms = KERNEL_FORMS_DEFAULT
    c.reserved0 = 0
    c.config_coef_3rd_order = 0.25
    for k, v in over.items():
        if not hasattr(c, k):
            raise AttributeError(k)
        setattr(c, k, v)
    return c


def mesh_ptrs(static: Dict[str, np.ndarray], dims: MpasDims):
    """Build an MpasMeshPtrs over numpy arrays (returned keep-alive list must outlive the call)."""
    m = MpasMeshPtrs()
    keep = []
    counts = {CELL: dims.nCells, EDGE: dims.nEdges, VERTEX: dims.nVertices}
    for name, dt, ent, wkey in MESH_MEMBERS:
        a = static.get(name)
        if a is None:
            setattr(m, name, None)
            continue
        w = wkey if isinstance(wkey, int) else (3 * dims.maxEdges if wkey == "maxEdges3" else getattr(dims, wkey))
        a = np.ascontiguousarray(a, dtype=dt)
        if wkey == "maxEdges3":
            a = a.reshape(a.shape[0], -1)
        want = (counts[ent],) if w == 1 else (counts[ent], w)
        if a.shape != want:
            raise ValueError(f"{name}: shape {a.shape}, expected {want}")
        keep.append(a)
        setattr(m, name, a.ctypes.data)
    return m, keep
