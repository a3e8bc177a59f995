"""JW baroclinic-wave style initial state + the rest of the harness inputs for the hot path.

Follows the formulas of ``init_atm_case_jw`` (reference: vertical_init/init_atm_cases.rg:
144-160 terrain/constants, 165-255 vertical grid, 257-263 zxu, 417-522 hydrostatic column
iterations, 530-596 zonal wind / ru / Coriolis, 616-665 zb, 681-704 rw and w, 716-723 v),
vectorised over columns, with u0=35, t0=288, t0b=250, dtdz=0.005, eta_t=0.2, zt=45000,
str=1.5.  The reference routine cannot be restated literally: it indexes regions with
swapped (level, cell) pairs far out of range (init_atm_cases.rg:266,268,419,447), uses
zw[k]=(k-1)*dz with 0-based k (:198) and sh[0]=-1 (:178).  This module is the CORRECTED
reading (what the MPAS Fortran does); it only *generates inputs* -- the kernels and the
oracle are pure functions of their inputs, so parity does not depend on it.

Then the ``atm_core_init`` chain (atm_core.rg:22-42) is applied through core_init.py, and
the fields the reference never writes (SURVEY.md 8c, rule M5) get deterministic,
non-degenerate values so that parity is not a comparison of zeros.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict

import numpy as np

from . import core_init
from .mesh import CORRECTED, FIFTEEN, LITERAL, MAX_EDGES, MAX_EDGES2, VERTEX_DEGREE, Mesh, resolve_ids

# constants.rg:27-38
SPHERE_RADIUS = 6371229.0
OMEGA = 7.29212e-5
RGAS = 287.0
CP = 7.0 * RGAS / 2.0
GRAVITY = 9.80616
PII = 3.141592653589793
SEED = 20261018


@dataclass
class HostState:
    """Host-side image of the regions: what the Regent program would hold after
    load_mesh + init_atm_case_jw + atm_core_init, restricted to hot-path fields."""

    nVertLevels: int
    policy: int
    mesh: Mesh                       # geometry scaled to the sphere
    static: Dict[str, np.ndarray] = field(default_factory=dict)   # level-0 fields (MpasMeshPtrs members)
    f: Dict[str, np.ndarray] = field(default_factory=dict)        # 3-D fields [n, L+1] (or [n, L+1, slots])
    vert: Dict[str, np.ndarray] = field(default_factory=dict)     # vertical_fs [L+1]
    extras: Dict[str, np.ndarray] = field(default_factory=dict)   # init-only inputs (coeffs_reconstruct, zb, ...)


def scale_mesh(mesh: Mesh, policy: int, a: float = SPHERE_RADIUS) -> Mesh:
    """init_atm_cases.rg:87-111.  kiteAreasOnVertex is NOT scaled under LITERAL: the reference
    writes element [vertexDegree], one past the array (:100)."""
    v = dict(mesh.v)
    for k in ("xCell", "yCell", "zCell", "xVertex", "yVertex", "zVertex", "xEdge", "yEdge", "zEdge", "dvEdge", "dcEdge"):
        v[k] = v[k] * a
    v["areaCell"] = v["areaCell"] * a ** 2.0
    v["areaTriangle"] = v["areaTriangle"] * a ** 2.0
    if policy == CORRECTED:
        v["kiteAreasOnVertex"] = v["kiteAreasOnVertex"] * a ** 2.0
    return Mesh(v=v, partition=mesh.partition, name=mesh.name)


def _smooth(modes, x, y, z, nlev1, amp, base=0.0):
    """low-order smooth field on the unit sphere x level, amplitude ~amp around base.  ``modes`` [nmodes, 6] rows
    (c0, c1, c2, c3, phase, wavenumber) from m5_draws; pointwise in (x, y, z), so any subset of rows evaluates alone."""
    out = np.full((x.shape[0], nlev1), base, dtype=np.float64)
    k = np.arange(nlev1) / max(nlev1 - 1, 1)
    nmodes = len(modes)
    for c in modes:
        horiz = c[0] * x + c[1] * y + c[2] * z + c[3] * x * y
        out += amp / nmodes * horiz[:, None] * np.cos(np.pi * c[5] * k + c[4])[None, :]
    return out


def m5_draws(nC: int, nE: int, L: int, seed: int = SEED) -> Dict[str, np.ndarray]:
    """Every random number the harness draws for the never-written fields (rule M5), in the order make_state has always
    drawn them: zb3 factor, deriv_two, defc_a / defc_b, ten _smooth mode sets, u_init / v_init, coeffs_reconstruct.
    Unscaled: make_static scales them with the mesh."""
    rng = np.random.default_rng(seed)
    d = dict(zb3_factor=rng.uniform(0.5, 1.5, size=(nE, 1, 2)), deriv_two=rng.normal(size=(nE, 2 * FIFTEEN)),
             defc_a=rng.normal(size=(nC, MAX_EDGES)), defc_b=rng.normal(size=(nC, MAX_EDGES)))
    modes = np.zeros((len(M5_SMOOTH), 4, 6))
    for f in range(len(M5_SMOOTH)):
        for m in range(4):
            modes[f, m, :4] = rng.normal(size=4)
            modes[f, m, 4] = rng.uniform(0, 2 * np.pi)
            modes[f, m, 5] = rng.integers(1, 3)
    d["modes"] = modes
    d["u_init"] = 10.0 + rng.normal(size=L)
    d["v_init"] = rng.normal(size=L)
    d["coeffs_reconstruct"] = rng.normal(size=(nC, MAX_EDGES, 3)) * 0.3
    return d


#: the M5 fields built from a _smooth mode set, in draw order: (field, cell or edge, amplitude, base, kind);
#: kind "factor" multiplies theta_m by (1 + smooth), "one_plus" is 1 + smooth
M5_SMOOTH = (("h", "cell", 50.0, 1000.0, "plain"), ("rt_diabatic_tend", "cell", 1e-4, 0.0, "plain"),
             ("t_init", "cell", 0.01, 0.0, "factor"), ("tend_rho_physics", "cell", 1e-6, 0.0, "plain"),
             ("tend_rtheta_physics", "cell", 1e-3, 0.0, "plain"), ("theta_m_save", "cell", 0.01, 0.0, "factor"),
             ("tend_ru_physics", "edge", 1e-4, 0.0, "plain"), ("u_tend", "edge", 1e-2, 0.0, "plain"),
             ("tend_ru", "edge", 1e-2, 0.0, "plain"), ("cqu", "edge", 0.01, 0.0, "one_plus"))


def m5_fields(modes: np.ndarray, cell_xyz, edge_xyz, theta_m: np.ndarray, rho_zz: np.ndarray, c1: np.ndarray,
              c2: np.ndarray) -> Dict[str, np.ndarray]:
    """The 3-D M5 fields on any set of rows: the _smooth ones are pointwise in the UNIT-sphere coordinates ``cell_xyz`` /
    ``edge_xyz``; t_init and theta_m_save scale ``theta_m`` of the same cells; rho_edge averages the coupled ``rho_zz`` of
    the cells c1 / c2 (0-based rows of rho_zz, len(rho_zz) = the zero pad).  Same keys and order as make_state's."""
    L1 = theta_m.shape[1]
    lev = np.arange(L1)[None, :] < L1 - 1
    out = {}
    rz_p = np.concatenate([rho_zz, np.zeros((1, L1))], 0)
    for i, (name, ent, amp, base, kind) in enumerate(M5_SMOOTH):
        if name == "tend_ru_physics":      # rho_edge sits between the cell and the edge fields
            with np.errstate(invalid="ignore", over="ignore"):
                out["rho_edge"] = np.where(lev, 0.5 * (rz_p[c1] + rz_p[c2]), 0.0)
        s = _smooth(modes[i], *(cell_xyz if ent == "cell" else edge_xyz), L1, amp, base)
        if kind == "factor":
            s = theta_m * (1.0 + s)
        elif kind == "one_plus":
            s = 1.0 + s
        out[name] = np.where(lev, s, 0.0)
    return out


def vertical_grid(L: int, zt: float = 45000.0, strf: float = 1.5):
    """init_atm_cases.rg:165-237, corrected indexing: zw[k] = k*dz."""
    dz = zt / L
    k = np.arange(L + 1, dtype=np.float64)
    zw = k * dz
    sh = (k * dz / zt) ** strf
    ah = 1.0 - np.cos(0.5 * PII * k * dz / zt) ** 6.0
    dzw = zw[1:] - zw[:-1]
    vert = {n: np.zeros(L + 1) for n in ("rdzw", "rdzu", "fzm", "fzp", "cf1", "cf2", "cf3", "u_init", "v_init", "cofrz")}
    vert["rdzw"][:L] = 1.0 / dzw
    dzu = np.zeros(L + 1)
    dzu[1:L] = 0.5 * (dzw[1:L] + dzw[0:L - 1])
    vert["rdzu"][1:L] = 1.0 / dzu[1:L]
    vert["fzp"][1:L] = 0.5 * dzw[1:L] / dzu[1:L]
    vert["fzm"][1:L] = 0.5 * dzw[0:L - 1] / dzu[1:L]
    cof1 = (2.0 * dzu[1] + dzu[2]) / (dzu[1] + dzu[2]) * dzw[0] / dzu[1]
    cof2 = dzu[1] / (dzu[1] + dzu[2]) * dzw[0] / dzu[2]
    vert["cf1"][0] = vert["fzp"][1] + cof1
    vert["cf2"][0] = vert["fzm"][1] - cof1 - cof2
    vert["cf3"][0] = cof2
    return zw, sh, ah, dzw, dzu, vert


def make_static(mesh_unit: Mesh, nVertLevels: int, policy: int = CORRECTED, m5: bool = True, seed: int = SEED):
    """The part of make_state that needs no 3-D array: level-0 ("static") data, the vertical grid with u_init / v_init,
    and the harness draws (rule M5).  Returns (HostState with static / vert / extras[coeffs_reconstruct, deriv_two] set
    and no fields, the m5_draws dict or None)."""
    L = nVertLevels
    mesh = scale_mesh(mesh_unit, policy)
    v = mesh.v
    nC, nE = mesh.nCells, mesh.nEdges
    st = HostState(nVertLevels=L, policy=policy, mesh=mesh)
    st.vert = vertical_grid(L)[-1]
    dr = m5_draws(nC, nE, L, seed) if m5 else None
    S = st.static
    S["fVertex"] = 2.0 * OMEGA * np.sin(v["latVertex"])
    sg = core_init.atm_compute_signs(mesh, policy)
    deriv_two = dr["deriv_two"] * (0.05 / (v["dcEdge"] ** 2))[:, None] if m5 else None
    adv = core_init.atm_adv_coef_compression(mesh, policy, deriv_two)
    adv3, _ = core_init.atm_couple_coef_3rd_order(0.25, adv["adv_coefs_3rd"], None)
    ms = core_init.atm_compute_mesh_scaling(mesh, policy, True)
    S.update(nEdgesOnCell=v["nEdgesOnCell"], edgesOnCell=v["edgesOnCell"], verticesOnCell=v["verticesOnCell"],
             kiteForCell=sg["kiteForCell"], edgesOnCellSign=sg["edgesOnCellSign"], latCell=v["latCell"],
             cellsOnEdge=v["cellsOnEdge"], verticesOnEdge=v["verticesOnEdge"], nEdgesOnEdge=v["nEdgesOnEdge"],
             edgesOnEdge_ECP=v["edgesOnEdge"], weightsOnEdge=v["weightsOnEdge"], dcEdge=v["dcEdge"], dvEdge=v["dvEdge"],
             angleEdge=v["angleEdge"], latEdge=v["latEdge"], nAdvCellsForEdge=adv["nAdvCellsForEdge"],
             advCellsForEdge=adv["advCellsForEdge"], adv_coefs=adv["adv_coefs"], adv_coefs_3rd=adv3,
             meshScalingDel2=ms["meshScalingDel2"], meshScalingDel4=ms["meshScalingDel4"],
             edgesOnVertex=v["edgesOnVertex"], edgesOnVertexSign=sg["edgesOnVertexSign"],
             kiteAreasOnVertex=v["kiteAreasOnVertex"],
             xCell=v["xCell"], yCell=v["yCell"], zCell=v["zCell"])
    S["isShared"] = np.zeros(nC, dtype=np.uint8)
    S["inCpr"] = np.ones(nC, dtype=np.uint8)
    S["bdyMaskCell"] = np.zeros(nC, dtype=np.int32)
    if m5:
        nEoC = v["nEdgesOnCell"]
        S["invAreaCell"] = 1.0 / v["areaCell"]
        S["invDcEdge"] = 1.0 / v["dcEdge"]
        S["invDvEdge"] = 1.0 / v["dvEdge"]
        S["invAreaTriangle"] = 1.0 / v["areaTriangle"]
        S["edgesOnCell_sign"] = sg["edgesOnCellSign"].copy()
        S["edgesOnVertex_sign"] = sg["edgesOnVertexSign"].copy()
        S["edgesOnEdge"] = v["edgesOnEdge"].copy()
        S["specZoneMaskCell"] = np.zeros(nC)
        S["specZoneMaskEdge"] = np.zeros(nE)
        slot = (np.arange(MAX_EDGES)[None, :] < nEoC[:, None])
        S["defc_a"] = np.where(slot, dr["defc_a"], 0.0) / np.sqrt(v["areaCell"])[:, None]
        S["defc_b"] = np.where(slot, dr["defc_b"], 0.0) / np.sqrt(v["areaCell"])[:, None]
        st.vert["u_init"][:L] = dr["u_init"]
        st.vert["v_init"][:L] = dr["v_init"]
        coeffs = dr["coeffs_reconstruct"]
    else:
        coeffs = np.zeros((nC, MAX_EDGES, 3))
    # inputs of the device-side init chain (mpasb200_init_coupled_diagnostics / mpasb200_reconstruct_2d)
    S["lonCell"] = v["lonCell"]
    S["coeffs_reconstruct"] = coeffs
    st.extras = dict(coeffs_reconstruct=coeffs, deriv_two=deriv_two)
    return st, dr


def make_state(mesh_unit: Mesh, nVertLevels: int, policy: int = CORRECTED, m5: bool = True,
               seed: int = SEED, diag_on_host: bool = True, keep_jw: bool = False) -> HostState:
    """Build every hot-path input.  ``m5`` = fill never-written fields (rule M5); with
    m5=False they stay zero (rule M1, the literal reading).  The level-0 data, the vertical grid and the draws come
    from make_static; this adds the 3-D fields."""
    L = nVertLevels
    L1 = L + 1
    st, dr = make_static(mesh_unit, L, policy, m5, seed)
    mesh = st.mesh
    v = mesh.v
    nC, nE, nV = mesh.nCells, mesh.nEdges, mesh.nVertices
    F = st.f
    S = st.static

    zw, sh, ah, dzw, dzu, _ = vertical_grid(L)
    vert = st.vert
    u0, t0, t0b, dtdz, eta_t, delta_t = 35.0, 288.0, 250.0, 0.005, 0.2, 4.8e5
    etavs0 = (1.0 - 0.252) * PII / 2.0
    p0 = 1.0e5
    zt = 45000.0
    r_earth = SPHERE_RADIUS

    def terrain(phi):
        return u0 / GRAVITY * np.cos(etavs0) ** 1.5 * (
            (-2.0 * np.sin(phi) ** 6 * (np.cos(phi) ** 2 + 1.0 / 3.0) + 10.0 / 63.0) * u0 * np.cos(etavs0) ** 1.5
            + (1.6 * np.cos(phi) ** 3 * (np.sin(phi) ** 2 + 2.0 / 3.0) - PII / 4.0) * r_earth * OMEGA)

    latC = v["latCell"]
    hx = terrain(latC)
    zgrid = (1.0 - ah)[None, :] * (sh[None, :] * (zt - hx[:, None]) + hx[:, None]) + (ah * sh)[None, :] * zt
    zz = np.zeros((nC, L1))
    zz[:, :L] = dzw[None, :] / (zgrid[:, 1:] - zgrid[:, :-1])
    F["zgrid"], F["zz"] = zgrid, zz

    c1 = resolve_ids(v["cellsOnEdge"][:, 0], nC, policy)
    c2 = resolve_ids(v["cellsOnEdge"][:, 1], nC, policy)
    pad = lambda a: np.concatenate([a, np.zeros((1,) + a.shape[1:], a.dtype)], 0)
    zg_p = pad(zgrid)
    zxu = np.zeros((nE, L1))
    zxu[:, :L] = 0.5 * (zg_p[c2, :L] - zg_p[c1, :L] + zg_p[c2, 1:] - zg_p[c1, 1:]) / v["dcEdge"][:, None]
    F["zxu"] = zxu

    # ---- hydrostatic base state + 10 x 25 iterations per column (:417-516), qv = 0.
    # The state is zonally symmetric, so the column iteration runs on a latitude table
    # (as the reference's own 2-D (z,lat) section does, :278-383) and pp, tt are
    # interpolated to the cells; rr is then recomputed pointwise so the column relations hold.
    def column_solve(lat_t):
        hx_t = terrain(lat_t)
        zg_t = (1.0 - ah)[None, :] * (sh[None, :] * (zt - hx_t[:, None]) + hx_t[:, None]) + (ah * sh)[None, :] * zt
        zz_t = dzw[None, :] / (zg_t[:, 1:] - zg_t[:, :-1])
        zt_t = 0.5 * (zg_t[:, 1:] + zg_t[:, :-1])
        ppb_t = p0 * np.exp(-GRAVITY * zt_t / (RGAS * t0b))
        rb_t = ppb_t / (RGAS * t0b * zz_t)
        pp_t = np.zeros_like(ppb_t)
        phi_t = lat_t[:, None]
        tt_t = None
        wgt = dzu[1:L] * GRAVITY
        for _itr in range(10):
            eta = (ppb_t + pp_t) / p0
            etav = (eta - 0.252) * PII / 2.0
            teta = t0 * eta ** (RGAS * dtdz / GRAVITY) + np.where(eta >= eta_t, 0.0, delta_t * np.maximum(eta_t - eta, 0.0) ** 5)
            cosv = np.maximum(np.cos(etav), 0.0)
            tt_t = teta + 0.75 * eta * PII * u0 / RGAS * np.sin(etav) * np.sqrt(cosv) * (
                (-2.0 * np.sin(phi_t) ** 6 * (np.cos(phi_t) ** 2 + 1.0 / 3.0) + 10.0 / 63.0) * 2.0 * u0 * cosv ** 1.5
                + (1.6 * np.cos(phi_t) ** 3 * (np.sin(phi_t) ** 2 + 2.0 / 3.0) - PII / 4.0) * r_earth * OMEGA)
            for _itrp in range(25):
                rr_t = (pp_t / (RGAS * zz_t) - rb_t * (tt_t - t0b)) / tt_t
                ppi0 = p0 - 0.5 * dzw[0] * GRAVITY * (1.25 * (rr_t[:, 0] + rb_t[:, 0]) - 0.25 * (rr_t[:, 1] + rb_t[:, 1])) - ppb_t[:, 0]
                term = wgt[None, :] * (rr_t[:, :-1] * vert["fzp"][None, 1:L] + rr_t[:, 1:] * vert["fzm"][None, 1:L])
                ppi = np.concatenate([ppi0[:, None], ppi0[:, None] - np.cumsum(term, axis=1)], axis=1)
                pp_t = 0.2 * ppi + 0.8 * pp_t
        return pp_t, tt_t

    nlat_t = 4097
    lat_t = np.linspace(-0.5 * PII, 0.5 * PII, nlat_t)
    pp_t, tt_t = column_solve(lat_t)
    fpos = (latC + 0.5 * PII) / (PII / (nlat_t - 1))
    i0 = np.clip(np.floor(fpos).astype(np.int64), 0, nlat_t - 2)
    wt = (fpos - i0)[:, None]
    pp = (1.0 - wt) * pp_t[i0] + wt * pp_t[i0 + 1]
    tt = (1.0 - wt) * tt_t[i0] + wt * tt_t[i0 + 1]
    ztemp = 0.5 * (zgrid[:, 1:] + zgrid[:, :-1])
    ppb = p0 * np.exp(-GRAVITY * ztemp / (RGAS * t0b))
    pb = (ppb / p0) ** (RGAS / CP)
    rb = ppb / (RGAS * t0b * zz[:, :L])
    tb = t0b / pb
    rr = (pp / (RGAS * zz[:, :L]) - rb * (tt - t0b)) / tt
    full = lambda a: np.concatenate([a, np.zeros((a.shape[0], 1))], 1)
    exner = ((ppb + pp) / p0) ** (RGAS / CP)
    theta_m = tt / exner
    F["rho_base"], F["pressure_p"], F["rho_p"] = full(rb), full(pp), full(rr)
    theta_base = full(tb)
    F["exner"], F["theta_m"] = full(exner), full(theta_m)
    F["rtheta_p"] = full(theta_m * rr + rb * (theta_m - tb))
    F["rho_zz"] = full(rb + rr)
    rho_zz_coupled = F["rho_zz"].copy()

    # ---- zonal wind on edges (:530-596)
    v1 = resolve_ids(v["verticesOnEdge"][:, 0], nV, policy)
    v2 = resolve_ids(v["verticesOnEdge"][:, 1], nV, policy)
    latV_p = np.concatenate([v["latVertex"], [0.0]])
    lat1, lat2 = latV_p[v1], latV_p[v2]
    flux = (0.5 * (lat2 - lat1) - 0.125 * (np.sin(4.0 * lat2) - np.sin(4.0 * lat1))) * SPHERE_RADIUS / v["dvEdge"]
    pf = pad(ppb + pp)
    etavs = (0.5 * (pf[c1] + pf[c2]) / p0 - 0.252) * PII / 2.0
    u = np.zeros((nE, L1))
    u[:, :L] = u0 * flux[:, None] * np.maximum(np.cos(etavs), 0.0) ** 1.5
    F["u"] = u
    rz_p = pad(F["rho_zz"])
    F["ru"] = 0.5 * (rz_p[c1] + rz_p[c2]) * u

    # ---- zb (:616-665), zb3 = 0
    z_edge = 0.5 * (zg_p[c1, :] + zg_p[c2, :])
    area_p = np.concatenate([v["areaCell"], [1.0]])
    zb = np.zeros((nE, L1, 2))
    zb[:, :L, 0] = ((z_edge - zg_p[c1]) * (v["dvEdge"] / area_p[c1])[:, None])[:, :L]
    zb[:, :L, 1] = ((z_edge - zg_p[c2]) * (v["dvEdge"] / area_p[c2])[:, None])[:, :L]
    zb3 = np.zeros((nE, L1, 2))
    if m5:   # non-degenerate 3rd-order metric terms
        zb3[:, :L, :] = 0.1 * zb[:, :L, :] * dr["zb3_factor"]

    # ---- rw / w (:681-704): rw accumulates on a zero field
    fzm, fzp = vert["fzm"], vert["fzp"]
    zz_p = pad(zz)
    rw = np.zeros((nC + 1, L1))
    fl = np.zeros((nE, L1))
    fl[:, 1:L] = fzm[None, 1:L] * F["ru"][:, 1:L] + fzp[None, 1:L] * F["ru"][:, 0:L - 1]
    zzf = np.zeros((nC + 1, L1))
    zzf[:, 1:L] = fzm[None, 1:L] * zz_p[:, 1:L] + fzp[None, 1:L] * zz_p[:, 0:L - 1]
    np.add.at(rw, c2, zzf[c2] * zb[:, :, 1] * fl)
    np.add.at(rw, c1, -zzf[c1] * zb[:, :, 0] * fl)
    rw = rw[:nC]
    w = np.zeros((nC, L1))
    w[:, 1:L] = rw[:, 1:L] / (fzp[None, 1:L] * F["rho_zz"][:, 0:L - 1] + fzm[None, 1:L] * F["rho_zz"][:, 1:L])
    F["rw"], F["w"] = rw, w

    if keep_jw:      # what init_atm_case_jw itself leaves in the regions (the device form, mpasb200_init_atm_case_jw, is checked against this)
        jw_snapshot = {k: F[k].copy() for k in ("zgrid", "zz", "zxu", "rho_base", "pressure_p", "rho_p", "exner", "theta_m", "rtheta_p",
                                                    "rho_zz", "u", "ru", "rw", "w")}
        jw_snapshot.update(theta_base=theta_base.copy(), zb=zb.copy())

    # ================= atm_core_init chain (atm_core.rg:22-42) =================
    sg = core_init.atm_compute_signs(mesh, policy, zb=zb, zb3=zb3, nlev1=L1)
    _, zb3c = core_init.atm_couple_coef_3rd_order(0.25, None, sg["zb3_cell"])
    F["zb_cell"], F["zb3_cell"] = sg["zb_cell"], zb3c

    # atm_init_coupled_diagnostics (dynamics_tasks.rg:651-725)
    eoc = resolve_ids(v["edgesOnCell"], nE, policy)
    nEoC = v["nEdgesOnCell"]
    F["rho_zz"][:, :L] = (F["rho_zz"][:, :L] * zz[:, :L]) / zz[:, :L]   # stored uncoupled (rho), coupled here (:674)
    rz_p = pad(F["rho_zz"])
    F["ru"][:, :L] = (0.5 * u * (rz_p[c1] + rz_p[c2]))[:, :L]
    ru_p = pad(F["ru"])
    rwn = np.zeros((nC, L1))
    rzf = np.zeros((nC, L1))
    rzf[:, 1:L] = fzp[None, 1:L] * F["rho_zz"][:, 0:L - 1] + fzm[None, 1:L] * F["rho_zz"][:, 1:L]
    zf = np.zeros((nC, L1))
    zf[:, 1:L] = fzp[None, 1:L] * zz[:, 0:L - 1] + fzm[None, 1:L] * zz[:, 1:L]
    rwn[:, 1:L] = (F["w"] * rzf * zf)[:, 1:L]
    for i in range(MAX_EDGES):
        use = (i < nEoC)[:, None]
        e = eoc[:, i]
        fx = np.zeros((nC, L1))
        fx[:, 1:L] = fzm[None, 1:L] * ru_p[e][:, 1:L] + fzp[None, 1:L] * ru_p[e][:, 0:L - 1]
        term = S["edgesOnCellSign"][:, i][:, None] * (F["zb_cell"][:, :, i] + np.copysign(1.0, fx) * F["zb3_cell"][:, :, i]) * fx * zf
        rwn[:, 1:L] -= np.where(use, term, 0.0)[:, 1:L]
    F["rw"] = rwn
    rho_base = F["rho_base"]
    F["rho_p"] = np.where(np.arange(L1)[None, :] < L, F["rho_zz"] - rho_base, 0.0)
    rtb = theta_base * rho_base
    F["rtheta_base"] = rtb
    F["rtheta_p"] = np.where(np.arange(L1)[None, :] < L, F["theta_m"] * F["rho_p"] + rho_base * (F["theta_m"] - theta_base), 0.0)
    rcv = RGAS / (CP - RGAS)
    with np.errstate(invalid="ignore"):
        ex = np.power(np.maximum(zz * (RGAS / 100000) * (F["rtheta_p"] + rtb), 0.0), rcv)
        exb = np.power(np.maximum(zz * (RGAS / 100000) * rtb, 0.0), rcv)
    lev = np.arange(L1)[None, :] < L
    F["exner"] = np.where(lev, ex, 0.0)
    F["exner_base"] = np.where(lev, exb, 0.0)
    F["pressure_p"] = np.where(lev, zz * RGAS * (F["exner"] * F["rtheta_p"] + rtb * (F["exner"] - F["exner_base"])), 0.0)

    F["dss"] = core_init.atm_compute_damping_coefs(zgrid, v["meshDensity"], L)

    # ---- fields the reference never writes (M1: zero;  M5: deterministic non-degenerate values)
    if m5:
        F.update(m5_fields(dr["modes"], [mesh_unit.v[k] for k in ("xCell", "yCell", "zCell")],
                           [mesh_unit.v[k] for k in ("xEdge", "yEdge", "zEdge")], F["theta_m"], F["rho_zz"], c1, c2))
    else:
        for k in ("h", "rt_diabatic_tend", "t_init", "tend_rho_physics", "tend_rtheta_physics", "theta_m_save"):
            F[k] = np.zeros((nC, L1))
        for k in ("rho_edge", "tend_ru_physics", "u_tend", "tend_ru", "cqu"):
            F[k] = np.zeros((nE, L1))
    coeffs, deriv_two = st.extras["coeffs_reconstruct"], st.extras["deriv_two"]
    st.extras = dict(coeffs_reconstruct=coeffs, theta_base=theta_base, zb=zb, zb3=zb3, deriv_two=deriv_two)
    if keep_jw:
        st.extras["jw"] = jw_snapshot
    F["theta_base"] = theta_base
    F["uReconstructZonal"], F["uReconstructMeridional"] = core_init.mpas_reconstruct_2d(mesh, policy, F["u"], coeffs, L)
    # v is produced by atm_compute_solve_diagnostics(rk_step=-1) at init (atm_core.rg:31): that is a
    # hot-path task and is run through the library (or the oracle) by the caller.  For callers that
    # want a complete host image without it, reconstruct here (dynamics_tasks.rg:431-438, loop from i=1).
    if diag_on_host:
        eoe = resolve_ids(v["edgesOnEdge"], nE, policy)
        u_p = pad(F["u"])
        vv = np.zeros((nE, L1))
        for i in range(1, MAX_EDGES2):
            use = (i < v["nEdgesOnEdge"])[:, None]
            vv[:, :L] += np.where(use, v["weightsOnEdge"][:, i][:, None] * u_p[eoe[:, i]][:, :L], 0.0)
        F["v"] = vv
    for k in list(F):
        F[k] = np.ascontiguousarray(F[k], dtype=np.float64)
    return st


# ---- the same state built on the device, one handle per partition -----------------------------------------------------
def jw_inputs(mesh_unit: Mesh, st: HostState, draws: Dict[str, np.ndarray], lm=None) -> Dict[str, np.ndarray]:
    """Per-entity inputs of init_on_device for the rows one handle holds (``lm`` a partition.LocalMesh, None = the whole
    mesh): latCell / areaCell / meshDensity / latVertex of the scaled mesh, the unit-sphere coordinates of cells and edges
    (rows x, y, z), the zb3 factors of the edges, and the _smooth mode sets (global)."""
    v, u = st.mesh.v, mesh_unit.v
    c, e, vx = (slice(None), slice(None), slice(None)) if lm is None else (lm.cells, lm.edges, lm.vertices)
    return dict(latCell=v["latCell"][c], areaCell=v["areaCell"][c], meshDensity=v["meshDensity"][c], latVertex=v["latVertex"][vx],
                cell_xyz=np.stack([u[k][c] for k in ("xCell", "yCell", "zCell")]),
                edge_xyz=np.stack([u[k][e] for k in ("xEdge", "yEdge", "zEdge")]),
                zb3_factor=np.ascontiguousarray(draws["zb3_factor"][e]), modes=draws["modes"])


def init_on_device(dyn, static: Dict[str, np.ndarray], jw: Dict[str, np.ndarray], vert: Dict[str, np.ndarray]) -> None:
    """make_state(m5=True)'s 3-D fields built on a handle whose mesh (``static``, from make_static or a static shard) is
    uploaded: init_atm_case_jw, rho_zz *= zz, zb3, zb_cell, the level-0 zb3 coupling, atm_init_coupled_diagnostics,
    atm_compute_damping_coefs, mpas_reconstruct_2d, then the M5 fields of the rows held (from the device theta_m and
    coupled rho_zz).  CORRECTED index policy.

    On a local mesh every owned entity comes out right; ghost ring 2 and the edges to cells that are not held do not
    (their stencils leave the rows held) until parallel.INIT_EXCHANGE runs.  atm_compute_solve_diagnostics(-1) is the
    caller's, as with uploaded inputs."""
    assert dyn.cfg.index_policy == CORRECTED, "init_on_device builds the CORRECTED reading"
    L = dyn.dims.nVertLevels
    dyn.init_atm_case_jw(jw["latCell"], jw["areaCell"], jw["latVertex"])
    with np.errstate(all="ignore"):          # rows outside the stencil's reach may hold inf / NaN until the exchange
        dyn.upload_field("rho_zz", dyn.download_field("rho_zz") * dyn.download_field("zz"))   # atm_init_coupled_diagnostics divides by zz
        zb = dyn.download_field("zb")
        zb3 = np.zeros_like(zb)
        zb3[:, :L, :] = 0.1 * zb[:, :L, :] * jw["zb3_factor"]
    dyn.upload_field("zb3", zb3)
    dyn.atm_compute_zb_cell()
    dyn.atm_couple_coef_3rd_order(0.25)
    dyn.atm_init_coupled_diagnostics()
    dyn.atm_compute_damping_coefs(jw["meshDensity"])
    dyn.mpas_reconstruct_2d(False, True)
    nC = dyn.dims.nCells
    c1, c2 = (resolve_ids(static["cellsOnEdge"][:, i], nC, CORRECTED) for i in (0, 1))
    with np.errstate(all="ignore"):
        F = m5_fields(jw["modes"], list(jw["cell_xyz"]), list(jw["edge_xyz"]), dyn.download_field("theta_m"),
                      dyn.download_field("rho_zz"), c1, c2)
    dyn.upload_state(F, {k: vert[k] for k in ("u_init", "v_init", "cofrz")})
