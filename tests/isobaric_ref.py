"""numpy restatement of mpasb200_isobaric_diagnostics (the definition in include/mpas_b200.h), written from that text and
independent of k_isobaric's warp form: whole columns at a time, every level and slot in the order the definition gives.
The library is built with --fmad=false, so everything but the interpolation weight a (np.log against the device's log)
is the same IEEE arithmetic, and the NaN masks and the surface pressure agree bit for bit."""
import numpy as np

from mpas_regent_b200 import _abi
from mpas_regent_b200.mesh import resolve_ids

#: the fields of the mirror the diagnostics read
INPUTS = ("pressure_base", "pressure_p", "theta_m", "exner", "zgrid", "w", "u", "vorticity")


def _pad(a):
    return np.concatenate([a, np.zeros((1,) + a.shape[1:], a.dtype)])


def level_fields(f, static, L, policy=_abi.INDEX_CORRECTED):
    """per mass level k = 0..L-1 of every cell: p, T, z, wm, uzon, umer, zeta, each [nCells, L]"""
    nC, nE, nV = f["theta_m"].shape[0], f["u"].shape[0], f["vorticity"].shape[0]
    zg, w = f["zgrid"], f["w"]
    out = {"p": f["pressure_base"][:, :L] + f["pressure_p"][:, :L],
           "T": f["theta_m"][:, :L] * f["exner"][:, :L],
           "z": 0.5 * (zg[:, :L] + zg[:, 1:L + 1]),
           "wm": 0.5 * (w[:, :L] + w[:, 1:L + 1])}
    n = static["nEdgesOnCell"]
    eoc = resolve_ids(static["edgesOnCell"], nE, policy)
    voc = resolve_ids(static["verticesOnCell"], nV, policy)
    kite = np.asarray(static["kiteForCell"])
    cf = np.asarray(static["coeffs_reconstruct"]).reshape(nC, -1, 3)
    u, vort = _pad(f["u"][:, :L]), _pad(f["vorticity"][:, :L])
    areas = _pad(np.asarray(static["kiteAreasOnVertex"]))
    # mpas_reconstruct_2d (dynamics_tasks.rg:1894-1948), on_a_sphere: sums from 0.0 over the cell's slots in order
    ux, uy, uz = np.zeros((nC, L)), np.zeros((nC, L)), np.zeros((nC, L))
    num, den = np.zeros((nC, L)), np.zeros(nC)
    for i in range(eoc.shape[1]):
        use = i < n
        ue = u[eoc[:, i]]
        ux = np.where(use[:, None], ux + cf[:, i, 0][:, None] * ue, ux)
        uy = np.where(use[:, None], uy + cf[:, i, 1][:, None] * ue, uy)
        uz = np.where(use[:, None], uz + cf[:, i, 2][:, None] * ue, uz)
        a = areas[voc[:, i], np.where(use, kite[:, i], 0)]
        num = np.where(use[:, None], num + a[:, None] * vort[voc[:, i]], num)
        den = np.where(use, den + a, den)
    lat, lon = np.asarray(static["latCell"]), np.asarray(static["lonCell"])
    clat, slat, clon, slon = (x[:, None] for x in (np.cos(lat), np.sin(lat), np.cos(lon), np.sin(lon)))
    out["uzon"] = -ux * slon + uy * clon
    out["umer"] = -(ux * clon + uy * slon) * slat + uz * clat
    with np.errstate(divide="ignore", invalid="ignore"):
        out["zeta"] = num / den[:, None]
    return out


#: the six interpolated values per level, in the row order of the C entry and under the names of Dynamics.isobaric_diagnostics
ROW = (("temperature", "T"), ("height", "z"), ("uzonal", "uzon"), ("umeridional", "umer"), ("w", "wm"), ("vorticity", "zeta"))


def isobaric_from_levels(lev, zgrid0, plev):
    """the surface pressure and the six fields on the pressure surfaces plev (Pa) from level_fields' columns"""
    p, z = lev["p"], lev["z"]
    nC, L = p.shape
    r = np.arange(nC)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        out = {"surface_pressure": p[:, 0] + (zgrid0 - z[:, 0]) * ((p[:, 1] - p[:, 0]) / (z[:, 1] - z[:, 0]))}
        for name, _ in ROW:
            out[name] = np.empty((nC, len(plev)))
        for j, P in enumerate(plev):
            P = float(P)
            bracket = (p[:, :L - 1] >= P) & (P >= p[:, 1:L])        # comparisons with NaN are false
            has = bracket.any(axis=1)
            k = np.argmax(bracket, axis=1)                           # the smallest such k
            pk, pk1 = p[r, k], p[r, k + 1]
            a = np.where(pk == pk1, 1.0, (np.log(P) - np.log(pk1)) / (np.log(pk) - np.log(pk1)))
            for name, key in ROW:
                fk, fk1 = lev[key][r, k], lev[key][r, k + 1]
                out[name][:, j] = np.where(has, fk1 + a * (fk - fk1), np.nan)
    return out


def isobaric_ref(f, static, L, plev, policy=_abi.INDEX_CORRECTED):
    """the diagnostics of every cell: f = full fields [n, L+1] of INPUTS (downloaded or host-built), static = the mesh
    arrays as uploaded"""
    return isobaric_from_levels(level_fields(f, static, L, policy), f["zgrid"][:, 0], plev)
