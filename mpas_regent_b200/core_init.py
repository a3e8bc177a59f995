"""Host-side (numpy) producers of the hot path's static inputs: the one-time setup tasks
``atm_core_init`` runs before the first step (reference: atm_core.rg:22-42).

These stay on the host in the drop-in design (they are CPU Regent tasks that run once);
the GPU library only consumes their outputs through ``mpasb200_upload_mesh`` /
``mpasb200_upload_field``.  They are vectorised re-statements that keep the reference's
quirks (SURVEY.md 8a Q-list), so that the harness feeds the kernels what the reference's
regions would hold.  tests/test_core_init.py checks them two ways: geometric properties under the
CORRECTED policy, and -- for ``atm_compute_signs`` and ``atm_couple_coef_3rd_order`` -- a literal loop-by-loop
restatement of the reference text under BOTH index policies on the bundled x1.2562 mesh (the oracle itself
has no init-chain functions: it starts from the uploaded static data).

Index policy: ``raw`` ids are the stored 1-based values.  ``R(raw, n)`` resolves them to
array indices with a zero pad entity at index n (mesh.resolve_ids).  Under LITERAL the
reference's raw-vs-0-based comparisons (Q33) are kept; under CORRECTED both the indexing
and those comparisons are corrected.
"""
from __future__ import annotations

import numpy as np

from .mesh import CORRECTED, FIFTEEN, LITERAL, MAX_EDGES, VERTEX_DEGREE, Mesh, resolve_ids


def _padrows(a: np.ndarray) -> np.ndarray:
    """append one zero row (the pad entity)."""
    return np.concatenate([a, np.zeros((1,) + a.shape[1:], dtype=a.dtype)], axis=0)


def _cmp_id(policy: int) -> int:
    """what a 0-based loop index must be offset by to compare equal with a stored id."""
    return 0 if policy == LITERAL else 1


def atm_compute_signs(mesh: Mesh, policy: int, zb: np.ndarray = None, zb3: np.ndarray = None, nlev1: int = 0):
    """dynamics_tasks.rg:46-130.  Returns dict with edgesOnVertexSign, edgesOnCellSign,
    kiteForCell and (if zb/zb3 given, shape [nEdges, nlev1, 2]) zb_cell / zb3_cell of
    shape [nCells, nlev1, maxEdges]."""
    v = mesh.v
    nC, nE, nV = mesh.nCells, mesh.nEdges, mesh.nVertices
    off = _cmp_id(policy)
    out = {}
    # -- edgesOnVertexSign (:60-72)
    eov = v["edgesOnVertex"]
    voe_p = _padrows(v["verticesOnEdge"])
    e_idx = resolve_ids(eov, nE, policy)
    sign = np.where(voe_p[e_idx, 1] == (np.arange(nV)[:, None] + off), 1.0, -1.0)
    out["edgesOnVertexSign"] = np.where(eov <= nE, sign, 0.0)
    # -- edgesOnCellSign (:74-86)
    eoc = v["edgesOnCell"]
    nEoC = v["nEdgesOnCell"]
    slot = np.arange(MAX_EDGES)[None, :] < nEoC[:, None]
    coe_p = _padrows(v["cellsOnEdge"])
    ce_idx = resolve_ids(eoc, nE, policy)
    is_c1 = coe_p[ce_idx, 0] == (np.arange(nC)[:, None] + off)
    s = np.where(eoc <= nE, np.where(is_c1, 1.0, -1.0), 0.0)
    out["edgesOnCellSign"] = np.where(slot, s, 0.0)
    # -- zb_cell / zb3_cell (:88-110): levels 0..nVertLevels (cell_range_2d)
    if zb is not None:
        zb_p, zb3_p = _padrows(zb), _padrows(zb3)
        zbc = np.zeros((nC, nlev1, MAX_EDGES))
        zb3c = np.zeros((nC, nlev1, MAX_EDGES))
        for i in range(MAX_EDGES):
            use = slot[:, i] & (eoc[:, i] <= nE)
            side = np.where(is_c1[:, i], 0, 1)
            e = ce_idx[:, i]
            zsel = np.take_along_axis(zb_p[e], side[:, None, None], axis=2)[:, :, 0]
            z3sel = np.take_along_axis(zb3_p[e], side[:, None, None], axis=2)[:, :, 0]
            zbc[:, :, i] = np.where(use[:, None], zsel, 0.0)
            zb3c[:, :, i] = np.where(use[:, None], z3sel, 0.0)
        out["zb_cell"], out["zb3_cell"] = zbc, zb3c
    # -- kiteForCell (:113-129): j runs 1..vertexDegree-1 only
    voc = v["verticesOnCell"]
    cov_p = _padrows(v["cellsOnVertex"])
    v_idx = resolve_ids(voc, nV, policy)
    kite = np.zeros((nC, MAX_EDGES), dtype=np.int32)
    me = np.arange(nC)[:, None] + off
    for j in range(VERTEX_DEGREE - 1, 0, -1):      # reverse so the smallest matching j wins (break)
        kite = np.where(cov_p[v_idx, j] == me, j, kite)
    kite = np.where(voc <= nV, kite, 1)
    out["kiteForCell"] = np.where(slot, kite, 0).astype(np.int32)
    return out


def atm_adv_coef_compression(mesh: Mesh, policy: int, deriv_two: np.ndarray = None):
    """dynamics_tasks.rg:133-269.  deriv_two: [nEdges, 2*FIFTEEN] (never written upstream;
    None = zeros).  Returns nAdvCellsForEdge, advCellsForEdge (raw ids), adv_coefs, adv_coefs_3rd.

    Kept quirks: ``n`` is the index of the last list element, the duplicate search and every
    ``for j = 0, n`` loop are exclusive of it, the list is capped at maxEdges-1 (:175), and
    nAdvCellsForEdge = n, so the last listed cell never enters the flux sum."""
    v = mesh.v
    nC, nE = mesh.nCells, mesh.nEdges
    if deriv_two is None:
        deriv_two = np.zeros((nE, 2 * FIFTEEN))
    coc_p = _padrows(v["cellsOnCell"])
    nEoC_p = _padrows(v["nEdgesOnCell"][:, None])[:, 0]
    cell1, cell2 = v["cellsOnEdge"][:, 0].astype(np.int64), v["cellsOnEdge"][:, 1].astype(np.int64)
    i1, i2 = resolve_ids(cell1, nC, policy), resolve_ids(cell2, nC, policy)
    n1, n2 = nEoC_p[i1], nEoC_p[i2]
    W = 2 + 2 * MAX_EDGES
    lst = np.zeros((nE, W), dtype=np.int64)
    lst[:, 0], lst[:, 1] = cell1, cell2
    n = np.ones(nE, dtype=np.int64)
    rows = np.arange(nE)
    for i in range(MAX_EDGES):
        cand = coc_p[i1, i].astype(np.int64)
        add = (i < n1) & (cand != cell2)
        n = n + add
        lst[rows[add], n[add]] = cand[add]
    cols = np.arange(W)[None, :]
    for i in range(MAX_EDGES):
        cand = coc_p[i2, i].astype(np.int64)
        dup = ((lst == cand[:, None]) & (cols < n[:, None])).any(axis=1)
        add = (i < n2) & ~dup & (n < MAX_EDGES - 1)
        n = n + add
        lst[rows[add], n[add]] = cand[add]
    nAdv = n.astype(np.int32)
    adv = np.zeros((nE, FIFTEEN), dtype=np.int32)
    valid = np.arange(FIFTEEN)[None, :] < n[:, None]
    adv[valid] = lst[:, :FIFTEEN][valid]

    def j_in(target):
        """last j < n with cell_list[j] == target, else 0 (:195-200)."""
        hit = (lst == target[:, None]) & (cols < n[:, None])
        idx = np.where(hit, cols, -1).max(axis=1)
        return np.where(idx < 0, 0, idx)

    a = np.zeros((nE, W))
    a3 = np.zeros((nE, W))

    def acc(j, val):
        np.add.at(a, (rows, j), val)
        np.add.at(a3, (rows, j), val)

    def d2(idx):
        """deriv_two : double[2*FIFTEEN]; the reference indexes it iCell*FIFTEEN + side (:211,234),
        which runs past the array for iCell >= 2 -- memory model: an out-of-range read is 0."""
        return deriv_two[:, idx] if idx < 2 * FIFTEEN else np.zeros(nE)

    acc(j_in(cell1), deriv_two[:, 0])
    for i in range(MAX_EDGES):
        use = i < n1
        acc(j_in(coc_p[i1, i].astype(np.int64)), np.where(use, d2(i * FIFTEEN + 0), 0.0))
    acc(j_in(cell2), deriv_two[:, 1])
    for i in range(MAX_EDGES):
        use = i < n2
        acc(j_in(coc_p[i2, i].astype(np.int64)), np.where(use, d2(i * FIFTEEN + 1), 0.0))
    dc, dv = v["dcEdge"], v["dvEdge"]   # already scaled to the sphere (init_atm_cases.rg:104-111)
    inrange = cols < n[:, None]
    scale = (-1.0 * (dc * dc))[:, None]
    a = np.where(inrange, scale * a / 12, a)
    a3 = np.where(inrange, scale * a3 / 12, a3)
    np.add.at(a, (rows, j_in(cell1)), 0.5)
    np.add.at(a, (rows, j_in(cell2)), 0.5)
    a = np.where(inrange, a * dv[:, None], a)
    a3 = np.where(inrange, a3 * dv[:, None], a3)
    return dict(nAdvCellsForEdge=nAdv, advCellsForEdge=adv,
                adv_coefs=np.ascontiguousarray(a[:, :FIFTEEN]), adv_coefs_3rd=np.ascontiguousarray(a3[:, :FIFTEEN]))


def atm_couple_coef_3rd_order(coef: float, adv_coefs_3rd: np.ndarray, zb3_cell: np.ndarray):
    """dynamics_tasks.rg:303-325: adv_coefs_3rd *= coef on every edge; zb3_cell *= coef at LEVEL 0 only.  Either may be
    None (the mesh-only half and the 3-D half run apart when the level-0 data is built without any 3-D field)."""
    if adv_coefs_3rd is not None:
        adv_coefs_3rd *= coef
    if zb3_cell is not None:
        zb3_cell[:, 0, :] *= coef
    return adv_coefs_3rd, zb3_cell


def atm_compute_mesh_scaling(mesh: Mesh, policy: int, scale_with_mesh: bool = True):
    """dynamics_tasks.rg:595-646 (meshDensity read through cellOne/cellTwo = cellsOnEdge)."""
    v = mesh.v
    nC = mesh.nCells
    md = np.concatenate([v["meshDensity"], [0.0]])
    c1 = resolve_ids(v["cellsOnEdge"][:, 0], nC, policy)
    c2 = resolve_ids(v["cellsOnEdge"][:, 1], nC, policy)
    if not scale_with_mesh:
        one = np.ones(mesh.nEdges)
        return dict(meshScalingDel2=one, meshScalingDel4=one.copy())
    with np.errstate(divide="ignore"):
        m = (md[c1] + md[c2]) / 2.0
        return dict(meshScalingDel2=1.0 / np.power(m, 0.25), meshScalingDel4=1.0 / np.power(m, 0.75))


def atm_compute_damping_coefs(zgrid: np.ndarray, meshDensity: np.ndarray, nVertLevels: int,
                              config_zd: float = 22000.0, config_xnutr: float = 0.2):
    """dynamics_tasks.rg:274-300.  zgrid [nCells, L+1] -> dss [nCells, L+1] (level L untouched = 0)."""
    L = nVertLevels
    pii = np.arccos(-1.0)
    dss = np.zeros_like(zgrid)
    zt = zgrid[:, L][:, None]
    z = 0.5 * (zgrid[:, :L] + zgrid[:, 1:L + 1])
    with np.errstate(invalid="ignore", divide="ignore"):
        val = config_xnutr * np.sin(0.5 * pii * (z - config_zd) / (zt - config_zd)) ** 2.0
        val = val / np.power(meshDensity[:, None], 0.25)
    dss[:, :L] = np.where(z > config_zd, val, 0.0)
    return dss


def mpas_reconstruct_2d(mesh: Mesh, policy: int, u: np.ndarray, coeffs_reconstruct: np.ndarray, nVertLevels: int):
    """dynamics_tasks.rg:1894-1948 with on_a_sphere = true.  u [nEdges, L+1];
    coeffs_reconstruct [nCells, maxEdges, 3] (never written upstream)."""
    v = mesh.v
    nC, nE, L = mesh.nCells, mesh.nEdges, nVertLevels
    u_p = _padrows(u)
    eoc = resolve_ids(v["edgesOnCell"], nE, policy)
    X = np.zeros((nC, L + 1)); Y = np.zeros((nC, L + 1)); Z = np.zeros((nC, L + 1))
    for i in range(MAX_EDGES):
        use = (i < v["nEdgesOnCell"])[:, None]
        ue = u_p[eoc[:, i]][:, :L]
        X[:, :L] += np.where(use, coeffs_reconstruct[:, i, 0][:, None] * ue, 0.0)
        Y[:, :L] += np.where(use, coeffs_reconstruct[:, i, 1][:, None] * ue, 0.0)
        Z[:, :L] += np.where(use, coeffs_reconstruct[:, i, 2][:, None] * ue, 0.0)
    clat, slat = np.cos(v["latCell"])[:, None], np.sin(v["latCell"])[:, None]
    clon, slon = np.cos(v["lonCell"])[:, None], np.sin(v["lonCell"])[:, None]
    zonal = np.zeros((nC, L + 1)); merid = np.zeros((nC, L + 1))
    zonal[:, :L] = (-X * slon + Y * clon)[:, :L]
    merid[:, :L] = (-(X * clon + Y * slon) * slat + Z * clat)[:, :L]
    return zonal, merid
