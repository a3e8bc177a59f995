"""A deterministic irregular Voronoi test mesh with cells of 4 to 10 sides, and an MPAS regional mask layout on it.

Every other test mesh has only pentagons and hexagons, so code that depends on a cell's degree (the switch over
n = 5, 6, 7 and the generic loop of k_rec_cell2, shared-memory rows of width maxEdges, the nEdgesOnEdge loop, the
maxEdges - 1 cap of atm_adv_coef_compression) and code that depends on the regional masks (bdyMaskCell beyond
nRelaxZone, specZoneMaskCell / specZoneMaskEdge, isShared) would otherwise never see other inputs.

The mesh starts from the generators of the 642-cell icosahedral mesh.  Around 7 well separated generators, every other
generator closer than 1.6 h (h = mean spacing) is removed and a ring of k points is put at radius ~h, which makes the
centre cell a k-gon.  All points are then jittered by 0.02 h.
"""
import functools

import numpy as np

from mpas_regent_b200 import icosa
from mpas_regent_b200.mesh import MAX_EDGES

RING_DEGREES = (4, 7, 8, 9, 10, 7, 8)
SEED = 3
N_RELAX_ZONE = 5          # MpasConfig.nRelaxZone of _abi.default_config


def generators():
    p, f = icosa._icosahedron()
    for _ in range(icosa.level_for_cells(642)):
        p, f = icosa._subdivide(p, f)
    h = icosa._arc(p[f[:, 0]], p[f[:, 1]]).mean()
    rng = np.random.default_rng(SEED)
    keep = np.ones(len(p), bool)
    ring, centres = [], []
    for k in RING_DEGREES:
        while True:                                     # a centre far from the earlier ones
            c = int(rng.integers(len(p)))
            if keep[c] and all(icosa._arc(p[c], p[o]) > 5 * h for o in centres):
                break
        centres.append(c)
        d = icosa._arc(p, p[c][None, :])
        keep &= ~((d > 0) & (d < 1.6 * h))
        n = p[c]
        t1 = np.cross(n, [0.3, 0.5, 0.8]); t1 /= np.linalg.norm(t1)
        t2 = np.cross(n, t1)
        r = h * (1.0 + 0.15 * max(0, k - 6))
        a = 2 * np.pi * np.arange(k) / k
        ring.append(np.cos(r) * n + np.sin(r) * (np.cos(a)[:, None] * t1 + np.sin(a)[:, None] * t2))
    pts = np.concatenate([p[keep]] + ring)
    pts += 0.02 * h * rng.standard_normal(pts.shape)
    return pts / np.linalg.norm(pts, axis=1, keepdims=True)


def adv_list_uncapped(mesh):
    """the last index of the list of distinct cells atm_adv_coef_compression gathers for each edge, before its
    maxEdges - 1 cap: both cells of the edge, every other neighbour of either, the two shared neighbours once."""
    n = mesh.v["nEdgesOnCell"].astype(np.int64)
    coe = mesh.v["cellsOnEdge"].astype(np.int64) - 1
    return n[coe[:, 0]] + n[coe[:, 1]] - 3


@functools.lru_cache(maxsize=None)
def irregular_mesh():
    m = icosa.make_voronoi_mesh(generators(), "irregular646")
    v = m.v
    deg = v["nEdgesOnCell"]
    assert set(range(4, 11)) <= set(np.unique(deg).tolist()), np.bincount(deg)
    assert v["nEdgesOnEdge"].max() >= 14
    assert (adv_list_uncapped(m) > MAX_EDGES - 1).any()
    return m


@functools.lru_cache(maxsize=None)
def regional_masks():
    """MPAS's regional layout around one side of the sphere: bdyMaskCell 1..5 are relaxation bands, 6..7 the specified
    zone (specZoneMaskCell = 1, specZoneMaskEdge = 1 on every edge of a specified cell), isShared on band 7.  The bands
    are rings of cells in graph distance from the 40 cells farthest from every irregular cell (degree other than 5 and
    6), so that those stay in the interior or the relaxation zone, where the code they are there to reach runs."""
    m = irregular_mesh()
    v = m.v
    nC = m.nCells
    deg = v["nEdgesOnCell"]
    coc = v["cellsOnCell"].astype(np.int64) - 1
    slot = np.arange(MAX_EDGES)[None, :] < deg[:, None]
    p = np.stack([v["xCell"], v["yCell"], v["zCell"]], 1)
    odd = np.flatnonzero((deg != 5) & (deg != 6))
    far = p @ p[odd].T                                   # cos of the distance to every irregular cell
    seed = np.argsort(far.max(axis=1))[:40]               # the 40 cells farthest from all of them
    dist = np.full(nC, -1)
    dist[seed] = 0
    front = seed
    while (dist < 0).any():                               # breadth-first rings of cells
        nb = coc[front][slot[front]]
        nb = np.unique(nb[dist[nb] < 0])
        dist[nb] = dist[front[0]] + 1
        front = nb
    bdy = np.where(dist <= 6, 7 - np.minimum(dist, 6), 0).astype(np.int32)   # 7, 6 specified; 5..1 relaxation; 0 interior
    spec_cell = (bdy >= 6).astype(np.float64)
    coe = v["cellsOnEdge"].astype(np.int64) - 1
    spec_edge = np.maximum(spec_cell[coe[:, 0]], spec_cell[coe[:, 1]])
    shared = (bdy == 7).astype(np.uint8)
    assert np.all(bdy[odd] <= N_RELAX_ZONE) and np.all(spec_cell[odd] == 0.0)
    for b in range(8):
        assert (bdy == b).any(), b
    return dict(bdyMaskCell=bdy, specZoneMaskCell=spec_cell, specZoneMaskEdge=spec_edge, isShared=shared)


def make_state(L, policy, masked=True, **kw):
    """init_jw.make_state on the irregular mesh, with the regional masks when ``masked``."""
    from mpas_regent_b200 import init_jw
    st = init_jw.make_state(irregular_mesh(), L, policy, **kw)
    if masked:
        st.static.update(regional_masks())
    return st
