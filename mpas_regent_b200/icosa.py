"""Synthetic icosahedral Voronoi meshes of 10*4**n + 2 cells (BASELINE.json configs 2-5), and Voronoi meshes of
arbitrary generators on the sphere.

Deterministic and seedless: recursive bisection of the icosahedron gives the Delaunay
triangulation (cells = triangulation points, Voronoi vertices = triangle circumcentres,
nEdges = 3n-6, nVertices = 2n-4, 12 pentagons).  ``make_voronoi_mesh`` takes the triangulation
from the convex hull instead, so its cells may have anywhere from 3 to MAX_EDGES sides.  The output carries the same 38 variables,
dimensions and conventions as the bundled ``x1.2562.grid.nc`` that ``load_mesh`` reads
(reference: mesh_loading/mesh_loading.rg:123-201): 1-based ids, unit sphere, counter-
clockwise ``edgesOnCell``/``verticesOnCell``/``cellsOnCell`` with edge i joining vertex i and
vertex i+1, ``verticesOnEdge`` ordered along k x n, TRiSK ``edgesOnEdge``/``weightsOnEdge``.
Those conventions were checked against the bundled file (tests/test_mesh.py).

Everything is vectorised numpy; x1.655362 takes a few seconds.
"""
from __future__ import annotations

import numpy as np

from .mesh import MAX_EDGES, MAX_EDGES2, Mesh

CELLS_FOR_LEVEL = {n: 10 * 4 ** n + 2 for n in range(0, 11)}


def level_for_cells(n_cells: int) -> int:
    for lvl, n in CELLS_FOR_LEVEL.items():
        if n == n_cells:
            return lvl
    raise ValueError(f"{n_cells} is not 10*4^n+2")


def _icosahedron():
    t = (1.0 + np.sqrt(5.0)) / 2.0
    p = np.array([
        (-1, t, 0), (1, t, 0), (-1, -t, 0), (1, -t, 0),
        (0, -1, t), (0, 1, t), (0, -1, -t), (0, 1, -t),
        (t, 0, -1), (t, 0, 1), (-t, 0, -1), (-t, 0, 1)], dtype=np.float64)
    p /= np.linalg.norm(p, axis=1, keepdims=True)
    f = np.array([
        (0, 11, 5), (0, 5, 1), (0, 1, 7), (0, 7, 10), (0, 10, 11),
        (1, 5, 9), (5, 11, 4), (11, 10, 2), (10, 7, 6), (7, 1, 8),
        (3, 9, 4), (3, 4, 2), (3, 2, 6), (3, 6, 8), (3, 8, 9),
        (4, 9, 5), (2, 4, 11), (6, 2, 10), (8, 6, 7), (9, 8, 1)], dtype=np.int64)
    # make every face counter-clockwise seen from outside
    a, b, c = p[f[:, 0]], p[f[:, 1]], p[f[:, 2]]
    flip = np.einsum("ij,ij->i", np.cross(b - a, c - a), a + b + c) < 0
    f[flip] = f[flip][:, [0, 2, 1]]
    return p, f


def _subdivide(p, f):
    n = p.shape[0]
    a, b, c = f[:, 0], f[:, 1], f[:, 2]
    e = np.concatenate([np.stack([a, b], 1), np.stack([b, c], 1), np.stack([c, a], 1)])
    key = np.minimum(e[:, 0], e[:, 1]) * n + np.maximum(e[:, 0], e[:, 1])
    uk, inv = np.unique(key, return_inverse=True)
    lo, hi = uk // n, uk % n
    mid = p[lo] + p[hi]
    mid /= np.linalg.norm(mid, axis=1, keepdims=True)
    nf = f.shape[0]
    ab, bc, ca = n + inv[:nf], n + inv[nf:2 * nf], n + inv[2 * nf:]
    f2 = np.concatenate([
        np.stack([a, ab, ca], 1), np.stack([b, bc, ab], 1),
        np.stack([c, ca, bc], 1), np.stack([ab, bc, ca], 1)])
    return np.concatenate([p, mid]), f2


def _arc(a, b):
    """great-circle distance between unit vectors (numerically robust)."""
    return 2.0 * np.arcsin(np.clip(0.5 * np.linalg.norm(a - b, axis=-1), 0.0, 1.0))


def _tri_area(a, b, c):
    """signed area of the spherical triangle (unit sphere): positive when a, b, c run counter-clockwise seen from
    outside.  A kite of a cell whose Voronoi vertex lies outside its triangle (an obtuse Delaunay triangle) is the sum
    of one positive and one negative part; with unsigned parts the cell areas would no longer tile the sphere."""
    num = np.einsum("ij,ij->i", a, np.cross(b, c))
    den = 1.0 + np.einsum("ij,ij->i", a, b) + np.einsum("ij,ij->i", b, c) + np.einsum("ij,ij->i", c, a)
    return 2.0 * np.arctan2(num, den)


def _latlon(p):
    lat = np.arcsin(np.clip(p[:, 2], -1.0, 1.0))
    lon = np.arctan2(p[:, 1], p[:, 0])
    return lat, lon


def trisk_weights(nEdgesOnCell, edgesOnCell, verticesOnCell, cellsOnEdge, cellsOnVertex,
                  kiteAreasOnVertex, areaCell, dcEdge, dvEdge):
    """TRiSK edgesOnEdge / weightsOnEdge (Thuburn et al. JCP 2009) from 0-based connectivity.

    For edge e and each of its two cells: walk the cell's other edges counter-clockwise
    starting after e, accumulating the kite-area fractions R of the vertices passed;
    w = +-(1/2 - sum R) * dv(e') / dc(e), sign by which side of e' the cell is on and
    by which of e's cells is being walked.
    """
    nE = cellsOnEdge.shape[0]
    nEoE = np.zeros(nE, dtype=np.int32)
    eoe = np.zeros((nE, MAX_EDGES2), dtype=np.int32)  # 1-based on output; 0 = none
    woe = np.zeros((nE, MAX_EDGES2), dtype=np.float64)
    eids = np.arange(nE)
    for side in (0, 1):
        c = cellsOnEdge[:, side]
        nc = nEdgesOnCell[c]
        i0 = np.argmax(edgesOnCell[c, :] == eids[:, None], axis=1)
        sum_r = np.zeros(nE)
        sgn_side = 1.0 if side == 0 else -1.0
        for i in range(1, int(nEdgesOnCell.max())):
            act = i < nc
            j = (i0 + i) % nc
            vtx = verticesOnCell[c, j]
            kj = np.argmax(cellsOnVertex[vtx, :] == c[:, None], axis=1)
            r = kiteAreasOnVertex[vtx, kj] / areaCell[c]
            sum_r = sum_r + np.where(act, r, 0.0)
            e2 = edgesOnCell[c, j]
            s2 = np.where(cellsOnEdge[e2, 0] == c, 1.0, -1.0)
            w = sgn_side * (0.5 - sum_r) * dvEdge[e2] / dcEdge * s2
            slot = nEoE + (i - 1)
            rows = eids[act]
            eoe[rows, slot[act]] = e2[act] + 1
            woe[rows, slot[act]] = w[act]
        nEoE = nEoE + (nc - 1).astype(np.int32)
    return nEoE, eoe, woe


def make_icosahedral_mesh(n_cells: int) -> Mesh:
    lvl = level_for_cells(n_cells)
    p, f = _icosahedron()
    for _ in range(lvl):
        p, f = _subdivide(p, f)
    assert p.shape[0] == n_cells
    m = mesh_from_triangulation(p, f, f"x1.{n_cells}")
    deg = m.v["nEdgesOnCell"]
    assert deg.min() == 5 and deg.max() <= 6 and int((deg == 5).sum()) == 12
    return m


def make_voronoi_mesh(points: np.ndarray, name: str) -> Mesh:
    """The spherical Voronoi mesh of arbitrary generators (unit vectors, [n, 3]).  The convex hull of points on a sphere
    is their spherical Delaunay triangulation; its faces are turned counter-clockwise seen from outside, as
    ``_icosahedron`` does.  Cells may have 3 to MAX_EDGES sides."""
    from scipy.spatial import ConvexHull
    p = np.ascontiguousarray(points, dtype=np.float64)
    f = ConvexHull(p).simplices.astype(np.int64)
    a, b, c = p[f[:, 0]], p[f[:, 1]], p[f[:, 2]]
    flip = np.einsum("ij,ij->i", np.cross(b - a, c - a), a + b + c) < 0
    f[flip] = f[flip][:, [0, 2, 1]]
    return mesh_from_triangulation(p, f, name)


def mesh_from_triangulation(p: np.ndarray, f: np.ndarray, name: str) -> Mesh:
    """The Voronoi mesh dual to a triangulation of the unit sphere: points ``p`` [nC, 3] become cells, the counter-
    clockwise triangles ``f`` [nV, 3] (0-based) become vertices placed at their circumcentres."""
    nC, nV = p.shape[0], f.shape[0]
    assert nV == 2 * nC - 4
    nE = 3 * nC - 6

    # ---- directed half-edges: triangle t lies to the left of a->b; around a, b is followed by c
    a = np.concatenate([f[:, 0], f[:, 1], f[:, 2]])
    b = np.concatenate([f[:, 1], f[:, 2], f[:, 0]])
    c = np.concatenate([f[:, 2], f[:, 0], f[:, 1]])
    t = np.concatenate([np.arange(nV)] * 3)
    key = a * nC + b
    order = np.argsort(key, kind="stable")
    key_s, a_s, b_s, c_s, t_s = key[order], a[order], b[order], c[order], t[order]

    def lookup(aa, bb):
        pos = np.searchsorted(key_s, aa * nC + bb)
        return pos

    # ---- undirected edges: cell1 < cell2
    und = a_s < b_s
    c1, c2 = a_s[und], b_s[und]
    assert c1.shape[0] == nE
    ekey = c1 * nC + c2                      # sorted ascending already
    t_left = t_s[und]                        # triangle left of c1->c2  (the +t side)
    t_right = t_s[lookup(c2, c1)]            # triangle left of c2->c1
    cellsOnEdge = np.stack([c1, c2], 1)
    verticesOnEdge = np.stack([t_right, t_left], 1)   # v1 -> v2 runs along k x n

    def edge_of(aa, bb):
        lo, hi = np.minimum(aa, bb), np.maximum(aa, bb)
        return np.searchsorted(ekey, lo * nC + hi)

    # ---- counter-clockwise rings around each cell
    first = np.searchsorted(a_s, np.arange(nC))           # first half-edge leaving each cell
    deg = np.searchsorted(a_s, np.arange(nC), side="right") - first
    nEdgesOnCell = deg.astype(np.int32)
    assert deg.min() >= 3 and deg.max() <= MAX_EDGES
    cellsOnCell = np.zeros((nC, MAX_EDGES), dtype=np.int64)
    triAfter = np.zeros((nC, MAX_EDGES), dtype=np.int64)   # triangle between neighbour i and i+1
    cur = b_s[first]
    me = np.arange(nC)
    for i in range(int(deg.max())):
        act = i < deg
        pos = lookup(me, cur)
        cellsOnCell[act, i] = cur[act]
        triAfter[act, i] = t_s[pos][act]
        cur = c_s[pos]
    edgesOnCell = np.zeros((nC, MAX_EDGES), dtype=np.int64)
    verticesOnCell = np.zeros((nC, MAX_EDGES), dtype=np.int64)
    for i in range(int(deg.max())):
        act = i < deg
        edgesOnCell[act, i] = edge_of(me, cellsOnCell[:, i])[act]
        # vertex i sits before edge i (between edge i-1 and edge i)
        prev = np.where(i == 0, deg - 1, i - 1)
        verticesOnCell[act, i] = triAfter[me, prev][act]

    # ---- vertices (triangles)
    cellsOnVertex = f.copy()
    edgesOnVertex = np.stack([edge_of(f[:, 0], f[:, 1]), edge_of(f[:, 1], f[:, 2]), edge_of(f[:, 2], f[:, 0])], 1)
    pa, pb, pc = p[f[:, 0]], p[f[:, 1]], p[f[:, 2]]
    pv = np.cross(pb - pa, pc - pa)
    pv /= np.linalg.norm(pv, axis=1, keepdims=True)
    pe = p[c1] + p[c2]
    pe /= np.linalg.norm(pe, axis=1, keepdims=True)

    # ---- metrics
    dcEdge = _arc(p[c1], p[c2])
    dvEdge = _arc(pv[t_right], pv[t_left])
    kite = np.zeros((nV, 3))
    for j in range(3):
        cj = f[:, j]
        e_next = edgesOnVertex[:, j]             # edge (cov[j], cov[j+1])
        e_prev = edgesOnVertex[:, (j + 2) % 3]   # edge (cov[j-1], cov[j])
        kite[:, j] = _tri_area(p[cj], pe[e_next], pv) + _tri_area(p[cj], pv, pe[e_prev])
    areaTriangle = kite.sum(1)
    areaCell = np.zeros(nC)
    np.add.at(areaCell, f.ravel(), kite.ravel())

    latC, lonC = _latlon(p)
    latE, lonE = _latlon(pe)
    latV, lonV = _latlon(pv)
    # angleEdge: angle of the edge normal (cell1 -> cell2) from local east at the edge point
    east = np.stack([-np.sin(lonE), np.cos(lonE), np.zeros(nE)], 1)
    north = np.stack([-np.sin(latE) * np.cos(lonE), -np.sin(latE) * np.sin(lonE), np.cos(latE)], 1)
    nrm = p[c2] - p[c1]
    nrm -= np.einsum("ij,ij->i", nrm, pe)[:, None] * pe
    angleEdge = np.arctan2(np.einsum("ij,ij->i", nrm, north), np.einsum("ij,ij->i", nrm, east))

    nEoE, eoe, woe = trisk_weights(nEdgesOnCell, edgesOnCell, verticesOnCell, cellsOnEdge,
                                   cellsOnVertex, kite, areaCell, dcEdge, dvEdge)

    def pad_last(arr, cnt):
        """1-based ids, unused slots repeat the last valid id (as in the bundled file)."""
        out = arr + 1
        last = out[np.arange(out.shape[0]), cnt - 1]
        mask = np.arange(out.shape[1])[None, :] >= cnt[:, None]
        out[mask] = np.broadcast_to(last[:, None], out.shape)[mask]
        return out.astype(np.int32)

    voc = verticesOnCell + 1
    voc[np.arange(MAX_EDGES)[None, :] >= deg[:, None]] = 0
    i32 = lambda x: np.ascontiguousarray(x, dtype=np.int32)
    f64 = lambda x: np.ascontiguousarray(x, dtype=np.float64)
    v = dict(
        latCell=f64(latC), lonCell=f64(lonC), meshDensity=np.ones(nC), xCell=f64(p[:, 0]), yCell=f64(p[:, 1]),
        zCell=f64(p[:, 2]), indexToCellID=i32(np.arange(1, nC + 1)),
        latEdge=f64(latE), lonEdge=f64(lonE), xEdge=f64(pe[:, 0]), yEdge=f64(pe[:, 1]), zEdge=f64(pe[:, 2]),
        indexToEdgeID=i32(np.arange(1, nE + 1)),
        latVertex=f64(latV), lonVertex=f64(lonV), xVertex=f64(pv[:, 0]), yVertex=f64(pv[:, 1]),
        zVertex=f64(pv[:, 2]), indexToVertexID=i32(np.arange(1, nV + 1)),
        cellsOnEdge=i32(cellsOnEdge + 1), nEdgesOnCell=i32(nEdgesOnCell), nEdgesOnEdge=i32(nEoE),
        edgesOnCell=pad_last(edgesOnCell, deg), edgesOnEdge=i32(eoe), weightsOnEdge=f64(woe),
        dvEdge=f64(dvEdge), dv1Edge=f64(_arc(pv[t_right], pe)), dv2Edge=f64(_arc(pv[t_left], pe)),
        dcEdge=f64(dcEdge), angleEdge=f64(angleEdge), areaCell=f64(areaCell), areaTriangle=f64(areaTriangle),
        cellsOnCell=pad_last(cellsOnCell, deg), verticesOnCell=i32(voc), verticesOnEdge=i32(verticesOnEdge + 1),
        edgesOnVertex=i32(edgesOnVertex + 1), cellsOnVertex=i32(cellsOnVertex + 1), kiteAreasOnVertex=f64(kite),
    )
    m = Mesh(v=v, partition=None, name=name)
    m.validate()
    return m
