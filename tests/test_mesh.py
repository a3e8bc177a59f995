"""Mesh reader, fixture and the synthetic icosahedral generator (CPU only)."""
import numpy as np
import pytest

from mpas_regent_b200 import icosa
from mpas_regent_b200 import mesh as M


def test_fixture_matches_survey_facts(grid2562):
    m = grid2562
    assert (m.nCells, m.nEdges, m.nVertices) == (2562, 7680, 5120)          # constants.rg:18-20
    assert int((m["nEdgesOnCell"] == 5).sum()) == 12                        # pentagons
    assert m.partition is not None and m.partition.shape == (2562,)
    sizes = np.bincount(m.partition, minlength=16).tolist()                 # SURVEY.md 8c cross-check
    assert sizes == [161, 155, 161, 156, 160, 161, 161, 159, 162, 159, 161, 162, 164, 160, 156, 164]


def test_literal_policy_pad_hits(grid2562):
    """valid-slot ids equal to N: indices one past the region under LITERAL (SURVEY.md 8c)."""
    m = grid2562
    v = m.v
    nC, nE, nV = m.nCells, m.nEdges, m.nVertices
    slotC = np.arange(10)[None, :] < v["nEdgesOnCell"][:, None]
    slotE = np.arange(20)[None, :] < v["nEdgesOnEdge"][:, None]
    assert int((v["edgesOnCell"][slotC] == nE).sum()) == 2
    assert int((v["cellsOnEdge"] == nC).sum()) == 6
    assert int((v["verticesOnEdge"] == nV).sum()) == 3
    assert int((v["edgesOnVertex"] == nE).sum()) == 2
    assert int((v["cellsOnCell"][slotC] == nC).sum()) == 6
    assert int((v["edgesOnEdge"][slotE] == nE).sum()) == 9
    for name, n in (("edgesOnCell", nE), ("cellsOnEdge", nC)):
        lit = M.resolve_ids(v[name], n, M.LITERAL)
        cor = M.resolve_ids(v[name], n, M.CORRECTED)
        assert lit.max() <= n and cor.max() <= n and lit.min() >= 0 and cor.min() >= 0


def test_trisk_weights_reproduce_the_bundled_file(grid2562):
    """the generator's TRiSK routine, fed the file's own connectivity, returns the file's weights."""
    v = grid2562.v
    nEoE, eoe, woe = icosa.trisk_weights(v["nEdgesOnCell"], v["edgesOnCell"] - 1, v["verticesOnCell"] - 1,
                                         v["cellsOnEdge"] - 1, v["cellsOnVertex"] - 1, v["kiteAreasOnVertex"],
                                         v["areaCell"], v["dcEdge"], v["dvEdge"])
    assert np.array_equal(nEoE, v["nEdgesOnEdge"])
    assert np.array_equal(eoe, v["edgesOnEdge"])
    assert np.abs(woe - v["weightsOnEdge"]).max() < 1e-14


@pytest.mark.parametrize("n", [12, 42, 642, 2562, 10242])
def test_icosahedral_mesh_invariants(n):
    m = icosa.make_icosahedral_mesh(n)
    v = m.v
    assert m.nCells == n and m.nEdges == 3 * n - 6 and m.nVertices == 2 * n - 4
    assert int((v["nEdgesOnCell"] == 5).sum()) == 12
    check_voronoi_invariants(m, trisk_edges=300)


def check_voronoi_invariants(m, trisk_edges=None):
    """what every closed spherical Voronoi mesh of the generator satisfies; TRiSK antisymmetry on the first
    ``trisk_edges`` edges (all when None)."""
    v = m.v
    n = m.nCells
    for k in ("areaCell", "areaTriangle", "kiteAreasOnVertex"):
        assert abs(v[k].sum() - 4 * np.pi) < 1e-9
    # every edge appears once in each of its two cells; ids are 1-based
    eoc, ne = v["edgesOnCell"], v["nEdgesOnCell"]
    slot = np.arange(10)[None, :] < ne[:, None]
    assert np.array_equal(np.bincount(eoc[slot] - 1, minlength=m.nEdges), np.full(m.nEdges, 2))
    assert v["cellsOnEdge"].min() == 1 and v["cellsOnEdge"].max() == n
    # convention of the bundled file: edge i of a cell joins vertex i and vertex i+1, for every slot up to the degree
    for i in range(int(ne.max())):
        c = np.flatnonzero(i < ne)
        e = eoc[c, i] - 1
        a = np.sort(v["verticesOnEdge"][e], axis=1)
        nxt = np.where(i + 1 < ne[c], i + 1, 0)
        b = np.sort(np.stack([v["verticesOnCell"][c, i], v["verticesOnCell"][c, nxt]], 1), axis=1)
        assert np.array_equal(a, b), i
    # TRiSK: weights are antisymmetric in energy norm  w_{e,e'} dc_e / dv_e' = - w_{e',e} dc_e' / dv_e
    nE = m.nEdges if trisk_edges is None else min(m.nEdges, trisk_edges)
    W = {}
    eoe, woe, neoe = v["edgesOnEdge"] - 1, v["weightsOnEdge"], v["nEdgesOnEdge"]
    for e in range(nE):
        for j in range(neoe[e]):
            W[(e, eoe[e, j])] = woe[e, j] * v["dcEdge"][e] / v["dvEdge"][eoe[e, j]]
    pairs = 0
    for (e, e2), w in W.items():
        if (e2, e) in W:
            assert abs(w + W[(e2, e)]) < 1e-12
            pairs += 1
    assert pairs > 0
    if trisk_edges is None:
        assert pairs == len(W)


# SHA-256 over (name, dtype, shape, bytes) of every array, in name order, from the generator before it was split into
# make_icosahedral_mesh + mesh_from_triangulation: the icosahedral meshes every other test runs on keep their bits.
ICOSA_DIGESTS = {
    642: "4efb030d31e3a27d1e402b51b6a910687107aa3491e2ef7a3b8ab880907dc0ed",
    10242: "de069213bdd3173199773d13bb1888eda43267c7fb1e1fc651dcef561a91cff4",
}


def mesh_digest(m):
    import hashlib
    h = hashlib.sha256()
    for k in sorted(m.v):
        a = np.ascontiguousarray(m.v[k])
        h.update(k.encode()); h.update(str(a.dtype).encode()); h.update(str(a.shape).encode()); h.update(a.tobytes())
    return h.hexdigest()


@pytest.mark.parametrize("n", sorted(ICOSA_DIGESTS))
def test_icosahedral_mesh_bits_are_pinned(n):
    m = icosa.make_icosahedral_mesh(n)
    assert m.name == f"x1.{n}"
    assert mesh_digest(m) == ICOSA_DIGESTS[n]


def test_icosahedral_generator_is_deterministic():
    a, b = icosa.make_icosahedral_mesh(642), icosa.make_icosahedral_mesh(642)
    for k in a.v:
        assert np.array_equal(a.v[k], b.v[k])


def test_level_for_cells():
    assert icosa.level_for_cells(40962) == 6 and icosa.level_for_cells(655362) == 8
    with pytest.raises(ValueError):
        icosa.level_for_cells(1000)
