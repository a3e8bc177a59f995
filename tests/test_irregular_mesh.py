"""The irregular mesh of tests/irregular.py (cells of 4 to 10 sides) and its regional masks, on the CPU: the generator's
invariants, the oracle against the array-at-a-time restatements with the masks on, and N ranks against one."""
import numpy as np
import pytest

from mpas_regent_b200 import _abi, core_init, dynamics, icosa, parallel
from mpas_regent_b200.mesh import MAX_EDGES
from tests import irregular, test_oracle_restatements as R
from tests.test_mesh import check_voronoi_invariants, mesh_digest
from tests.test_oracle import check_corrected_acoustic_restatement
from tests.test_parallel import _assert_owned_equal, _rank_backend, _single, _task_schedule


def test_degrees_edge_neighbours_and_adv_cap():
    m = irregular.irregular_mesh()
    v = m.v
    assert (m.nCells, m.nEdges, m.nVertices) == (646, 1932, 1288)
    deg, cnt = np.unique(v["nEdgesOnCell"], return_counts=True)
    assert dict(zip(deg.tolist(), cnt.tolist())) == {4: 3, 5: 44, 6: 569, 7: 25, 8: 3, 9: 1, 10: 1}
    assert v["nEdgesOnEdge"].max() == 14
    # atm_adv_coef_compression caps its cell list at index maxEdges - 1 (dynamics_tasks.rg:175): on some edges the list
    # holds fewer cells than the two cells and their neighbours
    adv = core_init.atm_adv_coef_compression(m, _abi.INDEX_CORRECTED, None)
    n_adv = adv["nAdvCellsForEdge"]
    capped = n_adv < irregular.adv_list_uncapped(m)
    assert capped.sum() > 0 and np.all(n_adv[capped] >= MAX_EDGES - 1)
    assert n_adv.max() == MAX_EDGES                # cell1's own neighbours are never capped: a 10-gon lists all of them


def test_invariants():
    m = irregular.irregular_mesh()
    check_voronoi_invariants(m)
    # the mesh is not well centred: 10 circumcentres lie outside their triangle, whose kite parts are signed
    kite = m.v["kiteAreasOnVertex"]
    assert int((kite < 0).sum()) == 10 and (m.v["areaCell"] > 0).all() and (m.v["areaTriangle"] > 0).all()


def test_generator_is_deterministic():
    a, b = irregular.irregular_mesh.__wrapped__(), irregular.irregular_mesh.__wrapped__()
    assert mesh_digest(a) == mesh_digest(b)
    assert mesh_digest(icosa.make_voronoi_mesh(irregular.generators(), "irregular646")) == mesh_digest(a)


def test_mask_layout():
    m, mk = irregular.irregular_mesh(), irregular.regional_masks()
    bdy = mk["bdyMaskCell"]
    assert np.bincount(bdy).tolist() == [363, 47, 47, 43, 39, 35, 32, 40]
    assert np.array_equal(mk["specZoneMaskCell"] == 1.0, bdy >= 6)
    assert np.array_equal(mk["isShared"] == 1, bdy == 7)
    coe = m.v["cellsOnEdge"] - 1
    assert np.array_equal(mk["specZoneMaskEdge"] == 1.0, (bdy[coe] >= 6).any(axis=1))
    # an edge between a specified and a relaxation cell, and one between two shared cells (divergence damping skips it)
    assert ((bdy[coe[:, 0]] >= 6) != (bdy[coe[:, 1]] >= 6)).any()
    assert (mk["isShared"][coe] == 1).all(axis=1).any()


# ---- the restatements of test_oracle_restatements.py on the irregular mesh with the masks: this module's `warmed`
# ---- fixture replaces that module's for the test functions imported here
@pytest.fixture(scope="module")
def warmed():
    from oracle.oracle import Oracle
    st = irregular.make_state(R.L, _abi.INDEX_CORRECTED)
    ora = Oracle(dynamics.dims_of(st.mesh, R.L), _abi.default_config(index_policy=_abi.INDEX_CORRECTED, rkarg_policy=_abi.RKARG_STAGE_INDEX))
    ora.upload_mesh(st.static); ora.upload_state(st.f, st.vert)
    ora.atm_compute_solve_diagnostics(False, -1)
    ora.atm_srk3(600.0)
    pre = ora.download_all()
    assert all(np.isfinite(a).all() for a in pre.values())
    yield st, ora, pre
    ora.close()


test_divergence_damping_3d = R.test_divergence_damping_3d
test_set_smlstep_pert_variables = R.test_set_smlstep_pert_variables
test_advance_acoustic_step_literal = R.test_advance_acoustic_step_literal
test_recover_large_step_variables = R.test_recover_large_step_variables
test_compute_vert_imp_coefs = R.test_compute_vert_imp_coefs
test_compute_solve_diagnostics = R.test_compute_solve_diagnostics
test_compute_dyn_tend = R.test_compute_dyn_tend
test_advance_scalars = R.test_advance_scalars
test_init_coupled_diagnostics_and_reconstruct_2d = R.test_init_coupled_diagnostics_and_reconstruct_2d


@pytest.mark.parametrize("small_step", [0, 1])
def test_corrected_physics_acoustic_step_matches_array_restatement(small_step):
    check_corrected_acoustic_restatement(irregular.irregular_mesh(), small_step, masks=irregular.regional_masks())


# ---- partitions: N ranks over the in-process exchange equal one rank, bitwise on owned entities ------------------------
def test_halo_lists_are_symmetric():
    m = irregular.irregular_mesh()
    st = irregular.make_state(6, _abi.INDEX_CORRECTED)
    shards = parallel.make_shards(st, 4)
    for ent, attr, n in (("cell", "cells", m.nCells), ("edge", "edges", m.nEdges), ("vertex", "vertices", m.nVertices)):
        e = ("cell", "edge", "vertex").index(ent)
        assert sum(sh["lm"].n_owned[e] for sh in shards) == n
        for h, sh in enumerate(shards):
            lm = sh["lm"]
            for o, ridx in lm.recv[ent].items():
                assert np.array_equal(getattr(lm, attr)[ridx], getattr(shards[o]["lm"], attr)[shards[o]["lm"].send[ent][h]])


@pytest.mark.parametrize("physics", [_abi.PHYSICS_LITERAL, _abi.PHYSICS_CORRECTED], ids=["literal", "corrected_physics"])
@pytest.mark.parametrize("world", [2, 4])
def test_n_ranks_equal_single_partition_bitwise(world, physics):
    from tests.test_parallel import L
    m = irregular.irregular_mesh()
    st = irregular.make_state(L, _abi.INDEX_CORRECTED)
    shards = parallel.make_shards(st, world)
    # every irregular cell is owned by some rank, and the masks travel with the shards
    for sh in shards:
        for k in ("bdyMaskCell", "specZoneMaskCell", "isShared"):
            assert np.array_equal(sh["static"][k], st.static[k][sh["lm"].cells]), k
    single = _single(m, st, 2, physics)
    backs = [_rank_backend(s, physics) for s in shards]
    ex = parallel.InProcessExchanger(backs, [s["lm"] for s in shards])
    exchanges = parallel.exchanges_for(backs[0].cfg)
    for b in backs:
        b.atm_compute_solve_diagnostics(False, -1)
    ex.exchange(exchanges["compute_solve_diagnostics"])
    seq = _task_schedule(backs[0].cfg)
    for _ in range(2):
        for name, args in seq:
            for b in backs:
                b._call(name, *args)
            spec = exchanges.get(parallel.exchange_key(name, args))
            if spec:
                ex.exchange(spec)
    for b, s in zip(backs, shards):
        _assert_owned_equal(single, b, s["lm"])
        b.close()
    single.close()
