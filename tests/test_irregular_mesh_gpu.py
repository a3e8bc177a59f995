"""The CUDA path against the oracle on the irregular mesh of tests/irregular.py (cells of 4 to 10 sides, up to 14 edge
neighbours, capped advection lists) with MPAS's regional masks on, and without them so that a failure can be put on
the mesh or on the masks.

In the default configuration every field the kernels write is bit-identical to the oracle's except q and tend_u, whose
edgesOnEdge sums run in another order, and exner / pressure_p after recover at rk_step 2, where exner is a device pow
(DESIGN.md §2); the task-by-task checks hold every other field to its bits."""
import numpy as np
import pytest

from mpas_regent_b200 import _abi, dynamics
from tests import irregular
from tests.test_parity_gpu import (ACOUSTIC_OUT, CORRECTED_TASKS, DT, L_SMALL, TASKS, _warm, acoustic_mode_parity,
                                   advance_scalars_parity, emulated_ranks_equal_single_partition,
                                   mesh_only_init_producers_equal_oracle, range_restricted_launches_equal_whole)
from tests.util import build_pair, compare

pytestmark = pytest.mark.gpu

NOT_BITWISE = ("q", "tend_u")
POW = ("exner", "pressure_p")
POLICIES = [_abi.INDEX_CORRECTED, _abi.INDEX_LITERAL]
VARIANTS = [(p, m) for m in (True, False) for p in POLICIES]
VARIANT_IDS = [f"{'corrected' if p == _abi.INDEX_CORRECTED else 'literal'}-{'masked' if m else 'unmasked'}" for p, m in VARIANTS]


def _pair(policy, masked=True, L=L_SMALL, **kw):
    return build_pair(irregular.irregular_mesh(), L, policy, masks=irregular.regional_masks() if masked else None, **kw)


def _bitwise(g, ora, what, skip=()):
    bad = [n for n, _, _ in _abi.FIELDS if n not in NOT_BITWISE + tuple(skip)
           and not np.array_equal(g.download_field(n), ora.download_field(n), equal_nan=True)]
    assert not bad, f"{what}: not bit-identical: {bad}"


def _same_bits(outs):
    for n in outs[0]:
        for o in outs[1:]:
            assert np.array_equal(outs[0][n], o[n], equal_nan=True), n


# ---- task by task, from one warmed snapshot ----------------------------------------------------------------------------
@pytest.fixture(scope="module", params=VARIANTS, ids=VARIANT_IDS)
def warmed(request):
    policy, masked = request.param
    st, ora, g = _pair(policy, masked)
    _warm(ora, g)
    snap = {n: ora.download_field(n) for (n, _, _) in _abi.FIELDS}
    yield ora, g, snap
    g.close(); ora.close()


@pytest.mark.parametrize("name,fn", TASKS, ids=[t[0] for t in TASKS])
def test_task_parity(warmed, name, fn):
    ora, g, snap = warmed
    for n, a in snap.items():
        ora.upload_field(n, a); g.upload_field(n, a)
    fn(ora); fn(g)
    compare(g, ora, what=name)
    _bitwise(g, ora, name, POW if name == "recover_rk2" else ())


@pytest.fixture(scope="module", params=VARIANTS, ids=VARIANT_IDS)
def warmed_physics(request):
    """state after one LITERAL step (finite everywhere), then both backends switched to CORRECTED physics."""
    policy, masked = request.param
    st, ora0, _ = _pair(policy, masked, gpu=False)
    ora0.atm_compute_solve_diagnostics(False, -1)
    ora0.atm_srk3(DT)
    snap = {n: ora0.download_field(n) for (n, _, _) in _abi.FIELDS}
    ora0.close()
    st, ora, g = _pair(policy, masked, physics_mode=_abi.PHYSICS_CORRECTED)
    yield ora, g, snap
    g.close(); ora.close()


@pytest.mark.parametrize("name,fn", CORRECTED_TASKS, ids=[t[0] for t in CORRECTED_TASKS])
def test_corrected_physics_task_parity(warmed_physics, name, fn):
    ora, g, snap = warmed_physics
    for n, a in snap.items():
        ora.upload_field(n, a); g.upload_field(n, a)
    fn(ora); fn(g)
    compare(g, ora, what="corrected physics " + name)
    _bitwise(g, ora, "corrected physics " + name, POW if name.endswith("recover") or name == "recover_rk2" else ())


def test_masks_reach_the_kernels():
    """the masked and the unmasked mesh give different results where the masks act: smlstep and recover skip cells beyond
    nRelaxZone, the acoustic step integrates specified columns, divergence damping leaves specified and shared edges."""
    outs = []
    for masked in (True, False):
        st, ora, g = _pair(_abi.INDEX_CORRECTED, masked, gpu=True, physics_mode=_abi.PHYSICS_CORRECTED)
        for b in (ora, g):
            b.atm_compute_solve_diagnostics(False, -1)
            b.atm_srk3(DT)
        outs.append(g.download_all())
        g.close(); ora.close()
    bdy = irregular.regional_masks()["bdyMaskCell"]
    for n in ("w", "rw_p", "rho_pp", "ru_p"):
        a, b = outs[0][n], outs[1][n]
        assert not np.array_equal(a, b), n
    assert not np.array_equal(outs[0]["w"][bdy > irregular.N_RELAX_ZONE], outs[1]["w"][bdy > irregular.N_RELAX_ZONE])


def test_divergence_damping_carries_masks_across_tiles():
    """k_divdamp's persistent blocks walk the edge tiles and load the next edge's specZoneMaskEdge and skip flag ahead of
    the current edge's arithmetic.  The carry only runs when a launch has more tiles than resident blocks, which the 646-cell
    mesh never has: x1.40962 (122880 edges) needs several passes at any occupancy.  Random masks make a value carried
    from the wrong edge visible."""
    from mpas_regent_b200 import icosa, init_jw
    from oracle.oracle import Oracle
    mesh = icosa.make_icosahedral_mesh(40962)
    L = L_SMALL
    st = init_jw.make_state(mesh, L, _abi.INDEX_CORRECTED)
    rng = np.random.default_rng(17)
    st.static["specZoneMaskEdge"] = rng.integers(0, 2, mesh.nEdges).astype(np.float64)
    st.static["isShared"] = (rng.random(mesh.nCells) < 0.3).astype(np.uint8)
    cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX)
    ora, g = Oracle(dynamics.dims_of(mesh, L), cfg), dynamics.Dynamics(dynamics.dims_of(mesh, L), cfg)
    cell, edge = st.f["theta_m"].shape, st.f["u"].shape
    f = {"rtheta_pp": rng.standard_normal(cell), "rtheta_pp_old": rng.standard_normal(cell), "theta_m": st.f["theta_m"],
         "ru_p": rng.standard_normal(edge)}
    for b in (ora, g):
        b.upload_mesh(st.static); b.upload_state(st.f, st.vert)
        for n, a in f.items():
            b.upload_field(n, a)
        b.atm_divergence_damping_3d(360.0)
    got, want = g.download_field("ru_p"), ora.download_field("ru_p")
    assert not np.array_equal(want, f["ru_p"])
    assert np.array_equal(got, want), int((got != want).any(axis=1).sum())
    g.close(); ora.close()


# ---- full steps ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("policy,masked", VARIANTS, ids=VARIANT_IDS)
@pytest.mark.parametrize("rkarg", [_abi.RKARG_STAGE_INDEX, _abi.RKARG_SUBSTEP_TRUNC], ids=["stage_index", "substep_trunc"])
def test_full_step_parity(policy, masked, rkarg):
    """one RK3 step, then 9 more inside the growth bound 1e-12 * (1 + step) of test_hundred_step_drift."""
    st, ora, g = _pair(policy, masked, rkarg=rkarg)
    for b in (ora, g):
        b.atm_compute_solve_diagnostics(False, -1)
    for step in range(1, 11):
        for b in (ora, g):
            b.atm_srk3(DT)
        compare(g, ora, tol=1e-12 * (1 + step) if step > 1 else 1e-12, what=f"after {step} steps")
    assert np.isfinite(ora.download_field("u")).all()
    g.close(); ora.close()


@pytest.mark.parametrize("policy,masked", VARIANTS, ids=VARIANT_IDS)
@pytest.mark.parametrize("rkarg", [_abi.RKARG_STAGE_INDEX, _abi.RKARG_SUBSTEP_TRUNC], ids=["stage_index", "substep_trunc"])
def test_corrected_physics_full_step_parity(policy, masked, rkarg):
    """the first CORRECTED step stays finite and within 1e-12; the second, where the reference's remaining quirks (Q17/Q27)
    begin to produce Inf/NaN, must have the oracle's NaN/Inf positions."""
    st, ora, g = _pair(policy, masked, rkarg=rkarg, physics_mode=_abi.PHYSICS_CORRECTED)
    u0 = ora.download_field("u")
    for b in (ora, g):
        b.atm_compute_solve_diagnostics(False, -1)
        b.atm_srk3(DT)
    assert np.isfinite(ora.download_field("u")).all() and not np.array_equal(u0, ora.download_field("u"))
    compare(g, ora, what="corrected physics, 1 step")
    for b in (ora, g):
        b.atm_srk3(DT)
    for n, _, _ in _abi.FIELDS:
        a, b = g.download_field(n), ora.download_field(n)
        assert np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(np.isinf(a), np.isinf(b)), n
    g.close(); ora.close()


# ---- acoustic forms, lane pipeline shapes, launch ranges -------------------------------------------------------------
@pytest.mark.parametrize("exact", [0, 1, 2, 3, 4], ids=["fused_affine", "two_kernel_exact", "fused_affine_tma", "split_gather_tma", "split_gather_lane_pipeline_default"])
def test_acoustic_modes(exact):
    acoustic_mode_parity(irregular.irregular_mesh(), exact, masks=irregular.regional_masks())


@pytest.mark.parametrize("levels", [4, 26, 58], ids=lambda v: f"L{v}")
def test_acoustic_lane_pipeline_shapes(levels):
    """k_acoustic_lane (32-column tiles, 8-level chunks) with specified-zone columns and cells of every degree: a full step
    bit-identical on the acoustic outputs, then a restricted cell range advances exactly the cells it covers."""
    st, ora, g = _pair(_abi.INDEX_CORRECTED, True, L=levels, acoustic_tma=3)
    for b in (ora, g):
        b.atm_compute_solve_diagnostics(False, -1)
        b.atm_srk3(300.0)
    compare(g, ora, what=f"L={levels}")
    for n in ACOUSTIC_OUT[2:]:
        assert np.array_equal(g.download_field(n), ora.download_field(n), equal_nan=True), n
    snap = {n: ora.download_field(n) for n in ACOUSTIC_OUT[2:]}
    g.set_range(_abi.CELL, 37, 301)
    g.atm_advance_acoustic_step(100.0, 1)
    ora.atm_advance_acoustic_step(100.0, 1)
    for n in ACOUSTIC_OUT[2:]:
        a, full = g.download_field(n), ora.download_field(n)
        touched = ~np.all(a == snap[n], axis=1)
        assert 0 < touched.sum() <= 301 - 37, n
        assert np.array_equal(a[touched], full[touched], equal_nan=True), n
    g.close(); ora.close()


@pytest.mark.parametrize("physics", [_abi.PHYSICS_LITERAL, _abi.PHYSICS_CORRECTED], ids=["literal", "corrected_physics"])
def test_range_restricted_launches_equal_whole(physics):
    range_restricted_launches_equal_whole(irregular.irregular_mesh(), irregular.make_state(9, _abi.INDEX_CORRECTED), physics)


# ---- bitwise invariance of launch forms, numbering and drivers -------------------------------------------------------
def _run(st, L, steps, mode="driver", **cfg_over):
    cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, use_graph=int(mode == "graph"), **cfg_over)
    g = dynamics.Dynamics(dynamics.dims_of(irregular.irregular_mesh(), L), cfg)
    g.upload_mesh(st.static); g.upload_state(st.f, st.vert)
    g.atm_compute_solve_diagnostics(False, -1)
    for _ in range(steps):
        g.atm_srk3_by_tasks(600.0) if mode == "tasks" else g.atm_srk3(600.0)
    out = g.download_all()
    g.close()
    return out


@pytest.mark.parametrize("physics", [_abi.PHYSICS_LITERAL, _abi.PHYSICS_CORRECTED], ids=["literal", "corrected_physics"])
def test_forms_numbering_and_drivers_are_bit_identical(physics):
    """kernel_forms 0 / 1, sfc_renumber 0 / 1, and the host task replay / the library's driver / its CUDA graph."""
    st = irregular.make_state(10, _abi.INDEX_CORRECTED)
    steps = 2 if physics == _abi.PHYSICS_LITERAL else 1
    base = _run(st, 10, steps, physics_mode=physics)
    _same_bits([base, _run(st, 10, steps, physics_mode=physics, kernel_forms=1)])
    _same_bits([base, _run(st, 10, steps, physics_mode=physics, sfc_renumber=0)])
    _same_bits([base, _run(st, 10, steps, "tasks", physics_mode=physics), _run(st, 10, steps, "graph", physics_mode=physics)])


# ---- scalar advection, mesh-only init producers, emulated ranks ------------------------------------------------------
@pytest.mark.parametrize("policy", POLICIES, ids=["corrected", "literal"])
def test_advance_scalars_parity(policy):
    advance_scalars_parity(irregular.irregular_mesh(), policy, masks=irregular.regional_masks())


@pytest.mark.parametrize("policy", POLICIES, ids=["corrected", "literal"])
def test_mesh_only_init_producers_on_the_device(policy):
    mesh_only_init_producers_equal_oracle(irregular.irregular_mesh(), policy)


@pytest.mark.parametrize("physics", [_abi.PHYSICS_LITERAL, _abi.PHYSICS_CORRECTED], ids=["literal", "corrected_physics"])
def test_emulated_ranks_on_one_gpu_equal_single_partition(physics):
    emulated_ranks_equal_single_partition(irregular.irregular_mesh(), irregular.make_state(6, _abi.INDEX_CORRECTED), physics, False)
