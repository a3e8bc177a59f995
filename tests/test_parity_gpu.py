"""Parity of the CUDA path (through the C ABI) against the CPU oracle -- the parity tests proper.

Reference: every hot-path task of dynamics/dynamics_tasks.rg and the driver rk_timestep.rg:361-500.
Tolerance per BASELINE.json: 1e-12 relative per field, identical NaN/Inf positions; integer
connectivity handling is exercised under both index policies.
"""
import numpy as np
import pytest

from mpas_regent_b200 import _abi
from tests.util import build_pair, compare, copy_state

pytestmark = pytest.mark.gpu

L_SMALL = 26
DT = 720.0


def _warm(ora, g, dt=DT):
    """populate every intermediate field with one oracle step, then mirror it onto the GPU."""
    ora.atm_compute_solve_diagnostics(False, -1)
    ora.atm_srk3(dt)
    copy_state(ora, g)


TASKS = [
    ("rk_integration_setup", lambda b: b.atm_rk_integration_setup()),
    ("compute_moist_coefficients", lambda b: b.atm_compute_moist_coefficients()),
    ("compute_vert_imp_coefs", lambda b: b.atm_compute_vert_imp_coefs(240.0)),
    ("compute_vert_imp_coefs_again", lambda b: (b.atm_compute_vert_imp_coefs(240.0), b.atm_compute_vert_imp_coefs(360.0))),
    ("dyn_tend_rk0", lambda b: b.atm_compute_dyn_tend(0, DT)),
    ("dyn_tend_rk1", lambda b: b.atm_compute_dyn_tend(1, DT)),
    ("dyn_tend_rk2", lambda b: b.atm_compute_dyn_tend(2, DT)),
    ("dyn_tend_neg", lambda b: b.atm_compute_dyn_tend(-1, DT)),
    ("dyn_tend_fixed", lambda b: b.atm_compute_dyn_tend(0, DT, config_horiz_mixing=_abi.MIX_2D_FIXED)),
    ("dyn_tend_other", lambda b: b.atm_compute_dyn_tend(0, DT, config_horiz_mixing=_abi.MIX_OTHER)),
    ("dyn_tend_cam", lambda b: b.atm_compute_dyn_tend(0, DT, config_mpas_cam_coef=0.2)),
    ("dyn_tend_rayleigh", lambda b: b.atm_compute_dyn_tend(1, DT, config_rayleigh_damp_u=True)),
    ("set_smlstep_pert_variables", lambda b: b.atm_set_smlstep_pert_variables()),
    ("acoustic_step0", lambda b: b.atm_advance_acoustic_step(240.0, 0)),
    ("acoustic_step1", lambda b: b.atm_advance_acoustic_step(360.0, 1)),
    ("acoustic_pair", lambda b: (b.atm_advance_acoustic_step(360.0, 0), b.atm_divergence_damping_3d(360.0),
                                 b.atm_advance_acoustic_step(360.0, 1), b.atm_divergence_damping_3d(360.0),
                                 b.atm_advance_acoustic_step(360.0, 2))),
    ("divergence_damping_3d", lambda b: b.atm_divergence_damping_3d(360.0)),
    ("recover_rk0", lambda b: b.atm_recover_large_step_variables(1, 0, DT)),
    ("recover_rk2", lambda b: b.atm_recover_large_step_variables(2, 2, DT)),
    ("solve_diagnostics_rk0", lambda b: b.atm_compute_solve_diagnostics(False, 0)),
    ("solve_diagnostics_rk2", lambda b: b.atm_compute_solve_diagnostics(False, 2)),
    ("solve_diagnostics_init", lambda b: b.atm_compute_solve_diagnostics(False, -1)),
    ("solve_diagnostics_hollingsworth", lambda b: b.atm_compute_solve_diagnostics(True, 2)),
    ("substep_finish_1_1", lambda b: b.atm_rk_dynamics_substep_finish(1, 1)),
    ("substep_finish_1_3", lambda b: b.atm_rk_dynamics_substep_finish(1, 3)),
    ("substep_finish_2_3", lambda b: b.atm_rk_dynamics_substep_finish(2, 3)),
    ("substep_finish_3_3", lambda b: b.atm_rk_dynamics_substep_finish(3, 3)),
]


@pytest.fixture(scope="module", params=[_abi.INDEX_CORRECTED, _abi.INDEX_LITERAL], ids=["corrected", "literal"])
def warmed(request, grid2562):
    st, ora, g = build_pair(grid2562, L_SMALL, request.param, m5=True)
    _warm(ora, g)
    snap = {n: ora.download_field(n) for (n, _, _) in _abi.FIELDS}
    yield ora, g, snap
    g.close(); ora.close()


@pytest.mark.parametrize("name,fn", TASKS, ids=[t[0] for t in TASKS])
def test_task_parity(warmed, name, fn):
    ora, g, snap = warmed
    for n, a in snap.items():          # same starting state for every task
        ora.upload_field(n, a); g.upload_field(n, a)
    fn(ora); fn(g)
    compare(g, ora, what=name)


@pytest.mark.parametrize("policy", [_abi.INDEX_CORRECTED, _abi.INDEX_LITERAL], ids=["corrected", "literal"])
@pytest.mark.parametrize("rkarg", [_abi.RKARG_STAGE_INDEX, _abi.RKARG_SUBSTEP_TRUNC], ids=["stage_index", "substep_trunc"])
def test_full_step_parity(grid2562, policy, rkarg):
    """one RK3 step after init (atm_core.rg:31 diagnostics + rk_timestep.rg:361-500), then 3 more."""
    st, ora, g = build_pair(grid2562, L_SMALL, policy, m5=True, rkarg=rkarg)
    for b in (ora, g):
        b.atm_compute_solve_diagnostics(False, -1)
        b.atm_srk3(DT)
    compare(g, ora, what="after 1 step")
    for b in (ora, g):
        for _ in range(3):
            b.atm_srk3(DT)
    compare(g, ora, what="after 4 steps")
    g.close(); ora.close()


def test_full_step_memory_model_m1(grid2562):
    """the literal reading: never-written fields are zero (rule M1), literal index policy, literal driver."""
    st, ora, g = build_pair(grid2562, L_SMALL, _abi.INDEX_LITERAL, m5=False, rkarg=_abi.RKARG_SUBSTEP_TRUNC)
    for b in (ora, g):
        b.atm_compute_solve_diagnostics(False, -1)
        b.atm_srk3(DT)
    compare(g, ora, what="M1 literal step")
    g.close(); ora.close()


def test_literal_driver_dt_zero_nan_masks(grid2562):
    """main.rg:66 passes the loop index as dt (Q1): the first step has dts = 0, coef_divdamp = inf,
    inf*0 = NaN in ru_p (dynamics_tasks.rg:1737-1759).  NaN masks must coincide."""
    st, ora, g = build_pair(grid2562, L_SMALL, _abi.INDEX_CORRECTED, m5=True, rkarg=_abi.RKARG_SUBSTEP_TRUNC)
    for b in (ora, g):
        b.atm_compute_solve_diagnostics(False, -1)
        b.atm_srk3(0.0)
        b.atm_srk3(1.0)
    assert np.isnan(ora.download_field("ru_p")).any()
    compare(g, ora, what="dt=0 then dt=1")
    g.close(); ora.close()


def test_by_tasks_equals_driver_and_graph(grid642):
    """the host replay of atm_srk3, the library's driver and its CUDA-graph replay are bit-identical."""
    from mpas_regent_b200 import dynamics, init_jw
    st = init_jw.make_state(grid642, 10, _abi.INDEX_CORRECTED)
    outs = []
    for mode in ("tasks", "driver", "graph"):
        cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, use_graph=int(mode == "graph"))
        g = dynamics.Dynamics(dynamics.dims_of(grid642, 10), cfg)
        g.upload_mesh(st.static); g.upload_state(st.f, st.vert)
        g.atm_compute_solve_diagnostics(False, -1)
        for _ in range(3):
            g.atm_srk3_by_tasks(600.0) if mode == "tasks" else g.atm_srk3(600.0)
        outs.append(g.download_all())
        assert g.launch_count > 0
        g.close()
    for n in outs[0]:
        assert np.array_equal(outs[0][n], outs[1][n], equal_nan=True), n
        assert np.array_equal(outs[0][n], outs[2][n], equal_nan=True), n


def test_sfc_renumbering_is_transparent(grid642):
    """results must not depend on the internal space-filling-curve numbering (bitwise)."""
    from mpas_regent_b200 import dynamics, init_jw
    st = init_jw.make_state(grid642, 10, _abi.INDEX_CORRECTED)
    outs = []
    for sfc in (0, 1):
        g = dynamics.Dynamics(dynamics.dims_of(grid642, 10), _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, sfc_renumber=sfc))
        g.upload_mesh(st.static); g.upload_state(st.f, st.vert)
        g.atm_compute_solve_diagnostics(False, -1)
        g.atm_srk3(600.0); g.atm_srk3(600.0)
        outs.append(g.download_all()); g.close()
    for n in outs[0]:
        assert np.array_equal(outs[0][n], outs[1][n], equal_nan=True), n


def test_vertical_mixing_branches(grid642):
    """config_v_mom_eddy_visc2 / config_v_theta_eddy_visc2 > 0 (dead with the shipped constants,
    dynamics_tasks.rg:1094-1146,1304-1314,1432-1473), both mix_full settings."""
    for mix_full in (0, 1):
        st, ora, g = build_pair(grid642, 12, _abi.INDEX_CORRECTED, config_v_mom_eddy_visc2=30.0,
                                config_v_theta_eddy_visc2=20.0, config_mix_full=mix_full)
        for b in (ora, g):
            b.atm_compute_solve_diagnostics(False, -1)
            b.atm_srk3(600.0)
        compare(g, ora, what=f"vertical mixing, mix_full={mix_full}")
        g.close(); ora.close()


def test_nonfinite_advection_coefficient_takes_the_literal_loop(grid642):
    """w_adv_curv multiplies every advection coefficient of the cell's last edge by an exact 0.0 (dynamics_tasks.rg:1170-1202): the
    kernel leaves those loads out when upload_mesh found every coefficient finite.  One NaN and one Inf coefficient must bring the
    literal loop back -- the NaN pattern they spread over w / tend_w / rw has to be the oracle's."""
    from mpas_regent_b200 import dynamics, init_jw
    from oracle.oracle import Oracle
    L = 12
    st = init_jw.make_state(grid642, L, _abi.INDEX_CORRECTED, m5=True)
    static = dict(st.static)
    ac = np.array(static["adv_coefs"], dtype=np.float64, copy=True); a3 = np.array(static["adv_coefs_3rd"], dtype=np.float64, copy=True)
    n_adv = np.asarray(static["nAdvCellsForEdge"])
    edges = np.flatnonzero(n_adv > 0)
    ac[edges[::7], 0] = np.nan
    a3[edges[3::11], 0] = np.inf
    static["adv_coefs"], static["adv_coefs_3rd"] = ac, a3
    cfg = _abi.default_config(index_policy=_abi.INDEX_CORRECTED, rkarg_policy=_abi.RKARG_STAGE_INDEX)
    ora = Oracle(dynamics.dims_of(grid642, L), cfg)
    g = dynamics.Dynamics(dynamics.dims_of(grid642, L), cfg)
    for b in (ora, g):
        b.upload_mesh(static)
        b.upload_state(st.f, st.vert)
        b.atm_compute_solve_diagnostics(False, -1)
        b.atm_compute_dyn_tend(1, 600.0)            # rk_step > 0: k_dt_cellC<false> evaluates w_adv_curv; nothing else feeds w here
    w = ora.download_field("w")
    bad_cells = np.isnan(w).any(axis=1).sum()
    assert 0 < bad_cells < w.shape[0], "the poisoned coefficients must reach w in some cells of the oracle, not all"
    compare(g, ora, what="non-finite advection coefficients, one dyn_tend")
    for b in (ora, g):
        b.atm_srk3(600.0)
    compare(g, ora, what="non-finite advection coefficients, full step")
    g.close(); ora.close()


def test_strided_region_layout(grid642):
    """upload/download with Legion-style byte strides (x-fastest instance): stride_x = 8, stride_k = 8*n."""
    import ctypes as C
    from mpas_regent_b200 import dynamics, init_jw
    st = init_jw.make_state(grid642, 10, _abi.INDEX_CORRECTED)
    g = dynamics.Dynamics(dynamics.dims_of(grid642, 10), _abi.default_config())
    g.upload_mesh(st.static)
    a = st.f["theta_m"]                      # [n, L1]
    at = np.ascontiguousarray(a.T)           # [L1, n]: x fastest
    n = a.shape[0]
    rc = g._lib.mpasb200_upload_field(g._h, _abi.FIELD_ID["theta_m"], at.ctypes.data, 8, 8 * n)
    assert rc == 0
    assert np.array_equal(g.download_field("theta_m"), a)
    back = np.zeros_like(at)
    rc = g._lib.mpasb200_download_field(g._h, _abi.FIELD_ID["theta_m"], back.ctypes.data, 8, 8 * n)
    assert rc == 0 and np.array_equal(back, at)
    g.close()


def test_error_paths(grid642):
    from mpas_regent_b200 import dynamics
    g = dynamics.Dynamics(dynamics.dims_of(grid642, 10), _abi.default_config())
    with pytest.raises(dynamics.MpasB200Error, match="upload_mesh"):
        g.atm_rk_integration_setup()
    g.close()


@pytest.mark.parametrize("exact", [0, 1, 2, 3, 4], ids=["fused_affine", "two_kernel_exact", "fused_affine_tma", "split_gather_tma", "split_gather_lane_pipeline_default"])
def test_acoustic_modes(grid2562, exact):
    """every evaluation of the acoustic column sweep agrees with the oracle (1e-12); the strictly ordered ones
    (acoustic_exact=1, and the default acoustic_tma=3) are additionally bit-identical on the fields the sweep produces."""
    acoustic_mode_parity(grid2562, exact)


def acoustic_mode_parity(mesh, exact, masks=None):
    st, ora, g = build_pair(mesh, L_SMALL, _abi.INDEX_CORRECTED, m5=True, masks=masks, acoustic_exact=int(exact == 1),
                            acoustic_tma=(exact - 1 if exact >= 2 else 0))
    _warm(ora, g)
    for b in (ora, g):
        for ss, dts in ((0, 360.0), (1, 360.0), (2, 360.0)):
            b.atm_advance_acoustic_step(dts, ss)
            b.atm_divergence_damping_3d(dts)
    compare(g, ora, what=f"acoustic exact={exact}")
    if exact in (1, 4):
        for n in ("rw_p", "rho_pp", "rtheta_pp", "wwAvg", "rtheta_pp_old", "ru_p"):
            assert np.array_equal(g.download_field(n), ora.download_field(n)), n
    g.close(); ora.close()


@pytest.mark.parametrize("policy", [_abi.INDEX_CORRECTED, _abi.INDEX_LITERAL], ids=["corrected", "literal"])
@pytest.mark.parametrize("tiles", [8, 408, 16, 216], ids=["te8_5blocks", "te8_4blocks", "te16_3blocks", "te16_2blocks"])
@pytest.mark.parametrize("levels", [L_SMALL, 55], ids=lambda v: f"L{v}")
def test_edge_tiles_bit_identical(grid2562, tiles, policy, levels):
    """(laboratory build only; measured slower, profiles/r2_edge_tiles.md)  MpasConfig.edge_tiles only changes HOW the edgesOnEdge columns reach k_dt_edge's arithmetic (the distinct columns of a tile of
    edges staged once in shared memory with cp.async.bulk instead of per-thread gathers): every field keeps its bytes on the real mesh
    (pentagons, the last tile partial), under both index policies (LITERAL ids scatter the neighbours: the not-staged fallback runs)."""
    import os
    from mpas_regent_b200 import dynamics, init_jw
    lab = os.path.join(os.path.dirname(dynamics._LIB_PATH), "libmpas_b200_lab.so")
    if not os.path.exists(lab):
        pytest.skip("laboratory build absent (make -C mpas_regent_b200/csrc lab): the tile-staged kernel is not in the shipped library")
    st = init_jw.make_state(grid2562, levels, policy)
    outs = []
    for t in (0, tiles):
        g = dynamics.Dynamics(dynamics.dims_of(grid2562, levels), _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, index_policy=policy, edge_tiles=t), lib_path=lab)
        g.upload_mesh(st.static); g.upload_state(st.f, st.vert)
        g.atm_compute_solve_diagnostics(False, -1)
        for _ in range(2):
            g.atm_srk3(DT)
        g.atm_compute_dyn_tend(1, DT, config_rayleigh_damp_u=True)
        outs.append(g.download_all())
        g.close()
    for n in outs[0]:
        assert np.array_equal(outs[0][n], outs[1][n], equal_nan=True), n


@pytest.mark.parametrize("policy", [_abi.INDEX_CORRECTED, _abi.INDEX_LITERAL], ids=["corrected", "literal"])
@pytest.mark.parametrize("levels", [L_SMALL, 55], ids=lambda v: f"L{v}")
def test_kernel_forms_bit_identical(grid2562, policy, levels):
    """MpasConfig.kernel_forms selects alternative launch forms of the same arithmetic (bit 0: k_dt_cellC as a w launch and a theta
    launch): every field keeps its bytes over two full steps and a mixing / Rayleigh variant of dyn_tend at rk_step 0."""
    from mpas_regent_b200 import dynamics, init_jw
    st = init_jw.make_state(grid2562, levels, policy)
    outs = []
    for forms in (0, 1):
        g = dynamics.Dynamics(dynamics.dims_of(grid2562, levels), _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, index_policy=policy, kernel_forms=forms,
                                                                                      config_v_mom_eddy_visc2=10.0, config_v_theta_eddy_visc2=10.0, config_h_mom_eddy_visc4=1e13, config_h_theta_eddy_visc4=1e13))
        g.upload_mesh(st.static); g.upload_state(st.f, st.vert)
        g.atm_compute_solve_diagnostics(False, -1)
        for _ in range(2):
            g.atm_srk3(DT)
        g.atm_compute_dyn_tend(0, DT, config_rayleigh_damp_u=True)
        outs.append(g.download_all())
        g.close()
    for n in outs[0]:
        assert np.array_equal(outs[0][n], outs[1][n], equal_nan=True), n


@pytest.mark.parametrize("mask", [0, 1, 2, 4, -1], ids=["plain", "dt_edge", "acoustic_gather", "theta_flux", "all"])
def test_staged_gathers_bit_identical(grid2562, mask):
    """(laboratory build only; measured slower, profiles/r2_staged_gathers.md)  MpasConfig.gather_stage only changes HOW neighbour columns reach the arithmetic (cp.async into shared-memory slots
    instead of index -> gather chains): every field keeps its bytes, on the real mesh (pentagons) and with a range set."""
    import os
    from mpas_regent_b200 import dynamics, init_jw
    lab = os.path.join(os.path.dirname(dynamics._LIB_PATH), "libmpas_b200_lab.so")
    if not os.path.exists(lab):
        pytest.skip("laboratory build absent (make -C mpas_regent_b200/csrc lab): the staged kernels are not in the shipped library")
    st = init_jw.make_state(grid2562, L_SMALL, _abi.INDEX_CORRECTED)
    outs = []
    for m in (0, mask):
        g = dynamics.Dynamics(dynamics.dims_of(grid2562, L_SMALL), _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, gather_stage=m), lib_path=lab)
        g.upload_mesh(st.static); g.upload_state(st.f, st.vert)
        g.atm_compute_solve_diagnostics(False, -1)
        for _ in range(2):
            g.atm_srk3(DT)
        g.set_range(_abi.CELL, 100, 1777)
        g.atm_advance_acoustic_step(240.0, 1)
        g.set_range(_abi.CELL)
        outs.append(g.download_all())
        g.close()
    for n in outs[0]:
        assert np.array_equal(outs[0][n], outs[1][n], equal_nan=True), n


@pytest.mark.parametrize("physics,split", [(_abi.PHYSICS_LITERAL, False), (_abi.PHYSICS_CORRECTED, False), (_abi.PHYSICS_LITERAL, True)],
                         ids=["literal", "corrected_physics", "literal_interior_boundary_split"])
def test_emulated_ranks_on_one_gpu_equal_single_partition(grid642, physics, split):
    """4 ranks emulated as 4 handles on one GPU (pack/unpack + the exchange schedule of parallel.exchanges_for):
    owned entities are bit-identical to the single-partition GPU run."""
    from mpas_regent_b200 import init_jw
    emulated_ranks_equal_single_partition(grid642, init_jw.make_state(grid642, 6, _abi.INDEX_CORRECTED), physics, split)


def emulated_ranks_equal_single_partition(mesh, st, physics, split):
    import torch
    from mpas_regent_b200 import dynamics, parallel
    from tests.test_parallel import _task_schedule, _assert_owned_equal
    Lh = st.nVertLevels
    cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, physics_mode=physics)
    exchanges = parallel.exchanges_for(cfg)
    single = dynamics.Dynamics(dynamics.dims_of(mesh, Lh), cfg)
    single.upload_mesh(st.static); single.upload_state(st.f, st.vert)
    single.atm_compute_solve_diagnostics(False, -1)
    shards = parallel.make_shards(st, 4)
    backs = []
    for sh in shards:
        lm = sh["lm"]
        b = dynamics.Dynamics(_abi.make_dims(len(lm.cells), len(lm.edges), len(lm.vertices), Lh), cfg)
        b.upload_mesh(sh["static"]); b.upload_state(sh["f"], sh["vert"])
        backs.append(b)
    # device-side exchange through k_pack / k_unpack and torch buffers (the building blocks NcclExchanger uses, minus the wire)
    lists = {}
    for h, sh in enumerate(shards):
        for ent in ("cell", "edge", "vertex"):
            for peer, idx in sh["lm"].send[ent].items():
                lists[("s", h, ent, peer)] = backs[h].register_list(parallel.ENT[ent], idx)
            for peer, idx in sh["lm"].recv[ent].items():
                lists[("r", h, ent, peer)] = backs[h].register_list(parallel.ENT[ent], idx)

    def exchange(spec):
        for b in backs:
            b.sync()
        for ent, names in spec.items():
            for h, sh in enumerate(shards):
                for o, ridx in sh["lm"].recv[ent].items():
                    buf = torch.empty(len(names) * len(ridx) * (Lh + 1), dtype=torch.float64, device="cuda")
                    backs[o].pack(lists[("s", o, ent, h)], names, buf.data_ptr()); backs[o].sync()
                    backs[h].unpack(lists[("r", h, ent, o)], names, buf.data_ptr()); backs[h].sync()

    for b in backs:
        b.atm_compute_solve_diagnostics(False, -1)
    exchange(exchanges["compute_solve_diagnostics"])
    seq = _task_schedule(cfg)
    CELL, EDGE = parallel.CELL, parallel.EDGE
    if split:      # the schedule of DistributedDynamics._acoustic_pair, with the blocking exchange in place of start()/finish()
        for b, sh in zip(backs, shards):
            lm = sh["lm"]
            c0, c1, c2 = (b.class_range(CELL, c) for c in (0, 1, 2))
            assert c0[0] == 0 and c0[1] == c1[0] and c1[1] == c2[0] == lm.n_owned[0] and c2[1] == len(lm.cells)
            assert c1[1] - c1[0] == len(np.unique(np.concatenate(list(lm.send["cell"].values()))))
            e0, e1 = b.class_range(EDGE, 0), b.class_range(EDGE, 1)
            assert e0[0] == 0 and e0[1] == e1[0] and e1[1] == len(lm.edges)
    for _ in range(2):
        single.atm_srk3(600.0)
        i = 0
        while i < len(seq):
            name, args = seq[i]
            if split and name == "advance_acoustic_step":
                dts = args[0]
                for b in backs:
                    b.set_range(CELL, *b.class_range(CELL, 1)); b._call(name, *args)
                exchange(exchanges[parallel.exchange_key(name, args)])
                for b in backs:
                    b.set_range(CELL, *b.class_range(CELL, 0)); b._call(name, *args)
                    b.set_range(EDGE, *b.class_range(EDGE, 0)); b.atm_divergence_damping_3d(dts)
                    b.set_range(EDGE, *b.class_range(EDGE, 1)); b.atm_divergence_damping_3d(dts)
                    b.set_range(CELL); b.set_range(EDGE)
                assert seq[i + 1][0] == "divergence_damping_3d"
                i += 2
                continue
            for b in backs:
                b._call(name, *args)
            if parallel.exchange_key(name, args) in exchanges:
                exchange(exchanges[parallel.exchange_key(name, args)])
            i += 1
    for b, sh in zip(backs, shards):
        _assert_owned_equal(single, b, sh["lm"])
        b.close()
    single.close()


def test_nccl_ranks_equal_single_gpu():
    """real multi-process run over NCCL when the box has >= 2 GPUs (gpurun --gpus N)."""
    import os
    import subprocess
    import sys
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    n = 2 if n < 4 else 4
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for physics, port in (("literal", "29533"), ("overlap", "29537"), ("corrected", "29535"), ("native", "29539"),
                          ("native_corrected", "29541"), ("native_scalars", "29543")):
        out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr", "127.0.0.1",
                              "--master-port", port, os.path.join(root, "tests", "run_multigpu_check.py"), physics],
                             capture_output=True, text=True, timeout=600, cwd=root)
        assert out.returncode == 0 and "MULTIGPU_OK" in out.stdout, physics + out.stdout[-2000:] + out.stderr[-3000:]


def test_hundred_step_drift(grid2562):
    """100 RK3 steps of the JW-style state (BASELINE.json config 2, at the bundled mesh's size): the deviation from the
    oracle must stay within the stated growth bound 1e-12 * (1 + step) per field."""
    st, ora, g = build_pair(grid2562, 10, _abi.INDEX_CORRECTED, m5=True, rkarg=_abi.RKARG_STAGE_INDEX)
    ora.set_threads(ora.max_threads())
    for b in (ora, g):
        b.atm_compute_solve_diagnostics(False, -1)
    done = 0
    for upto in (1, 10, 100):
        for b in (ora, g):
            for _ in range(upto - done):
                b.atm_srk3(DT)
        done = upto
        worst = compare(g, ora, tol=1e-12 * (1 + upto), what=f"after {upto} steps")
        assert worst[0] <= 1e-12 * (1 + upto)
    g.close(); ora.close()


# ---- MPASB200_PHYSICS_CORRECTED: u update + back-substitution + recover wired (SURVEY.md 8f rank 1) -----------------
CORRECTED_TASKS = [
    ("acoustic_step0", lambda b: b.atm_advance_acoustic_step(240.0, 0)),
    ("acoustic_step1", lambda b: b.atm_advance_acoustic_step(360.0, 1)),
    ("acoustic_loop", lambda b: [(b.atm_advance_acoustic_step(360.0, s), b.atm_divergence_damping_3d(360.0)) for s in range(3)]),
    ("recover_rk0", lambda b: b.atm_recover_large_step_variables(1, 0, DT)),
    ("recover_rk2", lambda b: b.atm_recover_large_step_variables(2, 2, DT)),
    ("acoustic_loop_then_recover", lambda b: ([(b.atm_advance_acoustic_step(360.0, s), b.atm_divergence_damping_3d(360.0)) for s in range(3)],
                                              b.atm_recover_large_step_variables(2, 2, DT))),
]
ACOUSTIC_OUT = ("ru_p", "ruAvg", "rw_p", "wwAvg", "rho_pp", "rtheta_pp", "rtheta_pp_old")


@pytest.fixture(scope="module", params=[_abi.INDEX_CORRECTED, _abi.INDEX_LITERAL], ids=["corrected", "literal"])
def warmed_physics(request, grid2562):
    """state after one LITERAL step (finite everywhere), then both backends switched to CORRECTED physics."""
    st, ora0, _ = build_pair(grid2562, L_SMALL, request.param, m5=True, gpu=False)
    ora0.atm_compute_solve_diagnostics(False, -1)
    ora0.atm_srk3(DT)
    snap = {n: ora0.download_field(n) for (n, _, _) in _abi.FIELDS}
    ora0.close()
    st, ora, g = build_pair(grid2562, L_SMALL, request.param, m5=True, physics_mode=_abi.PHYSICS_CORRECTED)
    yield ora, g, snap
    g.close(); ora.close()


@pytest.mark.parametrize("name,fn", CORRECTED_TASKS, ids=[t[0] for t in CORRECTED_TASKS])
def test_corrected_physics_task_parity(warmed_physics, name, fn):
    ora, g, snap = warmed_physics
    for n, a in snap.items():
        ora.upload_field(n, a); g.upload_field(n, a)
    fn(ora); fn(g)
    compare(g, ora, what="corrected physics " + name)
    if name.startswith("acoustic") and "recover" not in name:
        # the column solve runs strictly in the oracle's order (no FMA contraction): bit-identical
        for n in ACOUSTIC_OUT:
            assert np.array_equal(g.download_field(n), ora.download_field(n), equal_nan=True), n
        assert np.isfinite(ora.download_field("rw_p")).all() and np.abs(ora.download_field("ru_p")).max() > 0


@pytest.mark.parametrize("policy", [_abi.INDEX_CORRECTED, _abi.INDEX_LITERAL], ids=["corrected", "literal"])
def test_corrected_physics_full_step_parity(grid2562, policy):
    """atm_srk3 with the acoustic loop completed and recover called after it (rk_timestep.rg:459-460).  The first step
    stays finite; the reference's remaining quirks (cr.w / cr.theta_m used as tendencies, Q17/Q27) then drive the state
    to Inf/NaN, so the second step checks identical NaN/Inf masks."""
    st, ora, g = build_pair(grid2562, L_SMALL, policy, m5=True, physics_mode=_abi.PHYSICS_CORRECTED)
    u0 = ora.download_field("u")
    for b in (ora, g):
        b.atm_compute_solve_diagnostics(False, -1)
        b.atm_srk3(DT)
    assert np.isfinite(ora.download_field("u")).all() and not np.array_equal(u0, ora.download_field("u"))
    compare(g, ora, what="corrected physics, 1 step")
    for b in (ora, g):
        b.atm_srk3(DT)
    compare(g, ora, what="corrected physics, 2 steps")
    g.close(); ora.close()


def test_corrected_physics_by_tasks_equals_driver_and_graph(grid642):
    from mpas_regent_b200 import dynamics, init_jw
    st = init_jw.make_state(grid642, 10, _abi.INDEX_CORRECTED)
    outs = []
    for mode in ("tasks", "driver", "graph"):
        cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, use_graph=int(mode == "graph"), physics_mode=_abi.PHYSICS_CORRECTED)
        g = dynamics.Dynamics(dynamics.dims_of(grid642, 10), cfg)
        g.upload_mesh(st.static); g.upload_state(st.f, st.vert)
        g.atm_compute_solve_diagnostics(False, -1)
        g.atm_srk3_by_tasks(600.0) if mode == "tasks" else g.atm_srk3(600.0)
        outs.append(g.download_all())
        g.close()
    for n in outs[0]:
        assert np.array_equal(outs[0][n], outs[1][n], equal_nan=True), n
        assert np.array_equal(outs[0][n], outs[2][n], equal_nan=True), n


def test_pipelined_transfers_match_blocking(grid642):
    """mpasb200_upload_field_async / download_field_async / transfer_wait (copy streams + events) give the same bytes as
    the blocking transfers, batch after batch, with the host buffers reused between batches."""
    import torch
    from mpas_regent_b200 import dynamics, init_jw
    Lh = 9
    st = init_jw.make_state(grid642, Lh, _abi.INDEX_CORRECTED)
    names = ("u", "w", "theta_m", "rho_zz", "zb_cell")           # cell, edge and an array-typed field
    outs = ("u", "ru_p", "rtheta_pp", "pv_edge", "vorticity", "zb_cell")
    rng = np.random.default_rng(5)
    batches = [{n: st.f[n] * (1.0 + 1e-3 * rng.standard_normal(st.f[n].shape)) for n in names} for _ in range(3)]
    res = {}
    for mode in ("blocking", "pipelined"):
        g = dynamics.Dynamics(dynamics.dims_of(grid642, Lh), _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX))
        g.upload_mesh(st.static); g.upload_state(st.f, st.vert)
        g.atm_compute_solve_diagnostics(False, -1)
        got = []
        if mode == "blocking":
            for b in batches:
                for n in names:
                    g.upload_field(n, b[n])
                g.atm_srk3(500.0)
                got.append({n: g.download_field(n) for n in outs})
        else:
            hin = {n: torch.empty(g.field_shape(n), dtype=torch.float64).pin_memory() for n in names}
            hout = [{n: torch.empty(g.field_shape(n), dtype=torch.float64).pin_memory() for n in outs} for _ in batches]
            for i, b in enumerate(batches):
                g.transfer_wait() if i else None                 # the input buffers are reused: wait for their copies
                for n in names:
                    hin[n].numpy()[...] = b[n]
                    g.upload_field_async(n, hin[n].numpy())
                g.atm_srk3(500.0)
                for n in outs:
                    g.download_field_async(n, hout[i][n].numpy())
            g.transfer_wait()
            got = [{n: hout[i][n].numpy().copy() for n in outs} for i in range(len(batches))]
        res[mode] = got
        g.close()
    for a, b in zip(res["blocking"], res["pipelined"]):
        for n in outs:
            assert np.array_equal(a[n], b[n], equal_nan=True), n
    assert not np.array_equal(res["blocking"][0]["u"], res["blocking"][1]["u"])


@pytest.mark.parametrize("levels", [4, 30, 58, 100], ids=lambda v: f"L{v}")
def test_level_counts_that_change_the_block_shape(grid642, levels):
    """block = (LP/2, columns per block) is derived from nVertLevels; cover shapes where LP/2 does not divide a warp
    (L=58: 30 pair-threads per column), a very short column (L=4) and a tall column (L=100)."""
    for physics in (_abi.PHYSICS_LITERAL, _abi.PHYSICS_CORRECTED):
        st, ora, g = build_pair(grid642, levels, _abi.INDEX_CORRECTED, m5=True, physics_mode=physics)
        for b in (ora, g):
            b.atm_compute_solve_diagnostics(False, -1)
            b.atm_srk3(300.0)
        compare(g, ora, what=f"L={levels} physics={physics}")
        g.close(); ora.close()


@pytest.mark.parametrize("physics", [_abi.PHYSICS_LITERAL, _abi.PHYSICS_CORRECTED], ids=["literal", "corrected_physics"])
def test_range_restricted_launches_equal_whole(grid642, physics):
    """mpasb200_set_range: the acoustic step on cell ranges and the divergence damping on edge ranges, in any order of
    disjoint ranges that covers everything, give the bytes of the unrestricted launches; launch classes only permute the
    library's internal numbering."""
    from mpas_regent_b200 import init_jw
    range_restricted_launches_equal_whole(grid642, init_jw.make_state(grid642, 9, _abi.INDEX_CORRECTED), physics)


def range_restricted_launches_equal_whole(mesh, st, physics):
    from mpas_regent_b200 import dynamics
    Lh = st.nVertLevels
    cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, physics_mode=physics)
    nC, nE = mesh.nCells, mesh.nEdges
    rng = np.random.default_rng(11)
    outs = []
    for mode in ("whole", "ranges", "classes"):
        static = dict(st.static)
        if mode == "classes":
            static["cellClass"] = rng.integers(0, 3, nC).astype(np.uint8)
            static["edgeClass"] = rng.integers(0, 2, nE).astype(np.uint8)
        g = dynamics.Dynamics(dynamics.dims_of(mesh, Lh), cfg)
        g.upload_mesh(static); g.upload_state(st.f, st.vert)
        g.atm_compute_solve_diagnostics(False, -1)
        g.atm_srk3(500.0)                               # populate everything
        if mode == "whole":
            cuts_c, cuts_e = [(0, nC)], [(0, nE)]
        elif mode == "ranges":
            cuts_c, cuts_e = [(nC // 3, nC), (0, 5), (5, nC // 3), (7, 7)], [(100, nE), (0, 100)]
        else:
            cuts_c = [g.class_range(parallel_CELL, c) for c in (2, 0, 1)]
            cuts_e = [g.class_range(parallel_EDGE, c) for c in (1, 0)]
            assert sum(e - b for b, e in cuts_c) == nC and sum(e - b for b, e in cuts_e) == nE
            assert g.class_range(parallel_CELL, 1)[1] - g.class_range(parallel_CELL, 1)[0] == int((static["cellClass"] == 1).sum())
        for ss in range(3):
            if physics == _abi.PHYSICS_CORRECTED:      # the edge update precedes the cell part: edges first, one range at a time
                for be in cuts_e:
                    g.set_range(parallel_EDGE, *be); g.set_range(parallel_CELL, 0, 0); g.atm_advance_acoustic_step(360.0, ss)
                g.set_range(parallel_EDGE, 0, 0)
            for bc in cuts_c:
                g.set_range(parallel_CELL, *bc); g.atm_advance_acoustic_step(360.0, ss)
            g.set_range(parallel_CELL); g.set_range(parallel_EDGE)
            for be in cuts_e:
                g.set_range(parallel_EDGE, *be); g.atm_divergence_damping_3d(360.0)
            g.set_range(parallel_EDGE)
        outs.append(g.download_all())
        g.close()
    for n in outs[0]:
        assert np.array_equal(outs[0][n], outs[1][n], equal_nan=True), ("ranges", n)
        assert np.array_equal(outs[0][n], outs[2][n], equal_nan=True), ("classes", n)


from mpas_regent_b200._abi import CELL as parallel_CELL, EDGE as parallel_EDGE  # noqa: E402


# ---- atm_advance_scalars (SURVEY.md 8a row a11 / 8f rank 2; absent from the reference, parity unpinned) ---------------------
@pytest.mark.parametrize("policy", [_abi.INDEX_CORRECTED, _abi.INDEX_LITERAL], ids=["corrected", "literal"])
def test_advance_scalars_parity(grid2562, policy):
    """the task alone on a state where everything it reads is non-trivial, then the driver with config_scalar_advection on
    (setup saves scalars_old, every RK stage advances; rk_timestep.rg:465), plain and as a CUDA graph: bit-identical."""
    advance_scalars_parity(grid2562, policy)


def advance_scalars_parity(mesh, policy, masks=None):
    st, ora, g = build_pair(mesh, L_SMALL, policy, m5=True, masks=masks, config_scalar_advection=1)
    _warm(ora, g)
    rng = np.random.default_rng(9)
    nC = mesh.nCells
    q = 1e-3 * (1.0 + rng.random((nC, L_SMALL + 1, 8))); q_old = 1e-3 * (1.0 + rng.random((nC, L_SMALL + 1, 8)))
    ru = ora.download_field("ru") + 0.3 * rng.standard_normal((mesh.nEdges, L_SMALL + 1))
    ww = 0.05 * rng.standard_normal((nC, L_SMALL + 1))
    for b in (ora, g):
        for n, a in (("scalars", q), ("scalars_old", q_old), ("ruAvg", ru), ("wwAvg", ww)):
            b.upload_field(n, a)
        b.atm_advance_scalars(240.0, 0)
        b.atm_advance_scalars(720.0, 2)
    a, b_ = g.download_field("scalars"), ora.download_field("scalars")
    assert not np.array_equal(b_, q)
    assert np.array_equal(a, b_), float(np.abs(a - b_).max())
    for b in (ora, g):
        b.atm_srk3(DT); b.atm_srk3(DT)
    compare(g, ora, what="2 steps with scalar advection")
    assert np.array_equal(g.download_field("scalars"), ora.download_field("scalars"))
    assert np.array_equal(g.download_field("scalars_old"), ora.download_field("scalars_old"))
    g.set_use_graph(True)
    for b in (ora, g):
        b.atm_srk3(DT)
    assert np.array_equal(g.download_field("scalars"), ora.download_field("scalars"))
    g.close(); ora.close()


@pytest.mark.parametrize("levels", [4, 26, 30, 55, 58, 100], ids=lambda v: f"L{v}")
def test_acoustic_lane_pipeline_shapes(grid642, levels):
    """k_acoustic_lane (acoustic_tma = 3, the default: sweeper warp + mover warps, 8-level chunks, 32-column tiles): partial last chunk,
    partial last tile, level counts around the chunk size, a restricted cell range, spec-zone columns -- bit-identical
    acoustic outputs, full state inside the bound."""
    st, ora, g = build_pair(grid642, levels, _abi.INDEX_CORRECTED, m5=True, acoustic_tma=3)
    spec = np.zeros(grid642.nCells); spec[5::37] = 1.0
    ora.close(); g.close()
    st.static["specZoneMaskCell"] = spec
    from mpas_regent_b200 import dynamics
    from oracle.oracle import Oracle
    cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, acoustic_tma=3)
    ora = Oracle(dynamics.dims_of(grid642, levels), cfg); g = dynamics.Dynamics(dynamics.dims_of(grid642, levels), cfg)
    for b in (ora, g):
        b.upload_mesh(st.static); b.upload_state(st.f, st.vert)
        b.atm_compute_solve_diagnostics(False, -1)
        b.atm_srk3(300.0)
    compare(g, ora, what=f"L={levels}")
    for n in ACOUSTIC_OUT[2:]:
        assert np.array_equal(g.download_field(n), ora.download_field(n), equal_nan=True), n
    # a restricted range: cells [37, 301) only
    snap = {n: ora.download_field(n) for n in ACOUSTIC_OUT[2:]}
    g.set_range(_abi.CELL, 37, 301)
    g.atm_advance_acoustic_step(100.0, 1)
    ora.atm_advance_acoustic_step(100.0, 1)
    for n in ACOUSTIC_OUT[2:]:
        a, full = g.download_field(n), ora.download_field(n)
        lo, hi = g.class_range(_abi.CELL, 0)      # no classes: internal order == the curve; compare through the untouched set instead
        touched = ~np.all(a == snap[n], axis=1)
        assert touched.sum() <= 301 - 37, n
        assert np.array_equal(a[touched], full[touched], equal_nan=True), n
    g.close(); ora.close()


def test_strided_mesh_members_equal_dense_upload(grid642):
    """mpasb200_mesh_member + mpasb200_upload_mesh_staged (the Legion-instance form: one array per x with a byte stride between x,
    level 0 of a 2-D region) build the same mirror as the dense mpasb200_upload_mesh."""
    import ctypes as C
    from mpas_regent_b200 import dynamics, init_jw
    L = 8
    st = init_jw.make_state(grid642, L, _abi.INDEX_CORRECTED)
    cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX)
    outs = []
    for staged in (False, True):
        g = dynamics.Dynamics(dynamics.dims_of(grid642, L), cfg)
        if not staged:
            g.upload_mesh(st.static)
        else:
            keep = []
            for name, dt, ent, wkey in _abi.MESH_MEMBERS:
                a = st.static.get(name)
                if a is None:
                    continue
                a = np.ascontiguousarray(a, dtype=dt).reshape(a.shape[0], -1)
                pad = np.zeros((a.shape[0], a.shape[1] + 3), dtype=dt)            # a wider instance: byte stride > row size
                pad[:, :a.shape[1]] = a
                keep.append(pad)
                rc = g._lib.mpasb200_mesh_member(g._h, name.encode(), pad.ctypes.data, pad.strides[0])
                assert rc == 0, name
            assert g._lib.mpasb200_mesh_member(g._h, b"noSuchMember", keep[0].ctypes.data, 8) != 0
            assert g._lib.mpasb200_upload_mesh_staged(g._h) == 0
        g.upload_state(st.f, st.vert)
        g.atm_compute_solve_diagnostics(False, -1)
        g.atm_srk3(600.0)
        outs.append(g.download_all()); g.close()
    for n in outs[0]:
        assert np.array_equal(outs[0][n], outs[1][n], equal_nan=True), n


@pytest.mark.parametrize("policy", [_abi.INDEX_CORRECTED, _abi.INDEX_LITERAL], ids=["corrected", "literal"])
def test_init_chain_on_the_device(grid2562, policy):
    """SURVEY.md 8f rank 3: atm_init_coupled_diagnostics (dynamics_tasks.rg:651-725) and mpas_reconstruct_2d (:1894-1948) as
    device kernels: 1e-12 against the oracle (the two pow() calls are the only non-exact operations), everything else bitwise."""
    st, ora, g = build_pair(grid2562, L_SMALL, policy, m5=True)
    for b in (ora, g):
        b.atm_init_coupled_diagnostics()
        b.mpas_reconstruct_2d(False, True)
    compare(g, ora, what="init chain")
    for n in ("rho_zz", "ru", "rw", "rho_p", "rtheta_base", "rtheta_p", "uReconstructX", "uReconstructY", "uReconstructZ",
              "uReconstructZonal", "uReconstructMeridional"):
        assert np.array_equal(g.download_field(n), ora.download_field(n), equal_nan=True), n
    for b in (ora, g):
        b.mpas_reconstruct_2d(False, False)
    for n in ("uReconstructZonal", "uReconstructMeridional"):
        assert np.array_equal(g.download_field(n), ora.download_field(n), equal_nan=True), n
    g.close(); ora.close()


@pytest.mark.parametrize("policy", [_abi.INDEX_CORRECTED, _abi.INDEX_LITERAL], ids=["corrected", "literal"])
@pytest.mark.parametrize("which", ["x1.2562", "icosa642"])
def test_mesh_only_init_producers_on_the_device(grid2562, grid642, policy, which):
    """SURVEY.md 8f rank 3: atm_compute_signs (dynamics_tasks.rg:46-130), atm_adv_coef_compression (:133-269) and
    atm_couple_coef_3rd_order (:303-325) as device kernels, through the C ABI with the RAW stored ids: integer lists, signs and
    coefficients are bit-identical to the oracle's literal loops (and therefore to what the host chain fed every other test)."""
    mesh_only_init_producers_equal_oracle(grid2562 if which == "x1.2562" else grid642, policy)


def mesh_only_init_producers_equal_oracle(mesh, policy):
    from mpas_regent_b200 import dynamics, init_jw
    from oracle.oracle import Oracle
    from tests.test_core_init import _raw_mesh
    st = init_jw.make_state(mesh, L_SMALL, policy)
    raw = _raw_mesh(mesh, st.mesh, st.extras["deriv_two"])
    cfg = _abi.default_config(index_policy=policy)
    g = dynamics.Dynamics(dynamics.dims_of(mesh, L_SMALL), cfg)
    ora = Oracle(dynamics.dims_of(mesh, L_SMALL), cfg)
    sg, so = g.atm_compute_signs(raw), ora.atm_compute_signs(raw)           # before upload_mesh: their outputs feed it
    for k in so:
        assert np.array_equal(sg[k], so[k]), k
        assert np.array_equal(sg[k], st.static[k]), k
    ag, ao = g.atm_adv_coef_compression(raw), ora.atm_adv_coef_compression(raw)
    for k in ao:
        assert np.array_equal(ag[k], ao[k]), k
    raw0 = dict(raw); raw0.pop("deriv_two")                                  # deriv_two never written upstream: null = zeros
    a0g, a0o = g.atm_adv_coef_compression(raw0), ora.atm_adv_coef_compression(raw0)
    for k in a0o:
        assert np.array_equal(a0g[k], a0o[k]), k
    for b in (g, ora):
        b.upload_mesh(st.static)
        b.upload_field("zb", st.extras["zb"]); b.upload_field("zb3", st.extras["zb3"])
        b.atm_compute_zb_cell()
    a3g, a3o = ag["adv_coefs_3rd"].copy(), ao["adv_coefs_3rd"].copy()
    g.atm_couple_coef_3rd_order(0.25, a3g); ora.atm_couple_coef_3rd_order(0.25, a3o)
    assert np.array_equal(a3g, a3o) and np.array_equal(a3g, st.static["adv_coefs_3rd"])
    for n in ("zb_cell", "zb3_cell"):
        assert np.array_equal(g.download_field(n), ora.download_field(n)), n
        assert np.array_equal(g.download_field(n), st.f[n]), n
    g.close(); ora.close()


@pytest.mark.parametrize("which,levels", [("x1.2562", L_SMALL), ("icosa642", 55), ("icosa642", 10)], ids=["x1.2562_L26", "icosa642_L55", "icosa642_L10"])
def test_init_atm_case_jw_on_the_device(grid2562, grid642, which, levels):
    """SURVEY.md 8f rank 3: init_atm_case_jw (vertical_init/init_atm_cases.rg:24-743) as device kernels -- the corrected reading,
    compared field by field with the host generator (mpas_regent_b200/init_jw.py, what every parity test is fed by): 1e-12 of the
    field's largest value (libm and the device differ in the last place of exp / pow / sin / cos; rw and w also in the order the
    edge terms are summed), vertical-grid arrays included; then the whole atm_core_init chain on the device reproduces the inputs."""
    from mpas_regent_b200 import dynamics, init_jw
    mesh = grid2562 if which == "x1.2562" else grid642
    st = init_jw.make_state(mesh, levels, _abi.INDEX_CORRECTED, m5=False, keep_jw=True)
    g = dynamics.Dynamics(dynamics.dims_of(mesh, levels), _abi.default_config())
    g.upload_mesh(st.static)
    v = st.mesh.v
    g.init_atm_case_jw(v["latCell"], v["areaCell"], v["latVertex"])
    worst = {}
    for n, ref in list(st.extras["jw"].items()) + [(k, st.vert[k]) for k in ("rdzw", "rdzu", "fzm", "fzp", "cf1", "cf2", "cf3")]:
        a = g.download_field(n)
        scale = np.abs(ref).max()
        if n in ("rw", "w"):
            # rw is a sum of edge terms zzf * zb * (fzm ru + fzp ru) that cancel to ~1e-4 of their size (an almost balanced flow over
            # smooth terrain): the honest scale of its rounding error is the size of the terms, not of the sum
            jw = st.extras["jw"]
            scale = np.abs(jw["zz"]).max() * np.abs(jw["zb"]).max() * np.abs(jw["ru"]).max() * 2.0
            if n == "w":
                scale /= jw["rho_zz"][:, :levels].min()
        err = np.abs(a - ref).max()
        worst[n] = err / scale if scale > 0 else err
        assert np.isfinite(a).all(), n
        assert err <= 1e-12 * scale if scale > 0 else err == 0.0, (n, err, scale)
    assert not g.download_field("zb3").any()
    # the rest of atm_core_init on the device: zb_cell, coupled diagnostics -> the state the host chain produces
    g.atm_compute_zb_cell()
    g.upload_field("rho_zz", g.download_field("rho_zz") * g.download_field("zz"))     # the chain starts from the uncoupled density (:674)
    g.atm_init_coupled_diagnostics()
    for n in ("zb_cell", "zb3_cell", "rho_zz", "ru", "rw", "rho_p", "rtheta_base", "rtheta_p", "exner", "exner_base", "pressure_p"):
        a, ref = g.download_field(n), st.f[n]
        scale = np.abs(ref).max()
        if n == "rw":       # same cancellation: w * rho * zz against the edge terms zb_cell * ru * zz
            scale = max(scale, np.abs(st.f["zz"]).max() * np.abs(st.f["zb_cell"]).max() * np.abs(st.f["ru"]).max() * 2.0)
        assert np.abs(a - ref).max() <= 2e-12 * max(scale, 1e-300), (n, np.abs(a - ref).max(), scale)
    print("worst relative deviations:", {k: f"{x:.1e}" for k, x in worst.items()})
    g.close()


@pytest.mark.parametrize("policy", [_abi.INDEX_CORRECTED, _abi.INDEX_LITERAL], ids=["corrected", "literal"])
def test_mesh_scaling_and_damping_coefs_on_the_device(grid2562, policy):
    """atm_compute_mesh_scaling (dynamics_tasks.rg:595-646) and atm_compute_damping_coefs (:274-300) as device kernels against the
    oracle's loops on a non-uniform meshDensity: 1e-12 (one pow / sin each)."""
    from mpas_regent_b200 import dynamics, init_jw
    from oracle.oracle import Oracle
    st = init_jw.make_state(grid2562, L_SMALL, policy)
    md = np.random.default_rng(5).uniform(0.05, 1.0, grid2562.nCells)
    cfg = _abi.default_config(index_policy=policy)
    g, ora = dynamics.Dynamics(dynamics.dims_of(grid2562, L_SMALL), cfg), Oracle(dynamics.dims_of(grid2562, L_SMALL), cfg)
    raw = {"cellsOnEdge": grid2562.v["cellsOnEdge"]}
    a, b = g.atm_compute_mesh_scaling(raw, md, True), ora.atm_compute_mesh_scaling(raw, md, True)
    for k in b:
        assert np.allclose(a[k], b[k], rtol=1e-12, atol=0), k
    a1 = g.atm_compute_mesh_scaling(raw, md, False)
    assert (a1["meshScalingDel2"] == 1.0).all() and (a1["meshScalingDel4"] == 1.0).all()
    for x in (g, ora):
        x.upload_mesh(st.static); x.upload_field("zgrid", st.f["zgrid"])
        x.atm_compute_damping_coefs(md, 22000.0, 0.2)
    da, db = g.download_field("dss"), ora.download_field("dss")
    assert db.max() > 0 and np.allclose(da, db, rtol=1e-12, atol=0)
    g.close(); ora.close()
