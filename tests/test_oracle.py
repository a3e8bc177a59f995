"""The CPU oracle: pinned against the only observables the reference offers (SURVEY.md 8c) and
against hand-checkable properties of the task bodies."""
import numpy as np
import pytest

from mpas_regent_b200 import _abi, dynamics, init_jw
from tests.util import build_pair

L = 8


@pytest.fixture(scope="module")
def pair(grid642):
    st, ora, _ = build_pair(grid642, L, _abi.INDEX_CORRECTED, gpu=False)
    ora.atm_compute_solve_diagnostics(False, -1)
    yield st, ora
    ora.close()


def test_output_txt_observable_u_never_changes(grid2562):
    """output.txt prints er[{0,0}].u after every RK stage of 10 steps and it never changes: nothing on
    the shipped path writes u (acoustic u-update commented out :1585-1613, recover not called,
    rk_timestep.rg:460).  With the literal driver dt = step index (main.rg:66)."""
    st, ora, _ = build_pair(grid2562, 5, _abi.INDEX_LITERAL, m5=False, gpu=False, rkarg=_abi.RKARG_SUBSTEP_TRUNC)
    u0 = ora.download_field("u").copy()
    ora.atm_compute_solve_diagnostics(False, -1)
    for j in range(3):
        ora.atm_srk3(float(j))
    assert np.array_equal(ora.download_field("u"), u0)
    assert np.array_equal(ora.download_field("theta_m"), st.f["theta_m"])
    ora.close()


def test_setup_and_finish_are_copies(pair):
    st, ora = pair
    ora.atm_rk_integration_setup()
    for a, b in (("ru_save", "ru"), ("u_2", "u"), ("rw_save", "rw"), ("w_2", "w"), ("rho_zz_old_split", "rho_zz")):
        x, y = ora.download_field(a), ora.download_field(b)
        assert np.array_equal(x[:, :L], y[:, :L])
        assert not x[:, L].any()            # level nVertLevels is outside every hot-path loop


def test_moist_coefficients(pair):
    st, ora = pair
    ora.atm_compute_moist_coefficients()
    cqw = ora.download_field("cqw")
    assert np.all(cqw[:, 1:L] == 1.0) and np.all(cqw[:, 0] == 0.0)
    assert not ora.download_field("qtot").any()


def test_vert_imp_coefs_uses_previous_gamma(pair):
    """alpha_tri(k) reads gamma_tri(k-1) from the PREVIOUS call (:580-591), so two identical calls differ."""
    st, ora = pair
    ora.atm_compute_moist_coefficients()
    ora.upload_field("gamma_tri", np.zeros(ora.field_shape("gamma_tri")))
    ora.atm_compute_vert_imp_coefs(240.0)
    a1, b, g1 = ora.download_field("alpha_tri"), ora.download_field("b_tri"), ora.download_field("gamma_tri")
    assert np.allclose(a1[:, 1:L], 1.0 / b[:, 1:L], rtol=0, atol=0)        # gamma was all zero
    ora.atm_compute_vert_imp_coefs(240.0)
    a2 = ora.download_field("alpha_tri")
    a_tri = ora.download_field("a_tri")
    expect = 1.0 / (b[:, 2:L] - a_tri[:, 2:L] * g1[:, 1:L - 1])
    assert np.array_equal(a2[:, 2:L], expect)
    cofrz = ora.download_field("cofrz")
    assert np.array_equal(cofrz[:L], 0.5 * 240.0 * 1.1 * st.vert["rdzw"][:L])


def test_divergence_is_s_plus_u(pair, grid642):
    """Q6: divergence accumulates s + u, not s * u (:375)."""
    st, ora = pair
    from mpas_regent_b200.mesh import resolve_ids
    ora.atm_compute_solve_diagnostics(False, 0)
    div = ora.download_field("divergence")
    u = ora.download_field("u")
    S = st.static
    eoc = resolve_ids(S["edgesOnCell"], grid642.nEdges, _abi.INDEX_CORRECTED)
    c, k = 17, 3
    acc = 0.0
    for i in range(S["nEdgesOnCell"][c]):
        e = eoc[c, i]
        acc += S["edgesOnCellSign"][c, i] * S["dvEdge"][e] + u[e, k]
    assert div[c, k] == acc * S["invAreaCell"][c]


def test_v_only_on_stage_2_or_init(pair):
    st, ora = pair
    ora.upload_field("v", np.full(ora.field_shape("v"), 7.0))
    ora.atm_compute_solve_diagnostics(False, 0)
    assert np.all(ora.download_field("v") == 7.0)
    ora.atm_compute_solve_diagnostics(False, 2)
    assert not np.all(ora.download_field("v")[:, :L] == 7.0)


def test_srk3_call_sequence_counts(pair):
    """2 / 2 / 3 acoustic iterations per stage (rk_timestep.rg:450, output.txt)."""
    st, ora = pair
    calls = []
    ora.atm_srk3_by_tasks(600.0, hook=lambda name, *a: calls.append(name))
    assert calls.count("advance_acoustic_step") == 7 and calls.count("divergence_damping_3d") == 7
    assert calls.count("compute_dyn_tend") == 3 and calls.count("compute_vert_imp_coefs") == 2
    assert calls.count("compute_solve_diagnostics") == 3 and calls[-1] == "rk_dynamics_substep_finish"


def test_by_tasks_equals_driver(grid642):
    outs = []
    for mode in (0, 1):
        st, ora, _ = build_pair(grid642, L, _abi.INDEX_CORRECTED, gpu=False)
        ora.atm_compute_solve_diagnostics(False, -1)
        (ora.atm_srk3 if mode else ora.atm_srk3_by_tasks)(600.0)
        outs.append(ora.download_all()); ora.close()
    for n in outs[0]:
        assert np.array_equal(outs[0][n], outs[1][n], equal_nan=True), n


def test_threads_do_not_change_results(grid642):
    outs = []
    for t in (1, 4):
        st, ora, _ = build_pair(grid642, L, _abi.INDEX_CORRECTED, gpu=False)
        ora.set_threads(t)
        ora.atm_compute_solve_diagnostics(False, -1)
        ora.atm_srk3(600.0)
        outs.append(ora.download_all()); ora.close()
    for n in outs[0]:
        assert np.array_equal(outs[0][n], outs[1][n], equal_nan=True), n


def test_recover_writes_the_garbage_cell(pair):
    st, ora = pair
    ora.atm_recover_large_step_variables(1, 0, 600.0)
    assert np.all(ora.download_pad("rho_zz")[:L] == 1.0)                  # :1792-1794


# ---- MPASB200_PHYSICS_CORRECTED (SURVEY.md 8f rank 1): the three disabled pieces enabled ----------------------------
def _numpy_acoustic_corrected(st, f, vert, cfg, dts, small_step):
    """Independent array-at-a-time restatement of the corrected acoustic step (edge update :1581-1613, column-phased
    cell part :1615-1704 with the back-substitution :1674-1677) used to pin the oracle's loop form."""
    s = st.static
    nC, nE = s["nEdgesOnCell"].shape[0], s["cellsOnEdge"].shape[0]
    Lv = f["theta_m"].shape[1] - 1
    pad = lambda a: np.vstack([a, np.zeros((1,) + a.shape[1:])])
    idx = lambda ids, n: np.where(ids > 0, ids - 1, n)             # INDEX_CORRECTED: id-1, 0 -> pad entity
    c1, c2 = idx(s["cellsOnEdge"][:, 0], nC), idx(s["cellsOnEdge"][:, 1], nC)
    K = slice(0, Lv)
    epssm, rgas, cp, g = cfg.config_epssm, cfg.rgas, cfg.cp, cfg.gravity
    rcv = rgas / (cp - rgas); cc2 = cp * rcv; resm = (1.0 - epssm) / (1.0 + epssm)
    o = {k: f[k].copy() for k in ("ru_p", "ruAvg", "rw_p", "wwAvg", "rho_pp", "rtheta_pp", "rtheta_pp_old")}
    if small_step != 0:
        rpp, zz, ex, rho = pad(f["rtheta_pp"])[:, K], pad(f["zz"])[:, K], pad(f["exner"])[:, K], pad(f["rho_pp"])[:, K]
        pgrad = ((rpp[c2] - rpp[c1]) * s["invDcEdge"][:, None]) / (0.5 * (zz[c2] + zz[c1]))
        pgrad = pgrad * (f["cqu"][:, K] * 0.5 * cc2 * (ex[c1] + ex[c2]))
        pgrad = pgrad + 0.5 * f["zxu"][:, K] * g * (rho[c1] + rho[c2])
        o["ru_p"][:, K] = f["ru_p"][:, K] + dts * (f["tend_ru"][:, K] - (1.0 - s["specZoneMaskEdge"][:, None]) * pgrad)
        o["ruAvg"][:, K] = f["ruAvg"][:, K] + o["ru_p"][:, K]
    else:
        o["ru_p"][:, K] = dts * f["tend_ru"][:, K]
        o["ruAvg"][:, K] = o["ru_p"][:, K]
    rw_p, ww, rho_pp, rt_pp = o["rw_p"], o["wwAvg"], o["rho_pp"], o["rtheta_pp"]
    o["rtheta_pp_old"][:, K] = 0.0 if small_step == 0 else f["rtheta_pp"][:, K]
    if small_step == 0:
        rw_p[:] = 0; ww[:] = 0; rho_pp[:, K] = 0; rt_pp[:, K] = 0
    spec = s["specZoneMaskCell"] != 0.0
    before = [a[spec][:, K].copy() for a in (rho_pp, rt_pp, rw_p, ww)]
    rs, ts = np.zeros((nC, Lv)), np.zeros((nC, Lv))
    rup, tm = pad(o["ru_p"])[:, K], pad(f["theta_m"])[:, K]
    for i in range(s["edgesOnCell"].shape[1]):
        on = (i < s["nEdgesOnCell"])[:, None]
        e = idx(s["edgesOnCell"][:, i], nE)
        flux = s["edgesOnCellSign"][:, i][:, None] * dts * pad(s["dvEdge"][:, None])[e] * rup[e] * s["invAreaCell"][:, None]
        ec1, ec2 = np.append(c1, nC)[e], np.append(c2, nC)[e]
        rs = np.where(on, rs - flux, rs)
        ts = np.where(on, ts - flux * 0.5 * (tm[ec2] + tm[ec1]), ts)
    cofrz, rdzw, fzm, fzp = (vert[k][K] for k in ("cofrz", "rdzw", "fzm", "fzp"))
    coftz = f["coftz"]
    rs = rho_pp[:, K] + dts * f["tend_rho"][:, K] + rs - cofrz * resm * (rw_p[:, 1:] - rw_p[:, :-1])
    ts = rt_pp[:, K] + dts * f["theta_m"][:, K] + ts - resm * rdzw * (coftz[:, 1:] * rw_p[:, 1:] - coftz[:, :-1] * rw_p[:, :-1])
    k, m = slice(1, Lv), slice(0, Lv - 1)
    zz, w = f["zz"], f["w"]
    ww[:, k] += 0.5 * (1.0 - epssm) * rw_p[:, k]
    rw_p[:, k] += (dts * w[:, k] - f["cofwz"][:, k] * ((zz[:, k] * ts[:, k] - zz[:, m] * ts[:, m]) + resm * (zz[:, k] * rt_pp[:, k] - zz[:, m] * rt_pp[:, m]))
                   - f["cofwr"][:, k] * ((rs[:, k] + rs[:, m]) + resm * (rho_pp[:, k] + rho_pp[:, m]))
                   + f["cofwt"][:, k] * (ts[:, k] + resm * rt_pp[:, k])
                   + f["cofwt"][:, m] * (ts[:, m] + resm * rt_pp[:, m]))
    for kk in range(1, Lv):
        rw_p[:, kk] = (rw_p[:, kk] - f["a_tri"][:, kk] * rw_p[:, kk - 1]) * f["alpha_tri"][:, kk]
    for kk in range(Lv - 1, -1, -1):
        rw_p[:, kk] = rw_p[:, kk] - f["gamma_tri"][:, kk] * rw_p[:, kk + 1]
    d3 = f["rw_save"][:, k] - f["rw"][:, k]
    x = rw_p[:, k] + (d3 - dts * f["dss"][:, k] * (fzm[k] * zz[:, k] + fzp[k] * zz[:, m]) * (fzm[k] * f["rho_zz"][:, k] + fzp[k] * f["rho_zz"][:, m]) * w[:, k])
    x = x / (1.0 + dts * f["dss"][:, k])
    rw_p[:, k] = x - d3
    ww[:, k] += 0.5 * (1.0 + epssm) * rw_p[:, k]
    rho_pp[:, K] = rs - cofrz * (rw_p[:, 1:] - rw_p[:, :-1])
    rt_pp[:, K] = ts - rdzw * (coftz[:, 1:] * rw_p[:, 1:] - coftz[:, :-1] * rw_p[:, :-1])
    # specified-zone columns only integrate their tendencies, every level from 0 (:1698-1703)
    rho_pp[spec, K] = before[0] + dts * f["tend_rho"][spec][:, K]
    rt_pp[spec, K] = before[1] + dts * f["theta_m"][spec][:, K]
    rw_p[spec, K] = before[2] + dts * w[spec][:, K]
    ww[spec, K] = before[3] + 0.5 * (1.0 + epssm) * rw_p[spec][:, K]
    return o


@pytest.mark.parametrize("small_step", [0, 1])
def test_corrected_physics_acoustic_step_matches_array_restatement(grid642, small_step):
    check_corrected_acoustic_restatement(grid642, small_step)


def check_corrected_acoustic_restatement(mesh, small_step, masks=None):
    st, lit, _ = build_pair(mesh, L, _abi.INDEX_CORRECTED, gpu=False, masks=masks)
    lit.atm_compute_solve_diagnostics(False, -1)
    lit.atm_srk3(600.0)                                    # a finite, fully populated state
    pre = lit.download_all(); lit.close()
    st, ora, _ = build_pair(mesh, L, _abi.INDEX_CORRECTED, gpu=False, masks=masks, physics_mode=_abi.PHYSICS_CORRECTED)
    for n, a in pre.items():
        ora.upload_field(n, a)
    ora.atm_advance_acoustic_step(300.0, small_step)
    want = _numpy_acoustic_corrected(st, pre, {k: pre[k] for k in ("cofrz", "rdzw", "fzm", "fzp")}, ora.cfg, 300.0, small_step)
    for n, a in want.items():
        got = ora.download_field(n)
        assert np.isfinite(got).all(), n
        scale = np.abs(a).max()
        assert np.abs(got - a).max() <= 1e-13 * scale, (n, np.abs(got - a).max(), scale)
    assert np.abs(want["ru_p"]).max() > 0 and np.abs(want["rw_p"]).max() > 0
    ora.close()


def test_corrected_physics_u_evolves_and_recover_is_called(grid642):
    """the LITERAL observable (u never changes) is exactly what CORRECTED removes; one step stays finite."""
    st, ora, _ = build_pair(grid642, L, _abi.INDEX_CORRECTED, gpu=False, physics_mode=_abi.PHYSICS_CORRECTED)
    calls = []
    orig = ora._call
    ora._call = lambda name, *a: (calls.append(name), orig(name, *a))[1]
    u0 = ora.download_field("u").copy()
    ora.atm_compute_solve_diagnostics(False, -1)
    ora.atm_srk3_by_tasks(600.0)
    assert calls.count("recover_large_step_variables") == 3
    by_tasks = ora.download_all()
    assert all(np.isfinite(by_tasks[n]).all() for n in ("u", "w", "theta_m", "rho_zz", "ru", "rw"))
    assert not np.array_equal(by_tasks["u"], u0)
    assert np.all(ora.download_pad("rho_zz")[:L] == 1.0)
    ora.close()
    st, ora2, _ = build_pair(grid642, L, _abi.INDEX_CORRECTED, gpu=False, physics_mode=_abi.PHYSICS_CORRECTED)
    ora2.atm_compute_solve_diagnostics(False, -1)
    ora2.atm_srk3(600.0)
    for n, a in by_tasks.items():
        assert np.array_equal(a, ora2.download_field(n), equal_nan=True), n
    ora2.close()
