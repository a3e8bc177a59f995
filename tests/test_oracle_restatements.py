"""A second, array-at-a-time restatement (numpy, one level or one edge slot at a time) of four task bodies, written from the
reference text and independent of oracle/mpas_oracle.cpp's loop form.  It pins the oracle against transcription slips:
both must agree to rounding (1e-13 relative).  Memory-model rules as in the oracle header (M1-M4, level -1 reads 0)."""
import numpy as np
import pytest

from mpas_regent_b200 import _abi, dynamics
from tests.util import build_pair

L = 7
TOL = 1e-13


def _idx(ids, n):                       # INDEX_CORRECTED: stored id - 1, 0 -> pad entity n
    ids = np.asarray(ids).astype(np.int64)
    return np.where(ids > 0, ids - 1, n)


def _pad(a):                            # append the zero pad entity
    return np.concatenate([a, np.zeros((1,) + a.shape[1:], a.dtype)])


def _below(a):                          # a[:, k-1] with level -1 = 0
    return np.concatenate([np.zeros_like(a[:, :1]), a[:, :-1]], axis=1)


@pytest.fixture(scope="module")
def warmed(grid642):
    st, ora, _ = build_pair(grid642, L, _abi.INDEX_CORRECTED, gpu=False)
    ora.atm_compute_solve_diagnostics(False, -1)
    ora.atm_srk3(600.0)
    pre = ora.download_all()
    yield st, ora, pre
    ora.close()


def _reset(ora, pre):
    for n, a in pre.items():
        ora.upload_field(n, a)


def _check(ora, want):
    for n, a in want.items():
        got = ora.download_field(n)
        fin = np.isfinite(a)
        assert np.array_equal(fin, np.isfinite(got)), n
        scale = np.abs(a[fin]).max() if fin.any() else 0.0
        err = np.abs(got[fin] - a[fin]).max() if fin.any() else 0.0
        assert err <= TOL * scale, (n, err, scale)


def test_divergence_damping_3d(warmed):                                     # dynamics_tasks.rg:1736-1763
    st, ora, f = warmed
    _reset(ora, f)
    s, cfg = st.static, ora.cfg
    nC = s["nEdgesOnCell"].shape[0]
    dts = 300.0
    c1, c2 = _idx(s["cellsOnEdge"][:, 0], nC), _idx(s["cellsOnEdge"][:, 1], nC)
    coef = 2.0 * cfg.config_smdiv * cfg.config_len_disp * (1.0 / dts)
    rpp, rppo, tm = _pad(f["rtheta_pp"]), _pad(f["rtheta_pp_old"]), _pad(f["theta_m"])
    shared = _pad(np.asarray(s["isShared"]).astype(bool)) if s.get("isShared") is not None else np.zeros(nC + 1, bool)
    on = ~(shared[c1] & shared[c2])
    div1, div2 = -(rpp[c1] - rppo[c1]), -(rpp[c2] - rppo[c2])
    with np.errstate(all="ignore"):
        upd = f["ru_p"] + coef * (div2 - div1) * (1.0 - s["specZoneMaskEdge"][:, None]) / (tm[c1] + tm[c2])
    want = f["ru_p"].copy()
    want[on, :L] = upd[on, :L]
    ora.atm_divergence_damping_3d(dts)
    _check(ora, {"ru_p": want})
    assert not np.array_equal(want, f["ru_p"])


def test_set_smlstep_pert_variables(warmed):       # dynamics_tasks.rg:1503-1528, EVERY point of cpr: levels 0..L inclusive (Q22)
    st, ora, f = warmed
    _reset(ora, f)
    s, cfg = st.static, ora.cfg
    nE = s["cellsOnEdge"].shape[0]
    # make level L discriminating: the init leaves fzm/fzp/zz/u_tend/w of level L at zero (M1)
    rng = np.random.default_rng(7)
    f = dict(f)
    for n in ("fzm", "fzp", "zz", "u_tend", "w", "zb_cell", "zb3_cell"):
        a = f[n].copy()
        if a.ndim == 1:
            a[L] = 0.3 + rng.random()
        elif a.ndim == 2:
            a[:, L] = 0.5 + rng.random(a.shape[0])
        else:
            a[:, L, :] = 0.5 + rng.random((a.shape[0], a.shape[2]))
        f[n] = a
        ora.upload_field(n, a)
    fzm, fzp = f["fzm"], f["fzp"]
    ut = _pad(f["u_tend"])
    w = f["w"].copy()
    act = (s["bdyMaskCell"] <= cfg.nRelaxZone)[:, None]
    for i in range(s["edgesOnCell"].shape[1]):
        on = act & (i < s["nEdgesOnCell"])[:, None]
        e = _idx(s["edgesOnCell"][:, i], nE)
        u_k, u_m = ut[e], _below(ut[e])
        flux = s["edgesOnCell_sign"][:, i][:, None] * (fzm * u_k + fzp * u_m)
        w = np.where(on, w - (f["zb_cell"][:, :, i] + np.copysign(1.0, u_k) * f["zb3_cell"][:, :, i]) * flux, w)
    w = np.where(act, w * (fzm * f["zz"] + fzp * _below(f["zz"])), w)
    ora.atm_set_smlstep_pert_variables()
    _check(ora, {"w": w})
    assert np.abs(w[:, L]).max() > 0


@pytest.mark.parametrize("small_step", [0, 1])
def test_advance_acoustic_step_literal(warmed, small_step):                 # dynamics_tasks.rg:1615-1704, point by point
    st, ora, f = warmed
    _reset(ora, f)
    s, cfg = st.static, ora.cfg
    nC, nE = s["nEdgesOnCell"].shape[0], s["cellsOnEdge"].shape[0]
    dts = 300.0
    epssm = cfg.config_epssm
    resm = (1.0 - epssm) / (1.0 + epssm)
    cofrz, rdzw, fzm, fzp = (f[k] for k in ("cofrz", "rdzw", "fzm", "fzp"))
    o = {k: f[k].copy() for k in ("rw_p", "wwAvg", "rho_pp", "rtheta_pp", "rtheta_pp_old")}
    rw_p, ww, rho_pp, rt_pp = o["rw_p"], o["wwAvg"], o["rho_pp"], o["rtheta_pp"]
    o["rtheta_pp_old"][:, :L] = 0.0 if small_step == 0 else f["rtheta_pp"][:, :L]
    if small_step == 0:
        rw_p[:] = 0; ww[:] = 0
    c1, c2 = np.append(_idx(s["cellsOnEdge"][:, 0], nC), nC), np.append(_idx(s["cellsOnEdge"][:, 1], nC), nC)
    rup, tm = _pad(f["ru_p"]), _pad(f["theta_m"])
    dv = np.append(s["dvEdge"], 0.0)
    zz, w = f["zz"], f["w"]
    spec = s["specZoneMaskCell"] != 0.0
    for k in range(L):                                      # levels ascend (M4): level k sees the NEW level k-1
        if small_step == 0:
            rho_pp[:, k] = 0; rt_pp[:, k] = 0
        before = [a[spec, k].copy() for a in (rho_pp, rt_pp, rw_p, ww)]
        rs, ts = np.zeros(nC), np.zeros(nC)
        for i in range(s["edgesOnCell"].shape[1]):
            on = i < s["nEdgesOnCell"]
            e = _idx(s["edgesOnCell"][:, i], nE)
            flux = s["edgesOnCellSign"][:, i] * dts * dv[e] * rup[e, k] * s["invAreaCell"]
            rs = np.where(on, rs - flux, rs)
            ts = np.where(on, ts - flux * 0.5 * (tm[c2[e], k] + tm[c1[e], k]), ts)
        rs = rho_pp[:, k] + dts * f["tend_rho"][:, k] + rs - cofrz[k] * resm * (rw_p[:, k + 1] - rw_p[:, k])
        ts = rt_pp[:, k] + dts * f["theta_m"][:, k] + ts - resm * rdzw[k] * (f["coftz"][:, k + 1] * rw_p[:, k + 1] - f["coftz"][:, k] * rw_p[:, k])
        if k > 0:
            ww[:, k] += 0.5 * (1.0 - epssm) * rw_p[:, k]
            # rs[k-1] and ts[k-1] were re-zeroed at this point (Q25)
            rw_p[:, k] += (dts * w[:, k] - f["cofwz"][:, k] * ((zz[:, k] * ts - zz[:, k - 1] * 0.0) + resm * (zz[:, k] * rt_pp[:, k] - zz[:, k - 1] * rt_pp[:, k - 1]))
                           - f["cofwr"][:, k] * ((rs + 0.0) + resm * (rho_pp[:, k] + rho_pp[:, k - 1]))
                           + f["cofwt"][:, k] * (ts + resm * rt_pp[:, k])
                           + f["cofwt"][:, k - 1] * (0.0 + resm * rt_pp[:, k - 1]))
            rw_p[:, k] -= f["a_tri"][:, k] * rw_p[:, k - 1]
            rw_p[:, k] *= f["alpha_tri"][:, k]
            d3 = f["rw_save"][:, k] - f["rw"][:, k]
            rw_p[:, k] += d3 - dts * f["dss"][:, k] * (fzm[k] * zz[:, k] + fzp[k] * zz[:, k - 1]) * (fzm[k] * f["rho_zz"][:, k] + fzp[k] * f["rho_zz"][:, k - 1]) * w[:, k]
            rw_p[:, k] /= (1.0 + dts * f["dss"][:, k])
            rw_p[:, k] -= d3
            ww[:, k] += 0.5 * (1.0 + epssm) * rw_p[:, k]
        rho_pp[:, k] = rs - cofrz[k] * (rw_p[:, k + 1] - rw_p[:, k])
        rt_pp[:, k] = ts - rdzw[k] * (f["coftz"][:, k + 1] * rw_p[:, k + 1] - f["coftz"][:, k] * rw_p[:, k])
        # specified-zone columns only integrate their tendencies (:1698-1703); level 0 included
        rho_pp[spec, k] = before[0] + dts * f["tend_rho"][spec, k]
        rt_pp[spec, k] = before[1] + dts * f["theta_m"][spec, k]
        rw_p[spec, k] = before[2] + dts * w[spec, k]
        ww[spec, k] = before[3] + 0.5 * (1.0 + epssm) * rw_p[spec, k]
    ora.atm_advance_acoustic_step(dts, small_step)
    _check(ora, o)
    assert np.abs(o["rw_p"]).max() > 0


@pytest.mark.parametrize("fix", [False, True], ids=["literal", "corrected_physics"])
@pytest.mark.parametrize("rk_step", [0, 2])
def test_recover_large_step_variables(warmed, rk_step, fix):                # dynamics_tasks.rg:1786-1871, as written
    st, ora, f = warmed
    if fix:        # MPASB200_PHYSICS_CORRECTED restores four expressions (include/mpas_b200.h)
        from oracle.oracle import Oracle
        ora = Oracle(dynamics.dims_of(st.mesh, L), _abi.default_config(index_policy=_abi.INDEX_CORRECTED, rkarg_policy=_abi.RKARG_STAGE_INDEX,
                                                                      physics_mode=_abi.PHYSICS_CORRECTED))
        ora.upload_mesh(st.static); ora.upload_state(st.f, st.vert)
    _reset(ora, f)
    s, cfg = st.static, ora.cfg
    nC, nE = s["nEdgesOnCell"].shape[0], s["cellsOnEdge"].shape[0]
    ns, dt = 2, 600.0
    rgas = cfg.rgas; rcv = rgas / (cfg.cp - rgas); p0 = 100000
    fzm, fzp = f["fzm"][:L], f["fzp"][:L]
    K = slice(0, L)
    o = {k: f[k].copy() for k in ("rho_p", "rho_zz", "w", "wwAvg", "rw", "rtheta_p", "theta_m", "exner", "pressure_p", "ruAvg", "ru", "u")}
    invNs = 1 / float(ns)
    o["rho_p"][:, K] = f["rho_p_save"][:, K] + f["rho_pp"][:, K]
    o["rho_zz"][:, K] = o["rho_p"][:, K] + f["rho_base"][:, K]
    o["wwAvg"][:, K] = f["wwAvg"][:, K] * invNs + f["rw_save"][:, K]
    o["rw"][:, K] = f["rw_save"][:, K] + f["rw_p"][:, K]
    with np.errstate(all="ignore"):
        o["w"][:, K] = o["rw"][:, K] / (fzm * f["zz"][:, K] + fzp * _below(f["zz"])[:, K])
        if fix:
            o["w"][:, 0] = 0.0                                                    # MPAS: w(1) = 0, k = 2..nVertLevels (:1810)
        if rk_step == 2:
            o["rtheta_p"][:, K] = f["rtheta_p_save"][:, K] + f["rtheta_pp"][:, K] - dt * o["rho_zz"][:, K] * f["rt_diabatic_tend"][:, K]
            o["theta_m"][:, K] = (o["rtheta_p"][:, K] + f["rtheta_base"][:, K]) / o["rho_zz"][:, K]
            if fix:
                o["exner"][:, K] = np.power(f["zz"][:, K] * (rgas / p0) * (o["rtheta_p"][:, K] + f["rtheta_base"][:, K]), rcv)   # :1819
            else:
                o["exner"][:, K] = f["zz"][:, K] * (rgas / p0) * np.power(o["rtheta_p"][:, K] + f["rtheta_base"][:, K], rcv)
            o["pressure_p"][:, K] = f["zz"][:, K] * rgas * (o["exner"][:, K] * o["rtheta_p"][:, K] + f["rtheta_base"][:, K] * (o["exner"][:, K] - f["exner_base"][:, K]))
        else:
            o["rtheta_p"][:, K] = f["rtheta_p_save"][:, K] + f["rtheta_pp"][:, K]
            o["theta_m"][:, K] = (o["rtheta_p"][:, K] + f["rtheta_base"][:, K]) / o["rho_zz"][:, K]
        c1, c2 = _idx(s["cellsOnEdge"][:, 0], nC), _idx(s["cellsOnEdge"][:, 1], nC)
        rz = _pad(o["rho_zz"]); rz[nC, :L] = 1.0                                   # the "garbage cell" (:1792-1794)
        o["ruAvg"][:, K] = f["ruAvg"][:, K] * invNs + f["ru_save"][:, K]
        o["ru"][:, K] = f["ru_save"][:, K] + f["ru_p"][:, K] if fix else f["ru_save"][:, K] * f["ru_p"][:, K]   # a product, as written (:1840)
        o["u"][:, K] = 2 * o["ru"][:, K] / (rz[c1][:, K] + rz[c2][:, K])
        ru = _pad(o["ru"])
        cf1, cf2, cf3 = f["cf1"][0], f["cf2"][0], f["cf3"][0]
        act = s["bdyMaskCell"] <= cfg.nRelaxZone
        w = o["w"]
        for y in range(L):                                                        # the surface term is added at EVERY level's visit
            for i in range(s["edgesOnCell"].shape[1]):
                on = act & (i < s["nEdgesOnCell"])
                e = _idx(s["edgesOnCell"][:, i], nE)
                sg = s["edgesOnCell_sign"][:, i]
                flux = cf1 * ru[e, 0] + cf2 * ru[e, 1] + cf3 * ru[e, 2]
                w[:, 0] = np.where(on, w[:, 0] + sg * (f["zb_cell"][:, 0, i] + np.copysign(1.0, flux) * f["zb3_cell"][:, 0, i]) * flux, w[:, 0])
                ru_m = ru[e, y - 1] if y > 0 else np.zeros(nC)
                flux2 = fzm[y] * ru[e, y] + fzp[y] * ru_m if fix else fzm[y] * ru[e, y] * (fzp[y] * ru_m)          # :1856
                w[:, y] = np.where(on, w[:, y] + sg * (f["zb_cell"][:, y, i] + np.copysign(1.0, flux2) * f["zb3_cell"][:, y, i]) * flux2, w[:, y])
        w[:, 0] = np.where(act, w[:, 0] / (cf1 * o["rho_zz"][:, 0] + cf2 * o["rho_zz"][:, 1] + cf3 * o["rho_zz"][:, 2]), w[:, 0])
        for y in range(1, L):
            w[:, y] = np.where(act, w[:, y] / (fzm[y] * o["rho_zz"][:, y] + fzp[y] * o["rho_zz"][:, y - 1]), w[:, y])
    ora.atm_recover_large_step_variables(ns, rk_step, dt)
    _check(ora, o)
    assert np.all(ora.download_pad("rho_zz")[:L] == 1.0)
    if fix:
        assert np.isfinite(o["w"]).all()
        ora.close()


@pytest.mark.parametrize("twice", [False, True], ids=["once", "again_with_other_dts"])
def test_compute_vert_imp_coefs(warmed, twice):                             # dynamics_tasks.rg:513-592
    st, ora, f = warmed
    _reset(ora, f)
    cfg = ora.cfg
    rgas = cfg.rgas; rcv = rgas / (cfg.cp - rgas); c2 = cfg.cp * rcv; g = cfg.gravity
    cur = {k: f[k].copy() for k in ("cofrz", "cofwr", "cofwz", "coftz", "cofwt", "a_tri", "b_tri", "c_tri", "alpha_tri", "gamma_tri")}
    fzm, fzp, rdzw, rdzu = f["fzm"], f["fzp"], f["rdzw"], f["rdzu"]
    zz, ex, th = f["zz"], f["exner"], f["theta_m"]
    for dts in ((200.0, 300.0) if twice else (200.0,)):
        dtseps = .5 * dts * (1.0 + cfg.config_epssm)
        cur["cofrz"][:L] = dtseps * rdzw[:L]
        cofrz = cur["cofrz"]
        cur["gamma_tri"][:, 0] = 0.0
        k = np.arange(1, L)
        m = k - 1
        zf = fzm[k] * zz[:, k] + fzp[k] * zz[:, m]
        cur["cofwr"][:, k] = .5 * dtseps * g * zf
        cur["coftz"][:, :L] = 0.0
        cur["cofwz"][:, k] = dtseps * c2 * zf * rdzu[k] * f["cqw"][:, k] * (fzm[k] * ex[:, k] + fzp[k] * ex[:, m])
        cur["coftz"][:, k] = dtseps * (fzm[k] * th[:, k] + fzp[k] * th[:, m])
        K = slice(0, L)
        cur["cofwt"][:, K] = (.5 * dtseps * rcv * zz[:, K] * g * f["rho_base"][:, K] / (1.0 + f["qtot"][:, K]) * ex[:, K]
                              / ((f["rtheta_base"][:, K] + f["rtheta_p"][:, K]) * f["exner_base"][:, K]))
        cofwz, coftz, cofwr, cofwt = cur["cofwz"], cur["coftz"], cur["cofwr"], cur["cofwt"]
        cur["a_tri"][:, k] = (-1.0 * cofwz[:, k] * coftz[:, m] * rdzw[m] * zz[:, m] + cofwr[:, k] * cofrz[m]
                              - cofwt[:, m] * coftz[:, m] * rdzw[m])
        cur["b_tri"][:, k] = (1.0 + cofwz[:, k] * (coftz[:, k] * rdzw[k] * zz[:, k] + coftz[:, k] * rdzw[m] * zz[:, m])
                              - coftz[:, k] * (cofwt[:, k] * rdzw[k] - cofwt[:, k] * rdzw[m]) + cofwr[:, k] * ((cofrz[k] - cofrz[m])))
        cur["c_tri"][:, k] = (-1.0 * cofwz[:, k] * coftz[:, k + 1] * rdzw[k] * zz[:, k] - cofwr[:, k] * cofrz[k]
                              + cofwt[:, k] * coftz[:, k + 1] * rdzw[k])
        # alpha uses gamma_tri of level k-1 as it is BEFORE this call's gamma loop (Q10): a separate, earlier loop
        cur["alpha_tri"][:, k] = 1.0 / (cur["b_tri"][:, k] - cur["a_tri"][:, k] * cur["gamma_tri"][:, m])
        cur["gamma_tri"][:, k] = cur["c_tri"][:, k] * cur["alpha_tri"][:, k]
        ora.atm_compute_vert_imp_coefs(dts)
    _check(ora, cur)


@pytest.mark.parametrize("hollingsworth,rk_step", [(False, 0), (False, 2), (True, -1)])
def test_compute_solve_diagnostics(warmed, hollingsworth, rk_step):         # dynamics_tasks.rg:328-454
    st, ora, f = warmed
    _reset(ora, f)
    s = st.static
    nC, nE, nV = s["nEdgesOnCell"].shape[0], s["cellsOnEdge"].shape[0], s["edgesOnVertex"].shape[0]
    K = slice(0, L)
    zero = lambda n: np.zeros((n, L))
    get = lambda k, n: np.zeros(n) if s.get(k) is None else np.asarray(s[k], dtype=np.float64)
    c1, c2 = _idx(s["cellsOnEdge"][:, 0], nC), _idx(s["cellsOnEdge"][:, 1], nC)
    u = _pad(f["u"])[:, K]
    h = _pad(f["h"])[:, K]
    dc, dv = np.append(get("dcEdge", nE), 0.0), np.append(get("dvEdge", nE), 0.0)
    o = {k: f[k].copy() for k in ("h_edge", "ke_edge", "vorticity", "divergence", "ke", "ke_vertex", "v", "pv_vertex", "pv_edge")}
    o["h_edge"][:, K] = 0.5 * (h[c1] + h[c2])
    o["ke_edge"][:, K] = (dc[:nE] * dv[:nE])[:, None] * u[:nE] ** 2
    vort = zero(nV)
    for i in range(s["edgesOnVertex"].shape[1]):
        e = _idx(s["edgesOnVertex"][:, i], nE)
        vort = vort + (get("edgesOnVertexSign", (nV, 3))[:, i] * dc[e])[:, None] * u[e]
    o["vorticity"][:, K] = vort * get("invAreaTriangle", nV)[:, None]
    div, ke = zero(nC), zero(nC)
    kee = _pad(o["ke_edge"])[:, K]
    for i in range(s["edgesOnCell"].shape[1]):
        on = (i < s["nEdgesOnCell"])[:, None]
        e = _idx(s["edgesOnCell"][:, i], nE)
        div = np.where(on, div + ((s["edgesOnCellSign"][:, i] * dv[e])[:, None] + u[e]), div)         # "s + u", as written (:375)
        ke = np.where(on, ke + 0.25 * kee[e], ke)
    inva = get("invAreaCell", nC)[:, None]
    o["divergence"][:, K] = div * inva
    ke = ke * inva
    if hollingsworth:
        ev = [_idx(s["edgesOnVertex"][:, j], nE) for j in range(3)]
        o["ke_vertex"][:, K] = (kee[ev[0]] + kee[ev[1]] + kee[ev[2]]) * (0.25 * get("invAreaTriangle", nV))[:, None]
        ke_fact = 1.0 - 0.375
        ke = ke * ke_fact
        kev = _pad(o["ke_vertex"])[:, K]
        kav = np.concatenate([np.asarray(s["kiteAreasOnVertex"], dtype=np.float64), np.zeros((1, 3))])
        for i in range(s["edgesOnCell"].shape[1]):
            on = (i < s["nEdgesOnCell"])[:, None]
            vtx = _idx(s["verticesOnCell"][:, i], nV)
            j = np.asarray(s["kiteForCell"])[:, i]
            ke = np.where(on, ke + ((1.0 - ke_fact) * kav[vtx, j])[:, None] * kev[vtx] * inva, ke)
    o["ke"][:, K] = ke
    if not (rk_step != -1 and rk_step != 2):
        v = zero(nE)
        for i in range(1, s["edgesOnEdge_ECP"].shape[1]):                   # starts at 1, as written (:433)
            on = (i < s["nEdgesOnEdge"])[:, None]
            eoe = _idx(s["edgesOnEdge_ECP"][:, i], nE)
            v = np.where(on, v + s["weightsOnEdge"][:, i][:, None] * u[eoe], v)
        o["v"][:, K] = v
    o["pv_vertex"][:, K] = get("fVertex", nV)[:, None] + o["vorticity"][:, K]
    pvv = _pad(o["pv_vertex"])[:, K]
    v1, v2 = _idx(s["verticesOnEdge"][:, 0], nV), _idx(s["verticesOnEdge"][:, 1], nV)
    o["pv_edge"][:, K] = 0.5 * (pvv[v1] + pvv[v2])
    ora.atm_compute_solve_diagnostics(hollingsworth, rk_step)
    _check(ora, o)


# ---- atm_compute_dyn_tend_work, dynamics_tasks.rg:814-1480 ------------------------------------------------------------
def _flux4(q_im2, q_im1, q_i, q_ip1, ua):                                  # :781-783
    return ua * (7. * (q_i + q_im1) - (q_ip1 + q_im2)) / 12.0


def _flux3(q_im2, q_im1, q_i, q_ip1, ua, coef3):                           # :786-789
    return _flux4(q_im2, q_im1, q_i, q_ip1, ua) + coef3 * np.abs(ua) * ((q_ip1 - q_im2) - 3. * (q_i - q_im1)) / 12.0


def _np_dyn_tend(st, f, cfg, rk_step, dt, mixing, cam_coef, rayleigh):
    """array-at-a-time restatement for config_v_mom_eddy_visc2 = config_v_theta_eddy_visc2 = 0 (constants.rg)."""
    s = st.static
    nC, nE, nV = s["nEdgesOnCell"].shape[0], s["cellsOnEdge"].shape[0], s["edgesOnVertex"].shape[0]
    K = slice(0, L)
    ME = s["edgesOnCell"].shape[1]
    written = ("kdiff", "h_divergence", "tend_rho", "dpdz", "w", "ru_edge_w", "flux_arr", "delsq_w", "tend_w_euler", "wdwz",
               "tend_theta", "delsq_theta", "tend_theta_euler", "wdtz", "tend_rtheta_adv", "rthdynten", "delsq_divergence",
               "tend_u_euler", "wduz", "tend_u", "q", "delsq_u", "delsq_vorticity")
    o = {k: f[k].copy() for k in written}
    fzm, fzp, rdzw, rdzu = f["fzm"], f["fzp"], f["rdzw"], f["rdzu"]
    c1, c2 = _idx(s["cellsOnEdge"][:, 0], nC), _idx(s["cellsOnEdge"][:, 1], nC)
    v1, v2 = _idx(s["verticesOnEdge"][:, 0], nV), _idx(s["verticesOnEdge"][:, 1], nV)
    eoc = [_idx(s["edgesOnCell"][:, i], nE) for i in range(ME)]
    on = [(i < s["nEdgesOnCell"])[:, None] for i in range(ME)]
    sgn = s["edgesOnCell_sign"]
    dvE, invDcE = np.append(s["dvEdge"], 0.0), np.append(s["invDcEdge"], 0.0)
    del2E, del4E = np.append(s["meshScalingDel2"], 0.0), np.append(s["meshScalingDel4"], 0.0)
    c1E, c2E = np.append(c1, nC), np.append(c2, nC)
    inva = s["invAreaCell"][:, None]
    invDc, invDv = s["invDcEdge"][:, None], s["invDvEdge"][:, None]
    ld = cfg.config_len_disp
    prandtl_inv, invDt, r_earth = 1.0 / cfg.prandtl, 1.0 / dt, cfg.sphere_radius
    inv_r_earth = 1.0 / r_earth
    h_mom4, h_theta4 = cfg.config_h_mom_eddy_visc4, cfg.config_h_theta_eddy_visc4
    u, v, ru = _pad(f["u"]), _pad(f["v"]), _pad(f["ru"])
    rho_edge = _pad(f["rho_edge"])
    if rk_step == 0:                                                                                   # :858-917
        if mixing == _abi.MIX_2D_SMAGORINSKY:
            dd, do = np.zeros((nC, L)), np.zeros((nC, L))
            for i in range(ME):
                a, b = s["defc_a"][:, i][:, None], s["defc_b"][:, i][:, None]
                ue, ve = u[eoc[i]][:, K], v[eoc[i]][:, K]
                dd = np.where(on[i], dd + (a * ue - b * ve), dd)
                do = np.where(on[i], do + (b * ue + a * ve), do)
            o["kdiff"][:, K] = np.minimum((cfg.config_smagorinsky_coef * ld) ** 2.0 * np.sqrt(dd ** 2.0 + do ** 2.0), (0.01 * ld ** 2.0) * invDt)
            h_mom4 = cfg.config_visc4_2dsmag * ld ** 3.0
            h_theta4 = h_mom4
        elif mixing == _abi.MIX_2D_FIXED:
            o["kdiff"][:, K] = 0.0
        if cam_coef > 0.0:
            for k in range(L - 2, L):
                o["kdiff"][:, k] = np.maximum(o["kdiff"][:, k], 2.0 ** (k - (L - 2)) * 2.0833 * ld * cam_coef)
    kdiff = _pad(o["kdiff"])
    hd = np.zeros((nC, L))                                                                             # :924-938
    for i in range(ME):
        hd = np.where(on[i], hd + (sgn[:, i] * dvE[eoc[i]])[:, None] * ru[eoc[i]][:, K], hd)
    hd = hd * inva
    o["h_divergence"][:, K] = hd
    if rk_step == 0:                                                                                   # :942-951
        o["tend_rho"][:, K] = -hd - rdzw[K] * (f["rw"][:, 1:] - f["rw"][:, :-1] + f["tend_rho_physics"][:, K])
        o["dpdz"][:, K] = -cfg.gravity * (f["rho_base"][:, K] * f["qtot"][:, K] + f["rho_p_save"][:, K] * (1.0 + f["qtot"][:, K]))
    pp, zz, dpdz, rw, ke, hdp = _pad(f["pressure_p"]), _pad(f["zz"]), _pad(o["dpdz"]), _pad(f["rw"]), _pad(f["ke"]), _pad(o["h_divergence"])
    ue = f["u"]
    if rk_step == 0:                                                                                   # :964-970
        o["tend_u_euler"][:, K] = -f["cqu"][:, K] * ((pp[c2][:, K] - pp[c1][:, K]) * invDc / (0.5 * (zz[c2][:, K] + zz[c1][:, K]))
                                                     - 0.5 * f["zxu"][:, K] * (dpdz[c1][:, K] + dpdz[c2][:, K]))
    wduz = o["wduz"]
    wduz[:, K] = 0.0                                                                                   # :972-980
    rwavg = 0.5 * (rw[c1] + rw[c2])
    for k in range(L):
        if k == 1 or k == L - 1:
            wduz[:, k] = rwavg[:, k] * (fzm[k] * ue[:, k] + fzp[k] * ue[:, k - 1])
        if 1 < k < L - 1:
            wduz[:, k] = _flux3(ue[:, k - 2], ue[:, k - 1], ue[:, k], ue[:, k + 1], rwavg[:, k], 1.0)
    tend_u = -rdzw[K] * (wduz[:, 1:] - wduz[:, :-1])                                                   # :987
    q = np.zeros((nE, L))                                                                              # :991-1001, each term L times (Q14)
    pv = _pad(f["pv_edge"])
    for j in range(s["edgesOnEdge"].shape[1]):
        onj = (j < s["nEdgesOnEdge"])[:, None]
        eoe = _idx(s["edgesOnEdge"][:, j], nE)
        term = s["weightsOnEdge"][:, j][:, None] * u[eoe][:, K] * (0.5 * (f["pv_edge"][:, K] + pv[eoe][:, K]))
        for _ in range(L):
            q = np.where(onj, q + term, q)
    o["q"][:, K] = q
    re_ = f["rho_edge"][:, K]
    tend_u = tend_u + (re_ * (q - (ke[c2][:, K] - ke[c1][:, K]) * invDc) - ue[:, K] * 0.5 * (hdp[c1][:, K] + hdp[c2][:, K]))   # :1005-1007
    w_in = _pad(f["w"])                                                     # cr.w as it is BEFORE the w section resets it
    wsum = w_in[c1][:, :-1] + w_in[c1][:, 1:] + w_in[c2][:, :-1] + w_in[c2][:, 1:]
    cosang, coslat = np.cos(s["angleEdge"])[:, None], np.cos(s["latEdge"])[:, None]
    tend_u = tend_u - ((2.0 * cfg.omega * cosang * coslat * re_ * 0.25 * wsum) - (ue[:, K] * 0.25 * wsum * re_ * inv_r_earth))   # :1011-1017
    if rk_step == 0:
        div, vort = _pad(f["divergence"]), _pad(f["vorticity"])
        r_dv = np.minimum(invDv, 4 * invDc)
        u_diff = (div[c2][:, K] - div[c1][:, K]) * invDc - (vort[v2][:, K] - vort[v1][:, K]) * r_dv       # :1036-1047
        o["delsq_u"][:, K] = 0.0 + u_diff
        kdiffu = 0.5 * (kdiff[c1][:, K] + kdiff[c2][:, K])
        o["tend_u_euler"][:, K] += re_ * kdiffu * u_diff * s["meshScalingDel2"][:, None]
        if h_mom4 > 0.0:                                                                               # :1050-1090
            dsu = _pad(o["delsq_u"])
            dcE = np.append(s["dcEdge"], 0.0)
            dv_ = np.zeros((nV, L))
            for i in range(3):
                e = _idx(s["edgesOnVertex"][:, i], nE)
                dv_ = dv_ + (s["invAreaTriangle"] * dcE[e] * s["edgesOnVertex_sign"][:, i])[:, None] * dsu[e][:, K]
            o["delsq_vorticity"][:, K] = dv_
            dd_ = np.zeros((nC, L))
            for i in range(ME):
                dd_ = np.where(on[i], dd_ + (s["invAreaCell"] * dvE[eoc[i]] * sgn[:, i])[:, None] * dsu[eoc[i]][:, K], dd_)
            o["delsq_divergence"][:, K] = dd_
            ddp, dvp = _pad(o["delsq_divergence"]), _pad(o["delsq_vorticity"])
            scale = s["meshScalingDel4"][:, None] * h_mom4
            r_dc4 = scale * cfg.config_del4u_div_factor * invDc
            r_dv4 = scale * np.minimum(invDv, 4 * invDc)
            o["tend_u_euler"][:, K] -= re_ * ((ddp[c2][:, K] - ddp[c1][:, K]) * r_dc4 - (dvp[v2][:, K] - dvp[v1][:, K]) * r_dv4)
    if rayleigh:                                                                                       # :1152-1159
        nl = cfg.config_number_rayleigh_damp_u_levels
        inv = 1.0 / (float(nl) * (cfg.config_rayleigh_damp_u_timescale_days * 86400.0))
        for k in range(L):
            if k > L - nl + 1:
                tend_u[:, k] -= re_[:, k] * ue[:, k] * (float(k - (L - nl)) * inv)
    o["tend_u"][:, K] = tend_u + (o["tend_u_euler"][:, K] + f["tend_ru_physics"][:, K])                 # :1162
    # ---- w :1170-1320
    w = o["w"]
    w[:, K] = 0.0
    n = s["nEdgesOnCell"]
    has = n > 0
    last = _idx(s["edgesOnCell"][np.arange(nC), np.maximum(n - 1, 0)], nE)          # Q18: only the last edge's values survive
    rew = fzm[K] * ru[last][:, K] + fzp[K] * _below(ru[last])[:, K]
    o["ru_edge_w"][:, 1:L] = np.where(has[:, None], rew[:, 1:], o["ru_edge_w"][:, 1:L])
    fa = np.zeros((nC, L))
    nadv = np.append(s["nAdvCellsForEdge"], 0)
    advc = np.vstack([s["advCellsForEdge"], np.zeros((1, s["advCellsForEdge"].shape[1]), s["advCellsForEdge"].dtype)])
    ac, a3 = np.vstack([s["adv_coefs"], np.zeros((1, 15))]), np.vstack([s["adv_coefs_3rd"], np.zeros((1, 15))])
    wz = _pad(w)
    for j in range(advc.shape[1]):
        onj = (j < nadv[last])[:, None]
        cellj = _idx(advc[last, j], nC)
        sw = ac[last, j][:, None] + np.copysign(1.0, o["ru_edge_w"][:, K]) * a3[last, j][:, None]
        fa[:, 1:] = np.where(onj, fa + sw * wz[cellj][:, K], fa)[:, 1:]
    o["flux_arr"][:, K] = np.where(has[:, None], fa, o["flux_arr"][:, K])
    for i in range(ME):                                                                                # :1198-1204
        w[:, 1:L] = np.where(on[i], w[:, K] - sgn[:, i][:, None] * o["ru_edge_w"][:, K] * o["flux_arr"][:, K], w[:, K])[:, 1:]
    rz, uz, um = f["rho_zz"], f["uReconstructZonal"], f["uReconstructMeridional"]
    k, m = slice(1, L), slice(0, L - 1)
    rzf = rz[:, k] * fzm[k] + rz[:, m] * fzp[k]
    uzf, umf = fzm[k] * uz[:, k] + fzp[k] * uz[:, m], fzm[k] * um[:, k] + fzp[k] * um[:, m]
    w[:, k] += rzf * (uzf ** 2.0 + umf ** 2.0) / r_earth + 2.0 * cfg.omega * np.cos(s["latCell"])[:, None] * uzf * rzf   # :1208-1218
    if rk_step == 0:                                                                                   # :1222-1262
        dw, twe = np.zeros((nC, L)), np.zeros((nC, L))
        wp = _pad(w)
        for i in range(ME):
            e = eoc[i]
            es = (0.5 * s["invAreaCell"] * sgn[:, i] * dvE[e] * invDcE[e])[:, None]
            wtf = es * (rho_edge[e][:, K] + _below(rho_edge[e])[:, K]) * (wp[c2E[e]][:, K] - wp[c1E[e]][:, K])
            dw[:, 1:] = np.where(on[i], dw + wtf, dw)[:, 1:]
            wtf = wtf * (del2E[e][:, None] * 0.25 * (kdiff[c1E[e]][:, K] + kdiff[c2E[e]][:, K] + _below(kdiff[c1E[e]])[:, K] + _below(kdiff[c2E[e]])[:, K]))
            twe[:, 1:] = np.where(on[i], twe + wtf, twe)[:, 1:]
        o["delsq_w"][:, K] = dw
        if h_mom4 > 0.0:
            dwp = _pad(o["delsq_w"])
            for i in range(ME):
                e = eoc[i]
                es = (del4E[e] * (h_mom4 * s["invAreaCell"]) * dvE[e] * sgn[:, i] * invDcE[e])[:, None]
                twe[:, 1:] = np.where(on[i], twe - es * (dwp[c2E[e]][:, K] - dwp[c1E[e]][:, K]), twe)[:, 1:]
        o["tend_w_euler"][:, K] = twe
    wdwz = o["wdwz"]
    wdwz[:, K] = 0.0                                                                                   # :1266-1276
    rwc = f["rw"]
    for kk in range(L):
        if kk == 1 or kk == L - 1:
            wdwz[:, kk] = 0.25 * (rwc[:, kk] + rwc[:, kk - 1]) * (w[:, kk] + w[:, kk - 1])
        if 1 < kk < L - 1:
            wdwz[:, kk] = _flux3(w[:, kk - 2], w[:, kk - 1], w[:, kk], w[:, kk + 1], 0.5 * (rwc[:, kk] + rwc[:, kk - 1]), 1.0)
    w[:, k] = w[:, k] * (inva - rdzu[k] * (wdwz[:, 2:] - wdwz[:, 1:L]))                                # :1292 (Q19)
    if rk_step == 0:                                                                                   # :1294-1299
        ppc, dpc = f["pressure_p"], o["dpdz"]
        o["tend_w_euler"][:, k] -= f["cqw"][:, k] * (rdzu[k] * (ppc[:, k] - ppc[:, m]) - (fzm[k] * dpc[:, k] + fzp[k] * dpc[:, m]))
    w[:, k] += o["tend_w_euler"][:, k]                                                                  # :1316-1320
    # ---- theta :1322-1480
    tm, tms = _pad(f["theta_m"]), _pad(f["theta_m_save"])
    tt = np.zeros((nC, L))
    fa = o["flux_arr"][:, K].copy()
    for i in range(ME):
        e = eoc[i]
        fi = np.zeros((nC, L))
        for j in range(advc.shape[1]):
            onj = (j < nadv[e])[:, None]
            sw = ac[e, j][:, None] + np.copysign(1.0, ru[e][:, K]) * a3[e, j][:, None]
            fi = np.where(onj, fi + sw * tm[_idx(advc[e, j], nC)][:, K], fi)
        fa = np.where(on[i], fi, fa)
        tt = np.where(on[i], tt - sgn[:, i][:, None] * ru[e][:, K] * fi, tt)
    o["flux_arr"][:, K] = fa
    if rk_step > 0:                                                                                    # :1340-1352
        rus = _pad(f["ru_save"])
        for i in range(ME):
            e = eoc[i]
            flux = (sgn[:, i] * dvE[e])[:, None] * (rus[e][:, K] - ru[e][:, K]) * 0.5 * (tms[c2E[e]][:, K] + tms[c1E[e]][:, K])
            tt = np.where(on[i], tt - flux, tt)
    if rk_step == 0:                                                                                   # :1354-1394
        dth, tte = np.zeros((nC, L)), np.zeros((nC, L))
        for i in range(ME):
            e = eoc[i]
            es = (s["invAreaCell"] * sgn[:, i] * dvE[e] * invDcE[e])[:, None]
            pr_scale = (prandtl_inv * del2E[e])[:, None]
            ttf = es * (tm[c2E[e]][:, K] - tm[c1E[e]][:, K]) * rho_edge[e][:, K]
            dth = np.where(on[i], dth + ttf, dth)
            ttf = ttf * (0.5 * (kdiff[c1E[e]][:, K] + kdiff[c2E[e]][:, K]) * pr_scale)
            tte = np.where(on[i], tte + ttf, tte)
        o["delsq_theta"][:, K] = dth
        if h_theta4 > 0.0:
            dtp = _pad(o["delsq_theta"])
            for i in range(ME):
                e = eoc[i]
                es = (del4E[e] * (h_theta4 * prandtl_inv * s["invAreaCell"]) * dvE[e] * sgn[:, i] * invDcE[e])[:, None]
                tte = np.where(on[i], tte - es * (dtp[c2E[e]][:, K] - dtp[c1E[e]][:, K]), tte)
        o["tend_theta_euler"][:, K] = tte
    wdtz = o["wdtz"]
    wdtz[:, K] = 0.0                                                                                   # :1398-1412
    tmc, tmsc, rws = f["theta_m"], f["theta_m_save"], f["rw_save"]
    for kk in range(L):
        if 0 < kk < L - 1:
            wdtz[:, kk] = (rws[:, kk] - rwc[:, kk]) * (fzm[kk] * tmsc[:, kk] + fzp[kk] * tmsc[:, kk - 1])
        if kk == 1:
            wdtz[:, kk] += rwc[:, kk] * (fzm[kk] * tmc[:, kk] + fzp[kk] * tmc[:, kk - 1])
        if kk == L - 1:
            wdtz[:, kk] = rws[:, kk] * (fzm[kk] * tmsc[:, kk] + fzp[kk] * tmsc[:, kk - 1])
    tt = tt * (inva - rdzw[K] * (wdtz[:, 1:] - wdtz[:, :-1]))                                           # :1415 (Q19)
    o["tend_rtheta_adv"][:, K] = tt
    o["rthdynten"][:, K] = tt / f["rho_zz"][:, K]
    tt = tt + f["rho_zz"][:, K] * f["rt_diabatic_tend"][:, K]
    o["tend_theta"][:, K] = tt + (o["tend_theta_euler"][:, K] + f["tend_rtheta_physics"][:, K])        # :1478
    return o


@pytest.mark.parametrize("rk_step,mixing,cam,rayleigh", [
    (0, _abi.MIX_2D_SMAGORINSKY, 0.0, False), (1, _abi.MIX_2D_SMAGORINSKY, 0.0, False), (0, _abi.MIX_2D_FIXED, 0.2, False),
    (0, _abi.MIX_OTHER, 0.0, True), (2, _abi.MIX_2D_SMAGORINSKY, 0.0, True)],
    ids=["rk0_smagorinsky", "rk1", "rk0_fixed_cam", "rk0_other_rayleigh", "rk2_rayleigh"])
def test_compute_dyn_tend(warmed, rk_step, mixing, cam, rayleigh):
    st, ora, f0 = warmed
    _reset(ora, f0)
    # the warmed state already holds this task's own outputs (nothing on the literal path changes its inputs): perturb the
    # inputs so that every output has to move
    rng = np.random.default_rng(3)
    f = dict(f0)
    for n in ("u", "v", "ru", "rw", "w", "theta_m", "pv_edge", "ke", "pressure_p", "divergence", "vorticity", "rho_zz", "rho_p_save"):
        f[n] = f0[n] * (1.0 + 0.05 * rng.standard_normal(f0[n].shape))
        ora.upload_field(n, f[n])
    want = _np_dyn_tend(st, f, ora.cfg, rk_step, 600.0, mixing, cam, rayleigh)
    ora.atm_compute_dyn_tend(rk_step, 600.0, config_horiz_mixing=mixing, config_mpas_cam_coef=cam, config_rayleigh_damp_u=rayleigh)
    _check(ora, want)
    moved = [n for n in want if not np.array_equal(want[n], f[n], equal_nan=True)]
    for n in ("tend_u", "tend_theta", "w", "q", "h_divergence", "wduz", "wdwz", "wdtz", "flux_arr", "rthdynten"):
        assert n in moved and np.isfinite(want[n]).all() and np.abs(want[n]).max() > 0, n
    if rk_step == 0:
        for n in ("tend_u_euler", "tend_w_euler", "tend_theta_euler", "delsq_u", "delsq_w", "delsq_theta", "tend_rho", "dpdz"):
            assert n in moved, n
        if mixing != _abi.MIX_OTHER:
            assert "kdiff" in moved


def test_advance_scalars(warmed):
    """atm_advance_scalars is ABSENT from the reference (rk_timestep.rg:465 skips it; storage data_structures.rg:36): the oracle
    restates atm_advance_scalars_work of MPAS-A v7 loop by loop; this is the same routine array-at-a-time.  Parity unpinned."""
    st, ora, f = warmed
    _reset(ora, f)
    s, cfg = st.static, ora.cfg
    nC, nE = s["nEdgesOnCell"].shape[0], s["cellsOnEdge"].shape[0]
    rng = np.random.default_rng(5)
    NS = 8
    q = 1e-3 * (1.0 + rng.random((nC, L + 1, NS))); q_old = 1e-3 * (1.0 + rng.random((nC, L + 1, NS)))
    ru = (f["ru"] + 0.3 * rng.standard_normal(f["ru"].shape)); ww = 0.05 * rng.standard_normal(f["wwAvg"].shape)
    rzo = f["rho_zz"] * (1.0 + 0.01 * rng.random(f["rho_zz"].shape))
    for n, a in (("scalars", q), ("scalars_old", q_old), ("ruAvg", ru), ("wwAvg", ww), ("rho_zz_old_split", rzo)):
        ora.upload_field(n, a)
    dt = 200.0
    coef3 = cfg.config_coef_3rd_order
    fzm, fzp, rdzw = f["fzm"], f["fzp"], f["rdzw"]
    qp, rup = _pad(q), _pad(ru)
    flux = np.zeros((nE + 1, L, NS))
    for j in range(s["advCellsForEdge"].shape[1]):
        on = (j < s["nAdvCellsForEdge"])[:, None, None]
        c = _idx(s["advCellsForEdge"][:, j], nC)
        wgt = s["adv_coefs"][:, j][:, None] + np.copysign(1.0, ru[:, :L]) * s["adv_coefs_3rd"][:, j][:, None]
        flux[:nE] += np.where(on, wgt[:, :, None] * qp[c][:, :L, :], 0.0)
    tend = np.zeros((nC, L, NS))
    for i in range(s["edgesOnCell"].shape[1]):
        on = (i < s["nEdgesOnCell"])[:, None, None]
        e = _idx(s["edgesOnCell"][:, i], nE)
        tend -= np.where(on, (s["edgesOnCellSign"][:, i][:, None] * rup[e][:, :L])[:, :, None] * flux[e], 0.0)
    tend *= s["invAreaCell"][:, None, None]
    wdtn = np.zeros((nC, L + 1, NS))
    for k in (1, L - 1):
        wdtn[:, k] = ww[:, k, None] * (fzm[k] * q[:, k] + fzp[k] * q[:, k - 1])
    for k in range(2, L - 1):
        ua = ww[:, k, None]
        f4 = ua * (7.0 * (q[:, k] + q[:, k - 1]) - (q[:, k + 1] + q[:, k - 2])) / 12.0
        wdtn[:, k] = f4 + coef3 * np.abs(ua) * ((q[:, k + 1] - q[:, k - 2]) - 3.0 * (q[:, k] - q[:, k - 1])) / 12.0
    want = q.copy()
    want[:, :L] = (q_old[:, :L] * rzo[:, :L, None] + dt * (tend - rdzw[:L, None] * (wdtn[:, 1:] - wdtn[:, :-1]))) / f["rho_zz"][:, :L, None]
    ora.atm_advance_scalars(dt, 1)
    _check(ora, {"scalars": want})
    assert not np.allclose(want[:, :L], q[:, :L])
    # and the driver wiring: with config_scalar_advection on, the setup task saves scalars_old and every stage advances
    from oracle.oracle import Oracle
    from mpas_regent_b200 import dynamics
    o2 = Oracle(dynamics.dims_of(st.mesh, L), _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, config_scalar_advection=1))
    o2.upload_mesh(st.static); o2.upload_state(st.f, st.vert); o2.upload_field("scalars", q)
    o2.atm_compute_solve_diagnostics(False, -1)
    o2.atm_srk3(600.0)
    assert np.array_equal(o2.download_field("scalars_old")[:, :L], q[:, :L])
    assert np.isfinite(o2.download_field("scalars")).all()
    o2.close()


def test_init_coupled_diagnostics_and_reconstruct_2d(warmed):
    """the two one-time tasks of atm_core_init that are stencils over 3-D fields (SURVEY.md 8f rank 3), array-at-a-time:
    atm_init_coupled_diagnostics dynamics_tasks.rg:651-725, mpas_reconstruct_2d :1894-1948 (the latter also against the
    vectorised host producer core_init.mpas_reconstruct_2d the harness uses)."""
    from mpas_regent_b200 import core_init
    st, ora, f = warmed
    _reset(ora, f)
    s, cfg = st.static, ora.cfg
    nC, nE = s["nEdgesOnCell"].shape[0], s["cellsOnEdge"].shape[0]
    rgas = cfg.rgas; rcv = rgas / (cfg.cp - rgas)
    fzm, fzp = f["fzm"], f["fzp"]
    lev = np.arange(L + 1)[None, :] < L
    rho_zz = np.where(lev, f["rho_zz"] / np.where(lev, f["zz"], 1.0), f["rho_zz"])
    c1, c2 = _idx(s["cellsOnEdge"][:, 0], nC), _idx(s["cellsOnEdge"][:, 1], nC)
    rzp = _pad(rho_zz)
    ru = np.where(lev, 0.5 * f["u"] * (rzp[c1] + rzp[c2]), f["ru"])
    zz = f["zz"]
    zf = fzp * _below(zz) + fzm * zz
    rw = f["w"] * (fzp * _below(rho_zz) + fzm * rho_zz) * zf
    rw[:, 0] = 0.0
    rup = _pad(ru)
    for i in range(s["edgesOnCell"].shape[1]):
        on = (i < s["nEdgesOnCell"])[:, None] & (np.arange(L + 1)[None, :] > 0)
        e = _idx(s["edgesOnCell"][:, i], nE)
        flux = fzm * rup[e] + fzp * _below(rup[e])
        rw = np.where(on, rw - s["edgesOnCellSign"][:, i][:, None] * (f["zb_cell"][:, :, i] + np.copysign(1.0, flux) * f["zb3_cell"][:, :, i]) * flux * zf, rw)
    rho_p = rho_zz - f["rho_base"]
    rtb = f["theta_base"] * f["rho_base"]
    rtp = f["theta_m"] * rho_p + f["rho_base"] * (f["theta_m"] - f["theta_base"])
    with np.errstate(invalid="ignore"):
        ex = np.power(zz * (rgas / 100000) * (rtp + rtb), rcv); exb = np.power(zz * (rgas / 100000) * rtb, rcv)
    want = {"rho_zz": rho_zz, "ru": ru, "rw": np.where(lev, rw, f["rw"])}
    for n, a in (("rho_p", rho_p), ("rtheta_base", rtb), ("rtheta_p", rtp), ("exner", ex), ("exner_base", exb),
                 ("pressure_p", zz * rgas * (ex * rtp + rtb * (ex - exb))), ("pressure_base", zz * rgas * exb * rtb)):
        want[n] = np.where(lev, a, f[n])
    ora.atm_init_coupled_diagnostics()
    _check(ora, want)
    # reconstruct
    _reset(ora, f)
    ora.mpas_reconstruct_2d(False, True)
    zonal, merid = core_init.mpas_reconstruct_2d(st.mesh, _abi.INDEX_CORRECTED, f["u"], s["coeffs_reconstruct"], L)
    _check(ora, {"uReconstructZonal": np.where(lev, zonal, f["uReconstructZonal"]), "uReconstructMeridional": np.where(lev, merid, f["uReconstructMeridional"])})
    assert np.abs(ora.download_field("uReconstructX")).max() > 0
