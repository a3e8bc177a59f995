"""The numpy restatement of the pressure-level diagnostics (tests/isobaric_ref.py) pinned on hand-built columns, and a
physical check of it on the host-built JW state: surface pressure near p0 and the 850 hPa temperature near the analytic JW
temperature at eta = 0.85."""
import numpy as np
import pytest

from mpas_regent_b200 import _abi, init_jw
from mpas_regent_b200.init_jw import GRAVITY, OMEGA, PII, RGAS, SPHERE_RADIUS
from tests.isobaric_ref import ROW, isobaric_from_levels, isobaric_ref

KEYS = [k for _, k in ROW]


def _columns(p, fields=None, zgrid=None):
    """level_fields' layout for hand-built columns: p [n, L]; every one of the six fields = ``fields`` (default 0)"""
    p = np.atleast_2d(np.asarray(p, dtype=np.float64))
    n, L = p.shape
    zg = np.tile(np.arange(L + 1, dtype=np.float64) * 100.0, (n, 1)) if zgrid is None else np.atleast_2d(zgrid)
    lev = {k: np.zeros((n, L)) if fields is None else np.atleast_2d(np.asarray(fields, dtype=np.float64)).copy() for k in KEYS}
    lev["p"] = p
    lev["z"] = 0.5 * (zg[:, :L] + zg[:, 1:])
    return lev, zg[:, 0]


def test_field_linear_in_ln_p_is_reproduced():
    p = 1.0e5 * np.exp(-0.1 * np.arange(12))
    f = 3.0 + 2.0 * np.log(p)
    lev, zg0 = _columns(p, f)
    plev = np.array([99000.0, 85000.0, 70000.5, 50000.0, 40000.0, p[0], p[-1]])
    out = isobaric_from_levels(lev, zg0, plev)
    for name, key in ROW:
        if key == "z":
            continue
        assert np.allclose(out[name][0], 3.0 + 2.0 * np.log(plev), rtol=1e-14, atol=0.0), name


def test_outside_the_column_is_nan():
    p = [1000.0, 900.0, 800.0, 700.0]
    lev, zg0 = _columns(p, [1.0, 2.0, 3.0, 4.0])
    out = isobaric_from_levels(lev, zg0, [1000.5, 1000.0, 700.0, 699.5, 850.0])
    for name, _ in ROW:
        assert np.array_equal(np.isnan(out[name][0]), [True, False, False, True, False]), name


def test_nan_and_equal_neighbours():
    """a NaN level breaks only the brackets that touch it; equal adjacent pressures give a = 1: f(k+1) + (f(k) - f(k+1))"""
    p = [1000.0, np.nan, 800.0, 800.0, 700.0]
    T = [1.0, 2.0, 3.0 + 1e-9, 7.25, 5.0]
    lev, zg0 = _columns(p, T)
    out = isobaric_from_levels(lev, zg0, [900.0, 800.0, 750.0])["temperature"][0]
    assert np.isnan(out[0])
    assert out[1] == np.float64(7.25) + 1.0 * (np.float64(3.0 + 1e-9) - np.float64(7.25))     # k* = 2, the equal pair
    assert np.isfinite(out[2])


def test_first_bracket_wins_in_a_non_monotone_column():
    p = [1000.0, 800.0, 900.0, 700.0]
    T = [10.0, 20.0, 30.0, 40.0]
    lev, zg0 = _columns(p, T)
    out = isobaric_from_levels(lev, zg0, [850.0, 750.0, 950.0])["temperature"][0]
    a = (np.log(850.0) - np.log(800.0)) / (np.log(1000.0) - np.log(800.0))
    assert out[0] == 20.0 + a * (10.0 - 20.0)                                       # k* = 0, not 2
    assert 30.0 < out[1] < 40.0                                                     # only 900 >= 750 >= 700 brackets it
    assert 10.0 < out[2] < 20.0


def test_surface_pressure_is_exact_for_p_linear_in_z():
    zg = np.array([[0.0, 100.0, 300.0, 600.0], [1000.0, 1100.0, 1300.0, 1700.0]])
    z = 0.5 * (zg[:, :3] + zg[:, 1:])
    p = 1.0e5 - 2.0 * z
    lev, zg0 = _columns(p, zgrid=zg)
    ps = isobaric_from_levels(lev, zg0, [90000.0])["surface_pressure"]
    assert np.array_equal(ps, 1.0e5 - 2.0 * zg[:, 0])


def _T_jw(eta, phi, u0=35.0, t0=288.0, dtdz=0.005, eta_t=0.2, delta_t=4.8e5):
    """the analytic JW (2006) temperature init_jw's column solve uses, at one eta (eta >= eta_t here)"""
    assert eta >= eta_t
    etav = (eta - 0.252) * PII / 2.0
    teta = t0 * eta ** (RGAS * dtdz / GRAVITY)
    cosv = max(np.cos(etav), 0.0)
    return teta + 0.75 * eta * PII * u0 / RGAS * np.sin(etav) * np.sqrt(cosv) * (
        (-2.0 * np.sin(phi) ** 6 * (np.cos(phi) ** 2 + 1.0 / 3.0) + 10.0 / 63.0) * 2.0 * u0 * cosv ** 1.5
        + (1.6 * np.cos(phi) ** 3 * (np.sin(phi) ** 2 + 2.0 / 3.0) - PII / 4.0) * SPHERE_RADIUS * OMEGA)


def test_jw_state_surface_pressure_and_850_hpa_temperature(grid2562):
    """x1.2562, L = 26, the host generator.  make_state leaves pressure_base to atm_init_coupled_diagnostics on the device,
    so it is formed here as that task forms it (zz * rgas * exner_base * rtheta_base, dynamics_tasks.rg:651-725).
    Measured: ps - p0 lies in [+308.1, +379.5] Pa, and |T(850 hPa) - T_JW(eta = 0.85)| <= 0.418 K (T from 223.5 to
    301.8 K).  Bounds: ps - p0 in [0, 500] Pa and 0.6 K, about 30 % and 45 % above the measured extremes.  The surface
    pressure is the discrete state's, not the extrapolation's: linear in ln p and a hydrostatic half layer from level 0
    give 1003.4 - 1005.1 and 1003.4 - 1004.6 hPa.  The JW surface is at p0 = 1000 hPa, so the discrete hydrostatic
    balance of init_jw puts 3 - 4 hPa too much mass in the columns.  1000 hPa lies below the lowest mass level (979 - 985
    hPa) everywhere and is NaN."""
    L = 26
    st = init_jw.make_state(grid2562, L, _abi.INDEX_CORRECTED)
    f = dict(st.f)
    lev = np.arange(L + 1)[None, :] < L
    f["pressure_base"] = np.where(lev, f["zz"] * RGAS * f["exner_base"] * f["rtheta_base"], 0.0)
    f["vorticity"] = np.zeros((grid2562.nVertices, L + 1))
    out = isobaric_ref(f, st.static, L, [85000.0, 100000.0])
    dps = out["surface_pressure"] - 1.0e5
    assert 0.0 <= dps.min() and dps.max() <= 500.0, (dps.min(), dps.max())
    dT = np.abs(out["temperature"][:, 0] - _T_jw(0.85, st.static["latCell"]))
    assert dT.max() <= 0.6, dT.max()
    assert np.isnan(out["temperature"][:, 1]).all()
    for name, _ in ROW:
        assert np.isfinite(out[name][:, 0]).all(), name
