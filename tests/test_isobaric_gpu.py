"""Surface pressure and pressure-level diagnostics on the device (mpasb200_isobaric_diagnostics, k_isobaric) against the
numpy restatement of tests/isobaric_ref.py: the surface pressure and the NaN masks bit for bit, the interpolated values
within 1e-12 of each field's largest value, on three meshes, before and after RK3 steps, with the SFC renumbering on and
off; wild columns; L across one and two 32-level chunks; the call writes nothing; bad arguments; emulated ranks assemble to
the single handle's bits."""
import numpy as np
import pytest

from mpas_regent_b200 import _abi
from tests.isobaric_ref import INPUTS, ROW, isobaric_ref

pytestmark = pytest.mark.gpu

TOL = 1e-12
PLEV = 100.0 * np.array([1050, 1000, 925, 850, 700, 500, 300, 250, 200, 100, 50, 10], dtype=np.float64)
NAMES = ("surface_pressure",) + tuple(n for n, _ in ROW)


def _handle(mesh, L, physics=_abi.PHYSICS_LITERAL, sfc=1):
    """the device-built JW state (init_jw.init_on_device, which also forms pressure_base) and atm_core_init's diagnostics"""
    from tests.test_device_init_gpu import _single
    cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, physics_mode=physics, sfc_renumber=sfc)
    st, _, g = _single(mesh, L, cfg)
    g.atm_compute_solve_diagnostics(False, -1)
    return st, g


def _reference(g, static, plev):
    L = g.dims.nVertLevels
    return isobaric_ref({n: g.download_field(n) for n in INPUTS}, static, L, plev)


def _assert_matches(got, ref, what=""):
    """surface pressure and NaN masks identical; the rest within TOL x the field's largest finite |ref|"""
    assert np.array_equal(got["surface_pressure"], ref["surface_pressure"], equal_nan=True), what
    for name, _ in ROW:
        a, b = got[name], ref[name]
        assert a.shape == b.shape, (what, name)
        assert np.array_equal(np.isnan(a), np.isnan(b)), (what, name, int((np.isnan(a) != np.isnan(b)).sum()))
        fin = np.isfinite(b)
        assert np.array_equal(a[~fin], b[~fin], equal_nan=True), (what, name)
        if fin.any():
            scale = np.abs(b[fin]).max()
            err = np.abs(a[fin] - b[fin]).max()
            assert err <= TOL * scale, (what, name, err, scale)


def _bits_equal(x, y):
    return all(np.array_equal(x[n].view(np.uint64), y[n].view(np.uint64)) for n in NAMES)


def _irregular():
    from tests import irregular
    return irregular.irregular_mesh()


@pytest.mark.parametrize("physics", [_abi.PHYSICS_LITERAL, _abi.PHYSICS_CORRECTED], ids=["literal", "corrected_physics"])
@pytest.mark.parametrize("which", ["x1.2562", "icosa642", "irregular646"])
def test_parity_with_the_restatement(grid2562, grid642, which, physics):
    """initial state and after 3 RK3 steps; the SFC renumbering on and off give the same bits"""
    import bench
    mesh = {"x1.2562": grid2562, "icosa642": grid642}.get(which) or _irregular()
    L = 26
    dt = bench.dt_for(mesh.nCells)
    (st, on), (_, off) = _handle(mesh, L, physics, 1), _handle(mesh, L, physics, 0)
    for stage in ("initial", "3 steps"):
        if stage == "3 steps":
            for _ in range(3):
                on.atm_srk3(dt); off.atm_srk3(dt)
        got = on.isobaric_diagnostics(PLEV)
        ref = _reference(on, st.static, PLEV)
        _assert_matches(got, ref, f"{which} {stage}")
        assert _bits_equal(got, off.isobaric_diagnostics(PLEV)), f"{which} {stage}: sfc_renumber on and off differ"
        T = got["temperature"]
        assert np.isnan(T[:, 0]).all(), stage                                         # 1050 hPa lies below the lowest level
        if stage == "initial":
            assert np.isfinite(T[:, 3]).all() and np.isfinite(got["surface_pressure"]).all()
    on.close(); off.close()


def test_wild_columns(grid642):
    """random pressure columns: non-monotone, equal neighbours, NaN, targets equal to level pressures"""
    L = 12
    st, g = _handle(grid642, L)
    rng = np.random.default_rng(7)
    n = grid642.nCells
    pb = g.download_field("pressure_base")
    pp = rng.normal(0.0, 2.0e4, (n, L + 1))
    rows = rng.choice(n, 200, replace=False)
    for c in rows[:100]:                                  # equal neighbours: both parts equal, so the sums are equal
        k = rng.integers(0, L - 1)
        pb[c, k + 1], pp[c, k + 1] = pb[c, k], pp[c, k]
    pp[rows[100:150], rng.integers(0, L, 50)] = np.nan
    pp[rows[150:160], :] = np.nan
    g.upload_field("pressure_base", pb)
    g.upload_field("pressure_p", pp)
    p = (pb + pp)[:, :L]
    exact = p[rows[:100]][np.isfinite(p[rows[:100]]) & (p[rows[:100]] > 0)]
    plev = np.concatenate([PLEV, rng.choice(exact, 12, replace=False), [PLEV[3], PLEV[3]]])
    rng.shuffle(plev)
    got = g.isobaric_diagnostics(plev)
    ref = _reference(g, st.static, plev)
    _assert_matches(got, ref, "wild")
    T = got["temperature"]
    assert np.isnan(T).any() and np.isfinite(T).any()
    g.close()


@pytest.mark.parametrize("L", [4, 26, 58])
@pytest.mark.parametrize("nplev", [1, 32])
def test_shapes(grid642, L, nplev):
    """one level, and the most levels a call takes (in a shuffled order, with repeats); L = 58 spans two 32-level chunks"""
    st, g = _handle(grid642, L)
    if nplev == 1:
        plev = np.array([50000.0])                        # inside the column at every L here (at L = 4, 850 hPa is not)
    else:
        rng = np.random.default_rng(L)
        plev = np.concatenate([np.geomspace(104000.0, 50.0, 29), PLEV[[3, 3, 5]]])
        rng.shuffle(plev)
    got = g.isobaric_diagnostics(plev)
    assert got["temperature"].shape == (grid642.nCells, nplev)
    _assert_matches(got, _reference(g, st.static, plev), f"L={L} nplev={nplev}")
    assert np.isfinite(got["temperature"]).any()
    g.close()


def _fingerprint(g):
    out = {}
    for name, ent, slots in _abi.FIELDS:
        if ent != _abi.VERTICAL and slots == 1:
            out[name] = g.summarize_field(name)["checksum"]
        else:
            out[name] = g.download_field(name).tobytes()
    return out


def test_the_call_writes_nothing(grid642):
    """every field of the mirror unchanged by the call, and a step after the call bit-identical to a step without it"""
    L = 10
    _, a = _handle(grid642, L, _abi.PHYSICS_CORRECTED)
    _, b = _handle(grid642, L, _abi.PHYSICS_CORRECTED)
    a.atm_srk3(600.0); b.atm_srk3(600.0)
    before = _fingerprint(a)
    a.isobaric_diagnostics(PLEV)
    assert _fingerprint(a) == before
    assert _fingerprint(b) == before
    a.atm_srk3(600.0); b.atm_srk3(600.0)
    assert _fingerprint(a) == _fingerprint(b)
    a.close(); b.close()


def test_rejects_bad_arguments(grid642):
    from mpas_regent_b200 import dynamics
    L = 5
    fresh = dynamics.Dynamics(dynamics.dims_of(grid642, L), _abi.default_config())
    with pytest.raises(dynamics.MpasB200Error, match=r"\(-4\)"):          # before upload_mesh
        fresh.isobaric_diagnostics(PLEV)
    fresh.close()
    _, g = _handle(grid642, L)
    n = grid642.nCells
    for plev in ([], np.full(_abi.ISOBARIC_MAX_LEVELS + 1, 5e4), [5e4, np.nan], [np.inf], [0.0], [-1e4]):
        with pytest.raises(dynamics.MpasB200Error, match=r"\(-1\)"):
            g.isobaric_diagnostics(plev)
    for nf in (-1, n + 1):
        with pytest.raises(dynamics.MpasB200Error, match=r"\(-1\)"):
            g.isobaric_diagnostics(PLEV, n_first=nf)
    out = np.empty((n, 1 + 6 * 2))
    plev = np.array([85000.0, 50000.0])
    assert g._lib.mpasb200_isobaric_diagnostics(g._h, None, 2, n, out.ctypes.data) == -1
    assert g._lib.mpasb200_isobaric_diagnostics(g._h, plev.ctypes.data, 2, n, None) == -1
    assert g._lib.mpasb200_isobaric_diagnostics(None, plev.ctypes.data, 2, n, out.ctypes.data) == -1
    assert g.isobaric_diagnostics(PLEV, n_first=0)["temperature"].shape == (0, len(PLEV))
    some = g.isobaric_diagnostics(PLEV, n_first=17)
    whole = g.isobaric_diagnostics(PLEV)
    assert all(np.array_equal(some[k], whole[k][:17], equal_nan=True) for k in NAMES)
    g.close()


@pytest.mark.parametrize("physics", [_abi.PHYSICS_LITERAL, _abi.PHYSICS_CORRECTED], ids=["literal", "corrected_physics"])
@pytest.mark.parametrize("colouring", ["sfc", "random", "random_blocks"])
def test_emulated_ranks_assemble_to_the_single_handle(grid642, colouring, physics):
    """ranks as handles on one GPU (the colourings of test_device_init_gpu) and the single handle run 3 RK3 steps task by
    task with the exchange schedule: at the initial state and after every exchange that follows atm_compute_solve_diagnostics
    (the end of every RK stage), the rows parallel.isobaric_diagnostics assembles are bit-identical to the single handle's.
    Under CORRECTED physics the recover of the last stage of the first step drives this state's pressure out of the finite
    range (the CPU oracle does the same), so from there on every value is NaN; the stage boundaries before it, where
    recover has moved u and vorticity, are where that mode's rows are compared with finite values."""
    from mpas_regent_b200 import parallel
    from tests.test_device_init_gpu import _colouring, _PackUnpack, _ranks, _single
    from tests.test_parallel import _task_schedule
    L = 6
    cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, physics_mode=physics)
    st, draws, single = _single(grid642, L, cfg)
    col, world = _colouring(grid642, colouring)
    shards, backs = _ranks(grid642, L, cfg, st, draws, col, world)
    ex = _PackUnpack(backs, shards)
    ex.exchange(parallel.INIT_EXCHANGE)
    exchanges = parallel.exchanges_for(cfg)
    single.atm_compute_solve_diagnostics(False, -1)
    for b in backs:
        b.atm_compute_solve_diagnostics(False, -1)
    ex.exchange(exchanges["compute_solve_diagnostics"])
    lms = [sh["lm"] for sh in shards]
    seen = []

    def compare(when):
        want = single.isobaric_diagnostics(PLEV)
        assert _bits_equal(parallel.isobaric_diagnostics(backs, lms, PLEV), want), when
        seen.append(want)

    compare("initial state")
    seq = _task_schedule(cfg)
    for step in range(3):
        for name, args in seq:
            single._call(name, *args)
            for b in backs:
                b._call(name, *args)
            spec = exchanges.get(parallel.exchange_key(name, args))
            if spec:
                ex.exchange(spec)
            if name == "compute_solve_diagnostics":
                compare(f"step {step}, {name}{args}")
    assert len(seen) == 1 + 3 * 3
    # some stage boundary after the initial state has moved rows whose 500 hPa values are all finite
    moved = [w for w in seen[1:] if not _bits_equal(w, seen[0]) and all(np.isfinite(w[n][:, 5]).all() for n, _ in ROW)]
    assert moved, "no stage boundary with moved, finite 500 hPa rows"
    if physics == _abi.PHYSICS_LITERAL:
        assert all(np.isfinite(seen[-1][n][:, 5]).all() for n, _ in ROW)
    for b in backs:
        b.close()
    single.close()
