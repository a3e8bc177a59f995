"""Exact global integrals on the device (mpasb200_integrate, k_integrate): the limbs equal the exact sum of the numpy
products, with the SFC renumbering on and off; emulated ranks merge to the single handle's bits before and after RK3
steps; atm_advance_scalars conserves every tracer's mass at every RK stage; the N-GPU run over NCCL where the box has
the GPUs."""
import math
import os
import struct
import subprocess
import sys
from fractions import Fraction

import numpy as np
import pytest

from mpas_regent_b200 import _abi

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NL, BIAS = _abi.INTEGRAL_LIMBS, _abi.INTEGRAL_BIAS


def _canonical(N):
    out = []
    for _ in range(NL - 1):
        out.append(N & 0xffffffff)
        N >>= 32
    return np.array(out + [N], dtype=np.int64)


def _want(p):
    """limbs, counts and value of the exact sum of the finite products p"""
    fin = np.isfinite(p)
    N = 0
    for x in p[fin & (p != 0)].tolist():
        n, d = x.as_integer_ratio()
        N += n * ((1 << BIAS) // d)
    w = {"limbs": _canonical(N), "count": p.size, "n_nan": int(np.isnan(p).sum()), "n_pinf": int((p == np.inf).sum()),
         "n_ninf": int((p == -np.inf).sum())}
    if w["n_nan"] or (w["n_pinf"] and w["n_ninf"]):
        w["value"] = math.nan
    elif w["n_pinf"] or w["n_ninf"]:
        w["value"] = math.inf if w["n_pinf"] else -math.inf
    else:
        w["value"] = float(Fraction(N, 1 << BIAS))
    return w


def _assert_is(got, want, what):
    assert np.array_equal(got["limbs"], want["limbs"]), what
    assert all(got[k] == want[k] for k in ("count", "n_nan", "n_pinf", "n_ninf")), (what, got, want)
    assert struct.pack("<d", got["value"]) == struct.pack("<d", want["value"]) or (math.isnan(got["value"]) and math.isnan(want["value"])), \
        (what, got["value"], want["value"])


def _wild(rng, shape, nonfinite=False):
    """magnitudes 1e-300 .. 1e300, subnormals, pairs that cancel exactly, and (optionally) NaN / +Inf / -Inf"""
    x = rng.standard_normal(shape) * 10.0 ** rng.integers(-300, 301, shape)
    f = x.reshape(-1)
    idx = rng.permutation(f.size)
    m = f.size // 10
    f[idx[:m]] = rng.integers(-(1 << 40), 1 << 40, m) * 5e-324                     # subnormals (exact multiples of 2^-1074)
    f[idx[2 * m:3 * m]] = -f[idx[m:2 * m]]                                            # heavy cancellation
    if nonfinite:
        f[idx[-9:]] = [np.nan, np.inf, -np.inf, np.nan, np.inf, 1e300, 1e300, -1e300, 1e-300]
    return x


def _handle(mesh, L, sfc):
    from mpas_regent_b200 import dynamics, init_jw
    st, _ = init_jw.make_static(mesh, L, _abi.INDEX_CORRECTED)
    g = dynamics.Dynamics(dynamics.dims_of(mesh, L), _abi.default_config(sfc_renumber=sfc))
    g.upload_mesh(st.static)
    return g


@pytest.mark.parametrize("which", ["x1.2562", "icosa642"])
def test_integrate_is_the_exact_sum_of_the_numpy_products(grid2562, grid642, which):
    """((a * b) * wh) * wv with every multiply rounded once, as numpy does it; the device limbs are the exact sum of the
    finite products, the value that sum rounded once, the counts those of NaN / +Inf / -Inf; with sfc_renumber on and off"""
    mesh = grid2562 if which == "x1.2562" else grid642
    L = 7
    L1, n = L + 1, mesh.nCells
    rng = np.random.default_rng(7)
    a_wide = _wild(rng, (n, L1))
    a_nf, b_nf = _wild(rng, (n, L1), nonfinite=True), _wild(rng, (n, L1), nonfinite=True)
    theta = rng.standard_normal((n, L1)) * 300.0
    rho = rng.random((n, L1)) * 1.2
    q = rng.random((n, L1, 8)) * 10.0 ** rng.integers(-12, 3, (n, L1, 8))
    wh = rng.random(n) * 10.0 ** rng.integers(-150, 150, n)
    wh[::97] = 0.0
    wv = rng.random(L1) * 10.0 ** rng.integers(-100, 100, L1)
    ue = _wild(rng, (mesh.nEdges, L1))
    with np.errstate(all="ignore"):          # products overflow, underflow and meet 0 * inf on purpose
        cases = [  # (name, kwargs of integrate, products)
            ("wide", dict(a="w"), a_wide),
            ("wide_part", dict(a="w", n_first=n // 3, nlevels=L), a_wide[:n // 3, :L]),
            ("two_fields_both_weights", dict(a="theta_m", b="rho_zz", weight_id="wh", wv=wv), ((theta * rho) * wh[:, None]) * wv),
            ("nonfinite", dict(a="rtheta_p", b="rho_p"), a_nf * b_nf),
            ("nonfinite_weighted", dict(a="rtheta_p", b="rho_p", weight_id="wh", wv=wv), ((a_nf * b_nf) * wh[:, None]) * wv),
            ("scalars_slot", dict(a="scalars", slot_a=5, b="rho_zz", weight_id="wh", wv=wv[:L], nlevels=L),
             ((q[:, :L, 5] * rho[:, :L]) * wh[:, None]) * wv[:L]),
            ("scalar_is_b", dict(a="rho_zz", b="scalars", slot_b=2), rho * q[:, :, 2]),
            ("edges", dict(a="u", n_first=mesh.nEdges - 5), ue[:mesh.nEdges - 5]),
        ]
        cases = [(nm, kw, _want(np.asarray(p))) for nm, kw, p in cases]
    assert any(w["n_nan"] and w["n_pinf"] and w["n_ninf"] for _, _, w in cases)
    got = {}
    for sfc in (1, 0):
        g = _handle(mesh, L, sfc)
        for nm, arr in (("w", a_wide), ("rtheta_p", a_nf), ("rho_p", b_nf), ("theta_m", theta), ("rho_zz", rho), ("scalars", q), ("u", ue)):
            g.upload_field(nm, arr)
        wid = g.register_weights(_abi.CELL, wh)
        for nm, kw, want in cases:
            kw = dict(kw, weight_id=wid) if "weight_id" in kw else kw
            r = g.integrate(**kw)
            _assert_is(r, want, (which, sfc, nm))
            got[(sfc, nm)] = r["limbs"]
        g.close()
    for nm, _, _ in cases:
        assert np.array_equal(got[(1, nm)], got[(0, nm)]), nm


def test_integrate_rejects_bad_arguments(grid642):
    from mpas_regent_b200 import dynamics
    g = _handle(grid642, 5, 1)
    wid = g.register_weights(_abi.CELL, np.ones(grid642.nCells))
    eid = g.register_weights(_abi.EDGE, np.ones(grid642.nEdges))
    bad = [dict(a="rdzw"), dict(a="w", slot_a=1), dict(a="scalars", slot_a=8), dict(a="w", b="u"), dict(a="w", b="scalars", slot_b=-1),
           dict(a="w", weight_id=eid), dict(a="w", weight_id=7), dict(a="w", n_first=grid642.nCells + 1), dict(a="w", n_first=-1),
           dict(a="w", nlevels=0), dict(a="w", nlevels=7)]
    for kw in bad:
        with pytest.raises(dynamics.MpasB200Error, match=r"\(-1\)"):
            g.integrate(**kw)
    with pytest.raises(dynamics.MpasB200Error, match=r"\(-1\)"):
        g.register_weights(_abi.CELL, np.ones(grid642.nCells - 1))
    assert g.integrate("w", weight_id=wid, n_first=0)["count"] == 0
    g.close()


def _integrals(g, area_id, lm=None):
    """what an N-rank run compares: mass, a mass-weighted theta_m, ke (cells, areaCell x 1/rdzw), u and vorticity (plain)"""
    from mpas_regent_b200 import parallel
    own = (lambda e: None) if lm is None else (lambda e: lm.n_owned[e])
    L = g.dims.nVertLevels
    dz = 1.0 / g.download_field("rdzw")[:L]
    out = parallel.column_integrals(g, area_id, own(0), fields=("rho_zz", "ke"))
    out["theta_rho"] = g.integrate("theta_m", b="rho_zz", weight_id=area_id, wv=dz, n_first=own(0), nlevels=L)
    out["u"] = g.integrate("u", n_first=own(1))
    out["vorticity"] = g.integrate("vorticity", n_first=own(2))
    return out


def _assert_merged_equal(single, backs, shards, ids, area_id):
    from mpas_regent_b200 import parallel
    ref = _integrals(single, area_id)
    per = [_integrals(b, i, sh["lm"]) for b, i, sh in zip(backs, ids, shards)]
    for k, r in ref.items():
        m = parallel.merge_integrals([p[k] for p in per])
        assert np.array_equal(m["limbs"], r["limbs"]) and m["bits"] == r["bits"], k
        assert all(m[c] == r[c] for c in ("count", "n_nan", "n_pinf", "n_ninf")), k
    assert np.isfinite(ref["rho_zz"]["value"]) and ref["rho_zz"]["value"] > 0
    return ref


@pytest.mark.parametrize("physics", [_abi.PHYSICS_LITERAL, _abi.PHYSICS_CORRECTED], ids=["literal", "corrected_physics"])
@pytest.mark.parametrize("colouring", ["sfc", "random", "random_blocks"])
def test_emulated_ranks_merge_to_the_single_handle(grid642, colouring, physics):
    """ranks as handles on one GPU (the colourings of test_device_init_gpu): the merged integrals over owned entities have
    the single handle's limbs on the device-built initial state and after 3 RK3 steps"""
    from mpas_regent_b200 import init_jw, parallel
    from tests.test_device_init_gpu import _colouring, _PackUnpack, _ranks, _single
    from tests.test_parallel import DT, _task_schedule
    L = 6
    cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, physics_mode=physics)
    st, draws, single = _single(grid642, L, cfg)
    col, world = _colouring(grid642, colouring)
    shards, backs = _ranks(grid642, L, cfg, st, draws, col, world)
    ex = _PackUnpack(backs, shards)
    ex.exchange(parallel.INIT_EXCHANGE)
    area_id = single.register_weights(_abi.CELL, init_jw.jw_inputs(grid642, st, draws)["areaCell"])
    ids = [b.register_weights(_abi.CELL, init_jw.jw_inputs(grid642, st, draws, sh["lm"])["areaCell"]) for b, sh in zip(backs, shards)]
    before = _assert_merged_equal(single, backs, shards, ids, area_id)
    exchanges = parallel.exchanges_for(cfg)
    single.atm_compute_solve_diagnostics(False, -1)
    for b in backs:
        b.atm_compute_solve_diagnostics(False, -1)
    ex.exchange(exchanges["compute_solve_diagnostics"])
    seq = _task_schedule(cfg)
    for _ in range(3):
        single.atm_srk3(DT)
        for name, args in seq:
            for b in backs:
                b._call(name, *args)
            spec = exchanges.get(parallel.exchange_key(name, args))
            if spec:
                ex.exchange(spec)
    after = _assert_merged_equal(single, backs, shards, ids, area_id)
    assert any(before[k]["bits"] != after[k]["bits"] for k in before)      # LITERAL physics never updates u, but theta_m moves
    for b in backs:
        b.close()
    single.close()


@pytest.mark.parametrize("physics", [_abi.PHYSICS_CORRECTED, _abi.PHYSICS_LITERAL], ids=["corrected_physics", "literal"])
def test_advance_scalars_conserves_tracer_mass_at_every_stage(grid642, physics):
    """rho_zz * s = s_old * rho_zz_old_split + dt * (tend - rdzw * d(wdtn)): every edge flux enters its two cells with
    opposite signs and wdtn = 0 at levels 0 and L, so I(rho_zz * scalars[s]) after atm_advance_scalars equals
    I(rho_zz_old_split * scalars_old[s]) (areaCell x 1/rdzw, levels 0..L-1) to rounding, for every slot and RK stage.
    Under LITERAL physics ruAvg stays 0 and only the vertical flux moves the tracers.  Rounding is relative to the terms
    summed, so the bound is 1e-13 of the integral of |rho_zz * s|.  On this state the non-monotone transport drives the
    seeded positive tracers far negative within the first step (min s ~ -3 after stage 0, ~ -2e3 after stage 1, from
    1e-3), so the sum cancels and 1e-13 of the tracer mass itself holds at stage 0 only; in a second step CORRECTED
    physics reaches NaN.  Both are properties of the transport on this state, not of the flux form, which the test pins."""
    from mpas_regent_b200 import init_jw
    from tests.test_device_init_gpu import _single
    from tests.test_parallel import DT
    L = 6
    cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, physics_mode=physics, config_scalar_advection=1)
    st, draws, g = _single(grid642, L, cfg)
    g.atm_compute_solve_diagnostics(False, -1)
    g.upload_field("scalars", 1e-3 * (1.0 + np.random.default_rng(3).random((grid642.nCells, L + 1, 8))))
    area = init_jw.jw_inputs(grid642, st, draws)["areaCell"]
    area_id = g.register_weights(_abi.CELL, area)
    dz = 1.0 / g.download_field("rdzw")[:L]
    w = area[:, None] * dz[None, :]
    rows = []

    def hook(name, *args):
        if name == "advance_scalars":
            rho = g.download_field("rho_zz")[:, :L]
            q, q0 = g.download_field("scalars")[:, :L], g.download_field("scalars_old")[:, :L]
            for s in range(8):
                new = g.integrate("rho_zz", b="scalars", slot_b=s, weight_id=area_id, wv=dz, nlevels=L)["value"]
                old = g.integrate("rho_zz_old_split", b="scalars_old", slot_b=s, weight_id=area_id, wv=dz, nlevels=L)["value"]
                scale = float(np.abs(rho * q[:, :, s] * w).sum())
                rows.append((len(rows) // 8, s, new, old, abs(new - old) / scale, float(q[:, :, s].min()),
                             float(np.abs(q[:, :, s] - q0[:, :, s]).max())))
            if physics == _abi.PHYSICS_LITERAL:
                assert not g.download_field("ruAvg").any()

    g.atm_srk3_by_tasks(DT, hook)
    for r in rows:
        print("stage %d slot %d  new %.17g old %.17g  err/sum|terms| %.2e  min s %.3e  max|s-s_old| %.3e" % r)
    assert len(rows) == 3 * 8 and all(np.isfinite(r[2:]).all() for r in rows) and min(r[6] for r in rows) > 0.0
    bad = [r for r in rows if not r[4] <= 1e-13 or (r[0] == 0 and not abs(r[2] - r[3]) <= 1e-13 * abs(r[3]))]
    assert not bad, bad[:8]
    g.close()


def test_nccl_ranks_integrals_equal_single_gpu():
    """merged integrals of N ranks over NCCL (tests/run_integrals_multigpu.py) == one GPU, bitwise (>= 2 GPUs)"""
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    n = 2 if n < 4 else 4
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr",
                          "127.0.0.1", "--master-port", "29547", os.path.join(ROOT, "tests", "run_integrals_multigpu.py")],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0 and "MULTIGPU_INTEGRALS_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-3000:]
