"""Shared helpers for the parity tests."""
import numpy as np

from mpas_regent_b200 import _abi, dynamics, init_jw

TOL = 1e-12   # BASELINE.json north_star: "within 1e-12 relative (fp64) per field"


def build_pair(mesh, L, policy, m5=True, gpu=True, rkarg=_abi.RKARG_STAGE_INDEX, sfc=1, masks=None, **cfg_over):
    """(state, oracle, gpu-or-None) with identical mesh + fields uploaded; ``masks`` replaces level-0 arrays of the state
    (the regional masks bdyMaskCell, specZoneMaskCell, specZoneMaskEdge, isShared)."""
    from oracle.oracle import Oracle
    st = init_jw.make_state(mesh, L, policy, m5=m5)
    st.static.update(masks or {})
    dims = dynamics.dims_of(mesh, L)
    cfg = _abi.default_config(index_policy=policy, rkarg_policy=rkarg, sfc_renumber=sfc, **cfg_over)
    ora = Oracle(dims, cfg)
    ora.upload_mesh(st.static)
    ora.upload_state(st.f, st.vert)
    g = None
    if gpu:
        g = dynamics.Dynamics(_abi.make_dims(mesh.nCells, mesh.nEdges, mesh.nVertices, L), cfg)
        g.upload_mesh(st.static)
        g.upload_state(st.f, st.vert)
    return st, ora, g


def copy_state(src, dst, names=None):
    for n in (names or [f[0] for f in _abi.FIELDS]):
        dst.upload_field(n, src.download_field(n))


def compare(gpu, ora, names=None, tol=TOL, what=""):
    """Every field, every level 0..nVertLevels: max|gpu-ref| <= tol*max|ref|, NaN/Inf positions identical."""
    bad = []
    worst = (0.0, None)
    for n in (names or [f[0] for f in _abi.FIELDS]):
        a, b = gpu.download_field(n), ora.download_field(n)
        fin_a, fin_b = np.isfinite(a), np.isfinite(b)
        if not np.array_equal(np.isnan(a), np.isnan(b)) or not np.array_equal(np.isinf(a), np.isinf(b)):
            bad.append((n, "nan/inf mask differs", int((fin_a != fin_b).sum())))
            continue
        if not np.array_equal(a[~fin_b], b[~fin_b], equal_nan=True):
            bad.append((n, "inf sign differs", 0))
            continue
        ref = np.abs(b[fin_b]).max() if fin_b.any() else 0.0
        err = np.abs(a[fin_b] - b[fin_b]).max() if fin_b.any() else 0.0
        rel = err / ref if ref > 0 else (0.0 if err == 0 else np.inf)
        if rel > worst[0]:
            worst = (rel, n)
        if rel > tol:
            bad.append((n, f"rel {rel:.3e} (abs {err:.3e}, ref {ref:.3e})", int((np.abs(a - b) > tol * ref).sum())))
    assert not bad, f"{what}: {len(bad)} field(s) out of tolerance: {bad[:12]}"
    return worst


def ulp_histogram(a, b):
    """element-wise distance in units of the last place between two float64 arrays (the report behind the
    bit-identical claims: compare() above is norm-wise per field and says nothing about small-magnitude elements)."""
    a = np.ascontiguousarray(a, dtype=np.float64); b = np.ascontiguousarray(b, dtype=np.float64)
    both_nan = np.isnan(a) & np.isnan(b)
    one_nan = np.isnan(a) ^ np.isnan(b)

    def ordered(x):                                                     # monotone double -> uint64 (-0.0 sits 1 below +0.0)
        u = x.view(np.uint64)
        return np.where(u >> np.uint64(63) != 0, ~u, u | np.uint64(1 << 63))

    ka, kb = ordered(a), ordered(b)
    d = (np.maximum(ka, kb) - np.minimum(ka, kb)).astype(np.float64)       # exact below 2^53, which is all that matters here
    d[both_nan] = 0
    d[one_nan] = np.inf
    h = {"0": int((d == 0).sum()), "1": int((d == 1).sum()), "2-4": int(((d >= 2) & (d <= 4)).sum()),
         "5-16": int(((d > 4) & (d <= 16)).sum()), "17-256": int(((d > 16) & (d <= 256)).sum()),
         ">256": int((d > 256).sum()), "max_ulp": float(d.max()) if d.size else 0.0, "n": int(d.size)}
    return h
