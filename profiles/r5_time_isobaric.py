#!/usr/bin/env python
"""Time one call of the pressure-level diagnostics (mpasb200_isobaric_diagnostics, 10 pressure levels) against the
download of the fields a host-side tool would need for the same output, on a device-built state.

    python profiles/r5_time_isobaric.py [--mesh 655362] [--levels 55] [--reps 20] [--out FILE]

The state is the JW initial state built on the device (init_jw.init_on_device) plus atm_compute_solve_diagnostics(-1),
as run_device_init.py builds it at N = 1.  The call is synchronous: it is timed with the host clock around the call (the
launch, the kernel, the copy of the [nCells][1 + 6 x 10] result to pageable host memory and the synchronise), after one
warm-up call, and in a separate pass per kernel with CUDA events (mpasb200_enable_kernel_timing).  The same run times
download_field of pressure_base, pressure_p, theta_m, exner, zgrid, w, u and vorticity (median of --reps / 4 rounds).  At
x1.655362 x 55 the fields k_isobaric reads are several GB, far above the 126 MB of L2.

Algorithmic bytes of k_isobaric per cell (n = nEdgesOnCell, B = targets bracketed in the column, P = requested levels):
    16 L                   the pressure column, pressure_base + pressure_p at levels 0..L-1
  + 24                     zgrid levels 0..2 (surface pressure)
  + 40 + 44 n              map, nEdgesOnCell, four trig values; per slot edgesOnCell, verticesOnCell, kiteForCell (4 B each),
                           coeffs_reconstruct (24 B), kiteAreasOnVertex (8 B)
  + B (112 + 32 n)         per bracketed target: pressure_base, pressure_p, theta_m, exner at k*, k*+1 (64 B), zgrid and w at
                           k*..k*+2 (48 B), u and vorticity at k*, k*+1 on the cell's n edges and n vertices
  + 8 (1 + 6 P)            the output row
Prints one JSON line with the card's name and power limit (read, never set).
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PLEV_HPA = (1000, 925, 850, 700, 500, 300, 250, 200, 100, 50)
HOST_INPUTS = ("pressure_base", "pressure_p", "theta_m", "exner", "zgrid", "w", "u", "vorticity")


def algorithmic_bytes(L: int, n_edges: "np.ndarray", bracketed: "np.ndarray", P: int) -> int:
    """k_isobaric's algorithmic bytes summed over cells (see the module docstring)"""
    n = n_edges.astype(int)
    b = bracketed.astype(int)
    return int((16 * L + 24 + 40 + 44 * n + b * (112 + 32 * n) + 8 * (1 + 6 * P)).sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mesh", type=int, default=655362)
    ap.add_argument("--levels", type=int, default=55)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", type=str, default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    import numpy as np
    import torch
    from mpas_regent_b200 import _abi, dynamics, icosa, init_jw
    from run_device_init import card
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    L = args.levels
    mesh = icosa.make_icosahedral_mesh(args.mesh)
    st, draws = init_jw.make_static(mesh, L, _abi.INDEX_CORRECTED)
    jw = init_jw.jw_inputs(mesh, st, draws)
    g = dynamics.Dynamics(dynamics.dims_of(mesh, L), _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, device=0))
    g.upload_mesh(st.static)
    init_jw.init_on_device(g, st.static, jw, st.vert)
    g.atm_compute_solve_diagnostics(False, -1)
    plev = [100.0 * p for p in PLEV_HPA]
    first = g.isobaric_diagnostics(plev)
    host = []
    for _ in range(args.reps):
        t0 = time.perf_counter()
        r = g.isobaric_diagnostics(plev)
        host.append((time.perf_counter() - t0) * 1e3)
        assert all(np.array_equal(r[k].view(np.uint64), first[k].view(np.uint64)) for k in r)
    g.enable_kernel_timing(True)
    for _ in range(args.reps):
        g.isobaric_diagnostics(plev)
    kt = g.kernel_times()
    g.enable_kernel_timing(False)
    k_ms = kt["k_isobaric"][0] / kt["k_isobaric"][1]
    down = {n: [] for n in HOST_INPUTS}
    bufs = {n: np.empty(g.field_shape(n)) for n in HOST_INPUTS}
    for n in HOST_INPUTS:
        g.download_field(n, bufs[n])
    for _ in range(max(args.reps // 4, 1)):
        for n in HOST_INPUTS:
            t0 = time.perf_counter()
            g.download_field(n, bufs[n])
            down[n].append((time.perf_counter() - t0) * 1e3)
    down_ms = {n: float(np.median(v)) for n, v in down.items()}
    nbytes = algorithmic_bytes(L, st.static["nEdgesOnCell"], np.isfinite(first["temperature"]).sum(axis=1), len(plev))
    T = first["temperature"]
    line = {"what": "one isobaric_diagnostics call (10 pressure levels, all cells) vs download_field of its inputs",
            "mesh": args.mesh, "levels": L, "plev_hpa": list(PLEV_HPA), "reps": args.reps,
            "call_host_ms": {"median": float(np.median(host)), "min": min(host), "max": max(host)},
            "kernel_ms_per_call": {k: v[0] / v[1] for k, v in kt.items()},
            "algorithmic_bytes": nbytes, "k_isobaric_gb_per_s": nbytes / k_ms / 1e6,
            "output_bytes": int(8 * T.shape[0] * (1 + 6 * T.shape[1])),
            "download_field_ms": down_ms, "download_total_ms": sum(down_ms.values()),
            "download_bytes": int(sum(bufs[n].nbytes for n in HOST_INPUTS)),
            "ps_min_max": [float(first["surface_pressure"].min()), float(first["surface_pressure"].max())],
            "T_min_max": [[float(np.nanmin(T[:, j])), float(np.nanmax(T[:, j]))] if np.isfinite(T[:, j]).any() else None
                          for j in range(T.shape[1])],
            "card": card(0)}
    print(json.dumps(line), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(json.dumps(line) + "\n")
    g.close()


if __name__ == "__main__":
    main()
