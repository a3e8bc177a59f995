#!/usr/bin/env python
"""Time one exact integral (mpasb200_integrate: two fields, per-cell and per-level weights) next to the summarize_timestep
scan (mpasb200_summarize_field) of the same field, on a device-built state.

    python profiles/r4_time_integrate.py [--mesh 655362] [--levels 55] [--reps 20]

The state is the JW initial state built on the device (init_jw.init_on_device), as run_device_init.py builds it at N = 1.
Both calls are synchronous; each is timed with the host clock around the call (what a caller waits for, including the
result's copy to the host) and, in a separate pass, per kernel with CUDA events (mpasb200_enable_kernel_timing).  The two
calls alternate, after one warm-up call each.  Two fields of x1.655362 x 56 levels are 587 MB, well above the 126 MB of
L2, so every call reads its fields from HBM.  Prints one JSON line with the card's name and power limit.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mesh", type=int, default=655362)
    ap.add_argument("--levels", type=int, default=55)
    ap.add_argument("--reps", type=int, default=20)
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
    area = g.register_weights(_abi.CELL, jw["areaCell"])
    L1 = L + 1
    dz = np.ones(L1)
    dz[:L] = 1.0 / g.download_field("rdzw")[:L]
    integ = lambda: g.integrate("theta_m", b="rho_zz", weight_id=area, wv=dz)
    summ = lambda: g.summarize_field("theta_m")
    first = integ(), summ()
    host = {"integrate": [], "summarize_field": []}
    for _ in range(args.reps):
        for name, fn in (("integrate", integ), ("summarize_field", summ)):
            t0 = time.perf_counter()
            r = fn()
            host[name].append((time.perf_counter() - t0) * 1e3)
            if name == "integrate":
                assert np.array_equal(r["limbs"], first[0]["limbs"])
    g.enable_kernel_timing(True)
    for _ in range(args.reps):
        integ(); summ()
    kt = g.kernel_times()
    g.enable_kernel_timing(False)
    n = mesh.nCells * L1
    line = {"what": "one exact integral (theta_m x rho_zz x areaCell x dz, all cells and levels) vs summarize_field(theta_m)",
            "mesh": args.mesh, "levels": L, "points": n, "reps": args.reps,
            "integrate_host_ms": {"median": float(np.median(host["integrate"])), "min": min(host["integrate"])},
            "summarize_host_ms": {"median": float(np.median(host["summarize_field"])), "min": min(host["summarize_field"])},
            "kernel_ms_per_call": {k: v[0] / v[1] for k, v in kt.items()},
            "integrate_hbm_gb_per_s": 2 * 8 * n / (kt["k_integrate"][0] / kt["k_integrate"][1]) / 1e6,
            "value": first[0]["value"], "bits": first[0]["bits"], "card": card(0)}
    print(json.dumps(line), flush=True)
    g.close()


if __name__ == "__main__":
    main()
