#!/usr/bin/env python
"""Time restart.save and restart.load at x1.655362 x 55 on one GPU (the JW state built on the device).

    python profiles/r6_time_restart.py [--mesh CELLS] [--levels L] [--dir DIR] [--out JSON]

Prints one JSON line: the bytes of the restart set, the seconds of save and load, and their split into device-to-host
(host-to-device) copies, timed separately over the same fields, and the rest (file I/O and checksums); GB/s for each; the
share of ghost rows an N-rank save would copy for N = 2, 4, 8 (SFC colouring); the card's name and power limit.
"""
import argparse
import json
import os
import shutil
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mesh", type=int, default=655362)
    ap.add_argument("--levels", type=int, default=55)
    ap.add_argument("--dir", type=str, default=None, help="where the restart is written (default: a temporary directory)")
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    import run_device_init
    from mpas_regent_b200 import _abi, dynamics, icosa, init_jw, parallel, restart
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    L = args.levels
    mesh = icosa.make_icosahedral_mesh(args.mesh)
    st, draws = init_jw.make_static(mesh, L, _abi.INDEX_CORRECTED)
    cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, device=0)
    g = dynamics.Dynamics(dynamics.dims_of(mesh, L), cfg)
    g.upload_mesh(st.static)
    init_jw.init_on_device(g, st.static, init_jw.jw_inputs(mesh, st, draws), st.vert)
    g.atm_compute_solve_diagnostics(False, -1)
    g.atm_srk3(run_device_init.bench.dt_for(args.mesh))
    g.sync()
    names = _abi.restart_fields(cfg)
    nbytes = sum(int(np.prod(g.field_shape(n))) * 8 for n in names)
    # copies alone, the same fields into host memory and back
    t0 = time.perf_counter()
    host = {n: g.download_field(n) for n in names}
    t_d2h = time.perf_counter() - t0
    t0 = time.perf_counter()
    for n in names:
        g.upload_field(n, host[n])
    g.sync()
    t_h2d = time.perf_counter() - t0
    del host
    d = args.dir or tempfile.mkdtemp(prefix="mpas_b200_restart_")
    path = os.path.join(d, "restart")
    t0 = time.perf_counter()
    restart.save(path, g, None, 1, mesh)
    t_save = time.perf_counter() - t0
    h = dynamics.Dynamics(dynamics.dims_of(mesh, L), cfg)
    h.upload_mesh(st.static)
    t0 = time.perf_counter()
    restart.load(path, h, None, mesh)
    h.sync()
    t_load = time.perf_counter() - t0
    same = all(np.array_equal(g.download_field(n), h.download_field(n), equal_nan=True) for n in names)
    ghost = {}
    for world in (2, 4, 8):
        shards = parallel.make_static_shards(st, world)
        held = sum(len(s["lm"].cells) for s in shards)
        ghost[world] = round(1.0 - mesh.nCells / held, 4)
    if args.dir is None:
        shutil.rmtree(d, ignore_errors=True)
    gb = nbytes / 1e9
    line = {"what": "restart.save / restart.load of the restart set, one GPU", "mesh": args.mesh, "levels": L,
            "fields": len(names), "bytes": nbytes, "save_s": round(t_save, 3), "load_s": round(t_load, 3),
            "d2h_s": round(t_d2h, 3), "h2d_s": round(t_h2d, 3),
            "save_rest_s": round(t_save - t_d2h, 3), "load_rest_s": round(t_load - t_h2d, 3),
            "save_gbs": round(gb / t_save, 3), "load_gbs": round(gb / t_load, 3),
            "d2h_gbs": round(gb / t_d2h, 3), "h2d_gbs": round(gb / t_h2d, 3),
            "loaded_equals_saved": bool(same), "ghost_row_share_cells_sfc": ghost,
            "gpu": run_device_init.card(0)}
    print(json.dumps(line), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(line, fh)


if __name__ == "__main__":
    main()
