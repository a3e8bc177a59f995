#!/usr/bin/env python
"""run_device_init.py -- every rank builds its shard of the initial state on its own GPU, then runs the RK3 step.

    python run_device_init.py [--mesh CELLS] [--levels L] [--steps K] [--warmup W]                 (one GPU)
    torchrun --nproc-per-node N run_device_init.py [--mesh CELLS] [--levels L] [--steps K] [--warmup W]

Rank 0 builds the mesh and the level-0 data only (init_jw.make_static: no 3-D array exists on the host) and partitions it
(parallel.make_static_shards); the shards are staged as .npy files in a temporary directory (under /dev/shm when there is
one) and every rank loads its own.  Every rank then builds the JW state of the rows it holds on its GPU
(init_jw.init_on_device), repairs the ghost rows with one exchange (parallel.INIT_EXCHANGE, over NCCL), runs
atm_compute_solve_diagnostics(-1) with its exchange and K steps of the library's distributed driver (mpasb200_srk3_dist;
atm_srk3 on one GPU) with bench.dt_for(nCells).  bench.py itself keeps the host-generated inputs.

Prints one JSON line: init seconds (host mesh / level-0 data, shard loading, device), peak host RSS per rank, ms per step,
bench.run_check's combined checksum over owned entities (identical at every N when the N-rank state is bit-identical to
the single-partition one), the total mass (rho_zz x areaCell x 1/rdzw) and the same integral of ke, exact and merged
over ranks (parallel.column_integrals: the same bits at every N), and the name and power limit of the card (read, never
set).  --time-make-state also times, on rank 0 after everything else (so the peak RSS above is the device path's), the host generator bench.py uses for the same
mesh (icosa mesh + init_jw.make_state), for comparison with the init seconds.
"""
import argparse
import datetime
import json
import os
import resource
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402


def card(index: int) -> dict:
    """name and power limit of one GPU as nvidia-smi reports them (None when it cannot be asked)"""
    import torch
    out = {"name": torch.cuda.get_device_name(index), "power_limit_w": None}
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        name, limit = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        out.update(name=name, power_limit_w=float(limit))
    except Exception:
        pass
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mesh", type=int, default=163842)
    ap.add_argument("--levels", type=int, default=55)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--time-make-state", action="store_true", help="also time the host generator (make_state) on rank 0")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    import torch
    from mpas_regent_b200 import _abi, dynamics, icosa, init_jw, parallel

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("run_device_init.py needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        # ranks 1..N-1 wait in a collective while rank 0 builds the mesh and every shard in Python: at x1.2621442 that can
        # outlast the default process-group timeout, after which the watchdog aborts the job
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(hours=2))
    L, nC = args.levels, args.mesh
    dt = bench.dt_for(nC)
    cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, device=local_rank, gather_stage=-1)   # bench.py's step
    stream = torch.cuda.Stream()

    # ---- host: mesh and level-0 data on rank 0 only, one shard per rank ----
    t0 = time.perf_counter()
    lm = None
    if world == 1:
        mesh = icosa.make_icosahedral_mesh(nC)
        st, draws = init_jw.make_static(mesh, L, _abi.INDEX_CORRECTED)
        sh = dict(static=st.static, vert=st.vert, jw=init_jw.jw_inputs(mesh, st, draws))
        del mesh, st, draws
        t_host = time.perf_counter() - t0
        t_load = 0.0
    else:
        box = [None]
        if rank == 0:
            mesh = icosa.make_icosahedral_mesh(nC)
            st, draws = init_jw.make_static(mesh, L, _abi.INDEX_CORRECTED)
            stage = tempfile.mkdtemp(prefix="mpas_b200_shards_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
            for r, s in enumerate(parallel.make_static_shards(st, world)):
                s.update(vert=st.vert, jw=init_jw.jw_inputs(mesh, st, draws, s["lm"]))
                parallel.save_shard(os.path.join(stage, f"rank{r}"), s)
            del mesh, st, draws, s
            box = [stage]
        dist.broadcast_object_list(box, src=0)
        t_host = time.perf_counter() - t0
        t1 = time.perf_counter()
        sh = parallel.load_shard(os.path.join(box[0], f"rank{rank}"))
        lm = sh["lm"]
        dist.barrier()
        if rank == 0:
            shutil.rmtree(box[0], ignore_errors=True)
        t_load = time.perf_counter() - t1
    n_loc = (len(lm.cells), len(lm.edges), len(lm.vertices)) if lm is not None else (
        sh["static"]["nEdgesOnCell"].shape[0], sh["static"]["cellsOnEdge"].shape[0], sh["static"]["edgesOnVertex"].shape[0])

    # ---- device: the JW state of the rows held, the init exchange, the diagnostics of atm_core_init ----
    g = dynamics.Dynamics(_abi.make_dims(*n_loc, L), cfg)
    g.set_stream(stream.cuda_stream)
    g.upload_mesh(sh["static"])
    area_id = g.register_weights(_abi.CELL, sh["jw"]["areaCell"])
    g.sync(); torch.cuda.synchronize()
    t2 = time.perf_counter()
    with torch.cuda.stream(stream):
        init_jw.init_on_device(g, sh["static"], sh["jw"], sh["vert"])
        if world > 1:
            parallel.NcclExchanger(g, lm, stream).exchange(parallel.INIT_EXCHANGE)
            run = parallel.NativeDistributedDynamics(g, lm, rank, world)
            run.init_diagnostics()
            step = lambda: run.step(dt)
        else:
            g.atm_compute_solve_diagnostics(False, -1)
            step = lambda: g.atm_srk3(dt)
        g.sync(); torch.cuda.synchronize()
    t_dev = time.perf_counter() - t2
    del sh

    # ---- K steps, timed with CUDA events on the stream that carries them ----
    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            step()
        if world > 1:
            run.flush()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            step()
        if world > 1:
            run.flush()
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        check = bench.run_check(g, lm, dist, world)
        integrals = parallel.column_integrals(g, area_id, None if lm is None else lm.n_owned[0], dist if world > 1 else None)
    mine = {"ms": ms, "t_load": t_load, "t_dev": t_dev, "rss_gb": resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 2 ** 20,
            "card": card(local_rank)}
    ranks = [mine]
    if world > 1:
        ranks = [None] * world
        dist.all_gather_object(ranks, mine)
    host_gen = None
    if args.time_make_state and rank == 0:
        t3 = time.perf_counter()
        mesh = icosa.make_icosahedral_mesh(nC)
        t4 = time.perf_counter()
        init_jw.make_state(mesh, L, _abi.INDEX_CORRECTED, m5=True, diag_on_host=False)
        host_gen = {"icosa_mesh_s": round(t4 - t3, 3), "make_state_s": round(time.perf_counter() - t4, 3)}
        del mesh
    if rank == 0:
        line = {"what": "device-built initial state (init_jw.init_on_device per rank) + RK3 steps", "mesh": nC, "levels": L,
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "dt": dt,
                "ms_per_step": max(r["ms"] for r in ranks) / args.steps,
                "init_s": {"host_mesh_static": round(t_host, 3), "shard_load_max": round(max(r["t_load"] for r in ranks), 3),
                           "device_max": round(max(r["t_dev"] for r in ranks), 3)},
                "peak_host_rss_gb": [round(r["rss_gb"], 3) for r in ranks],
                "combined_checksum": check["combined_checksum"], "finite": check["finite"],
                "integrals": {"what": "exact sum over owned cells and levels 0..L-1 of field x areaCell x (1/rdzw)",
                              **{"mass" if f == "rho_zz" else f: {"value": r["value"], "bits": r["bits"]} for f, r in integrals.items()}},
                "gpus": [r["card"] for r in ranks], "host_generator": host_gen}
        print(json.dumps(line), flush=True)
    g.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
