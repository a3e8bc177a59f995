#!/usr/bin/env python
"""bench.py -- RK3 dynamics step throughput (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--mesh CELLS] [--levels L] [--impl reference] [--dump-outputs DIR]

One "step" = one atm_srk3 (reference: dynamics/rk_timestep.rg:361-500) over the whole synthetic
icosahedral mesh.  metric = cell-level updates/s = nCells * nVertLevels * steps / seconds (whole job).
Under torchrun (N > 1) the mesh is partitioned across ranks (strong scaling: the global mesh is fixed).

Timed with CUDA events on the stream the kernels are launched on, max over ranks, barrier +
synchronize on both sides.  Extra objects on the JSON line: roofline (dominant kernel, algorithmic
bytes / CUDA-event duration / measured HBM peak), cpu_baseline (the CPU oracle on a bounded sample,
rank 0, N=1), e2e (same metric through the C ABI with host buffers: H2D of the prognostic state from
pinned memory + step + D2H, every step), clocks, gpu_launches.

--impl reference times the reference's CPU implementation of the path.  The reference is Regent and
cannot be built here, so this arm runs the oracle port (oracle/, a literal C++ restatement) with all
host threads on a bounded sample of the same workload.

--dump-outputs DIR writes what the last timed step left in the fields the check scans (CHECK_FIELDS) as DIR/<field>.npy,
float64: the same seeded sample of rows (entities, every level) at every run with the same --mesh / --levels, so that two
builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "cell_level_updates_per_s"
UNIT = "cell-levels/s"
DT_REF = 720.0           # constants.rg:99, scaled with resolution to keep the CFL number (SURVEY.md 8d)
E2E_FIELDS = ("u", "ru", "w", "theta_m", "rho_zz", "rw", "rho_p", "rtheta_p", "exner", "pressure_p")
# fields scanned by the device form of summarize_timestep (rk_timestep.rg:29-359) after the timed loop: the prognostic state,
# the acoustic perturbation variables and the tendencies / diagnostics every task of the step feeds into
CHECK_FIELDS = ("u", "w", "theta_m", "rho_zz", "ru", "rw", "rho_p", "rtheta_p", "rtheta_pp", "rho_pp", "rw_p", "ru_p", "wwAvg",
                "ruAvg", "tend_u", "tend_theta", "tend_rho", "pv_edge", "ke", "divergence", "vorticity", "v")
DUMP_BYTES = 48 << 20    # --dump-outputs: all fields together; a field of the headline mesh is 0.3-0.9 GB, so rows are sampled
DUMP_SEED = 20260


def dt_for(n_cells: int) -> float:
    return DT_REF * (2562.0 / n_cells) ** 0.5


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and "Active" in r[col] and "Not" not in r[col]:
                    reasons.add(name)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def build_inputs(n_cells: int, L: int):
    """Synthetic mesh + JW-style state, generated on the host (deterministic).  The result is cached
    as raw .npy files under $MPAS_B200_CACHE (default /tmp/mpas_b200_cache) so that repeated
    invocations on one box (scaling runs, profiler passes) do not regenerate it."""
    from mpas_regent_b200 import _abi, icosa, init_jw
    from mpas_regent_b200.mesh import Mesh
    t0 = time.time()
    cache = os.path.join(os.environ.get("MPAS_B200_CACHE", "/tmp/mpas_b200_cache"), f"x1.{n_cells}_L{L}")
    done = os.path.join(cache, "DONE")
    if os.path.exists(done):
        def load(sub):
            d = os.path.join(cache, sub)
            return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d)) if f.endswith(".npy")}
        mesh = Mesh(v=load("mesh"), name=f"x1.{n_cells}")
        st = init_jw.HostState(nVertLevels=L, policy=_abi.INDEX_CORRECTED, mesh=mesh, static=load("static"), f=load("f"),
                               vert=load("vert"))
        return mesh, st, time.time() - t0
    mesh = icosa.make_icosahedral_mesh(n_cells)
    st = init_jw.make_state(mesh, L, _abi.INDEX_CORRECTED, m5=True, diag_on_host=False)
    try:
        for sub, d in (("mesh", st.mesh.v), ("static", st.static), ("f", st.f), ("vert", st.vert)):
            os.makedirs(os.path.join(cache, sub), exist_ok=True)
            for k, a in d.items():
                np.save(os.path.join(cache, sub, k + ".npy"), a)
        open(done, "w").write("ok")
    except OSError:
        pass
    return st.mesh, st, time.time() - t0


def run_check(g, lm=None, dist=None, world=1):
    """min / max / NaN / Inf / bit checksum per field over the OWNED entities (mpasb200_summarize_field), merged over ranks.
    Every merge is exact and order-independent, so the result must be identical at every N when the N-rank step is
    bit-identical to the single-partition one."""
    from mpas_regent_b200 import _abi
    if lm is not None:
        for ent, ids in ((_abi.CELL, lm.cells), (_abi.EDGE, lm.edges), (_abi.VERTEX, lm.vertices)):
            g.set_global_ids(ent, ids)
    loc = {}
    for n in CHECK_FIELDS:
        ent = _abi.FIELD_ENTITY[n]
        loc[n] = g.summarize_field(n, None if lm is None else lm.n_owned[ent])
    parts = [loc]
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, loc)
    return merge_checks(parts)


def merge_checks(parts):
    """merge per-rank summaries (owned entities, global ids): min / max with the first place, sums, checksum mod 2^64"""
    out, comb, finite = {}, 0, True
    for i, n in enumerate(CHECK_FIELDS):
        ps = [p[n] for p in parts]
        lo = min(ps, key=lambda p: (p["min"], p["min_at"] if p["min_at"][0] >= 0 else [1 << 62, 0]))
        hi = min(ps, key=lambda p: (-p["max"], p["max_at"] if p["max_at"][0] >= 0 else [1 << 62, 0]))
        cs = sum(int(p["checksum"], 16) for p in ps) & ((1 << 64) - 1)
        out[n] = {"min": lo["min"], "min_at": lo["min_at"], "max": hi["max"], "max_at": hi["max_at"],
                  "n_nan": sum(p["n_nan"] for p in ps), "n_inf": sum(p["n_inf"] for p in ps),
                  "count": sum(p["count"] for p in ps), "checksum": f"{cs:016x}"}
        finite = finite and out[n]["n_nan"] == 0 and out[n]["n_inf"] == 0
        comb = (comb * 0x100000001b3 + cs + i) & ((1 << 64) - 1)
    return {"what": "summarize_timestep (rk_timestep.rg:29-359) on the device over owned entities after the timed loop",
            "finite": finite, "combined_checksum": f"{comb:016x}", "fields": out}


def dump_outputs(g, out_dir: str):
    """CHECK_FIELDS as out_dir/<field>.npy (float64, rows = entities in mesh order, all levels): every row when the fields
    fit DUMP_BYTES, else the same seeded sample of rows for every field of one entity kind, in ascending order."""
    from mpas_regent_b200 import _abi
    os.makedirs(out_dir, exist_ok=True)
    for n in CHECK_FIELDS:
        a = g.download_field(n)
        ent, rows = _abi.FIELD_ENTITY[n], a.shape[0]
        k = min(rows, max(1, DUMP_BYTES // (len(CHECK_FIELDS) * a[0].nbytes)))
        if k < rows:
            a = a[np.sort(np.random.default_rng(DUMP_SEED + ent).permutation(rows)[:k])]
        np.save(os.path.join(out_dir, n + ".npy"), np.ascontiguousarray(a))


def host_threads() -> int:
    """host cores this process may use (torchrun exports OMP_NUM_THREADS=1; the oracle takes an explicit count)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_baseline(sample_cells: int, L: int, steps: int, warmup: int, threads: int):
    """The oracle (a port: the Regent reference cannot run here) on a bounded sample of the workload."""
    from mpas_regent_b200 import _abi, dynamics, icosa, init_jw
    from oracle.oracle import Oracle
    mesh = icosa.make_icosahedral_mesh(sample_cells)
    st = init_jw.make_state(mesh, L, _abi.INDEX_CORRECTED, m5=True, diag_on_host=False)
    cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX)
    o = Oracle(dynamics.dims_of(mesh, L), cfg, threads=threads)
    o.upload_mesh(st.static); o.upload_state(st.f, st.vert)
    o.atm_compute_solve_diagnostics(False, -1)
    dt = dt_for(sample_cells)
    for _ in range(warmup):
        o.atm_srk3(dt)
    t0 = time.perf_counter()
    for _ in range(steps):
        o.atm_srk3(dt)
    sec = time.perf_counter() - t0
    o.close()
    return sample_cells * L * steps / sec, sec / steps


def workload_config(n_cells: int, L: int, world: int, corrected: bool = False) -> dict:
    """the `config` object: identical for the b200 arm and the reference arm at the same N (run-specific facts live in `run_info`)"""
    dt = dt_for(n_cells)
    return {"workload": f"x1.{n_cells} synthetic icosahedral Voronoi mesh, {L} levels, JW-style analytic state, dt={dt:.2f}s, "
                        f"one atm_srk3 per step (canonical stage-index sequence: stage 0 takes the rk_step==0 branches)"
                        + ("; CORRECTED physics mode (u update, back-substitution, recover wired in)" if corrected else ""),
            "parallelism": "single partition" if world == 1 else f"{world}-way cell partition (SFC chunks), 2-ring halo exchange over NVLink",
            "l2": "working set (tens of GB) >> 126 MB L2; no flush needed"}


def mem_available_gb() -> float:
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) / 1048576.0
    except OSError:
        pass
    return 0.0


def cpu_sample_cells(requested: int, workload_cells: int) -> int:
    """bounded sample of the workload for the CPU legs: the largest mesh of the family that the host holds comfortably and that
    keeps a --steps 20 --warmup 5 run within a few minutes (x1.163842 x 55 ~ 3 s per step on 16 cores, BASELINE.md section 4)"""
    if requested > 0:
        return requested
    for n in (163842, 40962, 10242):
        if n <= workload_cells and mem_available_gb() >= 45.0 * n / 163842 + 4:
            return n
    return 2562


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    n_s = cpu_sample_cells(args.cpu_sample_cells, args.mesh)
    val, sec = cpu_baseline(n_s, args.levels, max(1, args.steps), max(0, args.warmup), threads)
    sample = (f"oracle port (literal C++ restatement of the reference's task bodies, OpenMP over the outer entity loop, {threads} threads) on a "
              f"bounded sample of the workload: x1.{n_s} mesh of the same family x {args.levels} levels "
              f"({n_s / args.mesh:.3f} of the workload's cells; the rate per cell-level is what is reported"
              + (", i.e. extrapolated to the workload" if n_s != args.mesh else "") + f"), {args.steps} RK3 steps after {args.warmup} warm-up")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.mesh, args.levels, max(1, args.gpus), args.physics == "corrected"),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    _emit(line)


_REAL_STDOUT = None


def _quiet_stdout():
    """Route everything that libraries print on stdout (e.g. "NCCL version ...") to stderr, so that stdout carries
    exactly ONE line: the JSON result."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def _emit(line: dict):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (json.dumps(line) + "\n").encode())


def main():
    _quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--mesh", type=int, default=int(os.environ.get("MPAS_BENCH_CELLS", "655362")))
    ap.add_argument("--levels", type=int, default=55)
    ap.add_argument("--cpu-sample-cells", type=int, default=0, help="0 = the largest of x1.163842 / 40962 / 10242 the host holds")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--graph", type=int, default=0)
    ap.add_argument("--gather-stage", type=int, default=-1, help="MpasConfig.gather_stage bit mask (ablation: 0 = the plain gather kernels)")
    ap.add_argument("--edge-tiles", type=int, default=None, help="MpasConfig.edge_tiles (0 = plain k_dt_edge; 8 / 16 = tile-staged form)")
    ap.add_argument("--timeline", default="", help="write the launch timeline of ONE step (both streams, rank 0) to this file and exit")
    ap.add_argument("--kernel-forms", type=int, default=None, help="MpasConfig.kernel_forms bit mask (1 = k_dt_cellC as two launches)")
    ap.add_argument("--acoustic", type=int, default=3, help="MpasConfig.acoustic_tma (3 = exact column-per-lane pipeline, 2 = affine sweep)")
    ap.add_argument("--physics", choices=("literal", "corrected"), default="literal",
                    help="literal = the reference as it executes (headline); corrected = acoustic u update + back-substitution + "
                         "recover wired in (SURVEY.md 8f rank 1, MPASB200_PHYSICS_CORRECTED)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the fields the last timed step left (a fixed, seeded sample of rows) to DIR/<field>.npy; one GPU only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    from mpas_regent_b200 import _abi, dynamics, traffic

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs samples the fields of a single partition: run it on one GPU")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    L, nC = args.levels, args.mesh
    dt = dt_for(nC)
    corrected = args.physics == "corrected"
    cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, device=local_rank, use_graph=args.graph,
                              physics_mode=_abi.PHYSICS_CORRECTED if corrected else _abi.PHYSICS_LITERAL, gather_stage=args.gather_stage, acoustic_tma=args.acoustic,
                              **({} if args.edge_tiles is None else {"edge_tiles": args.edge_tiles}),
                              **({} if args.kernel_forms is None else {"kernel_forms": args.kernel_forms}))
    stream = torch.cuda.Stream()

    if world == 1:
        mesh, st, t_init = build_inputs(nC, L)
        g = dynamics.Dynamics(dynamics.dims_of(mesh, L), cfg)
        g.set_stream(stream.cuda_stream)
        g.upload_mesh(st.static)
        g.upload_state(st.f, st.vert)
        # pinned host images of the prognostic state for the end-to-end leg
        host = {}
        if not args.no_e2e:
            for n in E2E_FIELDS:
                t = torch.from_numpy(st.f[n]).pin_memory()
                host[n] = t
        del st
        g.atm_compute_solve_diagnostics(False, -1)       # atm_core_init, atm_core.rg:31
        step = lambda: g.atm_srk3(dt)
        n_owned_total = nC
        parallelism = "single partition"
    else:
        from mpas_regent_b200 import parallel
        parallel.DistributedDynamics.KEEP_HOST_FIELDS = () if args.no_e2e else E2E_FIELDS
        run = parallel.DistributedDynamics.for_bench(nC, L, cfg, stream, rank, world)
        g = run.dyn
        host = {n: torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for n, a in run.host_fields.items()}
        step = lambda: run.step(dt)
        n_owned_total = nC
        parallelism = (f"{world}-way cell partition (SFC chunks), 2-ring halo exchange over NCCL send/recv"
                       + (", exchanges overlapped with interior compute on a communication stream" if getattr(run, "overlap", False) else ""))
        t_init = run.t_init

    def barrier():
        if world > 1:
            dist.barrier()

    with torch.cuda.stream(stream):
        for _ in range(max(args.warmup, 3)):
            step()
        g.sync()
        launches0 = g.launch_count
        sampler = ClockSampler(local_rank) if rank == 0 else None
        torch.cuda.synchronize(); barrier()
        if args.timeline:
            # one step with an event pair around every launch on both of the handle's streams: where the exchanges sit in time
            g.enable_kernel_timing(2)
            step()
            if world > 1:
                run.flush()
            g.sync(); torch.cuda.synchronize()
            tl = g.timeline()
            g.enable_kernel_timing(False)
            if rank == 0:
                with open(args.timeline, "w") as fh:
                    json.dump({"n_gpus": world, "mesh": nC, "levels": L, "rank": 0, "entries": tl}, fh)
            barrier()
            if world > 1:
                dist.destroy_process_group()
            return
        # ---- the timed region: K steps, nothing else on the stream (per-kernel events are a separate pass below) ----
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            step()
        if world > 1:
            run.flush()          # the last halo exchange (travelling on the communication stream) belongs to the timed region
        e1.record(stream)
        torch.cuda.synchronize(); barrier()
        ms = e0.elapsed_time(e1)
        launches = g.launch_count - launches0
        if args.dump_outputs:
            dump_outputs(g, args.dump_outputs)      # the state after the last timed step, before the per-kernel pass advances it
        # ---- the same K steps again with a CUDA-event pair around every launch (on the launching stream): per-kernel times.
        # Kept out of the headline region because two event records per launch inflate a step of ~100 short kernels;
        # graph replay is off here (events cannot bracket the nodes of a replayed graph).
        k_steps = min(args.steps, 5)
        if args.graph:
            g.set_use_graph(False)
        g.reset_kernel_timing(); g.enable_kernel_timing(True)
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e2.record(stream)
        for _ in range(k_steps):
            step()
        if world > 1:
            run.flush()
        e3.record(stream)
        torch.cuda.synchronize(); barrier()
        ms_k = e2.elapsed_time(e3)
        clocks = sampler.stop() if sampler else {}
        ktimes = g.kernel_times()
        g.enable_kernel_timing(False)
        if args.graph:
            g.set_use_graph(True)
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        tl = torch.tensor([launches], device="cuda", dtype=torch.int64)
        dist.all_reduce(tl, op=dist.ReduceOp.SUM)
        launches = int(tl.item())
    value = n_owned_total * L * args.steps / (ms * 1e-3)
    # ---- the step's own sanity scan, before anything else touches the state ----
    with torch.cuda.stream(stream):
        check = run_check(g, run.lm if world > 1 else None, dist if world > 1 else None, world)
    check["steps_from_initial_state"] = max(args.warmup, 3) + args.steps + k_steps

    # ---- roofline of the dominant kernel (rank 0's kernels; cells of this rank) ----
    peak, peak_src = peaks()
    n_local = g.dims.nCells
    roof = None
    if ktimes:
        name, (kms, kn) = max(ktimes.items(), key=lambda kv: kv[1][0])
        key = traffic.lookup(name)
        if key is not None and kn > 0:
            u = traffic.units(key, scratch=False)
            bytes_per_launch = u * 8.0 * n_local * L
            achieved = bytes_per_launch / (kms / kn * 1e-3) / 1e9
            # dram__bytes_read.sum + dram__bytes_write.sum per launch: NOT measured in this run (ncu cannot run under a bench) --
            # taken from the committed ncu capture and stamped with where it came from, so a stale entry is visible
            traffic_bytes, traffic_src = None, None
            tj = os.path.join(ROOT, "profiles", "ncu_traffic.json")
            if world == 1 and nC == 655362 and L == 55 and os.path.exists(tj):
                td = json.load(open(tj))
                traffic_bytes = td["bytes_per_launch"].get(name)
                traffic_src = {k: td.get(k) for k in ("source", "kernel_source_commit", "captured")}
            roof = {"bound": "hbm", "kernel": name, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic_bytes, "traffic_source": traffic_src, "peak_source": peak_src, "algorithmic_bytes_per_launch": bytes_per_launch,
                    "avg_launch_ms": kms / kn, "launches_timed": kn, "share_of_step": kms / ms_k,
                    "timed_over": f"{k_steps} steps with an event pair per launch ({ms_k / k_steps:.3f} ms/step; the headline "
                                  f"region runs without them)"}
    step_units = traffic.step_units(True, scratch=False, corrected_physics=True) if corrected else traffic.SURVEY_STEP_UNITS_CANONICAL
    step_bytes = step_units * 8.0 * nC * L
    step_gbs = step_bytes / (ms / args.steps * 1e-3) / 1e9

    # ---- end to end through the C ABI with host buffers ----
    # Every step uploads its inputs from pinned host memory and reads its results back.  `e2e` uses the pipelined
    # transfer entries (H2D of the next batch and D2H of the previous one overlap the step on separate copy streams);
    # `e2e.sync` is the same loop through the blocking upload_field / download_field calls.
    e2e = None
    if world == 1 and not args.no_e2e:
        k_e = max(3, min(args.steps, 5))
        h2d = sum(t.numel() * 8 for t in host.values())
        outs = {n: torch.empty_like(t).pin_memory() for n, t in host.items()}
        with torch.cuda.stream(stream):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(2):
                for n, t in host.items():
                    g.upload_field(n, t.numpy())
                g.atm_srk3(dt)
                for n, t in outs.items():
                    g.download_field(n, t.numpy())
            torch.cuda.synchronize()
            sec_sync = (time.perf_counter() - t0) / 2
            ref_out = {n: t.clone() for n, t in outs.items()}
            # pipelined: one untimed batch fills the pipeline buffers, then k_e timed batches
            for n, t in host.items():
                g.upload_field_async(n, t.numpy())
            g.atm_srk3(dt)
            for n, t in outs.items():
                g.download_field_async(n, t.numpy())
            g.transfer_wait()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(k_e):
                for n, t in host.items():
                    g.upload_field_async(n, t.numpy())
                g.atm_srk3(dt)
                for n, t in outs.items():
                    g.download_field_async(n, t.numpy())
            g.transfer_wait()
            torch.cuda.synchronize()
            sec = time.perf_counter() - t0
        same = all(torch.equal(ref_out[n], outs[n]) for n in outs)      # every batch has the same inputs: results must be identical
        e2e = {"value": nC * L * k_e / sec, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": h2d,
               "steps": k_e, "fields": list(E2E_FIELDS), "ms_per_step": sec / k_e * 1e3, "pipelined": True,
               "results_equal_blocking_path": bool(same),
               "sync": {"value": nC * L / sec_sync, "ms_per_step": sec_sync * 1e3}}

    if world > 1 and not args.no_e2e:
        # every rank moves ITS shard (owned + ghost columns) of the prognostic state host -> device before and device -> host after
        # every step, through the pipelined C-ABI transfers; wall clock between barriers, max over ranks
        k_e = max(3, min(args.steps, 5))
        outs = {n: torch.empty_like(t).pin_memory() for n, t in host.items()}
        with torch.cuda.stream(stream):
            for n, t in host.items():
                g.upload_field_async(n, t.numpy())
            step()
            for n, t in outs.items():
                g.download_field_async(n, t.numpy())
            g.transfer_wait(); run.flush(); torch.cuda.synchronize(); barrier()
            t0 = time.perf_counter()
            for _ in range(k_e):
                for n, t in host.items():
                    g.upload_field_async(n, t.numpy())
                step()
                for n, t in outs.items():
                    g.download_field_async(n, t.numpy())
            g.transfer_wait(); run.flush(); torch.cuda.synchronize(); barrier()
            sec = time.perf_counter() - t0
        tt = torch.tensor([sec, float(sum(t.numel() * 8 for t in host.values()))], device="cuda", dtype=torch.float64)
        tmax = tt.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(tt, op=dist.ReduceOp.SUM)
        sec, h2d = float(tmax[0].item()), float(tt[1].item())
        e2e = {"value": nC * L * k_e / sec, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": h2d, "steps": k_e,
               "fields": list(E2E_FIELDS), "ms_per_step": sec / k_e * 1e3, "pipelined": True,
               "note": "bytes are summed over ranks and include every rank's ghost columns; wall clock between barriers, max over ranks"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        thr = host_threads()
        n_s = cpu_sample_cells(args.cpu_sample_cells, nC)
        n_1 = min(n_s, 40962)
        v1, s1 = cpu_baseline(n_1, L, 1, 0, 1)
        vN, sN = cpu_baseline(n_s, L, 3, 1, thr)
        cpu = {"value": vN, "unit": UNIT, "cores": thr, "kind": "port",
               "sample": f"oracle port (the Regent reference cannot be built here) on a bounded sample of the workload: x1.{n_s} x {L} levels "
                         f"({n_s / nC:.3f} of the cells, rate per cell-level), 3 RK3 steps after 1 warm-up with {thr} OpenMP threads "
                         f"({sN:.2f} s/step); 1 thread (how the reference runs: one serial leaf task at a time, main.rg:55) on x1.{n_1}: "
                         f"{v1:.4g} {UNIT} ({s1:.2f} s/step)",
               "single_thread_value": v1}

    if rank == 0:
        top = sorted(ktimes.items(), key=lambda kv: -kv[1][0])
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": workload_config(nC, L, world, corrected),
            "run_info": {"parallelism_detail": parallelism, "host_init_s": round(t_init, 1), "device_bytes": g.device_bytes,
                         "cuda_graph": bool(args.graph), "acoustic_tma": args.acoustic, "edge_tiles": int(cfg.edge_tiles), "kernel_forms": int(cfg.kernel_forms), "ms_per_step_with_kernel_events": ms_k / k_steps},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": roof,
            "step_hbm": {"algorithmic_bytes_per_step": step_bytes, "achieved_gbs_per_gpu": step_gbs / world,
                         "frac_of_peak": step_gbs / world / peak},
            "kernels_ms_per_step": {k: round(v[0] / k_steps, 4) for k, v in top},
            "kernels_launches_per_step": {k: round(v[1] / k_steps, 2) for k, v in top},
            "e2e": e2e, "cpu_baseline": cpu, "check": check,
        }
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
