"""Launched by torchrun on N >= 2 GPUs (tests/test_restart_gpu.py::test_nccl_restart_resumes_at_n_and_at_one): every rank
builds its shard of the initial state on its own GPU and runs the library's distributed step (NativeDistributedDynamics).
A restart saved at step 3, resumed at N and on one GPU and run to step 6, must give the combined checksum of an
uninterrupted N-rank run."""
import os
import sys
import tempfile

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from mpas_regent_b200 import _abi, dynamics, icosa, init_jw, parallel, restart  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    L, dt = 12, 400.0
    mesh = icosa.make_icosahedral_mesh(2562)
    st, draws = init_jw.make_static(mesh, L, _abi.INDEX_CORRECTED)
    cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, device=local)
    stream = torch.cuda.Stream()
    sh = parallel.make_static_shards(st, world)[rank]
    lm = sh["lm"]
    box = [tempfile.mkdtemp(prefix="mpas_b200_restart_") if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    path = os.path.join(box[0], "r3")

    def handle():
        d = dynamics.Dynamics(_abi.make_dims(len(lm.cells), len(lm.edges), len(lm.vertices), L), cfg)
        d.set_stream(stream.cuda_stream)
        d.upload_mesh(sh["static"])
        return d

    # uninterrupted, saving at step 3 on the way
    d = handle()
    with torch.cuda.stream(stream):
        init_jw.init_on_device(d, sh["static"], init_jw.jw_inputs(mesh, st, draws, lm), st.vert)
        parallel.NcclExchanger(d, lm, stream).exchange(parallel.INIT_EXCHANGE)
        run = parallel.NativeDistributedDynamics(d, lm, rank, world)
        run.init_diagnostics()
        for k in range(6):
            run.step(dt)
            if k == 2:
                run.flush()
                torch.cuda.synchronize()
                restart.save(path, d, lm, 3, mesh, dist)
        run.flush()
        torch.cuda.synchronize()
    want = bench.run_check(d, lm, dist, world)["combined_checksum"]
    d.close()

    # resumed at N
    d = handle()
    with torch.cuda.stream(stream):
        assert restart.load(path, d, lm, mesh, dist) == 3
        run = parallel.NativeDistributedDynamics(d, lm, rank, world)
        for _ in range(3):
            run.step(dt)
        run.flush()
        torch.cuda.synchronize()
    got_n = bench.run_check(d, lm, dist, world)["combined_checksum"]
    d.close()

    # resumed on one GPU (rank 0)
    got_1 = None
    if rank == 0:
        g = dynamics.Dynamics(dynamics.dims_of(mesh, L), cfg)
        g.upload_mesh(st.static)
        assert restart.load(path, g, None, mesh) == 3
        for _ in range(3):
            g.atm_srk3(dt)
        g.sync()
        got_1 = bench.run_check(g)["combined_checksum"]
        g.close()
    dist.barrier()
    if rank == 0:
        assert got_n == want and got_1 == want, (want, got_n, got_1)
        import shutil
        shutil.rmtree(box[0], ignore_errors=True)
        print(f"MULTIGPU_RESTART_OK world={world} checksum={want}")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
