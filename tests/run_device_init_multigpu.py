"""Launched by torchrun on N >= 2 GPUs (tests/test_device_init_gpu.py::test_nccl_ranks_from_device_init_equal_single_gpu):
every rank builds its rows of the initial state on its own GPU from its static shard (init_jw.init_on_device), repairs its
ghosts with parallel.INIT_EXCHANGE through NcclExchanger and runs the library's distributed step; OWNED entities must be
bit-identical to a single-GPU run from the device-built global state."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mpas_regent_b200 import _abi, dynamics, icosa, init_jw, parallel  # noqa: E402
from tests.test_parallel import _assert_owned_equal  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    L, dt, steps = 12, 400.0, 3
    mesh = icosa.make_icosahedral_mesh(2562)
    st, draws = init_jw.make_static(mesh, L, _abi.INDEX_CORRECTED)
    cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, device=local)
    stream = torch.cuda.Stream()
    sh = parallel.make_static_shards(st, world)[rank]
    lm = sh["lm"]
    d = dynamics.Dynamics(_abi.make_dims(len(lm.cells), len(lm.edges), len(lm.vertices), L), cfg)
    d.set_stream(stream.cuda_stream)
    d.upload_mesh(sh["static"])
    with torch.cuda.stream(stream):
        init_jw.init_on_device(d, sh["static"], init_jw.jw_inputs(mesh, st, draws, lm), st.vert)
        parallel.NcclExchanger(d, lm, stream).exchange(parallel.INIT_EXCHANGE)
    run = parallel.NativeDistributedDynamics(d, lm, rank, world)
    run.init_diagnostics()
    for _ in range(steps):
        run.step(dt)
    run.flush()
    torch.cuda.synchronize()
    single = dynamics.Dynamics(dynamics.dims_of(mesh, L), cfg)
    single.upload_mesh(st.static)
    init_jw.init_on_device(single, st.static, init_jw.jw_inputs(mesh, st, draws), st.vert)
    single.atm_compute_solve_diagnostics(False, -1)
    for _ in range(steps):
        single.atm_srk3(dt)
    _assert_owned_equal(single, d, lm)
    dist.barrier()
    if rank == 0:
        print(f"MULTIGPU_INIT_OK world={world} owned_cells={lm.n_owned[0]} ghosts={len(lm.cells) - lm.n_owned[0]}")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
