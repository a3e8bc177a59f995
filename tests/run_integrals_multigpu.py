"""Launched by torchrun on N >= 2 GPUs (tests/test_integrals_gpu.py::test_nccl_ranks_integrals_equal_single_gpu): every
rank builds its shard of the initial state on its own GPU and runs the library's distributed step; the integrals of
parallel.column_integrals over its owned cells, merged over torch.distributed (parallel.merge_integrals), must have the
limbs and bits of the same integrals on one GPU, on the initial state and after the steps."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mpas_regent_b200 import _abi, dynamics, icosa, init_jw, parallel  # noqa: E402


def _same(a, b, what):
    for k in a:
        assert np.array_equal(a[k]["limbs"], b[k]["limbs"]) and a[k]["bits"] == b[k]["bits"], (what, k, a[k]["value"], b[k]["value"])


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
    jw = init_jw.jw_inputs(mesh, st, draws, lm)
    area = d.register_weights(_abi.CELL, jw["areaCell"])
    with torch.cuda.stream(stream):
        init_jw.init_on_device(d, sh["static"], jw, st.vert)
        parallel.NcclExchanger(d, lm, stream).exchange(parallel.INIT_EXCHANGE)
    got = [parallel.column_integrals(d, area, lm.n_owned[0], dist, fields=("rho_zz", "ke", "theta_m"))]
    run = parallel.NativeDistributedDynamics(d, lm, rank, world)
    run.init_diagnostics()
    for _ in range(steps):
        run.step(dt)
    run.flush()
    torch.cuda.synchronize()
    got.append(parallel.column_integrals(d, area, lm.n_owned[0], dist, fields=("rho_zz", "ke", "theta_m")))

    single = dynamics.Dynamics(dynamics.dims_of(mesh, L), cfg)
    single.upload_mesh(st.static)
    jw1 = init_jw.jw_inputs(mesh, st, draws)
    area1 = single.register_weights(_abi.CELL, jw1["areaCell"])
    init_jw.init_on_device(single, st.static, jw1, st.vert)
    want = [parallel.column_integrals(single, area1, fields=("rho_zz", "ke", "theta_m"))]
    single.atm_compute_solve_diagnostics(False, -1)
    for _ in range(steps):
        single.atm_srk3(dt)
    want.append(parallel.column_integrals(single, area1, fields=("rho_zz", "ke", "theta_m")))
    _same(got[0], want[0], "initial state")
    _same(got[1], want[1], f"after {steps} steps")
    dist.barrier()
    if rank == 0:
        print(f"MULTIGPU_INTEGRALS_OK world={world} mass={got[1]['rho_zz']['value']!r} bits={got[1]['rho_zz']['bits']}")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
