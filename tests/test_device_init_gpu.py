"""The initial state built on the device, one handle per partition (init_jw.init_on_device + parallel.INIT_EXCHANGE): against
the host generator on one handle, then N emulated ranks on one GPU against the single handle, bitwise, before and after
the RK3 steps; the N = 1 runner; the N-GPU run over NCCL where the box has the GPUs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from mpas_regent_b200 import _abi

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _single(mesh, L, cfg):
    from mpas_regent_b200 import dynamics, init_jw
    st, draws = init_jw.make_static(mesh, L, _abi.INDEX_CORRECTED)
    g = dynamics.Dynamics(dynamics.dims_of(mesh, L), cfg)
    g.upload_mesh(st.static)
    init_jw.init_on_device(g, st.static, init_jw.jw_inputs(mesh, st, draws), st.vert)
    return st, draws, g


@pytest.mark.parametrize("which,levels", [("x1.2562", 26), ("icosa642", 55)], ids=["x1.2562_L26", "icosa642_L55"])
def test_device_init_matches_make_state(grid2562, grid642, which, levels):
    """every field make_state(m5=True) hands the step, and v from atm_compute_solve_diagnostics(-1), within 1e-12 of the
    field's largest value; rw and w against the size of the edge terms they sum (they cancel to ~1e-4 of it, as in
    test_init_atm_case_jw_on_the_device).  All finite."""
    from mpas_regent_b200 import init_jw
    mesh = grid2562 if which == "x1.2562" else grid642
    ref = init_jw.make_state(mesh, levels, _abi.INDEX_CORRECTED, m5=True)
    _, _, g = _single(mesh, levels, _abi.default_config())
    g.atm_compute_solve_diagnostics(False, -1)
    f = ref.f
    term = np.abs(f["zz"]).max() * np.abs(f["ru"]).max() * 2.0
    bad, worst = [], {}
    for n, r in list(f.items()) + [(k, ref.vert[k]) for k in ref.vert]:
        a = g.download_field(n)
        scale = np.abs(r).max()
        if n == "rw":
            scale = max(scale, term * np.abs(f["zb_cell"]).max())
        elif n == "w":
            scale = term * np.abs(ref.extras["zb"]).max() / f["rho_zz"][:, :levels].min()
        err = np.abs(a - r).max()
        worst[n] = err / scale if scale > 0 else err
        if not np.isfinite(a).all() or not (err <= 1e-12 * scale if scale > 0 else err == 0.0):
            bad.append((n, err, scale, bool(np.isfinite(a).all())))
    print("worst relative deviations:", {k: f"{x:.1e}" for k, x in worst.items()})
    assert not bad, bad
    g.close()


class _PackUnpack:
    """owner -> holder through k_pack / k_unpack and a device buffer per (holder, owner) pair: NcclExchanger minus the wire"""

    def __init__(self, backs, shards):
        from mpas_regent_b200 import parallel
        self.backs, self.shards, self.lists = backs, shards, {}
        for h, sh in enumerate(shards):
            for ent in ("cell", "edge", "vertex"):
                for peer, idx in sh["lm"].send[ent].items():
                    self.lists[("s", h, ent, peer)] = backs[h].register_list(parallel.ENT[ent], idx)
                for peer, idx in sh["lm"].recv[ent].items():
                    self.lists[("r", h, ent, peer)] = backs[h].register_list(parallel.ENT[ent], idx)

    def exchange(self, spec):
        import torch
        from mpas_regent_b200 import parallel
        backs = self.backs
        for b in backs:
            b.sync()
        L1 = backs[0].dims.nVertLevels + 1
        for ent, all_names in spec.items():
            for names in parallel.pack_groups(all_names):
                width = sum(_abi.FIELD_SLOTS[n] for n in names) * L1
                for h, sh in enumerate(self.shards):
                    for o, ridx in sh["lm"].recv[ent].items():
                        buf = torch.empty(len(ridx) * width, dtype=torch.float64, device="cuda")
                        backs[o].pack(self.lists[("s", o, ent, h)], names, buf.data_ptr()); backs[o].sync()
                        backs[h].unpack(self.lists[("r", h, ent, o)], names, buf.data_ptr()); backs[h].sync()


def _ranks(mesh, L, cfg, st, draws, colours, world):
    """one handle per rank: its static shard uploaded, its rows built on the device (before INIT_EXCHANGE)"""
    from mpas_regent_b200 import dynamics, init_jw, parallel
    shards = parallel.make_static_shards(st, world, colours)
    backs = []
    for sh in shards:
        lm = sh["lm"]
        b = dynamics.Dynamics(_abi.make_dims(len(lm.cells), len(lm.edges), len(lm.vertices), L), cfg)
        b.upload_mesh(sh["static"])
        init_jw.init_on_device(b, sh["static"], init_jw.jw_inputs(mesh, st, draws, lm), st.vert)
        backs.append(b)
    return shards, backs


def _colouring(mesh, kind):
    """(colours or None for the SFC default, world)"""
    from mpas_regent_b200 import partition
    rng = np.random.default_rng(1)
    if kind == "sfc":
        return None, 4
    if kind == "random":
        return rng.integers(0, 3, mesh.nCells).astype(np.int32), 3
    return rng.integers(0, 3, 24).astype(np.int32)[partition.sfc_colouring(mesh, 24)], 3


def _rows_equal(single, b, lm, name):
    rows = {_abi.CELL: lm.cells, _abi.EDGE: lm.edges, _abi.VERTEX: lm.vertices}
    ent = _abi.FIELD_ENTITY[name]
    ref = single.download_field(name)
    return np.array_equal(b.download_field(name), ref if ent == _abi.VERTICAL else ref[rows[ent]], equal_nan=True)


@pytest.mark.parametrize("exchanger", ["pack_unpack", "in_process"])
@pytest.mark.parametrize("colouring", ["sfc", "random", "random_blocks"])
def test_emulated_ranks_after_init_exchange_equal_single_handle(grid642, colouring, exchanger):
    """4 SFC ranks, the 3-rank `random` colouring of test_irregular_colourings_still_match_single_partition, and 3 ranks
    that each own scattered blocks (24 SFC chunks dealt out at random), as handles on one GPU: after INIT_EXCHANGE every
    field of every rank, ghost rows included, is bit-identical to the single-handle device init at the rank's rows.  Under
    SFC and scattered blocks ranks do not hold the whole mesh and some ghost row is wrong before the exchange; the
    cell-by-cell random colouring's two rings reach every cell, so there every rank is right before it too."""
    from mpas_regent_b200 import parallel
    L = 10
    cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX)
    st, draws, single = _single(grid642, L, cfg)
    col, world = _colouring(grid642, colouring)
    shards, backs = _ranks(grid642, L, cfg, st, draws, col, world)
    fields = [n for n, _, _ in _abi.FIELDS]
    wrong_before = [[n for n in fields if not _rows_equal(single, b, sh["lm"], n)] for b, sh in zip(backs, shards)]
    whole = [len(sh["lm"].cells) == grid642.nCells for sh in shards]
    if colouring != "random":
        assert not any(whole) and all(wrong_before), wrong_before
        assert all(set(w) <= set(parallel.INIT_EXCHANGE["cell"]) | set(parallel.INIT_EXCHANGE["edge"]) for w in wrong_before)
    else:
        assert all(whole) and not any(wrong_before), wrong_before
    ex = _PackUnpack(backs, shards) if exchanger == "pack_unpack" else parallel.InProcessExchanger(backs, [s["lm"] for s in shards])
    ex.exchange(parallel.INIT_EXCHANGE)
    for b, sh in zip(backs, shards):
        bad = [n for n in fields if not _rows_equal(single, b, sh["lm"], n)]
        assert not bad, (sh["lm"].rank, bad)
        b.close()
    single.close()


@pytest.mark.parametrize("physics", [_abi.PHYSICS_LITERAL, _abi.PHYSICS_CORRECTED], ids=["literal", "corrected_physics"])
def test_emulated_ranks_from_device_init_step_like_single_partition(grid642, physics):
    """then atm_compute_solve_diagnostics(-1) and 3 RK3 steps with the exchange schedule of parallel.exchanges_for: owned
    entities are bit-identical to the single-partition run from the device-initialized global state"""
    from mpas_regent_b200 import parallel
    from tests.test_parallel import DT, _assert_owned_equal, _task_schedule
    L = 6
    cfg = _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, physics_mode=physics)
    st, draws, single = _single(grid642, L, cfg)
    shards, backs = _ranks(grid642, L, cfg, st, draws, None, 4)
    ex = _PackUnpack(backs, shards)
    ex.exchange(parallel.INIT_EXCHANGE)
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
    assert np.isfinite(single.download_field("u")).any()
    for b, sh in zip(backs, shards):
        _assert_owned_equal(single, b, sh["lm"])
        b.close()
    single.close()


def test_runner_on_one_gpu_is_reproducible():
    """run_device_init.py at N = 1 twice: the same finite checksum"""
    lines = []
    for _ in range(2):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "run_device_init.py"), "--mesh", "10242", "--levels", "26",
                              "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
        lines.append(json.loads(out.stdout.strip().splitlines()[-1]))
    assert lines[0]["finite"] and lines[0]["combined_checksum"] == lines[1]["combined_checksum"], lines


def test_nccl_ranks_from_device_init_equal_single_gpu():
    """rank-local device init, INIT_EXCHANGE through NcclExchanger, then the library's distributed step (>= 2 GPUs)"""
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    n = 2 if n < 4 else 4
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr",
                          "127.0.0.1", "--master-port", "29545", os.path.join(ROOT, "tests", "run_device_init_multigpu.py")],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0 and "MULTIGPU_INIT_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-3000:]
