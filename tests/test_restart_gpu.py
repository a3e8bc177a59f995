"""Restart files with the CUDA library: the same bytes at every rank count, resume across rank counts, the C ABI of the
restart set.  Ranks are emulated on one GPU (InProcessExchanger); tests/run_restart_multigpu.py runs them over NCCL."""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

from mpas_regent_b200 import _abi, dynamics, icosa, init_jw, parallel, partition, restart
from mpas_regent_b200._abi import CELL, EDGE, VERTEX, VERTICAL

pytestmark = pytest.mark.gpu

L = 6
DT = 600.0
NAMES = [n for n, _, _ in _abi.FIELDS]


@pytest.fixture(scope="module")
def problem():
    mesh = icosa.make_icosahedral_mesh(642)
    return mesh, init_jw.make_state(mesh, L, _abi.INDEX_CORRECTED)


def _cfg(**over):
    return _abi.default_config(rkarg_policy=_abi.RKARG_STAGE_INDEX, device=0, **over)


def _with_scalars(mesh, st):
    return init_jw.HostState(nVertLevels=st.nVertLevels, policy=st.policy, mesh=st.mesh, static=st.static, vert=st.vert,
                             f=dict(st.f, scalars=1e-3 * (1.0 + np.random.default_rng(2).random((mesh.nCells, L + 1, 8)))))


def _shards(st, world, sfc_colouring=True):
    if world == 1:
        return parallel.make_shards(st, 1)
    col = partition.sfc_colouring(st.mesh, world) if sfc_colouring else np.random.default_rng(5).integers(0, world, st.mesh.nCells).astype(np.int32)
    return parallel.make_shards(st, world, colours=col)


def _handles(shards, cfg, with_state=True):
    out = []
    for sh in shards:
        lm = sh["lm"]
        g = dynamics.Dynamics(_abi.make_dims(len(lm.cells), len(lm.edges), len(lm.vertices), L), cfg)
        g.upload_mesh(sh["static"])
        if with_state:
            g.upload_state(sh["f"], sh["vert"])
        out.append(g)
    return out


def _steps(gs, lms, steps, init):
    """``steps`` RK3 steps: atm_srk3 on one handle, the task sequence with its exchanges on emulated ranks"""
    if len(gs) == 1:
        if init:
            gs[0].atm_compute_solve_diagnostics(False, -1)
        for _ in range(steps):
            gs[0].atm_srk3(DT)
        gs[0].sync()
        return
    ex = parallel.InProcessExchanger(gs, lms)
    exchanges = parallel.exchanges_for(gs[0].cfg)
    if init:
        for g in gs:
            g.atm_compute_solve_diagnostics(False, -1)
        ex.exchange(exchanges["compute_solve_diagnostics"])
    seq = []

    class Rec(dynamics.TaskAPI):
        def __init__(self):
            self.cfg, self.dims = gs[0].cfg, None

        def _call(self, name, *args):
            seq.append((name, args))

    Rec().atm_srk3_by_tasks(DT)
    for _ in range(steps):
        for name, args in seq:
            for g in gs:
                g._call(name, *args)
            spec = exchanges.get(parallel.exchange_key(name, args))
            if spec:
                ex.exchange(spec)
    for g in gs:
        g.sync()


def _digests(path):
    return {f: hashlib.sha256(open(os.path.join(path, f), "rb").read()).hexdigest()
            for f in sorted(os.listdir(path)) if f.endswith(".npy")}


def _assert_owned_equal(single, gs, lms):
    for g, lm in zip(gs, lms):
        rows = {CELL: lm.cells, EDGE: lm.edges, VERTEX: lm.vertices} if lm is not None else None
        for name, ent, _ in _abi.FIELDS:
            a, ref = g.download_field(name), single.download_field(name)
            if ent == VERTICAL or lm is None:
                assert np.array_equal(a, ref, equal_nan=True), name
            else:
                n = lm.n_owned[ent]
                assert np.array_equal(a[:n], ref[rows[ent][:n]], equal_nan=True), (name, lm.rank)


@pytest.mark.parametrize("sfc", [1, 0], ids=["sfc_renumber", "no_renumber"])
def test_same_bytes_one_handle_and_emulated_ranks(tmp_path, problem, sfc):
    mesh, st = problem
    cfg = _cfg(sfc_renumber=sfc)
    ref = None
    for world in (1, 3, 4):
        shards = _shards(st, world)
        gs = _handles(shards, cfg)
        lms = [None] if world == 1 else [s["lm"] for s in shards]
        _steps(gs, lms, 2, True)
        p = str(tmp_path / f"n{world}")
        restart.save(p, gs, lms, 2, mesh)
        d = _digests(p)
        ref = ref or d
        assert d == ref, world
        for g in gs:
            g.close()


CASES = [("literal", {}, 1, 3, 0), ("literal", {}, 3, 1, 1), ("corrected", dict(physics_mode=_abi.PHYSICS_CORRECTED), 2, 4, 0),
         ("corrected", dict(physics_mode=_abi.PHYSICS_CORRECTED), 4, 2, 1),
         ("scalars", dict(physics_mode=_abi.PHYSICS_CORRECTED, config_scalar_advection=1), 3, 1, 0),
         ("scalars", dict(physics_mode=_abi.PHYSICS_CORRECTED, config_scalar_advection=1), 1, 3, 1)]


@pytest.mark.parametrize("what,over,n_save,m_load,graph", CASES, ids=[f"{c[0]}-{c[2]}to{c[3]}-graph{c[4]}" for c in CASES])
def test_resume_across_rank_counts(tmp_path, problem, what, over, n_save, m_load, graph):
    """a fresh handle set holds only what the file gives it; K1 + K2 steps must equal the uninterrupted single handle"""
    import bench
    mesh, st = problem
    if over.get("config_scalar_advection"):
        st = _with_scalars(mesh, st)
    cfg = _cfg(**over)
    k1, k2 = 1, 2
    shards = _shards(st, n_save)
    gs = _handles(shards, cfg)
    lms = [None] if n_save == 1 else [s["lm"] for s in shards]
    _steps(gs, lms, k1, True)
    p = str(tmp_path / "r")
    restart.save(p, gs, lms, k1, mesh)
    for g in gs:
        g.close()
    shards = _shards(st, m_load, sfc_colouring=False)
    gs = _handles(shards, _cfg(use_graph=graph, **over), with_state=False)
    lms = [None] if m_load == 1 else [s["lm"] for s in shards]
    assert restart.load(p, gs, lms, mesh) == k1
    _steps(gs, lms, k2, False)
    single = _handles(_shards(st, 1), cfg)[0]
    _steps([single], [None], k1 + k2, True)
    _assert_owned_equal(single, gs, lms)
    want = bench.run_check(single)
    got = bench.merge_checks([bench.run_check(g, lm)["fields"] for g, lm in zip(gs, lms)])
    assert got["combined_checksum"] == want["combined_checksum"]


def test_resume_from_device_init_on_emulated_ranks(tmp_path):
    """step 0 written right after init_jw.init_on_device (+ the init exchange and the diagnostics) on 3 emulated ranks,
    resumed on one handle: equal to the single handle's device init and steps"""
    mesh = icosa.make_icosahedral_mesh(642)
    stt, draws = init_jw.make_static(mesh, L, _abi.INDEX_CORRECTED)
    cfg = _cfg()
    shards = parallel.make_static_shards(stt, 3)
    gs, lms = [], []
    for sh in shards:
        lm = sh["lm"]
        g = dynamics.Dynamics(_abi.make_dims(len(lm.cells), len(lm.edges), len(lm.vertices), L), cfg)
        g.upload_mesh(sh["static"])
        init_jw.init_on_device(g, sh["static"], init_jw.jw_inputs(mesh, stt, draws, lm), stt.vert)
        gs.append(g); lms.append(lm)
    parallel.InProcessExchanger(gs, lms).exchange(parallel.INIT_EXCHANGE)
    _steps(gs, lms, 0, True)
    p = str(tmp_path / "r0")
    restart.save(p, gs, lms, 0, mesh)
    single = dynamics.Dynamics(dynamics.dims_of(mesh, L), cfg)
    single.upload_mesh(stt.static)
    init_jw.init_on_device(single, stt.static, init_jw.jw_inputs(mesh, stt, draws), stt.vert)
    _steps([single], [None], 2, True)
    g = dynamics.Dynamics(dynamics.dims_of(mesh, L), cfg)
    g.upload_mesh(stt.static)
    assert restart.load(p, g, None, mesh) == 0
    _steps([g], [None], 2, False)
    _assert_owned_equal(single, [g], [None])


def test_restart_fields_abi_equals_declaration():
    lib = dynamics.load_library()
    for cfg in (_cfg(), _cfg(physics_mode=_abi.PHYSICS_CORRECTED), _cfg(config_scalar_advection=1)):
        want = [_abi.FIELD_ID[n] for n in _abi.restart_fields(cfg)]
        ids = np.full(128, -7, np.int32)
        assert lib.mpasb200_restart_fields(C.byref(cfg), ids.ctypes.data, 128) == len(want)
        assert ids[:len(want)].tolist() == want and np.all(ids[len(want):] == -7)
        few = np.full(4, -7, np.int32)
        assert lib.mpasb200_restart_fields(C.byref(cfg), few.ctypes.data, 3) == len(want)     # too small: the full count
        assert few[:3].tolist() == want[:3] and few[3] == -7
        assert lib.mpasb200_restart_fields(C.byref(cfg), None, 0) == len(want)
    assert lib.mpasb200_restart_fields(None, None, 0) == _abi.E_INVAL


def test_nccl_restart_resumes_at_n_and_at_one():
    """save at step 3 at N over NCCL, resume at N and on one GPU, run to step 6 (tests/run_restart_multigpu.py; >= 2 GPUs)"""
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                          "127.0.0.1", "--master-port", "29549", os.path.join(root, "tests", "run_restart_multigpu.py")],
                         capture_output=True, text=True, timeout=900, cwd=root)
    assert out.returncode == 0 and "MULTIGPU_RESTART_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-3000:]
