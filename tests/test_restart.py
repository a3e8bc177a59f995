"""Restart files (mpas_regent_b200/restart.py) and the restart set (include/mpas_b200_restart.def), on the CPU oracle.

The restart set is found again here by poisoning: at a step boundary every field OUTSIDE the set is overwritten, with NaN
and with seeded random finite bits, and 2 steps must give the same mirror as without the poison.  The entries the step never
writes keep the poison; in the unpoisoned run they must be zero, which is what a fresh handle holds (rule M1)."""
import hashlib
import os

import numpy as np
import pytest

from mpas_regent_b200 import _abi, dynamics, icosa, init_jw, parallel, partition, restart
from mpas_regent_b200._abi import CELL, EDGE, VERTEX, VERTICAL

from . import irregular

L = 6
DT = 600.0
NAMES = [n for n, _, _ in _abi.FIELDS]


def _cfg(physics=_abi.PHYSICS_LITERAL, rkarg=_abi.RKARG_STAGE_INDEX, scalars=False, **over):
    return _abi.default_config(physics_mode=physics, rkarg_policy=rkarg, config_scalar_advection=int(scalars), **over)


_MESHES = {}


def _problem(kind, scalars):
    """(global mesh, HostState) on x1.642 or the masked irregular mesh, with tracers when ``scalars``"""
    if kind not in _MESHES:
        if kind == "x1.642":
            mesh = icosa.make_icosahedral_mesh(642)
            st = init_jw.make_state(mesh, L, _abi.INDEX_CORRECTED)
        else:
            mesh = irregular.irregular_mesh()
            st = irregular.make_state(L, _abi.INDEX_CORRECTED)
        _MESHES[kind] = (mesh, st)
    mesh, st = _MESHES[kind]
    if scalars:
        st = init_jw.HostState(nVertLevels=st.nVertLevels, policy=st.policy, mesh=st.mesh, static=st.static, vert=st.vert,
                               f=dict(st.f, scalars=1e-3 * (1.0 + np.random.default_rng(2).random((mesh.nCells, L + 1, 8)))))
    return mesh, st


def _single(mesh, st, cfg, steps):
    from oracle.oracle import Oracle
    o = Oracle(dynamics.dims_of(mesh, L), cfg)
    o.upload_mesh(st.static); o.upload_state(st.f, st.vert)
    o.atm_compute_solve_diagnostics(False, -1)
    for _ in range(steps):
        o.atm_srk3(DT)
    return o


def _poisoned_run(mesh, st, cfg, pre, poison, how):
    o = _single(mesh, st, cfg, pre)
    rng = np.random.default_rng(11)
    for n in poison:
        shp = o.field_shape(n)
        if how == "nan":
            a = np.full(shp, np.nan)
        else:                       # random finite bits: a random sign, exponent and mantissa, not inf / NaN
            bits = rng.integers(0, 1 << 63, size=shp, dtype=np.int64).view(np.uint64)
            bits &= ~np.uint64(0x7ff0000000000000) | np.uint64(0x3ff0000000000000)
            bits |= rng.integers(0, 2, size=shp, dtype=np.uint64) << np.uint64(63)
            a = bits.view(np.float64)
        o.upload_field(n, a)
    out = []
    for _ in range(2):
        o.atm_srk3(DT)
        out.append(o.download_all())
    return out


POISON_CASES = [(mk, ph, rk, sc, pre) for mk in ("x1.642", "irregular") for ph in (_abi.PHYSICS_LITERAL, _abi.PHYSICS_CORRECTED)
                for rk in (_abi.RKARG_SUBSTEP_TRUNC, _abi.RKARG_STAGE_INDEX) for sc in (False, True) for pre in (0, 1)]


@pytest.mark.parametrize("mk,physics,rkarg,scalars,pre", POISON_CASES,
                         ids=[f"{c[0]}-{'corr' if c[1] else 'lit'}-rkarg{c[2]}-{'scal' if c[3] else 'noscal'}-step{c[4]}" for c in POISON_CASES])
def test_restart_set_is_complete(mk, physics, rkarg, scalars, pre):
    mesh, st = _problem(mk, scalars)
    cfg = _cfg(physics, rkarg, scalars)
    keep = set(_abi.restart_fields(cfg))
    poison = [n for n in NAMES if n not in keep]
    refs = _poisoned_run(mesh, st, cfg, pre, [], "nan")
    nans = _poisoned_run(mesh, st, cfg, pre, poison, "nan")
    rnds = _poisoned_run(mesh, st, cfg, pre, poison, "random")
    for step, (ref, got_nan, got_rnd) in enumerate(zip(refs, nans, rnds), 1):     # after each of the 2 steps
        for n in NAMES:
            if n in keep:
                assert np.array_equal(got_nan[n], ref[n], equal_nan=True), (step, n)
                assert np.array_equal(got_rnd[n], ref[n], equal_nan=True), (step, n)
                continue
            written = ~np.isnan(got_nan[n])          # what the step wrote, and NaN the unpoisoned run has too
            assert np.array_equal(got_nan[n][written], ref[n][written], equal_nan=True), (step, n)
            assert np.array_equal(got_rnd[n][written], ref[n][written], equal_nan=True), (step, n)
            rest = ref[n][~written]
            assert np.all((rest == 0) | np.isnan(rest)), (step, n, "an entry the step never writes is not zero")


def test_restart_set_has_no_dead_entry():
    """each field of the set, poisoned alone with NaN at step 0, changes the mirror 2 steps later"""
    mesh, st = _problem("x1.642", True)
    cfg = _cfg(_abi.PHYSICS_LITERAL, _abi.RKARG_SUBSTEP_TRUNC, True)
    ref = _poisoned_run(mesh, st, cfg, 0, [], "nan")[-1]
    for n in _abi.restart_fields(cfg):
        got = _poisoned_run(mesh, st, cfg, 0, [n], "nan")[-1]
        assert any(not np.array_equal(got[m], ref[m], equal_nan=True) for m in NAMES), n


def test_restart_declaration_parsed():
    when = [w for _, w in _abi.RESTART]
    assert (when.count("ALWAYS"), when.count("CORRECTED"), when.count("SCALARS")) == (62, 0, 1)
    assert len({n for n, _ in _abi.RESTART}) == len(_abi.RESTART)
    assert _abi.restart_fields(_cfg()) == [n for n, w in _abi.RESTART if w == "ALWAYS"]
    assert _abi.restart_fields(_cfg(scalars=True))[-1] == "scalars"
    assert _abi.restart_fields(_cfg(physics=_abi.PHYSICS_CORRECTED)) == _abi.restart_fields(_cfg())


# ---- N ranks in one process ----------------------------------------------------------------------------------------
def _colours(mesh, world, kind):
    if kind == "sfc":
        return partition.sfc_colouring(mesh, world)
    if kind == "random":
        return np.random.default_rng(5).integers(0, world, mesh.nCells).astype(np.int32)
    return ((np.arange(mesh.nCells) // 16) % world).astype(np.int32)     # scattered blocks


def _shards(st, world, colouring):
    return parallel.make_shards(st, world, colours=None if world == 1 else _colours(st.mesh, world, colouring))


def _backends(shards, cfg, with_state=True):
    from oracle.oracle import Oracle
    out = []
    for sh in shards:
        lm = sh["lm"]
        o = Oracle(_abi.make_dims(len(lm.cells), len(lm.edges), len(lm.vertices), L), cfg)
        o.upload_mesh(sh["static"])
        if with_state:
            o.upload_state(sh["f"], sh["vert"])
        out.append(o)
    return out


def _schedule(cfg):
    seq = []

    class Rec(dynamics.TaskAPI):
        def __init__(self):
            self.cfg, self.dims = cfg, None

        def _call(self, name, *args):
            seq.append((name, args))

    Rec().atm_srk3_by_tasks(DT)
    return seq


def _lockstep(backs, lms, steps, init):
    ex = parallel.InProcessExchanger(backs, lms)
    exchanges = parallel.exchanges_for(backs[0].cfg)
    if init:
        for b in backs:
            b.atm_compute_solve_diagnostics(False, -1)
        ex.exchange(exchanges["compute_solve_diagnostics"])
    seq = _schedule(backs[0].cfg)
    for _ in range(steps):
        for name, args in seq:
            for b in backs:
                b._call(name, *args)
            spec = exchanges.get(parallel.exchange_key(name, args))
            if spec:
                ex.exchange(spec)


def _digests(path):
    return {f: hashlib.sha256(open(os.path.join(path, f), "rb").read()).hexdigest()
            for f in sorted(os.listdir(path)) if f.endswith(".npy")}


def _save_at(tmp, mesh, st, cfg, world, colouring, steps, tag):
    shards = _shards(st, world, colouring)
    backs = _backends(shards, cfg)
    lms = [s["lm"] for s in shards]
    _lockstep(backs, lms, steps, True)
    p = str(tmp / tag)
    restart.save(p, backs, lms, steps, mesh)
    return p


@pytest.mark.parametrize("physics", [_abi.PHYSICS_LITERAL, _abi.PHYSICS_CORRECTED], ids=["literal", "corrected"])
@pytest.mark.parametrize("steps", [0, 2])
def test_same_bytes_at_every_rank_count(tmp_path, physics, steps):
    mesh, st = _problem("x1.642", False)
    cfg = _cfg(physics)
    ref = _digests(_save_at(tmp_path, mesh, st, cfg, 1, "sfc", steps, "n1"))
    assert len(ref) == len(_abi.restart_fields(cfg))
    for world, colouring in ((2, "sfc"), (3, "random"), (4, "blocks"), (4, "sfc")):
        p = _save_at(tmp_path, mesh, st, cfg, world, colouring, steps, f"n{world}_{colouring}")
        assert _digests(p) == ref, (world, colouring)
        assert restart._check_meta(p, cfg, dynamics.dims_of(mesh, L), mesh) is None


def _assert_owned_equal(single, backs, lms):
    rows = lambda lm: {CELL: lm.cells, EDGE: lm.edges, VERTEX: lm.vertices}
    for b, lm in zip(backs, lms):
        for name, ent, _ in _abi.FIELDS:
            a, ref = b.download_field(name), single.download_field(name)
            if ent == VERTICAL:
                assert np.array_equal(a, ref, equal_nan=True), name
            else:
                n = lm.n_owned[ent]
                assert np.array_equal(a[:n], ref[rows(lm)[ent][:n]], equal_nan=True), (name, lm.rank)


RESUME_CASES = [(n, m, ph, sc) for (n, m) in ((1, 3), (3, 1), (2, 4), (4, 2))
                for (ph, sc) in ((_abi.PHYSICS_LITERAL, False), (_abi.PHYSICS_CORRECTED, False), (_abi.PHYSICS_CORRECTED, True))]


@pytest.mark.parametrize("n_save,m_load,physics,scalars", RESUME_CASES,
                         ids=[f"{c[0]}to{c[1]}-{'corr' if c[2] else 'lit'}{'-scal' if c[3] else ''}" for c in RESUME_CASES])
def test_resume_at_another_rank_count(tmp_path, n_save, m_load, physics, scalars):
    import bench
    mesh, st = _problem("x1.642", scalars)
    cfg = _cfg(physics, scalars=scalars)
    k1, k2 = 1, 1
    p = _save_at(tmp_path, mesh, st, cfg, n_save, "sfc", k1, "r")
    shards = _shards(st, m_load, "random")
    backs = _backends(shards, cfg, with_state=False)
    lms = [s["lm"] for s in shards]
    assert restart.load(p, backs, lms, mesh) == k1
    _lockstep(backs, lms, k2, False)
    single = _single(mesh, st, cfg, k1 + k2)
    _assert_owned_equal(single, backs, lms)
    want = bench.run_check(single)
    got = bench.merge_checks([bench.run_check(b, lm)["fields"] for b, lm in zip(backs, lms)])
    assert got["combined_checksum"] == want["combined_checksum"]


def _one(mesh, st, cfg):
    from oracle.oracle import Oracle
    o = Oracle(dynamics.dims_of(mesh, L), cfg)
    o.upload_mesh(st.static)
    return o


@pytest.mark.parametrize("case", ["mesh", "levels", "config", "no_meta", "byte", "execution_only"])
def test_refusals(tmp_path, case):
    mesh, st = _problem("x1.642", False)
    cfg = _cfg()
    p = str(tmp_path / "r")
    restart.save(p, _single(mesh, st, cfg, 0), None, 0, mesh)
    if case == "mesh":
        m2, st2 = _problem("irregular", False)
        with pytest.raises(ValueError, match="nCells|topology"):
            restart.load(p, _one(m2, st2, cfg), None, m2)
        other = icosa.make_icosahedral_mesh(642)                 # same dims, other connectivity
        other.v["cellsOnEdge"] = other.v["cellsOnEdge"][:, ::-1].copy()
        with pytest.raises(ValueError, match="topology_sha256"):
            restart.load(p, _one(mesh, st, cfg), None, other)
        return
    if case == "levels":
        st2 = init_jw.make_state(mesh, L + 1, _abi.INDEX_CORRECTED)
        from oracle.oracle import Oracle
        o = Oracle(dynamics.dims_of(mesh, L + 1), cfg)
        o.upload_mesh(st2.static)
        with pytest.raises(ValueError, match="nVertLevels"):
            restart.load(p, o, None, mesh)
        return
    if case == "config":
        with pytest.raises(ValueError, match="config_epssm"):
            restart.load(p, _one(mesh, st, _cfg(config_epssm=0.2)), None, mesh)
        with pytest.raises(ValueError, match="acoustic_tma"):
            restart.load(p, _one(mesh, st, _cfg(acoustic_tma=2)), None, mesh)
        return
    if case == "no_meta":
        os.remove(os.path.join(p, "meta.json"))
        with pytest.raises(ValueError, match="meta.json"):
            restart.load(p, _one(mesh, st, cfg), None, mesh)
        return
    if case == "byte":
        f = os.path.join(p, "theta_m.npy")
        raw = bytearray(open(f, "rb").read())
        raw[len(raw) // 2] ^= 0x01
        open(f, "wb").write(bytes(raw))
        with pytest.raises(ValueError, match="theta_m"):
            restart.load(p, _one(mesh, st, cfg), None, mesh)
        return
    o = _one(mesh, st, _cfg(sfc_renumber=0, use_graph=1, kernel_forms=1, device=3))
    assert restart.load(p, o, None, mesh) == 0


# ---- torch.distributed (gloo): two processes save, one resumes ------------------------------------------------------
def _gloo_worker(rank, world, port, tmp):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        mesh, st = _problem("x1.642", False)
        cfg = _cfg()
        sh = parallel.make_shards(st, world)[rank]
        b = _backends([sh], cfg)[0]
        run = parallel.DistributedDynamics(b, parallel.HostDistExchanger(b, sh["lm"]))
        run.init_diagnostics()
        run.step(DT)
        run.flush()
        restart.save(os.path.join(tmp, "r"), b, sh["lm"], 1, mesh if rank == 0 else None, dist)
        open(os.path.join(tmp, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def test_gloo_world_size_2(tmp_path):
    import socket
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_gloo_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert os.path.exists(tmp_path / "ok0") and os.path.exists(tmp_path / "ok1")
    mesh, st = _problem("x1.642", False)
    cfg = _cfg()
    assert _digests(str(tmp_path / "r")) == _digests(_save_at(tmp_path, mesh, st, cfg, 1, "sfc", 1, "n1"))
    o = _one(mesh, st, cfg)
    assert restart.load(str(tmp_path / "r"), o, None, mesh) == 1
    o.atm_srk3(DT)
    single = _single(mesh, st, cfg, 2)
    for n in NAMES:
        assert np.array_equal(o.download_field(n), single.download_field(n), equal_nan=True), n
