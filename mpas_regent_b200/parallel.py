"""One process per GPU: owned/ghost partitions of the mesh and the halo exchanges of the RK3 step.

The reference computes the owned / ghost partitions (mesh_loading.rg:399-483) but never runs more
than one of them (main.rg:54-55; CURIS_2021_DependentPartitioning_BearE.md:50-58).  Here every rank
holds [owned | ghost ring 1 | ghost ring 2] cells plus all their edges and vertices, runs every task
on all of them (ghost entities are recomputed redundantly) and repairs the ghost values that the
stencils invalidate with packed neighbour exchanges.  With 2 rings the literal dataflow needs these
exchanges per RK stage (10 per step; SURVEY.md 8e, Appendix B):

    after the first acoustic step         cells    w                       (atm_compute_dyn_tend's w tendency; read at cellsOnEdge by the next stage's tend_u)
    after every atm_advance_acoustic_step cells    rtheta_pp, rtheta_pp_old (read at cellsOnEdge by divergence damping)
    after atm_compute_solve_diagnostics   cells    ke, divergence ; edges pv_edge, v ; vertices vorticity

Everything else on the path is pointwise or column-local and keeps ghost values valid.  Owned results
are bit-identical to the single-partition run: each entity sums over its own slots in the same order
whatever rank computes it (tests/test_parallel.py, CPU: world_size-2 gloo; GPU: tests/test_parity_gpu.py).

The wire is torch.distributed (NCCL send/recv over NVLink on the GPU box, gloo in the CPU tests);
pack / unpack run in libmpas_b200 (k_pack / k_unpack).  DistributedDynamics.enable_overlap() moves the exchanges to a
communication stream and hides them under interior compute (launch classes + TaskAPI.restrict); without it they run
on the stream that carries the step.
"""
from __future__ import annotations

import os
import time
from typing import Callable, Dict, List, Optional, Sequence

import numpy as np

from . import _abi, partition
from ._abi import CELL, EDGE, FIELD_ENTITY, FIELD_SLOTS, VERTEX
from .dynamics import TaskAPI, merge_integrals as _merge_integrals

ENT = {"cell": CELL, "edge": EDGE, "vertex": VERTEX}

#: task name (hook key) -> {entity: [fields]} exchanged right after it.  atm_compute_dyn_tend leaves `w` (the w tendency,
#: Q17) invalid on the outer ghost ring; nothing reads it across cells before the next stage's tend_u, and
#: atm_set_smlstep_pert_variables rewrites it column by column, so it rides on the exchange after the FIRST acoustic
#: step of the stage (10 exchanges per step instead of 13).
EXCHANGES: Dict[str, Dict[str, List[str]]] = {
    "advance_acoustic_step:first": {"cell": ["w", "rtheta_pp", "rtheta_pp_old"]},
    "advance_acoustic_step": {"cell": ["rtheta_pp", "rtheta_pp_old"]},
    "compute_solve_diagnostics": {"cell": ["ke", "divergence"], "edge": ["pv_edge", "v"], "vertex": ["vorticity"]},
    # config_scalar_advection: the advection stencil reads `scalars` two rings out (rk_timestep.rg:469 = MPAS's halo update)
    "advance_scalars": {"cell": ["scalars"]},
}

#: MPASB200_PHYSICS_CORRECTED: the acoustic edge update reads rho_pp across cells and atm_recover_large_step_variables runs,
#: so everything the acoustic step leaves invalid on the outer ghost ring is repaired, and so is what recover derives
#: from ru_p on the outermost edges (u, ru, ruAvg) and gathers from them (w).
EXCHANGES_CORRECTED: Dict[str, Dict[str, List[str]]] = {
    "advance_acoustic_step:first": {"cell": ["w", "rtheta_pp", "rtheta_pp_old", "rho_pp", "rw_p", "wwAvg"]},
    "advance_acoustic_step": {"cell": ["rtheta_pp", "rtheta_pp_old", "rho_pp", "rw_p", "wwAvg"]},
    "recover_large_step_variables": {"cell": ["w"], "edge": ["u", "ru", "ruAvg"]},
    "compute_solve_diagnostics": {"cell": ["ke", "divergence"], "edge": ["pv_edge", "v"], "vertex": ["vorticity"]},
    "advance_scalars": {"cell": ["scalars"]},
}


#: init_jw.init_on_device run on a local mesh computes every owned entity right (its stencils reach ring 1 at most) but
#: leaves ghost ring 2 and the edges to cells not held wrong (inf / NaN on some); this one exchange after it copies every
#: cell and edge field the device init writes from owner to holder, after which each rank equals the single-partition
#: device init restricted to its rows, ghosts included.
INIT_EXCHANGE: Dict[str, List[str]] = {
    "cell": ["zgrid", "zz", "rho_base", "pressure_p", "rho_p", "theta_base", "exner", "theta_m", "rtheta_p", "rho_zz", "rw", "w",
             "zb_cell", "zb3_cell", "rtheta_base", "exner_base", "pressure_base", "dss", "uReconstructX", "uReconstructY",
             "uReconstructZ", "uReconstructZonal", "uReconstructMeridional", "h", "rt_diabatic_tend", "t_init", "tend_rho_physics",
             "tend_rtheta_physics", "theta_m_save"],
    "edge": ["zxu", "u", "ru", "zb", "zb3", "rho_edge", "tend_ru_physics", "u_tend", "tend_ru", "cqu"],
}

#: k_pack / k_unpack move at most this many buffer entries (fields x slots) per launch (mpasb200_pack)
PACK_MAX_ENTRIES = 32


def pack_groups(names: Sequence[str]) -> List[List[str]]:
    """split a field list into consecutive groups that one pack / unpack launch can carry"""
    groups, n = [[]], 0
    for name in names:
        s = FIELD_SLOTS[name]
        if n + s > PACK_MAX_ENTRIES:
            groups.append([]); n = 0
        groups[-1].append(name); n += s
    return groups


def exchange_key(name: str, args=()) -> str:
    """hook key of a task call: the first acoustic step of a stage (small_step == 0) has its own."""
    return "advance_acoustic_step:first" if name == "advance_acoustic_step" and len(args) >= 2 and int(args[1]) == 0 else name


def exchanges_for(cfg) -> Dict[str, Dict[str, List[str]]]:
    return EXCHANGES_CORRECTED if cfg.physics_mode == _abi.PHYSICS_CORRECTED else EXCHANGES


def launch_classes(lm: partition.LocalMesh, static: Dict[str, np.ndarray]):
    """(cellClass, edgeClass) of a local mesh for MpasMeshPtrs: cells 0 = owned and not sent, 1 = owned and sent to some
    rank, 2 = ghost; edges 0 = both cells owned, 1 = the rest.  The acoustic step of class-1 cells can run first, its
    results travel while class 0 is computed; class-0 edges can be damped before the ghosts arrive."""
    n_own = lm.n_owned[0]
    cc = np.zeros(len(lm.cells), np.uint8)
    cc[n_own:] = 2
    for idx in lm.send["cell"].values():
        cc[idx] = 1
    coe = np.asarray(static["cellsOnEdge"]).reshape(-1, 2).astype(np.int64) - 1          # local ids are 1-based, 0 = absent
    owned = (coe >= 0) & (coe < n_own)
    ec = np.where(owned.all(axis=1), 0, 1).astype(np.uint8)
    return cc, ec


def split_state(fields: Dict[str, np.ndarray], lm: partition.LocalMesh) -> Dict[str, np.ndarray]:
    """restrict global 3-D fields to a rank's local entities (rows in local order)."""
    rows = {CELL: lm.cells, EDGE: lm.edges, VERTEX: lm.vertices}
    out = {}
    for k, a in fields.items():
        if k not in FIELD_ENTITY:
            continue
        out[k] = np.ascontiguousarray(a[rows[FIELD_ENTITY[k]]])
    return out


class Exchanger:
    """moves ghost columns of a set of fields; subclasses provide the wire."""

    def exchange(self, spec: Dict[str, List[str]]):
        raise NotImplementedError


class InProcessExchanger(Exchanger):
    """All ranks live in one process (tests, and the single-GPU emulation of an N-rank run): ghost columns are
    copied owner -> holder through download_field / upload_field."""

    def __init__(self, backends: Sequence[TaskAPI], locals_: Sequence[partition.LocalMesh]):
        self.b, self.l = list(backends), list(locals_)

    def exchange(self, spec: Dict[str, List[str]]):
        for ent, names in spec.items():
            for name in names:
                arrs = [b.download_field(name) for b in self.b]
                for h, lm in enumerate(self.l):
                    for o, ridx in lm.recv[ent].items():
                        arrs[h][ridx] = arrs[o][self.l[o].send[ent][h]]
                for b, a in zip(self.b, arrs):
                    b.upload_field(name, a)


class HostDistExchanger(Exchanger):
    """torch.distributed with host tensors (gloo): the CPU test of the N > 1 plumbing.  Works with any TaskAPI
    backend through download_field / upload_field."""

    def __init__(self, backend: TaskAPI, lm: partition.LocalMesh):
        import torch.distributed as dist
        self.dist, self.b, self.lm = dist, backend, lm

    def exchange(self, spec: Dict[str, List[str]]):
        import torch
        dist = self.dist
        for ent, names in spec.items():
            arrs = {n: self.b.download_field(n) for n in names}
            ops, recvs = [], []
            for peer in sorted(set(self.lm.send[ent]) | set(self.lm.recv[ent])):
                width = [int(np.prod(arrs[n].shape[1:])) for n in names]       # levels x slots per listed entity
                if peer in self.lm.send[ent]:
                    sidx = self.lm.send[ent][peer]
                    buf = torch.from_numpy(np.ascontiguousarray(np.concatenate([arrs[n][sidx].reshape(len(sidx), -1) for n in names], axis=1)))
                    ops.append(dist.P2POp(dist.isend, buf, peer))
                if peer in self.lm.recv[ent]:
                    ridx = self.lm.recv[ent][peer]
                    rbuf = torch.empty((len(ridx), sum(width)), dtype=torch.float64)
                    ops.append(dist.P2POp(dist.irecv, rbuf, peer))
                    recvs.append((ridx, rbuf, width))
            if ops:
                for r in dist.batch_isend_irecv(ops):
                    r.wait()
            for ridx, rbuf, width in recvs:
                a, o = rbuf.numpy(), 0
                for n, wd in zip(names, width):
                    arrs[n][ridx] = a[:, o:o + wd].reshape((len(ridx),) + arrs[n].shape[1:])
                    o += wd
            for n in names:
                self.b.upload_field(n, arrs[n])


    # the overlapped schedule of DistributedDynamics on the CPU: same call sequence, the exchange simply blocks in start()
    def start(self, spec: Dict[str, List[str]]):
        self.exchange(spec)

    def finish(self):
        pass


class NcclExchanger(Exchanger):
    """GPU path: k_pack -> NCCL send/recv (NVLink) -> k_unpack, all ordered on the step's stream.

    Per entity type ONE send list and ONE recv list (all peers concatenated) are registered, so an exchange is one
    pack launch, one grouped NCCL send/recv and one unpack launch per entity type; the rows of a peer are a
    contiguous slice of the [i][field][level] buffer.  Buffers and the P2P descriptors are built once per
    exchange kind."""

    def __init__(self, dyn, lm: partition.LocalMesh, stream):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.dyn, self.lm, self.stream = torch, dist, dyn, lm, stream
        self.L1 = dyn.dims.nVertLevels + 1
        self.ent = {}
        for ent in ("cell", "edge", "vertex"):
            peers_s, peers_r = sorted(lm.send[ent]), sorted(lm.recv[ent])
            s_idx = np.concatenate([lm.send[ent][p] for p in peers_s]) if peers_s else np.zeros(0, np.int32)
            r_idx = np.concatenate([lm.recv[ent][p] for p in peers_r]) if peers_r else np.zeros(0, np.int32)
            s_off = np.cumsum([0] + [len(lm.send[ent][p]) for p in peers_s])
            r_off = np.cumsum([0] + [len(lm.recv[ent][p]) for p in peers_r])
            self.ent[ent] = dict(peers_s=peers_s, peers_r=peers_r, s_off=s_off, r_off=r_off, ns=len(s_idx), nr=len(r_idx),
                                 ls=dyn.register_list(ENT[ent], s_idx) if len(s_idx) else -1,
                                 lr=dyn.register_list(ENT[ent], r_idx) if len(r_idx) else -1)
        self.plans = {}

    def _plan(self, spec):
        key = tuple((e, tuple(n)) for e, n in sorted(spec.items()))
        if key in self.plans:
            return self.plans[key]
        torch, dist = self.torch, self.dist
        items, ops = [], []
        for ent, all_names in spec.items():
            for names in pack_groups(all_names):
                E, nf = self.ent[ent], sum(FIELD_SLOTS[n] for n in names)       # one buffer entry per slot of an array-typed field
                row = nf * self.L1
                sbuf = torch.empty(max(E["ns"] * row, 1), dtype=torch.float64, device="cuda")
                rbuf = torch.empty(max(E["nr"] * row, 1), dtype=torch.float64, device="cuda")
                for i, p in enumerate(E["peers_s"]):
                    ops.append(dist.P2POp(dist.isend, sbuf[E["s_off"][i] * row:E["s_off"][i + 1] * row], p))
                for i, p in enumerate(E["peers_r"]):
                    ops.append(dist.P2POp(dist.irecv, rbuf[E["r_off"][i] * row:E["r_off"][i + 1] * row], p))
                items.append((E, names, sbuf, rbuf))
        self.plans[key] = (items, ops)
        return self.plans[key]

    # ---- the same exchange on a communication stream, so that compute enqueued after start() overlaps it ----------
    def start(self, spec: Dict[str, List[str]]):
        """everything enqueued on the compute stream so far is visible to the pack; returns at once."""
        torch, dist = self.torch, self.dist
        if not hasattr(self, "comm"):
            self.comm = torch.cuda.Stream()
            self.ev_ready, self.ev_done = torch.cuda.Event(), torch.cuda.Event()
        items, ops = self._plan(spec)
        self.ev_ready.record(self.stream)
        self.comm.wait_event(self.ev_ready)
        self.dyn.set_stream(self.comm.cuda_stream)
        try:
            with torch.cuda.stream(self.comm):
                for E, names, sbuf, _ in items:
                    if E["ls"] >= 0:
                        self.dyn.pack(E["ls"], names, sbuf.data_ptr())
                if ops:
                    for r in dist.batch_isend_irecv(ops):
                        r.wait()
                for E, names, _, rbuf in items:
                    if E["lr"] >= 0:
                        self.dyn.unpack(E["lr"], names, rbuf.data_ptr())
                self.ev_done.record(self.comm)
        finally:
            self.dyn.set_stream(self.stream.cuda_stream)

    def finish(self):
        """compute enqueued after this sees the unpacked ghosts."""
        self.stream.wait_event(self.ev_done)

    def exchange(self, spec: Dict[str, List[str]]):
        torch, dist = self.torch, self.dist
        items, ops = self._plan(spec)
        with torch.cuda.stream(self.stream):
            for E, names, sbuf, _ in items:
                if E["ls"] >= 0:
                    self.dyn.pack(E["ls"], names, sbuf.data_ptr())
            if ops:
                for r in dist.batch_isend_irecv(ops):
                    r.wait()          # stream-ordered for NCCL: makes the current stream wait, not the host
            for E, names, _, rbuf in items:
                if E["lr"] >= 0:
                    self.dyn.unpack(E["lr"], names, rbuf.data_ptr())


class NativeDistributedDynamics:
    """The same step with the whole exchange schedule INSIDE libmpas_b200 (mpasb200_dist_init / _set_halo / _srk3_dist):
    NCCL send/recv issued from the C++ driver on the library's own communication stream, overlap by launch classes.
    The host only hands over the NCCL unique id (here through torch.distributed) and the halo lists."""

    def __init__(self, dyn, lm: partition.LocalMesh, rank: int, world: int):
        import torch.distributed as dist
        self.dyn, self.lm = dyn, lm
        box = [dyn.dist_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        dyn.dist_init(rank, world, box[0])
        for ent in ("cell", "edge", "vertex"):
            dyn.dist_set_halo(ENT[ent], lm.send[ent], lm.recv[ent])
        self.overlap = True
        self.t_init = 0.0

    def init_diagnostics(self):
        self.dyn.atm_compute_solve_diagnostics(False, -1)
        self.dyn.dist_exchange(_abi.X_DIAG)

    def step(self, dt: float):
        self.dyn.atm_srk3_dist(dt)

    def flush(self):
        self.dyn.dist_flush()


class DistributedDynamics:
    """atm_srk3 on one rank of an N-rank run: the reference's task sequence (rk_timestep.rg:378-481) with the
    exchanges of EXCHANGES after the tasks that need them."""

    def __init__(self, dyn: TaskAPI, exchanger):
        self.dyn, self.ex = dyn, exchanger
        self.exchanges = exchanges_for(dyn.cfg)
        self.t_init = 0.0

    def _hook(self, name: str, *args):
        if getattr(self, "overlap", False):
            # the exchange after atm_compute_solve_diagnostics of stages 0 and 2 is needed by the next atm_compute_dyn_tend
            # only: it travels under atm_compute_vert_imp_coefs (stage 1) or under substep_finish + the next step's
            # setup / moist / vert_imp coefficients, none of which touches the exchanged fields
            if name == "compute_vert_imp_coefs":
                self.flush()
            elif name == "compute_solve_diagnostics" and len(args) >= 2 and int(args[1]) in (0, 2):
                self.ex.start(self.exchanges[name])
                self._pending = True
                return
        spec = self.exchanges.get(exchange_key(name, args))
        if spec:
            self.ex.exchange(spec)

    def flush(self):
        """complete an exchange that is still travelling (call before reading ghosts from outside a step)."""
        if getattr(self, "_pending", False):
            self.ex.finish()
            self._pending = False

    def init_diagnostics(self):
        """atm_core_init's atm_compute_solve_diagnostics(..., -1) (atm_core.rg:31)."""
        self.dyn.atm_compute_solve_diagnostics(False, -1)
        self._hook("compute_solve_diagnostics")

    def enable_overlap(self):
        """Overlap the acoustic-loop exchanges with interior compute (needs launch classes in the uploaded mesh and an
        exchanger with start()/finish()): boundary-owned cells first, their columns travel while the interior is advanced
        and the interior edges are damped; the edges next to ghosts follow after the unpack.  Ghost cells are never
        advanced: everything the owned entities read from them arrives by exchange.  LITERAL physics only: with
        physics_mode CORRECTED the acoustic edge update belongs to the same task call and must not run once per cell class."""
        self.overlap = (hasattr(self.ex, "start") and hasattr(self.dyn, "restrict")
                        and self.dyn.cfg.physics_mode == _abi.PHYSICS_LITERAL)
        return self.overlap

    def _acoustic_pair(self, dts: float, small_step: int):
        d = self.dyn
        spec = self.exchanges[exchange_key("advance_acoustic_step", (dts, small_step))]
        d.restrict(CELL, 1); d.atm_advance_acoustic_step(dts, small_step)      # sent cells first
        self.ex.start(spec)
        d.restrict(CELL, 0); d.atm_advance_acoustic_step(dts, small_step)      # interior, overlaps the exchange
        d.restrict(EDGE, 0); d.atm_divergence_damping_3d(dts)
        self.ex.finish()
        d.restrict(EDGE, 1); d.atm_divergence_damping_3d(dts)
        d.restrict(CELL); d.restrict(EDGE)

    def step(self, dt: float):
        pair = self._acoustic_pair if getattr(self, "overlap", False) else None
        self.dyn.atm_srk3_by_tasks(dt, hook=self._hook, acoustic_pair=pair)

    # ---- bench helper: rank 0 builds + partitions the global problem, every rank loads its shard -------------
    @classmethod
    def for_bench(cls, n_cells: int, L: int, cfg, stream, rank: int, world: int):
        import torch.distributed as dist
        from . import dynamics
        t0 = time.time()
        shm = os.environ.get("MPAS_B200_SHARDS", "/dev/shm/mpas_b200_shards")
        tag = os.path.join(shm, f"x1.{n_cells}_L{L}_w{world}")
        if rank == 0:
            import bench
            mesh, st, _ = bench.build_inputs(n_cells, L)
            shards = make_shards(st, world)
            os.makedirs(tag, exist_ok=True)
            for r, sh in enumerate(shards):
                save_shard(os.path.join(tag, f"rank{r}"), sh)
            del shards, st
        dist.barrier()
        sh = load_shard(os.path.join(tag, f"rank{rank}"))
        lm, static, fields, vert = sh["lm"], sh["static"], sh["f"], sh["vert"]
        dims = _abi.make_dims(len(lm.cells), len(lm.edges), len(lm.vertices), L)
        dyn = dynamics.Dynamics(dims, cfg)
        dyn.set_stream(stream.cuda_stream)
        dyn.upload_mesh(static)
        dyn.upload_state(fields, vert)
        host_fields = {n: fields[n] for n in getattr(cls, "KEEP_HOST_FIELDS", ()) if n in fields}     # bench.py's end-to-end leg
        del fields
        if os.environ.get("MPAS_B200_NATIVE_DIST", "1") != "0":
            run = NativeDistributedDynamics(dyn, lm, rank, world)
        else:
            run = cls(dyn, NcclExchanger(dyn, lm, stream))
            if cfg.physics_mode == _abi.PHYSICS_LITERAL and os.environ.get("MPAS_B200_OVERLAP", "1") != "0":
                run.enable_overlap()
        run.lm = lm
        run.host_fields = host_fields
        run.init_diagnostics()
        run.t_init = time.time() - t0
        return run


# ---- shards --------------------------------------------------------------------------------------------------
def merge_integrals(parts: Sequence[dict], dist=None) -> dict:
    """Exact global integral from per-partition ones (Dynamics.integrate over each partition's owned entities).  ``parts``
    are the results this process holds; with ``dist`` (torch.distributed, initialised) every process's parts are gathered
    first, limbs as int64 arrays, so no float enters the merge and every rank returns the same bits."""
    parts = list(parts)
    if dist is not None and dist.get_world_size() > 1:
        every = [None] * dist.get_world_size()
        dist.all_gather_object(every, parts)
        parts = [p for ps in every for p in ps]
    return _merge_integrals(parts)


def column_integrals(dyn, area_id: int, n_owned: Optional[int] = None, dist=None, fields: Sequence[str] = ("rho_zz", "ke")) -> dict:
    """{field: exact integral of field x areaCell x (1/rdzw)} over the first ``n_owned`` cells (default all) and levels
    0..nVertLevels-1, merged over ranks (merge_integrals): the total mass for rho_zz.  ``area_id`` = the handle's
    register_weights(CELL, areaCell of the rows it holds)."""
    L = dyn.dims.nVertLevels
    dz = 1.0 / dyn.download_field("rdzw")[:L]
    return {f: merge_integrals([dyn.integrate(f, weight_id=area_id, wv=dz, n_first=n_owned, nlevels=L)], dist) for f in fields}


def isobaric_diagnostics(dyn, lm, plev_pa, dist=None) -> Optional[Dict[str, np.ndarray]]:
    """Dynamics.isobaric_diagnostics of the owned cells of every rank, assembled in global cell order on rank 0 (other ranks
    get None).  ``dyn`` / ``lm`` are this rank's handle and LocalMesh (``lm`` None: one rank holding the whole mesh), or
    equal-length lists of them for ranks emulated in one process; with ``dist`` (torch.distributed, initialised) the rows
    travel to rank 0 over it.  The values are column-local, so the assembled arrays have the same bits at every rank count."""
    dyns, lms = (list(dyn), list(lm)) if isinstance(dyn, (list, tuple)) else ([dyn], [lm])
    parts = []
    for d, m in zip(dyns, lms):
        n = d.dims.nCells if m is None else m.n_owned[0]
        cells = np.arange(n) if m is None else np.asarray(m.cells[:n])
        parts.append((cells, d.isobaric_diagnostics(plev_pa, n_first=n)))
    if dist is not None and dist.get_world_size() > 1:
        every = [None] * dist.get_world_size() if dist.get_rank() == 0 else None
        dist.gather_object(parts, every, dst=0)
        if dist.get_rank() != 0:
            return None
        parts = [p for ps in every for p in ps]
    n = sum(len(c) for c, _ in parts)
    out = {k: np.empty((n,) + v.shape[1:], dtype=np.float64) for k, v in parts[0][1].items()}
    seen = np.zeros(n, dtype=bool)
    for cells, r in parts:
        seen[cells] = True
        for k, v in r.items():
            out[k][cells] = v
    if not seen.all():
        raise ValueError("isobaric_diagnostics: the ranks' owned cells do not cover the mesh")
    return out


def make_static_shards(st, world: int, colours: Optional[np.ndarray] = None):
    """partition the level-0 data of a HostState (CORRECTED policy; init_jw.make_static is enough, no 3-D field is read)
    into per-rank {lm, static}, launch classes included."""
    mesh = st.mesh
    n_global = (mesh.nCells, mesh.nEdges, mesh.nVertices)
    col = colours if colours is not None else (mesh.partition if mesh.partition is not None and mesh.partition.max() + 1 == world
                                               else partition.sfc_colouring(mesh, world))
    part = partition.partition_regions(mesh, col, world, _abi.INDEX_CORRECTED)
    locs, statics = [], []
    for r in range(world):
        lm, loc = partition.build_local(st.static, n_global, col, part, r, mesh.v["cellsOnVertex"])
        locs.append(lm); statics.append(loc)
    partition.build_halo_lists(locs)
    for lm, loc in zip(locs, statics):
        loc["cellClass"], loc["edgeClass"] = launch_classes(lm, loc)
    return [dict(lm=lm, static=loc) for lm, loc in zip(locs, statics)]


def make_shards(st, world: int, colours: Optional[np.ndarray] = None):
    """partition a global HostState (CORRECTED policy) into per-rank {lm, static, f, vert}."""
    return [dict(lm=sh["lm"], static=sh["static"], f=split_state(st.f, sh["lm"]), vert=dict(st.vert))
            for sh in make_static_shards(st, world, colours)]


#: the array dictionaries a shard may carry: level-0 data, 3-D fields, vertical fields, inputs of init_jw.init_on_device
SHARD_PARTS = ("static", "f", "vert", "jw")


def save_shard(path: str, sh):
    os.makedirs(path, exist_ok=True)
    lm = sh["lm"]
    meta = dict(rank=lm.rank, n_owned=np.asarray(lm.n_owned), cells=lm.cells, edges=lm.edges, vertices=lm.vertices,
                interior=lm.interior_cells)
    for ent in ("cell", "edge", "vertex"):
        meta[f"owner_{ent}"] = lm.owner[ent]
        for peer, idx in lm.send[ent].items():
            meta[f"send_{ent}_{peer}"] = idx
        for peer, idx in lm.recv[ent].items():
            meta[f"recv_{ent}_{peer}"] = idx
    np.savez(os.path.join(path, "lm.npz"), **meta)
    for sub in SHARD_PARTS:
        if sub not in sh:
            continue
        os.makedirs(os.path.join(path, sub), exist_ok=True)
        for k, a in sh[sub].items():
            np.save(os.path.join(path, sub, k + ".npy"), a)


def load_shard(path: str):
    z = np.load(os.path.join(path, "lm.npz"))
    lm = partition.LocalMesh(rank=int(z["rank"]), n_owned=tuple(int(v) for v in z["n_owned"]), cells=z["cells"], edges=z["edges"],
                             vertices=z["vertices"], owner={e: z[f"owner_{e}"] for e in ("cell", "edge", "vertex")})
    lm.interior_cells = z["interior"]
    for ent in ("cell", "edge", "vertex"):
        lm.send[ent], lm.recv[ent] = {}, {}
    for k in z.files:
        for kind in ("send", "recv"):
            if k.startswith(kind + "_"):
                _, ent, peer = k.split("_")
                getattr(lm, kind)[ent][int(peer)] = z[k]
    out = dict(lm=lm)
    for sub in SHARD_PARTS:
        d = os.path.join(path, sub)
        if not os.path.isdir(d):
            continue
        out[sub] = {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d)) if f.endswith(".npy")}
    return out
