"""Restart files that any rank count can resume from, bit for bit.

A restart is a directory:

* ``<field>.npy`` for every field of the restart set (include/mpas_b200_restart.def, ``_abi.restart_fields``): float64 of
  global shape [nGlobal][nVertLevels+1] ([..][slots] for array-typed fields, [nVertLevels+1] for vertical ones), rows in
  global entity order.  Owned rows of every field equal the single partition's rows, so the files have the same bytes
  whatever the rank count and colouring that wrote them.
* ``meta.json``: format version, step count, global dims, nVertLevels, the whole MpasConfig, a SHA-256 of the global
  connectivity and one checksum per field.  It is written last: a directory without it is an incomplete save.

The checksum of a field is the MpasFieldSummary checksum (mpas_b200.h) over every row in global numbering, merged over
ranks by a sum mod 2^64.  An array-typed field counts as nVertLevels+1 x slots levels; it and the vertical fields are
summed on the host, because the device scan (mpasb200_summarize_field) takes scalar 3-D fields only.

``save`` / ``load`` take one handle (any TaskAPI) and its partition.LocalMesh (None: the handle holds the whole mesh), or
equal-length lists of them for ranks emulated in one process.  With ``dist`` (torch.distributed, initialised) the ranks
are processes, and the directory must be on a file system every rank sees.  ``mesh`` is the global Mesh; with ``dist`` only
rank 0 reads it.  Save at a step boundary, after the last exchange has landed (DistributedDynamics.flush,
mpasb200_dist_flush).
"""
from __future__ import annotations

import hashlib
import json
import os
from typing import Dict, List, Optional

import numpy as np

from . import _abi
from ._abi import CELL, EDGE, FIELD_ENTITY, FIELD_SLOTS, VERTEX, VERTICAL

FORMAT_VERSION = 1
META = "meta.json"

#: MpasConfig fields that select how a step is executed and not its bits (mpas_b200.h): a restart written under one value
#: resumes under another.  The acoustic forms (acoustic_exact, acoustic_tma) are a few ulp apart and are not listed.
EXECUTION_ONLY = ("sfc_renumber", "device", "use_graph", "kernel_forms", "gather_stage", "edge_tiles")

#: the connectivity the fingerprint covers
TOPOLOGY = ("cellsOnEdge", "edgesOnCell", "verticesOnCell", "cellsOnVertex", "edgesOnVertex")

_M64 = (1 << 64) - 1


def fingerprint(mesh) -> str:
    """SHA-256 of the global connectivity (TOPOLOGY, raw stored ids as int32, names and shapes included)"""
    h = hashlib.sha256()
    for name in TOPOLOGY:
        a = np.ascontiguousarray(mesh.v[name], dtype=np.int32)
        h.update(f"{name}{a.shape}".encode())
        h.update(a.tobytes())
    return h.hexdigest()


def _config_dict(cfg) -> Dict[str, float]:
    return {k: (float(getattr(cfg, k)) if t is _abi.C.c_double else int(getattr(cfg, k))) for k, t in cfg._fields_}


def _parts(dyn, lm):
    return (list(dyn), list(lm)) if isinstance(dyn, (list, tuple)) else ([dyn], [lm])


def _rows(d, m, ent):
    """(global ids of the local rows, number of owned rows) of one handle"""
    n = d.entity_count(ent)
    if m is None:
        return np.arange(n), n
    gid = {CELL: m.cells, EDGE: m.edges, VERTEX: m.vertices}[ent]
    return np.asarray(gid), m.n_owned[ent]


def _set_global_ids(d, m):
    for ent, attr in ((CELL, "cells"), (EDGE, "edges"), (VERTEX, "vertices")):
        d.set_global_ids(ent, None if m is None else getattr(m, attr))


def _mix64(z: np.ndarray) -> np.ndarray:
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xbf58476d1ce4e5b9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94d049bb133111eb)
    return z ^ (z >> np.uint64(31))


def _host_checksum(a: np.ndarray, gid, chunk: int = 1 << 14) -> int:
    """the MpasFieldSummary checksum of rows ``a`` with global ids ``gid``, every trailing axis flattened into levels"""
    a = a.reshape(a.shape[0], -1)
    nl = a.shape[1]
    lev = np.arange(nl, dtype=np.uint64)[None, :]
    cs = 0
    with np.errstate(over="ignore"):
        for i in range(0, a.shape[0], chunk):
            x = np.ascontiguousarray(a[i:i + chunk], dtype=np.float64)
            bits = x.view(np.uint64).copy()
            bits[np.isnan(x)] = np.uint64(0x7ff8000000000000)
            ids = np.asarray(gid[i:i + chunk]).astype(np.uint64)[:, None] * np.uint64(nl) + lev
            cs += int(_mix64(bits + np.uint64(0x9e3779b97f4a7c15) * (ids + np.uint64(1))).sum(dtype=np.uint64))
    return cs & _M64


def _checksum(d, name: str, n_own: int, rows: np.ndarray, gid) -> int:
    """checksum of the owned rows of ``name``: the device scan for scalar 3-D fields (after _set_global_ids), else the
    host restatement over ``rows`` (the handle's rows as uploaded or downloaded)"""
    if FIELD_SLOTS[name] == 1:
        return int(d.summarize_field(name, n_own)["checksum"], 16)
    return _host_checksum(rows[:n_own], gid[:n_own])


def _global_shape(name: str, n_global: Dict[int, int], L1: int):
    ent, s = FIELD_ENTITY[name], FIELD_SLOTS[name]
    if ent == VERTICAL:
        return (L1,)
    return (n_global[ent], L1) if s == 1 else (n_global[ent], L1, s)


def _sum_over_ranks(cs: Dict[str, int], dist) -> Dict[str, int]:
    if dist is None or dist.get_world_size() == 1:
        return cs
    every = [None] * dist.get_world_size()
    dist.all_gather_object(every, cs)
    return {k: sum(p[k] for p in every) & _M64 for k in cs}


def _fsync(path: str):
    fd = os.open(path, os.O_RDONLY)
    try:
        os.fsync(fd)
    finally:
        os.close(fd)


def save(path: str, dyn, lm, step: int, mesh, dist=None) -> None:
    """write the restart set of ``dyn`` (one handle, or a list of emulated ranks) to the directory ``path``"""
    dyns, lms = _parts(dyn, lm)
    rank0 = dist is None or dist.get_rank() == 0
    cfg, L1 = dyns[0].cfg, dyns[0].dims.nVertLevels + 1
    names = _abi.restart_fields(cfg)
    files = {n: os.path.join(path, n + ".npy") for n in names}
    if rank0:
        os.makedirs(path, exist_ok=True)
        if os.path.exists(os.path.join(path, META)):
            os.remove(os.path.join(path, META))
        n_global = {CELL: mesh.nCells, EDGE: mesh.nEdges, VERTEX: mesh.nVertices}
        for n in names:
            mm = np.lib.format.open_memmap(files[n], mode="w+", dtype=np.float64, shape=_global_shape(n, n_global, L1))
            del mm
    if dist is not None:
        dist.barrier()
    for d, m in zip(dyns, lms):
        _set_global_ids(d, m)
    cs = {n: 0 for n in names}
    for n in names:
        ent = FIELD_ENTITY[n]
        if ent == VERTICAL:
            if rank0:
                a = dyns[0].download_field(n)
                mm = np.lib.format.open_memmap(files[n], mode="r+")
                mm[:] = a
                mm.flush()
                del mm
                cs[n] = _host_checksum(a[None, :], np.zeros(1, np.int64))
            continue
        mm = np.lib.format.open_memmap(files[n], mode="r+")
        for d, m in zip(dyns, lms):
            a = d.download_field(n)
            gid, n_own = _rows(d, m, ent)
            mm[gid[:n_own]] = a[:n_own]
            cs[n] = (cs[n] + _checksum(d, n, n_own, a, gid)) & _M64
        mm.flush()
        del mm
    for n in names:
        _fsync(files[n])
    cs = _sum_over_ranks(cs, dist)
    if dist is not None:
        dist.barrier()
    if rank0:
        d0 = dyns[0].dims
        meta = {"format": "mpas_b200 restart", "version": FORMAT_VERSION, "step": int(step),
                "dims": {"nCells": mesh.nCells, "nEdges": mesh.nEdges, "nVertices": mesh.nVertices, "nVertLevels": int(d0.nVertLevels)},
                "config": _config_dict(cfg), "topology_sha256": fingerprint(mesh), "fields": names,
                "checksums": {n: f"{cs[n]:016x}" for n in names}}
        tmp = os.path.join(path, META + ".tmp")
        with open(tmp, "w") as fh:
            json.dump(meta, fh, indent=1)
            fh.flush()
            os.fsync(fh.fileno())
        os.replace(tmp, os.path.join(path, META))
        _fsync(path)
    if dist is not None:
        dist.barrier()


def _check_meta(path: str, cfg, dims, mesh) -> Optional[str]:
    """None, or why the restart at ``path`` cannot be loaded into handles of ``cfg`` / ``dims`` on ``mesh``"""
    p = os.path.join(path, META)
    if not os.path.exists(p):
        return f"{path}: no {META} (an incomplete save, or not a restart)"
    with open(p) as fh:
        meta = json.load(fh)
    if meta.get("version") != FORMAT_VERSION:
        return f"{META}: version {meta.get('version')}, this library reads {FORMAT_VERSION}"
    want = {"nCells": mesh.nCells, "nEdges": mesh.nEdges, "nVertices": mesh.nVertices, "nVertLevels": int(dims.nVertLevels)}
    for k, v in want.items():
        if meta["dims"][k] != v:
            return f"{META}: {k} = {meta['dims'][k]}, the handle has {v}"
    if meta["topology_sha256"] != fingerprint(mesh):
        return f"{META}: topology_sha256 differs: the restart was written on another mesh"
    mine = _config_dict(cfg)
    for k, v in mine.items():
        if k not in EXECUTION_ONLY and meta["config"].get(k) != v:
            return f"{META}: config {k} = {meta['config'].get(k)}, the handle has {v}"
    if meta["fields"] != _abi.restart_fields(cfg):
        return f"{META}: fields {meta['fields']} are not the restart set of this library"
    return None


def load(path: str, dyn, lm, mesh, dist=None) -> int:
    """upload the restart at ``path`` into ``dyn`` (one handle or a list; upload_mesh done, any rank count and colouring)
    and return its step count.  Raises ValueError naming the key or field on any mismatch."""
    dyns, lms = _parts(dyn, lm)
    rank0 = dist is None or dist.get_rank() == 0
    err = _check_meta(path, dyns[0].cfg, dyns[0].dims, mesh) if rank0 else None
    if dist is not None and dist.get_world_size() > 1:
        box = [err]
        dist.broadcast_object_list(box, src=0)
        err = box[0]
    if err is not None:
        raise ValueError(err)
    with open(os.path.join(path, META)) as fh:
        meta = json.load(fh)
    names = meta["fields"]
    L1 = dyns[0].dims.nVertLevels + 1
    n_global = {CELL: meta["dims"]["nCells"], EDGE: meta["dims"]["nEdges"], VERTEX: meta["dims"]["nVertices"]}
    for d, m in zip(dyns, lms):
        _set_global_ids(d, m)
    cs = {n: 0 for n in names}
    for n in names:
        a = np.load(os.path.join(path, n + ".npy"), mmap_mode="r")
        ent = FIELD_ENTITY[n]
        want = _global_shape(n, n_global, L1)
        if a.dtype != np.float64 or a.shape != want:
            raise ValueError(f"{n}.npy: {a.dtype} {a.shape}, expected float64 {want}")
        if ent == VERTICAL:
            v = np.array(a)
            for d in dyns:
                d.upload_field(n, v)
            if rank0:
                cs[n] = _host_checksum(v[None, :], np.zeros(1, np.int64))
            continue
        for d, m in zip(dyns, lms):
            gid, n_own = _rows(d, m, ent)
            rows = np.ascontiguousarray(a[gid])
            d.upload_field(n, rows)
            cs[n] = (cs[n] + _checksum(d, n, n_own, rows, gid)) & _M64
        del a
    cs = _sum_over_ranks(cs, dist)
    for n in names:
        if f"{cs[n]:016x}" != meta["checksums"][n]:
            raise ValueError(f"{n}: checksum {cs[n]:016x} of the uploaded rows, {META} has {meta['checksums'][n]}")
    return int(meta["step"])
