"""The mesh-only half of the initial state (init_jw.make_static, parallel.make_static_shards), on the CPU: it must be exactly
what make_state / make_shards hand over, so that a rank can build its shard of the 3-D state on its own GPU
(init_jw.init_on_device; tests/test_device_init_gpu.py) from this alone."""
import numpy as np
import pytest

from mpas_regent_b200 import _abi, init_jw, parallel, partition
from mpas_regent_b200.mesh import CORRECTED, resolve_ids

L = 6


def _colours(mesh, kind):
    if kind == "sfc":
        return None, 4
    rng = np.random.default_rng(1)
    if kind == "random":
        return rng.integers(0, 3, mesh.nCells).astype(np.int32), 3      # test_parallel's `random` colouring
    return rng.integers(0, 3, 24).astype(np.int32)[partition.sfc_colouring(mesh, 24)], 3    # scattered blocks


def _same(a, b, what):
    assert a.keys() == b.keys(), what
    for k in a:
        assert a[k].dtype == b[k].dtype and np.array_equal(a[k], b[k]), (what, k)


@pytest.mark.parametrize("kind", ["sfc", "random", "random_blocks"])
def test_static_shards_equal_make_shards(grid642, kind):
    col, world = _colours(grid642, kind)
    full = parallel.make_shards(init_jw.make_state(grid642, L, _abi.INDEX_CORRECTED), world, colours=col)
    st, _ = init_jw.make_static(grid642, L, _abi.INDEX_CORRECTED)
    stat = parallel.make_static_shards(st, world, colours=col)
    assert len(stat) == len(full)
    for a, b in zip(full, stat):
        la, lb = a["lm"], b["lm"]
        assert la.rank == lb.rank and la.n_owned == lb.n_owned
        for attr in ("cells", "edges", "vertices", "interior_cells"):
            assert np.array_equal(getattr(la, attr), getattr(lb, attr)), attr
        for ent in ("cell", "edge", "vertex"):
            assert np.array_equal(la.owner[ent], lb.owner[ent])
            for kind_ in ("send", "recv"):
                da, db = getattr(la, kind_)[ent], getattr(lb, kind_)[ent]
                assert da.keys() == db.keys() and all(np.array_equal(da[p], db[p]) for p in da), (kind_, ent)
        _same(a["static"], b["static"], "static")


@pytest.mark.parametrize("which", ["x1.2562", "icosa642"])
def test_make_static_is_make_state_without_fields(grid2562, grid642, which):
    """level-0 data, vertical grid (u_init / v_init drawn) and the mesh-only extras, bit for bit, under both M5 readings"""
    mesh = grid2562 if which == "x1.2562" else grid642
    for m5 in (True, False):
        full = init_jw.make_state(mesh, L, _abi.INDEX_CORRECTED, m5=m5)
        st, draws = init_jw.make_static(mesh, L, _abi.INDEX_CORRECTED, m5=m5)
        assert (draws is not None) == m5 and not st.f
        assert list(st.static) == list(full.static)
        _same(st.static, full.static, "static")
        _same(st.vert, full.vert, "vert")
        assert np.array_equal(st.extras["coeffs_reconstruct"], full.extras["coeffs_reconstruct"])
        if m5:
            assert np.array_equal(st.extras["deriv_two"], full.extras["deriv_two"])
            assert np.array_equal(full.extras["zb3"][:, :L, :], 0.1 * full.extras["zb"][:, :L, :] * draws["zb3_factor"])
        else:
            assert st.extras["deriv_two"] is None and full.extras["deriv_two"] is None


@pytest.mark.parametrize("kind", ["sfc", "random", "random_blocks"])
def test_m5_fields_on_local_rows(grid642, kind):
    """what init_on_device computes on the host from a shard's inputs: the pointwise M5 fields equal make_state's on every
    local row; rho_edge on every edge whose two cells are held (the rest is repaired by parallel.INIT_EXCHANGE)."""
    col, world = _colours(grid642, kind)
    full = init_jw.make_state(grid642, L, _abi.INDEX_CORRECTED)
    st, draws = init_jw.make_static(grid642, L, _abi.INDEX_CORRECTED)
    for sh in parallel.make_static_shards(st, world, colours=col):
        lm, loc = sh["lm"], sh["static"]
        jw = init_jw.jw_inputs(grid642, st, draws, lm)
        assert np.array_equal(jw["latCell"], st.mesh.v["latCell"][lm.cells]) and np.array_equal(jw["latCell"], loc["latCell"])
        c1, c2 = (resolve_ids(loc["cellsOnEdge"][:, i], len(lm.cells), CORRECTED) for i in (0, 1))
        F = init_jw.m5_fields(jw["modes"], list(jw["cell_xyz"]), list(jw["edge_xyz"]), full.f["theta_m"][lm.cells],
                              full.f["rho_zz"][lm.cells], c1, c2)
        assert set(F) == {m[0] for m in init_jw.M5_SMOOTH} | {"rho_edge"}
        both = (loc["cellsOnEdge"] > 0).all(axis=1)
        assert both[:lm.n_owned[1]].all()
        for k, a in F.items():
            ent = _abi.FIELD_ENTITY[k]
            ref = full.f[k][lm.cells if ent == _abi.CELL else lm.edges]
            if k == "rho_edge":
                assert np.array_equal(a[both], ref[both]), k
            else:
                assert np.array_equal(a, ref), k


def test_init_exchange_covers_what_the_device_init_writes(grid642):
    """every field in the spec lives on its entity, fits the pack launches, and the step-input fields make_state
    produces (other than v, made by atm_compute_solve_diagnostics) are all in it"""
    spec = parallel.INIT_EXCHANGE
    ent = {"cell": _abi.CELL, "edge": _abi.EDGE}
    for e, names in spec.items():
        assert len(set(names)) == len(names)
        assert all(_abi.FIELD_ENTITY[n] == ent[e] for n in names)
        groups = parallel.pack_groups(names)
        assert sum(groups, []) == names
        assert all(sum(_abi.FIELD_SLOTS[n] for n in g) <= parallel.PACK_MAX_ENTRIES for g in groups)
    full = init_jw.make_state(grid642, L, _abi.INDEX_CORRECTED, diag_on_host=False)
    assert set(full.f) <= set(spec["cell"]) | set(spec["edge"])


def test_shard_roundtrip_with_device_init_inputs(grid642, tmp_path):
    st, draws = init_jw.make_static(grid642, L, _abi.INDEX_CORRECTED)
    sh = parallel.make_static_shards(st, 2)[1]
    sh["jw"] = init_jw.jw_inputs(grid642, st, draws, sh["lm"])
    sh["vert"] = st.vert
    parallel.save_shard(str(tmp_path / "r1"), sh)
    back = parallel.load_shard(str(tmp_path / "r1"))
    assert "f" not in back
    for sub in ("static", "jw", "vert"):
        _same(back[sub], sh[sub], sub)


def _digest(arrays):
    import hashlib
    h = hashlib.sha256()
    for k in sorted(arrays):
        a = np.ascontiguousarray(arrays[k])
        h.update(f"{k}:{a.dtype}:{a.shape}".encode()); h.update(a.tobytes())
    return h.hexdigest()


def test_harness_draws_are_pinned(grid2562):
    """make_static and make_state share m5_draws, so comparing them cannot see a reordered or dropped draw: pin the draws
    themselves, and what make_state derives from them with + - * / and sqrt only (bit-identical on every IEEE platform;
    the fields that also pass through sin / cos / exp / pow are left out, numpy's vectorised transcendental functions differ
    in the last place between CPUs).  The second digest is the same at the commit before make_static existed."""
    d = init_jw.m5_draws(grid2562.nCells, grid2562.nEdges, 26)
    assert _digest(d) == "15692751af97bbb0a1d5e08b366ccfc5fb28595644d8f8f0a014d81717a69836"
    st = init_jw.make_state(grid2562, 26, _abi.INDEX_CORRECTED)
    sel = {f"static/{k}": st.static[k] for k in ("defc_a", "defc_b", "coeffs_reconstruct", "adv_coefs", "adv_coefs_3rd")}
    sel.update({f"vert/{k}": st.vert[k] for k in ("u_init", "v_init")})
    sel["extras/deriv_two"] = st.extras["deriv_two"]
    assert _digest(sel) == "af6f197c55872209eec4fa5e9c834693082f6c0cd58d508529e85aaabf4a164e"
