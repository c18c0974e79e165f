"""Equiangulation (the ``u`` command) on the device: ``ms_equiangulate.cuh`` through the host emulator in the CPU tier,
``ms_ctx_equiangulate`` / ``DeviceMesh.equiangulate`` / ``DeviceMinimizer.equiangulate`` in the GPU tier, against the
host twin ``geometry.equiangulate.equiangulate_triangles``: the same rows, flip count and sweep count."""

import ctypes
import json
import os
import subprocess
import types

import numpy as np
import pytest

import ms_test_helpers as H

from membrane_solver_b200 import _lib as L
from membrane_solver_b200.geometry.equiangulate import equiangulate_triangles
from membrane_solver_b200.synthetic import icosphere

ITERATIONS = [1, 2, 100]


# ---- meshes ------------------------------------------------------------------------------------------------------

def jittered_sphere(freq, seed=0):
    """Icosphere with tangential noise of 0.3 x the mean edge length, back on the unit sphere."""
    pos, tri = icosphere(freq, perturb=False)
    rng = np.random.default_rng(seed)
    h = np.mean(np.linalg.norm(pos[tri[:, 1]] - pos[tri[:, 0]], axis=1))
    q = pos + 0.3 * h * rng.normal(size=pos.shape)
    return q / np.linalg.norm(q, axis=1)[:, None], tri


def _sheet():
    """The jittered planar sheet with random diagonals of test_equiangulate.py."""
    rng = np.random.default_rng(7)
    nx, ny = 14, 11
    xs, ys = np.meshgrid(np.arange(nx, dtype=float), np.arange(ny, dtype=float), indexing="ij")
    pts = np.stack([xs.ravel(), ys.ravel()], axis=1)
    interior = (xs.ravel() > 0) & (xs.ravel() < nx - 1) & (ys.ravel() > 0) & (ys.ravel() < ny - 1)
    pts[interior] += rng.uniform(-0.35, 0.35, size=(int(interior.sum()), 2))
    vid = np.arange(nx * ny).reshape(nx, ny)
    a, b, c, d = vid[:-1, :-1].ravel(), vid[1:, :-1].ravel(), vid[1:, 1:].ravel(), vid[:-1, 1:].ravel()
    flip = rng.random(a.size) < 0.5
    tri = np.concatenate([np.where(flip[:, None], np.stack([a, b, d], 1), np.stack([a, b, c], 1)),
                          np.where(flip[:, None], np.stack([b, c, d], 1), np.stack([a, c, d], 1))]).astype(np.int32)
    return np.concatenate([pts, np.zeros((len(pts), 1))], axis=1), tri


def _three_facet_edge():
    """The sheet with a third facet on one interior edge and one facet turned over (an orientation defect)."""
    pos, tri = _sheet()
    e = tri[40, :2]
    pos = np.concatenate([pos, [[pos[e, 0].mean(), pos[e, 1].mean(), 0.7]]])
    tri = np.concatenate([tri, [[e[0], e[1], len(pos) - 1]]]).astype(np.int32)
    tri[100] = tri[100, ::-1]
    return pos, tri


def _same_new_diagonal():
    """Two quads a1-b1 and a2-b2 whose flips would both create the diagonal c-d: only the first may flip."""
    pos = np.array([[0, 0.2, 0], [0, -0.2, 0], [-1, 0, 0], [1, 0, 0], [0, 0, -1], [0, 0, 1]], float)
    c, d, a1, b1, a2, b2 = range(6)
    tri = np.array([[a1, b1, c], [b1, a1, d], [a2, b2, c], [b2, a2, d]], np.int32)
    return pos, tri


def _ellipse_fan(n=50, axis=10.0):
    """Fan of an elongated convex polygon from one tip: the candidates form a chain of shared facets in ascending
    key, so a sweep's selection needs many rounds (17 in the first sweep) and the mesh many sweeps.  The tip has
    valence 48, the most a packed mesh allows."""
    t = np.linspace(0, 2 * np.pi, n, endpoint=False)
    pos = np.stack([axis * np.cos(t), np.sin(t), np.zeros(n)], axis=1)
    tri = np.stack([np.zeros(n - 2, int), np.arange(1, n - 1), np.arange(2, n)], axis=1).astype(np.int32)
    return pos, tri


def _mesh(name):
    """(pos, tri, fixed or None)"""
    if name == "sheet":
        return (*_sheet(), None)
    if name.startswith("sphere"):
        return (*jittered_sphere(32, seed=int(name[-1])), None)
    if name == "catenoid":
        g = np.load(os.path.join(H.GOLDEN, "equiangulate.npz"))
        return g["pos"], g["tri"], np.asarray(g["fixed"], bool)
    if name == "fixed_edges":
        pos, tri = jittered_sphere(12, seed=4)
        return pos, tri, np.random.default_rng(4).uniform(size=len(pos)) < 0.3
    if name.startswith("odd"):
        pos, tri = H.odd_mesh(int(name[-1]), nfan=30)[:2]
        return pos, tri, None
    if name == "three_facet_edge":
        return (*_three_facet_edge(), None)
    if name == "same_new_diagonal":
        return (*_same_new_diagonal(), None)
    if name == "ellipse_fan":
        return (*_ellipse_fan(), None)
    raise KeyError(name)


MESHES = ["sheet", "sphere0", "sphere1", "sphere2", "catenoid", "fixed_edges", "odd1", "odd2", "three_facet_edge",
          "same_new_diagonal", "ellipse_fan"]


def twin(pos, tri, fixed, max_iterations):
    """The twin's rows and flips, and its sweep count: sweeps that flipped, one max_iterations=1 call at a time."""
    rows, flips = equiangulate_triangles(pos, tri, fixed, max_iterations=max_iterations)
    cur, sweeps, total = np.asarray(tri, np.int32), 0, 0
    while sweeps < max_iterations:
        cur, f = equiangulate_triangles(pos, cur, fixed, max_iterations=1)
        if f == 0:
            break
        sweeps += 1
        total += f
    assert total == flips and np.array_equal(cur, rows)
    return rows, flips, sweeps


# ---- CPU tier: the predicate and the selection, compiled for the host ---------------------------------------------

@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    """tests/emul/equiangulate_emul.cpp compiled for the host into a temporary directory (the tree may be
    read-only).  No fp contraction: the host side rounds every operation, as the twin does."""
    out = str(tmp_path_factory.mktemp("eq_emul") / "libms_eq_emul.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-o", out,
                           os.path.join(H.ROOT, "tests", "emul", "equiangulate_emul.cpp")])
    lib = ctypes.CDLL(out)
    lib.emul_equiangulate.restype = ctypes.c_int
    return lib


def emulate(lib, pos, tri, fixed, max_iterations, key_id=None):
    """(rows, flips, sweeps, rounds per sweep run)"""
    rows = np.array(tri, dtype=np.int32, order="C", copy=True)
    pos = np.ascontiguousarray(pos, dtype=np.float64)
    fx = None if fixed is None else np.ascontiguousarray(fixed, dtype=np.uint8)
    kid = None if key_id is None else np.ascontiguousarray(key_id, dtype=np.int32)
    flips, sweeps = ctypes.c_int64(0), ctypes.c_int32(0)
    rounds = np.zeros(max(max_iterations, 1), np.int32)
    rc = lib.emul_equiangulate(ctypes.c_int32(len(pos)), ctypes.c_int32(len(rows)), L.iptr(rows), L.dptr(pos),
                               L.bptr(fx), L.iptr(kid), ctypes.c_int32(max_iterations), ctypes.byref(flips),
                               ctypes.byref(sweeps), L.iptr(rounds))
    assert rc == 0
    n_run = min(sweeps.value + 1, max_iterations)
    return rows, flips.value, sweeps.value, rounds[:n_run]


@pytest.mark.parametrize("name", MESHES)
def test_emulated_sweeps_match_the_twin(emul, name):
    pos, tri, fixed = _mesh(name)
    for it in ITERATIONS:
        want, flips, sweeps = twin(pos, tri, fixed, it)
        rows, f, s, _ = emulate(emul, pos, tri, fixed, it)
        assert (f, s) == (flips, sweeps), (it, f, s, flips, sweeps)
        assert np.array_equal(rows, want), it
    assert flips > 0 or name == "same_new_diagonal"


@pytest.mark.parametrize("name", ["sphere0", "odd1", "three_facet_edge", "ellipse_fan"])
def test_emulated_sweeps_in_a_permuted_vertex_order(emul, name):
    """Rows held in another vertex numbering (as the device's Morton order) with keys taken in the caller's: the
    same flips, mapped back."""
    pos, tri, fixed = _mesh(name)
    perm = np.random.default_rng(9).permutation(len(pos)).astype(np.int32)   # internal -> caller
    inv = np.empty_like(perm)
    inv[perm] = np.arange(len(pos), dtype=np.int32)
    want, flips, sweeps = twin(pos, tri, fixed, 100)
    rows, f, s, _ = emulate(emul, pos[perm], inv[tri], None if fixed is None else fixed[perm], 100, key_id=perm)
    assert (f, s) == (flips, sweeps)
    assert np.array_equal(perm[rows], want)


def test_same_new_diagonal_flips_once(emul):
    pos, tri, _ = _mesh("same_new_diagonal")
    rows, f, s, _ = emulate(emul, pos, tri, None, 100)
    assert (f, s) == (1, 1)
    assert np.array_equal(rows[2:], tri[2:])


def test_selection_of_a_long_conflict_chain_takes_many_rounds(emul):
    pos, tri, _ = _mesh("ellipse_fan")
    _, f, s, rounds = emulate(emul, pos, tri, None, 100)
    print(f"ellipse fan: {f} flips in {s} sweeps, selection rounds per sweep {rounds.tolist()}")
    assert rounds[0] >= 16 and rounds[-1] == 0 and s >= 30


def disk_fan_start(n_rim=60):
    """A centre and n_rim points on a circle, triangulated with spokes to every other rim point and ears between
    them (centre valence n_rim / 2): it packs, but its equiangulation is the full fan of valence n_rim."""
    t = 2 * np.pi * np.arange(n_rim) / n_rim
    pos = np.concatenate([[[0.0, 0.0, 0.0]], np.stack([np.cos(t), np.sin(t), np.zeros(n_rim)], axis=1)])
    k = np.arange(0, n_rim, 2)
    r = lambda i: 1 + i % n_rim                                               # noqa: E731
    tri = np.concatenate([np.stack([np.zeros_like(k), r(k), r(k + 2)], axis=1),
                          np.stack([r(k), r(k + 1), r(k + 2)], axis=1)]).astype(np.int32)
    return pos, tri


def test_the_disk_equiangulates_to_a_fan_above_the_pack_limit():
    pos, tri = disk_fan_start()
    rows, flips = equiangulate_triangles(pos, tri)
    assert flips == 30 and np.count_nonzero(rows == 0) == 60 > 48 and np.count_nonzero(tri == 0) == 30


def test_partitions_refuse_equiangulation():
    from membrane_solver_b200.runtime.device_minimizer import DeviceMinimizer
    from membrane_solver_b200.runtime.partitioned_minimizer import PartitionedDevice

    dev = PartitionedDevice(types.SimpleNamespace(dm=None, dist=None, torch=None))
    with pytest.raises(L.B200Error, match="single GPU only"):
        DeviceMinimizer(dm=dev, modules=L.MOD_SURFACE).equiangulate()


# ---- GPU tier: the C ABI, DeviceMesh and DeviceMinimizer ---------------------------------------------------------

@pytest.fixture(scope="module")
def gpu():
    if L.device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu tier must run on the B200 box")


def _device(pos, tri, *, fixed=None, hint=False, **kw):
    from membrane_solver_b200.context import DeviceMesh

    dm = DeviceMesh(0)
    dm.set_topology(len(pos), tri, fixed_mask=fixed, order_hint=pos if hint else None, **kw)
    dm.set_positions(pos)
    return dm


@pytest.mark.gpu
@pytest.mark.parametrize("hint", [False, True], ids=["caller-order", "morton-order"])
@pytest.mark.parametrize("name", MESHES)
def test_device_sweeps_match_the_twin(gpu, name, hint):
    pos, tri, fixed = _mesh(name)
    for it in ITERATIONS:
        want, flips, sweeps = twin(pos, tri, fixed, it)
        dm = _device(pos, tri, fixed=fixed, hint=hint)
        info = dm.pack_info()
        f = dm.equiangulate(it)
        assert (f, dm.last_equiangulate_sweeps) == (flips, sweeps), it
        assert np.array_equal(dm.triangles(), want), it
        assert np.array_equal(dm.download(L.ARR_POSITIONS).view(np.uint64), pos.view(np.uint64))
        if flips == 0:
            assert dm.pack_info() == info
        if it == 100:
            info = dm.pack_info()
            assert dm.equiangulate(100) == 0 and dm.pack_info() == info
            assert np.array_equal(dm.triangles(), want)
        dm.close()


@pytest.mark.gpu
def test_device_repeats_are_bitwise_and_rounds_are_reported(gpu):
    pos, tri, _ = _mesh("ellipse_fan")
    rows, stats = [], []
    for _ in range(3):
        dm = _device(pos, tri, hint=True)
        dm.equiangulate(100)
        rows.append(dm.triangles())
        stats.append(dm.equiangulate_stats())
        dm.close()
    assert all(np.array_equal(r, rows[0]) for r in rows)
    assert all(s["rounds"] == stats[0]["rounds"] for s in stats)
    print("ellipse fan rounds per sweep:", stats[0]["rounds"])
    assert stats[0]["rounds"][0] >= 16


def _eval(dm, body):
    mods = L.MOD_SURFACE | L.MOD_BENDING | (L.MOD_VOLUME if body is not None else 0)
    res = dm.eval(dm.options(mods, constraint_mode=0 if body is not None else -1, want_grad=True, apply_fixed=True))
    return res.scalars.copy(), dm.download(L.ARR_GRAD)


def _prepared(pos, tri, *, fixed, boundary, body, gamma, kappa, c0):
    dm = _device(pos, tri, fixed=fixed, hint=True, is_boundary=boundary, body_mask=body)
    dm.set_surface_tension(gamma)
    dm.set_bending_params(kappa, c0)
    return dm


@pytest.mark.gpu
def test_evaluation_after_equiangulation_equals_a_fresh_context(gpu):
    pos, tri = jittered_sphere(32, seed=1)
    nv, nf = len(pos), len(tri)
    rng = np.random.default_rng(11)
    kw = dict(fixed=(rng.uniform(size=nv) < 0.05).astype(np.uint8), boundary=(rng.uniform(size=nv) < 0.05).astype(np.uint8),
              body=(rng.uniform(size=nf) < 0.8).astype(np.uint8), gamma=rng.uniform(0.5, 1.5, size=nf),
              kappa=rng.uniform(0.5, 1.5, size=nv), c0=rng.uniform(-0.2, 0.2, size=nv))
    want_rows, _ = equiangulate_triangles(pos, tri, kw["fixed"].astype(bool))
    dm = _prepared(pos, tri, **kw)
    assert dm.equiangulate() > 0
    assert np.array_equal(dm.triangles(), want_rows)
    got = _eval(dm, kw["body"])
    fresh = _prepared(pos, want_rows, **kw)
    want = _eval(fresh, kw["body"])
    assert dm.pack_info() == fresh.pack_info()
    assert np.array_equal(got[0].view(np.uint64), want[0].view(np.uint64))
    assert np.array_equal(got[1].view(np.uint64), want[1].view(np.uint64))
    dm.close()
    fresh.close()


@pytest.mark.gpu
def test_device_refusals(gpu):
    from membrane_solver_b200.context import DeviceMesh

    pos, tri, _ = _mesh("sheet")
    dm = DeviceMesh(0)
    dm.set_topology(len(pos), tri)
    with pytest.raises(L.B200Error, match="no positions"):
        dm.equiangulate()
    dm.set_positions(pos)
    with pytest.raises(L.B200Error, match="max_iterations"):
        dm.equiangulate(-1)
    dm.set_topology(len(pos), tri, n_owned=len(pos) - 5)
    dm.set_positions(pos)
    with pytest.raises(L.B200Error, match="partitioned"):
        dm.equiangulate()
    bad = tri.copy()
    bad[3, 1] = len(pos)
    dm.set_topology(len(pos), bad)
    dm.set_positions(pos)
    with pytest.raises(L.B200Error, match="outside"):
        dm.equiangulate()
    assert np.array_equal(dm.triangles(), bad)
    dm.close()


@pytest.mark.gpu
def test_leaflet_selection_must_be_set_again_after_a_flip(gpu):
    pos, tri, _ = _mesh("sheet")
    dm = _device(pos, tri)
    dm.set_tilts(np.zeros_like(pos))
    dm.upload(L.ARR_TILTS_IN, 0.01 * np.ones_like(pos))
    dm.set_leaflet(0, div_sign=1.0, kappa=1.0, k_tilt=1.0)
    before = dm.eval_leaflet(0, L.MOD_TILT | L.MOD_BENDING_TILT)
    assert dm.equiangulate() > 0
    with pytest.raises(L.B200Error, match="set_leaflet"):
        dm.eval_leaflet(0, L.MOD_TILT | L.MOD_BENDING_TILT)
    dm.set_leaflet(0, div_sign=1.0, kappa=1.0, k_tilt=1.0)
    after = dm.eval_leaflet(0, L.MOD_TILT | L.MOD_BENDING_TILT)
    assert np.all(np.isfinite(before)) and np.all(np.isfinite(after))
    dm.close()


@pytest.mark.gpu
def test_a_flip_result_that_does_not_pack_leaves_the_context_as_it_was(gpu):
    pos, tri = disk_fan_start()
    dm = _device(pos, tri, hint=True)
    dm.set_surface_tension(np.linspace(0.5, 1.5, len(tri)))
    dm.set_bending_params(1.0, 0.0)
    info = dm.pack_info()
    before = _eval(dm, None)
    with pytest.raises(L.B200Error, match="48"):
        dm.equiangulate()
    assert np.array_equal(dm.triangles(), tri) and dm.pack_info() == info
    after = _eval(dm, None)
    assert np.array_equal(after[0].view(np.uint64), before[0].view(np.uint64))
    assert np.array_equal(after[1].view(np.uint64), before[1].view(np.uint64))
    dm.close()


@pytest.mark.gpu
def test_bending_cube_replay_with_device_u_equals_the_twin(gpu):
    """``r, u, g 50, r, u, g 100, V`` of the bending cube (``replay.npz``, from its state after the first ``r``), once
    with ``DeviceMinimizer.equiangulate`` and once with the twin + ``set_topology``: energies and positions agree to
    1e-12 after every instruction."""
    from membrane_solver_b200.context import DeviceMesh
    from membrane_solver_b200.geometry.refine import refine_triangles
    from membrane_solver_b200.runtime.device_minimizer import DeviceMinimizer

    gold = np.load(os.path.join(H.GOLDEN, "replay.npz"))
    prm = json.loads(str(gold["bcube_params_json"]))
    a = "bcube_00_"
    pos0, tri0, fixed0 = gold[a + "pos"], gold[a + "tri"], np.asarray(gold[a + "fixed"], bool)
    body0 = np.zeros(len(tri0), np.uint8)
    body0[gold[a + "body_rows_0"]] = 1
    target = float(gold[a + "body_target_0"])
    kappa = float(prm["bending_modulus"])
    instructions = [str(gold[f"bcube_{k:02d}_instruction"]).replace(" ", "") for k in range(1, int(gold["bcube_count"]))]
    assert instructions == ["u", "g50", "r", "u", "g100", "V"]

    def run(device_u):
        dm = DeviceMesh(0)
        # hint: the positions that chose the internal vertex order; the twin's path keeps it across its set_topology,
        # so both paths evaluate with the same packing and must agree bit for bit
        state = dict(pos=pos0, tri=tri0, fixed=fixed0, body=body0, hint=pos0)

        def load(pos, tri, fixed, body, hint):
            dm.set_topology(len(pos), tri, fixed_mask=fixed.astype(np.uint8) if fixed.any() else None, body_mask=body,
                            order_hint=hint)
            dm.set_positions(pos)
            dm.set_surface_tension(float(prm["surface_tension"]))
            dm.set_bending_params(kappa, float(prm["spontaneous_curvature"]))
            return DeviceMinimizer(dm, L.MOD_BENDING, volume_mode="lagrange", v_target=target, enforce_volume=True)

        mz = load(**state)
        trace = []
        for ins in instructions:
            pos = dm.download(L.ARR_POSITIONS)
            if ins == "u":
                if device_u:
                    mz.equiangulate()
                    state["tri"] = dm.triangles()
                else:
                    state["tri"], _ = equiangulate_triangles(pos, state["tri"], state["fixed"])
                    step, mz = mz.step_size, load(pos, state["tri"], state["fixed"], state["body"], state["hint"])
                    mz.step_size = step
                    mz._enforce(trial=False, max_iter=12)
            elif ins == "r":
                p, t, f, parent = refine_triangles(pos, state["tri"], state["fixed"])
                step = mz.step_size
                state.update(pos=p, tri=t, fixed=np.asarray(f, bool), body=state["body"][parent], hint=p)
                mz = load(**state)
                mz.step_size = step
            elif ins[0] == "g":
                mz.minimize(n_steps=int(ins[1:]))
            elif ins == "V":
                mz.vertex_average(1)
            trace.append((mz.energy(), dm.download(L.ARR_POSITIONS), dm.triangles()))
        dm.close()
        return trace

    dev, host = run(True), run(False)
    for ins, (e1, p1, t1), (e2, p2, t2) in zip(instructions, dev, host):
        assert np.array_equal(t1, t2), ins
        assert abs(e1 - e2) <= 1e-12 * max(1.0, abs(e2)), (ins, e1, e2)
        assert np.max(np.abs(p1 - p2)) <= 1e-12, ins


@pytest.mark.gpu
def test_device_equiangulation_at_size(gpu):
    """About 1 M facets (icosphere frequency 224, tangential jitter): the rows equal the twin's."""
    pos, tri = jittered_sphere(224)
    assert len(tri) == 1_003_520
    want, flips = equiangulate_triangles(pos, tri)
    dm = _device(pos, tri, hint=True)
    assert dm.equiangulate() == flips
    assert np.array_equal(dm.triangles(), want)
    dm.close()
