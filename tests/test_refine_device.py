"""Refinement (the ``r`` command) on the device: ``ms_refine.cuh`` through the host emulator in the CPU tier,
``ms_ctx_refine`` / ``DeviceMesh.refine`` / ``DeviceMinimizer.refine`` in the GPU tier, against the host twin
``geometry.refine.refine_triangles``: the same rows, positions (bitwise), fixed and boundary flags, and a context
indistinguishable from one set up from the twin's output."""

import ctypes
import json
import os
import subprocess
import types

import numpy as np
import pytest

import ms_test_helpers as H

from membrane_solver_b200 import _lib as L
from membrane_solver_b200.geometry.array_mesh import ArrayMesh
from membrane_solver_b200.geometry.refine import cube_mesh, refine_triangles
from membrane_solver_b200.synthetic import icosphere, open_sheet


# ---- meshes ------------------------------------------------------------------------------------------------------

def jittered_sphere(freq, seed=0):
    """Icosphere with tangential noise of 0.3 x the mean edge length, back on the unit sphere."""
    pos, tri = icosphere(freq, perturb=False)
    rng = np.random.default_rng(seed)
    h = np.mean(np.linalg.norm(pos[tri[:, 1]] - pos[tri[:, 0]], axis=1))
    q = pos + 0.3 * h * rng.normal(size=pos.shape)
    return q / np.linalg.norm(q, axis=1)[:, None], tri


def topological_boundary(pos, tri):
    mask = np.zeros(len(pos), bool)
    mask[sorted(ArrayMesh(pos, tri).boundary_vertex_ids)] = True
    return mask


def _mesh(name):
    """(pos, tri, fixed or None, boundary or None)"""
    if name == "cube":
        return (*cube_mesh(), None, None)
    if name == "catenoid":
        g = np.load(os.path.join(H.GOLDEN, "equiangulate.npz"))
        pos, tri = g["pos"], g["tri"]
        return pos, tri, np.asarray(g["fixed"], bool), topological_boundary(pos, tri)
    if name == "fixed_sphere":
        pos, tri = jittered_sphere(12, seed=4)
        return pos, tri, np.random.default_rng(4).uniform(size=len(pos)) < 0.3, None
    if name.startswith("odd"):
        pos, tri = H.odd_mesh(int(name[-1]), nfan=30)[:2]
        fixed = np.random.default_rng(int(name[-1])).uniform(size=len(pos)) < 0.2
        return pos, tri, fixed, topological_boundary(pos, tri)
    if name == "sheet":
        pos, tri = open_sheet(14, 11, jitter=0.2)
        pos[:, 2] = 0.0
        return pos, tri, None, topological_boundary(pos, tri)
    raise KeyError(name)


CASES = [("cube", 1), ("cube", 2), ("cube", 3), ("catenoid", 1), ("catenoid", 2), ("fixed_sphere", 1),
         ("fixed_sphere", 2), ("odd1", 1), ("odd2", 2), ("sheet", 1), ("sheet", 2)]
CASE_IDS = [f"{n}-{k}" for n, k in CASES]


def twin(pos, tri, fixed, boundary, levels):
    """``refine_triangles`` ``levels`` times; the boundary rule of ``ms_ctx_refine`` restated: a midpoint is a
    boundary vertex when its edge has one half-edge and both ends are.  Returns (pos, tri, fixed, boundary, parent)."""
    p, t, f, b = pos, np.asarray(tri, np.int32), fixed, boundary
    parent = np.arange(len(t))
    for _ in range(levels):
        nv = len(p)
        e = np.stack([t[:, [0, 1]], t[:, [1, 2]], t[:, [2, 0]]], axis=1).reshape(-1, 2).astype(np.int64)
        uniq, counts = np.unique(e.min(axis=1) * nv + e.max(axis=1), return_counts=True)
        if b is not None:
            b = np.concatenate([b, (counts == 1) & b[uniq // nv] & b[uniq % nv]])
        p, t, f, par = refine_triangles(p, t, f)
        parent = parent[par]
    return p, t, f, b, parent


# ---- CPU tier: the per-element bodies, compiled for the host ------------------------------------------------------

@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    """tests/emul/refine_emul.cpp compiled for the host into a temporary directory (the tree may be read-only).  No
    fp contraction: the host side rounds every operation, as the twin does."""
    out = str(tmp_path_factory.mktemp("rf_emul") / "libms_rf_emul.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-o", out,
                           os.path.join(H.ROOT, "tests", "emul", "refine_emul.cpp")])
    lib = ctypes.CDLL(out)
    lib.emul_refine.restype = ctypes.c_int
    return lib


def emulate(lib, pos, tri, fixed, boundary, levels, key_id=None):
    """(pos, tri, fixed or None, boundary or None) of the refined mesh, in the caller's numbering"""
    nv, nf = len(pos), len(tri)
    nv_cap = nv + nf * (4 ** levels - 1)   # >= nv + sum over levels of 3 nf_l
    out_pos = np.zeros((nv_cap, 3))
    out_tri = np.zeros((nf * 4 ** levels, 3), np.int32)
    out_fx, out_bd = np.zeros(nv_cap, np.uint8), np.zeros(nv_cap, np.uint8)
    fx = None if fixed is None else np.ascontiguousarray(fixed, np.uint8)
    bd = None if boundary is None else np.ascontiguousarray(boundary, np.uint8)
    kid = None if key_id is None else np.ascontiguousarray(key_id, np.int32)
    nv_out = ctypes.c_int32(0)
    rows = np.ascontiguousarray(tri, np.int32)
    rc = lib.emul_refine(ctypes.c_int32(nv), ctypes.c_int32(nf), L.iptr(rows),
                         L.dptr(np.ascontiguousarray(pos, np.float64)), L.bptr(fx), L.bptr(bd), L.iptr(kid),
                         ctypes.c_int32(levels), L.dptr(out_pos), L.iptr(out_tri), L.bptr(out_fx), L.bptr(out_bd),
                         ctypes.byref(nv_out))
    assert rc == 0
    n = nv_out.value
    return (out_pos[:n], out_tri, None if fixed is None else out_fx[:n].astype(bool),
            None if boundary is None else out_bd[:n].astype(bool))


def assert_same(got, want):
    p, t, f, b = got
    assert p.shape == want[0].shape and np.array_equal(p.view(np.uint64), want[0].view(np.uint64))
    assert np.array_equal(t, want[1])
    assert (f is None) == (want[2] is None) and (f is None or np.array_equal(f, want[2]))
    assert (b is None) == (want[3] is None) and (b is None or np.array_equal(b, want[3]))


@pytest.mark.parametrize("name,levels", CASES, ids=CASE_IDS)
def test_emulated_refinement_matches_the_twin(emul, name, levels):
    pos, tri, fixed, boundary = _mesh(name)
    want = twin(pos, tri, fixed, boundary, levels)
    assert_same(emulate(emul, pos, tri, fixed, boundary, levels), want)


@pytest.mark.parametrize("levels", [1, 2])
def test_midpoint_boundary_flags_are_the_refined_topological_boundary(levels):
    """For flags derived from the topology the boundary rule is ``boundary_vertex_ids`` of the refined mesh."""
    for name in ("catenoid", "sheet"):
        pos, tri, fixed, boundary = _mesh(name)
        p, t, _, b, _ = twin(pos, tri, fixed, boundary, levels)
        assert b.any() and np.array_equal(b, topological_boundary(p, t)), name


@pytest.mark.parametrize("name,levels", [("cube", 2), ("catenoid", 1), ("fixed_sphere", 1), ("odd1", 2),
                                         ("sheet", 1)])
def test_emulated_refinement_in_a_permuted_vertex_order(emul, name, levels):
    """Rows held in another vertex numbering (as the device's Morton order) with keys and the result taken in the
    caller's: the twin's mesh."""
    pos, tri, fixed, boundary = _mesh(name)
    perm = np.random.default_rng(9).permutation(len(pos)).astype(np.int32)   # internal -> caller
    inv = np.empty_like(perm)
    inv[perm] = np.arange(len(pos), dtype=np.int32)
    got = emulate(emul, pos[perm], inv[tri], None if fixed is None else fixed[perm],
                  None if boundary is None else boundary[perm], levels, key_id=perm)
    assert_same(got, twin(pos, tri, fixed, boundary, levels))


def test_partitions_refuse_refinement():
    from membrane_solver_b200.runtime.device_minimizer import DeviceMinimizer
    from membrane_solver_b200.runtime.partitioned_minimizer import PartitionedDevice

    dev = PartitionedDevice(types.SimpleNamespace(dm=None, dist=None, torch=None))
    with pytest.raises(L.B200Error, match="single GPU only"):
        DeviceMinimizer(dm=dev, modules=L.MOD_SURFACE).refine()


# ---- GPU tier: the C ABI, DeviceMesh and DeviceMinimizer ---------------------------------------------------------

@pytest.fixture(scope="module")
def gpu():
    if L.device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu tier must run on the B200 box")


def _u8(a):
    return None if a is None else np.asarray(a, np.uint8)


def _device(pos, tri, *, fixed=None, boundary=None, body=None, hint=False):
    from membrane_solver_b200.context import DeviceMesh

    dm = DeviceMesh(0)
    dm.set_topology(len(pos), tri, fixed_mask=_u8(fixed), is_boundary=_u8(boundary), body_mask=_u8(body),
                    order_hint=pos if hint else None)
    dm.set_positions(pos)
    return dm


def _eval(dm, body=None):
    """Scalars, gradient and dV/dx of a surface + bending (+ volume) evaluation with the fixed rows zeroed."""
    mods = L.MOD_SURFACE | L.MOD_BENDING | (L.MOD_VOLUME if body is not None else 0)
    res = dm.eval(dm.options(mods, constraint_mode=0 if body is not None else -1, want_grad=True, apply_fixed=True))
    return res.scalars.copy(), dm.download(L.ARR_GRAD), dm.download(L.ARR_VOLGRAD)


def _bitwise(a, b):
    return all(np.array_equal(np.asarray(x).view(np.uint64), np.asarray(y).view(np.uint64)) for x, y in zip(a, b))


@pytest.mark.gpu
@pytest.mark.parametrize("hint", [False, True], ids=["caller-order", "morton-order"])
@pytest.mark.parametrize("name,levels", CASES, ids=CASE_IDS)
def test_device_refinement_matches_the_twin(gpu, name, levels, hint):
    """Rows and positions bitwise; the fixed and boundary flags through an evaluation bitwise equal to a fresh context
    set up from the twin's output with the refined positions as order hint (same order, same packing)."""
    pos, tri, fixed, boundary = _mesh(name)
    p2, t2, f2, b2, parent = twin(pos, tri, fixed, boundary, levels)
    dm = _device(pos, tri, fixed=fixed, boundary=boundary, hint=hint)
    dm.set_bending_params(1.0, 0.1)
    got_parent = dm.refine(levels)
    assert (dm.nv, dm.nf) == (len(p2), len(t2)) and np.array_equal(got_parent, parent)
    assert np.array_equal(dm.triangles(), t2)
    assert np.array_equal(dm.download(L.ARR_POSITIONS).view(np.uint64), p2.view(np.uint64))
    fresh = _device(p2, t2, fixed=f2, boundary=b2, hint=True)
    fresh.set_bending_params(1.0, 0.1)
    assert np.array_equal(dm.permutation(), fresh.permutation())
    assert dm.pack_info() == fresh.pack_info()
    got, want = _eval(dm), _eval(fresh)
    assert _bitwise(got, want)
    if f2 is not None:
        assert np.all(got[1][f2] == 0)
    dm.close()
    fresh.close()


@pytest.mark.gpu
def test_device_repeats_are_bitwise_and_times_are_reported(gpu):
    pos, tri, fixed, boundary = _mesh("odd2")
    out = []
    for _ in range(2):
        dm = _device(pos, tri, fixed=fixed, boundary=boundary, hint=True)
        dm.refine(2)
        out.append((dm.triangles(), dm.download(L.ARR_POSITIONS), dm.permutation(), _eval(dm)))
        stats = dm.refine_stats()
        dm.close()
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][2], out[1][2])
    assert _bitwise([out[0][1]], [out[1][1]]) and _bitwise(out[0][3], out[1][3])
    assert set(stats) == {"device_ms", "d2h_ms", "pack_ms", "upload_ms"} and stats["device_ms"] > 0


def _prepared(pos, tri, *, fixed, boundary, body, gamma, hint):
    dm = _device(pos, tri, fixed=fixed, boundary=boundary, body=body, hint=hint)
    dm.set_surface_tension(gamma)
    dm.set_bending_params(1.3, -0.2)
    return dm


@pytest.mark.gpu
@pytest.mark.parametrize("levels", [1, 2])
def test_evaluation_after_refinement_equals_a_fresh_context(gpu, levels):
    """Per-facet surface tension, uniform kappa / c0, a body mask, fixed and boundary flags survive, expanded to the
    refined mesh: packing and evaluation (scalars, gradient, dV/dx) equal a fresh context's, bitwise."""
    pos, tri = jittered_sphere(16, seed=1)
    nv, nf = len(pos), len(tri)
    rng = np.random.default_rng(11)
    fixed, boundary = rng.uniform(size=nv) < 0.05, rng.uniform(size=nv) < 0.1
    body, gamma = rng.uniform(size=nf) < 0.8, rng.uniform(0.5, 1.5, size=nf)
    p2, t2, f2, b2, parent = twin(pos, tri, fixed, boundary, levels)
    dm = _prepared(pos, tri, fixed=fixed, boundary=boundary, body=body, gamma=gamma, hint=False)
    _eval(dm, body)
    dm.direction_from_gradient()
    dm.make_trial(1e-3)   # trial positions and a direction of the old size are dropped
    assert np.array_equal(dm.refine(levels), parent)
    fresh = _prepared(p2, t2, fixed=f2, boundary=b2, body=body[parent], gamma=gamma[parent], hint=True)
    assert dm.pack_info() == fresh.pack_info()
    assert _bitwise(_eval(dm, body[parent]), _eval(fresh, body[parent]))
    with pytest.raises(L.B200Error, match="trial"):
        dm.eval(dm.options(L.MOD_SURFACE, want_grad=False, use_trial=True))
    dm.close()
    fresh.close()


@pytest.mark.gpu
def test_refusals_leave_the_context_as_it_was(gpu):
    from membrane_solver_b200.context import DeviceMesh

    pos, tri, fixed, boundary = _mesh("sheet")
    dm = DeviceMesh(0)
    with pytest.raises(L.B200Error, match="set_topology"):
        dm.refine()
    dm.set_topology(len(pos), tri)
    with pytest.raises(L.B200Error, match="no positions"):
        dm.refine()
    dm.set_topology(len(pos), tri, n_owned=len(pos) - 5)
    dm.set_positions(pos)
    with pytest.raises(L.B200Error, match="partitioned"):
        dm.refine()
    dm.close()

    dm = _device(pos, tri, fixed=fixed, boundary=boundary, hint=True)
    dm.set_surface_tension(np.linspace(0.5, 1.5, len(tri)))
    dm.set_bending_params(1.0, 0.1)
    state = lambda: (dm.triangles(), dm.pack_info(), dm.nv, dm.nf, _eval(dm))     # noqa: E731

    def refused(match, levels=1):
        before = state()
        with pytest.raises(L.B200Error, match=match):
            dm.refine(levels)
        now = state()
        assert np.array_equal(now[0], before[0]) and now[1:4] == before[1:4] and _bitwise(now[4], before[4])

    before = state()
    dm.refine(0)
    now = state()
    assert np.array_equal(now[0], before[0]) and now[1:4] == before[1:4] and _bitwise(now[4], before[4])
    refused("levels", -1)
    refused("2\\^31", 16)                                  # 308 x 4^15 facets: refused before any allocation
    dm.set_bending_params(np.linspace(0.5, 1.5, len(pos)), 0.1)
    refused("kappa")
    dm.set_bending_params(1.0, np.linspace(-0.1, 0.1, len(pos)))
    refused("refine_triangles")
    dm.set_bending_params(1.0, 0.1)
    dm.set_tilts(np.zeros_like(pos))
    refused("tilt")
    bad = tri.copy()
    bad[3, 1] = len(pos)
    dm.set_topology(len(pos), bad)
    dm.set_positions(pos)
    with pytest.raises(L.B200Error, match="outside"):
        dm.refine()
    assert np.array_equal(dm.triangles(), bad)
    dm.close()


@pytest.mark.gpu
def test_leaflet_selection_must_be_set_again_after_refinement(gpu):
    pos, tri, _, _ = _mesh("sheet")
    dm = _device(pos, tri)
    dm.set_leaflet(0, div_sign=1.0, kappa=1.0, k_tilt=1.0)
    dm.refine()
    dm.set_tilts(np.zeros((dm.nv, 3)))
    dm.upload(L.ARR_TILTS_IN, 0.01 * np.ones((dm.nv, 3)))
    with pytest.raises(L.B200Error, match="set_leaflet"):
        dm.eval_leaflet(0, L.MOD_TILT | L.MOD_BENDING_TILT)
    dm.set_leaflet(0, div_sign=1.0, kappa=1.0, k_tilt=1.0)
    assert np.all(np.isfinite(dm.eval_leaflet(0, L.MOD_TILT | L.MOD_BENDING_TILT)))
    dm.close()


@pytest.mark.gpu
def test_bending_cube_gogo_with_every_mesh_operation_on_the_device(gpu):
    """``gogo`` of ``meshes/bending_cube.yaml`` (``r, u, g 50, r, u, g 100, V``) from ``cube_mesh()``, once with
    ``DeviceMinimizer.refine`` and once with the twin + ``set_topology(order_hint=...)``, both with device ``u`` and
    ``V``: rows equal, energies and positions within 1e-12 after every instruction.  After the first ``r`` the vertex
    set is the reference's (``replay.npz`` ``bcube_00``)."""
    from membrane_solver_b200.context import DeviceMesh
    from membrane_solver_b200.runtime.device_minimizer import DeviceMinimizer

    gold = np.load(os.path.join(H.GOLDEN, "replay.npz"))
    prm = json.loads(str(gold["bcube_params_json"]))
    target = float(gold["bcube_00_body_target_0"])
    instructions = [str(gold[f"bcube_{k:02d}_instruction"]).replace(" ", "") for k in range(int(gold["bcube_count"]))]
    assert instructions == ["r", "u", "g50", "r", "u", "g100", "V"]
    pos0, tri0 = cube_mesh()

    def run(device_r):
        dm = DeviceMesh(0)

        def load(pos, tri, body):
            dm.set_topology(len(pos), tri, body_mask=body, order_hint=pos)
            dm.set_positions(pos)
            dm.set_surface_tension(float(prm["surface_tension"]))
            dm.set_bending_params(float(prm["bending_modulus"]), float(prm["spontaneous_curvature"]))
            return DeviceMinimizer(dm, L.MOD_BENDING, volume_mode="lagrange", v_target=target, enforce_volume=True)

        body = np.ones(len(tri0), np.uint8)
        mz = load(pos0, tri0, body)
        trace = []
        for ins in instructions:
            if ins == "r":
                if device_r:
                    body = body[mz.refine()]
                else:
                    p, t, _, parent = refine_triangles(dm.download(L.ARR_POSITIONS), dm.triangles())
                    step, body = mz.step_size, body[parent]
                    mz = load(p, t, body)
                    mz.step_size = step
            elif ins == "u":
                mz.equiangulate()
            elif ins[0] == "g":
                mz.minimize(n_steps=int(ins[1:]))
            elif ins == "V":
                mz.vertex_average(1)
            trace.append((mz.energy(), dm.download(L.ARR_POSITIONS), dm.triangles()))
        dm.close()
        return trace

    dev, host = run(True), run(False)
    want = gold["bcube_00_pos"]
    key = lambda x: x[np.lexsort(np.round(x, 9).T[::-1])]                            # noqa: E731
    assert dev[0][1].shape == want.shape and np.max(np.abs(key(dev[0][1]) - key(want))) <= 1e-12
    for ins, (e1, p1, t1), (e2, p2, t2) in zip(instructions, dev, host):
        assert np.array_equal(t1, t2), ins
        assert abs(e1 - e2) <= 1e-12 * max(1.0, abs(e2)), (ins, e1, e2)
        assert np.max(np.abs(p1 - p2)) <= 1e-12, ins


@pytest.mark.gpu
def test_device_refinement_at_size(gpu):
    """About 1 M facets (icosphere frequency 224, tangential jitter) refined once: rows and positions equal the
    twin's."""
    pos, tri = jittered_sphere(224)
    assert len(tri) == 1_003_520
    p2, t2, _, _ = refine_triangles(pos, tri)
    dm = _device(pos, tri, hint=True)
    dm.refine()
    assert np.array_equal(dm.triangles(), t2)
    assert np.array_equal(dm.download(L.ARR_POSITIONS).view(np.uint64), p2.view(np.uint64))
    dm.close()
