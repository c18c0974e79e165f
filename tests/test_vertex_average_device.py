"""Vertex averaging (the ``V`` command) on the device: ``ms_vertex_average.cuh`` through the host emulator in the CPU
tier, ``ms_ctx_vertex_average`` / ``DeviceMesh.vertex_average`` / ``DeviceMinimizer.vertex_average`` in the GPU tier,
against the host twin ``geometry.vertex_average.vertex_average_arrays`` and the reference's golden vectors."""

import ctypes
import json
import os
import subprocess
import types

import numpy as np
import pytest

import ms_test_helpers as H

from membrane_solver_b200 import _lib as L
from membrane_solver_b200.geometry.vertex_average import vertex_average_arrays

TOL = 1e-13
SEEDS = [1, 2, 3]


def _golden():
    return np.load(os.path.join(H.GOLDEN, "vertex_average.npz"))


def _odd(seed):
    """odd_mesh with a valence-30 fan (unused vertices, repeated-index and duplicated facets, two components), a
    random fixed set and pin groups on a few vertices."""
    pos, tri, _, _, _ = H.odd_mesh(seed, nfan=30)
    rng = np.random.default_rng(100 + seed)
    fixed = rng.uniform(size=len(pos)) < 0.1
    group = np.full(len(pos), -1, np.int32)
    group[rng.choice(len(pos), size=len(pos) // 5, replace=False)] = rng.integers(0, 3, size=len(pos) // 5)
    return pos, tri, fixed, group


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    """tests/emul/vertex_average_emul.cpp with the packer's CSR builder, compiled for the host into a temporary
    directory (the tree may be read-only)."""
    csrc = os.path.join(H.ROOT, "membrane_solver_b200", "csrc")
    out = str(tmp_path_factory.mktemp("va_emul") / "libms_va_emul.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-fPIC", "-shared", "-o", out,
                           os.path.join(H.ROOT, "tests", "emul", "vertex_average_emul.cpp"),
                           os.path.join(csrc, "ms_pack.cpp")])
    lib = ctypes.CDLL(out)
    lib.emul_vertex_average.restype = ctypes.c_int
    return lib


def _emulate(lib, pos, tri, *, fixed=None, group=None, rounds=1):
    out = np.array(pos, dtype=np.float64, order="C", copy=True)
    tri = np.ascontiguousarray(tri, dtype=np.int32)
    fx = None if fixed is None else np.ascontiguousarray(fixed, dtype=np.uint8)
    gr = None if group is None else np.ascontiguousarray(group, dtype=np.int32)
    rc = lib.emul_vertex_average(ctypes.c_int32(len(out)), ctypes.c_int32(len(tri)), L.iptr(tri), L.bptr(fx),
                                 L.iptr(gr), ctypes.c_int32(rounds), L.dptr(out))
    assert rc == 0
    return out


def _twin(pos, tri, *, fixed=None, group=None, rounds=1):
    for _ in range(rounds):
        pos = vertex_average_arrays(pos, tri, movable=None if fixed is None else ~np.asarray(fixed, bool), group=group)
    return pos


# ---- CPU tier: the per-vertex body, compiled for the host --------------------------------------------------------

@pytest.mark.parametrize("name", ["cube", "catenoid"])
def test_emulated_averaging_matches_the_reference_golden(emul, name):
    g = _golden()
    pos0, tri, fixed = g[name + "_pos0"], g[name + "_tri"], g[name + "_fixed"]
    out = _emulate(emul, pos0, tri, fixed=fixed)
    assert np.max(np.abs(out - g[name + "_pos1"])) <= TOL
    assert np.array_equal(out[fixed].view(np.uint64), pos0[fixed].view(np.uint64))


def test_emulated_pin_groups_match_the_twin(emul):
    g = _golden()
    pos0, tri = g["cube_pos0"], g["cube_tri"]
    group = np.full(len(pos0), -1, np.int32)
    group[:5] = 0
    out = _emulate(emul, pos0, tri, group=group)
    assert np.max(np.abs(out - _twin(pos0, tri, group=group))) <= TOL
    assert not np.allclose(out[:5], g["cube_pos1"][:5])


@pytest.mark.parametrize("seed", SEEDS)
def test_emulated_odd_meshes_match_the_twin(emul, seed):
    pos, tri, fixed, group = _odd(seed)
    assert np.bincount(tri.ravel()).max() >= 30
    for kw in (dict(), dict(fixed=fixed), dict(fixed=fixed, group=group)):
        out = _emulate(emul, pos, tri, rounds=2, **kw)
        assert np.max(np.abs(out - _twin(pos, tri, rounds=2, **kw))) <= TOL, kw


def test_partitions_refuse_vertex_averaging():
    from membrane_solver_b200.runtime.device_minimizer import DeviceMinimizer
    from membrane_solver_b200.runtime.partitioned_minimizer import PartitionedDevice

    dev = PartitionedDevice(types.SimpleNamespace(dm=None, dist=None, torch=None))
    with pytest.raises(L.B200Error, match="single GPU only"):
        DeviceMinimizer(dm=dev, modules=L.MOD_SURFACE).vertex_average(1)


# ---- GPU tier: the C ABI, DeviceMesh and DeviceMinimizer ---------------------------------------------------------

@pytest.fixture(scope="module")
def gpu():
    if L.device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu tier must run on the B200 box")


def _device(pos, tri, *, fixed=None, hint=False, body=None):
    from membrane_solver_b200.context import DeviceMesh

    dm = DeviceMesh(0)
    dm.set_topology(len(pos), tri, fixed_mask=fixed, body_mask=body, order_hint=pos if hint else None)
    dm.set_positions(pos)
    return dm


def _on_device(pos, tri, *, fixed=None, group=None, rounds=1, hint=False):
    dm = _device(pos, tri, fixed=fixed, hint=hint)
    dm.vertex_average(rounds, group=group)
    out = dm.download(L.ARR_POSITIONS)
    dm.close()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("hint", [False, True], ids=["caller-order", "morton-order"])
@pytest.mark.parametrize("name", ["cube", "catenoid"])
def test_device_averaging_matches_the_reference_golden(gpu, name, hint):
    g = _golden()
    pos0, tri, fixed = g[name + "_pos0"], g[name + "_tri"], g[name + "_fixed"]
    out = _on_device(pos0, tri, fixed=fixed, hint=hint)
    assert np.max(np.abs(out - g[name + "_pos1"])) <= TOL
    assert np.array_equal(out[fixed].view(np.uint64), pos0[fixed].view(np.uint64))
    group = np.full(len(pos0), -1, np.int32)
    group[:5] = 0
    out = _on_device(pos0, tri, group=group, hint=hint)
    assert np.max(np.abs(out - _twin(pos0, tri, group=group))) <= TOL


@pytest.mark.gpu
@pytest.mark.parametrize("seed", SEEDS)
def test_device_odd_meshes_match_the_twin(gpu, seed):
    pos, tri, fixed, group = _odd(seed)
    for hint in (False, True):
        for kw in (dict(), dict(fixed=fixed, group=group)):
            out = _on_device(pos, tri, hint=hint, **kw)
            assert np.max(np.abs(out - _twin(pos, tri, **kw))) <= TOL, (hint, kw)


@pytest.mark.gpu
def test_device_rounds_and_repeats_are_bitwise(gpu):
    pos, tri, fixed, group = _odd(1)
    dm = _device(pos, tri, fixed=fixed, hint=True)
    dm.vertex_average(2, group=group)
    two = dm.download(L.ARR_POSITIONS)
    dm.set_positions(pos)
    dm.vertex_average(1, group=group)
    dm.vertex_average(1, group=group)
    assert np.array_equal(dm.download(L.ARR_POSITIONS).view(np.uint64), two.view(np.uint64))
    dm.set_positions(pos)
    dm.vertex_average(2, group=group)
    assert np.array_equal(dm.download(L.ARR_POSITIONS).view(np.uint64), two.view(np.uint64))
    dm.set_positions(pos)
    dm.vertex_average(0)
    assert np.array_equal(dm.download(L.ARR_POSITIONS), pos)
    with pytest.raises(L.B200Error):
        dm.vertex_average(-1)
    dm.close()


@pytest.mark.gpu
def test_device_refusals(gpu):
    from membrane_solver_b200.context import DeviceMesh

    pos, tri, _, _ = _odd(2)
    dm = DeviceMesh(0)
    dm.set_topology(len(pos), tri)
    with pytest.raises(L.B200Error, match="no positions"):
        dm.vertex_average(1)
    dm.set_topology(len(pos), tri, n_owned=len(pos) - 5)
    dm.set_positions(pos)
    with pytest.raises(L.B200Error, match="partitioned"):
        dm.vertex_average(1)
    dm.close()


@pytest.mark.gpu
def test_device_replay_of_the_V_instructions(gpu):
    """Every ``V``/``Vn`` of the cube and bending-cube lists (``replay.npz``), applied with
    ``DeviceMinimizer.vertex_average`` (hard volume projection as stored) to the reference's state before it, lands on
    the reference's state after it -- the tolerance of test_mesh_operations_of_the_instruction_lists_on_arrays.  The
    catenoid's ``V`` stays out: its rims are pinned by pin_to_circle, which is not on the path."""
    from membrane_solver_b200.runtime.device_minimizer import DeviceMinimizer

    gold = np.load(os.path.join(H.GOLDEN, "replay.npz"))
    checked = 0
    for name in ("cube", "bcube"):
        prm = json.loads(str(gold[f"{name}_params_json"]))
        for k in range(1, int(gold[f"{name}_count"])):
            ins = str(gold[f"{name}_{k:02d}_instruction"]).replace(" ", "")
            cons = [str(x) for x in gold[f"{name}_{k:02d}_constraints"]]
            if ins[0] != "V" or cons not in ([], ["volume"]):
                continue
            a, b = f"{name}_{k - 1:02d}_", f"{name}_{k:02d}_"
            pos, tri, fixed = gold[a + "pos"], gold[a + "tri"], np.asarray(gold[a + "fixed"], bool)
            body = None
            if cons == ["volume"]:
                assert prm.get("volume_constraint_mode", "lagrange") in ("lagrange", "projection")
                body = np.zeros(len(tri), np.uint8)
                body[gold[a + "body_rows_0"]] = 1
            dm = _device(pos, tri, fixed=fixed, body=body, hint=True)
            mz = DeviceMinimizer(dm=dm, modules=L.MOD_SURFACE, enforce_volume=cons == ["volume"],
                                 v_target=float(gold[a + "body_target_0"]) if body is not None else 0.0)
            mz.vertex_average(int(ins[1:] or 1))
            out = dm.download(L.ARR_POSITIONS)
            dm.close()
            assert np.max(np.abs(out - gold[b + "pos"])) <= 1e-12, (name, k, ins)
            checked += 1
    assert checked >= 5


@pytest.mark.gpu
def test_device_averaging_at_size(gpu):
    """10 M facets (synthetic.icosphere(708)): the device result against the host twin."""
    from membrane_solver_b200.synthetic import icosphere

    pos, tri = icosphere(708)
    assert len(tri) == 10_025_280
    out = _on_device(pos, tri, hint=True)
    assert np.max(np.abs(out - vertex_average_arrays(pos, tri))) <= 1e-12
