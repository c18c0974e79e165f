"""Patch packing on the device (``ms_pack_device.cuh``) against the host packer ``ms::pack_patches``: byte for byte
the same headers, halo ids, records, slot facets, statistics and return codes.  The CPU tier runs the device bodies
through the host emulator (tests/emul/pack_emul.cpp); the GPU tier reads the context's packing back
(``DeviceMesh.packing``) after ``set_topology``, ``refine`` and ``equiangulate``."""

import numpy as np
import pytest

import ms_pack_helpers as P
import ms_test_helpers as H

from membrane_solver_b200.geometry.refine import cube_mesh, refine_triangles
from membrane_solver_b200.synthetic import icosphere, open_sheet


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    return P.build_pack_emulator(tmp_path_factory.mktemp("pack_emul"))


def random_order(pos, tri, seed=0):
    perm = np.random.default_rng(seed).permutation(len(pos))
    inv = np.empty_like(perm)
    inv[perm] = np.arange(len(pos))
    return pos[perm], inv[tri].astype(np.int32)


def meshes():
    """name -> (pos, tri, body or None)"""
    out = {}
    for n in (5, 12):
        p, t = icosphere(n)
        out[f"ico{n}"] = (p, t, None)
        out[f"ico{n}_random"] = (*random_order(p, t, n), None)
    p, t, _, b, _ = H.odd_mesh(0, 30)
    out["odd_fan30"] = (p, t, b)
    p, t = cube_mesh()
    for _ in range(4):
        p, t, _, _ = refine_triangles(p, t)
    out["cube_r4"] = (p, t.astype(np.int32), (np.arange(len(t)) % 3 == 0).astype(np.uint8))
    p, t = open_sheet(40, 30, jitter=0.1)
    out["sheet"] = (p, t, None)
    return out


MESHES = meshes()


def assert_same(emul, tri, nv, **kw):
    """The emulated device packer equals the host packer; returns the host's (rc, stats)."""
    rc_d, st_d, arr_d = P.pack_emulated(emul, True, tri, nv, **kw)
    rc_h, st_h, arr_h = P.pack_emulated(emul, False, tri, nv, **kw)
    assert rc_d == rc_h, (rc_d, rc_h)
    if rc_h == 0:
        assert st_d == st_h
        for k in arr_h:
            assert arr_d[k].tobytes() == arr_h[k].tobytes(), k
    return rc_h, st_h


# ---- CPU tier ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", sorted(MESHES))
def test_corner_csr_matches_host(emul, name):
    pos, tri, _ = MESHES[name]
    pd, idd = P.corner_csr_emulated(emul, True, tri, len(pos))
    ph, ih = P.corner_csr_emulated(emul, False, tri, len(pos))
    assert np.array_equal(pd, ph) and np.array_equal(idd, ih)


def test_corner_csr_skips_out_of_range_facets(emul):
    pos, tri = icosphere(3)
    tri = np.concatenate([tri, [[0, 1, len(pos)], [-1, 2, 3], [4, 4, 5]]]).astype(np.int32)
    pd, idd = P.corner_csr_emulated(emul, True, tri, len(pos))
    ph, ih = P.corner_csr_emulated(emul, False, tri, len(pos))
    assert np.array_equal(pd, ph) and np.array_equal(idd, ih)
    assert pd[-1] == 3 * (len(tri) - 2)   # the degenerate facet is valid: the CSR lists it


@pytest.mark.parametrize("name", sorted(MESHES))
@pytest.mark.parametrize("threads", [32, 64, 96, 128])
def test_device_packer_matches_host(emul, name, threads):
    pos, tri, body = MESHES[name]
    threads_ok = 32 if name.startswith("odd") else threads   # the valence-30 fan packs with 32 lanes only
    rc, st = assert_same(emul, tri, len(pos), body=body, threads=threads_ok)
    assert rc == 0 and st["n_listed"] >= st["n_valid"] - 2


@pytest.mark.parametrize("fill_pct", [50, 87, 100])
@pytest.mark.parametrize("repair_sweeps", [0, 1, 3])
def test_tuning(emul, fill_pct, repair_sweeps):
    pos, tri, _ = MESHES["ico12_random"]
    rc, _ = assert_same(emul, tri, len(pos), fill_pct=fill_pct, repair_sweeps=repair_sweeps)
    assert rc == 0


@pytest.mark.parametrize("name", ["ico12", "ico12_random", "cube_r4", "sheet"])
@pytest.mark.parametrize("max_owned,max_local", [(32, 64), (100, 160), (512, 896)])
def test_patch_sizes(emul, name, max_owned, max_local):
    pos, tri, body = MESHES[name]
    rc, _ = assert_same(emul, tri, len(pos), body=body, max_owned=max_owned, max_local=max_local)
    assert rc == 0


def test_trimming(emul):
    """Full-size patches are trimmed to whole rounds: the largest patch owns fewer than max_owned rows."""
    pos, tri, _ = MESHES["ico12"]
    rc, st = assert_same(emul, tri, len(pos))
    assert rc == 0 and 64 < st["max_owned"] < 512 and st["n_patches"] > 1


def test_max_local_halving(emul):
    """A max_local below the neighbourhood of max_owned rows halves the patches (no trimming at 64 rows)."""
    pos, tri, _ = MESHES["ico12_random"]
    rc, st = assert_same(emul, tri, len(pos), max_owned=64, max_local=96)
    assert rc == 0 and st["max_owned"] < 64 and st["max_local"] <= 96


def test_slot_capacity_halving(emul):
    """256 lanes: the seven first rounds exceed 1536 slots, so patches are halved until they fit."""
    pos, tri, _ = MESHES["ico5"]
    rc, st = assert_same(emul, tri, len(pos), threads=256)
    assert rc == 0 and st["max_owned"] < 512 and st["max_slots"] <= 1536


def test_partition(emul):
    pos, tri, _ = MESHES["ico12_random"]
    for n_owned in (len(pos) // 3, len(pos) - 5):
        rc, st = assert_same(emul, tri, len(pos), n_owned=n_owned, max_owned=64, max_local=200)
        assert rc == 0 and st["n_patches"] > 1


def test_several_chunks(emul):
    """Chunks of 32 max_owned rows are packed independently and concatenated."""
    pos, tri, _ = MESHES["ico12_random"]
    rc, st = assert_same(emul, tri, len(pos), max_owned=8, max_local=64)
    assert rc == 0 and len(pos) > 4 * 32 * 8


def test_error_codes(emul):
    pos, tri, _ = MESHES["ico5"]
    assert assert_same(emul, tri, len(pos), max_owned=4, max_local=5)[0] == -2
    assert assert_same(emul, tri, len(pos), fill_pct=5)[0] == -1
    assert assert_same(emul, tri, len(pos), max_slots=16)[0] == -1


def test_narrower_rounds_retry(emul):
    """The valence-30 fan: -3 at 96 and 64 lanes, packs at 32 (pack_rows retries in that order)."""
    pos, tri, body = MESHES["odd_fan30"]
    assert assert_same(emul, tri, len(pos), body=body, threads=96)[0] == -3
    assert assert_same(emul, tri, len(pos), body=body, threads=64)[0] == -3
    assert assert_same(emul, tri, len(pos), body=body, threads=32)[0] == 0
    p, t, _, b, _ = H.odd_mesh(1, 60)   # valence 60: no width fits
    assert assert_same(emul, t, len(p), body=b, threads=32)[0] == -3


# ---- GPU tier ----------------------------------------------------------------------------------------------------

def internal_rows(dm):
    perm = dm.permutation()
    inv = np.empty_like(perm)
    inv[perm] = np.arange(len(perm), dtype=perm.dtype)
    tri = dm.triangles()
    ok = (tri >= 0) & (tri < dm.nv)
    return np.where(ok, inv[np.clip(tri, 0, dm.nv - 1)], tri).astype(np.int32)


def assert_context_matches(emul, dm, body=None, **kw):
    info = dm.pack_info()
    got = dm.packing()
    rc, st, want = P.pack_emulated(emul, False, internal_rows(dm), dm.nv, body=body, threads=info["threads"],
                                   n_owned=dm.n_owned, **kw)
    assert rc == 0
    for k in ("n_patches", "n_halo", "n_slots", "max_owned", "max_local", "max_rounds", "max_slots", "n_round_slots",
              "n_listed", "n_valid", "n_lane_conflicts", "n_hw_groups", "n_hw_excess"):
        assert info[k] == st[k], k
    for k in want:
        assert got[k].tobytes() == want[k].tobytes(), k


def _dm(**kw):
    from membrane_solver_b200.context import DeviceMesh
    return DeviceMesh(0, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(MESHES))
@pytest.mark.parametrize("hint", [False, True])
def test_context_packing(emul, name, hint):
    pos, tri, body = MESHES[name]
    dm = _dm()
    dm.set_topology(len(pos), tri, body_mask=body, order_hint=pos if hint else None)
    assert_context_matches(emul, dm, body=body)


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(threads=32, max_owned=64, max_local=128), dict(threads=128),
                                dict(fill_pct=50, repair_sweeps=3), dict(fill_pct=100, repair_sweeps=0)])
def test_context_packing_params(emul, kw):
    pos, tri, _ = MESHES["ico12_random"]
    dm = _dm(**kw)
    dm.set_topology(len(pos), tri, order_hint=pos)
    tun = {k: kw[k] for k in ("fill_pct", "repair_sweeps") if k in kw}
    size = {k: kw[k] for k in ("max_owned", "max_local") if k in kw}
    assert_context_matches(emul, dm, **tun, **size)


@pytest.mark.gpu
def test_context_partition(emul):
    pos, tri, _ = MESHES["ico12"]
    dm = _dm(max_owned=64, max_local=200)
    dm.set_topology(len(pos), tri, n_owned=len(pos) // 2)
    assert_context_matches(emul, dm, max_owned=64, max_local=200)


@pytest.mark.gpu
@pytest.mark.parametrize("levels", [1, 2])
def test_packing_after_refine(emul, levels):
    pos, tri, body = MESHES["cube_r4"]
    dm = _dm()
    dm.set_topology(len(pos), tri, body_mask=body, order_hint=pos)
    dm.set_positions(pos)
    dm.refine(levels)
    child_body = body[np.arange(dm.nf) % len(tri)]
    assert_context_matches(emul, dm, body=child_body)


@pytest.mark.gpu
def test_packing_after_equiangulate(emul):
    pos, tri = icosphere(12, perturb=False)
    rng = np.random.default_rng(5)
    h = np.mean(np.linalg.norm(pos[tri[:, 1]] - pos[tri[:, 0]], axis=1))
    q = pos + 0.3 * h * rng.normal(size=pos.shape)
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    body = (rng.uniform(size=len(tri)) < 0.5).astype(np.uint8)
    dm = _dm()
    dm.set_topology(len(q), tri, body_mask=body, order_hint=q)
    dm.set_positions(q)
    assert dm.equiangulate(10) > 0
    assert_context_matches(emul, dm, body=body)


@pytest.mark.gpu
def test_failed_pack_leaves_the_context(emul):
    from membrane_solver_b200 import _lib as L
    pos, tri, body = MESHES["odd_fan30"]
    dm = _dm(max_owned=4, max_local=5)
    with pytest.raises(Exception):
        dm.set_topology(len(pos), tri, body_mask=body)
    # refine / equiangulate that cannot pack: a small max_local set after the topology
    p, t = icosphere(6)
    dm = _dm()
    dm.set_topology(len(p), t, order_hint=p)
    dm.set_positions(p)
    before = (dm.packing(), dm.pack_info(), dm.triangles())
    L.check(dm._lib.ms_ctx_set_pack_params(dm._h, 96, 4, 5))
    with pytest.raises(Exception):
        dm.refine(1)
    assert dm.nf == len(t)
    after = (dm.packing(), dm.pack_info(), dm.triangles())
    assert all(before[0][k].tobytes() == after[0][k].tobytes() for k in before[0])
    assert before[1] == after[1] and np.array_equal(before[2], after[2])


@pytest.mark.gpu
@pytest.mark.parametrize("levels", [0, 1])
def test_packing_at_size(emul, levels):
    """The 10 M-facet icosphere, and its refinement to 40 M facets."""
    pos, tri = icosphere(708, perturb=False)
    dm = _dm()
    dm.set_topology(len(pos), tri, order_hint=pos)
    if levels:
        dm.set_positions(pos)
        dm.refine(levels)
    assert_context_matches(emul, dm)
