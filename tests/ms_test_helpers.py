"""Shared helpers for the test-suite (unique module name: an unrelated ``tests`` package is installed in this image)."""

import glob
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def golden_module_files():
    return sorted(glob.glob(os.path.join(GOLDEN, "modules_*.npz")))


def golden_ids():
    return [os.path.basename(p)[len("modules_"):-4] for p in golden_module_files()]


def rel_err(a, b):
    """max|a-b| / max|b|: the gradient parity measure (SURVEY.md §7 hard part 5)."""
    a = np.asarray(a, dtype=float)
    b = np.asarray(b, dtype=float)
    if b.size == 0:
        return 0.0
    scale = max(float(np.max(np.abs(b))), 1e-300)
    return float(np.max(np.abs(a - b))) / scale


def volgrad_close(got, want, pos, tol=1e-12):
    """dV/dx_v = 1/6 sum_i p_i x p_(i+1) cancels from O(|p|^2) summands down to O(h^2): on fine meshes the
    reference's own result moves by more than 1e-12 of its magnitude when its sum is re-ordered.  The bound is
    therefore 1e-12 relative to the size of the summands, and 1e-10 relative to max |dV/dx|."""
    err = float(np.abs(np.asarray(got) - np.asarray(want)).max())
    summand = float((np.asarray(pos) ** 2).sum(axis=1).max()) / 6.0
    assert err <= tol * summand, (err, summand)
    assert err <= 1e-10 * float(np.abs(want).max()), (err, float(np.abs(want).max()))


# --------------------------------------------------------------------------
# Host emulator of the patch kernels (tests/emul/emul.cpp) -- TEST ONLY.
# --------------------------------------------------------------------------
import ctypes
import subprocess

MOD_SURFACE, MOD_VOLUME, MOD_BENDING, MOD_TILT, MOD_BENDING_TILT = 1, 2, 4, 8, 16
FLAG_WILLMORE, FLAG_APPROX = 1, 2
_EMUL = None


def build_emulator():
    src = os.path.join(ROOT, "tests", "emul", "emul.cpp")
    csrc = os.path.join(ROOT, "membrane_solver_b200", "csrc")
    out = os.path.join(ROOT, "tests", "emul", "_build", "libms_emul.so")
    deps = [src] + [os.path.join(csrc, f) for f in ("ms_pack.cpp", "ms_pack.h", "ms_math.cuh", "ms_patch_body.cuh", "ms_bt.cuh",
                                                         "ms_leaflet.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-fPIC", "-shared", "-o", out, src,
                               os.path.join(csrc, "ms_pack.cpp")])
    return out


def emulate(pos, tri, *, modules, flags=0, want_grad=True, is_boundary=None, body_mask=None,
            tilts=None, gamma=None, gamma_u=1.0, kappa=None, c0=None, kappa_u=0.0, c0_u=0.0,
            k_tilt=0.0, threads=96, max_owned=512, max_local=896, n_owned=-1, phase=0, seeds=None):
    """Run the emulator; returns a dict of scalars and arrays."""
    global _EMUL
    if _EMUL is None:
        _EMUL = ctypes.CDLL(build_emulator())
        _EMUL.emul_eval.restype = ctypes.c_int
    pos = np.ascontiguousarray(pos, dtype=np.float64)
    tri = np.ascontiguousarray(tri, dtype=np.int32)
    nv, nf = pos.shape[0], tri.shape[0]

    def dptr(a):
        return None if a is None else a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))

    def bptr(a):
        return None if a is None else a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))

    keep = []

    def f64(a):
        if a is None:
            return None
        a = np.ascontiguousarray(a, dtype=np.float64)
        keep.append(a)
        return a

    def u8(a):
        if a is None:
            return None
        a = np.ascontiguousarray(a, dtype=np.uint8)
        keep.append(a)
        return a

    scal = np.zeros(8)
    out = dict(grad=np.zeros((nv, 3)), volgrad=np.zeros((nv, 3)), tilt_grad=np.zeros((nv, 3)),
               seeds=(np.zeros((nv, 5)) if seeds is None else np.ascontiguousarray(seeds, dtype=np.float64).copy()),
               k_vecs=np.zeros((nv, 3)), a_vor=np.zeros(nv),
               a_eff=np.zeros(nv), e_vertex=np.zeros(nv))
    stats = np.zeros(8, dtype=np.int64)
    rc = _EMUL.emul_eval(
        ctypes.c_int32(nv), ctypes.c_int32(nf), tri.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
        bptr(u8(is_boundary)), bptr(u8(body_mask)), dptr(pos), dptr(f64(tilts)), dptr(f64(gamma)),
        ctypes.c_double(gamma_u), dptr(f64(kappa)), dptr(f64(c0)), ctypes.c_double(kappa_u),
        ctypes.c_double(c0_u), ctypes.c_double(k_tilt), ctypes.c_uint32(modules), ctypes.c_uint32(flags),
        ctypes.c_int32(1 if want_grad else 0), ctypes.c_int32(threads), ctypes.c_int32(max_owned),
        ctypes.c_int32(max_local), dptr(scal), dptr(out["grad"]), dptr(out["volgrad"]),
        dptr(out["tilt_grad"]), dptr(out["seeds"]), dptr(out["k_vecs"]), dptr(out["a_vor"]),
        dptr(out["a_eff"]), dptr(out["e_vertex"]), stats.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)),
        ctypes.c_int32(n_owned), ctypes.c_int32(phase))
    if rc:
        raise RuntimeError(f"emul_eval failed: {rc}")
    out.update(E_surface=scal[0], area=scal[1], volume=scal[2], E_bending=scal[3], E_tilt=scal[4],
               E_bending_tilt=scal[5],
               pack=dict(n_patches=int(stats[0]), n_slots=int(stats[1]), n_listed=int(stats[2]),
                         max_rounds=int(stats[3]), max_local=int(stats[4]),
                         lane_conflicts=int(stats[5]), hw_groups=int(stats[6]), hw_excess=int(stats[7])))
    return out


def emulate_leaflet(pos, tri, tilts, *, sign, keep=None, is_boundary=None, interior=None, base_zero=None,
                    kappa=None, c0=None, kappa_u=0.0, c0_u=0.0, row_weight=None, consistent=None,
                    consistent_u=False, k_tilt=0.0, k_smooth=0.0, with_bt=True, with_tilt=False, with_smooth=False,
                    want_grad=True, want_tilt_grad=True):
    """Leaflet modules through the emulator (same ms_leaflet.cuh bodies as the device kernels)."""
    global _EMUL
    if _EMUL is None:
        _EMUL = ctypes.CDLL(build_emulator())
        _EMUL.emul_eval.restype = ctypes.c_int
    pos = np.ascontiguousarray(pos, dtype=np.float64)
    tri = np.ascontiguousarray(tri, dtype=np.int32)
    tilts = np.ascontiguousarray(tilts, dtype=np.float64)
    nv, nf = pos.shape[0], tri.shape[0]
    keepalive = []

    def conv(a, dt, ct):
        if a is None:
            return None
        a = np.ascontiguousarray(a, dtype=dt)
        keepalive.append(a)
        return a.ctypes.data_as(ctypes.POINTER(ct))

    grad = np.zeros((nv, 3)) if want_grad else None
    tg = np.zeros((nv, 3)) if want_tilt_grad else None
    e2 = np.zeros(3)
    dp = ctypes.POINTER(ctypes.c_double)
    rc = _EMUL.emul_leaflet(
        ctypes.c_int32(nv), ctypes.c_int32(nf), tri.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
        pos.ctypes.data_as(dp), tilts.ctypes.data_as(dp), conv(keep, np.uint8, ctypes.c_uint8),
        conv(is_boundary, np.uint8, ctypes.c_uint8), conv(interior, np.uint8, ctypes.c_uint8),
        conv(base_zero, np.uint8, ctypes.c_uint8), conv(kappa, np.float64, ctypes.c_double),
        conv(c0, np.float64, ctypes.c_double), ctypes.c_double(kappa_u), ctypes.c_double(c0_u),
        conv(row_weight, np.float64, ctypes.c_double), conv(consistent, np.uint8, ctypes.c_uint8),
        ctypes.c_int32(int(bool(consistent_u))), ctypes.c_double(k_tilt), ctypes.c_double(k_smooth), ctypes.c_double(sign),
        ctypes.c_int32(int(with_bt)), ctypes.c_int32(int(with_tilt)), ctypes.c_int32(int(with_smooth)),
        None if grad is None else grad.ctypes.data_as(dp), None if tg is None else tg.ctypes.data_as(dp),
        e2.ctypes.data_as(dp))
    if rc:
        raise RuntimeError(f"emul_leaflet failed: {rc}")
    return dict(E_bt=float(e2[0]), E_tilt=float(e2[1]), E_smooth=float(e2[2]), grad=grad, tilt_grad=tg)


def odd_mesh(seed: int, nfan: int):
    """A mesh the benchmark shapes never produce (see test_odd_topologies_against_the_oracle) with per-facet surface
    tension, a partial body and the oracle's surface / volume results: (pos, tri, gamma, body, (E, g, V, dV/dx))."""
    from membrane_solver_b200.synthetic import icosphere, open_sheet
    from oracle import ref_modules as ref

    rng = np.random.default_rng(seed)
    pa, ta = icosphere(4)
    pb, tb = open_sheet(5, 4, jitter=0.1)
    pb = pb + np.array([3.0, 0.0, 0.0])
    ring = np.stack([np.cos(np.linspace(0, 2 * np.pi, nfan, endpoint=False)),
                     np.sin(np.linspace(0, 2 * np.pi, nfan, endpoint=False)), np.zeros(nfan)], axis=1)
    pc = np.concatenate([[[0.0, 0.0, 0.4]], ring]) + np.array([0.0, 4.0, 0.0])
    tc = np.stack([np.zeros(nfan, int), 1 + np.arange(nfan), 1 + (np.arange(nfan) + 1) % nfan], axis=1)
    pos = np.concatenate([pa, pb, pc, rng.normal(size=(7, 3))])                 # 7 vertices nobody uses
    tri = np.concatenate([ta, tb + len(pa), tc + len(pa) + len(pb)])
    tri = np.concatenate([tri, tri[3:4], [[5, 5, 9], [2, 7, 2]]])               # duplicate facet, two degenerate ones
    perm = rng.permutation(len(pos))                                            # random vertex order
    inv = np.empty_like(perm)
    inv[perm] = np.arange(len(pos))
    pos, tri = pos[perm], inv[tri].astype(np.int32)
    pos = pos + 0.01 * rng.normal(size=pos.shape)
    nf = tri.shape[0]
    gamma = rng.uniform(0.5, 1.5, size=nf)
    body = (rng.uniform(size=nf) < 0.6).astype(np.uint8)
    want_g = np.zeros_like(pos)
    want_e = ref.surface_energy_and_gradient(pos, tri, gamma, want_g)
    want_vg = np.zeros_like(pos)
    tri_body = tri[body.astype(bool)]
    want_v = ref.body_volume(pos, tri_body)
    ref.accumulate_volume_gradient(pos, tri_body, want_vg, 1.0)
    return pos, tri, gamma, body, (want_e, want_g, want_v, want_vg)
