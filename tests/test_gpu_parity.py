"""GPU parity tests proper: the CUDA path, called through the C ABI, against the
CPU oracle (pinned to the reference by tests/test_oracle_golden.py) and against
the golden vectors produced by the real reference.

Tolerance: 1e-12 relative (fp64), measured as max|a-b|/max|b| for vectors
(BASELINE.json north_star; SURVEY.md section 7 hard part 5).
"""

import ctypes

import numpy as np
import pytest

from ms_test_helpers import golden_ids, golden_module_files, rel_err, volgrad_close

pytestmark = pytest.mark.gpu

TOL = 1e-12
BENDING_TAGS = {
    "helfrich_analytic": (0, 0),
    "helfrich_c0": (0, 0),
    "helfrich_approx": (0, 2),
    "willmore_analytic": (1, 0),
}


@pytest.fixture(scope="module")
def L():
    from membrane_solver_b200 import _lib

    if _lib.device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu tier must run on the B200 box")
    return _lib


def _ctx(nv, tri, **kw):
    from membrane_solver_b200.context import DeviceMesh

    pack = {k: kw.pop(k) for k in ("threads", "max_owned", "max_local") if k in kw}
    dm = DeviceMesh(0, **pack)
    dm.set_topology(nv, tri, **kw)
    return dm


def _scalar_close(a, b, tol=TOL):
    assert abs(a - b) <= tol * max(1.0, abs(b)), (a, b)


# ------------------------------------------------------------------ shims
def test_shim_grad_cotan(L, kernels_golden):
    g = kernels_golden
    for tag in ("gc4", "gc17", "gcd"):
        u, v = np.ascontiguousarray(g[f"{tag}_u"]), np.ascontiguousarray(g[f"{tag}_v"])
        gu, gv = np.empty_like(u), np.empty_like(v)
        L.check(L.lib().ms_grad_cotan_batch(u.shape[0], L.dptr(u), L.dptr(v), L.dptr(gu), L.dptr(gv)))
        assert rel_err(gu, g[f"{tag}_gu"]) <= TOL
        assert rel_err(gv, g[f"{tag}_gv"]) <= TOL
    assert np.array_equal(gu[2], np.zeros(3))


def test_shim_laplacian(L, kernels_golden):
    g = kernels_golden
    w, tri, field = (np.ascontiguousarray(g[k]) for k in ("lap_w", "lap_tri", "lap_field"))
    out = np.full_like(field, np.nan)
    L.check(L.lib().ms_apply_beltrami_laplacian(field.shape[1], field.shape[0], tri.shape[0], L.dptr(w),
                                                L.iptr(tri), L.dptr(field), L.dptr(out), 1))
    assert rel_err(out, g["lap_out"]) <= TOL
    # one-based indices give the same answer
    tri1 = np.ascontiguousarray(tri + 1)
    out1 = np.empty_like(field)
    L.check(L.lib().ms_apply_beltrami_laplacian(field.shape[1], field.shape[0], tri.shape[0], L.dptr(w),
                                                L.iptr(tri1), L.dptr(field), L.dptr(out1), 0))
    assert np.array_equal(out, out1)


def test_shim_p1_divergence(L, kernels_golden):
    g = kernels_golden
    pos, tl, tri = (np.ascontiguousarray(g[k]) for k in ("p1_pos", "p1_tilts", "p1_tri"))
    nf = tri.shape[0]
    div, area = np.empty(nf), np.empty(nf)
    g0, g1, g2 = np.empty((nf, 3)), np.empty((nf, 3)), np.empty((nf, 3))
    L.check(L.lib().ms_p1_triangle_divergence(pos.shape[0], nf, L.dptr(pos), L.dptr(tl), L.iptr(tri),
                                              L.dptr(div), L.dptr(area), L.dptr(g0), L.dptr(g1), L.dptr(g2), 1))
    for a, name in ((div, "p1_div"), (area, "p1_area"), (g0, "p1_g0"), (g1, "p1_g1"), (g2, "p1_g2")):
        assert rel_err(a, g[name]) <= TOL, name


def test_shim_curvature_data(L, kernels_golden):
    g = kernels_golden
    pos, tri = np.ascontiguousarray(g["cd_pos"]), np.ascontiguousarray(g["cd_tri"])
    nv, nf = pos.shape[0], tri.shape[0]
    k, a, w = np.empty((nv, 3)), np.empty(nv), np.empty((nf, 3))
    va = [np.empty(nf) for _ in range(3)]
    L.check(L.lib().ms_compute_curvature_data(nv, nf, L.dptr(pos), L.iptr(tri), L.dptr(k), L.dptr(a),
                                              L.dptr(w), 1, L.dptr(va[0]), L.dptr(va[1]), L.dptr(va[2])))
    for x, name in ((k, "cd_k"), (a, "cd_a"), (w, "cd_w"), (va[0], "cd_va0"), (va[1], "cd_va1"), (va[2], "cd_va2")):
        assert rel_err(x, g[name]) <= TOL, name
    # the optional corner outputs may be omitted (tilt_kernels.f90:96)
    L.check(L.lib().ms_compute_curvature_data(nv, nf, L.dptr(pos), L.iptr(tri), L.dptr(k), L.dptr(a),
                                              L.dptr(w), 1, None, None, None))
    assert rel_err(k, g["cd_k"]) <= TOL


def test_shim_surface_soup(L, kernels_golden):
    """Random triangle soup incl. repeated indices; out-of-range facets are skipped."""
    from oracle import ref_modules as ref

    g = kernels_golden
    pos, tri, gamma = (np.ascontiguousarray(g[k]) for k in ("sf_pos", "sf_tri", "sf_gamma"))
    grad_ref = np.ones_like(pos)
    e_ref = ref.surface_energy_and_gradient(pos, tri, gamma, grad_ref)
    grad = np.ones_like(pos)  # the kernel accumulates into the caller's array
    e = ctypes.c_double(0.0)
    L.check(L.lib().ms_surface_energy_and_gradient(pos.shape[0], tri.shape[0], L.dptr(pos), L.iptr(tri),
                                                   L.dptr(gamma), L.dptr(grad), ctypes.byref(e), 1))
    _scalar_close(e.value, e_ref)
    assert rel_err(grad, grad_ref) <= TOL
    bad = tri.copy()
    bad[3, 1] = pos.shape[0] + 5
    bad[4, 0] = -1
    keep = np.ones(len(tri), bool)
    keep[[3, 4]] = False
    grad_ref = np.zeros_like(pos)
    e_ref = ref.surface_energy_and_gradient(pos, tri[keep], gamma[keep], grad_ref)
    grad = np.zeros_like(pos)
    L.check(L.lib().ms_surface_energy_and_gradient(pos.shape[0], bad.shape[0], L.dptr(pos), L.iptr(bad),
                                                   L.dptr(gamma), L.dptr(grad), ctypes.byref(e), 1))
    _scalar_close(e.value, e_ref)
    assert rel_err(grad, grad_ref) <= TOL


def test_shim_empty_inputs(L):
    e = ctypes.c_double(1.0)
    pos = np.zeros((3, 3))
    grad = np.zeros((3, 3))
    L.check(L.lib().ms_surface_energy_and_gradient(3, 0, L.dptr(pos), None, None, L.dptr(grad), ctypes.byref(e), 1))
    assert e.value == 0.0 and not grad.any()
    L.check(L.lib().ms_grad_cotan_batch(0, None, None, None, None))


# ------------------------------------------------------------- golden meshes
@pytest.mark.parametrize("path", golden_module_files(), ids=golden_ids())
def test_context_vs_reference_golden(L, path):
    g = dict(np.load(path))
    pos, tri = g["pos"], g["tri"]
    nv, nf = pos.shape[0], tri.shape[0]
    body = np.zeros(nf, np.uint8)
    if "body_rows_0" in g:
        body[g["body_rows_0"]] = 1
    for pack in (dict(), dict(threads=32, max_owned=16, max_local=120)):
        dm = _ctx(nv, tri, is_boundary=g["is_boundary"], body_mask=body, **pack)
        dm.set_surface_tension(g["gamma"])
        dm.set_positions(pos)
        dm.set_tilts(g["tilts"])
        dm.set_tilt_rigidity(float(g["k_tilt"]))

        r = dm.eval(dm.options(L.MOD_SURFACE | L.MOD_VOLUME))
        _scalar_close(r.e_surface, float(g["E_surface"]))
        assert rel_err(dm.download(L.ARR_GRAD), g["g_surface"]) <= TOL
        if "g_volume" in g:
            _scalar_close(r.volume, float(g["volumes"][0]))
            assert rel_err(dm.download(L.ARR_VOLGRAD), g["g_volume"][0]) <= TOL

        for tag, (wil, apx) in BENDING_TAGS.items():
            kappa, c0 = g[f"param_{tag}"]
            dm.set_bending_params(kappa, c0)
            r = dm.eval(dm.options(L.MOD_BENDING, flags=wil | apx, diagnostics=True))
            _scalar_close(r.e_bending, float(g[f"E_bending_{tag}"]))
            grad = dm.download(L.ARR_GRAD)
            if apx:
                grad[g["is_boundary"]] = 0.0  # bending.py:163-167, applied by the host module
            assert rel_err(grad, g[f"g_bending_{tag}"]) <= 2e-12, tag
            assert rel_err(dm.download(L.ARR_E_VERTEX), g[f"Ev_bending_{tag}"]) <= TOL
            # energy-only evaluation (line search) gives the same energy
            r2 = dm.eval(dm.options(L.MOD_BENDING, flags=wil | apx, want_grad=False))
            assert r2.e_bending == r.e_bending
        assert rel_err(dm.download(L.ARR_K_VECS), g["k_vecs"]) <= TOL
        assert rel_err(dm.download(L.ARR_A_VOR), g["a_vor"]) <= TOL
        assert rel_err(dm.download(L.ARR_A_EFF), g["a_eff"]) <= TOL

        r = dm.eval(dm.options(L.MOD_TILT))
        _scalar_close(r.e_tilt, float(g["E_tilt"]))
        assert rel_err(dm.download(L.ARR_GRAD), g["g_tilt"]) <= TOL
        assert rel_err(dm.download(L.ARR_TILT_GRAD), g["tg_tilt"]) <= TOL
        r2 = dm.eval(dm.options(L.MOD_TILT, want_grad=False))
        _scalar_close(r2.e_tilt, float(g["E_tilt"]))
        dm.close()


def test_minimizer_golden(L, minimizer_golden):
    """Fused evaluation + KKT / penalty / fixed-mask post-processing against
    Minimizer.compute_energy_and_gradient_array of the reference."""
    g = minimizer_golden
    # cube: surface + volume penalty
    pos, tri = g["cube_pos"], g["cube_tri"]
    body = np.zeros(len(tri), np.uint8)
    body[g["cube_body_rows_0"]] = 1
    dm = _ctx(pos.shape[0], tri, is_boundary=g["cube_is_boundary"], body_mask=body, fixed_mask=g["cube_fixed"])
    dm.set_surface_tension(g["cube_gamma"])
    dm.set_positions(pos)
    k, v0 = float(g["cube_kvol"]), float(g["cube_body_target_0"])
    r = dm.eval(dm.options(L.MOD_SURFACE | L.MOD_VOLUME, constraint_mode=1, k_vol=k, v_target=v0, apply_fixed=True))
    e = r.e_surface + 0.5 * k * (r.volume - v0) ** 2
    _scalar_close(e, float(g["cube_E"]))
    assert rel_err(dm.download(L.ARR_GRAD), g["cube_g"]) <= TOL
    dm.close()
    # bending cube: bending + lagrange volume constraint
    pos, tri = g["bcube_pos"], g["bcube_tri"]
    body = np.zeros(len(tri), np.uint8)
    body[g["bcube_body_rows_0"]] = 1
    dm = _ctx(pos.shape[0], tri, is_boundary=g["bcube_is_boundary"], body_mask=body, fixed_mask=g["bcube_fixed"])
    dm.set_bending_params(float(g["bcube_kappa"]), float(g["bcube_c0"]))
    dm.set_positions(pos)
    r = dm.eval(dm.options(L.MOD_BENDING | L.MOD_VOLUME, constraint_mode=0, apply_fixed=True))
    _scalar_close(r.e_bending, float(g["bcube_E"]))
    assert rel_err(dm.download(L.ARR_GRAD), g["bcube_g"]) <= 2e-12
    dm.close()


# -------------------------------------------------------------- synthetic
@pytest.mark.parametrize("n,pack", [(6, dict()), (40, dict()), (40, dict(threads=64, max_owned=200, max_local=420)),
                                    (120, dict(threads=128, max_owned=384, max_local=700)), (120, dict(threads=160, max_owned=512, max_local=896))])
def test_icosphere_fused_vs_oracle(L, n, pack):
    from membrane_solver_b200.synthetic import icosphere
    from oracle import ref_modules as ref

    pos, tri = icosphere(n)
    nv, nf = pos.shape[0], tri.shape[0]
    ref_out = ref.fused_surface_bending_volume(pos, tri, np.ones(nf), 1.0, 0.05, np.zeros(nv, bool))
    dm = _ctx(nv, tri, body_mask=np.ones(nf, np.uint8), **pack)
    dm.set_bending_params(1.0, 0.05)
    dm.set_positions(pos)
    r = dm.eval(dm.options(L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME))
    _scalar_close(r.e_surface, ref_out["E_surface"])
    _scalar_close(r.e_bending, ref_out["E_bending"])
    _scalar_close(r.volume, ref_out["volume"])
    _scalar_close(r.area, ref_out["area"])
    g1 = dm.download(L.ARR_GRAD)
    assert rel_err(g1, ref_out["grad"]) <= TOL
    assert rel_err(dm.download(L.ARR_VOLGRAD), ref_out["vol_grad"]) <= TOL
    # run-to-run reproducibility: bitwise identical results
    r2 = dm.eval(dm.options(L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME))
    assert np.array_equal(r.scalars, r2.scalars)
    assert np.array_equal(g1, dm.download(L.ARR_GRAD))
    # end-to-end call with host buffers returns the same numbers
    grad = np.empty_like(pos)
    volgrad = np.empty_like(pos)
    r3 = dm.eval_host(dm.options(L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME), pos, grad=grad, volgrad=volgrad)
    assert np.array_equal(r3.scalars[:6], r.scalars[:6])
    assert np.array_equal(grad, g1)
    dm.close()


def test_open_sheet_boundary_and_flat_normals(L):
    """Open flat sheet: boundary redistribution + |K|=0 normal fallback with c0 != 0."""
    from membrane_solver_b200.synthetic import open_sheet
    from oracle import ref_modules as ref

    for jitter in (0.0, 0.08):
        pos, tri = open_sheet(9, 7, jitter=jitter)
        nv = pos.shape[0]
        is_b = ref.boundary_mask_from_triangles(tri, nv)
        grad_ref = np.zeros_like(pos)
        e_ref = ref.bending_energy_and_gradient(pos, tri, 1.5, 0.3, is_b, grad_ref)
        dm = _ctx(nv, tri, is_boundary=is_b, threads=32, max_owned=24, max_local=100)
        dm.set_bending_params(1.5, 0.3)
        dm.set_positions(pos)
        r = dm.eval(dm.options(L.MOD_BENDING))
        _scalar_close(r.e_bending, e_ref)
        assert rel_err(dm.download(L.ARR_GRAD), grad_ref) <= TOL
        dm.close()


def test_per_entity_parameters(L):
    """Per-facet surface tension and per-vertex kappa / c0 arrays."""
    from membrane_solver_b200.synthetic import icosphere
    from oracle import ref_modules as ref

    pos, tri = icosphere(12)
    nv, nf = pos.shape[0], tri.shape[0]
    rng = np.random.default_rng(11)
    gamma = rng.uniform(0.5, 2.0, nf)
    kappa = rng.uniform(0.5, 2.0, nv)
    c0 = rng.uniform(-0.3, 0.3, nv)
    grad_ref = np.zeros_like(pos)
    e_s = ref.surface_energy_and_gradient(pos, tri, gamma, grad_ref)
    e_b = ref.bending_energy_and_gradient(pos, tri, kappa, c0, np.zeros(nv, bool), grad_ref)
    dm = _ctx(nv, tri)
    dm.set_surface_tension(gamma)
    dm.set_bending_params(kappa, c0)
    dm.set_positions(pos)
    r = dm.eval(dm.options(L.MOD_SURFACE | L.MOD_BENDING))
    _scalar_close(r.e_surface, e_s)
    _scalar_close(r.e_bending, e_b)
    assert rel_err(dm.download(L.ARR_GRAD), grad_ref) <= TOL
    dm.close()


def test_degenerate_and_empty_meshes(L):
    from oracle import ref_modules as ref

    # empty mesh
    dm = _ctx(0, np.zeros((0, 3), np.int32))
    r = dm.eval(dm.options(L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME))
    assert not r.scalars[:6].any()
    dm.close()
    # vertices without facets + degenerate (repeated index, zero area) facets
    pos = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0.2], [5, 5, 5], [2, 0, 0]], dtype=float)
    tri = np.array([[0, 1, 2], [1, 3, 2], [0, 0, 1], [0, 1, 5]], dtype=np.int32)
    grad_ref = np.zeros_like(pos)
    e_s = ref.surface_energy_and_gradient(pos, tri, np.ones(4), grad_ref)
    is_b = ref.boundary_mask_from_triangles(tri[:2], 6)
    e_b = ref.bending_energy_and_gradient(pos, tri, 1.0, 0.1, is_b, grad_ref)
    dm = _ctx(6, tri, is_boundary=is_b)
    dm.set_bending_params(1.0, 0.1)
    dm.set_positions(pos)
    r = dm.eval(dm.options(L.MOD_SURFACE | L.MOD_BENDING))
    _scalar_close(r.e_surface, e_s)
    _scalar_close(r.e_bending, e_b)
    assert rel_err(dm.download(L.ARR_GRAD), grad_ref) <= TOL
    dm.close()


def test_trial_positions_energy_only(L):
    """x + alpha d on the device, energy-only evaluation (line_search.py:358-382)."""
    from membrane_solver_b200.synthetic import icosphere
    from oracle import ref_modules as ref

    pos, tri = icosphere(10)
    nv, nf = pos.shape[0], tri.shape[0]
    rng = np.random.default_rng(4)
    d = 0.01 * rng.normal(size=pos.shape)
    dm = _ctx(nv, tri, body_mask=np.ones(nf, np.uint8))
    dm.set_bending_params(1.0, 0.0)
    dm.set_positions(pos)
    dm.set_direction(d)
    dm.make_trial(0.37)
    r = dm.eval(dm.options(L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME, want_grad=False, use_trial=True))
    x = pos + 0.37 * d
    ref_out = ref.fused_surface_bending_volume(x, tri, np.ones(nf), 1.0, 0.0, np.zeros(nv, bool))
    _scalar_close(r.e_surface, ref_out["E_surface"])
    _scalar_close(r.e_bending, ref_out["E_bending"])
    _scalar_close(r.volume, ref_out["volume"])
    dm.accept_trial()
    assert rel_err(dm.download(L.ARR_POSITIONS), x) <= 1e-15
    dm.close()


def test_repeatability_stress(L):
    """The persistent kernels hand buffers between producer, consumer groups and epilogue warps
    through barriers: 40 back-to-back evaluations at several pack geometries must be bitwise
    identical (a race would show up as a last-bit or gross difference)."""
    from membrane_solver_b200.synthetic import icosphere

    pos, tri = icosphere(150)
    nv, nf = pos.shape[0], tri.shape[0]
    mods = L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME
    for pack in (dict(), dict(threads=32, max_owned=64, max_local=200), dict(threads=160, max_owned=512, max_local=896),
                 dict(threads=64, max_owned=256, max_local=512)):
        dm = _ctx(nv, tri, body_mask=np.ones(nf, np.uint8), **pack)
        dm.set_bending_params(1.0, 0.1)
        dm.set_positions(pos)
        opts = dm.options(mods, constraint_mode=0)
        first = dm.eval(opts)
        g0, v0, s0 = dm.download(L.ARR_GRAD), dm.download(L.ARR_VOLGRAD), dm.download(L.ARR_SEEDS)
        for _ in range(40):
            dm.eval_async(opts)
        again = dm.read_scalars()
        assert np.array_equal(first.scalars, again.scalars), pack
        assert np.array_equal(g0, dm.download(L.ARR_GRAD)), pack
        assert np.array_equal(v0, dm.download(L.ARR_VOLGRAD)), pack
        assert np.array_equal(s0, dm.download(L.ARR_SEEDS)), pack
        dm.close()


@pytest.mark.parametrize("path", golden_module_files(), ids=golden_ids())
def test_bending_tilt_vs_reference_golden(L, path):
    """bending_tilt through the C ABI: coupling stage (divergence, seeds, energy, tilt gradient) +
    pass B back-propagation, against the reference's vectors; tilt-only evaluation; combined with
    the tilt-magnitude module."""
    g = dict(np.load(path))
    pos, tri = g["pos"], g["tri"]
    nv = pos.shape[0]
    is_b = g["is_boundary"].astype(np.uint8) if g["is_boundary"].any() else None
    for pack in (dict(), dict(threads=32, max_owned=24, max_local=100)):
        dm = _ctx(nv, tri, is_boundary=is_b, **pack)
        dm.set_tilts(g["tilts"])
        dm.set_tilt_rigidity(float(g["k_tilt"]))
        for tag, (wil, apx) in BENDING_TAGS.items():
            if wil:
                continue
            kappa, c0 = g[f"param_{tag}"]
            dm.set_bending_params(float(kappa), float(c0))
            grad, tg = np.empty_like(pos), np.empty_like(pos)
            r = dm.eval_host(dm.options(L.MOD_BENDING_TILT, flags=apx), pos, grad=grad, tilt_grad=tg)
            _scalar_close(float(r.scalars[L.SC_E_BENDING_TILT]), float(g[f"E_bending_tilt_{tag}"]))
            assert r.e_bending == 0.0
            if apx:
                grad[g["is_boundary"]] = 0.0
            assert rel_err(grad, g[f"g_bending_tilt_{tag}"]) <= 2e-12, tag
            assert rel_err(tg, g[f"tg_bending_tilt_{tag}"]) <= TOL, tag
            tg2 = np.empty_like(pos)
            r = dm.eval_host(dm.options(L.MOD_BENDING_TILT, flags=apx, want_grad=False, want_tilt_grad=True), pos,
                             tilt_grad=tg2)
            _scalar_close(float(r.scalars[L.SC_E_BENDING_TILT]), float(g[f"E_bending_tilt_{tag}"]))
            assert rel_err(tg2, g[f"tgonly_bending_tilt_{tag}"]) <= TOL, tag
        # together with the tilt-magnitude module: energies separate, tilt gradients summed
        kappa, c0 = g["param_helfrich_analytic"]
        dm.set_bending_params(float(kappa), float(c0))
        grad, tg = np.empty_like(pos), np.empty_like(pos)
        r = dm.eval_host(dm.options(L.MOD_BENDING_TILT | L.MOD_TILT), pos, grad=grad, tilt_grad=tg)
        _scalar_close(r.e_tilt, float(g["E_tilt"]))
        _scalar_close(float(r.scalars[L.SC_E_BENDING_TILT]), float(g["E_bending_tilt_helfrich_analytic"]))
        assert rel_err(grad, g["g_tilt"] + g["g_bending_tilt_helfrich_analytic"]) <= 2e-12
        assert rel_err(tg, g["tg_tilt"] + g["tg_bending_tilt_helfrich_analytic"]) <= TOL
        with pytest.raises(L.B200Error):
            dm.eval(dm.options(L.MOD_BENDING_TILT | L.MOD_BENDING))
        dm.close()


def test_internal_reordering_is_transparent(L):
    """A mesh in RANDOM vertex order: with the order hint the context packs compact patches
    (few ring-facet listings) and every upload / download stays in the caller's order."""
    from membrane_solver_b200.context import DeviceMesh
    from membrane_solver_b200.synthetic import icosphere
    from oracle import ref_modules as ref

    pos0, tri0 = icosphere(60)
    nv, nf = pos0.shape[0], tri0.shape[0]
    rng = np.random.default_rng(3)
    old_of_new = rng.permutation(nv)
    new_of_old = np.empty(nv, np.int64)
    new_of_old[old_of_new] = np.arange(nv)
    pos = np.ascontiguousarray(pos0[old_of_new])
    tri = np.ascontiguousarray(new_of_old[tri0].astype(np.int32))
    kappa = 1.0 + 0.3 * rng.random(nv)
    c0 = 0.05 * rng.random(nv)
    gamma = 1.0 + 0.2 * rng.random(nf)
    want = ref.fused_surface_bending_volume(pos, tri, gamma, kappa, c0, np.zeros(nv, bool))
    listed = {}
    for hint in (None, pos):
        dm = DeviceMesh(0)
        dm.set_topology(nv, tri, body_mask=np.ones(nf, np.uint8), order_hint=hint)
        listed[hint is None] = dm.pack_info()["n_listed"]
        dm.set_surface_tension(gamma)
        dm.set_bending_params(kappa, c0)
        grad, volgrad = np.empty_like(pos), np.empty_like(pos)
        r = dm.eval_host(dm.options(L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME), pos, grad=grad, volgrad=volgrad)
        _scalar_close(r.e_surface, want["E_surface"])
        _scalar_close(r.e_bending, want["E_bending"])
        _scalar_close(r.volume, want["volume"])
        assert rel_err(grad, want["grad"]) <= 2e-12
        assert rel_err(volgrad, want["vol_grad"]) <= TOL
        assert np.array_equal(dm.download(L.ARR_GRAD), grad)            # ms_ctx_get_array: caller's order too
        assert np.array_equal(dm.download(L.ARR_POSITIONS), pos)
        perm = dm.permutation()
        assert sorted(perm.tolist()) == list(range(nv))
        if hint is None:
            assert np.array_equal(perm, np.arange(nv))
        dm.close()
    assert listed[False] < 0.5 * listed[True], listed   # hint: ~1.2 x nf listings instead of ~3 x nf


def test_full_size_invariants(L):
    """BASELINE.json configs[4] at its full single-GPU size (10 M facets), where the oracle is too
    slow: size-independent properties of the exact gradients.
      * Euler's theorem: surface energy is homogeneous of degree 2 in x, volume of degree 3, the
        Helfrich energy with c0 = 0 of degree 0  ->  <g_S, x> = 2 E_S, <dV/dx, x> = 3 V, <g_B, x> = 0;
      * translation invariance: every gradient sums to zero over the closed surface;
      * scaling x -> s x and a rigid rotation change the scalars exactly as the degrees predict;
      * the KKT-projected gradient is orthogonal to dV/dx."""
    from membrane_solver_b200.synthetic import frequency_for_facets, icosphere

    n = frequency_for_facets(10_000_000)
    pos, tri = icosphere(n)
    nv, nf = pos.shape[0], tri.shape[0]
    assert nf >= 10_000_000
    dm = _ctx(nv, tri, body_mask=np.ones(nf, np.uint8))
    dm.set_surface_tension(1.0)
    dm.set_bending_params(1.0, 0.0)
    dm.set_positions(pos)
    x = pos.reshape(-1)

    def run(mods, **kw):
        r = dm.eval(dm.options(mods, **kw))
        return r, dm.download(L.ARR_GRAD), dm.download(L.ARR_VOLGRAD)

    rs, gs, gv = run(L.MOD_SURFACE | L.MOD_VOLUME)
    assert abs(gs.reshape(-1) @ x - 2.0 * rs.e_surface) <= 1e-10 * rs.e_surface
    assert abs(gv.reshape(-1) @ x - 3.0 * rs.volume) <= 1e-10 * rs.volume
    assert np.abs(gs.sum(axis=0)).max() <= 1e-9 and np.abs(gv.sum(axis=0)).max() <= 1e-9
    rb, gb, _ = run(L.MOD_BENDING)
    gscale = np.abs(gb).max()
    assert abs(gb.reshape(-1) @ x) <= 1e-9 * rb.e_bending            # scale invariance of the Willmore/Helfrich(c0=0) energy
    assert np.abs(gb.sum(axis=0)).max() <= 1e-7 * gscale * np.sqrt(nv)
    # fused evaluation = sum of the parts; projection removes the dV/dx component
    rf, gf, gvf = run(L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME)
    assert rel_err(gf, gs + gb) <= 1e-12 and rel_err(gvf, gv) <= 1e-12  # other instantiation: rounding of (v1 x v2) only
    rp, gp, _ = run(L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME, constraint_mode=0)
    lam = rp.kkt_lambda
    assert rel_err(gp, gf - lam * gv) <= 1e-12
    assert abs(gp.reshape(-1) @ gv.reshape(-1)) <= 1e-9 * np.linalg.norm(gp) * np.linalg.norm(gv)
    # scaling and rotation
    s = 1.37
    c, sn = np.cos(0.7), np.sin(0.7)
    rot = np.array([[c, -sn, 0.0], [sn, c, 0.0], [0.0, 0.0, 1.0]]) @ np.array([[1, 0, 0], [0, c, -sn], [0, sn, c]])
    dm.set_positions(s * pos @ rot.T)
    r2, g2, _ = run(L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME)
    assert abs(r2.e_surface - s * s * rf.e_surface) <= 1e-11 * r2.e_surface
    assert abs(r2.volume - s**3 * rf.volume) <= 1e-11 * r2.volume
    assert abs(r2.e_bending - rf.e_bending) <= 1e-10 * rf.e_bending
    assert abs(r2.area - s * s * rf.area) <= 1e-11 * r2.area
    dm.close()


# -------------------------------------------------------------- parity at size (BASELINE.json configs[2], configs[4])
def test_million_facet_icosphere_vs_oracle(L):
    """1 003 520 facets: the largest mesh on which the whole-mesh oracle runs in seconds; energies, gradient and
    dV/dx of the fused evaluation and of the KKT-projected evaluation at 1e-12 relative."""
    from membrane_solver_b200.synthetic import icosphere
    from oracle import ref_modules as ref

    pos, tri = icosphere(224)
    nv, nf = pos.shape[0], tri.shape[0]
    assert nf >= 1_000_000
    want = ref.fused_surface_bending_volume(pos, tri, np.ones(nf), 1.0, 0.05, np.zeros(nv, bool))
    dm = _ctx(nv, tri, body_mask=np.ones(nf, np.uint8))
    dm.set_bending_params(1.0, 0.05)
    dm.set_positions(pos)
    mods = L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME
    r = dm.eval(dm.options(mods))
    for got, name in ((r.e_surface, "E_surface"), (r.e_bending, "E_bending"), (r.volume, "volume"), (r.area, "area")):
        _scalar_close(got, want[name])
    g = dm.download(L.ARR_GRAD)
    gv = dm.download(L.ARR_VOLGRAD)
    assert rel_err(g, want["grad"]) <= TOL
    volgrad_close(gv, want["vol_grad"], pos)
    rp = dm.eval(dm.options(mods, constraint_mode=0))
    lam = float(np.vdot(want["grad"], want["vol_grad"]) / np.vdot(want["vol_grad"], want["vol_grad"]))
    assert abs(rp.kkt_lambda - lam) <= 1e-10 * abs(lam)
    assert rel_err(dm.download(L.ARR_GRAD), want["grad"] - lam * want["vol_grad"]) <= TOL
    dm.close()


def test_bending_cube_r8_vs_oracle(L):
    """BASELINE.json configs[2] at its stated size: the cube of meshes/bending_cube.yaml refined to
    24 * 4^8 = 1 572 864 facets (array refinement, geometry/refine.py), jittered so that no vertex is flat;
    Helfrich bending + volume against the oracle."""
    from membrane_solver_b200.geometry.refine import cube_mesh, refine_triangles
    from oracle import ref_modules as ref

    pos, tri = cube_mesh()
    for _ in range(8):
        pos, tri, _, _ = refine_triangles(pos, tri)
    nv, nf = pos.shape[0], tri.shape[0]
    assert nf == 1_572_864
    rng = np.random.default_rng(8)
    pos = pos + 2.0e-4 * rng.normal(size=pos.shape)
    want = ref.fused_surface_bending_volume(pos, tri, np.zeros(nf), 1.0, 0.0, np.zeros(nv, bool))
    dm = _ctx(nv, tri, body_mask=np.ones(nf, np.uint8), order_hint=pos)  # refinement order -> Morton order inside
    dm.set_surface_tension(0.0)
    dm.set_bending_params(1.0, 0.0)
    dm.set_positions(pos)
    r = dm.eval(dm.options(L.MOD_BENDING | L.MOD_VOLUME))
    _scalar_close(r.e_bending, want["E_bending"])
    _scalar_close(r.volume, want["volume"])
    assert rel_err(dm.download(L.ARR_GRAD), want["grad"]) <= 2e-12
    volgrad_close(dm.download(L.ARR_VOLGRAD), want["vol_grad"], pos)
    dm.close()


def _sample_submeshes(tri, nv, n_seeds, radius, rng):
    """Around each random seed vertex: the vertices within `radius` rings (the sample rows S0) and the facets touching
    S0 or a neighbour of S0 -- everything the gradient rows of S0 depend on (seeds of the 1-ring need the 2-ring)."""
    order = np.argsort(tri.reshape(-1), kind="stable")
    corner_vertex = tri.reshape(-1)[order]
    ptr = np.searchsorted(corner_vertex, np.arange(nv + 1))
    facet_of = order // 3

    def facets_of(vs):
        return np.unique(np.concatenate([facet_of[ptr[v]:ptr[v + 1]] for v in vs]))

    for seed in rng.integers(0, nv, size=n_seeds):
        s0 = np.array([seed])
        for _ in range(radius):
            s0 = np.unique(tri[facets_of(s0)].reshape(-1))
        s1 = np.unique(tri[facets_of(s0)].reshape(-1))
        f = facets_of(s1)
        yield s0, f


def test_ten_million_facets_sampled_patches_vs_oracle(L):
    """BASELINE.json configs[4] at 10 025 280 facets: the oracle cannot run on the whole mesh, so it runs on 48
    random sub-meshes (each the closure the gradient rows of its sample vertices depend on) and the sampled
    gradient / dV/dx rows of the full-size device evaluation must agree at 1e-12 relative to the mesh-wide scale."""
    from membrane_solver_b200.synthetic import frequency_for_facets, icosphere
    from oracle import ref_modules as ref

    pos, tri = icosphere(frequency_for_facets(10_000_000))
    nv, nf = pos.shape[0], tri.shape[0]
    dm = _ctx(nv, tri, body_mask=np.ones(nf, np.uint8))
    dm.set_bending_params(1.0, 0.05)
    dm.set_positions(pos)
    dm.eval(dm.options(L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME))
    g = dm.download(L.ARR_GRAD)
    gv = dm.download(L.ARR_VOLGRAD)
    dm.close()
    g_scale, gv_scale = np.abs(g).max(), np.abs(gv).max()
    rng = np.random.default_rng(2026)
    n_rows = 0
    for s0, f in _sample_submeshes(tri, nv, 48, 4, rng):
        verts, local = np.unique(tri[f].reshape(-1), return_inverse=True)
        sub_tri = local.reshape(-1, 3).astype(np.int32)
        want = ref.fused_surface_bending_volume(pos[verts], sub_tri, np.ones(len(f)), 1.0, 0.05,
                                                np.zeros(len(verts), bool))
        rows = np.searchsorted(verts, s0)
        assert np.abs(g[s0] - want["grad"][rows]).max() <= TOL * g_scale
        assert np.abs(gv[s0] - want["vol_grad"][rows]).max() <= max(1e-10 * gv_scale, 0.0)
        assert np.abs(gv[s0] - want["vol_grad"][rows]).max() <= TOL * float((pos ** 2).sum(axis=1).max()) / 6.0
        n_rows += len(s0)
    assert n_rows >= 48 * 30


def test_pipelined_host_evaluation_matches_staged_path(L):
    """ms_ctx_eval_host on a large mesh overlaps the chunked position upload with the patch kernels
    (patches launched in the order their rows arrive).  The per-vertex sums do not depend on the launch
    order, so the raw gradients are BITWISE those of upload -> ms_ctx_eval -> ms_ctx_get_array; the
    scalars are summed over a different number of per-CTA rows (rounding only)."""
    from membrane_solver_b200.synthetic import icosphere

    pos, tri = icosphere(330)    # 1.09 M facets, 545 k vertices: above the pipelining threshold
    nv, nf = pos.shape[0], tri.shape[0]
    rng = np.random.default_rng(11)
    pos = pos * (1.0 + 0.01 * rng.standard_normal((nv, 1)))
    dm = _ctx(nv, tri, body_mask=np.ones(nf, np.uint8), fixed_mask=(rng.random(nv) < 0.05).astype(np.uint8))
    kappa, c0 = 1.0 + 0.3 * rng.random(nv), 0.05 * rng.random(nv)
    gamma = 1.0 + 0.2 * rng.random(nf)
    sbv = L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME
    # (modules, options, per-vertex kappa / c0, per-facet gamma)
    for mods, kw, per_vertex, per_facet in (
            (sbv, {}, False, False),
            (sbv, dict(constraint_mode=0), False, False),
            (L.MOD_SURFACE | L.MOD_VOLUME, {}, False, False),
            (sbv, dict(want_grad=0), False, False),
            (sbv, {}, True, False),                                 # kind 3 through the pipeline
            (L.MOD_SURFACE | L.MOD_VOLUME, {}, False, True),        # kind 0 pass B summing the scalars itself
            (sbv, dict(use_trial=1), False, False),                 # the rows travel into the trial positions
            (sbv, dict(constraint_mode=1, k_vol=2.0, v_target=3.9, apply_fixed=1), False, False)):
        dm.set_bending_params(kappa if per_vertex else 1.3, c0 if per_vertex else 0.02)
        dm.set_surface_tension(gamma if per_facet else 1.0)
        opts = dm.options(mods, **kw)
        target = L.ARR_TRIAL if kw.get("use_trial") else L.ARR_POSITIONS
        dm.upload(target, pos)
        want = dm.eval(opts)
        want_g, want_v = dm.download(L.ARR_GRAD), dm.download(L.ARR_VOLGRAD)
        dm.upload(target, np.zeros_like(pos))      # the pipelined call must bring every row itself
        g, v = np.full_like(pos, np.nan), np.full_like(pos, np.nan)
        got = dm.eval_host(opts, pos, grad=g, volgrad=v)
        for name in ("e_surface", "e_bending", "area", "volume"):
            _scalar_close(getattr(got, name), getattr(want, name))
        if kw.get("want_grad", 1):
            if "constraint_mode" in kw:
                assert rel_err(g, want_g) <= 1e-12      # the coefficient comes from the re-grouped sums
            else:
                assert np.array_equal(g, want_g)
            assert np.array_equal(v, want_v)
            g2 = np.empty_like(pos)
            dm.eval_host(opts, pos, grad=g2)
            assert np.array_equal(g2, g)               # and it repeats bitwise
        assert np.array_equal(dm.download(target), pos)
    dm.close()


def test_split_interior_boundary_evaluation(L):
    """Partition context (owned + ghost rows): evaluating the interior patches and the patches that
    read ghost rows as two launches gives the same gradients bit for bit, and the same scalars up to
    the summation order of the per-CTA partial sums."""
    from membrane_solver_b200.context import DeviceMesh
    from membrane_solver_b200.partition import split_mesh
    from membrane_solver_b200.synthetic import icosphere

    pos, tri = icosphere(90)
    lm = split_mesh(pos.shape[0], tri, 2, 0)
    rows = lm.global_rows()
    dm = DeviceMesh(0)
    dm.set_topology(lm.nv_local, lm.tri, n_owned=lm.n_owned, body_mask=np.ones(lm.tri.shape[0], np.uint8))
    dm.set_surface_tension(1.0)
    dm.set_bending_params(1.0, 0.1)
    dm.set_positions(pos[rows])
    mods = L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME
    full = dm.options(mods)
    # reference: the whole partition in one launch per pass (ghost seeds: take them from a full-mesh run)
    whole = _ctx(pos.shape[0], tri, body_mask=np.ones(tri.shape[0], np.uint8))
    whole.set_surface_tension(1.0)
    whole.set_bending_params(1.0, 0.1)
    whole.set_positions(pos)
    whole.eval(whole.options(mods))
    seeds_all = whole.download(L.ARR_SEEDS)

    def run(parts):
        for o in parts:
            dm.eval_pass_a(o)
        s = dm.download(L.ARR_SEEDS)
        s[lm.n_owned:] = seeds_all[rows[lm.n_owned:]]          # what the seed halo exchange delivers
        dm.upload(L.ARR_SEEDS, s)
        for o in parts:
            dm.eval_pass_b(o)
        dm.eval_reduce(parts[-1])
        sc = dm.read_scalars().scalars.copy()
        return sc, dm.download(L.ARR_GRAD)[:lm.n_owned], dm.download(L.ARR_VOLGRAD)[:lm.n_owned]

    sc1, g1, v1 = run([full])
    inner, outer = dm.options(mods, patch_count=L.PATCHES_INTERIOR), dm.options(mods, patch_count=L.PATCHES_BOUNDARY)
    sc2, g2, v2 = run([inner, outer])
    assert np.array_equal(g1, g2) and np.array_equal(v1, v2)
    assert np.allclose(sc1[:12], sc2[:12], rtol=1e-13, atol=0)
    # and the owned rows agree with the single-context evaluation of the whole mesh
    assert rel_err(g1, whole.download(L.ARR_GRAD)[rows[:lm.n_owned]]) <= 1e-13
    dm.close()
    whole.close()


def test_random_soups_with_repeated_and_wild_indices(L):
    """Random triangle soups through the PATCH path: repeated vertices inside a facet, facets listed
    twice, out-of-range indices, isolated vertices, a very high valence vertex -- against the oracle."""
    from oracle import ref_modules as ref

    rng = np.random.default_rng(123)
    for trial in range(6):
        nv = int(rng.integers(40, 400))
        nf = int(rng.integers(nv, 3 * nv))                             # mean valence 3..9, tails to ~25
        pos = rng.normal(size=(nv, 3))
        tri = rng.integers(0, nv - 5, size=(nf, 3)).astype(np.int32)   # the last 5 vertices stay isolated
        tri[rng.integers(0, nf, 8), 1] = tri[rng.integers(0, nf, 8), 0]   # some facets name a vertex twice ...
        rep = rng.integers(0, nf, 5)
        tri[rep, 1] = tri[rep, 0]                                           # ... for sure
        tri[rng.integers(0, nf, 4)] = tri[rng.integers(0, nf, 4)]           # duplicated facets
        tri[:28, 0] = 3                                                     # a hub of valence ~30 (needs narrow rounds)
        bad = tri.copy()
        bad[1, 2] = nv + 7
        bad[2, 0] = -3
        gamma = 0.5 + rng.random(nf)
        for t in (tri, bad):
            ok = np.all((t >= 0) & (t < nv), axis=1)
            tv, gv = np.ascontiguousarray(t[ok]), gamma[ok]
            for is_b in (ref.boundary_mask_from_triangles(tv, nv), np.zeros(nv, bool)):
                want_g = np.zeros_like(pos)
                e_s = ref.surface_energy_and_gradient(pos, tv, gv, want_g)
                e_b = ref.bending_energy_and_gradient(pos, tv, 1.3, 0.2, is_b, want_g)
                dm = _ctx(nv, t, is_boundary=is_b.astype(np.uint8) if is_b.any() else None,
                          body_mask=np.ones(nf, np.uint8), threads=32 * int(rng.integers(1, 4)), max_owned=64,
                          max_local=600)
                dm.set_surface_tension(gamma)
                dm.set_bending_params(1.3, 0.2)
                grad = np.empty_like(pos)
                r = dm.eval_host(dm.options(L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME), pos, grad=grad)
                _scalar_close(r.e_surface, e_s, 1e-12)
                _scalar_close(r.e_bending, e_b, 1e-11)
                _scalar_close(r.volume, ref.body_volume(pos, tv), 1e-12)
                assert rel_err(grad, want_g) <= 1e-11
                dm.close()


@pytest.mark.parametrize("seed", [1, 2])
def test_odd_topologies_through_the_c_abi(L, seed):
    """The mesh of tests/test_emulator.py::test_odd_topologies_against_the_oracle with a fan of valence 30 (more rounds
    than a 96-lane patch can hold: ms_ctx_set_topology narrows the rounds), unused vertices, degenerate and duplicated
    facets, two components, random vertex order, per-facet surface tension and a partial body -- with and without the
    internal Morton re-ordering -- against the oracle at 1e-12."""
    import ms_test_helpers as H

    pos, tri, gamma, body, (want_e, want_g, want_v, want_vg) = H.odd_mesh(seed, nfan=30)
    for hint in (None, pos):
        dm = _ctx(pos.shape[0], tri, body_mask=body, order_hint=hint)
        dm.set_surface_tension(gamma)
        dm.set_positions(pos)
        res = dm.eval(dm.options(L.MOD_SURFACE | L.MOD_VOLUME))
        assert abs(res.e_surface - want_e) <= 1e-12 * abs(want_e)
        assert abs(res.volume - want_v) <= 1e-12 * max(1.0, abs(want_v))
        assert rel_err(dm.download(L.ARR_GRAD), want_g) <= 1e-12
        assert rel_err(dm.download(L.ARR_VOLGRAD), want_vg) <= 1e-12
        assert dm.pack_info()["threads"] < 96        # the fan forced narrower rounds
        dm.close()
