"""The small kernels of the device-resident minimiser loop and the deferred gradient projection, against a plain
float64 NumPy reference of each ABI call (``math.fsum`` for the dot products).

Every scenario is one script run against a mesh object: ``FakeDeviceMesh`` (tests/fake_device.py, the NumPy
restatement the CPU tier of the minimiser tests relies on) in the CPU tier, ``DeviceMesh`` over libms_b200.so in
the GPU tier, so the fake is held to the same reference as the kernels.

The meshes are chosen where reductions and grids go wrong: facet counts at warp and CTA edges, ``3 nv`` around
multiples of the 592 fixed chunks of ``k_dots`` and far above 592 x 256 (every chunk loops), the shortest edge and
the largest direction row planted in the first, the last and a warp-edge slot, with and without the internal
(Morton) vertex order and a fixed mask."""

import math

import numpy as np
import pytest


from fake_device import FakeDeviceMesh
from membrane_solver_b200 import _lib as L
from membrane_solver_b200.runtime.device_minimizer import DeviceMinimizer
from membrane_solver_b200.synthetic import icosphere, sfc_order, tangent_tilts

EPS = np.finfo(np.float64).eps
BACKENDS = [pytest.param("emulator", id="emulator"), pytest.param("gpu", id="gpu", marks=pytest.mark.gpu)]


def _device(backend):
    if backend == "emulator":
        return FakeDeviceMesh(0)
    from membrane_solver_b200.context import DeviceMesh

    if L.device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu tier must run on the B200 box")
    return DeviceMesh(0)


@pytest.fixture
def dm(backend):
    d = _device(backend)
    yield d
    d.close()


def _load(dm, pos, tri, *, fixed=None, body=None, hint=False):
    dm.set_topology(len(pos), tri, fixed_mask=fixed, body_mask=body, order_hint=pos if hint else None)
    dm.set_positions(pos)
    if hint:  # a mesh already in Morton order would leave the internal order the identity
        identity = np.arange(len(pos))
        assert not np.array_equal(sfc_order(pos, tri)[2], identity), "the order hint would not move any vertex"
        if not isinstance(dm, FakeDeviceMesh):  # the emulator keeps the caller's order
            assert not np.array_equal(dm.permutation(), identity)


def _write_through_device_ptr(dm, which, values):
    """Overwrite a (nv,3) array through ``ms_ctx_device_ptr`` (internal row order)."""
    internal = np.ascontiguousarray(values[dm.permutation()])
    view = dm.device_view(which)
    if isinstance(view, np.ndarray):  # the fake hands out its own array
        view[...] = internal
        return
    import torch

    dm.sync()
    torch.as_tensor(view, device=f"cuda:{dm.device}").copy_(torch.from_numpy(internal))
    torch.cuda.synchronize(dm.device)


# ---- the float64 reference ---------------------------------------------------------------------------------------
def fdot(a, b):
    return math.fsum((np.asarray(a) * np.asarray(b)).ravel())


def fdot_bound(a, b):
    """Allowed error of a dot product: 1e-13 * sum |a_i b_i|."""
    return 1e-13 * math.fsum(np.abs(np.asarray(a) * np.asarray(b)).ravel())


def ref_min_edge(pos, tri):
    if len(tri) == 0:
        return 0.0
    p = pos[tri]
    e = np.concatenate([p[:, 2] - p[:, 1], p[:, 0] - p[:, 2], p[:, 1] - p[:, 0]])
    return float(np.sqrt((e * e).sum(axis=1).min()))


def ref_max_row(d):
    return float(np.sqrt((d * d).sum(axis=1).max()))


def ref_normal_change_ok(pos, trial, tri, limit):
    """A facet with |n0| > 1e-12 fails when |n1| < 1e-12, when cos(angle) < cos(limit), or when its trial normal is
    NaN; the step is fine when no facet fails."""
    def normals(p):
        return np.cross(p[tri[:, 1]] - p[tri[:, 0]], p[tri[:, 2]] - p[tri[:, 0]])

    n0, n1 = normals(pos), normals(trial)
    ok = True
    for a, b in zip(n0, n1):
        m0, m1 = math.sqrt(fdot(a, a)), math.sqrt(fdot(b, b)) if np.all(np.isfinite(b)) else math.nan
        if not m0 > 1e-12:
            continue
        if m1 < 1e-12 or not fdot(a, b) / (m0 * m1) >= math.cos(limit):
            ok = False
    return ok


def ref_cg_direction(g, pg, pd, fixed):
    """Per-vertex Polak-Ribiere: beta = g.(g - pg) / (pg.pg + 1e-20); d = -g + beta pd, or -g where beta < 0;
    fixed rows zero.  Also returns beta and the error scale of each row."""
    nv = len(g)
    d = np.empty_like(g)
    beta = np.empty(nv)
    scale = np.empty(nv)
    for v in range(nv):
        den = fdot(pg[v], pg[v]) + 1e-20
        beta[v] = fdot(g[v], g[v] - pg[v]) / den
        d[v] = -g[v] + beta[v] * pd[v] if beta[v] >= 0.0 else -g[v]
        cond = math.fsum(np.abs(g[v] * (g[v] - pg[v]))) / den
        scale[v] = np.linalg.norm(g[v]) + (abs(beta[v]) + cond) * np.linalg.norm(pd[v])
    if fixed is not None:
        d[fixed.astype(bool)] = 0.0
        scale[fixed.astype(bool)] = 0.0
    return d, beta, scale


def ref_projection(g, gc, volume, fixed, mode, k_vol=0.0, v_target=0.0):
    """P = g + coef gC with fixed rows zeroed; Lagrange coef = -<g,gC>/<gC,gC>, penalty coef = k_vol (V - V0)."""
    coef = -fdot(g, gc) / fdot(gc, gc) if mode == "lagrange" else k_vol * (volume - v_target)
    p = g + coef * gc
    if fixed is not None:
        p[fixed.astype(bool)] = 0.0
    return p, coef


def assert_ulps(got, want, ulps, what):
    err = abs(got - want)
    assert err <= ulps * EPS * abs(want), f"{what}: got {got!r}, want {want!r} ({err / (EPS * abs(want)):.1f} ulp)"


def assert_dot(got, a, b, what):
    want, tol = fdot(a, b), fdot_bound(a, b)
    assert abs(got - want) <= tol, f"{what}: got {got!r}, fsum {want!r}, |diff| {abs(got - want):.3e} > {tol:.3e}"


# ---- meshes ------------------------------------------------------------------------------------------------------
def _soup(nf, nv, seed):
    """``nf`` disjoint near-equilateral facets (edges 0.7 .. 1.3, bent out of plane) scattered in a box, plus
    unused vertices up to ``nv``: every facet owns its vertices, so one facet can be changed alone."""
    rng = np.random.default_rng(seed)
    base = np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.5, math.sqrt(3.0) / 2.0, 0.0]])
    pts = base[None] + rng.uniform(-50.0, 50.0, (nf, 1, 3)) + 0.05 * rng.normal(size=(nf, 3, 3))
    extra = rng.uniform(-50.0, 50.0, (nv - 3 * nf, 3))
    pos = np.concatenate([pts.reshape(-1, 3), extra])
    return pos, np.arange(3 * nf, dtype=np.int32).reshape(nf, 3)


# (nf, nv): facet counts at warp / CTA edges; 3 nv around the 592 dot chunks (3 * 197 = 591, 3 * 198 = 594,
# 3 * 592 = 1776 = 3 chunks each) and far above 592 * 256 so that every chunk loops
SIZES = [(1, 3), (31, 93), (32, 96), (33, 99), (255, 765), (256, 768), (257, 771), (4000, 12000),
         (65, 197), (66, 198), (197, 591), (197, 592), (197, 593), (116_666, 350_000)]


def _slot(n, where, width=32):
    """first / last / warp: the last lane of the last full warp (the lane before a partial one), mid-warp if none."""
    if where == "first":
        return 0
    if where == "last":
        return n - 1
    return width * (n // width) - 1 if n >= width else n // 2


# ---- 1. line-search statistics -----------------------------------------------------------------------------------
@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("fixed", [False, True], ids=["free", "fixed"])
@pytest.mark.parametrize("hint", [False, True], ids=["caller_order", "order_hint"])
@pytest.mark.parametrize("where", ["first", "last", "warp"])
@pytest.mark.parametrize("nf,nv", SIZES, ids=[f"nf{a}_nv{b}" for a, b in SIZES])
def test_line_search_stats(dm, backend, nf, nv, where, hint, fixed):
    rng = np.random.default_rng(nf * 7 + nv)
    pos, tri = _soup(nf, nv, seed=nv)
    f = _slot(nf, where)
    a, b = tri[f, (f + 1) % 3], tri[f, (f + 2) % 3]  # edge e_(f % 3) of facet f: the unique shortest edge
    u = (pos[b] - pos[a]) / np.linalg.norm(pos[b] - pos[a])
    pos[b] = pos[a] + 0.01 * u
    fx = (rng.uniform(size=nv) < 0.2).astype(np.uint8) if fixed else None
    _load(dm, pos, tri, fixed=fx, hint=hint)
    perm = dm.permutation()
    mid_warp = min(32 * ((nv - 1) // 64) + 13, nv - 1)
    row = {"first": 0, "last": nv - 1, "warp": mid_warp}[where]  # internal row of the largest direction row
    d = rng.normal(size=(nv, 3))
    d /= np.linalg.norm(d, axis=1)[:, None] * rng.uniform(1.0, 2.0, size=(nv, 1))
    d[perm[row]] = 3.0 * d[perm[row]] / np.linalg.norm(d[perm[row]])
    if fixed:  # a pending fixed-row projection: the dot products run the projected kernel
        dm.eval(dm.options(L.MOD_SURFACE, want_grad=True))
        g = dm.download(L.ARR_GRAD)
        dm.eval(dm.options(L.MOD_SURFACE, want_grad=True, apply_fixed=True))
        g[fx.astype(bool)] = 0.0
    else:
        g = rng.normal(size=(nv, 3))
        dm.upload(L.ARR_GRAD, g)
    dm.set_direction(d)
    min_edge, max_dir, g_d, g_g = stats = dm.line_search_stats()
    assert_ulps(min_edge, ref_min_edge(pos, tri), 4, "min edge")
    assert abs(min_edge - 0.01) < 1e-9
    assert_ulps(max_dir, ref_max_row(d), 4, "max direction row")
    assert abs(max_dir - 3.0) < 1e-12
    assert_dot(g_d, g, d, "<g,d>")
    assert_dot(g_g, g, g, "<g,g>")
    assert dm.line_search_stats() == stats  # bitwise repeatable


@pytest.mark.parametrize("backend", BACKENDS)
def test_line_search_stats_without_facets(dm, backend):
    rng = np.random.default_rng(5)
    pos = rng.normal(size=(40, 3))
    _load(dm, pos, np.zeros((0, 3), np.int32))
    d, g = rng.normal(size=(40, 3)), rng.normal(size=(40, 3))
    dm.upload(L.ARR_GRAD, g)
    dm.set_direction(d)
    min_edge, max_dir, g_d, g_g = dm.line_search_stats()
    assert min_edge == 0.0
    assert_ulps(max_dir, ref_max_row(d), 4, "max direction row")
    assert_dot(g_d, g, d, "<g,d>")
    assert_dot(g_g, g, g, "<g,g>")


# ---- 2. normal-change guard --------------------------------------------------------------------------------------
def _rotated(p3, angle):
    """The facet's three points turned by `angle` about an in-plane axis through their centroid: the normal turns
    by exactly `angle`."""
    c = p3.mean(axis=0)
    n = np.cross(p3[1] - p3[0], p3[2] - p3[0])
    n /= np.linalg.norm(n)
    k = (p3[1] - p3[0]) / np.linalg.norm(p3[1] - p3[0])
    k = k - (k @ n) * n
    k /= np.linalg.norm(k)
    x = p3 - c
    rot = (x * math.cos(angle) + np.cross(k, x) * math.sin(angle) + np.outer(x @ k, k) * (1.0 - math.cos(angle)))
    return c + rot


NC_NF = 1000  # 31 full warps and a partial one of 8 facets
NC_SLOTS = {"first_warp": 3, "middle_warp": 500, "last_partial_warp": 997}


def _normal_case(case, f, limit):
    """(pos, trial, tri, expected ok) with facet f affected as `case` says and every other facet turned slightly."""
    rng = np.random.default_rng(f)
    pos, tri = _soup(NC_NF, 3 * NC_NF, seed=11)
    pos[:, 2] = 0.0  # flat
    trial = pos + 1e-4 * rng.normal(size=pos.shape)  # turns of ~1e-4 rad everywhere else
    v = tri[f]
    p3 = pos[v].copy()
    if case == "turn_below":
        trial[v], ok = _rotated(p3, limit - 1e-6), True
    elif case == "turn_above":
        trial[v], ok = _rotated(p3, limit + 1e-6), False
    elif case == "line":  # collapsed to a line
        trial[v] = p3
        trial[v[2]] = 0.5 * (p3[0] + p3[1])
        ok = False
    elif case == "shrunk":  # |n1| ~ 1e-14: collapsed, yet the normal keeps its direction
        trial[v] = p3.mean(axis=0) + 1e-7 * (p3 - p3.mean(axis=0))
        ok = False
    elif case == "flip":
        trial[v], ok = _rotated(p3, math.pi), False
    elif case == "degenerate_before":  # not judged: |n0| <= 1e-12
        pos[v[2]] = 0.5 * (p3[0] + p3[1])
        trial[v], ok = _rotated(p3, math.pi), True
    elif case == "nan":
        trial[v] = p3
        trial[v[1], 0] = math.nan
        ok = False
    return pos, trial, tri, ok


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("limit", [0.1, 0.5, 2.0])
@pytest.mark.parametrize("slot", list(NC_SLOTS))
@pytest.mark.parametrize("case", ["turn_below", "turn_above", "line", "shrunk", "flip", "degenerate_before", "nan"])
def test_normal_change_guard(dm, backend, case, slot, limit):
    pos, trial, tri, ok = _normal_case(case, NC_SLOTS[slot], limit)
    assert ref_normal_change_ok(pos, trial, tri, limit) == ok
    _load(dm, pos, tri)
    dm.upload(L.ARR_TRIAL, trial)
    assert dm.normal_change_ok(limit) == ok
    # the untouched mesh passes: only the planted facet decides
    dm.upload(L.ARR_TRIAL, pos + 1e-4 * np.random.default_rng(1).normal(size=pos.shape))
    assert dm.normal_change_ok(limit)


@pytest.mark.parametrize("backend", BACKENDS)
def test_normal_change_limit_range(dm, backend):
    """At limit = pi every finite turn passes and a NaN still fails; limits outside [0, pi] are refused."""
    f = NC_SLOTS["last_partial_warp"]
    pos, trial, tri, _ = _normal_case("nan", f, math.pi)
    _load(dm, pos, tri)
    dm.upload(L.ARR_TRIAL, trial)
    assert not dm.normal_change_ok(math.pi)
    trial[tri[f]] = _rotated(pos[tri[f]], 3.0)
    dm.upload(L.ARR_TRIAL, trial)
    assert dm.normal_change_ok(math.pi)
    assert not dm.normal_change_ok(2.9)
    for bad in (math.pi + 1e-3, -1e-3, 7.0, math.nan):
        with pytest.raises(L.B200Error):
            dm.normal_change_ok(bad)


# ---- 3. conjugate-gradient direction -----------------------------------------------------------------------------
def _cg_rows(nv, rng):
    """previous gradient pg, previous direction pd and gradient g whose rows give beta > 0, beta < 0, beta = 0, and
    pg = 0 (the 1e-20 guard, with and without g = 0)."""
    pg = rng.normal(size=(nv, 3))
    pd = rng.normal(size=(nv, 3))
    noise = 0.1 * rng.normal(size=(nv, 3))
    kind = np.arange(nv) % 5
    g = np.where((kind == 0)[:, None], 1.5 * pg + noise, 0.5 * pg + noise)  # beta > 0 / beta < 0
    g[kind == 2] = pg[kind == 2]                                          # beta == 0 exactly
    pg[kind == 3] = 0.0                                                   # pg == 0: beta = |g|^2 * 1e20
    pg[kind == 4] = 0.0                                                   # pg == 0 and g == 0: beta = 0
    g[kind == 4] = 0.0
    return g, pg, pd


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("hint", [False, True], ids=["caller_order", "order_hint"])
def test_cg_direction(dm, backend, hint):
    rng = np.random.default_rng(21)
    nf, nv = 333, 1003
    pos, tri = _soup(nf, nv, seed=21)
    fx = (rng.uniform(size=nv) < 0.15).astype(np.uint8)
    _load(dm, pos, tri, fixed=fx, hint=hint)
    g, pg, pd = _cg_rows(nv, rng)
    dm.upload(L.ARR_GRAD, pg)
    dm.set_direction(pd)
    dm.cg_commit()
    dm.upload(L.ARR_GRAD, g)
    dm.cg_direction(False)
    got = dm.download(L.ARR_DIRECTION)
    want, beta, scale = ref_cg_direction(g, pg, pd, fx)
    free = ~fx.astype(bool)
    assert (beta[free] > 0).any() and (beta[free] < 0).any() and (beta[free] == 0).any()
    err = np.linalg.norm(got - want, axis=1)
    assert np.all(err <= 1e-14 * scale), (np.argmax(err - 1e-14 * scale), err.max())
    assert np.all(got[fx.astype(bool)] == 0.0)
    assert np.all(np.isfinite(got))
    # restart: -g as stored, whatever the history
    dm.cg_direction(True)
    assert np.array_equal(dm.download(L.ARR_DIRECTION), -g)
    # a new topology drops the history: the next direction is -g
    _load(dm, pos, tri, fixed=fx, hint=hint)
    dm.upload(L.ARR_GRAD, g)
    dm.cg_direction(False)
    assert np.array_equal(dm.download(L.ARR_DIRECTION), -g)


# ---- 4. the deferred projection as a state machine ---------------------------------------------------------------
INTERMEDIATES = ["none", "energy_only", "line_search_stats", "set_fixed_mask", "upload_volgrad", "axpy_volgrad",
                 "device_ptr_volgrad"]
CONSUMERS = ["direction", "line_search_stats", "dots", "download"]
K_VOL = 3.0


def _projection_setup(dm, mode, hint, modules=L.MOD_SURFACE | L.MOD_VOLUME):
    """Mesh with a fixed cap, raw g / gC / V of an evaluation without projection, then the evaluation with the
    projection pending.  Returns the state the consumers are checked against."""
    pos, tri = icosphere(6, reorder=False)  # not in Morton order: the order hint permutes the rows
    nv = len(pos)
    fx = (pos[:, 2] > 0.7).astype(np.uint8)
    _load(dm, pos, tri, fixed=fx, body=np.ones(len(tri), np.uint8), hint=hint)
    d0 = np.random.default_rng(3).normal(size=(nv, 3))
    dm.set_direction(d0)
    dm.make_trial(1e-3)
    raw = dm.eval(dm.options(modules, want_grad=True))
    g, gc = dm.download(L.ARR_GRAD), dm.download(L.ARR_VOLGRAD)
    v_target = 0.97 * raw.volume
    opts = dict(constraint_mode={"lagrange": 0, "penalty": 1}[mode], k_vol=K_VOL, v_target=v_target)
    dm.eval(dm.options(modules, want_grad=True, apply_fixed=True, **opts))
    p, coef = ref_projection(g, gc, raw.volume, fx, mode, K_VOL, v_target)
    return dict(pos=pos, tri=tri, fixed=fx, d0=d0, g=g, gc=gc, p=p, coef=coef, opts=opts, modules=modules)


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("hint", [False, True], ids=["caller_order", "order_hint"])
@pytest.mark.parametrize("consumer", CONSUMERS)
@pytest.mark.parametrize("between", INTERMEDIATES)
@pytest.mark.parametrize("mode", ["lagrange", "penalty"])
def test_deferred_projection(dm, backend, mode, between, consumer, hint):
    s = _projection_setup(dm, mode, hint)
    p, gc, d0 = s["p"], s["gc"], s["d0"]
    new_gc = np.random.default_rng(8).normal(size=gc.shape)
    if between == "energy_only":
        dm.eval(dm.options(s["modules"], want_grad=False, apply_fixed=True, **s["opts"]))
        dm.eval(dm.options(s["modules"], want_grad=False, apply_fixed=True, use_trial=True, **s["opts"]))
    elif between == "line_search_stats":
        dm.line_search_stats()
    elif between == "set_fixed_mask":  # the pending projection keeps the mask it was asked with
        dm.set_fixed_mask((s["pos"][:, 2] < -0.7).astype(np.uint8))
    elif between == "upload_volgrad":
        dm.upload(L.ARR_VOLGRAD, new_gc)
        gc = new_gc
    elif between == "axpy_volgrad":
        dm.axpy(L.ARR_VOLGRAD, L.ARR_DIRECTION, 0.5, skip_fixed=False)
        gc = gc + 0.5 * d0
    elif between == "device_ptr_volgrad":
        _write_through_device_ptr(dm, L.ARR_VOLGRAD, new_gc)
        gc = new_gc
    tol = 1e-12 * (np.abs(s["g"]).max() + abs(s["coef"]) * np.abs(s["gc"]).max())
    if consumer == "direction":
        dm.direction_from_gradient(-0.75)
        got = dm.download(L.ARR_DIRECTION)
        assert np.abs(got - (-0.75 * p)).max() <= tol
    elif consumer == "line_search_stats":
        _, _, g_d, g_g = dm.line_search_stats()
        assert abs(g_d - fdot(p, d0)) <= 1e-12 * math.fsum(np.abs(p * d0).ravel())
        assert abs(g_g - fdot(p, p)) <= 1e-12 * fdot(p, p)
    elif consumer == "dots":
        dm.dots()
        sc = dm.read_scalars().scalars
        assert abs(sc[L.SC_G_G] - fdot(p, p)) <= 1e-12 * fdot(p, p)
        assert abs(sc[L.SC_G_GC] - fdot(p, gc)) <= 1e-12 * math.fsum(np.abs(p * gc).ravel())
        assert abs(sc[L.SC_GC_GC] - fdot(gc, gc)) <= 1e-13 * fdot(gc, gc)
    else:
        got = dm.download(L.ARR_GRAD)
        assert np.abs(got - p).max() <= tol, np.abs(got - p).max()
        assert np.all(got[s["fixed"].astype(bool)] == 0.0)


@pytest.mark.parametrize("backend", BACKENDS)
def test_tilt_only_evaluation_replaces_the_gradients(dm, backend):
    """A tilt-only evaluation (MS_MOD_TILT, want_grad = 0, want_tilt_grad = 1) runs pass B: MS_ARR_GRAD and
    MS_ARR_VOLGRAD then hold the raw gradients of the modules, and the pending projection is gone."""
    pos, tri = icosphere(6)
    mods = L.MOD_SURFACE | L.MOD_VOLUME | L.MOD_TILT
    fx = (pos[:, 2] > 0.7).astype(np.uint8)
    _load(dm, pos, tri, fixed=fx, body=np.ones(len(tri), np.uint8))
    dm.set_tilt_rigidity(0.7)
    dm.set_tilts(tangent_tilts(pos, tri))
    dm.eval(dm.options(mods, want_grad=True))
    g, gc = dm.download(L.ARR_GRAD), dm.download(L.ARR_VOLGRAD)
    dm.eval(dm.options(mods, want_grad=True, constraint_mode=0, apply_fixed=True))
    dm.eval(dm.options(mods, want_grad=False, want_tilt_grad=True))
    got_g, got_gc = dm.download(L.ARR_GRAD), dm.download(L.ARR_VOLGRAD)
    assert np.abs(got_g - g).max() <= 1e-12 * np.abs(g).max()
    assert np.abs(got_gc - gc).max() <= 1e-12 * np.abs(gc).max()
    assert np.abs(got_g[fx.astype(bool)]).max() > 0.0  # not projected: the fixed rows keep their gradient


# ---- 5. axpy and trial moves -------------------------------------------------------------------------------------
def _ulp_close(got, y, alpha, x):
    """|got - (y + alpha x)| within one ulp of the result and of the product (fused or not)."""
    want = y + alpha * x
    return np.all(np.abs(got - want) <= np.spacing(np.abs(want)) + np.spacing(np.abs(alpha * x)))


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("skip_fixed", [False, True], ids=["all_rows", "skip_fixed"])
@pytest.mark.parametrize("src", [L.ARR_VOLGRAD, L.ARR_DIRECTION], ids=["src_volgrad", "src_direction"])
@pytest.mark.parametrize("dst", [L.ARR_POSITIONS, L.ARR_TRIAL, L.ARR_VOLGRAD],
                         ids=["dst_positions", "dst_trial", "dst_volgrad"])
def test_axpy_and_trial(dm, backend, dst, src, skip_fixed):
    rng = np.random.default_rng(31)
    nf, nv = 333, 1003
    pos, tri = _soup(nf, nv, seed=31)
    fx = (rng.uniform(size=nv) < 0.2).astype(np.uint8)
    _load(dm, pos, tri, fixed=fx, hint=True)  # the fixed mask is permuted with the rows
    d, gc = rng.normal(size=(nv, 3)), rng.normal(size=(nv, 3))
    dm.set_direction(d)
    dm.upload(L.ARR_VOLGRAD, gc)
    dm.make_trial(0.25)
    trial = dm.download(L.ARR_TRIAL)
    assert _ulp_close(trial, pos, 0.25, d)  # every row, the fixed ones included
    arrays = {L.ARR_POSITIONS: pos, L.ARR_TRIAL: trial, L.ARR_VOLGRAD: gc, L.ARR_DIRECTION: d}
    y, x = arrays[dst], arrays[src]
    alpha = -0.37
    dm.axpy(dst, src, alpha, skip_fixed=skip_fixed)
    got = dm.download(dst)
    moved = ~fx.astype(bool) if skip_fixed else np.ones(nv, bool)
    assert _ulp_close(got[moved], y[moved], alpha, x[moved])
    assert np.array_equal(got[~moved], y[~moved])
    dm.accept_trial()
    assert np.array_equal(dm.download(L.ARR_POSITIONS), dm.download(L.ARR_TRIAL))


# ---- 6. the loop at size -----------------------------------------------------------------------------------------
LOOP_FREQ = 56  # 62 720 facets


def _loop_run(backend, stepper):
    pos, tri = icosphere(LOOP_FREQ, reorder=False)  # not in Morton order: the order hint permutes the rows
    nf = len(tri)
    dm = _device(backend)
    try:
        fx = (pos[:, 2] > 0.85).astype(np.uint8)
        _load(dm, pos, tri, fixed=fx, body=np.ones(nf, np.uint8), hint=True)
        dm.set_surface_tension(1.0)
        dm.set_bending_params(0.05, 0.0)
        v0 = dm.eval(dm.options(L.MOD_VOLUME, want_grad=False)).volume
        mini = DeviceMinimizer(dm, L.MOD_SURFACE | L.MOD_BENDING, volume_mode="lagrange", v_target=0.98 * v0,
                               enforce_volume=True, stepper=stepper, step_size=1e-2)
        out = mini.minimize(n_steps=5)
        return mini.history, out, dm.download(L.ARR_POSITIONS)
    finally:
        dm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("stepper", ["gd", "cg"])
def test_loop_at_size_matches_emulator(stepper):
    """DeviceMinimizer with a Lagrange volume, its enforcement and a fixed cap on a 62 720-facet perturbed icosphere:
    the device (internal vertex order) against FakeDeviceMesh, per accepted energy, step and success, and the final
    positions at 1e-9.  The emulator side, which keeps the caller's vertex order, takes about 5 s per
    stepper on one CPU core."""
    h_ref, out_ref, pos_ref = _loop_run("emulator", stepper)
    h, out, pos = _loop_run("gpu", stepper)
    assert len(h) == len(h_ref) == 5
    assert any(s for *_, s in h)
    for (i, e, step, ok), (i_r, e_r, step_r, ok_r) in zip(h, h_ref):
        assert (i, ok) == (i_r, ok_r)
        assert abs(e - e_r) <= 1e-9 * abs(e_r), (i, e, e_r)
        assert abs(step - step_r) <= 1e-12 * step_r
    assert abs(out["energy"] - out_ref["energy"]) <= 1e-9 * abs(out_ref["energy"])
    assert np.abs(pos - pos_ref).max() <= 1e-9
