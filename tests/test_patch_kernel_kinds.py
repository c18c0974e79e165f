"""Every compile-time instantiation of the patch kernel ``k_patch<PASS, KIND, 448>``, every grid size and every launch
form, against a float64 reference assembled from ``oracle/ref_modules.py``.

The meshes are large enough that each persistent CTA works through several patches: that is where the kernel's
scheduling runs (the second input buffer, the ``bar_empty`` / ``bar_free`` waits from the third patch on, the mbarrier
parity flips, the consumer token ring carried from one patch to the next, the shared-memory accumulators zeroed by the
epilogue for the next patch).  The grid caps of ``ms_ctx_set_max_ctas`` put up to a few hundred patches on one CTA and
move the number of per-CTA rows that the last-CTA fold (``finalize_scalars``, 32 rows) and ``k_reduce_partials``
(64 rows) add up across their row-group edges.

CPU tier: every scenario through the host emulator (tests/emul, the same per-facet and per-vertex bodies and the same
packer) at the GPU tolerances, which checks the reference assembly and the packing at these sizes.  GPU tier: the same
scenarios through libms_b200.so, then the grid caps, the four launch forms and repeats against each other."""

import functools
from dataclasses import dataclass

import numpy as np
import pytest

import ms_test_helpers as H
from membrane_solver_b200 import _lib as L
from membrane_solver_b200.synthetic import icosphere, open_sheet, tangent_tilts
from ms_test_helpers import rel_err, volgrad_close
from oracle import ref_modules as ref

S, V, B, T, BT = L.MOD_SURFACE, L.MOD_VOLUME, L.MOD_BENDING, L.MOD_TILT, L.MOD_BENDING_TILT
TOL = 1e-12
GAMMA_U, KAPPA_U, C0_U, K_TILT = 1.2, 1.3, 0.05, 0.7
K_VOL, ALPHA = 3.0, 0.37
# threads=32: 14 consumer groups of 32 lanes instead of 4 of 96, and several times more patches
PACKS = {"default": {}, "narrow": dict(threads=32, max_owned=64, max_local=200)}
CAPS = [1, 2, 3, 31, 32, 33, 140, 1000]
FORMS = ["fused", "stages", "staged", "host"]


# ---- meshes ------------------------------------------------------------------------------------------------------
@dataclass
class Mesh:
    pos: np.ndarray
    tri: np.ndarray
    is_b: np.ndarray | None      # boundary flags (None: closed)
    hint: bool                   # set_topology with order_hint: the internal (Morton) order differs from the caller's
    gamma: np.ndarray            # per-facet surface tension
    kappa: np.ndarray            # per-vertex bending parameters
    c0: np.ndarray
    tilts: np.ndarray
    body: np.ndarray             # partial body (facet mask)
    fixed: np.ndarray            # fixed vertices
    direction: np.ndarray        # search direction of the trial positions x + ALPHA d


def _sheet(nx, ny):
    pos, tri = open_sheet(nx, ny, jitter=0.05)
    return pos, tri, ref.boundary_mask_from_triangles(tri, len(pos))


@functools.lru_cache(maxsize=None)
def mesh(name):
    is_b, hint = None, False
    if name == "ico120":          # 288 000 facets, closed
        pos, tri = icosphere(120)
    elif name == "ico60perm":     # 72 000 facets in random vertex order, packed in Morton order
        pos0, tri0 = icosphere(60, reorder=False)
        old_of_new = np.random.default_rng(7).permutation(len(pos0))
        new_of_old = np.empty_like(old_of_new)
        new_of_old[old_of_new] = np.arange(len(pos0))
        pos, tri, hint = np.ascontiguousarray(pos0[old_of_new]), new_of_old[tri0].astype(np.int32), True
    elif name == "sheet":         # 120 000 facets with a boundary
        pos, tri, is_b = _sheet(300, 200)
    elif name == "sheet65534":    # below the two-stage fixed-order sum of the bending-tilt stage (2^16 facets) ...
        pos, tri, is_b = _sheet(217, 151)
    elif name == "sheet65536":    # ... and at it
        pos, tri, is_b = _sheet(256, 128)
    else:
        raise KeyError(name)
    nv, nf = len(pos), len(tri)
    rng = np.random.default_rng(nf)
    h = float(np.sqrt(ref.triangle_areas(pos, tri).mean()))
    return Mesh(pos=pos, tri=np.ascontiguousarray(tri, dtype=np.int32), is_b=is_b, hint=hint,
                gamma=1.0 + 0.3 * rng.random(nf), kappa=1.0 + 0.3 * rng.random(nv), c0=0.1 * rng.random(nv) - 0.05,
                tilts=tangent_tilts(pos, tri), body=(rng.random(nf) < 0.6).astype(np.uint8),
                fixed=(rng.random(nv) < 0.05).astype(np.uint8), direction=0.05 * h * rng.normal(size=pos.shape))


# ---- scenarios ---------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Scenario:
    name: str
    mesh: str
    modules: int
    expect: frozenset            # the (pass, kind) instantiations the fused evaluation launches
    flags: int = 0
    facet_gamma: bool = False
    vertex_bending: bool = False  # per-vertex kappa / c0 (else uniform)
    want_grad: bool = True
    want_tilt_grad: bool = False
    diagnostics: bool = False
    constraint_mode: int = -1
    partial_body: bool = False
    fixed: bool = False           # fixed mask + apply_fixed
    trial: bool = False           # evaluate at x + ALPHA d made on the device (use_trial)

    @property
    def projected(self):
        return self.want_grad and (self.constraint_mode >= 0 or self.fixed)

    @property
    def bending(self):
        return bool(self.modules & (B | BT))

    @property
    def tilt_fields(self):
        return bool(self.modules & (T | BT))


def _k(*pairs):
    return frozenset(pairs)


SCENARIOS = [
    # kind 1: S+B+V, uniform parameters, closed mesh, no diagnostics
    Scenario("k1_sbv", "ico120", S | B | V, _k((0, 1), (1, 1))),
    Scenario("k1_sbv_lagrange_fixed", "ico120", S | B | V, _k((0, 1), (1, 1)), constraint_mode=0, partial_body=True,
             fixed=True),
    Scenario("k1_sbv_energy", "ico120", S | B | V, _k((0, 1)), want_grad=False),
    # kind 2: surface and/or volume, uniform gamma; pass A only for energy-only evaluations
    Scenario("k2_sv", "ico120", S | V, _k((1, 2))),
    Scenario("k2_sv_energy", "ico120", S | V, _k((0, 2)), want_grad=False),
    Scenario("k2_v", "ico120", V, _k((1, 2))),
    Scenario("k2_v_energy", "ico120", V, _k((0, 2)), want_grad=False),
    Scenario("k2_s", "sheet", S, _k((1, 2))),
    Scenario("k2_s_energy", "sheet", S, _k((0, 2)), want_grad=False),
    Scenario("k2_sv_penalty_fixed", "ico120", S | V, _k((1, 2)), constraint_mode=1, partial_body=True, fixed=True),
    # kind 3: bending with run-time parameters, boundary flags, flags or diagnostics, no tilt
    Scenario("k3_sbv_vertex_facet", "ico120", S | B | V, _k((0, 3), (1, 3)), facet_gamma=True, vertex_bending=True),
    Scenario("k3_willmore_boundary", "sheet", B, _k((0, 3), (1, 3)), flags=L.FLAG_WILLMORE),
    Scenario("k3_approx_boundary", "sheet", B, _k((0, 3), (1, 3)), flags=L.FLAG_APPROX),
    Scenario("k3_diagnostics", "ico120", B, _k((0, 3), (1, 3)), diagnostics=True),
    Scenario("k3_sbv_lagrange_fixed", "ico60perm", S | B | V, _k((0, 3), (1, 3)), vertex_bending=True,
             constraint_mode=0, partial_body=True, fixed=True),
    # kind 0: everything else (tilt, per-facet gamma without bending)
    Scenario("k0_sbvt_facet", "ico120", S | B | V | T, _k((0, 0), (1, 0)), facet_gamma=True),
    Scenario("k0_sbt_boundary", "sheet", S | B | T, _k((0, 0), (1, 0))),
    Scenario("k0_sv_facet", "ico120", S | V, _k((1, 0)), facet_gamma=True),
    Scenario("k0_tilt_only", "ico120", T, _k((0, 0), (1, 0)), want_grad=False, want_tilt_grad=True),
    Scenario("k0_svt_penalty_fixed", "ico120", S | V | T, _k((1, 0)), facet_gamma=True, constraint_mode=1,
             partial_body=True, fixed=True),
]
# bending-tilt (kind 3 in the patch kernels; kind 0 together with the tilt module) on both sides of the two-stage sum,
# with per-vertex kappa / c0 in Morton order and on the bounded sheet; at the positions and at trial positions.  At
# 65 536 facets the last of the 592 chunks of that sum is empty (591 x 111 >= 65 536); the 120 000-facet sheet fills it.
for _m, _vb in (("sheet65534", False), ("sheet65536", False), ("ico60perm", True), ("sheet", False)):
    for _mods, _pairs in ((BT, _k((0, 3), (1, 3))), (BT | T, _k((0, 0), (1, 0)))):
        for _trial in (False, True):
            SCENARIOS.append(Scenario(f"bt{'_tilt' if _mods & T else ''}_{_m}{'_trial' if _trial else ''}", _m, _mods,
                                      _pairs, vertex_bending=_vb, trial=_trial))
BY_NAME = {sc.name: sc for sc in SCENARIOS}
assert len(BY_NAME) == len(SCENARIOS)


# ---- kernel selection, restated from ms_kernels.cu (kernel_kind, launch_pass_a, launch_pass_b) ------------------
def kernel_kind(sc):
    """``kernel_kind``: the patch kernels see bending_tilt as bending with the diagnostic arrays attached
    (``fill_launch``); the seed and dV/dx arrays always exist on a context."""
    mods = (sc.modules & ~BT) | B if sc.modules & BT else sc.modules
    diag = sc.diagnostics or bool(sc.modules & BT)
    boundary = mesh_has_boundary(sc.mesh)
    if mods == S | B | V and sc.flags == 0 and not boundary and not sc.facet_gamma and not sc.vertex_bending and not diag:
        return 1
    if mods & ~(S | V) == 0 and mods and not sc.facet_gamma and not diag:
        return 2
    if not mods & T and mods & B:
        return 3
    return 0


def launched(sc):
    """(pass, kind) of the patch kernels one evaluation launches: pass A runs for bending and for energies, pass B
    for gradients and for the tilt gradient of the tilt module (``eval_pass_a_impl`` / ``eval_pass_b_impl``)."""
    kind, bending = kernel_kind(sc), sc.bending
    out = set()
    if bending or not sc.want_grad:
        out.add((0, kind))
    if sc.want_grad or (sc.want_tilt_grad and sc.modules & T):
        if kind == 1 and bending:
            out.add((1, 1))
        elif kind == 2 and not bending:
            out.add((1, 2))
        elif kind == 3 and bending:
            out.add((1, 3))
        else:
            out.add((1, 0))
    return out


def mesh_has_boundary(name):
    return name.startswith("sheet")


def test_scenarios_select_their_stated_kinds():
    for sc in SCENARIOS:
        assert launched(sc) == set(sc.expect), sc.name


def test_scenarios_reach_every_pass_and_kind():
    reached = set().union(*(launched(sc) for sc in SCENARIOS))
    assert reached == {(p, k) for p in (0, 1) for k in (0, 1, 2, 3)}
    # each kind also runs a volume constraint on a partial body with fixed vertices, both constraint modes overall
    for kind in range(4):
        assert any(kernel_kind(sc) == kind and sc.constraint_mode >= 0 and sc.partial_body and sc.fixed
                   for sc in SCENARIOS), kind
    assert {sc.constraint_mode for sc in SCENARIOS if sc.partial_body} == {0, 1}
    assert any(sc.trial and sc.modules == BT for sc in SCENARIOS)
    assert any(sc.trial and sc.modules == BT | T for sc in SCENARIOS)


# ---- the float64 reference ---------------------------------------------------------------------------------------
def inputs(sc):
    """Positions the evaluation sees, and the parameters, as the oracle takes them."""
    m = mesh(sc.mesh)
    pos = m.pos + ALPHA * m.direction if sc.trial else m.pos
    nv, nf = len(m.pos), len(m.tri)
    return dict(pos=pos, tri=m.tri, is_b=m.is_b if m.is_b is not None else np.zeros(nv, bool),
                gamma=m.gamma if sc.facet_gamma else np.full(nf, GAMMA_U),
                kappa=m.kappa if sc.vertex_bending else KAPPA_U, c0=m.c0 if sc.vertex_bending else C0_U,
                body=m.body if sc.partial_body else np.ones(nf, np.uint8))


def reference(sc):
    x = inputs(sc)
    pos, tri, is_b = x["pos"], x["tri"], x["is_b"]
    tilts = mesh(sc.mesh).tilts
    g, tg = np.zeros_like(pos), np.zeros_like(pos)
    out = {}
    if sc.modules & S:
        out["E_surface"] = ref.surface_energy_and_gradient(pos, tri, x["gamma"], g)
        out["area"] = float(ref.triangle_areas(pos, tri).sum())
    if sc.modules & B:
        model = "willmore" if sc.flags & L.FLAG_WILLMORE else "helfrich"
        mode = "approx" if sc.flags & L.FLAG_APPROX else "analytic"
        out["E_bending"] = ref.bending_energy_and_gradient(pos, tri, x["kappa"], x["c0"], is_b, g, model, mode)
    if sc.modules & T:
        out["E_tilt"] = ref.tilt_energy_and_gradient(pos, tri, tilts, K_TILT, g, tg)
    if sc.modules & BT:
        out["E_bending_tilt"] = ref.bending_tilt_energy_and_gradient(pos, tri, tilts, x["kappa"], x["c0"], is_b, g, tg)
    out["grad"] = g
    if sc.tilt_fields:
        out["tilt_grad"] = tg
    if sc.modules & V:
        tb = tri[x["body"].astype(bool)]
        out["volume"] = ref.body_volume(pos, tb)
        out["vol_grad"] = np.zeros_like(pos)
        ref.accumulate_volume_gradient(pos, tb, out["vol_grad"], 1.0)
    if sc.projected:
        p = g.copy()
        if sc.constraint_mode == 0:
            vg = out["vol_grad"]
            coef = -float(np.vdot(g, vg) / np.vdot(vg, vg))
            out["lambda"] = -coef
        elif sc.constraint_mode == 1:
            coef = K_VOL * (out["volume"] - v_target(sc))
            out["lambda"] = coef
        if sc.constraint_mode >= 0:
            p += coef * out["vol_grad"]
        if sc.fixed:
            p[mesh(sc.mesh).fixed.astype(bool)] = 0.0
        out["projected"] = p
    if sc.diagnostics:
        k_vecs, a_vor, w = ref.curvature_data(pos, tri)[:3]
        out["k_vecs"], out["a_vor"] = k_vecs, a_vor
        out["a_eff"] = ref.effective_areas(pos, tri, w, is_b)[0]
        out["e_vertex"] = ref.bending_energy_per_vertex(pos, tri, x["kappa"], x["c0"], is_b)
    return out


def v_target(sc):
    """Penalty target: 3 % below the body volume at the positions, so the penalty force is not small."""
    x = inputs(sc)
    return 0.97 * ref.body_volume(mesh(sc.mesh).pos, x["tri"][x["body"].astype(bool)])


@pytest.fixture(scope="module")
def references():
    cache = {}

    def get(sc):
        if sc.name not in cache:
            cache[sc.name] = reference(sc)
        return cache[sc.name]

    return get


def grad_tol(sc):
    return 2e-12 if sc.bending else TOL


def scalar_close(got, want, what, tol=TOL):
    assert abs(got - want) <= tol * max(1.0, abs(want)), (what, got, want)


SCALAR_NAMES = (("E_surface", L.SC_E_SURFACE), ("area", L.SC_AREA), ("volume", L.SC_VOLUME),
                ("E_bending", L.SC_E_BENDING), ("E_tilt", L.SC_E_TILT), ("E_bending_tilt", L.SC_E_BENDING_TILT))


def check_against_reference(sc, want, scalars, arrays):
    """``arrays``: raw gradient (approx mode: boundary rows zeroed by the caller, as the host module does), dV/dx,
    tilt gradient, projected gradient, diagnostics -- whatever the scenario produces."""
    for name, slot in SCALAR_NAMES:
        if name in want:
            scalar_close(float(scalars[slot]), want[name], name)
    if not sc.want_grad:
        if sc.want_tilt_grad:
            assert rel_err(arrays["tilt_grad"], want["tilt_grad"]) <= TOL
        return
    grad = arrays["grad"].copy()
    if sc.flags & L.FLAG_APPROX:
        grad[mesh(sc.mesh).is_b] = 0.0        # bending.py: the host module zeroes the boundary rows in approx mode
    assert rel_err(grad, want["grad"]) <= grad_tol(sc)
    if sc.modules & V:
        volgrad_close(arrays["vol_grad"], want["vol_grad"], inputs(sc)["pos"])
    if sc.tilt_fields:
        assert rel_err(arrays["tilt_grad"], want["tilt_grad"]) <= TOL
    if "projected" in want and "projected" in arrays:
        assert rel_err(arrays["projected"], want["projected"]) <= grad_tol(sc)
        if "lambda" in want:
            assert abs(float(scalars[L.SC_LAMBDA]) - want["lambda"]) <= 1e-10 * abs(want["lambda"])
    for name in ("k_vecs", "a_vor", "a_eff", "e_vertex"):
        if name in want:
            assert rel_err(arrays[name], want[name]) <= TOL, name


# ---- CPU tier: the host emulator ---------------------------------------------------------------------------------
SC_IDS = [sc.name for sc in SCENARIOS]


@pytest.mark.parametrize("pack", list(PACKS))
@pytest.mark.parametrize("name", SC_IDS)
def test_emulator_matches_reference(references, name, pack):
    sc = BY_NAME[name]
    m, x = mesh(sc.mesh), inputs(sc)
    # the emulator makes the tilt gradient in its gradient pass only
    out = H.emulate(x["pos"], x["tri"], modules=sc.modules, flags=sc.flags, want_grad=sc.want_grad or sc.want_tilt_grad,
                    is_boundary=m.is_b, body_mask=x["body"], tilts=m.tilts if sc.tilt_fields else None,
                    gamma=m.gamma if sc.facet_gamma else None, gamma_u=GAMMA_U,
                    kappa=m.kappa if sc.vertex_bending else None, c0=m.c0 if sc.vertex_bending else None,
                    kappa_u=KAPPA_U, c0_u=C0_U, k_tilt=K_TILT, **PACKS[pack])
    # at the smallest cap that still differs from one CTA per SM, a CTA takes several patches
    assert out["pack"]["n_patches"] > 33, out["pack"]
    want = references(sc)
    scalars = np.zeros(L.SC_COUNT)
    for name_, slot in SCALAR_NAMES:
        scalars[slot] = out[name_]
    arrays = dict(grad=out["grad"], vol_grad=out["volgrad"], tilt_grad=out["tilt_grad"], k_vecs=out["k_vecs"],
                  a_vor=out["a_vor"], a_eff=out["a_eff"], e_vertex=out["e_vertex"])
    check_against_reference(sc, want, scalars, arrays)


# ---- GPU tier ----------------------------------------------------------------------------------------------------
def _context(sc, pack):
    from membrane_solver_b200.context import DeviceMesh

    if L.device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu tier must run on the B200 box")
    m, x = mesh(sc.mesh), inputs(sc)
    dm = DeviceMesh(0, **PACKS[pack])
    dm.set_topology(len(m.pos), m.tri, is_boundary=m.is_b, body_mask=x["body"],
                    fixed_mask=m.fixed if sc.fixed else None, order_hint=m.pos if m.hint else None)
    if m.hint:
        assert not np.array_equal(dm.permutation(), np.arange(len(m.pos)))
    dm.set_surface_tension(m.gamma if sc.facet_gamma else GAMMA_U)
    dm.set_bending_params(m.kappa if sc.vertex_bending else KAPPA_U, m.c0 if sc.vertex_bending else C0_U)
    dm.set_tilt_rigidity(K_TILT)
    dm.set_positions(m.pos)
    if sc.tilt_fields:
        dm.set_tilts(m.tilts)
    if sc.trial:
        dm.set_direction(m.direction)
        dm.make_trial(ALPHA)
    return dm


def _options(dm, sc, raw=False):
    return dm.options(sc.modules, flags=sc.flags, want_grad=sc.want_grad, want_tilt_grad=sc.want_tilt_grad,
                      diagnostics=sc.diagnostics, use_trial=sc.trial,
                      constraint_mode=-1 if raw else sc.constraint_mode, k_vol=K_VOL,
                      v_target=v_target(sc) if sc.constraint_mode == 1 else 0.0, apply_fixed=sc.fixed and not raw)


def _outputs(sc):
    """Arrays an evaluation of the scenario writes."""
    names = []
    if sc.want_grad:
        names.append(("grad", L.ARR_GRAD))
        if sc.modules & V:
            names.append(("vol_grad", L.ARR_VOLGRAD))
    if sc.tilt_fields and (sc.want_grad or sc.want_tilt_grad):
        names.append(("tilt_grad", L.ARR_TILT_GRAD))
    if sc.bending:
        names.append(("seeds", L.ARR_SEEDS))
    if sc.diagnostics:
        names += [("k_vecs", L.ARR_K_VECS), ("a_vor", L.ARR_A_VOR), ("a_eff", L.ARR_A_EFF), ("e_vertex", L.ARR_E_VERTEX)]
    return names


def _run(dm, sc, opts, form):
    """One evaluation in the given launch form; every output array is poisoned with NaN first, so a row the
    evaluation does not write shows up."""
    names = _outputs(sc)
    for _, which in names:
        dm.upload(which, np.full(int(dm._lib.ms_ctx_array_len(dm._h, which)), np.nan))
    host = {}
    if form == "fused":
        scalars = dm.eval(opts).scalars
    elif form == "stages":
        dm.eval_stage(opts, 0)
        dm.eval_stage(opts, 1)
        scalars = dm.read_scalars().scalars
    elif form == "staged":                     # separate passes, rows reduced by k_reduce_partials
        dm.eval_pass_a(opts)
        dm.eval_pass_b(opts)
        dm.eval_finish(opts)
        scalars = dm.read_scalars().scalars
    else:                                      # ms_ctx_eval_host below the pipelining size
        pos = None if sc.trial else mesh(sc.mesh).pos
        kw = {}
        for key, which, arg in (("grad", L.ARR_GRAD, "grad"), ("vol_grad", L.ARR_VOLGRAD, "volgrad"),
                                ("tilt_grad", L.ARR_TILT_GRAD, "tilt_grad")):
            if (key, which) in names:
                kw[arg] = host[key] = np.full_like(mesh(sc.mesh).pos, np.nan)
        scalars = dm.eval_host(opts, pos, **kw).scalars
    out = {"scalars": scalars.copy()}
    for key, which in names:
        out[key] = host[key] if key in host else dm.download(which)
        assert np.all(np.isfinite(out[key])), (key, form)
    return out


def _collect(dm, sc, form):
    """Raw outputs of the scenario; with a projection also the projected gradient (a second evaluation)."""
    if not sc.projected:
        return _run(dm, sc, _options(dm, sc), form)
    raw = _run(dm, sc, _options(dm, sc, raw=True), form)
    got = _run(dm, sc, _options(dm, sc), form)
    got["projected"] = got.pop("grad")
    got["grad"] = raw["grad"]
    return got


def _scalar_slots(sc):
    return list(range(6)) + ([L.SC_G_G, L.SC_G_GC, L.SC_GC_GC, L.SC_LAMBDA, L.SC_COEF] if sc.want_grad else [])


def _assert_equivalent(sc, base, got, what, bitwise_scalars=False):
    """Raw arrays bitwise; scalars within 1e-13 relative (the per-CTA rows are added in another grouping); the
    projected gradient, whose coefficient comes from those scalars, at 1e-12."""
    for key, _ in _outputs(sc):
        a, b = base[key], got[key]
        assert np.array_equal(a.view(np.uint64), b.view(np.uint64)), (what, key, rel_err(b, a))
    if "projected" in base:
        assert rel_err(got["projected"], base["projected"]) <= TOL, what
    s0, s1 = base["scalars"], got["scalars"]
    for k in _scalar_slots(sc):
        if bitwise_scalars:
            assert s0[k].view(np.uint64) == s1[k].view(np.uint64), (what, k, s0[k], s1[k])
            continue
        scale = abs(s0[k])
        if k == L.SC_G_GC:                     # a sum with cancellation: Cauchy-Schwarz scale
            scale = max(scale, float(np.sqrt(s0[L.SC_G_G] * s0[L.SC_GC_GC])))
        if k in (L.SC_LAMBDA, L.SC_COEF) and s0[L.SC_GC_GC] > 0:
            scale = max(scale, float(np.sqrt(s0[L.SC_G_G] / s0[L.SC_GC_GC])))
        assert abs(s1[k] - s0[k]) <= 1e-13 * scale, (what, k, s0[k], s1[k])


def _set_cap(dm, n):
    L.check(L.lib().ms_ctx_set_max_ctas(dm._h, n))


@pytest.mark.gpu
@pytest.mark.parametrize("pack", list(PACKS))
@pytest.mark.parametrize("name", SC_IDS)
def test_patch_kernels_vs_reference_across_grids_and_forms(references, name, pack):
    sc = BY_NAME[name]
    dm = _context(sc, pack)
    try:
        # the oracle, at one CTA per SM, fused
        base = _collect(dm, sc, "fused")
        check_against_reference(sc, references(sc), base["scalars"], base)
        # grid caps on the same context
        for n in CAPS:
            _set_cap(dm, n)
            _assert_equivalent(sc, base, _collect(dm, sc, "fused"), f"cap {n}", bitwise_scalars=n >= 1000)
        assert L.lib().ms_ctx_set_max_ctas(dm._h, -1) != 0
        # launch forms at caps 0 and 1
        for cap in (0, 1):
            _set_cap(dm, cap)
            for form in FORMS:
                got = _collect(dm, sc, form)
                _assert_equivalent(sc, base, got, f"cap {cap} {form}")
                # repeats: the same cap and form give the same bits, scalars included
                if form in ("fused", "staged"):
                    _assert_equivalent(sc, got, _collect(dm, sc, form), f"repeat cap {cap} {form}", bitwise_scalars=True)
        _set_cap(dm, 33)
        first = _collect(dm, sc, "fused")
        _assert_equivalent(sc, first, _collect(dm, sc, "fused"), "repeat cap 33", bitwise_scalars=True)
    finally:
        dm.close()
