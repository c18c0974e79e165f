"""Generate golden input/output vectors by running the REAL reference.

Needs a checkout of the original membrane_solver:

    MEMBRANE_REFERENCE_ROOT=<checkout> PYTHONDONTWRITEBYTECODE=1 python tests/golden/generate_golden.py

It imports the unmodified reference from that checkout (read-only; NumPy path, without
its Fortran kernels), evaluates the hot-path modules
on the reference's own mesh files, and stores dense inputs + outputs as small
``.npz`` files next to this script.  The fixtures travel; the reference does not.

Each ``modules_*.npz`` holds one mesh state:
  pos (nv,3) f64, tri (nf,3) i32, gamma (nf), is_boundary (nv) bool,
  fixed (nv) bool, kappa (nv), c0 (nv), tilts (nv,3),
  body_rows_<i> (facet rows of body i), body_target_<i>,
and per evaluated module ``E_<tag>``, ``g_<tag>`` (+ ``tg_<tag>`` tilt grads).
"""

from __future__ import annotations

import importlib.util
import os
import sys

import numpy as np

REF = os.environ.get("MEMBRANE_REFERENCE_ROOT")
if not REF:
    sys.exit("set MEMBRANE_REFERENCE_ROOT to a checkout of the original membrane_solver")
HERE = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True
sys.path.insert(0, REF)

from core.parameters.global_parameters import GlobalParameters  # noqa: E402
from core.parameters.resolver import ParameterResolver  # noqa: E402
from geometry.bending_derivatives import grad_cotan, grad_triangle_area  # noqa: E402
from geometry.curvature import compute_curvature_data  # noqa: E402
from geometry.geom_io import load_data, parse_geometry  # noqa: E402
from geometry.tilt_operators import p1_triangle_shape_gradients  # noqa: E402
from modules.constraints import volume as volume_constraint  # noqa: E402
from modules.energy import bending, bending_tilt, surface, tilt  # noqa: E402
from modules.energy import volume as volume_energy  # noqa: E402
from modules.energy.bending_math import _apply_beltrami_laplacian  # noqa: E402
from modules.energy.bending_utils import _compute_effective_areas, _vertex_normals  # noqa: E402
from runtime.constraint_manager import ConstraintModuleManager  # noqa: E402
from runtime.energy_manager import EnergyModuleManager  # noqa: E402
from runtime.minimizer import Minimizer  # noqa: E402
from runtime.refinement import refine_triangle_mesh  # noqa: E402
from runtime.steppers.gradient_descent import GradientDescent  # noqa: E402


def _load_ref_test_module(name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(REF, "tests", name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


# ------------------------------------------------------------------ kernels
def kernel_vectors():
    """Same seeded inputs as the reference's tests/test_fortran_kernels.py:46-376."""
    out = {}
    for n in (4, 17):
        rng = np.random.default_rng(123)
        u = rng.normal(size=(n, 3))
        v = rng.normal(size=(n, 3))
        v += 0.3 * rng.normal(size=(n, 3))
        gu, gv = grad_cotan(u, v)
        tu, tv = grad_triangle_area(u, v)
        out.update({f"gc{n}_u": u, f"gc{n}_v": v, f"gc{n}_gu": gu, f"gc{n}_gv": gv,
                    f"gc{n}_tu": tu, f"gc{n}_tv": tv})
    # degenerate grad_cotan rows (S <= 1e-15 -> zeros)
    u = np.array([[1.0, 0, 0], [0, 0, 0], [1, 2, 3.0]])
    v = np.array([[2.0, 0, 0], [1, 1, 1], [1, 2, 3.0]])
    gu, gv = grad_cotan(u, v)
    out.update(gcd_u=u, gcd_v=v, gcd_gu=gu, gcd_gv=gv)

    rng = np.random.default_rng(456)
    nv, nf, dim = 11, 8, 3
    w = rng.normal(size=(nf, 3))
    tri = rng.integers(0, nv, size=(nf, 3), dtype=np.int32)
    field = rng.normal(size=(nv, dim))
    os.environ["MEMBRANE_DISABLE_FORTRAN_BENDING"] = "1"
    out.update(lap_w=w, lap_tri=tri, lap_field=field,
               lap_out=_apply_beltrami_laplacian(w, tri, field))

    rng = np.random.default_rng(999)
    nv, nf = 10, 7
    pos = rng.normal(size=(nv, 3))
    tl = rng.normal(size=(nv, 3))
    tri = rng.integers(0, nv, size=(nf, 3), dtype=np.int32)
    area, g0, g1, g2 = p1_triangle_shape_gradients(positions=pos, tri_rows=tri)
    div = (np.einsum("ij,ij->i", tl[tri[:, 0]], g0) + np.einsum("ij,ij->i", tl[tri[:, 1]], g1)
           + np.einsum("ij,ij->i", tl[tri[:, 2]], g2))
    out.update(p1_pos=pos, p1_tilts=tl, p1_tri=tri, p1_div=div, p1_area=area,
               p1_g0=g0, p1_g1=g1, p1_g2=g2)

    ref_test = _load_ref_test_module("test_fortran_kernels")
    rng = np.random.default_rng(2024)
    nv, nf = 12, 9
    pos = rng.normal(size=(nv, 3)).astype(np.float64)
    tri = rng.integers(0, nv, size=(nf, 3), dtype=np.int32)
    k, a, wts, va0, va1, va2 = ref_test._curvature_data_reference(pos, tri)
    out.update(cd_pos=pos, cd_tri=tri, cd_k=k, cd_a=a, cd_w=wts, cd_va0=va0, cd_va1=va1, cd_va2=va2)

    # surface kernel: random soup incl. repeated indices (degenerate facets are skipped)
    rng = np.random.default_rng(7)
    nv, nf = 15, 20
    pos = rng.normal(size=(nv, 3))
    tri = rng.integers(0, nv, size=(nf, 3), dtype=np.int32)
    gamma = rng.uniform(0.5, 2.0, size=nf)
    out.update(sf_pos=pos, sf_tri=tri, sf_gamma=gamma)
    np.savez_compressed(os.path.join(HERE, "kernels.npz"), **out)
    print("kernels.npz", len(out), "arrays")


# ------------------------------------------------------------------ modules
def _dense_state(mesh):
    mesh.build_position_cache()
    pos = np.array(mesh.positions_view(), dtype=np.float64, order="C")
    tri, _ = mesh.triangle_row_cache()
    tri = np.ascontiguousarray(tri, dtype=np.int32)
    nv = pos.shape[0]
    idx = mesh.vertex_index_to_row
    is_b = np.zeros(nv, dtype=bool)
    for vid in mesh.boundary_vertex_ids:
        if vid in idx:
            is_b[idx[vid]] = True
    fixed = np.zeros(nv, dtype=bool)
    for vid, v in mesh.vertices.items():
        if getattr(v, "fixed", False):
            fixed[idx[int(vid)]] = True
    state = dict(pos=pos, tri=tri, is_boundary=is_b, fixed=fixed,
                 gamma=np.asarray(mesh.get_facet_parameter_array("surface_tension"), dtype=np.float64))
    facet_row = mesh.facet_to_triangle_row
    for i, body in enumerate(mesh.bodies.values()):
        rows = np.array([facet_row[abs(int(f))] for f in body.facet_indices], dtype=np.int32)
        state[f"body_rows_{i}"] = rows
        tv = body.target_volume
        if tv is None:
            tv = body.options.get("target_volume")
        state[f"body_target_{i}"] = np.float64(np.nan if tv is None else tv)
    return state


def _module_outputs(mesh, gp, state, tag_params):
    """Evaluate the hot-path modules with the reference's own functions."""
    resolver = ParameterResolver(gp)
    pos = mesh.positions_view()
    idx = mesh.vertex_index_to_row
    out = {}

    g = np.zeros_like(pos)
    out["E_surface"] = surface.compute_energy_and_gradient_array(
        mesh, gp, resolver, positions=pos, index_map=idx, grad_arr=g)
    out["g_surface"] = g

    if mesh.bodies:
        gcs = []
        for body in mesh.bodies.values():
            gc = np.zeros_like(pos)
            body.accumulate_volume_gradient(mesh, pos, gc, factor=1.0)
            gcs.append(gc)
            out.setdefault("volumes", []).append(body.compute_volume(mesh, positions=np.array(pos)))
        out["g_volume"] = np.stack(gcs)
        out["volumes"] = np.array(out["volumes"])

    for tag, (model, mode, kappa, c0) in tag_params.items():
        gp.set("bending_modulus", kappa)
        gp.set("spontaneous_curvature", c0)
        gp.set("bending_energy_model", model)
        gp.set("bending_gradient_mode", mode)
        if hasattr(mesh, "_bending_vertex_param_cache"):
            mesh._bending_vertex_param_cache = None
        g = np.zeros_like(pos)
        out[f"E_bending_{tag}"] = bending.compute_energy_and_gradient_array(
            mesh, gp, resolver, positions=pos, index_map=idx, grad_arr=g)
        out[f"g_bending_{tag}"] = g
        out[f"Ev_bending_{tag}"] = bending.compute_energy_array(mesh, gp, pos, idx)
        if model == "helfrich":
            tl = state["tilts"]
            g = np.zeros_like(pos)
            tg = np.zeros_like(pos)
            out[f"E_bending_tilt_{tag}"] = bending_tilt.compute_energy_and_gradient_array(
                mesh, gp, resolver, positions=pos, index_map=idx, grad_arr=g,
                tilts=tl, tilt_grad_arr=tg)
            out[f"g_bending_tilt_{tag}"] = g
            out[f"tg_bending_tilt_{tag}"] = tg
            tg2 = np.zeros_like(pos)
            e2 = bending_tilt.compute_energy_and_gradient_array(
                mesh, gp, resolver, positions=pos, index_map=idx, grad_arr=None,
                tilts=tl, tilt_grad_arr=tg2)
            assert abs(e2 - out[f"E_bending_tilt_{tag}"]) <= 1e-12 * max(1.0, abs(e2))
            out[f"tgonly_bending_tilt_{tag}"] = tg2

    gp.set("tilt_rigidity", 1.7)
    g = np.zeros_like(pos)
    tg = np.zeros_like(pos)
    out["E_tilt"] = tilt.compute_energy_and_gradient_array(
        mesh, gp, resolver, positions=pos, index_map=idx, grad_arr=g,
        tilts=state["tilts"], tilt_grad_arr=tg)
    out["g_tilt"] = g
    out["tg_tilt"] = tg
    out["k_tilt"] = np.float64(1.7)

    # intermediates (curvature data, effective areas, normals) for kernel-level parity
    k_vecs, a_vor, weights, _ = compute_curvature_data(mesh, np.array(pos), idx)
    a_eff, va0, va1, va2 = _compute_effective_areas(mesh, np.array(pos), state["tri"], weights, idx)
    out.update(k_vecs=np.array(k_vecs), a_vor=np.array(a_vor), weights=np.array(weights),
               a_eff=np.array(a_eff), va_eff=np.stack([va0, va1, va2], axis=1),
               normals=_vertex_normals(mesh, np.array(pos), state["tri"]))
    return out


BENDING_TAGS = {
    "helfrich_analytic": ("helfrich", "analytic", 1.0, 0.0),
    "helfrich_c0": ("helfrich", "analytic", 2.5, 0.35),
    "helfrich_approx": ("helfrich", "approx", 1.0, 0.2),
    "willmore_analytic": ("willmore", "analytic", 1.3, 0.0),
}


def _save_state(name, mesh, rng, jitter=0.0):
    gp = mesh.global_parameters
    if jitter:
        for v in mesh.vertices.values():
            v.position = np.asarray(v.position, dtype=float) + jitter * rng.normal(size=3)
        mesh.increment_version()
    state = _dense_state(mesh)
    nv = state["pos"].shape[0]
    state["tilts"] = 0.1 * rng.normal(size=(nv, 3))
    params = {}
    for tag, (model, mode, kappa, c0) in BENDING_TAGS.items():
        params[f"param_{tag}"] = np.array([kappa, c0])
    out = _module_outputs(mesh, gp, state, BENDING_TAGS)
    np.savez_compressed(os.path.join(HERE, f"modules_{name}.npz"), **state, **params, **out)
    print(f"modules_{name}.npz nv={nv} nf={state['tri'].shape[0]} nb={int(state['is_boundary'].sum())}")


def _refined(path, levels):
    mesh = parse_geometry(load_data(path))
    for _ in range(levels):
        mesh = refine_triangle_mesh(mesh)
    return mesh


def module_vectors():
    rng = np.random.default_rng(20261018)
    m = os.path.join(REF, "meshes")
    b = os.path.join(REF, "benchmarks", "inputs")
    _save_state("cube_r0", _refined(os.path.join(m, "cube.json"), 0), rng)
    _save_state("cube_r2_jit", _refined(os.path.join(m, "cube.json"), 2), rng, jitter=0.02)
    _save_state("catenoid_r2", _refined(os.path.join(m, "catenoid.json"), 2), rng)
    _save_state("catenoid_r2_jit", _refined(os.path.join(m, "catenoid.json"), 2), rng, jitter=0.01)
    _save_state("bending_cube_r2", _refined(os.path.join(m, "bending_cube.yaml"), 2), rng, jitter=0.01)
    _save_state("sphere_r1_jit", _refined(os.path.join(b, "bench_bending_analytic.json"), 1), rng, jitter=0.03)
    _save_state("flat_sheet", _refined(os.path.join(m, "flat_sheet_4x4.yaml"), 1), rng)
    _save_state("flat_sheet_jit", _refined(os.path.join(m, "flat_sheet_4x4.yaml"), 1), rng, jitter=0.05)


# ------------------------------------------------------------- minimizer
def minimizer_vectors():
    """Total energy + projected gradient through Minimizer (KKT + fixed mask)."""
    out = {}
    for name, path, levels in (
        ("cube", os.path.join(REF, "meshes", "cube.json"), 1),
        ("bcube", os.path.join(REF, "meshes", "bending_cube.yaml"), 1),
    ):
        mesh = _refined(path, levels)
        rng = np.random.default_rng(5)
        for v in mesh.vertices.values():
            v.position = np.asarray(v.position, dtype=float) + 0.01 * rng.normal(size=3)
        mesh.increment_version()
        gp = mesh.global_parameters
        mini = Minimizer(mesh, gp, GradientDescent(), EnergyModuleManager(mesh.energy_modules),
                         ConstraintModuleManager(mesh.constraint_modules), quiet=True)
        e, g = mini.compute_energy_and_gradient_array()
        st = _dense_state(mesh)
        for k, v in st.items():
            out[f"{name}_{k}"] = v
        out[f"{name}_E"] = np.float64(e)
        out[f"{name}_g"] = np.array(g)
        out[f"{name}_modules"] = np.array(list(mesh.energy_modules))
        out[f"{name}_constraints"] = np.array(list(mesh.constraint_modules))
        out[f"{name}_mode"] = np.array(str(gp.get("volume_constraint_mode", "lagrange")))
        out[f"{name}_kvol"] = np.float64(gp.get("volume_stiffness", 0.0) or 0.0)
        out[f"{name}_kappa"] = np.float64(gp.get("bending_modulus", 0.0) or 0.0)
        out[f"{name}_c0"] = np.float64(gp.get("spontaneous_curvature", 0.0) or 0.0)
        out[f"{name}_model"] = np.array(str(gp.get("bending_energy_model", "helfrich")))
        bd = mini.compute_energy_breakdown()
        for k, v in bd.items():
            out[f"{name}_E_{k}"] = np.float64(v)
        print(name, list(mesh.energy_modules), list(mesh.constraint_modules), e,
              str(gp.get("volume_constraint_mode", "lagrange")))
    np.savez_compressed(os.path.join(HERE, "minimizer.npz"), **out)


def trajectory_vectors():
    """Gradient-descent trajectories of the reference Minimizer (GD + Armijo, trial-energy fast path:
    no enforceable constraints) for the device-resident loop: initial dense state, per-step energies,
    final positions."""
    out = {}
    for name, path, levels, steps, tweak in (
        ("cube", os.path.join(REF, "meshes", "cube.json"), 2, 12, None),                 # surface + volume penalty
        ("bcube", os.path.join(REF, "meshes", "bending_cube.yaml"), 1, 6, "no_constraints"),  # + Helfrich bending
        ("cubecg", os.path.join(REF, "meshes", "cube.json"), 2, 14, "cg"),               # conjugate gradient stepper
        # hard volume constraint, projected in every trial.  (With volume_projection_during_minimization=False the
        # reference's final projection starts from a STALE volume gradient -- Body.compute_volume refreshes the
        # cached version but not the cached gradient, geometry/body.py:70-148 vs 401-410 -- so that trajectory is a
        # property of the reference's host-side cache, kept by the drop-in path but not by the device loop.)
        ("bcubep", os.path.join(REF, "meshes", "bending_cube.yaml"), 1, 5, "constrained_proj"),
        # the same with the conjugate-gradient stepper: the volume-only evaluations of the Newton projection run
        # between the direction and the history update
        ("bcubepcg", os.path.join(REF, "meshes", "bending_cube.yaml"), 1, 8, "constrained_proj_cg"),
    ):
        mesh = _refined(path, levels)
        rng = np.random.default_rng(11)
        for v in mesh.vertices.values():
            v.position = np.asarray(v.position, dtype=float) + 0.01 * rng.normal(size=3)
        mesh.increment_version()
        gp = mesh.global_parameters
        if tweak == "no_constraints":
            # keep the trial-energy fast path: the volume enters as a penalty, not as a hard constraint
            mesh.constraint_modules = []
            gp.set("volume_constraint_mode", "penalty")
            if "volume" not in mesh.energy_modules:
                mesh.energy_modules = list(mesh.energy_modules) + ["volume"]
        if tweak in ("cg", "constrained_proj_cg"):
            from runtime.steppers.conjugate_gradient import ConjugateGradient

            stepper = ConjugateGradient()
        else:
            stepper = GradientDescent()
        mini = Minimizer(mesh, gp, stepper, EnergyModuleManager(mesh.energy_modules),
                         ConstraintModuleManager(mesh.constraint_modules), quiet=True)
        if tweak in ("constrained_proj", "constrained_proj_cg"):
            gp.set("volume_projection_during_minimization", True)
        assert mini._has_enforceable_constraints == (tweak in ("constrained", "constrained_proj", "constrained_proj_cg"))
        st = _dense_state(mesh)
        for k, v in st.items():
            out[f"{name}_{k}"] = v
        energies = []
        if tweak in ("cg", "constrained_proj_cg"):
            # one call: the stepper keeps its history across the iterations of a single minimize()
            res = mini.minimize(n_steps=steps)
            energies = [res["energy"]] * steps
        else:
            for i in range(steps):
                res = mini.minimize(n_steps=1)
                energies.append(res["energy"])
        out[f"{name}_energies"] = np.array(energies)
        out[f"{name}_final_pos"] = np.array(mesh.positions_view())
        out[f"{name}_step_size"] = np.float64(mini.step_size)
        out[f"{name}_modules"] = np.array(list(mesh.energy_modules))
        out[f"{name}_mode"] = np.array(str(gp.get("volume_constraint_mode", "lagrange")))
        out[f"{name}_kvol"] = np.float64(gp.get("volume_stiffness", 0.0) or 0.0)
        out[f"{name}_kappa"] = np.float64(gp.get("bending_modulus", 0.0) or 0.0)
        out[f"{name}_c0"] = np.float64(gp.get("spontaneous_curvature", 0.0) or 0.0)
        out[f"{name}_steps"] = np.int64(steps)
        out[f"{name}_enforce"] = np.bool_(mini._has_enforceable_constraints)
        out[f"{name}_proj_flag"] = np.bool_(gp.get("volume_projection_during_minimization", True))
        out[f"{name}_vol_tol"] = np.float64(gp.get("volume_tolerance", 1e-3))
        print(name, list(mesh.energy_modules), energies[0], energies[-1], mini.step_size)
    np.savez_compressed(os.path.join(HERE, "trajectory.npz"), **out)


def leaflet_vectors():
    """BASELINE config 4: the four leaflet modules of the reference's caveolin free-disk mesh
    (bending_tilt_in/out, tilt_in/out) with the selections the reference derives from the mesh options
    stored as plain masks.  One ``leaflet.npz``; keys ``<state>_<leaflet>_<what>``."""
    from modules.energy import (bending_tilt_in, bending_tilt_out, tilt_in, tilt_out, tilt_smoothness_in,
                                tilt_smoothness_out)
    from modules.energy.tilt_smoothness_utils import _resolve_smoothness_rigidity
    from modules.energy.bt_params import (_assume_J0_center_xy, _assume_J0_presets, _assume_J0_radius_max,
                                          _per_vertex_params_leaflet)
    from modules.energy.bt_selection import (_base_term_region_zero_rows, _collect_preset_rows,
                                             _interior_mask_leaflet)
    from modules.energy.leaflet_presence import leaflet_absent_vertex_mask, leaflet_present_triangle_mask
    from modules.energy.tilt_params import _resolve_tilt_mass_mode, _resolve_tilt_modulus

    path = os.path.join(REF, "meshes", "caveolin",
                        "kozlov_1disk_3d_tensionless_single_leaflet_profile_hard_rim_R12_free_disk.yaml")
    out = {}
    for state, levels, jitter, mass in (("r0", 0, 0.02, None), ("r1", 1, 0.05, None), ("r1c", 1, 0.03, "consistent")):
        mesh = _refined(path, levels)
        gp = mesh.global_parameters
        if mass:
            gp.set("tilt_mass_mode", mass)
        res = ParameterResolver(gp)
        rng = np.random.default_rng(77 + levels)
        pos = np.array(mesh.positions_view())
        pos[:, 2] += jitter * rng.standard_normal(len(pos))
        nv = len(pos)
        idx = mesh.vertex_index_to_row
        tri = np.ascontiguousarray(mesh.triangle_row_cache()[0], dtype=np.int32)
        tilts = {"in": 0.1 * rng.standard_normal((nv, 3)), "out": 0.1 * rng.standard_normal((nv, 3))}
        isb = np.zeros(nv, bool)
        for vid in mesh.boundary_vertex_ids:
            isb[idx[vid]] = True
        out[f"{state}_pos"], out[f"{state}_tri"], out[f"{state}_is_boundary"] = pos, tri, isb
        # the mesh options the selections are derived from (leaflet_selection.py re-derives them on arrays): the
        # vertex presets / group tags / numeric overrides, the mesh's own positions and the global parameters
        opt_keys = ("preset", "rim_slope_match_group", "tilt_thetaB_group", "tilt_thetaB_group_in",
                    "tilt_thetaB_group_out", "bending_modulus", "bending_modulus_in", "bending_modulus_out",
                    "spontaneous_curvature", "spontaneous_curvature_in", "spontaneous_curvature_out",
                    "intrinsic_curvature")
        vopts = {}
        for row, vid in enumerate(mesh.vertex_ids):
            o = getattr(mesh.vertices[int(vid)], "options", None) or {}
            keep_o = {k: o[k] for k in opt_keys if k in o and o[k] is not None}
            if keep_o:
                vopts[int(row)] = keep_o
        import json as _json

        gp_dump = {}
        for k in gp.to_dict() if hasattr(gp, "to_dict") else dict(getattr(gp, "_params", {})):
            v = gp.get(k)
            try:
                _json.dumps(v)
            except TypeError:
                continue
            gp_dump[k] = v
        out[f"{state}_vertex_options_json"] = np.array(_json.dumps(vopts))
        out[f"{state}_global_params_json"] = np.array(_json.dumps(gp_dump))
        out[f"{state}_mesh_pos"] = np.array(mesh.positions_view())
        for leaf, sign, bt, tm, sm in (("in", -1.0, bending_tilt_in, tilt_in, tilt_smoothness_in),
                                       ("out", 1.0, bending_tilt_out, tilt_out, tilt_smoothness_out)):
            pre = f"{state}_{leaf}_"
            am = leaflet_absent_vertex_mask(mesh, gp, leaflet=leaf)
            keep = leaflet_present_triangle_mask(mesh, tri, absent_vertex_mask=am)
            keep = np.ones(len(tri), bool) if keep.size == 0 else np.asarray(keep, bool)
            inter = _interior_mask_leaflet(mesh, gp, cache_tag=leaf, index_map=idx)
            kap, c0 = _per_vertex_params_leaflet(mesh, gp, model="helfrich", kappa_key=f"bending_modulus_{leaf}",
                                                 cache_tag=leaf)
            bz = np.zeros(nv, bool)
            presets = _assume_J0_presets(gp, cache_tag=leaf)
            if presets:
                rows = _collect_preset_rows(mesh, presets=presets, cache_tag=leaf, index_map=idx,
                                            radius_max=_assume_J0_radius_max(gp, cache_tag=leaf),
                                            center_xy=_assume_J0_center_xy(gp))
                bz[rows] = True
            bz[_base_term_region_zero_rows(mesh, gp, cache_tag=leaf, index_map=idx)] = True
            out[pre + "tilts"], out[pre + "keep"], out[pre + "interior"] = tilts[leaf], keep, np.asarray(inter, bool)
            out[pre + "base_zero"], out[pre + "kappa"], out[pre + "c0"] = bz, np.array(kap), np.array(c0)
            out[pre + "sign"] = np.float64(sign)
            out[pre + "k_tilt"] = np.float64(_resolve_tilt_modulus(res, leaf))
            out[pre + "consistent"] = np.bool_(_resolve_tilt_mass_mode(res, leaf) == "consistent")
            out[pre + "k_smooth"] = np.float64(_resolve_smoothness_rigidity(res, leaf))
            for tag, mod in (("bt", bt), ("tilt", tm), ("smooth", sm)):
                g, tgi, tgo = np.zeros_like(pos), np.zeros_like(pos), np.zeros_like(pos)
                e = mod.compute_energy_and_gradient_array(mesh, gp, res, positions=pos, index_map=idx, grad_arr=g,
                                                          tilts_in=tilts["in"], tilts_out=tilts["out"],
                                                          tilt_in_grad_arr=tgi, tilt_out_grad_arr=tgo)
                out[pre + f"E_{tag}"], out[pre + f"g_{tag}"] = np.float64(e), g
                out[pre + f"tg_{tag}"] = tgi if leaf == "in" else tgo
                assert not np.any(tgo if leaf == "in" else tgi)
                # tilt-only evaluation (grad_arr=None): the inner relaxation loop's call
                tgi, tgo = np.zeros_like(pos), np.zeros_like(pos)
                e2 = mod.compute_energy_and_gradient_array(mesh, gp, res, positions=pos, index_map=idx, grad_arr=None,
                                                           tilts_in=tilts["in"], tilts_out=tilts["out"],
                                                           tilt_in_grad_arr=tgi, tilt_out_grad_arr=tgo)
                out[pre + f"E_{tag}_tiltonly"] = np.float64(e2)
                out[pre + f"tg_{tag}_tiltonly"] = tgi if leaf == "in" else tgo
                print(state, leaf, tag, e, e2, int(keep.sum()), int(inter.sum()), int(bz.sum()))
    np.savez_compressed(os.path.join(HERE, "leaflet.npz"), **out)


def _replay(path, lines, *, step_size=None):
    """Drive the UNMODIFIED reference through an instruction list the way its benchmarks do
    (benchmarks/benchmark_profile_relax_light.py:12-31): yields (instruction, context) after every instruction."""
    from commands.context import CommandContext
    from commands.executor import execute_command_line

    mesh = parse_geometry(load_data(path))
    stepper = GradientDescent()
    mini = Minimizer(mesh, mesh.global_parameters, stepper, EnergyModuleManager(mesh.energy_modules),
                     ConstraintModuleManager(mesh.constraint_modules), quiet=True)
    mini.step_size = mesh.global_parameters.get("step_size", 1e-3) if step_size is None else step_size
    ctx = CommandContext(mesh, mini, stepper)
    for line in lines:
        execute_command_line(ctx, line)
        yield line, ctx


def replay_vectors():
    """SURVEY.md appendix B: the instruction lists of the reference's own benchmark inputs, replayed through the
    unmodified reference; the dense state after EVERY instruction (positions, triangles, masks, bodies), the
    reference's per-module energies and its total projected gradient there.  The device path re-evaluates every
    stored state (1e-12) and the end points are the survey's known answers (1e-9)."""
    import json

    cases = (
        ("cube", os.path.join(REF, "benchmarks", "inputs", "bench_cube.json"), None),
        ("catenoid", os.path.join(REF, "benchmarks", "inputs", "bench_catenoid.json"), None),
        ("bcube", os.path.join(REF, "meshes", "bending_cube.yaml"), ["r", "u", "g 50", "r", "u", "g 100", "V"]),  # macro gogo
    )
    out = {}
    for name, path, lines in cases:
        if lines is None:
            lines = [str(x) for x in load_data(path).get("instructions", [])]
        k = 0
        for line, ctx in _replay(path, lines):
            mesh, mini = ctx.mesh, ctx.minimizer
            gp = mesh.global_parameters
            st = _dense_state(mesh)
            pre = f"{name}_{k:02d}_"
            for key, v in st.items():
                out[pre + key] = v
            bd = mini.compute_energy_breakdown()
            for mod, e in bd.items():
                out[pre + f"E_{mod}"] = np.float64(e)
            e, g = mini.compute_energy_and_gradient_array()
            out[pre + "E"], out[pre + "g"] = np.float64(e), np.array(g)
            out[pre + "instruction"] = np.array(line)
            out[pre + "modules"] = np.array(list(mesh.energy_modules))
            out[pre + "constraints"] = np.array(list(mesh.constraint_modules))
            for body in mesh.bodies.values():
                out[pre + "volume"] = np.float64(body.compute_volume(mesh))
                break
            k += 1
        out[f"{name}_count"] = np.int64(k)
        out[f"{name}_params_json"] = np.array(json.dumps({
            "surface_tension": gp.get("surface_tension", 1.0), "bending_modulus": gp.get("bending_modulus", 0.0) or 0.0,
            "spontaneous_curvature": gp.get("spontaneous_curvature", gp.get("intrinsic_curvature", 0.0)) or 0.0,
            "bending_energy_model": str(gp.get("bending_energy_model", "helfrich")),
            "bending_gradient_mode": str(gp.get("bending_gradient_mode", "analytic")),
            "volume_constraint_mode": str(gp.get("volume_constraint_mode", "lagrange")),
            "volume_stiffness": gp.get("volume_stiffness", 0.0) or 0.0}))
        print(name, k, "states; end:", {m: float(v) for m, v in bd.items()}, "nf", len(st["tri"]), "nv", len(st["pos"]))
    # BASELINE configs[3]: the caveolin free-disk mesh after its macro profile_relax_light (SURVEY.md appendix B):
    # end state (positions, both tilt fields, the mesh options the leaflet selections derive from) and the
    # reference's module energies there
    import json as _json

    path = os.path.join(REF, "meshes", "caveolin",
                        "kozlov_1disk_3d_tensionless_single_leaflet_profile_hard_rim_R12_free_disk.yaml")
    for line, ctx in _replay(path, ["profile_relax_light"]):
        mesh, mini = ctx.mesh, ctx.minimizer
    gp = mesh.global_parameters
    st = _dense_state(mesh)
    out["caveolin_pos"], out["caveolin_tri"], out["caveolin_is_boundary"] = st["pos"], st["tri"], st["is_boundary"]
    out["caveolin_tilts_in"] = np.array(mesh.tilts_in_view())
    out["caveolin_tilts_out"] = np.array(mesh.tilts_out_view())
    opt_keys = ("preset", "rim_slope_match_group", "tilt_thetaB_group", "tilt_thetaB_group_in", "tilt_thetaB_group_out",
                "bending_modulus", "bending_modulus_in", "bending_modulus_out", "spontaneous_curvature",
                "spontaneous_curvature_in", "spontaneous_curvature_out", "intrinsic_curvature")
    vopts = {}
    for row, vid in enumerate(mesh.vertex_ids):
        o = getattr(mesh.vertices[int(vid)], "options", None) or {}
        keep_o = {k: o[k] for k in opt_keys if k in o and o[k] is not None}
        if keep_o:
            vopts[int(row)] = keep_o
    gp_dump = {}
    for k in gp.to_dict():
        v = gp.get(k)
        try:
            _json.dumps(v)
        except TypeError:
            continue
        gp_dump[k] = v
    out["caveolin_vertex_options_json"] = np.array(_json.dumps(vopts))
    out["caveolin_global_params_json"] = np.array(_json.dumps(gp_dump))
    bd = mini.compute_energy_breakdown()
    for mod, e in bd.items():
        out[f"caveolin_E_{mod}"] = np.float64(e)
    print("caveolin", len(st["pos"]), len(st["tri"]), {m: float(v) for m, v in bd.items()})
    np.savez_compressed(os.path.join(HERE, "replay.npz"), **out)


def equiangulate_vectors():
    """runtime/equiangulation.py on the jittered r2 catenoid (the case where the reference's traversal makes
    consistent flips): input, the reference's output, and the flip criterion's violation counts (should_flip_edge
    applied to every interior edge) before / after."""
    from runtime.equiangulation import equiangulate_mesh, should_flip_edge

    mesh = _refined(os.path.join(REF, "meshes", "catenoid.json"), 2)
    rng = np.random.default_rng(3)
    for v in mesh.vertices.values():
        if not getattr(v, "fixed", False):
            v.position = np.asarray(v.position, dtype=float) + 0.06 * rng.normal(size=3)
    mesh.increment_version()

    def violations(m):
        m.build_connectivity_maps()
        n = 0
        for ei, edge in m.edges.items():
            fs = m.get_facets_of_edge(ei)
            if len(fs) == 2 and should_flip_edge(m, edge, fs[0], fs[1]):
                n += 1
        return n

    st = _dense_state(mesh)
    before = violations(mesh)
    out = equiangulate_mesh(mesh)
    st2 = _dense_state(out)
    assert np.array_equal(st["pos"], st2["pos"])
    np.savez_compressed(os.path.join(HERE, "equiangulate.npz"), pos=st["pos"], tri=st["tri"], fixed=st["fixed"],
                        tri_ref=st2["tri"], violations_before=np.int64(before), violations_ref=np.int64(violations(out)))
    print("equiangulate", len(st["tri"]), before, violations(out))


def p1_vertex_vectors():
    """geometry/tilt_operators.py:414-465 on a jittered catenoid (open mesh) with a random tilt field."""
    from geometry.tilt_operators import p1_vertex_divergence

    mesh = _refined(os.path.join(REF, "meshes", "catenoid.json"), 2)
    rng = np.random.default_rng(11)
    pos = np.array(mesh.positions_view()) + 0.01 * rng.standard_normal((len(mesh.vertex_ids), 3))
    tri = np.ascontiguousarray(mesh.triangle_row_cache()[0], dtype=np.int32)
    tilts = 0.2 * rng.standard_normal(pos.shape)
    div_v, area_v = p1_vertex_divergence(n_vertices=len(pos), positions=pos, tilts=tilts, tri_rows=tri)
    # single-field tilt smoothness (modules/energy/tilt_smoothness.py) on the same state
    from modules.energy import tilt_smoothness

    gp = mesh.global_parameters
    gp.set("tilt_smoothness_rigidity", 0.7)
    tg, g = np.zeros_like(pos), np.zeros_like(pos)
    e_s = tilt_smoothness.compute_energy_and_gradient_array(mesh, gp, ParameterResolver(gp), positions=pos,
                                                            index_map=mesh.vertex_index_to_row, grad_arr=g, tilts=tilts,
                                                            tilt_grad_arr=tg)
    assert not g.any()
    np.savez_compressed(os.path.join(HERE, "p1_vertex.npz"), pos=pos, tri=tri, tilts=tilts, div_v=div_v, area_v=area_v,
                        smooth_k=np.float64(0.7), smooth_E=np.float64(e_s), smooth_tg=tg)
    print("p1_vertex", len(pos), len(tri), float(np.abs(div_v).max()))


def tilt_relaxation_vectors():
    """Row f3: the reference's leaflet tilt relaxation (``TiltRelaxationManager.relax_leaflet_tilts``, gradient-
    descent solver, frozen geometry) on the caveolin free-disk mesh with its four leaflet energy modules and NO
    tilt constraint modules.  Stores the initial state, the selections as masks and the relaxed tilt fields."""
    from modules.energy.bt_params import (_assume_J0_center_xy, _assume_J0_presets, _assume_J0_radius_max,
                                          _per_vertex_params_leaflet)
    from modules.energy.bt_selection import _collect_preset_rows, _interior_mask_leaflet
    from modules.energy.leaflet_presence import leaflet_absent_vertex_mask, leaflet_present_triangle_mask

    path = os.path.join(REF, "meshes", "caveolin",
                        "kozlov_1disk_3d_tensionless_single_leaflet_profile_hard_rim_R12_free_disk.yaml")
    out = {}
    for case, steps, step_size, solver, extra in (("gd5", 5, 0.15, "gd", {}), ("gd4small", 4, 0.003, "gd", {}),
                                                  ("gdreject", 3, 40.0, "gd", {}), ("cg6", 6, 0.15, "cg", {}),
                                                  ("cg5plain", 5, 0.15, "cg", {"tilt_cg_preconditioner": "none"}),
                                                  ("cg6big", 6, 1.0, "cg", {"tilt_cg_rejection_fallback": "gd"})):
        mesh = _refined(path, 1)
        gp = mesh.global_parameters
        gp.set("tilt_solver", solver)
        for k_extra, v_extra in extra.items():
            gp.set(k_extra, v_extra)
        gp.set("tilt_solve_mode", "nested")
        gp.set("tilt_inner_steps", steps)
        gp.set("tilt_step_size", step_size)
        gp.set("tilt_tol", 0.0)
        rng = np.random.default_rng(31)
        nv = len(mesh.vertex_ids)
        for row, vid in enumerate(mesh.vertex_ids):
            v = mesh.vertices[int(vid)]
            v.position = np.asarray(v.position, dtype=float) + np.array([0.0, 0.0, 0.05 * rng.standard_normal()])
            if not getattr(v, "tilt_fixed_in", False):
                v.tilt_in = 0.05 * rng.standard_normal(3)
            if not getattr(v, "tilt_fixed_out", False):
                v.tilt_out = 0.05 * rng.standard_normal(3)
        mesh.increment_version()
        if hasattr(mesh, "touch_tilts_in"):
            mesh.touch_tilts_in()
            mesh.touch_tilts_out()
        names = ["bending_tilt_in", "bending_tilt_out", "tilt_in", "tilt_out"]
        mesh.energy_modules = list(names)
        mesh.constraint_modules = []
        mini = Minimizer(mesh, gp, GradientDescent(), EnergyModuleManager(names), ConstraintModuleManager([]), quiet=True)
        pos = np.array(mesh.positions_view())
        idx = mesh.vertex_index_to_row
        tri = np.ascontiguousarray(mesh.triangle_row_cache()[0], dtype=np.int32)
        isb = np.zeros(nv, bool)
        for vid in mesh.boundary_vertex_ids:
            isb[idx[vid]] = True
        pre = case + "_"
        out[pre + "pos"], out[pre + "tri"], out[pre + "is_boundary"] = pos, tri, isb
        out[pre + "tilts_in0"], out[pre + "tilts_out0"] = np.array(mesh.tilts_in_view()), np.array(mesh.tilts_out_view())
        out[pre + "fixed_in"], out[pre + "fixed_out"] = np.array(mini._tilt_fixed_mask_in()), np.array(mini._tilt_fixed_mask_out())
        for leaf in ("in", "out"):
            am = leaflet_absent_vertex_mask(mesh, gp, leaflet=leaf)
            keep = leaflet_present_triangle_mask(mesh, tri, absent_vertex_mask=am)
            out[pre + f"{leaf}_keep"] = np.ones(len(tri), bool) if keep.size == 0 else np.asarray(keep, bool)
            out[pre + f"{leaf}_interior"] = np.asarray(_interior_mask_leaflet(mesh, gp, cache_tag=leaf, index_map=idx), bool)
            bz = np.zeros(nv, bool)
            presets = _assume_J0_presets(gp, cache_tag=leaf)
            if presets:
                bz[_collect_preset_rows(mesh, presets=presets, cache_tag=leaf, index_map=idx,
                                        radius_max=_assume_J0_radius_max(gp, cache_tag=leaf),
                                        center_xy=_assume_J0_center_xy(gp))] = True
            out[pre + f"{leaf}_base_zero"] = bz
            kap, c0 = _per_vertex_params_leaflet(mesh, gp, model="helfrich", kappa_key=f"bending_modulus_{leaf}",
                                                 cache_tag=leaf)
            out[pre + f"{leaf}_kappa"], out[pre + f"{leaf}_c0"] = np.array(kap), np.array(c0)
            out[pre + f"{leaf}_k_tilt"] = np.float64(gp.get(f"tilt_modulus_{leaf}"))
        stats = mini._relax_leaflet_tilts(positions=mesh.positions_view(), mode="nested")
        out[pre + "tilts_in1"], out[pre + "tilts_out1"] = np.array(mesh.tilts_in_view()), np.array(mesh.tilts_out_view())
        for k in ("accepted_steps", "backtracking_steps", "initial_energy", "final_energy", "initial_gradient_norm",
                  "final_gradient_norm"):
            out[pre + k] = np.float64(stats[k])
        out[pre + "steps"], out[pre + "step_size"] = np.int64(steps), np.float64(step_size)
        out[pre + "solver"] = np.array(solver)
        out[pre + "preconditioner"] = np.bool_(extra.get("tilt_cg_preconditioner", "jacobi") == "jacobi")
        out[pre + "gd_fallback"] = np.bool_(extra.get("tilt_cg_rejection_fallback", "off") == "gd")
        out[pre + "k_smooth_in"] = np.float64(gp.get("bending_modulus_in") or gp.get("bending_modulus") or 0.0)
        out[pre + "k_smooth_out"] = np.float64(gp.get("bending_modulus_out") or gp.get("bending_modulus") or 0.0)
        out[pre + "rejected_steps"] = np.float64(stats["rejected_steps"])
        out[pre + "stop_reason"] = np.array(str(stats["stop_reason"]))
        print(case, {k: stats[k] for k in ("accepted_steps", "backtracking_steps", "stop_reason", "initial_energy",
                                           "final_energy", "initial_gradient_norm", "final_gradient_norm")})
    np.savez_compressed(os.path.join(HERE, "tilt_relaxation.npz"), **out)


def tilt_relaxation_constrained_vectors():
    """Row f3 with the tilt CONSTRAINT modules configs[3] ships (``tilt_thetaB_boundary_in``, ``rim_slope_match_out``
    next to ``rigid_disk`` / ``pin_to_plane`` / ``pin_to_circle``): the reference's ``relax_leaflet_tilts`` on the
    caveolin free-disk mesh with its constraint manager in place.  The two places where the constraint manager
    touches the loop are recorded call by call -- arrays going in, arrays coming out -- so that the device relaxer
    can be driven along the same trajectory without the reference: ``{case}_ghook_{k}_*`` for
    ``apply_tilt_gradient_modifications_array`` and ``{case}_refresh_{k}_*`` for ``enforce_tilt_constraints``."""
    from modules.energy.bt_params import (_assume_J0_center_xy, _assume_J0_presets, _assume_J0_radius_max,
                                          _per_vertex_params_leaflet)
    from modules.energy.bt_selection import _collect_preset_rows, _interior_mask_leaflet
    from modules.energy.leaflet_presence import leaflet_absent_vertex_mask, leaflet_present_triangle_mask

    path = os.path.join(REF, "meshes", "caveolin",
                        "kozlov_1disk_3d_tensionless_single_leaflet_profile_hard_rim_R12_free_disk.yaml")
    out = {}
    for case, steps, step_size, solver, extra in (("cgd4", 4, 0.15, "gd", {}), ("ccg5", 5, 0.15, "cg", {}),
                                                  ("cgd6i2", 6, 0.05, "gd", {"tilt_projection_interval": 2}),
                                                  ("ccg4pass", 4, 0.15, "cg", {"tilt_projection_cadence": "per_pass"})):
        mesh = _refined(path, 1)
        gp = mesh.global_parameters
        gp.set("tilt_solver", solver)
        for k_extra, v_extra in extra.items():
            gp.set(k_extra, v_extra)
        gp.set("tilt_solve_mode", "nested")
        gp.set("tilt_inner_steps", steps)
        gp.set("tilt_step_size", step_size)
        gp.set("tilt_tol", 0.0)
        rng = np.random.default_rng(37)
        nv = len(mesh.vertex_ids)
        for row, vid in enumerate(mesh.vertex_ids):
            v = mesh.vertices[int(vid)]
            if not getattr(v, "fixed", False):
                v.position = np.asarray(v.position, dtype=float) + np.array([0.0, 0.0, 0.02 * rng.standard_normal()])
            if not getattr(v, "tilt_fixed_in", False):
                v.tilt_in = 0.05 * rng.standard_normal(3)
            if not getattr(v, "tilt_fixed_out", False):
                v.tilt_out = 0.05 * rng.standard_normal(3)
        mesh.increment_version()
        if hasattr(mesh, "touch_tilts_in"):
            mesh.touch_tilts_in()
            mesh.touch_tilts_out()
        names = ["bending_tilt_in", "bending_tilt_out", "tilt_in", "tilt_out"]
        mesh.energy_modules = list(names)
        cons = list(mesh.constraint_modules)
        assert "tilt_thetaB_boundary_in" in cons and "rim_slope_match_out" in cons, cons
        cm = ConstraintModuleManager(cons)
        mini = Minimizer(mesh, gp, GradientDescent(), EnergyModuleManager(names), cm, quiet=True)
        pos = np.array(mesh.positions_view())
        idx = mesh.vertex_index_to_row
        tri = np.ascontiguousarray(mesh.triangle_row_cache()[0], dtype=np.int32)
        isb = np.zeros(nv, bool)
        for vid in mesh.boundary_vertex_ids:
            isb[idx[vid]] = True
        pre = case + "_"
        out[pre + "pos"], out[pre + "tri"], out[pre + "is_boundary"] = pos, tri, isb
        out[pre + "tilts_in0"], out[pre + "tilts_out0"] = np.array(mesh.tilts_in_view()), np.array(mesh.tilts_out_view())
        out[pre + "fixed_in"], out[pre + "fixed_out"] = np.array(mini._tilt_fixed_mask_in()), np.array(mini._tilt_fixed_mask_out())
        for leaf in ("in", "out"):
            am = leaflet_absent_vertex_mask(mesh, gp, leaflet=leaf)
            keep = leaflet_present_triangle_mask(mesh, tri, absent_vertex_mask=am)
            out[pre + f"{leaf}_keep"] = np.ones(len(tri), bool) if keep.size == 0 else np.asarray(keep, bool)
            out[pre + f"{leaf}_interior"] = np.asarray(_interior_mask_leaflet(mesh, gp, cache_tag=leaf, index_map=idx), bool)
            bz = np.zeros(nv, bool)
            presets = _assume_J0_presets(gp, cache_tag=leaf)
            if presets:
                bz[_collect_preset_rows(mesh, presets=presets, cache_tag=leaf, index_map=idx,
                                        radius_max=_assume_J0_radius_max(gp, cache_tag=leaf),
                                        center_xy=_assume_J0_center_xy(gp))] = True
            out[pre + f"{leaf}_base_zero"] = bz
            kap, c0 = _per_vertex_params_leaflet(mesh, gp, model="helfrich", kappa_key=f"bending_modulus_{leaf}",
                                                 cache_tag=leaf)
            out[pre + f"{leaf}_kappa"], out[pre + f"{leaf}_c0"] = np.array(kap), np.array(c0)
            out[pre + f"{leaf}_k_tilt"] = np.float64(gp.get(f"tilt_modulus_{leaf}"))
        # -- record the two hooks call by call
        ghook, refresh = [], []
        orig_mod, orig_enf = cm.apply_tilt_gradient_modifications_array, cm.enforce_tilt_constraints

        def rec_mod(g_in, g_out, *a, **kw):
            before = (np.array(g_in), np.array(g_out), np.array(kw["tilts_in"]), np.array(kw["tilts_out"]))
            orig_mod(g_in, g_out, *a, **kw)
            ghook.append(before + (np.array(g_in), np.array(g_out)))

        def rec_enf(m, **kw):
            before = (np.array(m.tilts_in_view()), np.array(m.tilts_out_view()))
            orig_enf(m, **kw)
            refresh.append(before + (np.array(m.tilts_in_view()), np.array(m.tilts_out_view())))

        cm.apply_tilt_gradient_modifications_array = rec_mod
        cm.enforce_tilt_constraints = rec_enf
        stats = mini._relax_leaflet_tilts(positions=mesh.positions_view(), mode="nested")
        assert np.array_equal(np.array(mesh.positions_view()), pos), "the tilt block moved the geometry"
        out[pre + "tilts_in1"], out[pre + "tilts_out1"] = np.array(mesh.tilts_in_view()), np.array(mesh.tilts_out_view())
        out[pre + "n_ghook"], out[pre + "n_refresh"] = np.int64(len(ghook)), np.int64(len(refresh))
        for k, (gi, go, ti, to, gi2, go2) in enumerate(ghook):
            q = pre + f"ghook_{k}_"
            if k < 2:      # full arrays for the first calls, then their norms + the rows that change (fixture size)
                out[q + "g_in"], out[q + "g_out"], out[q + "t_in"], out[q + "t_out"] = gi, go, ti, to
            out[q + "norms"] = np.array([np.linalg.norm(x) for x in (gi, go, ti, to)])
            out[q + "old_in"], out[q + "old_out"] = gi[np.flatnonzero(np.any(gi2 != gi, axis=1))], go[np.flatnonzero(np.any(go2 != go, axis=1))]
            rows_in = np.flatnonzero(np.any(gi2 != gi, axis=1))
            rows_out = np.flatnonzero(np.any(go2 != go, axis=1))
            out[q + "rows_in"], out[q + "new_in"] = rows_in, gi2[rows_in]        # sparse: a few rim rows change
            out[q + "rows_out"], out[q + "new_out"] = rows_out, go2[rows_out]
        for k, (ti, to, ti2, to2) in enumerate(refresh):
            q = pre + f"refresh_{k}_"
            if k < 2:
                out[q + "t_in"], out[q + "t_out"] = ti, to
            out[q + "norms"] = np.array([np.linalg.norm(x) for x in (ti, to)])
            rows_in = np.flatnonzero(np.any(ti2 != ti, axis=1))
            rows_out = np.flatnonzero(np.any(to2 != to, axis=1))
            out[q + "old_in"], out[q + "old_out"] = ti[rows_in], to[rows_out]
            out[q + "rows_in"], out[q + "new_in"] = rows_in, ti2[rows_in]
            out[q + "rows_out"], out[q + "new_out"] = rows_out, to2[rows_out]
        for k in ("accepted_steps", "backtracking_steps", "initial_energy", "final_energy", "initial_gradient_norm",
                  "final_gradient_norm"):
            out[pre + k] = np.float64(stats[k])
        out[pre + "steps"], out[pre + "step_size"] = np.int64(steps), np.float64(step_size)
        out[pre + "solver"] = np.array(solver)
        out[pre + "interval"] = np.int64(extra.get("tilt_projection_interval", 1))
        out[pre + "cadence"] = np.array(extra.get("tilt_projection_cadence", "per_step"))
        out[pre + "preconditioner"] = np.bool_(True)
        out[pre + "gd_fallback"] = np.bool_(False)
        out[pre + "k_smooth_in"] = np.float64(gp.get("bending_modulus_in") or gp.get("bending_modulus") or 0.0)
        out[pre + "k_smooth_out"] = np.float64(gp.get("bending_modulus_out") or gp.get("bending_modulus") or 0.0)
        out[pre + "rejected_steps"] = np.float64(stats["rejected_steps"])
        out[pre + "stop_reason"] = np.array(str(stats["stop_reason"]))
        print(case, len(ghook), len(refresh),
              {k: stats[k] for k in ("accepted_steps", "backtracking_steps", "stop_reason", "initial_energy",
                                     "final_energy", "initial_gradient_norm", "final_gradient_norm")},
              "changed rows per gradient hook", [int(len(out[pre + f"ghook_{k}_rows_in"])) for k in range(len(ghook))][:3],
              [int(len(out[pre + f"ghook_{k}_rows_out"])) for k in range(len(ghook))][:3])
    np.savez_compressed(os.path.join(HERE, "tilt_relaxation_constrained.npz"), **out)


def vertex_average_vectors():
    """runtime/vertex_average.py on a jittered refined cube (closed) and on the catenoid (fixed rims)."""
    from runtime.vertex_average import vertex_average

    out = {}
    for name, path, levels in (("cube", os.path.join(REF, "meshes", "cube.json"), 2),
                               ("catenoid", os.path.join(REF, "meshes", "catenoid.json"), 2)):
        mesh = _refined(path, levels)
        rng = np.random.default_rng(13)
        for v in mesh.vertices.values():
            if not getattr(v, "fixed", False):
                v.position = np.asarray(v.position, dtype=float) + 0.03 * rng.normal(size=3)
        mesh.increment_version()
        out[f"{name}_pos0"] = np.array(mesh.positions_view())
        out[f"{name}_tri"] = np.ascontiguousarray(mesh.triangle_row_cache()[0], dtype=np.int32)
        out[f"{name}_fixed"] = np.array([bool(mesh.vertices[int(v)].fixed) for v in mesh.vertex_ids])
        vertex_average(mesh)
        out[f"{name}_pos1"] = np.array(mesh.positions_view())
        print("vertex_average", name, len(mesh.vertex_ids), float(np.abs(out[f"{name}_pos1"] - out[f"{name}_pos0"]).max()))
    np.savez_compressed(os.path.join(HERE, "vertex_average.npz"), **out)


if __name__ == "__main__":
    _ = (volume_constraint, volume_energy)
    if len(sys.argv) > 1 and sys.argv[1] == "leaflet":
        leaflet_vectors()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "tiltrelax":
        tilt_relaxation_vectors()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "tilt_relaxation_constrained":
        tilt_relaxation_constrained_vectors()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "vertexaverage":
        vertex_average_vectors()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "equiangulate":
        equiangulate_vectors()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "replay":
        replay_vectors()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "p1vertex":
        p1_vertex_vectors()
        sys.exit(0)
    kernel_vectors()
    module_vectors()
    minimizer_vectors()
    trajectory_vectors()
    replay_vectors()
    leaflet_vectors()
    p1_vertex_vectors()
    tilt_relaxation_vectors()
    tilt_relaxation_constrained_vectors()
    vertex_average_vectors()
    equiangulate_vectors()
