"""Drop-in proof against the REAL reference: runs when ``MEMBRANE_REFERENCE_ROOT`` names a checkout of the
original membrane_solver, and skips otherwise.  Every test here runs the original's own code on both sides of the
comparison, so none of them can run from stored vectors alone.  Only part of what they compare has a stored-output
twin under tests/golden/:

* compute_energy_and_gradient_array of the Minimizer: cube r1 and bending_cube r1 (seed 5) in minimizer.npz
  (test_plugins.py); no catenoid case.  GD trajectories of the reference are in trajectory.npz
  (test_device_minimizer.py), but not the three CASES below (cube 6 steps, bending_cube 3, catenoid 4).
* leaflet entry points of the EvaluationManager: leaflet.npz (test_leaflet.py).
* config-4 trajectory (3 full steps on the caveolin disk): NOT stored; test_replay.py checks only the reference's
  stored end state of that mesh.
* tilt relaxer with the reference's constraint manager: its hook calls are recorded in
  tilt_relaxation_constrained.npz (test_leaflet.py).
* instruction lists: the state after every instruction is in replay.npz (test_replay.py); the ``r`` and ``V``
  steps are replayed on arrays.  The ``g``, ``u`` and ``cg`` steps are not, because the stepper state the reference
  carries from one instruction to the next is not stored.
* enforce_constraint: replay.npz holds the reference's positions after ``V`` (``mesh_operation`` context, 12
  iterations), replayed in test_replay.py.  The default 3 iterations and ``force_projection`` from a fresh mesh are
  NOT stored; test_plugins.py checks those only against this project's own Newton step.

Storing what is missing needs generate_golden.py extended and run against a checkout of the original.

The reference's own ``Minimizer`` / ``EnergyModuleManager`` / ``ConstraintModuleManager`` run
unmodified; ``membrane_solver_b200.runtime.energy_manager.install()`` binds the B200 plugin twins
under the reference's module names.  On the CPU tier the device is the host emulator, so what is
proven here is the CONTRACT (names, signatures, accumulate semantics, version-keyed residency)
and the per-facet code; the kernels themselves are proven by the gpu tier."""

import importlib
import os
import sys

import numpy as np
import pytest

REF = os.environ.get("MEMBRANE_REFERENCE_ROOT", "")
pytestmark = pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, "runtime")),
                                reason="runs the original membrane_solver: set MEMBRANE_REFERENCE_ROOT to a checkout of it")

CASES = [("meshes/cube.json", 1, 6), ("meshes/bending_cube.yaml", 1, 3), ("meshes/catenoid.json", 1, 4)]


def _ref_imports():
    sys.dont_write_bytecode = True
    if REF not in sys.path:
        sys.path.insert(0, REF)
    from geometry.geom_io import load_data, parse_geometry
    from runtime.constraint_manager import ConstraintModuleManager
    from runtime.energy_manager import EnergyModuleManager
    from runtime.minimizer import Minimizer
    from runtime.refinement import refine_triangle_mesh
    from runtime.steppers.gradient_descent import GradientDescent

    return load_data, parse_geometry, ConstraintModuleManager, EnergyModuleManager, Minimizer, refine_triangle_mesh, GradientDescent


def _build(path, levels, seed=5):
    load_data, parse_geometry, CMM, EMM, Minimizer, refine, GD = _ref_imports()
    mesh = parse_geometry(load_data(os.path.join(REF, path)))
    for _ in range(levels):
        mesh = refine(mesh)
    rng = np.random.default_rng(seed)
    for v in mesh.vertices.values():
        if not getattr(v, "fixed", False):
            v.position = np.asarray(v.position, dtype=float) + 0.01 * rng.normal(size=3)
    mesh.increment_version()
    gp = mesh.global_parameters
    mini = Minimizer(mesh, gp, GD(), EMM(mesh.energy_modules), CMM(mesh.constraint_modules), quiet=True)
    return mesh, mini


@pytest.fixture
def b200_installed(monkeypatch):
    from fake_device import FakeDeviceMesh

    from membrane_solver_b200.runtime import device_state, energy_manager

    _ref_imports()
    saved = {k: sys.modules.get(k) for k in list(sys.modules) if k.startswith("modules.energy.")}
    import modules.constraints.volume as ref_cv

    saved_cv = (ref_cv.constraint_gradients_array, ref_cv.constraint_gradients, ref_cv.enforce_constraint)
    monkeypatch.setattr(device_state, "DEVICE_MESH_FACTORY", FakeDeviceMesh)
    yield energy_manager.install
    for name in energy_manager.NAMES:
        key = f"modules.energy.{name}"
        if saved.get(key) is not None:
            sys.modules[key] = saved[key]
        else:
            sys.modules.pop(key, None)
            importlib.import_module(key)
        import modules.energy as pkg

        setattr(pkg, name, sys.modules[key])
    ref_cv.constraint_gradients_array, ref_cv.constraint_gradients, ref_cv.enforce_constraint = saved_cv


@pytest.mark.parametrize("path,levels,steps", CASES, ids=[c[0].split("/")[-1] for c in CASES])
def test_reference_minimizer_runs_on_b200_plugins(b200_installed, path, levels, steps):
    # 1. the unmodified reference
    mesh_ref, mini_ref = _build(path, levels)
    e_ref, g_ref = mini_ref.compute_energy_and_gradient_array()
    bd_ref = mini_ref.compute_energy_breakdown()
    res_ref = mini_ref.minimize(n_steps=steps)
    # 2. the same driver code with the B200 plugins bound under the reference's names
    bound = b200_installed()
    assert "modules.energy.surface" in bound
    mesh, mini = _build(path, levels)
    for name, mod in zip(mini.energy_module_names if hasattr(mini, "energy_module_names") else mesh.energy_modules,
                         mini.energy_modules):
        if name in ("surface", "volume", "bending", "tilt"):
            assert mod.__name__.startswith("membrane_solver_b200."), (name, mod.__name__)
    e, g = mini.compute_energy_and_gradient_array()
    assert abs(e - e_ref) <= 1e-12 * max(1.0, abs(e_ref))
    assert np.max(np.abs(g - g_ref)) <= 1e-11 * max(1.0, np.max(np.abs(g_ref)))
    bd = mini.compute_energy_breakdown()
    for k, v in bd_ref.items():
        assert abs(bd[k] - v) <= 1e-11 * max(1.0, abs(v)), k
    # topology was packed once; every evaluation re-sent positions only
    assert mesh._b200_state.uploads == 1
    # 3. minimised-energy trajectory (BASELINE.json north_star: agree within 1e-9)
    res = mini.minimize(n_steps=steps)
    e_end_ref, e_end = mini_ref.compute_energy(), mini.compute_energy()
    assert abs(e_end - e_end_ref) <= 1e-9 * max(1.0, abs(e_end_ref)), (e_end, e_end_ref)
    p_ref = np.array([mesh_ref.vertices[v].position for v in sorted(mesh_ref.vertices)])
    p = np.array([mesh.vertices[v].position for v in sorted(mesh.vertices)])
    assert np.max(np.abs(p - p_ref)) <= 1e-9
    _ = (res, res_ref)


CAVEOLIN = "meshes/caveolin/kozlov_1disk_3d_tensionless_single_leaflet_profile_hard_rim_R12_free_disk.yaml"


def _build_caveolin(seed=3):
    load_data, parse_geometry, CMM, EMM, Minimizer, refine, GD = _ref_imports()
    mesh = refine(parse_geometry(load_data(os.path.join(REF, CAVEOLIN))))
    rng = np.random.default_rng(seed)
    nv = len(mesh.vertex_ids)
    pos = np.array(mesh.positions_view())
    pos[:, 2] += 0.03 * rng.standard_normal(nv)
    tilts_in, tilts_out = 0.1 * rng.standard_normal((nv, 3)), 0.1 * rng.standard_normal((nv, 3))
    gp = mesh.global_parameters
    mini = Minimizer(mesh, gp, GD(), EMM(mesh.energy_modules), CMM(mesh.constraint_modules), quiet=True)
    return mesh, mini, pos, tilts_in, tilts_out


def test_reference_leaflet_entry_points_run_on_b200_plugins(b200_installed):
    """BASELINE config 4 (caveolin free disk: bending_tilt_in/out, tilt_in/out + a contact module that stays the
    reference's): the reference's own EvaluationManager drives the B200 leaflet twins; selections come from the
    reference's helpers (leaflet presence, base-term rows, per-vertex parameters)."""

    def run(mini, pos, ti, to):
        ev = mini._evaluation_manager if hasattr(mini, "_evaluation_manager") else mini.evaluation_manager
        gi, go = np.zeros_like(pos), np.zeros_like(pos)
        e_t = ev.compute_energy_and_leaflet_tilt_gradients_array(positions=pos, tilts_in=ti, tilts_out=to,
                                                                 tilt_in_grad_arr=gi, tilt_out_grad_arr=go)
        gi2, go2 = np.zeros_like(pos), np.zeros_like(pos)
        e_only = ev.compute_energy_and_leaflet_tilt_gradients_array(positions=pos, tilts_in=ti, tilts_out=to,
                                                                    tilt_in_grad_arr=gi2, tilt_out_grad_arr=go2,
                                                                    tilt_only=True)
        e_dep = ev.compute_tilt_dependent_energy_with_leaflet_tilts(positions=pos, tilts_in=ti, tilts_out=to)
        e_tot = ev.compute_energy_array_with_leaflet_tilts(positions=pos, tilts_in=ti, tilts_out=to)
        return e_t, gi, go, e_only, gi2, go2, e_dep, e_tot

    mesh_ref, mini_ref, pos, ti, to = _build_caveolin()
    want = run(mini_ref, pos, ti, to)
    mods_ref = {n: m for n, m in zip(mesh_ref.energy_modules, mini_ref.energy_modules)}
    shape_ref = {}
    for name in ("bending_tilt_in", "bending_tilt_out", "tilt_in", "tilt_out"):
        g = np.zeros_like(pos)
        e = mods_ref[name].compute_energy_and_gradient_array(
            mesh_ref, mesh_ref.global_parameters, mini_ref.param_resolver, positions=pos,
            index_map=mesh_ref.vertex_index_to_row, grad_arr=g, tilts_in=ti, tilts_out=to,
            tilt_in_grad_arr=np.zeros_like(pos), tilt_out_grad_arr=np.zeros_like(pos))
        shape_ref[name] = (e, g)

    bound = b200_installed()
    assert "modules.energy.bending_tilt_in" in bound and "modules.energy.tilt_out" in bound
    mesh, mini, pos2, ti2, to2 = _build_caveolin()
    assert np.array_equal(pos, pos2)
    mods = {n: m for n, m in zip(mesh.energy_modules, mini.energy_modules)}
    for name in ("bending_tilt_in", "bending_tilt_out", "tilt_in", "tilt_out"):
        assert mods[name].__name__.startswith("membrane_solver_b200."), mods[name].__name__
    assert not mods["tilt_thetaB_contact_in"].__name__.startswith("membrane_solver_b200.")
    got = run(mini, pos, ti, to)
    for a, b in zip(got, want):
        if np.ndim(b) == 0:
            assert abs(a - b) <= 1e-12 * max(1.0, abs(b)), (a, b)
        else:
            assert np.max(np.abs(a - b)) <= 1e-12 * max(1.0, np.max(np.abs(b)))
    for name, (e_ref, g_ref) in shape_ref.items():
        g = np.zeros_like(pos)
        e = mods[name].compute_energy_and_gradient_array(
            mesh, mesh.global_parameters, mini.param_resolver, positions=pos, index_map=mesh.vertex_index_to_row,
            grad_arr=g, tilts_in=ti, tilts_out=to, tilt_in_grad_arr=np.zeros_like(pos),
            tilt_out_grad_arr=np.zeros_like(pos))
        assert abs(e - e_ref) <= 1e-12 * max(1.0, abs(e_ref)), name
        assert np.max(np.abs(g - g_ref)) <= 1e-12 * max(1.0, np.max(np.abs(g_ref))), name
    assert mesh._b200_state.uploads == 1


def test_reference_minimizer_config4_trajectory_on_b200_leaflet_plugins(b200_installed):
    """BASELINE configs[3]: the reference's full step on the caveolin free-disk mesh -- leaflet tilt relaxation
    (``TiltRelaxationManager.relax_leaflet_tilts``, coupled mode), shape step, rigid-disk / pin / rim constraints --
    unmodified, with the four leaflet energy modules replaced by the B200 twins: same energies, positions and
    tilt fields step by step (north_star: trajectories within 1e-9)."""
    load_data, parse_geometry, CMM, EMM, Minimizer, refine, GD = _ref_imports()

    def run(steps=3):
        mesh = parse_geometry(load_data(os.path.join(REF, CAVEOLIN)))
        mini = Minimizer(mesh, mesh.global_parameters, GD(), EMM(mesh.energy_modules), CMM(mesh.constraint_modules),
                         quiet=True)
        energies = [mini.minimize(n_steps=1)["energy"] for _ in range(steps)]
        return (mini, np.array(energies), np.array(mesh.positions_view()), np.array(mesh.tilts_in_view()),
                np.array(mesh.tilts_out_view()))

    _, e_ref, p_ref, ti_ref, to_ref = run()
    b200_installed()
    mini, e, p, ti, to = run()
    names = [m.__name__ for m in mini.energy_modules]
    assert sum(n.startswith("membrane_solver_b200.") for n in names) == 4, names
    assert np.max(np.abs(e - e_ref)) <= 1e-9 * max(1.0, np.max(np.abs(e_ref))), (e, e_ref)
    assert np.max(np.abs(p - p_ref)) <= 1e-9
    assert np.max(np.abs(ti - ti_ref)) <= 1e-9 and np.max(np.abs(to - to_ref)) <= 1e-9
    assert e[-1] < e[0]


@pytest.mark.parametrize("solver", ["gd", "cg"])
def test_device_tilt_relaxer_with_the_references_constraint_manager(b200_installed, solver):
    """Row f3 on configs[3] AS SHIPPED: the leaflet tilt inner solve of the caveolin free-disk mesh with its tilt
    constraint modules (``tilt_thetaB_boundary_in``, ``rim_slope_match_out``).  The device relaxer
    (``device_tilt_relaxer.relax_leaflet_tilts``) keeps fields, gradients and trials on the device and calls the
    reference's OWN constraint manager through its two hooks; the result is the reference's
    ``TiltRelaxationManager.relax_leaflet_tilts`` (tilt fields 1e-9, energies, step counts)."""
    load_data, parse_geometry, CMM, EMM, Minimizer, refine, GD = _ref_imports()
    from membrane_solver_b200.runtime.device_tilt_relaxer import relax_leaflet_tilts

    def build():
        mesh = refine(parse_geometry(load_data(os.path.join(REF, CAVEOLIN))))
        gp = mesh.global_parameters
        gp.set("tilt_solver", solver)
        gp.set("tilt_solve_mode", "nested")
        gp.set("tilt_inner_steps", 4)
        gp.set("tilt_step_size", 0.15)
        gp.set("tilt_tol", 0.0)
        rng = np.random.default_rng(41)
        for vid in mesh.vertex_ids:
            v = mesh.vertices[int(vid)]
            if not getattr(v, "fixed", False):
                v.position = np.asarray(v.position, dtype=float) + np.array([0.0, 0.0, 0.02 * rng.standard_normal()])
            if not getattr(v, "tilt_fixed_in", False):
                v.tilt_in = 0.05 * rng.standard_normal(3)
            if not getattr(v, "tilt_fixed_out", False):
                v.tilt_out = 0.05 * rng.standard_normal(3)
        mesh.increment_version()
        mesh.touch_tilts_in()
        mesh.touch_tilts_out()
        names = ["bending_tilt_in", "bending_tilt_out", "tilt_in", "tilt_out"]
        mesh.energy_modules = list(names)
        cm = CMM(list(mesh.constraint_modules))
        mini = Minimizer(mesh, gp, GD(), EMM(names), cm, quiet=True)
        return mesh, gp, cm, mini

    mesh_ref, _, _, mini_ref = build()
    want = mini_ref._relax_leaflet_tilts(positions=mesh_ref.positions_view(), mode="nested")
    ti_ref, to_ref = np.array(mesh_ref.tilts_in_view()), np.array(mesh_ref.tilts_out_view())
    assert want["accepted_steps"] > 0

    b200_installed()
    mesh, gp, cm, mini = build()
    start = np.array(mesh.tilts_in_view())
    got = relax_leaflet_tilts(mesh, gp, mini.param_resolver, constraint_manager=cm,
                              positions=np.array(mesh.positions_view()), mode="nested")
    assert got["hook_calls"]["gradient"] >= 4 and got["hook_calls"]["refresh"] >= 2     # the constraint manager was in the loop
    for k in ("accepted_steps", "backtracking_steps"):
        assert got[k] == want[k], k
    assert got["stop_reason"] == want["stop_reason"]
    for k in ("initial_energy", "final_energy", "initial_gradient_norm", "final_gradient_norm"):
        assert abs(got[k] - want[k]) <= 1e-10 * max(1.0, abs(want[k])), k
    assert np.max(np.abs(np.array(mesh.tilts_in_view()) - ti_ref)) <= 1e-9
    assert np.max(np.abs(np.array(mesh.tilts_out_view()) - to_ref)) <= 1e-9
    assert np.max(np.abs(ti_ref - start)) > 1e-3


# ----------------------------------------------------------------------- SURVEY.md appendix B: instruction lists
REPLAY = [
    ("cube", "benchmarks/inputs/bench_cube.json", None, {"surface": 4.840039760362666}),
    ("catenoid", "benchmarks/inputs/bench_catenoid.json", None, {"surface": 34.63728489557314}),
    ("bcube", "meshes/bending_cube.yaml", ["r", "u", "g 50", "r", "u", "g 100", "V"], {"bending": 24.75545218783622}),
]


@pytest.mark.parametrize("name,path,lines,end", REPLAY, ids=[r[0] for r in REPLAY])
def test_benchmark_instruction_lists_replay_on_b200_plugins(b200_installed, name, path, lines, end):
    """The reference's own benchmark inputs (BASELINE configs[0..2]) driven through its own command language
    (g / r / u / V / cg: refinement, equiangulation, vertex averaging, GD and CG steppers, constraint enforcement --
    all the reference's) with the energy modules and the volume constraint gradient on the B200 plugins: the state
    after EVERY instruction follows the unmodified reference's (tests/golden/replay.npz) and the end point is the
    survey's known answer, within 1e-9 (north_star)."""
    from commands.context import CommandContext
    from commands.executor import execute_command_line

    load_data, parse_geometry, CMM, EMM, Minimizer, refine, GD = _ref_imports()
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "replay.npz"))
    bound = b200_installed()
    assert "modules.energy.surface" in bound
    data = load_data(os.path.join(REF, path))
    mesh = parse_geometry(data)
    stepper = GD()
    mini = Minimizer(mesh, mesh.global_parameters, stepper, EMM(mesh.energy_modules), CMM(mesh.constraint_modules),
                     quiet=True)
    mini.step_size = mesh.global_parameters.get("step_size", 1e-3)
    for mod in mini.energy_modules:
        assert mod.__name__.startswith("membrane_solver_b200."), mod.__name__
    ctx = CommandContext(mesh, mini, stepper)
    if lines is None:
        lines = [str(x) for x in data.get("instructions", [])]
    assert int(gold[f"{name}_count"]) == len(lines)
    for k, line in enumerate(lines):
        execute_command_line(ctx, line)
        m = ctx.mesh
        pre = f"{name}_{k:02d}_"
        assert str(gold[pre + "instruction"]) == line
        pos = np.array(m.positions_view())
        assert pos.shape == gold[pre + "pos"].shape, (line, pos.shape)
        assert np.max(np.abs(pos - gold[pre + "pos"])) <= 1e-9, (k, line)
        bd = ctx.minimizer.compute_energy_breakdown()
        for mod, e in bd.items():
            want = float(gold[pre + f"E_{mod}"])
            assert abs(e - want) <= 1e-9 * max(1.0, abs(want)), (k, line, mod, e, want)
    bd = ctx.minimizer.compute_energy_breakdown()
    for mod, want in end.items():
        assert abs(bd[mod] - want) <= 1e-9 * abs(want), (mod, bd[mod], want)


def test_enforce_constraint_twin_matches_the_reference_from_a_fresh_state(b200_installed):
    """modules/constraints/volume.py:69-149 on arrays (SURVEY section 8f rank 2): from a freshly built mesh (no
    cached volume gradient in the reference) the hard projection lands on the same positions, for the default
    3 iterations and for the 12 of the mesh_operation context, with fixed vertices left alone."""
    import modules.constraints.volume as ref_cv

    ref_enforce = ref_cv.enforce_constraint
    from membrane_solver_b200.modules.constraints import volume as twin

    for kwargs in ({}, {"context": "mesh_operation"}, {"force_projection": True, "max_iter": 5}):
        meshes = []
        for _ in range(2):
            mesh, _ = _build("meshes/cube.json", 2, seed=9)
            for k, v in enumerate(mesh.vertices.values()):
                v.position = 1.07 * np.asarray(v.position, dtype=float)      # 22 % too much volume
                if k % 17 == 0:
                    v.fixed = True
            mesh.global_parameters.set("volume_constraint_mode", "lagrange")   # cube.json itself is penalty mode
            mesh.increment_version()
            if hasattr(mesh, "_touch_fixed_flags"):
                mesh._touch_fixed_flags()
            meshes.append(mesh)
        gp = meshes[0].global_parameters
        ref_enforce(meshes[0], global_params=gp, **kwargs)
        b200_installed()
        twin.enforce_constraint(meshes[1], global_params=meshes[1].global_parameters, **kwargs)
        p_ref, p = np.array(meshes[0].positions_view()), np.array(meshes[1].positions_view())
        assert np.max(np.abs(p - p_ref)) <= 1e-12, kwargs
        body = next(iter(meshes[1].bodies.values()))
        if kwargs.get("context") == "mesh_operation":
            assert abs(body.compute_volume(meshes[1]) - 1.0) <= 1e-10
        from membrane_solver_b200.runtime.device_state import get_state

        assert get_state(meshes[1], np.array(meshes[1].positions_view())).uploads == 1   # topology stayed resident
