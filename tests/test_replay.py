"""SURVEY.md appendix B / BASELINE configs[0..2]: the reference's benchmark instruction lists.

``tests/golden/replay.npz`` (``generate_golden.py replay_vectors``) holds the dense state after EVERY instruction of
``benchmarks/inputs/bench_cube.json``, ``bench_catenoid.json`` and the ``gogo`` macro of ``meshes/bending_cube.yaml``
as the UNMODIFIED reference produced them, with its per-module energies and its total projected gradient.  Here every
stored state is re-evaluated through the plugin layer (``EnergyModuleManager`` / ``EvaluationManager`` twins) -- on
the host emulator in the CPU tier, on the device through the C ABI in the GPU tier -- at 1e-12, and the end points
must be the survey's known answers.  The replay of the instruction lists THROUGH the plugins (reference command
language, refinement, equiangulation, steppers) is ``test_dropin_reference.py``, which needs a checkout of the
original project (``MEMBRANE_REFERENCE_ROOT``)."""

import json

import numpy as np
import pytest

import ms_test_helpers as H
from ms_test_helpers import rel_err

from membrane_solver_b200 import _lib as L
from membrane_solver_b200.geometry.array_mesh import ArrayBody, ArrayMesh, GlobalParams, ParamResolver
from membrane_solver_b200.runtime import device_state
from membrane_solver_b200.runtime.energy_manager import EnergyModuleManager
from membrane_solver_b200.runtime.evaluation_manager import EvaluationManager

END_POINTS = {"cube": ("surface", 4.840039760362666, 0.9999999999999997),
              "catenoid": ("surface", 34.63728489557314, None),
              "bcube": ("bending", 24.75545218783622, 1.0000000000000002)}


@pytest.fixture(scope="module")
def gold():
    return np.load(H.GOLDEN + "/replay.npz")


@pytest.fixture(params=[pytest.param("emulator", id="emulator"),
                        pytest.param("gpu", id="gpu", marks=pytest.mark.gpu)])
def backend(request, monkeypatch):
    if request.param == "emulator":
        from fake_device import FakeDeviceMesh

        monkeypatch.setattr(device_state, "DEVICE_MESH_FACTORY", FakeDeviceMesh)
    elif L.device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu tier must run on the B200 box")
    return request.param


def _state(gold, name, k):
    pre = f"{name}_{k:02d}_"
    prm = json.loads(str(gold[f"{name}_params_json"]))
    gp = GlobalParams(**prm)
    bodies = {}
    if pre + "body_rows_0" in gold.files:
        t = float(gold[pre + "body_target_0"])
        bodies[0] = ArrayBody(gold[pre + "body_rows_0"], target_volume=None if np.isnan(t) else t)
    mesh = ArrayMesh(gold[pre + "pos"], gold[pre + "tri"], global_params=gp,
                     facet_params={"surface_tension": gold[pre + "gamma"]}, bodies=bodies, fixed=gold[pre + "fixed"])
    names = [str(x) for x in gold[pre + "modules"]]
    mgr = EnergyModuleManager(names)
    ev = EvaluationManager(mesh=mesh, global_params=gp, param_resolver=ParamResolver(gp),
                           energy_modules=[mgr.get_module(n) for n in names], energy_module_names=names)
    return pre, mesh, ev, names, [str(x) for x in gold[pre + "constraints"]]


@pytest.mark.parametrize("name", ["cube", "catenoid", "bcube"])
def test_every_replayed_state_re_evaluates_like_the_reference(backend, gold, name):
    n = int(gold[f"{name}_count"])
    assert n >= 7
    for k in range(n):
        pre, mesh, ev, names, cons = _state(gold, name, k)
        pos = mesh.positions_view()
        assert set(mesh.boundary_vertex_ids) == set(np.nonzero(gold[pre + "is_boundary"])[0].tolist())
        if "volume" in cons:   # single volume constraint: KKT projection + fixed mask on the device
            e, g, res = ev.compute_energy_and_projected_gradient(positions=pos)
            assert abs(res.volume - float(gold[pre + "volume"])) <= 1e-12 * abs(float(gold[pre + "volume"]))
        else:                  # catenoid: the pinned rims are fixed rows; no multiplier
            e, g = ev.compute_energy_and_gradient_array(positions=pos)
            g[np.asarray(gold[pre + "fixed"], bool)] = 0.0
        want_e, want_g = float(gold[pre + "E"]), gold[pre + "g"]
        assert abs(e - want_e) <= 1e-12 * max(1.0, abs(want_e)), (k, str(gold[pre + "instruction"]))
        tol = 2e-12 if "bending" in names else 1e-12
        assert rel_err(g, want_g) <= tol, (k, str(gold[pre + "instruction"]), rel_err(g, want_g))
        bd = ev.compute_energy_breakdown(positions=pos)
        for mod in names:
            want = float(gold[pre + f"E_{mod}"])
            assert abs(bd[mod] - want) <= 1e-12 * max(1.0, abs(want)), (k, mod)
    # the end point is the survey's known answer (appendix B)
    mod, e_end, v_end = END_POINTS[name]
    pre, mesh, ev, names, cons = _state(gold, name, n - 1)
    bd = ev.compute_energy_breakdown(positions=mesh.positions_view())
    assert abs(bd[mod] - e_end) <= 1e-9 * abs(e_end), (bd[mod], e_end)
    if v_end is not None:
        _, _, res = ev.compute_energy_and_projected_gradient(positions=mesh.positions_view())
        assert abs(res.volume - v_end) <= 1e-12


CAVEOLIN_END = {"bending_tilt_in": 0.24157305138432794, "bending_tilt_out": 0.008943176191835553,
                "tilt_in": 0.45430920811328745, "tilt_out": 0.0006887388044462964}


def test_caveolin_end_state_module_energies(backend, gold):
    """BASELINE configs[3]: the state the reference reaches with its macro ``profile_relax_light`` on the caveolin
    free-disk mesh (1 129 vertices / 2 208 facets).  The four leaflet modules of the path, fed with the mesh OPTIONS
    (selections derived by leaflet_selection.py), give the reference's energies -- the survey's known answers; the
    fifth module of that mesh (tilt_thetaB_contact_in) is not on the path."""
    import importlib

    vopts = {int(k): v for k, v in json.loads(str(gold["caveolin_vertex_options_json"])).items()}
    gp = GlobalParams(json.loads(str(gold["caveolin_global_params_json"])))
    mesh = ArrayMesh(gold["caveolin_pos"], gold["caveolin_tri"], global_params=gp, vertex_options=vopts,
                     tilts_in=gold["caveolin_tilts_in"], tilts_out=gold["caveolin_tilts_out"])
    assert gold["caveolin_tri"].shape == (2208, 3) and gold["caveolin_pos"].shape == (1129, 3)
    res = ParamResolver(gp)
    pos = mesh.positions_view()
    for name, want in CAVEOLIN_END.items():
        mod = importlib.import_module(f"membrane_solver_b200.modules.energy.{name}")
        e = mod.compute_energy_array(mesh, gp, res, positions=pos, index_map=mesh.vertex_index_to_row)
        assert abs(e - float(gold[f"caveolin_E_{name}"])) <= 1e-12 * max(1.0, abs(want)), (name, e)
        assert abs(e - want) <= 1e-9 * abs(want), (name, e, want)
    # the manager's leaflet entry point sums them in one paired device evaluation
    names = list(CAVEOLIN_END)
    mgr = EnergyModuleManager(names)
    ev = EvaluationManager(mesh=mesh, global_params=gp, param_resolver=res,
                           energy_modules=[mgr.get_module(n) for n in names], energy_module_names=names)
    total = ev.compute_tilt_dependent_energy_with_leaflet_tilts(positions=pos, tilts_in=mesh.tilts_in_view(),
                                                                tilts_out=mesh.tilts_out_view())
    assert abs(total - sum(CAVEOLIN_END.values())) <= 1e-9 * sum(CAVEOLIN_END.values())


def test_mesh_operations_of_the_instruction_lists_on_arrays(backend, gold):
    """Rows f2 / f4 on the benchmark sequences: every ``r`` and ``V`` instruction of the three lists, applied to the
    reference's state BEFORE it with the array twins -- 1->4 refinement (``geometry/refine.py``), vertex averaging
    (``geometry/vertex_average.py``) followed, as ``commands/mesh_ops.py:45-53`` does, by the hard volume projection
    (``modules/constraints/volume.py::enforce_constraint`` with volume and dV/dx from the device, 12 iterations of the
    ``mesh_operation`` context) -- must land on the reference's state AFTER it: vertex averaging 1e-12 on the
    positions, refinement the same vertex set and facet count (the reference numbers the new vertices differently)
    and the same energy."""
    from membrane_solver_b200.geometry.refine import refine_triangles
    from membrane_solver_b200.geometry.vertex_average import vertex_average_arrays
    from membrane_solver_b200.modules.constraints import volume as volume_constraint

    checked = {"r": 0, "V": 0}
    for name in ("cube", "catenoid", "bcube"):
        prm = json.loads(str(gold[f"{name}_params_json"]))
        for k in range(1, int(gold[f"{name}_count"])):
            ins = str(gold[f"{name}_{k:02d}_instruction"]).replace(" ", "")
            a, b = f"{name}_{k - 1:02d}_", f"{name}_{k:02d}_"
            pos, tri, fixed = gold[a + "pos"], gold[a + "tri"], np.asarray(gold[a + "fixed"], bool)
            cons = [str(x) for x in gold[b + "constraints"]]
            if ins[0] == "r":
                p, t, f = pos, tri, fixed
                for _ in range(int(ins[1:] or 1)):
                    out = refine_triangles(p, t, f)
                    p, t, f = out[0], out[1], (out[2] if len(out) > 2 else None)
                want = gold[b + "pos"]
                assert p.shape == want.shape and t.shape == gold[b + "tri"].shape
                assert np.array_equal(p[: pos.shape[0]], pos)                  # old vertices keep their rows
                key = lambda x: x[np.lexsort(np.round(x, 9).T[::-1])]          # noqa: E731
                assert np.max(np.abs(key(p) - key(want))) <= 1e-12, (name, k)
                checked["r"] += 1
            elif ins[0] == "V" and cons in ([], ["volume"]):
                if name == "catenoid":
                    continue                        # its rims are pinned by pin_to_circle, which is not on the path
                p = pos
                for _ in range(int(ins[1:] or 1)):
                    p = vertex_average_arrays(p, tri, movable=~fixed)
                if cons == ["volume"]:
                    gp = GlobalParams(**prm)
                    mesh = ArrayMesh(p, tri, global_params=gp, fixed=fixed,
                                     bodies={0: ArrayBody(gold[a + "body_rows_0"],
                                                          target_volume=float(gold[a + "body_target_0"]))})
                    volume_constraint.enforce_constraint(mesh, global_params=gp, context="mesh_operation")
                    p = np.array(mesh.positions_view())
                assert np.max(np.abs(p - gold[b + "pos"])) <= 1e-12, (name, k, ins)
                checked["V"] += 1
    assert checked["r"] >= 4 and checked["V"] >= 5, checked
