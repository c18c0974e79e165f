"""The minimiser loop under device control (``ms_ctx_minimize``, ``csrc/ms_minimize.cuh``) against the host loop of
``DeviceMinimizer.minimize_host``.

CPU tier: the control code compiled for the host (tests/emul/minimize_emul.cpp) drives the emulated device
(tests/fake_device.py) action by action; the action sequence with its arguments, the positions, the step sizes, the
history, the conjugate-gradient state and the returned dict must equal the host loop's bit for bit -- on every case of
tests/golden/trajectory.npz and on scripted cases that reach each branch of the loop.

GPU tier: twin contexts, one minimised by the device loop, one by the host loop through the single calls; the same
quantities must agree bitwise, and every call synchronises with the host once."""

import ctypes
import os
import subprocess

import numpy as np
import pytest

import ms_test_helpers as H
from fake_device import FakeDeviceMesh
from membrane_solver_b200 import _lib as L
from membrane_solver_b200.runtime.device_minimizer import DeviceMinimizer

(EVAL_GRAD, DIRECTION, STATS, EVAL_ENERGY, MAKE_TRIAL, GUARD, ENF_EVAL_POS, ENF_EVAL_TRIAL, ENF_AXPY_POS,
 ENF_AXPY_TRIAL, EVAL_TRIAL, ACCEPT, DRIFT_EVAL, DONE) = range(14)
CASES = ["cube", "bcube", "cubecg", "bcubep", "bcubepcg"]


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    """tests/emul/minimize_emul.cpp compiled for the host into a temporary directory (the tree may be read-only)."""
    out = str(tmp_path_factory.mktemp("mn_emul") / "libms_mn_emul.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-o", out,
                           os.path.join(H.ROOT, "tests", "emul", "minimize_emul.cpp")])
    lib = ctypes.CDLL(out)
    assert lib.emul_min_opts_bytes() == ctypes.sizeof(L.MinimizeOpts)
    return lib


# -- the two drivers on the emulated device -------------------------------------------------------------------------
class Recording(FakeDeviceMesh):
    """The emulated device with a log of the loop's calls as (action, argument) and optional scripted answers."""

    def __init__(self, *, trial_energy=None, guard=None, stats=None):
        super().__init__(0)
        self.log = []
        self.trial_energy, self.guard, self.stats = trial_energy, guard, stats
        self.n_trial_evals = self.n_guards = 0

    def eval(self, opts):
        m, grad, trial = opts["modules"], bool(opts.get("want_grad", True)), bool(opts.get("use_trial"))
        if m == L.MOD_VOLUME and opts.get("constraint_mode", -1) == -1 and not opts.get("apply_fixed"):
            act = (ENF_EVAL_TRIAL if trial else ENF_EVAL_POS) if grad else DRIFT_EVAL
        else:
            act = EVAL_GRAD if grad else (EVAL_TRIAL if trial else EVAL_ENERGY)
        self.log.append((act, None))
        res = super().eval(opts)
        if act == EVAL_TRIAL and self.trial_energy is not None:
            off = self.trial_energy(self.n_trial_evals)  # added to every energy term _total may read
            for k in (L.SC_E_SURFACE, L.SC_E_BENDING):
                res.scalars[k] += off
            self.scalars = res.scalars.copy()
            self.n_trial_evals += 1
        return res

    def direction_from_gradient(self, scale=-1.0):
        self.log.append((DIRECTION, None))
        super().direction_from_gradient(scale)

    def cg_direction(self, restart):
        self.log.append((DIRECTION, bool(restart)))
        super().cg_direction(restart)

    def line_search_stats(self):
        self.log.append((STATS, None))
        out = super().line_search_stats()
        return self.stats(out) if self.stats else out

    def make_trial(self, alpha):
        self.log.append((MAKE_TRIAL, float(alpha).hex()))
        super().make_trial(alpha)

    def normal_change_ok(self, limit=0.5):
        self.log.append((GUARD, None))
        ok = super().normal_change_ok(limit)
        if self.guard is not None:
            ok = self.guard(self.n_guards, ok)
        self.n_guards += 1
        return ok

    def axpy(self, dst, src, alpha, skip_fixed=True):
        self.log.append((ENF_AXPY_TRIAL if dst == L.ARR_TRIAL else ENF_AXPY_POS, float(alpha).hex()))
        super().axpy(dst, src, alpha, skip_fixed)

    def accept_trial(self):
        self.log.append((ACCEPT, None))
        super().accept_trial()


def drive(lib, mini, n_steps):
    """DeviceMinimizer.minimize with the control code of ms_ctx_minimize taking every decision (the emulated device
    runs the actions); returns the result dict and updates the minimiser like the device path does."""
    dm = mini.dm
    opts = mini.minimize_options()
    state = ctypes.create_string_buffer(lib.emul_min_state_bytes())
    lib.emul_min_init.argtypes = [ctypes.c_void_p, ctypes.c_double, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                  ctypes.c_int32]
    lib.emul_min_init(state, mini.step_size, mini._cg_iter, int(mini._cg_have_history), int(dm._pg is not None),
                      int(n_steps))
    cap = max(int(n_steps), 1)
    hist = np.zeros((cap, 4))
    sc, ls, ok = np.zeros(L.SC_COUNT), np.zeros(4), 1
    alpha, neg_lam, restart = ctypes.c_double(), ctypes.c_double(), ctypes.c_int32()
    while True:
        act = lib.emul_min_step(ctypes.byref(opts), state, L.dptr(sc), L.dptr(ls), int(ok), L.dptr(hist), cap)
        if act == DONE:
            break
        lib.emul_min_args(state, ctypes.byref(alpha), ctypes.byref(neg_lam), ctypes.byref(restart))
        if act == EVAL_GRAD:
            sc = dm.eval(mini._opts(want_grad=True)).scalars
        elif act == DIRECTION:
            if mini.stepper == "cg":
                dm.cg_direction(bool(restart.value))
                dm.cg_commit()
            else:
                dm.direction_from_gradient(-1.0)
        elif act == STATS:
            ls = np.array(dm.line_search_stats())
        elif act in (EVAL_ENERGY, EVAL_TRIAL):
            sc = dm.eval(mini._opts(want_grad=False, use_trial=act == EVAL_TRIAL)).scalars
        elif act == MAKE_TRIAL:
            dm.make_trial(alpha.value)
        elif act == GUARD:
            ok = int(dm.normal_change_ok(0.5))
        elif act in (ENF_EVAL_POS, ENF_EVAL_TRIAL):
            sc = dm.eval(dm.options(L.MOD_VOLUME, want_grad=True, use_trial=act == ENF_EVAL_TRIAL)).scalars
        elif act in (ENF_AXPY_POS, ENF_AXPY_TRIAL):
            dm.axpy(L.ARR_TRIAL if act == ENF_AXPY_TRIAL else L.ARR_POSITIONS, L.ARR_VOLGRAD, neg_lam.value, skip_fixed=True)
        elif act == ACCEPT:
            dm.accept_trial()
        elif act == DRIFT_EVAL:
            sc = dm.eval(dm.options(L.MOD_VOLUME, want_grad=False)).scalars
        sc = np.array(sc, dtype=np.float64)
    d3, i9 = np.zeros(3), np.zeros(9, dtype=np.int32)
    lib.emul_min_result(state, L.dptr(d3), L.iptr(i9))
    cg_iter, have, iters, early, success, has_gn, n_hist = (int(x) for x in i9[:7])
    mini.step_size, mini._cg_iter, mini._cg_have_history = float(d3[0]), cg_iter, bool(have)
    mini.history.extend((int(h[0]), float(h[1]), float(h[2]), bool(h[3])) for h in hist[:min(n_hist, cap)])
    out = {"energy": float(d3[1]), "iterations": iters, "terminated_early": bool(early), "step_success": bool(success)}
    if has_gn:
        out["grad_norm"] = float(d3[2])
    return out


def golden_case(case):
    z = np.load(H.GOLDEN + "/trajectory.npz")
    return {k[len(case) + 1:]: z[k] for k in z.files if k.startswith(case + "_")}


def setup_case(dm, g, **kw):
    """The trajectory case's mesh on dm and its DeviceMinimizer (as tests/test_device_minimizer.py builds it)."""
    pos, tri = g["pos"], g["tri"]
    nv, nf = pos.shape[0], tri.shape[0]
    body = np.zeros(nf, np.uint8)
    body[g["body_rows_0"]] = 1
    fixed = g["fixed"].astype(np.uint8) if g["fixed"].any() else None
    is_b = g["is_boundary"].astype(np.uint8) if g["is_boundary"].any() else None
    dm.set_topology(nv, tri, body_mask=body, fixed_mask=fixed, is_boundary=is_b)
    dm.set_surface_tension(g["gamma"])
    dm.set_bending_params(float(g["kappa"]), float(g["c0"]))
    dm.set_positions(pos)
    names = [str(n) for n in g["modules"]]
    mods = (L.MOD_SURFACE if "surface" in names else 0) | (L.MOD_BENDING if "bending" in names else 0)
    cg = "cg" if str(kw.pop("stepper", "")) == "cg" else "gd"
    if bool(g["enforce"]):
        args = dict(volume_mode="lagrange", v_target=float(g["body_target_0"]), enforce_volume=True,
                    projection_during_minimization=bool(g["proj_flag"]), volume_tolerance=float(g["vol_tol"]))
    else:
        args = dict(volume_mode="penalty", k_vol=float(g["kvol"]), v_target=float(g["body_target_0"]))
    args.update(kw)
    return DeviceMinimizer(dm, mods, stepper=cg, **args)


def assert_same(a, b, ra, rb):
    """Two minimisers (a, b) after the same calls, with the dicts they returned (ra, rb): bitwise equal."""
    assert ra == rb or (np.isnan(ra["energy"]) and np.isnan(rb["energy"])
                        and {k: v for k, v in ra.items() if k != "energy"} == {k: v for k, v in rb.items() if k != "energy"})
    assert a.step_size.hex() == b.step_size.hex()
    assert (a._cg_iter, a._cg_have_history) == (b._cg_iter, b._cg_have_history)
    assert [(i, e.hex(), s.hex(), ok) for i, e, s, ok in a.history] == [(i, e.hex(), s.hex(), ok) for i, e, s, ok in b.history]
    assert np.array_equal(a.dm.download(L.ARR_POSITIONS), b.dm.download(L.ARR_POSITIONS))


def run_pair(emul, g, n_calls, n_steps, make_dm=Recording, **kw):
    host_dm, dev_dm = make_dm(), make_dm()
    host, dev = setup_case(host_dm, g, **kw), setup_case(dev_dm, g, **kw)
    for _ in range(n_calls):
        rh = host.minimize_host(n_steps)
        rd = drive(emul, dev, n_steps)
        assert_same(host, dev, rh, rd)
    assert host_dm.log == dev_dm.log
    return host_dm.log, rh


# -- CPU tier -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES)
def test_controller_replays_the_trajectory_cases(emul, case):
    g = golden_case(case)
    steps = int(g["steps"])
    log, _ = run_pair(emul, g, 1, steps, stepper="cg" if case.endswith("cg") else "gd")
    assert sum(a == ACCEPT for a, _ in log) > 0
    if not case.endswith("cg"):  # one step per call: step size and state carry across calls
        run_pair(emul, g, steps, 1)


def test_controller_stops_when_g_dot_d_is_not_negative(emul):
    g = golden_case("bcubep")
    log, res = run_pair(emul, g, 1, 3, make_dm=lambda: Recording(stats=lambda o: (o[0], o[1], abs(o[2]) + 1.0, o[3])))
    assert not any(a == MAKE_TRIAL for a, _ in log) and not res["step_success"]


def test_controller_ends_the_call_after_max_zero_steps(emul):
    g = golden_case("bcubep")
    log, res = run_pair(emul, g, 1, 20, make_dm=lambda: Recording(trial_energy=lambda n: 1.0e6),
                        step_size_floor=1.0, max_zero_steps=3)
    assert res["terminated_early"] and not res["step_success"] and res["iterations"] == 3
    assert not any(a == ACCEPT for a, _ in log)


def test_controller_alpha_floor_ends_the_search(emul):
    g = golden_case("bcubep")
    log, _ = run_pair(emul, g, 1, 2, make_dm=lambda: Recording(trial_energy=lambda n: 1.0e6),
                      step_size=2e-8, beta=0.1)
    assert sum(a == MAKE_TRIAL for a, _ in log) == 2  # one trial per search: 2e-9 < 1e-8 ends it


def test_controller_normal_guard_rejections(emul):
    g = golden_case("bcubep")
    log, _ = run_pair(emul, g, 1, 3, make_dm=lambda: Recording(guard=lambda n, ok: n >= 3),
                      step_size=10.0, alpha_max_factor=1e3)
    assert sum(a == GUARD for a, _ in log) > 3


def test_controller_nan_trial_energy_is_rejected(emul):
    g = golden_case("cube")
    log, _ = run_pair(emul, g, 1, 3, make_dm=lambda: Recording(trial_energy=lambda n: float("nan") if n == 0 else 0.0))
    assert sum(a == EVAL_TRIAL for a, _ in log) > sum(a == ACCEPT for a, _ in log)


def test_controller_tolerance_stop_at_step_zero(emul):
    g = golden_case("cube")
    log, res = run_pair(emul, g, 1, 5, tol=1.0e30)
    assert res["terminated_early"] and res["iterations"] == 1 and "grad_norm" in res
    assert [a for a, _ in log if a in (EVAL_GRAD, DIRECTION, STATS)] == [EVAL_GRAD, DIRECTION, STATS]


def test_controller_drift_triggered_projection(emul):
    g = golden_case("bcubep")
    assert bool(g["enforce"])
    log, _ = run_pair(emul, g, 1, 3, projection_during_minimization=False, volume_tolerance=0.0, stepper="cg")
    assert any(a == DRIFT_EVAL for a, _ in log) and any(a == ENF_AXPY_POS for a, _ in log)


def test_controller_cg_reset_after_a_failed_step(emul):
    g = golden_case("bcubepcg")
    fail_second = lambda n: 1.0e6 if 1 <= n < 1 + 10 else 0.0  # noqa: E731 -- every trial of the 2nd search
    log, _ = run_pair(emul, g, 1, 4, make_dm=lambda: Recording(trial_energy=fail_second), stepper="cg")
    restarts = [arg for a, arg in log if a == DIRECTION]
    assert restarts[0] and not restarts[1] and restarts[2]  # the failed search resets the history


@pytest.mark.parametrize("enforce", [False, True])
def test_controller_zero_steps_still_projects(emul, enforce):
    g = golden_case("cube")
    log, res = run_pair(emul, g, 1, 0, enforce_volume=enforce)
    assert res["iterations"] == 0 and not res["terminated_early"]
    assert (log[0][0] == ENF_EVAL_POS) == enforce and log[-1][0] == EVAL_ENERGY


# -- GPU tier -------------------------------------------------------------------------------------------------------
def _gpu_dm():
    from membrane_solver_b200.context import DeviceMesh

    if L.device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu tier must run on the B200 box")
    return DeviceMesh(0)


class HostLog:
    """Records the host loop's trial step sizes and normal-flip answers on a real context."""

    def __init__(self, dm):
        self.alphas, self.guards = [], []
        make_trial, guard = dm.make_trial, dm.normal_change_ok

        def rec_trial(alpha):
            self.alphas.append(float(alpha))
            make_trial(alpha)

        def rec_guard(limit=0.5):
            ok = guard(limit)
            self.guards.append(ok)
            return ok
        dm.make_trial, dm.normal_change_ok = rec_trial, rec_guard


def twin_step(dev, host, n):
    """One call of n steps: the device loop on dev, the host loop on host, compared bitwise."""
    log = HostLog(host.dm)
    rd = dev.minimize(n)
    st = dev.dm.minimize_stats()
    rh = host.minimize_host(n)
    assert_same(dev, host, rd, rh)
    for w in (L.ARR_GRAD, L.ARR_DIRECTION, L.ARR_TRIAL):
        assert np.array_equal(dev.dm.download(w), host.dm.download(w)), w
    assert st["trials"] == len(log.alphas)
    assert (st["guards"], st["guard_rejects"]) == (len(log.guards), log.guards.count(False))
    return st, log


def twin_minimize(make_twin, calls):
    """make_twin() -> DeviceMinimizer on a fresh context; `calls` step counts: device loop on one twin, host loop on
    the other, compared bitwise after every call.  Every call waits for the device once (set_topology left the
    triangle rows on the device)."""
    dev, host = make_twin(), make_twin()
    dev.device_loop = True
    logs = []
    for n in calls:
        st, log = twin_step(dev, host, n)
        assert st["host_syncs"] == 1
        logs.append(log)
    return dev, host, logs


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_device_loop_matches_host_loop_on_trajectory_cases(case):
    g = golden_case(case)
    steps = int(g["steps"])
    cg = "cg" if case.endswith("cg") else "gd"
    twin_minimize(lambda: setup_case(_gpu_dm(), g, stepper=cg), [steps, 0, 1])
    if cg == "gd":
        twin_minimize(lambda: setup_case(_gpu_dm(), g), [1] * steps)


@pytest.mark.gpu
@pytest.mark.parametrize("op", ["refine", "equiangulate", "set_topology"])
def test_device_loop_after_the_context_dropped_the_cg_history(op):
    """CG steps build a history; a topology change through the DeviceMesh API drops the context's committed pair while
    the minimiser still believes it has one.  The host loop restarts (ms_ctx_cg_direction finds no pair); so must the
    device loop."""
    g = golden_case("bcubepcg")
    dev, host, _ = twin_minimize(lambda: setup_case(_gpu_dm(), g, stepper="cg"), [3])
    assert dev._cg_have_history and host._cg_have_history
    for m in (dev, host):
        if op == "refine":
            m.dm.refine(1)
        elif op == "equiangulate":
            m.dm.set_positions(m.dm.download(L.ARR_POSITIONS) * np.array([1.0, 1.3, 0.8]))  # make flips likely
            m.dm.equiangulate()
        else:
            pos, tri = m.dm.download(L.ARR_POSITIONS), m.dm.triangles()
            body = np.zeros(len(tri), np.uint8)
            body[g["body_rows_0"]] = 1
            m.dm.set_topology(len(pos), tri, body_mask=body,
                              fixed_mask=g["fixed"].astype(np.uint8) if g["fixed"].any() else None)
            m.dm.set_positions(pos)
    assert dev._cg_have_history
    for n in (3, 2):
        st, _ = twin_step(dev, host, n)
        assert st["host_syncs"] == 1


@pytest.mark.gpu
@pytest.mark.parametrize("stepper", ["gd", "cg"])
def test_gogo_replay_device_loop_matches_host_loop(stepper):
    """``gogo`` of the bending cube (``r, u, g 50, r, u, g 100, V``) with device ``r``, ``u`` and ``V`` on twin
    contexts: ``g`` by the device loop on one, by the host loop on the other; bitwise equal after every instruction."""
    import json

    from membrane_solver_b200.context import DeviceMesh
    from membrane_solver_b200.geometry.refine import cube_mesh

    gold = np.load(os.path.join(H.GOLDEN, "replay.npz"))
    prm = json.loads(str(gold["bcube_params_json"]))
    target = float(gold["bcube_00_body_target_0"])
    pos0, tri0 = cube_mesh()

    def make(device_loop):
        dm = DeviceMesh(0)
        dm.set_topology(len(pos0), tri0, body_mask=np.ones(len(tri0), np.uint8), order_hint=pos0)
        dm.set_positions(pos0)
        dm.set_surface_tension(float(prm["surface_tension"]))
        dm.set_bending_params(float(prm["bending_modulus"]), float(prm["spontaneous_curvature"]))
        return DeviceMinimizer(dm, L.MOD_BENDING, volume_mode="lagrange", v_target=target, enforce_volume=True,
                               stepper=stepper, device_loop=device_loop)

    dev, host = make(True), make(False)
    for ins in ["r", "u", "g50", "r", "u", "g100", "V"]:
        out = []
        for m in (dev, host):
            if ins == "r":
                out.append(m.refine())
            elif ins == "u":
                out.append(m.equiangulate())
            elif ins[0] == "g":
                out.append(m.minimize(n_steps=int(ins[1:])))
            else:
                out.append(m.vertex_average(1))
        if ins[0] == "g":
            assert_same(dev, host, *out)
            assert dev.dm.minimize_stats()["host_syncs"] == 1
        else:
            assert np.array_equal(out[0], out[1]) if ins == "r" else out[0] == out[1], ins
        assert np.array_equal(dev.dm.triangles(), host.dm.triangles()), ins
        assert np.array_equal(dev.dm.download(L.ARR_POSITIONS), host.dm.download(L.ARR_POSITIONS)), ins
        assert dev.energy().hex() == host.energy().hex(), ins


MILLION = [
    dict(volume_mode="lagrange", stepper="gd"),
    dict(volume_mode="lagrange", stepper="cg"),
    dict(volume_mode="penalty", k_vol=50.0, stepper="gd"),
    dict(volume_mode="penalty", k_vol=50.0, stepper="cg"),
    dict(volume_mode="lagrange", enforce_volume=True, projection_during_minimization=True),
    dict(volume_mode="lagrange", enforce_volume=True, projection_during_minimization=False, volume_tolerance=1e-12,
         stepper="cg"),
    dict(volume_mode="lagrange", edge_fraction=0.05, step_size=1.0, expect="clamp"),
    dict(volume_mode="lagrange", step_size=100.0, alpha_max_factor=1e3, expect="guard"),
    dict(volume_mode=None, tilt=True),
]


@pytest.fixture(scope="module")
def sphere_1m():
    from membrane_solver_b200.synthetic import frequency_for_facets, icosphere

    pos, tri = icosphere(frequency_for_facets(1_000_000))
    return pos, tri


@pytest.mark.gpu
@pytest.mark.parametrize("kw", MILLION, ids=[str(i) for i in range(len(MILLION))])
def test_device_loop_matches_host_loop_at_one_million_facets(sphere_1m, kw):
    from membrane_solver_b200.synthetic import tangent_tilts

    pos, tri = sphere_1m
    kw = dict(kw)
    tilt = kw.pop("tilt", False)
    expect = kw.pop("expect", None)
    v0 = 4.0 / 3.0 * np.pi * 0.97

    def make():
        dm = _gpu_dm()
        dm.set_topology(pos.shape[0], tri, body_mask=np.ones(tri.shape[0], np.uint8), order_hint=pos)
        dm.set_surface_tension(1.0)
        dm.set_bending_params(0.1, 0.0)
        dm.set_positions(pos)
        mods = L.MOD_SURFACE | L.MOD_BENDING
        if tilt:  # a frozen tilt field: the tilt energy takes part, the tilts do not move
            dm.set_tilt_rigidity(0.5)
            dm.set_tilts(tangent_tilts(pos, tri))
            mods |= L.MOD_TILT
        return DeviceMinimizer(dm, mods, v_target=v0, step_size=kw.pop("step_size", 1e-3), **kw)

    kw0 = dict(kw)
    step0 = kw0.get("step_size", 1e-3)
    _, _, logs = twin_minimize(lambda: (kw.update(kw0), make())[1], [3, 1])
    if expect == "clamp":  # the first trial takes edge_fraction * min edge / max |d|, below the step size
        assert logs[0].alphas[0] < step0
    if expect == "guard":  # large steps: the guard runs and rejects trials
        assert len(logs[0].guards) > 0 and logs[0].guards.count(False) > 0


@pytest.mark.gpu
def test_minimize_refusals_leave_the_context_unchanged():
    g = golden_case("bcubep")
    mini = setup_case(_gpu_dm(), g)
    dm = mini.dm
    before = dm.download(L.ARR_POSITIONS)
    step = mini.step_size
    bad = [(mini.minimize_options(), -1)]
    o = mini.minimize_options()
    o.max_iter = 1 << 21
    bad.append((o, 2))
    o = mini.minimize_options()
    o.modules |= L.MOD_BENDING_TILT
    bad.append((o, 2))
    o = mini.minimize_options()
    o.restart_interval = 0
    bad.append((o, 2))
    for opts, n in bad:
        with pytest.raises(L.B200Error):
            dm.minimize(opts, n, step_size=step)
        assert np.array_equal(dm.download(L.ARR_POSITIONS), before)
    # a partition context
    pos, tri = g["pos"], g["tri"]
    part = _gpu_dm()
    part.set_topology(pos.shape[0], tri, n_owned=pos.shape[0] - 2)
    part.set_positions(pos)
    with pytest.raises(L.B200Error, match="partition"):
        part.minimize(mini.minimize_options(), 1, step_size=step)
    assert np.array_equal(part.download(L.ARR_POSITIONS), pos)
    # the refused calls left the context fit to minimise as before
    assert mini.minimize(1)["iterations"] == 1
