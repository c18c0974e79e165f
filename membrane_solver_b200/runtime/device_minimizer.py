"""Device-resident gradient descent with Armijo backtracking.

SURVEY.md section 8(f) rank 1.  In the reference the energy/gradient evaluation is ~13 % of a
minimiser step; the rest is per-vertex Python around it (``positions_view`` rebuilds, line-search
vertex writes, ...).  This driver keeps positions, gradient, search direction and trial positions
on the GPU and moves only scalars across PCIe, mirroring -- for the case without enforceable
constraints and without tilts --

* ``Minimizer.minimize`` (``runtime/minimizer.py:1189-1535``): evaluate energy + projected gradient,
  stop on ``|g| < tol``, step, adapt the step size, count zero-steps;
* ``GradientDescent.step`` (``runtime/steppers/gradient_descent.py:35-84``): direction ``-g``, or
  ``ConjugateGradient.step`` (``runtime/steppers/conjugate_gradient.py:63-119``): per-vertex
  Polak-Ribiere direction with periodic restart;
* the trial-energy fast path of ``backtracking_line_search_array``
  (``runtime/steppers/line_search.py:267-430``): Armijo rule ``E(x + a d) <= E0 + c a <g,d>``,
  backtracking factor ``beta``, growth ``gamma``, the normal-flip guard of
  ``runtime/topology.py:13-48`` for steps larger than 0.3 x the shortest edge.

With ``device_loop=True`` on a ``DeviceMesh`` the loop itself runs under device control (``ms_ctx_minimize``,
``csrc/ms_minimize.cuh``): one CUDA graph and one host synchronisation per ``minimize`` call, with the decisions of
the host loop (``minimize_host``) bit for bit.  It is opt-in because it measures slower than the host loop on one
B200 (DESIGN.md section 1, row f1).  The host loop is the default; it also serves ``PartitionedDevice``
(cross-rank reductions) and is the reference of the tests.

It is an optional consumer of the hot path, not part of it: the reference's own minimiser keeps
working on the plugin modules (INTEGRATION.md section 2).
"""

from __future__ import annotations

from dataclasses import dataclass, field

from .. import _lib as L


@dataclass
class DeviceMinimizer:
    dm: object                     # membrane_solver_b200.context.DeviceMesh with topology, parameters, positions
    modules: int                   # MS_MOD_* bits of the energy terms
    flags: int = 0
    volume_mode: str | None = None  # None | "lagrange" (KKT projection of the gradient) | "penalty"
    projection_during_minimization: bool = True   # global parameter volume_projection_during_minimization
    volume_tolerance: float = 1e-3                # global parameter volume_tolerance
    enforce_volume: bool = False   # hard volume constraint: Newton projection of the positions inside the line
                                   # search and around the loop (modules/constraints/volume.py:69-149)
    k_vol: float = 0.0
    v_target: float = 0.0
    step_size: float = 1e-3
    tol: float = 1e-6
    max_zero_steps: int = 10
    step_size_floor: float = 1e-8
    max_iter: int = 10
    beta: float = 0.7
    c: float = 1e-4
    gamma: float = 1.5
    alpha_max_factor: float = 10.0
    edge_fraction: float = 0.0     # global parameter shape_step_edge_fraction
    stepper: str = "gd"            # "gd" | "cg" (per-vertex Polak-Ribiere, conjugate_gradient.py:63-119)
    restart_interval: int = 10
    device_loop: bool = False      # run minimize() under device control (DeviceMesh.minimize), opt-in: measured slower
    _cg_iter: int = 0
    _cg_have_history: bool = False
    history: list = field(default_factory=list)

    # -- energy of the loaded module set from the scalar vector ---------------------------------
    def _total(self, res) -> float:
        e = 0.0
        if self.modules & L.MOD_SURFACE:
            e += res.e_surface
        if self.modules & L.MOD_BENDING:
            e += res.e_bending
        if self.modules & L.MOD_TILT:
            e += res.e_tilt
        if self.volume_mode == "penalty":
            d = res.volume - self.v_target
            e += 0.5 * self.k_vol * d * d
        return float(e)

    def _mods(self) -> int:
        return self.modules | (L.MOD_VOLUME if self.volume_mode else 0)

    def _opts(self, *, want_grad: bool, use_trial: bool = False):
        mode = {"lagrange": 0, "penalty": 1}.get(self.volume_mode, -1)
        return self.dm.options(self._mods(), flags=self.flags, want_grad=want_grad, constraint_mode=mode,
                               k_vol=self.k_vol, v_target=self.v_target, apply_fixed=True, use_trial=use_trial)

    def energy(self, *, trial: bool = False) -> float:
        """Energy-only evaluation (pass A alone) at the positions or at the trial positions."""
        return self._total(self.dm.eval(self._opts(want_grad=False, use_trial=trial)))

    def energy_and_gradient(self) -> float:
        """Energy; the projected, fixed-masked gradient stays in MS_ARR_GRAD."""
        return self._total(self.dm.eval(self._opts(want_grad=True)))

    # -- hard volume constraint (constraints/volume.py:116-149) -----------------------------------------
    def _enforce(self, *, trial: bool, max_iter: int = 3, tol: float = 1e-12) -> None:
        dm = self.dm
        target = L.ARR_TRIAL if trial else L.ARR_POSITIONS
        for _ in range(max_iter):
            res = dm.eval(dm.options(L.MOD_VOLUME, want_grad=True, use_trial=trial))
            delta = res.volume - self.v_target
            if abs(delta) < tol:
                break
            lam = delta / (float(res.scalars[L.SC_GC_GC]) + 1e-12)
            dm.axpy(target, L.ARR_VOLGRAD, -lam, skip_fixed=True)

    # -- the V[n] command (commands/mesh_ops.py:45-53) --------------------------------------------------
    def vertex_average(self, n: int = 1) -> None:
        """``n`` rounds of vertex averaging on the device (``DeviceMesh.vertex_average``; fixed rows stay), then,
        with ``enforce_volume``, the hard volume projection of the ``mesh_operation`` context (12 iterations).  The
        positions jump, so the conjugate-gradient history is discarded: the next ``cg`` step restarts from the
        steepest-descent direction, as after a failed step."""
        self.dm.vertex_average(int(n))
        if self.enforce_volume:
            self._enforce(trial=False, max_iter=12)
        self._cg_have_history = False
        self._cg_iter = 0

    # -- the u command (commands/mesh_ops.py) ----------------------------------------------------------
    def equiangulate(self, max_iterations: int = 100) -> int:
        """Equiangulation on the device (``DeviceMesh.equiangulate``), then, with ``enforce_volume``, the hard volume
        projection of the ``mesh_operation`` context (12 iterations).  The conjugate-gradient history is discarded,
        as after ``vertex_average``.  Returns the number of flips."""
        flips = self.dm.equiangulate(int(max_iterations))
        if self.enforce_volume:
            self._enforce(trial=False, max_iter=12)
        self._cg_have_history = False
        self._cg_iter = 0
        return flips

    # -- the r command (commands/mesh_ops.py) ----------------------------------------------------------
    def refine(self, n: int = 1):
        """``n`` levels of midpoint refinement on the device (``DeviceMesh.refine``).  The reference projects no
        volume after ``r`` (the midpoints of a closed surface lie inside it), so neither does this; step size and
        ``v_target`` stay, the conjugate-gradient history is discarded.  Returns the composed ``parent``."""
        parent = self.dm.refine(int(n))
        self._cg_have_history = False
        self._cg_iter = 0
        return parent

    # -- one line search (line_search.py:267-430) --------------------------------------------------
    def _line_search(self, step_size: float):
        dm = self.dm
        energy0 = self.energy()
        min_edge, max_dir_norm, g_dot_d, _ = dm.line_search_stats()
        safe_step_limit = 0.3 * min_edge if min_edge > 0 else float("inf")
        if g_dot_d >= 0.0:
            return False, step_size, energy0
        alpha = step_size
        if self.edge_fraction > 0.0 and min_edge > 0.0 and max_dir_norm > 0.0:
            alpha = min(alpha, self.edge_fraction * min_edge / max_dir_norm)
        alpha_max = self.alpha_max_factor * step_size
        for _ in range(self.max_iter):
            dm.make_trial(alpha)
            if not (alpha * max_dir_norm < safe_step_limit) and not dm.normal_change_ok(0.5):
                alpha *= self.beta
                if alpha < 1e-8:
                    break
                continue
            if self.enforce_volume and self.projection_during_minimization:
                # line_search.py:449-451: constraint_enforcer(mesh) before the trial energy; the volume module is
                # skipped there when the projection is left to the drift check (constraint_manager.py:877-885)
                self._enforce(trial=True)
            trial_energy = self.energy(trial=True)
            if trial_energy <= energy0 + self.c * alpha * g_dot_d:
                dm.accept_trial()
                return True, min(alpha * self.gamma, alpha_max), trial_energy
            alpha *= self.beta
            if alpha < 1e-8:
                break
        reduced = max(alpha * self.beta, 0.0)
        return False, max(reduced, step_size * self.beta), energy0

    # -- the loop (minimizer.py:1189-1535) ------------------------------------------------------------
    def minimize_options(self):
        """The options of the device-controlled loop (``ms_minimize_opts``)."""
        return L.MinimizeOpts(
            modules=self.modules, flags=self.flags, volume_mode={"lagrange": 0, "penalty": 1}.get(self.volume_mode, -1),
            enforce_volume=int(bool(self.enforce_volume)), projection_during=int(bool(self.projection_during_minimization)),
            stepper={"gd": 0, "cg": 1}[self.stepper], max_zero_steps=self.max_zero_steps, max_iter=self.max_iter,
            restart_interval=self.restart_interval, k_vol=self.k_vol, v_target=self.v_target, tol=self.tol,
            step_size_floor=self.step_size_floor, beta=self.beta, c=self.c, gamma=self.gamma,
            alpha_max_factor=self.alpha_max_factor, edge_fraction=self.edge_fraction,
            volume_tolerance=self.volume_tolerance)

    def minimize(self, n_steps: int = 1) -> dict:
        """``n_steps`` minimiser steps: the host loop (``minimize_host``) or, with ``device_loop``, the whole loop under
        device control (``DeviceMesh.minimize``: one host synchronisation per call).  Both take the same decisions bit
        for bit."""
        if self.device_loop:
            if not hasattr(self.dm, "minimize"):
                raise L.B200Error("device_loop needs a single-context DeviceMesh (ms_ctx_minimize)")
            res, rows = self.dm.minimize(self.minimize_options(), int(n_steps), step_size=self.step_size,
                                         cg_iter=self._cg_iter, cg_have_history=self._cg_have_history)
            self.step_size = float(res.step_size)
            self._cg_iter, self._cg_have_history = int(res.cg_iter), bool(res.cg_have_history)
            self.history.extend(rows)
            out = {"energy": float(res.energy), "iterations": int(res.iterations),
                   "terminated_early": bool(res.terminated_early), "step_success": bool(res.step_success)}
            if res.has_grad_norm:
                out["grad_norm"] = float(res.grad_norm)
            return out
        return self.minimize_host(n_steps)

    def minimize_host(self, n_steps: int = 1) -> dict:
        """The host loop: every decision on the host, one scalar read per evaluation and statistic."""
        zero_steps = 0
        success = True
        energy = float("nan")
        if self.enforce_volume and n_steps > 0:  # minimizer.py:1223-1226 (context mesh_operation: 12 iterations)
            self._enforce(trial=False, max_iter=12)
        for i in range(n_steps):
            energy = self.energy_and_gradient()
            if self.stepper == "cg":
                restart = (not self._cg_have_history) or (self._cg_iter % self.restart_interval == 0)
                self.dm.cg_direction(restart)
                # remember gradient and direction NOW: the volume-only evaluations of the constraint
                # enforcement inside the line search overwrite MS_ARR_GRAD (conjugate_gradient.py:104-119
                # stores the gradient the step was computed from); a failed step discards the history below
                self.dm.cg_commit()
            else:
                self.dm.direction_from_gradient(-1.0)
            _, _, _, g_dot_g = self.dm.line_search_stats()
            grad_norm = g_dot_g ** 0.5
            if grad_norm < self.tol:
                return {"energy": energy, "iterations": i + 1, "terminated_early": True, "step_success": True,
                        "grad_norm": grad_norm}
            step_in = self.step_size
            success, self.step_size, accepted = self._line_search(step_in)
            self.history.append((i, float(accepted), float(step_in), bool(success)))
            if self.stepper == "cg":
                if success:
                    self._cg_have_history = True
                    self._cg_iter += 1
                else:  # minimizer.py:1461-1463: a failed step resets the stepper
                    self._cg_have_history = False
                    self._cg_iter = 0
            if not success:
                if self.step_size <= self.step_size_floor:
                    zero_steps += 1
                    if zero_steps >= self.max_zero_steps:
                        return {"energy": self.energy(), "iterations": i + 1, "terminated_early": True,
                                "step_success": False}
                else:
                    zero_steps = 0
            else:
                zero_steps = 0
                if self.enforce_volume and self.volume_mode == "lagrange" and not self.projection_during_minimization:
                    # minimizer.py:1476-1510: geometric projection only when the volume drifted beyond tolerance
                    vol = self.dm.eval(self.dm.options(L.MOD_VOLUME, want_grad=False)).volume
                    if abs(vol - self.v_target) / max(abs(self.v_target), 1.0) > self.volume_tolerance:
                        self._enforce(trial=False, max_iter=12)
                        self._cg_have_history = False
                        self._cg_iter = 0
        if self.enforce_volume:  # minimizer.py:1518-1521: final projection (context finalize)
            self._enforce(trial=False, max_iter=12)
        return {"energy": self.energy(), "iterations": n_steps, "terminated_early": False,
                "step_success": success}
