import numpy as np, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from membrane_solver_b200 import _lib as L
from membrane_solver_b200.context import DeviceMesh
from membrane_solver_b200.synthetic import icosphere
pos, tri = icosphere(708)
nv, nf = pos.shape[0], tri.shape[0]
rng = np.random.default_rng(0)
def run(label, **cfg):
    dm = DeviceMesh(0)
    is_b = None
    if cfg.get('boundary'):
        is_b = np.zeros(nv, np.uint8); is_b[rng.integers(0, nv, 2000)] = 1
    dm.set_topology(nv, tri, body_mask=np.ones(nf, np.uint8), is_boundary=is_b)
    dm.set_surface_tension(1.0 + 0.1*rng.random(nf) if cfg.get('gamma') else 1.0)
    dm.set_bending_params(1.0 + 0.1*rng.random(nv) if cfg.get('kappa') else 1.0, 0.0)
    dm.set_positions(pos)
    mods = cfg.get('mods', L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME)
    if mods & (L.MOD_TILT | L.MOD_BENDING_TILT):
        t = 0.1*rng.normal(size=(nv,3)); dm.set_tilts(t); dm.set_tilt_rigidity(1.0)
    opts = dm.options(mods, constraint_mode=0 if mods & L.MOD_VOLUME else -1, flags=cfg.get('flags', 0), want_grad=cfg.get('want_grad', True))
    for _ in range(3): dm.eval_async(opts)
    dm.sync(); dm.timer_start()
    for _ in range(10): dm.eval_async(opts)
    ms = dm.timer_stop()/10
    print(f"{label:40s} {ms:.3f} ms  {nf/ms/1e6:.2f} Gf/s"); dm.close()
run("FAST S+B+V")
run("generic: per-vertex kappa", kappa=True)
run("generic: per-facet gamma", gamma=True)
run("generic: boundary flags", boundary=True)
run("generic: willmore", flags=L.FLAG_WILLMORE)
run("surface+volume only", mods=L.MOD_SURFACE | L.MOD_VOLUME)
run("surface only", mods=L.MOD_SURFACE)
run("energy only S+B+V (line search)", want_grad=False)
run("S+B+V+tilt", mods=L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME | L.MOD_TILT)
run("bending_tilt + tilt", mods=L.MOD_BENDING_TILT | L.MOD_TILT)

# device-resident minimiser steps (only scalars cross PCIe): surface + bending + volume penalty
from membrane_solver_b200.runtime.device_minimizer import DeviceMinimizer
for stepper in ("gd", "cg"):
    dm = DeviceMesh(0)
    dm.set_topology(nv, tri, body_mask=np.ones(nf, np.uint8))
    dm.set_surface_tension(1.0); dm.set_bending_params(1.0, 0.0); dm.set_positions(pos)
    mini = DeviceMinimizer(dm, L.MOD_SURFACE | L.MOD_BENDING, volume_mode="penalty", k_vol=1000.0, v_target=4.18,
                           step_size=1e-7, stepper=stepper)
    mini.minimize(n_steps=3)
    t0 = time.perf_counter(); r = mini.minimize(n_steps=20); dm.sync(); dt = time.perf_counter() - t0
    evals = sum(1 for h in mini.history)
    print(f"device-resident {stepper} step (10M facets)      {dt/20*1e3:.3f} ms/step  energy {r['energy']:.6f}  accepted {sum(h[3] for h in mini.history)}/{len(mini.history)}")
    dm.close()
