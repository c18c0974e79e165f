#!/usr/bin/env python
"""Minimiser steps with the loop under device control (``DeviceMinimizer(device_loop=True)`` -> ``ms_ctx_minimize``:
one CUDA graph, one host synchronisation per call) against the host loop (``minimize_host``: a scalar read per evaluation and
statistic), on twin contexts in the same run, alternating, with a bitwise comparison of positions, step sizes, history
and returned dicts after every call.

Cases: the 10 M-facet icosphere (surface + bending + volume: lagrange GD, CG, hard volume constraint), the bending cube
refined 8 times (1.57 M facets, hard volume constraint) and 3 times (1 536 facets: overheads only).

    python tools/minimize_bench.py [--out profiles/minimize_bench.jsonl] [--steps 10] [--rounds 3] [--quick]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from membrane_solver_b200 import _lib as L  # noqa: E402
from membrane_solver_b200.context import DeviceMesh  # noqa: E402
from membrane_solver_b200.geometry.refine import cube_mesh, refine_triangles  # noqa: E402
from membrane_solver_b200.runtime.device_minimizer import DeviceMinimizer  # noqa: E402
from membrane_solver_b200.synthetic import frequency_for_facets, icosphere  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def sphere_case(facets, **kw):
    pos, tri = icosphere(frequency_for_facets(facets))
    v0 = 4.0 / 3.0 * np.pi * 0.97

    def make():
        dm = DeviceMesh(0)
        dm.set_topology(pos.shape[0], tri, body_mask=np.ones(tri.shape[0], np.uint8), order_hint=pos)
        dm.set_surface_tension(1.0)
        dm.set_bending_params(0.1, 0.0)
        dm.set_positions(pos)
        return DeviceMinimizer(dm, L.MOD_SURFACE | L.MOD_BENDING, volume_mode="lagrange", v_target=v0, **kw)
    return make, tri.shape[0]


def cube_case(levels):
    pos, tri = cube_mesh()
    for _ in range(levels):
        pos, tri, _, _ = refine_triangles(pos, tri)

    def make():
        dm = DeviceMesh(0)
        dm.set_topology(pos.shape[0], tri, body_mask=np.ones(tri.shape[0], np.uint8), order_hint=pos)
        dm.set_surface_tension(0.0)
        dm.set_bending_params(1.0, 0.0)
        dm.set_positions(pos)
        return DeviceMinimizer(dm, L.MOD_BENDING, volume_mode="lagrange", v_target=1.0, enforce_volume=True,
                               projection_during_minimization=True)
    return make, tri.shape[0]


def same(a, b, ra, rb):
    return (ra == rb and a.step_size == b.step_size and (a._cg_iter, a._cg_have_history) == (b._cg_iter, b._cg_have_history)
            and a.history == b.history
            and np.array_equal(a.dm.download(L.ARR_POSITIONS), b.dm.download(L.ARR_POSITIONS)))


def run(name, make, nf, steps, rounds, gpu):
    dev, host = make(), make()
    dev.device_loop = True
    ok = same(dev, host, dev.minimize(1), host.minimize_host(1))  # warm-up: kernel loads, lazy arrays
    t_dev, t_host, dev_ms, build_ms = [], [], [], []
    for _ in range(rounds):
        t0 = time.perf_counter()
        rd = dev.minimize(steps)
        t_dev.append(time.perf_counter() - t0)
        st = dev.dm.minimize_stats()
        dev_ms.append(st["device_ms"])
        build_ms.append(st["build_ms"])
        t0 = time.perf_counter()
        rh = host.minimize_host(steps)
        host.dm.sync()
        t_host.append(time.perf_counter() - t0)
        ok = ok and same(dev, host, rd, rh)
    rec = {"case": name, "facets": int(nf), "steps_per_call": steps, "rounds": rounds, "gpu": gpu,
           "device_loop_ms_per_step": 1e3 * float(np.median(t_dev)) / steps,
           "host_loop_ms_per_step": 1e3 * float(np.median(t_host)) / steps,
           "device_graph_ms_per_step": float(np.median(dev_ms)) / steps,
           "graph_build_ms_per_call": float(np.median(build_ms)),
           "last_call": {k: st[k] for k in ("steps", "trials", "evaluations", "host_syncs", "actions", "guards")},
           "bitwise_equal": bool(ok)}
    for m in (dev, host):
        m.dm.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--quick", action="store_true", help="small meshes only")
    a = ap.parse_args()
    if L.device_count() < 1:
        raise SystemExit("no CUDA device: this benchmark measures the B200")
    gpu = gpu_info()
    cases = [("bending_cube_r3", *cube_case(3))]
    if not a.quick:
        cases += [("bending_cube_r8_hard_volume", *cube_case(8))]
        for label, kw in (("gd_lagrange", {}), ("cg_lagrange", {"stepper": "cg"}),
                          ("gd_hard_volume", {"enforce_volume": True})):
            cases.append((f"icosphere_10m_{label}", *sphere_case(10_000_000, **kw)))
    recs = []
    for name, make, nf in cases:
        small = nf < 100_000  # overheads only: more steps and rounds, so that the window is not scheduling noise
        rec = run(name, make, nf, 5 * a.steps if small else a.steps, max(10, a.rounds) if small else a.rounds, gpu)
        print(json.dumps(rec), flush=True)
        recs.append(rec)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for r in recs:
                f.write(json.dumps(r) + "\n")
    if not all(r["bitwise_equal"] for r in recs):
        raise SystemExit("the device loop and the host loop disagree")


if __name__ == "__main__":
    main()
