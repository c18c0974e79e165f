"""Device equiangulation (``ms_ctx_equiangulate``, the ``u`` command) on a large jittered icosphere, optionally
against the host twin ``geometry.equiangulate.equiangulate_triangles``.

Prints one JSON line per mesh: sweeps, flips and selection rounds per sweep; the device time of the sweeps (CUDA
events) in total and per sweep; the row download, host packing and upload of the new packing (host clock); the
whole call (host clock around the call, which ends synchronised); with ``--twin`` the twin's time on the same mesh
and whether its rows equal the device's.  The GPU name and power limit are read in the same run.  The mesh is the
icosphere of the requested size with tangential noise of 0.3 x the mean edge length (``default_rng(0)``), projected
back onto the sphere.

    python tools/equiangulate_bench.py                       # 10 M facets, device only
    python tools/equiangulate_bench.py --twin --out result.jsonl
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from membrane_solver_b200 import _lib as L  # noqa: E402
from membrane_solver_b200.context import DeviceMesh  # noqa: E402
from membrane_solver_b200.geometry.equiangulate import equiangulate_triangles  # noqa: E402
from membrane_solver_b200.synthetic import frequency_for_facets, icosphere  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30, check=True).stdout.strip()
        name, power = (x.strip() for x in out.split(",", 1))
        return name, power
    except (OSError, subprocess.SubprocessError, ValueError) as exc:
        return None, f"not read: {exc}"


def jittered_sphere(target_facets: int):
    pos, tri = icosphere(frequency_for_facets(target_facets), perturb=False)
    h = np.mean(np.linalg.norm(pos[tri[:, 1]] - pos[tri[:, 0]], axis=1))
    q = pos + 0.3 * h * np.random.default_rng(0).normal(size=pos.shape)
    return q / np.linalg.norm(q, axis=1)[:, None], tri


def run(target_facets: int, max_iterations: int, twin: bool) -> dict:
    pos, tri = jittered_sphere(target_facets)
    nv, nf = pos.shape[0], tri.shape[0]
    dm = DeviceMesh(0)
    dm.set_topology(nv, tri, order_hint=pos)
    dm.set_positions(pos)
    dm.sync()
    t0 = time.perf_counter()
    flips = dm.equiangulate(max_iterations)
    call_ms = 1e3 * (time.perf_counter() - t0)
    st = dm.equiangulate_stats()
    rows = dm.triangles()
    dm.close()
    out = {"facets": nf, "vertices": nv, "max_iterations": max_iterations, "sweeps": dm.last_equiangulate_sweeps,
           "sweeps_run": st["sweeps_run"], "flips": flips, "selection_rounds_per_sweep": st["rounds"],
           "device_sweeps_ms": st["sweep_ms"], "device_ms_per_sweep": st["sweep_ms"] / max(st["sweeps_run"], 1),
           "d2h_rows_ms": st["d2h_ms"], "host_pack_ms": st["pack_ms"], "upload_ms": st["upload_ms"],
           "call_ms": call_ms}
    if twin:
        t0 = time.perf_counter()
        want, twin_flips = equiangulate_triangles(pos, tri, max_iterations=max_iterations)
        out["twin_s"] = time.perf_counter() - t0
        out["twin_flips"] = twin_flips
        out["rows_equal_twin"] = bool(np.array_equal(rows, want))
    return out


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--facets", type=int, action="append", help="icosphere size (repeatable), default 10 M")
    ap.add_argument("--max-iterations", type=int, default=100)
    ap.add_argument("--twin", action="store_true", help="also run the host twin (minutes at 10 M facets)")
    ap.add_argument("--out", help="also append the JSON lines to this file")
    args = ap.parse_args()
    if L.device_count() < 1:
        raise SystemExit("equiangulate_bench needs a CUDA device; there is no CPU fallback")
    name, power = gpu_info()
    for facets in args.facets or [10_000_000]:
        res = {"gpu": name, "power_limit": power, **run(facets, args.max_iterations, args.twin)}
        line = json.dumps(res)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as fh:
                fh.write(line + "\n")


if __name__ == "__main__":
    main()
