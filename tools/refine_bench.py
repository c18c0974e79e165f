"""Device refinement (``ms_ctx_refine``, the ``r`` command) of the synthetic icosphere, optionally against the host
twin ``geometry.refine.refine_triangles``.

Prints one JSON line per mesh: the sizes before and after; the device time of the levels, the Morton order and the
gathers (CUDA events); the download of the rows and the order, the host packing, and the commit with the upload of
the new packing (host clock); the whole call (host clock around the call, which ends synchronised); with ``--twin``
the twin's time on the same mesh (its NumPy refinement alone, without the set-up of a new context) and whether its
rows and positions equal the device's, bitwise.  The GPU name and power limit are read in the same run.  The mesh is
``synthetic.icosphere`` of the requested size in its Morton order, uploaded with itself as order hint; a refinement
of a 2 k-facet icosphere first loads the kernels.

    python tools/refine_bench.py                       # 10 M facets -> 40 M, device only
    python tools/refine_bench.py --twin --out result.jsonl
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
from membrane_solver_b200.geometry.refine import refine_triangles  # noqa: E402
from membrane_solver_b200.synthetic import frequency_for_facets, icosphere  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30, check=True).stdout.strip()
        name, power = (x.strip() for x in out.split(",", 1))
        return name, power
    except (OSError, subprocess.SubprocessError, ValueError) as exc:
        return None, f"not read: {exc}"


def refined_on_device(pos, tri, levels):
    dm = DeviceMesh(0)
    dm.set_topology(len(pos), tri, order_hint=pos)
    dm.set_positions(pos)
    dm.sync()
    t0 = time.perf_counter()
    dm.refine(levels)
    call_ms = 1e3 * (time.perf_counter() - t0)
    return dm, call_ms


def run(target_facets: int, levels: int, twin: bool) -> dict:
    pos, tri = icosphere(frequency_for_facets(target_facets))
    nv, nf = pos.shape[0], tri.shape[0]
    dm, call_ms = refined_on_device(pos, tri, levels)
    st = dm.refine_stats()
    out = {"facets": nf, "vertices": nv, "levels": levels, "refined_facets": dm.nf, "refined_vertices": dm.nv,
           "device_ms": st["device_ms"], "d2h_ms": st["d2h_ms"], "host_pack_ms": st["pack_ms"],
           "commit_upload_ms": st["upload_ms"], "call_ms": call_ms}
    if twin:
        rows, got_pos = dm.triangles(), dm.download(L.ARR_POSITIONS)
        dm.close()
        t0 = time.perf_counter()
        p, t = pos, tri
        for _ in range(levels):
            p, t, _, _ = refine_triangles(p, t)
        out["twin_s"] = time.perf_counter() - t0
        out["rows_positions_equal_twin"] = bool(np.array_equal(rows, t)
                                                and np.array_equal(got_pos.view(np.uint64), p.view(np.uint64)))
    else:
        dm.close()
    return out


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--facets", type=int, action="append", help="icosphere size (repeatable), default 10 M")
    ap.add_argument("--levels", type=int, default=1)
    ap.add_argument("--twin", action="store_true", help="also run the host twin")
    ap.add_argument("--out", help="also append the JSON lines to this file")
    args = ap.parse_args()
    if L.device_count() < 1:
        raise SystemExit("refine_bench needs a CUDA device; there is no CPU fallback")
    name, power = gpu_info()
    warm, _ = refined_on_device(*icosphere(10), 1)
    warm.close()
    for facets in args.facets or [10_000_000]:
        res = {"gpu": name, "power_limit": power, **run(facets, args.levels, args.twin)}
        line = json.dumps(res)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as fh:
                fh.write(line + "\n")


if __name__ == "__main__":
    main()
