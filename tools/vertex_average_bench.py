"""Device vertex averaging (``ms_ctx_vertex_average``, the ``V`` command) against the host twin
``geometry.vertex_average.vertex_average_arrays`` on large icospheres.

For each mesh it prints one JSON line: the first call (it includes the host build and upload of the corner CSR), the
device time per round from CUDA events after warm-up (even round counts: no copy back), the time of a single-round call
(odd: includes the copy from the trial buffer back to the positions), the host twin's time, the largest difference of
the two results, and the compulsory bytes of one round over the kernel time against the HBM figure ``bench.py`` uses.
The GPU name and power limit are read in the same run.

    python tools/vertex_average_bench.py                     # 10 M facets
    python tools/vertex_average_bench.py --facets 10000000 --facets 100000000 --out result.jsonl
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
from membrane_solver_b200.geometry.vertex_average import vertex_average_arrays  # noqa: E402
from membrane_solver_b200.synthetic import frequency_for_facets, icosphere  # noqa: E402

L2_BYTES = 126 * 2**20
DESIGN_HBM_GBS = 6544.7  # DESIGN.md section 3.4: copy-measured on a B200


def hbm_peak():
    """The HBM figure of bench.py: MEASURED_PEAKS.json when present, else the copy-measured DESIGN.md figure."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "MEASURED_PEAKS.json"
    except (OSError, KeyError, ValueError):
        return DESIGN_HBM_GBS, "DESIGN.md section 3.4 (copy-measured, MEASURED_PEAKS.json absent)"


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30, check=True).stdout.strip()
        name, power = (x.strip() for x in out.split(",", 1))
        return name, power
    except (OSError, subprocess.SubprocessError, ValueError) as exc:
        return None, f"not read: {exc}"


def compulsory_bytes(nv: int, nf: int) -> int:
    """One round: positions read and written (24 B per vertex each), triangle rows (12 B per facet), corner CSR
    (4 B per corner, 3 per facet, plus 4 B per vertex pointer)."""
    return 48 * nv + 12 * nf + 4 * 3 * nf + 4 * (nv + 1)


def run(target_facets: int, rounds: int, host: bool) -> dict:
    pos, tri = icosphere(frequency_for_facets(target_facets))
    nv, nf = pos.shape[0], tri.shape[0]
    dm = DeviceMesh(0)
    dm.set_topology(nv, tri, order_hint=pos)
    dm.set_positions(pos)
    dm.sync()
    t0 = time.perf_counter()
    dm.vertex_average(1)
    dm.sync()
    first_ms = 1e3 * (time.perf_counter() - t0)
    dm.vertex_average(4)                      # warm-up
    dm.sync()
    dm.timer_start()
    dm.vertex_average(rounds)
    round_ms = dm.timer_stop() / rounds
    dm.timer_start()
    for _ in range(rounds):
        dm.vertex_average(1)
    call_ms = dm.timer_stop() / rounds
    dm.set_positions(pos)
    dm.vertex_average(1)
    dev = dm.download(L.ARR_POSITIONS)
    dm.close()
    out = {"facets": nf, "vertices": nv, "first_call_ms": first_ms, "device_ms_per_round": round_ms,
           "device_ms_per_single_round_call": call_ms, "rounds_timed": rounds}
    if host:
        t0 = time.perf_counter()
        want = vertex_average_arrays(pos, tri)
        out["host_twin_s"] = time.perf_counter() - t0
        out["max_abs_diff_vs_host_twin"] = float(np.max(np.abs(dev - want)))
    nbytes = compulsory_bytes(nv, nf)
    peak, source = hbm_peak()
    achieved = nbytes / (round_ms * 1e-3) / 1e9
    out.update(compulsory_bytes_per_round=nbytes, achieved_gbs=achieved, hbm_peak_gbs=peak, hbm_peak_source=source,
               share_of_hbm_peak=achieved / peak,
               l2_note=(f"working set {nbytes / 2**20:.0f} MiB > {L2_BYTES >> 20} MiB L2: rounds stream from HBM"
                        if nbytes > L2_BYTES else f"working set {nbytes / 2**20:.0f} MiB fits the L2"))
    return out


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--facets", type=int, action="append", help="icosphere size (repeatable), default 10 M")
    ap.add_argument("--rounds", type=int, default=20, help="rounds per timed window")
    ap.add_argument("--no-host", action="store_true", help="skip the host twin (time and difference)")
    ap.add_argument("--out", help="also append the JSON lines to this file")
    args = ap.parse_args()
    if L.device_count() < 1:
        raise SystemExit("vertex_average_bench needs a CUDA device; there is no CPU fallback")
    if args.rounds < 2 or args.rounds % 2:
        raise SystemExit("--rounds must be even and >= 2 (an even count ends in the positions without a copy)")
    name, power = gpu_info()
    for facets in args.facets or [10_000_000]:
        res = {"gpu": name, "power_limit": power, **run(facets, args.rounds, not args.no_host)}
        line = json.dumps(res)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as fh:
                fh.write(line + "\n")


if __name__ == "__main__":
    main()
