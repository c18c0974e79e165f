"""Patch packing on the device against the host packer ``ms::pack_patches``, on the 10 M-facet icosphere and its
40 M-facet refinement.

Prints one JSON line per case:
  - ``set_topology``: the whole call at 10 M facets (host clock; it uploads the rows and packs them on the device);
  - ``equiangulate``: a jittered 10 M-facet icosphere, ``ms_ctx_equiangulate_stats`` (its slot ``pack_ms`` is the
    device packing of the flipped rows, CUDA events);
  - ``refine``: 10 M -> 40 M facets, ``ms_ctx_refine_stats`` (``pack_ms`` = device packing of the 40 M rows);
each with the host reference ``pack_patches`` on the same internal-order rows in the same run (compiled as the test
emulator is, all host threads) and whether the two layouts are byte-identical.  A refinement of a small mesh first
loads the kernels.  The GPU name and power limit are read in the same run.

    python tools/pack_bench.py --out profiles/pack_bench_10m.jsonl
"""

from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import ms_pack_helpers as P  # noqa: E402
from membrane_solver_b200.context import DeviceMesh  # noqa: E402
from membrane_solver_b200.synthetic import frequency_for_facets, icosphere  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "tools"))
from refine_bench import gpu_info  # noqa: E402


def internal_rows(dm):
    perm = dm.permutation()
    inv = np.empty_like(perm)
    inv[perm] = np.arange(len(perm), dtype=perm.dtype)
    return inv[dm.triangles()].astype(np.int32)


def host_reference(lib, dm):
    """Host pack_patches of the context's rows with its parameters: (ms, byte-identical to the context's packing)."""
    info = dm.pack_info()
    rows = internal_rows(dm)
    t0 = time.perf_counter()
    rc, st, want = P.pack_emulated(lib, False, rows, dm.nv, threads=info["threads"])
    host_ms = 1e3 * (time.perf_counter() - t0)
    got = dm.packing()
    same = rc == 0 and all(info[k] == st[k] for k in P.PACK_STATS) and \
        all(got[k].tobytes() == want[k].tobytes() for k in want)
    return host_ms, bool(same), info


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--facets", type=int, default=10_000_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    name, power = gpu_info()
    out = open(args.out, "w") if args.out else None

    def emit(line):
        line.update(gpu=name, power_limit=power, host_threads=os.cpu_count())
        print(json.dumps(line), flush=True)
        if out:
            out.write(json.dumps(line) + "\n")
            out.flush()

    with tempfile.TemporaryDirectory() as tmp:
        lib = P.build_pack_emulator(tmp)
        p, t = icosphere(10)   # warm-up: loads every kernel of the packing and the refinement
        w = DeviceMesh(0)
        w.set_topology(len(p), t, order_hint=p)
        w.set_positions(p)
        w.refine(1)
        w.close()

        pos, tri = icosphere(frequency_for_facets(args.facets), perturb=False)
        dm = DeviceMesh(0)
        t0 = time.perf_counter()
        dm.set_topology(len(pos), tri, order_hint=pos)
        call_ms = 1e3 * (time.perf_counter() - t0)
        host_ms, same, info = host_reference(lib, dm)
        emit(dict(case="set_topology", nf=dm.nf, call_ms=round(call_ms, 1), host_pack_ms=round(host_ms, 1),
                          identical=same, n_patches=info["n_patches"], threads=info["threads"]))

        rng = np.random.default_rng(0)
        h = float(np.mean(np.linalg.norm(pos[tri[:, 1]] - pos[tri[:, 0]], axis=1)))
        q = pos + 0.3 * h * rng.normal(size=pos.shape)
        q /= np.linalg.norm(q, axis=1, keepdims=True)
        de = DeviceMesh(0)
        de.set_topology(len(q), tri, order_hint=q)
        de.set_positions(q)
        t0 = time.perf_counter()
        flips = de.equiangulate(9)
        call_ms = 1e3 * (time.perf_counter() - t0)
        st = de.equiangulate_stats()
        host_ms, same, _ = host_reference(lib, de)
        emit(dict(case="equiangulate", nf=de.nf, flips=flips, call_ms=round(call_ms, 1),
                          stats={k: (round(v, 2) if isinstance(v, float) else v) for k, v in st.items() if k != "rounds"},
                          host_pack_ms=round(host_ms, 1), identical=same))
        de.close()

        dm.set_positions(pos)
        t0 = time.perf_counter()
        dm.refine(1)
        call_ms = 1e3 * (time.perf_counter() - t0)
        st = dm.refine_stats()
        host_ms, same, _ = host_reference(lib, dm)
        emit(dict(case="refine", nf=dm.nf, call_ms=round(call_ms, 1),
                          stats={k: round(v, 2) for k, v in st.items()}, host_pack_ms=round(host_ms, 1),
                          identical=same))
        dm.close()
    if out:
        out.close()


if __name__ == "__main__":
    main()
