#!/usr/bin/env python
"""Throughput benchmark of the fused energy+gradient evaluation (BASELINE.json metric).

One *step* = one evaluation of surface + Helfrich bending + body volume (energies,
shape gradient, dV/dx, KKT projection of the volume constraint) over the whole mesh:
pass A, pass B, partial-sum reduction, dot products, projection.

    python bench.py --gpus 1 --steps 50 --warmup 5
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference            # CPU arm (oracle port, all host cores)
    python bench.py --gpus 1 --steps 50 --warmup 5 --dump-outputs DIR   # + what the last timed step computed
                                                # (1 GPU only; DESIGN.md "Measurement")

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every key.
"""

from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree, which may be read-only

METRIC = "Gfacet-evals/s (energy+grad)"
UNIT = "Gfacet-evals/s"
# Algorithmic bytes per facet-eval (SURVEY.md section 8d, closed manifold nv = nf/2,
# uniform gamma/kappa/c0): pass A reads tri 12 + pos 12 and writes 40 B/vertex = 20;
# pass B reads tri 12 + pos 12 + seeds 20 and writes grad 12 + dV/dx 12.
B_PASS_A = 44.0
B_PASS_B = 68.0
B_STEP = B_PASS_A + B_PASS_B  # 112 B, the headline figure
B_STRICT = 72.0
# --dump-outputs keeps at most this many vertex rows of each per-vertex array: 2 x 24 MiB of float64 in all
DUMP_ROWS = 1 << 20


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """Samples SM clocks and throttle reasons through NVML while `active` is set."""

    def __init__(self, index: int):
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.active = threading.Event()
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        except Exception as exc:  # NVML missing: report that, do not invent clocks
            self._nv = None
            self.error = str(exc)

    _NAMES = {
        0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
        0x4: "sw_power_cap", 0x80: "hw_power_brake", 0x2: "applications_clocks_setting",
        0x100: "display_clock_setting", 0x10: "sync_boost",
    }

    def _run(self):
        nv = self._nv
        while not self._stop.is_set():
            if self.active.is_set():
                try:
                    self.samples.append(int(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                    try:
                        mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                    except Exception:
                        mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
                    for bit, name in self._NAMES.items():
                        if mask & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
            time.sleep(0.004)

    def close(self):
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=1.0)

    def summary(self):
        if not self._nv:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "error": getattr(self, "error", "nvml unavailable")}
        med = int(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def _cpu_eval_worker(args):
    """One oracle evaluation of the sample mesh (C restatement of the Fortran kernels
    injected through the loader seam = the 'Fortran-enabled' reference path)."""
    n_freq, reps = args
    from membrane_solver_b200.synthetic import icosphere
    from oracle import ckernels
    from oracle import ref_modules as ref

    ref.use_c_kernels(ckernels)
    pos, tri = icosphere(n_freq)
    nv, nf = pos.shape[0], tri.shape[0]
    gamma = np.ones(nf)
    bnd = np.zeros(nv, bool)
    ref.fused_surface_bending_volume(pos, tri, gamma, 1.0, 0.0, bnd)  # warm caches / imports
    t0 = time.perf_counter()
    for _ in range(reps):
        out = ref.fused_surface_bending_volume(pos, tri, gamma, 1.0, 0.0, bnd)
        ref.kkt_project_single(out["grad"], out["vol_grad"])
    return nf * reps, time.perf_counter() - t0


def cpu_baseline(n_freq: int, reps: int, workers: int):
    """Gfacet-evals/s of the CPU oracle on `workers` processes, each evaluating its own
    copy of a frequency-`n_freq` icosphere `reps` times."""
    from oracle import ckernels

    ckernels.build()
    if workers <= 1:
        facets, secs = _cpu_eval_worker((n_freq, reps))
        return facets / secs / 1e9, 20 * n_freq * n_freq
    import multiprocessing as mp

    ctx = mp.get_context("spawn")
    t0 = time.perf_counter()
    with ctx.Pool(workers) as pool:
        res = pool.map(_cpu_eval_worker, [(n_freq, reps)] * workers)
    del t0
    # every worker ran concurrently: aggregate = total facets / slowest worker
    facets = sum(r[0] for r in res)
    secs = max(r[1] for r in res)
    return facets / secs / 1e9, 20 * n_freq * n_freq


def _time_oracle_eval(pos, tri, reps_warm: int, reps: int):
    """Seconds per whole evaluation (energies, gradient, dV/dx, KKT projection) of the CPU arm, one process."""
    from oracle import ref_modules as ref

    nv, nf = pos.shape[0], tri.shape[0]
    gamma = np.ones(nf)
    bnd = np.zeros(nv, bool)
    times = []
    for i in range(reps_warm + reps):
        t0 = time.perf_counter()
        out = ref.fused_surface_bending_volume(pos, tri, gamma, 1.0, 0.0, bnd)
        ref.kkt_project_single(out["grad"], out["vol_grad"])
        if i >= reps_warm:
            times.append(time.perf_counter() - t0)
    return times


def run_reference(args):
    """CPU arm: the reference's algorithm for this path on the host (oracle port with the C restatement of the
    Fortran kernels = the 'Fortran-enabled' path; the reference itself cannot hold these meshes in its
    dict-of-objects Mesh and gfortran is absent).  The reference's array path is single threaded, so `value` is ONE
    process; one step = one evaluation of a bounded sample of the workload (a 1 003 520-facet perturbed icosphere,
    same modules).  Extra keys: one evaluation of the full 10 M-facet mesh, and the all-core replica aggregate."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = "1"  # the reference pins these too (tools/tilt_perf_guardrails.py:22-28)
    from membrane_solver_b200.synthetic import frequency_for_facets, icosphere
    from oracle import ckernels
    from oracle import ref_modules as ref

    ckernels.build()
    ref.use_c_kernels(ckernels)
    t_wall = time.perf_counter()
    steps, warm = max(1, args.steps), max(0, args.warmup)
    n_sample = 224
    pos, tri = icosphere(n_sample)
    nf = tri.shape[0]
    times = _time_oracle_eval(pos, tri, warm, steps)
    sec_step = float(np.mean(times))
    value = nf / sec_step / 1e9
    sample = (f"1 process, {steps} timed + {warm} warm-up evaluations of a {nf}-facet perturbed icosphere (a bounded "
              "sample of the workload: same modules, energy + gradient + dV/dx + KKT projection); NumPy oracle with the C "
              "restatement of fortran_kernels/*.f90 injected (gfortran absent)")
    extra = {}
    if not args.no_full_mesh:
        try:  # the workload itself, once: the per-facet rate does not depend on the size
            n_full = frequency_for_facets(args.facets)
            pf, tf = icosphere(n_full)
            t_full = _time_oracle_eval(pf, tf, 0, 1)[0]
            extra["full_mesh"] = {"facets": int(tf.shape[0]), "seconds_per_evaluation": t_full,
                                  "value": tf.shape[0] / t_full / 1e9, "unit": UNIT, "processes": 1}
            del pf, tf
        except MemoryError as exc:
            extra["full_mesh"] = {"unavailable": str(exc)}
    cores = max(1, min(len(os.sched_getaffinity(0)), 64))
    if cores > 1:
        agg, nf_rep = cpu_baseline(100, 2, cores)
        extra["all_core_replicas"] = {"value": agg, "unit": UNIT, "processes": cores, "facets_per_process": nf_rep,
                                      "note": "independent replicas on every host core: scales with the box, not the path"}
    cfg = workload_config(args, args.gpus)
    cfg["reference_sample"] = {"facets": int(nf), "frequency": n_sample, "processes": 1}
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": 1e3 * sec_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t_wall, **extra,
    }
    print(json.dumps(line))
    return 0


def workload_config(args, n_gpus):
    from membrane_solver_b200.synthetic import frequency_for_facets

    n = frequency_for_facets(args.facets * n_gpus)
    return {
        "workload": "synthetic perturbed icosphere, surface + Helfrich bending + body-volume "
                    "(lagrange KKT) energy+gradient sweep (BASELINE.json configs[4])",
        "frequency": n, "facets": 20 * n * n, "vertices": 10 * n * n + 2,
        "facets_per_gpu": 20 * n * n // n_gpus,
        "modules": ["surface", "bending(helfrich,analytic)", "volume(lagrange)"],
        "l2": "working set (>=700 MB per 10M facets) exceeds the 126 MB L2; no explicit flush",
    }


def dump_outputs(dm, out_dir):
    """Writes what the last evaluation hands its caller: the 16 scalars (energies, area, volume, dot products, KKT
    multiplier and coefficient; include/ms_b200.h MS_SC_*), the projected gradient and dV/dx, all float64.  A mesh
    with more than DUMP_ROWS vertices keeps the same seeded sample of rows (ascending) in both arrays."""
    from membrane_solver_b200 import _lib as L

    os.makedirs(out_dir, exist_ok=True)
    scalars = dm.read_scalars().scalars
    grad, volgrad = dm.download(L.ARR_GRAD), dm.download(L.ARR_VOLGRAD)
    rows = slice(None)
    if grad.shape[0] > DUMP_ROWS:
        rows = np.sort(np.random.default_rng(0).choice(grad.shape[0], DUMP_ROWS, replace=False))
    np.save(os.path.join(out_dir, "scalars.npy"), scalars)
    np.save(os.path.join(out_dir, "grad.npy"), grad[rows])
    np.save(os.path.join(out_dir, "volgrad.npy"), volgrad[rows])


def run_b200(args):
    from membrane_solver_b200 import _lib as L
    from membrane_solver_b200.context import DeviceMesh
    from membrane_solver_b200.synthetic import frequency_for_facets, icosphere

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    if world > 1:
        from membrane_solver_b200 import partition

        return partition.bench_multi_gpu(args, rank, world, local, sys.modules[__name__])
    if L.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: the B200 path has no CPU fallback")

    t_setup = time.perf_counter()
    n = frequency_for_facets(args.facets)
    pos, tri = icosphere(n)
    nv, nf = pos.shape[0], tri.shape[0]
    t_gen = time.perf_counter() - t_setup
    dm = DeviceMesh(local, threads=args.threads, max_owned=args.max_owned, max_local=args.max_local,
                    fill_pct=args.fill,
                    repair_sweeps=args.repair)
    t0 = time.perf_counter()
    dm.set_topology(nv, tri, body_mask=np.ones(nf, np.uint8))
    t_pack = time.perf_counter() - t0
    dm.set_surface_tension(1.0)
    dm.set_bending_params(1.0, 0.0)
    dm.set_positions(pos)
    info = dm.pack_info()
    mods = L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME
    opts = dm.options(mods, constraint_mode=0, apply_fixed=False)
    launches_per_step = 2  # pass A, pass B (its last CTA reduces the sums and writes the KKT coefficient)

    sampler = ClockSampler(local)
    for _ in range(max(3, args.warmup)):
        dm.eval_async(opts)
    dm.sync()

    # ---- timed region: K steps, device-resident, CUDA events on the context stream ----
    sampler.active.set()
    dm.timer_start()
    for _ in range(args.steps):
        dm.eval_async(opts)
    ms_total = dm.timer_stop()
    sampler.active.clear()
    if args.dump_outputs:  # before the legs below overwrite the results
        dump_outputs(dm, args.dump_outputs)
    ms_step = ms_total / args.steps
    value = nf / (ms_step * 1e-3) / 1e9

    # ---- per-kernel durations (same stream, events between the launches) ----
    k_steps = max(5, min(args.steps, 50))
    sampler.active.set()
    for i in range(k_steps):
        dm.event_record(4 * i)
        dm.eval_stage(opts, 0)
        dm.event_record(4 * i + 1)
        dm.eval_stage(opts, 1)
        dm.event_record(4 * i + 2)
        dm.eval_pass_b(opts)        # the same pass without the fused finalisation: the difference is its cost
        dm.event_record(4 * i + 3)
    dm.sync()
    sampler.active.clear()
    t_a = float(np.mean([dm.event_elapsed(4 * i, 4 * i + 1) for i in range(k_steps)]))
    t_b = float(np.mean([dm.event_elapsed(4 * i + 1, 4 * i + 2) for i in range(k_steps)]))
    t_b_plain = float(np.mean([dm.event_elapsed(4 * i + 2, 4 * i + 3) for i in range(k_steps)]))
    t_f = max(0.0, t_b - t_b_plain)

    # ---- end to end through the C ABI with HOST buffers (pinned): H2D positions,
    #      evaluation, D2H projected gradient + scalars, every step ----
    grad = np.empty_like(pos)
    lib = L.lib()
    L.check(lib.ms_host_register(pos.ctypes.data, pos.nbytes))
    L.check(lib.ms_host_register(grad.ctypes.data, grad.nbytes))
    for _ in range(2):
        dm.eval_host(opts, pos, grad=grad)
    e2e_steps = max(3, min(args.steps, 20))
    sampler.active.set()
    dm.timer_start()
    for _ in range(e2e_steps):
        res = dm.eval_host(opts, pos, grad=grad)
    ms_e2e = dm.timer_stop() / e2e_steps
    sampler.active.clear()
    L.check(lib.ms_host_unregister(pos.ctypes.data))
    L.check(lib.ms_host_unregister(grad.ctypes.data))
    e2e_value = nf / (ms_e2e * 1e-3) / 1e9
    sampler.close()

    peak, peak_kind = _peaks()
    dominant = "pass_b" if t_b >= t_a else "pass_a"
    b_dom, t_dom = (B_PASS_B, t_b) if dominant == "pass_b" else (B_PASS_A, t_a)
    achieved = b_dom * nf / (t_dom * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            with open(tpath) as fh:
                tj = json.load(fh)
            if tj.get("facets") == nf:
                traffic = tj.get(dominant)
        except Exception:
            pass

    cpu_reps = 3
    cpu_val, cpu_nf = cpu_baseline(224, cpu_reps, 1) if not args.no_cpu else (None, 0)

    # ---- strong-scaling leg: the north_star's 100 M-facet mesh on this one GPU (the N > 1 lines carry the same
    #      mesh cut over N GPUs; speed-up = this ms_per_step / theirs) ----
    strong = None
    if args.strong_facets > 0:
        dm.close()
        t0 = time.perf_counter()
        n_s = frequency_for_facets(args.strong_facets)
        pos_s, tri_s = icosphere(n_s)
        t_gen_s = time.perf_counter() - t0
        dms = DeviceMesh(local, threads=args.threads, max_owned=args.max_owned, max_local=args.max_local,
                         fill_pct=args.fill, repair_sweeps=args.repair)
        t0 = time.perf_counter()
        dms.set_topology(pos_s.shape[0], tri_s, body_mask=np.ones(tri_s.shape[0], np.uint8))
        t_pack_s = time.perf_counter() - t0
        dms.set_surface_tension(1.0)
        dms.set_bending_params(1.0, 0.0)
        dms.set_positions(pos_s)
        for _ in range(3):
            dms.eval_async(opts)
        dms.sync()
        s_steps = max(3, min(args.steps, 10))
        dms.timer_start()
        for _ in range(s_steps):
            dms.eval_async(opts)
        ms_s = dms.timer_stop() / s_steps
        rs = dms.read_scalars()
        strong = {"scaling": "strong", "facets": int(tri_s.shape[0]), "n_gpus": 1, "ms_per_step": ms_s,
                  "value": tri_s.shape[0] / (ms_s * 1e-3) / 1e9, "unit": UNIT, "steps": s_steps,
                  "energies": {"surface": rs.e_surface, "bending": rs.e_bending, "volume": rs.volume},
                  "setup_seconds": t_gen_s + t_pack_s}
        dms.close()
        del pos_s, tri_s

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, 1),
        "roofline": {
            "bound": "hbm", "kernel": dominant, "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "traffic": traffic, "peak_source": f"MEASURED_PEAKS.json ({peak_kind})",
            "bytes_per_facet": b_dom,
            "step_gbs_112": B_STEP * nf / (ms_step * 1e-3) / 1e9,
            "step_frac_112": B_STEP * nf / (ms_step * 1e-3) / 1e9 / peak,
            "step_frac_72": B_STRICT * nf / (ms_step * 1e-3) / 1e9 / peak,
        },
        "kernels_ms": {"pass_a": t_a, "pass_b": t_b, "reduce+kkt": t_f},
        "fp64": {"peak_tflops_measured": 33.9, "note": "tools/fp64_peak.cu on this pool's B200; the kernels are "
                 "instruction-issue / latency bound at 12 consumer warps per SM, see DESIGN.md section 3.4"},
        "cpu_baseline": None if cpu_val is None else {
            "value": cpu_val, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"1 process, {cpu_reps} evaluations of a {cpu_nf}-facet perturbed icosphere (a bounded sample of the "
                      "workload, same modules); NumPy oracle with the C restatement of fortran_kernels/*.f90 (gfortran "
                      "absent).  The reference's array path is single threaded: see --impl reference for the all-core "
                      "replica figure"},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(pos.nbytes),
                "d2h_bytes_per_step": int(grad.nbytes + 8 * L.SC_COUNT), "ms_per_step": ms_e2e,
                "api": "ms_ctx_eval_host (pinned host positions in, projected gradient + scalars out)"},
        "gpu_launches": launches_per_step * args.steps,
        "clocks": sampler.summary(),
        "pack": {**info, "seconds": t_pack, "mesh_gen_seconds": t_gen},
        "energies": {"surface": res.e_surface, "bending": res.e_bending, "volume": res.volume},
    }
    if strong is not None:
        line["strong"] = strong
    print(json.dumps(line))
    if strong is None:
        dm.close()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--facets", type=int, default=10_000_000, help="facets per GPU")
    ap.add_argument("--threads", type=int, default=None)
    ap.add_argument("--max-owned", type=int, default=None)
    ap.add_argument("--max-local", type=int, default=None)
    ap.add_argument("--fill", type=int, default=None, help="packer: target percent of record slots holding a facet")
    ap.add_argument("--repair", type=int, default=None, help="packer: lane-placement repair passes")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--strong-facets", type=int, default=100_000_000,
                    help="total facets of the strong-scaling leg (BASELINE.json north_star: 100 M); 0 = skip")
    ap.add_argument("--no-full-mesh", action="store_true", help="reference arm: skip the one full-size evaluation")
    ap.add_argument("--no-parity", action="store_true", help="N>1: skip the comparison with one GPU on the same mesh")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="1 GPU: write the scalars, gradient and dV/dx of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.gpus != 1):
        ap.error("--dump-outputs needs --impl b200 --gpus 1")
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
