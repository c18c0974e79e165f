"""Helpers of the patch-packing tests (unique module name: an unrelated ``tests`` package is installed in this image):
the test-only host emulator of the device packer, tests/emul/pack_emul.cpp, through ctypes."""

import ctypes
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# --------------------------------------------------------------------------
# Host emulator of the device patch packer (tests/emul/pack_emul.cpp) -- TEST ONLY.
# --------------------------------------------------------------------------
PACK_STATS = ("n_patches", "n_halo", "n_slots", "max_owned", "max_local", "max_rounds", "max_slots", "n_round_slots",
              "n_listed", "n_valid", "n_lane_conflicts", "n_hw_groups", "n_hw_excess")


def build_pack_emulator(out_dir):
    """tests/emul/pack_emul.cpp with the host packer ms_pack.cpp, compiled into out_dir (the tree may be read-only)."""
    out = os.path.join(str(out_dir), "libms_pack_emul.so")
    csrc = os.path.join(ROOT, "membrane_solver_b200", "csrc")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-pthread", "-fPIC", "-shared", "-o", out,
                           os.path.join(ROOT, "tests", "emul", "pack_emul.cpp"), os.path.join(csrc, "ms_pack.cpp")])
    lib = ctypes.CDLL(out)
    lib.emul_pack.restype = ctypes.c_int
    lib.emul_corner_csr.restype = ctypes.c_int64
    return lib


def pack_emulated(lib, device, tri, nv, *, body=None, threads=96, max_owned=512, max_local=896, max_slots=1536,
                  fill_pct=87, repair_sweeps=1, n_owned=-1):
    """(rc, stats dict, arrays dict or None) of the emulated device packer (device=True) or ms::pack_patches."""
    tri = np.ascontiguousarray(tri, dtype=np.int32).reshape(-1, 3)
    body = None if body is None else np.ascontiguousarray(body, dtype=np.uint8)
    st = np.zeros(len(PACK_STATS), dtype=np.int64)
    ip = ctypes.POINTER(ctypes.c_int32)
    rc = lib.emul_pack(int(device), int(nv), len(tri), tri.ctypes.data_as(ip),
                       None if body is None else body.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), int(threads),
                       int(max_owned), int(max_local), int(max_slots), int(fill_pct), int(repair_sweeps), int(n_owned),
                       st.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)))
    stats = dict(zip(PACK_STATS, (int(x) for x in st)))
    if rc:
        return rc, stats, None
    arr = {"headers": np.zeros((stats["n_patches"], 32), dtype=np.uint8),
           "halo_ids": np.zeros(stats["n_halo"], dtype=np.int32),
           "recs": np.zeros((stats["n_slots"], 4), dtype=np.uint16),
           "slot_facet": np.zeros(stats["n_slots"], dtype=np.int32)}
    lib.emul_pack_fetch(int(device), arr["headers"].ctypes.data_as(ctypes.c_void_p), arr["halo_ids"].ctypes.data_as(ip),
                        arr["recs"].ctypes.data_as(ctypes.c_void_p), arr["slot_facet"].ctypes.data_as(ip))
    return rc, stats, arr


def corner_csr_emulated(lib, device, tri, nv):
    """(ptr, idx) of the device corner sort (device=True) or ms::build_corner_csr."""
    tri = np.ascontiguousarray(tri, dtype=np.int32).reshape(-1, 3)
    ptr = np.zeros(nv + 1, dtype=np.int32)
    idx = np.zeros(3 * len(tri) + 1, dtype=np.int32)
    ip = ctypes.POINTER(ctypes.c_int32)
    n = lib.emul_corner_csr(int(device), int(nv), len(tri), tri.ctypes.data_as(ip), ptr.ctypes.data_as(ip),
                            idx.ctypes.data_as(ip))
    return ptr, idx[:n]


def header_fields(headers):
    """Structured view of (n, 32) uint8 patch headers."""
    dt = np.dtype([("v_lo", "<i4"), ("n_owned", "<i4"), ("halo_off", "<i4"), ("n_halo", "<i4"), ("slot_off", "<i8"),
                   ("reserved", "<i4"), ("n_rounds", "<i4")])
    return np.ascontiguousarray(headers).view(dt).reshape(-1)
