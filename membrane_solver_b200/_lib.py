"""ctypes binding of ``libms_b200.so`` (the C ABI declared in ``include/ms_b200.h``).

This is the host side of the drop-in boundary: it replaces the dispatch of
``fortran_kernels/loader.py`` for the energy+gradient path.  There is no CPU
fallback -- a missing library or a missing CUDA device raises.
"""

from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MS_B200_LIB") or os.path.join(_PKG, "libms_b200.so")  # override: A/B builds
CSRC = os.path.join(_PKG, "csrc")

MOD_SURFACE, MOD_VOLUME, MOD_BENDING, MOD_TILT, MOD_BENDING_TILT = 1, 2, 4, 8, 16
MOD_TILT_SMOOTHNESS = 32
FLAG_WILLMORE, FLAG_APPROX = 1, 2
PATCHES_ALL, PATCHES_INTERIOR, PATCHES_BOUNDARY = -1, -2, -3

SC_E_SURFACE, SC_AREA, SC_VOLUME, SC_E_BENDING, SC_E_TILT, SC_E_BENDING_TILT = 0, 1, 2, 3, 4, 5
SC_G_G, SC_G_GC, SC_GC_GC, SC_LAMBDA, SC_COEF, SC_COUNT = 8, 9, 10, 11, 12, 16

ARR_POSITIONS, ARR_GRAD, ARR_VOLGRAD, ARR_SEEDS, ARR_TILTS, ARR_TILT_GRAD = 0, 1, 2, 3, 4, 5
ARR_SCALARS, ARR_K_VECS, ARR_A_VOR, ARR_A_EFF, ARR_E_VERTEX, ARR_TRIAL, ARR_DIRECTION = 6, 7, 8, 9, 10, 11, 12
ARR_TILTS_IN, ARR_TILTS_OUT, ARR_TILT_GRAD_IN, ARR_TILT_GRAD_OUT = 13, 14, 15, 16
ARR_TILTS_FIELD, ARR_TILT_GRAD_FIELD = 17, 18
LEAFLET_IN, LEAFLET_OUT, LEAFLET_FIELD = 0, 1, 2
IPC_FLAGS, IPC_HANDLE_BYTES, FLAG_POSITIONS, FLAG_SEEDS = 100, 64, 0, 1
ACC_GRAD, ACC_TILT_GRAD = 1, 2
ARRAY_WIDTH = {ARR_POSITIONS: 3, ARR_GRAD: 3, ARR_VOLGRAD: 3, ARR_SEEDS: 5, ARR_TILTS: 3,
               ARR_TILT_GRAD: 3, ARR_SCALARS: 1, ARR_K_VECS: 3, ARR_A_VOR: 1, ARR_A_EFF: 1,
               ARR_E_VERTEX: 1, ARR_TRIAL: 3, ARR_DIRECTION: 3, ARR_TILTS_IN: 3, ARR_TILTS_OUT: 3,
               ARR_TILT_GRAD_IN: 3, ARR_TILT_GRAD_OUT: 3, ARR_TILTS_FIELD: 3, ARR_TILT_GRAD_FIELD: 3}


class B200Error(RuntimeError):
    """Raised for every non-zero return code of the C ABI (no silent fallback)."""


class EvalOpts(ctypes.Structure):
    _fields_ = [
        ("modules", ctypes.c_uint32),
        ("flags", ctypes.c_uint32),
        ("want_grad", ctypes.c_int32),
        ("constraint_mode", ctypes.c_int32),
        ("k_vol", ctypes.c_double),
        ("v_target", ctypes.c_double),
        ("apply_fixed", ctypes.c_int32),
        ("use_trial", ctypes.c_int32),
        ("patch_begin", ctypes.c_int32),
        ("patch_count", ctypes.c_int32),
        ("diagnostics", ctypes.c_int32),
        ("want_tilt_grad", ctypes.c_int32),
    ]


class LeafletDesc(ctypes.Structure):
    """struct ms_leaflet_desc (include/ms_b200.h)."""
    _fields_ = [
        ("facet_keep", ctypes.POINTER(ctypes.c_uint8)),
        ("interior", ctypes.POINTER(ctypes.c_uint8)),
        ("base_zero", ctypes.POINTER(ctypes.c_uint8)),
        ("kappa", ctypes.POINTER(ctypes.c_double)),
        ("c0", ctypes.POINTER(ctypes.c_double)),
        ("tilt_row_weight", ctypes.POINTER(ctypes.c_double)),
        ("facet_consistent", ctypes.POINTER(ctypes.c_uint8)),
        ("kappa_default", ctypes.c_double),
        ("c0_default", ctypes.c_double),
        ("k_tilt", ctypes.c_double),
        ("k_smooth", ctypes.c_double),
        ("div_sign", ctypes.c_double),
        ("consistent_default", ctypes.c_int32),
        ("reserved", ctypes.c_int32),
    ]


class PackInfo(ctypes.Structure):
    _fields_ = [
        ("nv", ctypes.c_int32), ("nf", ctypes.c_int32),
        ("n_patches", ctypes.c_int32), ("threads", ctypes.c_int32),
        ("max_owned", ctypes.c_int32), ("max_local", ctypes.c_int32),
        ("max_rounds", ctypes.c_int32), ("max_slots", ctypes.c_int32),
        ("n_slots", ctypes.c_int64), ("n_listed", ctypes.c_int64),
        ("n_valid", ctypes.c_int64), ("n_halo", ctypes.c_int64),
        ("n_round_slots", ctypes.c_int64), ("n_lane_conflicts", ctypes.c_int64),
        ("n_hw_groups", ctypes.c_int64), ("n_hw_excess", ctypes.c_int64),
    ]


_D = ctypes.POINTER(ctypes.c_double)
_I = ctypes.POINTER(ctypes.c_int32)
_B = ctypes.POINTER(ctypes.c_uint8)
_V = ctypes.c_void_p
_i32, _i64, _f64 = ctypes.c_int32, ctypes.c_int64, ctypes.c_double

# name -> (restype, argtypes); every symbol include/ms_b200.h declares
SIGNATURES = {
    "ms_last_error": (ctypes.c_char_p, []),
    "ms_version": (ctypes.c_int, []),
    "ms_device_count": (ctypes.c_int, [ctypes.POINTER(ctypes.c_int)]),
    "ms_ctx_create": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(_V)]),
    "ms_ctx_destroy": (ctypes.c_int, [_V]),
    "ms_ctx_set_pack_params": (ctypes.c_int, [_V, _i32, _i32, _i32]),
    "ms_ctx_set_pack_tuning": (ctypes.c_int, [_V, _i32, _i32]),
    "ms_ctx_set_max_ctas": (ctypes.c_int, [_V, _i32]),
    "ms_ctx_set_vertex_order_hint": (ctypes.c_int, [_V, _i32, _D]),
    "ms_ctx_get_permutation": (ctypes.c_int, [_V, _I]),
    "ms_ctx_set_topology": (ctypes.c_int, [_V, _i32, _i32, _I, _B, _B, _B]),
    "ms_ctx_set_topology_partition": (ctypes.c_int, [_V, _i32, _i32, _i32, _I, _B, _B, _B]),
    "ms_ctx_set_send_rows": (ctypes.c_int, [_V, _I, _i64]),
    "ms_ctx_pack_send": (ctypes.c_int, [_V, ctypes.c_int, _V]),
    "ms_ctx_set_fixed_mask": (ctypes.c_int, [_V, ctypes.POINTER(ctypes.c_uint8)]),
    "ms_ctx_pack_info": (ctypes.c_int, [_V, ctypes.POINTER(PackInfo)]),
    "ms_ctx_patch_ranges": (ctypes.c_int, [_V, _I]),
    "ms_ctx_halo_rows": (ctypes.c_int, [_V, _i32, _i32, _i32, _i32, _I, ctypes.POINTER(_i64)]),
    "ms_ctx_set_surface_tension": (ctypes.c_int, [_V, _D, _f64]),
    "ms_ctx_set_bending_params": (ctypes.c_int, [_V, _D, _D, _f64, _f64]),
    "ms_ctx_set_tilt_rigidity": (ctypes.c_int, [_V, _f64]),
    "ms_ctx_set_positions": (ctypes.c_int, [_V, _D]),
    "ms_ctx_set_tilts": (ctypes.c_int, [_V, _D]),
    "ms_ctx_upload": (ctypes.c_int, [_V, ctypes.c_int, _D, _i64, _i64]),
    "ms_ctx_get_array": (ctypes.c_int, [_V, ctypes.c_int, _D, _i64, _i64]),
    "ms_ctx_device_ptr": (_V, [_V, ctypes.c_int]),
    "ms_ctx_array_len": (_i64, [_V, ctypes.c_int]),
    "ms_ctx_set_stream": (ctypes.c_int, [_V, _V]),
    "ms_ctx_eval_async": (ctypes.c_int, [_V, ctypes.POINTER(EvalOpts)]),
    "ms_ctx_self_check": (ctypes.c_int, [_V, ctypes.POINTER(ctypes.c_int32)]),
    "ms_ctx_eval_stage": (ctypes.c_int, [_V, ctypes.POINTER(EvalOpts), _i32]),
    "ms_ctx_eval_pass_a": (ctypes.c_int, [_V, ctypes.POINTER(EvalOpts)]),
    "ms_ctx_eval_pass_b": (ctypes.c_int, [_V, ctypes.POINTER(EvalOpts)]),
    "ms_ctx_eval_finish": (ctypes.c_int, [_V, ctypes.POINTER(EvalOpts)]),
    "ms_ctx_eval_reduce": (ctypes.c_int, [_V, ctypes.POINTER(EvalOpts)]),
    "ms_ctx_eval_project": (ctypes.c_int, [_V, ctypes.POINTER(EvalOpts)]),
    "ms_ctx_read_scalars": (ctypes.c_int, [_V, _D]),
    "ms_ctx_eval": (ctypes.c_int, [_V, ctypes.POINTER(EvalOpts), _D]),
    "ms_ctx_eval_host": (ctypes.c_int, [_V, ctypes.POINTER(EvalOpts), _D, _D, _D, _D, _D]),
    "ms_ctx_set_leaflet": (ctypes.c_int, [_V, _i32, ctypes.POINTER(LeafletDesc)]),
    "ms_ctx_eval_leaflet": (ctypes.c_int, [_V, _i32, ctypes.c_uint32, _i32, _i32, ctypes.c_uint32, _i32, _D]),
    "ms_ctx_set_leaflet_fixed": (ctypes.c_int, [_V, _i32, _B]),
    "ms_ctx_update_vertex_normals": (ctypes.c_int, [_V]),
    "ms_ctx_leaflet_project_tilts": (ctypes.c_int, [_V, _i32]),
    "ms_ctx_leaflet_gradient_norm2": (ctypes.c_int, [_V, _i32, _D]),
    "ms_ctx_eval_leaflet_pair": (ctypes.c_int, [_V, ctypes.c_uint32, _i32, _i32, ctypes.c_uint32, _i32]),
    "ms_ctx_leaflet_results": (ctypes.c_int, [_V, _D]),
    "ms_ctx_leaflet_make_trial": (ctypes.c_int, [_V, _i32, _f64, _i32]),
    "ms_ctx_leaflet_build_preconditioner": (ctypes.c_int, [_V, _i32, _f64, _i32]),
    "ms_ctx_leaflet_rz": (ctypes.c_int, [_V, _i32, _i32, _D]),
    "ms_ctx_leaflet_cg_direction": (ctypes.c_int, [_V, _i32, _f64, _i32, _i32]),
    "ms_ctx_leaflet_swap_trial": (ctypes.c_int, [_V, _i32]),
    "ms_ctx_ipc_export": (ctypes.c_int, [_V, _i32, _B]),
    "ms_ctx_peer_close": (ctypes.c_int, [_V]),
    "ms_ctx_peer_open": (ctypes.c_int, [_V, _i32, _i32, _B]),
    "ms_ctx_peer_set_pointer": (ctypes.c_int, [_V, _i32, _i32, _V]),
    "ms_ctx_flag_words_ptr": (_V, [_V]),
    "ms_ctx_set_ghost_sources": (ctypes.c_int, [_V, _i32, _I, _I]),
    "ms_ctx_halo_prepare": (ctypes.c_int, [_V]),
    "ms_ctx_halo_signal": (ctypes.c_int, [_V, _i32]),
    "ms_ctx_halo_pull": (ctypes.c_int, [_V, _i32, _i32]),
    "ms_ctx_set_rank_slot": (ctypes.c_int, [_V, _i32, _i32]),
    "ms_ctx_allreduce_scalars": (ctypes.c_int, [_V, _i32]),
    "ms_ctx_halo_error": (ctypes.c_int, [_V, _I]),
    "ms_ctx_eval_partition": (ctypes.c_int, [_V, ctypes.POINTER(EvalOpts), _i32]),
    "ms_ctx_set_push_targets": (ctypes.c_int, [_V, _i32, _I, _I, _I]),
    "ms_ctx_halo_push": (ctypes.c_int, [_V, _i32, _i32]),
    "ms_ctx_make_trial": (ctypes.c_int, [_V, _f64]),
    "ms_ctx_accept_trial": (ctypes.c_int, [_V]),
    "ms_ctx_dots": (ctypes.c_int, [_V]),
    "ms_ctx_direction_from_gradient": (ctypes.c_int, [_V, _f64]),
    "ms_ctx_axpy": (ctypes.c_int, [_V, ctypes.c_int, ctypes.c_int, _f64, _i32]),
    "ms_ctx_vertex_average": (ctypes.c_int, [_V, _I, _i32]),
    "ms_ctx_equiangulate": (ctypes.c_int, [_V, _i32, ctypes.POINTER(_i64), ctypes.POINTER(_i32)]),
    "ms_ctx_equiangulate_stats": (ctypes.c_int, [_V, _D, _I, _i32, ctypes.POINTER(_i32)]),
    "ms_ctx_get_triangles": (ctypes.c_int, [_V, _I]),
    "ms_ctx_cg_direction": (ctypes.c_int, [_V, _i32]),
    "ms_ctx_cg_commit": (ctypes.c_int, [_V]),
    "ms_ctx_line_search_stats": (ctypes.c_int, [_V, _D]),
    "ms_ctx_normal_change_ok": (ctypes.c_int, [_V, _f64, _I]),
    "ms_ctx_timer_start": (ctypes.c_int, [_V]),
    "ms_ctx_timer_stop": (ctypes.c_int, [_V, ctypes.POINTER(ctypes.c_float)]),
    "ms_ctx_sync": (ctypes.c_int, [_V]),
    "ms_ctx_event_record": (ctypes.c_int, [_V, _i32]),
    "ms_ctx_event_elapsed": (ctypes.c_int, [_V, _i32, _i32, ctypes.POINTER(ctypes.c_float)]),
    "ms_ctx_flush_l2": (ctypes.c_int, [_V, _i64]),
    "ms_host_register": (ctypes.c_int, [_V, _i64]),
    "ms_host_unregister": (ctypes.c_int, [_V]),
    "ms_surface_energy_and_gradient": (ctypes.c_int, [_i32, _i32, _D, _I, _D, _D, _D, _i32]),
    "ms_grad_cotan_batch": (ctypes.c_int, [_i32, _D, _D, _D, _D]),
    "ms_apply_beltrami_laplacian": (ctypes.c_int, [_i32, _i32, _i32, _D, _I, _D, _D, _i32]),
    "ms_p1_triangle_divergence": (ctypes.c_int, [_i32, _i32, _D, _D, _I, _D, _D, _D, _D, _D, _i32]),
    "ms_p1_vertex_divergence": (ctypes.c_int, [_i32, _i32, _D, _D, _I, _D, _D, _i32]),
    "ms_compute_curvature_data": (ctypes.c_int, [_i32, _i32, _D, _I, _D, _D, _D, _i32, _D, _D, _D]),
    "ms_volume_and_gradient": (ctypes.c_int, [_i32, _i32, _D, _I, _f64, _D, _D]),
}

_lib = None


def build(force: bool = False) -> str:
    """Compile the CUDA extension in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    if force and os.path.exists(LIB_PATH):
        os.remove(LIB_PATH)
    subprocess.check_call(["make", "-s", "-C", CSRC, "all"])
    return LIB_PATH


def lib() -> ctypes.CDLL:
    """Load the shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B200Error(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`"
                " (there is no CPU fallback for the B200 path)")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().ms_last_error()
        raise B200Error(f"libms_b200 error {rc}: {msg.decode() if msg else '?'}")


def device_count() -> int:
    n = ctypes.c_int(0)
    rc = lib().ms_device_count(ctypes.byref(n))
    return int(n.value) if rc == 0 else 0


def dptr(a):
    return None if a is None else a.ctypes.data_as(_D)


def iptr(a):
    return None if a is None else a.ctypes.data_as(_I)


def bptr(a):
    return None if a is None else a.ctypes.data_as(_B)


def as_f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None and a.shape != shape:
        raise ValueError(f"expected shape {shape}, got {a.shape}")
    return a
