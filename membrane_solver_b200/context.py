"""Device-resident mesh context: the B200 twin of ``runtime/energy_context.py``.

``DeviceMesh`` owns one ``ms_ctx`` (C ABI): packed topology, positions, tilts,
per-entity parameters and all outputs live in HBM across minimiser steps and are
re-uploaded only when the reference bumps the matching version counter
(SURVEY.md section 3.5): topology <- ``_facet_loops_version`` / ``_vertex_ids_version``
/ ``_topology_version``; positions <- every evaluation that passes a host array.
"""

from __future__ import annotations

import ctypes
from dataclasses import dataclass

import numpy as np

from . import _lib as L


@dataclass
class EvalResult:
    """Host copy of the scalar vector of one evaluation."""

    scalars: np.ndarray

    @property
    def e_surface(self) -> float:
        return float(self.scalars[L.SC_E_SURFACE])

    @property
    def area(self) -> float:
        return float(self.scalars[L.SC_AREA])

    @property
    def volume(self) -> float:
        return float(self.scalars[L.SC_VOLUME])

    @property
    def e_bending(self) -> float:
        return float(self.scalars[L.SC_E_BENDING])

    @property
    def e_tilt(self) -> float:
        return float(self.scalars[L.SC_E_TILT])

    @property
    def kkt_lambda(self) -> float:
        return float(self.scalars[L.SC_LAMBDA])


class _CudaArrayView:
    """Exposes a device buffer of the context through ``__cuda_array_interface__``
    so that ``torch.as_tensor(view, device=...)`` aliases it without a copy."""

    def __init__(self, ptr: int, shape, owner):
        self._owner = owner  # keeps the context alive
        self.__cuda_array_interface__ = {
            "shape": tuple(int(s) for s in shape),
            "typestr": "<f8",
            "data": (int(ptr), False),
            "version": 3,
            "strides": None,
        }


class DeviceMesh:
    """One mesh resident on one GPU."""

    def __init__(self, device: int = 0, *, threads: int | None = None, max_owned: int | None = None,
                 max_local: int | None = None,
                 fill_pct: int | None = None, repair_sweeps: int | None = None):
        self._lib = L.lib()
        handle = ctypes.c_void_p()
        L.check(self._lib.ms_ctx_create(int(device), ctypes.byref(handle)))
        self._h = handle
        self.device = int(device)
        self.nv = 0
        self.nf = 0
        self.n_owned = 0
        if threads is not None or max_owned is not None or max_local is not None:
            L.check(self._lib.ms_ctx_set_pack_params(self._h, int(threads or 96), int(max_owned or 512),
                                                     int(max_local or 896)))
        if fill_pct is not None or repair_sweeps is not None:
            L.check(self._lib.ms_ctx_set_pack_tuning(self._h, int(87 if fill_pct is None else fill_pct),
                                                     int(1 if repair_sweeps is None else repair_sweeps)))

    # -- lifetime -----------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.ms_ctx_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- topology and parameters --------------------------------------------
    def set_topology(self, nv: int, tri: np.ndarray, *, is_boundary=None, body_mask=None,
                     fixed_mask=None, n_owned: int | None = None, order_hint=None) -> None:
        """``n_owned`` < nv marks rows [n_owned, nv) as ghosts of other partitions (multi-GPU).
        ``order_hint``: positions (nv,3) used only to pick the internal (Morton) vertex order."""
        tri = np.ascontiguousarray(tri, dtype=np.int32).reshape(-1, 3)
        keep = [tri]

        def mask(a, n):
            if a is None:
                return None
            a = np.ascontiguousarray(a, dtype=np.uint8)
            if a.shape != (n,):
                raise ValueError(f"mask must have shape ({n},)")
            keep.append(a)
            return a

        b = mask(is_boundary, nv)
        bm = mask(body_mask, tri.shape[0])
        fx = mask(fixed_mask, nv)
        self.n_owned = int(nv if n_owned is None else n_owned)
        if order_hint is not None and self.n_owned == int(nv):
            hint = L.as_f64(order_hint, (int(nv), 3))
            L.check(self._lib.ms_ctx_set_vertex_order_hint(self._h, int(nv), L.dptr(hint)))
        L.check(self._lib.ms_ctx_set_topology_partition(self._h, int(nv), self.n_owned, int(tri.shape[0]),
                                                        L.iptr(tri), L.bptr(b), L.bptr(bm), L.bptr(fx)))
        self.nv = int(nv)
        self.nf = int(tri.shape[0])

    def set_fixed_mask(self, fixed_mask) -> None:
        """Replace the fixed-vertex mask (None: no fixed vertex); the packed topology stays as it is."""
        if fixed_mask is None:
            L.check(self._lib.ms_ctx_set_fixed_mask(self._h, None))
            return
        m = np.ascontiguousarray(fixed_mask, dtype=np.uint8)
        if m.shape != (self.nv,):
            raise ValueError(f"mask must have shape ({self.nv},)")
        L.check(self._lib.ms_ctx_set_fixed_mask(self._h, L.bptr(m)))

    def permutation(self) -> np.ndarray:
        """Internal row -> caller's vertex row."""
        out = np.empty(self.nv, dtype=np.int32)
        L.check(self._lib.ms_ctx_get_permutation(self._h, L.iptr(out)))
        return out

    def pack_info(self) -> dict:
        info = L.PackInfo()
        L.check(self._lib.ms_ctx_pack_info(self._h, ctypes.byref(info)))
        return {name: int(getattr(info, name)) for name, _ in L.PackInfo._fields_}

    def packing(self) -> dict:
        """The current packing as NumPy arrays (``ms_ctx_get_packing``): ``headers`` ((n_patches, 32) uint8, the
        32-byte patch headers), ``halo_ids`` (int32), ``recs`` ((n_slots, 4) uint16: a, b, c, flags) and ``slot_facet``
        (int32, -1 for an empty slot).  It is what the host packer makes of the internal-order rows."""
        info = self.pack_info()
        out = {"headers": np.zeros((info["n_patches"], 32), dtype=np.uint8),
               "halo_ids": np.zeros(info["n_halo"], dtype=np.int32),
               "recs": np.zeros((info["n_slots"], 4), dtype=np.uint16),
               "slot_facet": np.zeros(info["n_slots"], dtype=np.int32)}
        L.check(self._lib.ms_ctx_get_packing(self._h, out["headers"].ctypes.data_as(ctypes.c_void_p),
                                             L.iptr(out["halo_ids"]), out["recs"].ctypes.data_as(ctypes.c_void_p),
                                             L.iptr(out["slot_facet"])))
        return out

    def patch_ranges(self) -> np.ndarray:
        n = self.pack_info()["n_patches"]
        out = np.empty(n + 1, dtype=np.int32)
        L.check(self._lib.ms_ctx_patch_ranges(self._h, L.iptr(out)))
        return out

    def halo_rows(self, patch_begin: int, patch_count: int, own_lo: int, own_hi: int) -> np.ndarray:
        n = ctypes.c_int64(0)
        L.check(self._lib.ms_ctx_halo_rows(self._h, patch_begin, patch_count, own_lo, own_hi, None,
                                           ctypes.byref(n)))
        out = np.empty(int(n.value), dtype=np.int32)
        if out.size:
            L.check(self._lib.ms_ctx_halo_rows(self._h, patch_begin, patch_count, own_lo, own_hi,
                                               L.iptr(out), ctypes.byref(n)))
        return out

    def set_surface_tension(self, gamma) -> None:
        """Scalar (uniform) or per-facet array, as ``Mesh.get_facet_parameter_array`` builds it."""
        if np.ndim(gamma) == 0:
            L.check(self._lib.ms_ctx_set_surface_tension(self._h, None, float(gamma)))
            return
        g = L.as_f64(gamma, (self.nf,))
        if g.size and np.all(g == g[0]):
            L.check(self._lib.ms_ctx_set_surface_tension(self._h, None, float(g[0])))
        else:
            L.check(self._lib.ms_ctx_set_surface_tension(self._h, L.dptr(g), 0.0))

    def set_bending_params(self, kappa, c0) -> None:
        def split(x):
            if np.ndim(x) == 0:
                return None, float(x)
            a = L.as_f64(x, (self.nv,))
            if a.size and np.all(a == a[0]):
                return None, float(a[0])
            return a, 0.0

        ka, ku = split(kappa)
        ca, cu = split(c0)
        L.check(self._lib.ms_ctx_set_bending_params(self._h, L.dptr(ka), L.dptr(ca), ku, cu))

    def set_tilt_rigidity(self, k_tilt: float) -> None:
        L.check(self._lib.ms_ctx_set_tilt_rigidity(self._h, float(k_tilt)))

    # -- leaflet tilt modules (tilt_in/out, bending_tilt_in/out) ------------
    def set_leaflet(self, leaflet: int, *, div_sign: float, kappa=0.0, c0=0.0, k_tilt: float = 0.0, k_smooth: float = 0.0,
                    facet_keep=None, interior=None, base_zero=None, tilt_row_weight=None,
                    facet_consistent=None, consistent: bool = False) -> None:
        """Selections and parameters of one leaflet (``struct ms_leaflet_desc``).  ``kappa`` / ``c0``:
        scalar or (nv,) array; masks in the caller's vertex / facet order, None = absent."""
        hold = []

        def mask(a, n):
            if a is None:
                return None
            a = np.ascontiguousarray(a, dtype=np.uint8)
            if a.shape != (n,):
                raise ValueError(f"mask must have shape ({n},)")
            hold.append(a)
            return a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))

        def vec(a):
            if a is None or np.ndim(a) == 0:
                return None
            a = L.as_f64(a, (self.nv,))
            hold.append(a)
            return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))

        d = L.LeafletDesc(
            facet_keep=mask(facet_keep, self.nf), interior=mask(interior, self.nv), base_zero=mask(base_zero, self.nv),
            kappa=vec(kappa), c0=vec(c0), tilt_row_weight=vec(tilt_row_weight),
            facet_consistent=mask(facet_consistent, self.nf),
            kappa_default=float(kappa) if np.ndim(kappa) == 0 else 0.0,
            c0_default=float(c0) if np.ndim(c0) == 0 else 0.0,
            k_tilt=float(k_tilt), k_smooth=float(k_smooth), div_sign=float(div_sign), consistent_default=int(bool(consistent)), reserved=0)
        L.check(self._lib.ms_ctx_set_leaflet(self._h, int(leaflet), ctypes.byref(d)))

    # -- leaflet tilt relaxation primitives (tilt_relaxation.py:426-1057, GD solver) --
    def set_leaflet_fixed(self, leaflet: int, fixed_rows) -> None:
        m = None
        if fixed_rows is not None:
            m = np.ascontiguousarray(fixed_rows, dtype=np.uint8)
            if m.shape != (self.nv,):
                raise ValueError(f"mask must have shape ({self.nv},)")
        L.check(self._lib.ms_ctx_set_leaflet_fixed(self._h, int(leaflet), L.bptr(m)))

    def update_vertex_normals(self) -> None:
        L.check(self._lib.ms_ctx_update_vertex_normals(self._h))

    def leaflet_project_tilts(self, leaflet: int) -> None:
        L.check(self._lib.ms_ctx_leaflet_project_tilts(self._h, int(leaflet)))

    def leaflet_gradient_norm2(self, leaflet: int, read: bool = True) -> float | None:
        if not read:                                   # result stays on the device: leaflet_results()
            L.check(self._lib.ms_ctx_leaflet_gradient_norm2(self._h, int(leaflet), None))
            return None
        out = np.zeros(1)
        L.check(self._lib.ms_ctx_leaflet_gradient_norm2(self._h, int(leaflet), L.dptr(out)))
        return float(out[0])

    def eval_leaflet_pair(self, modules: int, *, want_grad: bool = False, want_tilt_grad: bool = True,
                          accumulate: int = 0, use_trial: bool = False) -> None:
        """Inner and outer leaflet together (one launch on small meshes); read with ``leaflet_results()``."""
        L.check(self._lib.ms_ctx_eval_leaflet_pair(self._h, int(modules), int(bool(want_grad)), int(bool(want_tilt_grad)),
                                                   int(accumulate), int(bool(use_trial))))

    def leaflet_results(self) -> np.ndarray:
        """One synchronisation for everything the leaflet calls left on the device: rows = leaflet slots,
        columns = E_bending_tilt, E_tilt, E_tilt_smoothness, |g|^2, r.z."""
        out = np.zeros(15)
        L.check(self._lib.ms_ctx_leaflet_results(self._h, L.dptr(out)))
        return out.reshape(3, 5)

    def leaflet_make_trial(self, leaflet: int, step: float, along_direction: bool = False) -> None:
        L.check(self._lib.ms_ctx_leaflet_make_trial(self._h, int(leaflet), float(step), int(bool(along_direction))))

    def leaflet_build_preconditioner(self, leaflet: int, k_smooth: float, kept_facets_only: bool) -> None:
        L.check(self._lib.ms_ctx_leaflet_build_preconditioner(self._h, int(leaflet), float(k_smooth),
                                                              int(bool(kept_facets_only))))

    def leaflet_rz(self, leaflet: int, preconditioned: bool, read: bool = True) -> float | None:
        if not read:
            L.check(self._lib.ms_ctx_leaflet_rz(self._h, int(leaflet), int(bool(preconditioned)), None))
            return None
        out = np.zeros(1)
        L.check(self._lib.ms_ctx_leaflet_rz(self._h, int(leaflet), int(bool(preconditioned)), L.dptr(out)))
        return float(out[0])

    def leaflet_cg_direction(self, leaflet: int, beta: float, restart: bool, preconditioned: bool) -> None:
        L.check(self._lib.ms_ctx_leaflet_cg_direction(self._h, int(leaflet), float(beta), int(bool(restart)),
                                                      int(bool(preconditioned))))

    def leaflet_swap_trial(self, leaflet: int) -> None:
        L.check(self._lib.ms_ctx_leaflet_swap_trial(self._h, int(leaflet)))

    def eval_leaflet(self, leaflet: int, modules: int, *, want_grad: bool = True, want_tilt_grad: bool = True,
                     accumulate: int = 0, use_trial: bool = False, read: bool = True):
        """(E_bending_tilt, E_tilt, E_tilt_smoothness) of the leaflet's modules; gradients stay on the device
        (``ARR_GRAD``, ``ARR_TILT_GRAD_IN`` / ``_OUT``)."""
        if not read:                                   # energies stay on the device: leaflet_results()
            L.check(self._lib.ms_ctx_eval_leaflet(self._h, int(leaflet), int(modules), int(bool(want_grad)),
                                                  int(bool(want_tilt_grad)), int(accumulate), int(bool(use_trial)),
                                                  None))
            return None
        e = np.zeros(3)
        L.check(self._lib.ms_ctx_eval_leaflet(self._h, int(leaflet), int(modules), int(bool(want_grad)),
                                              int(bool(want_tilt_grad)), int(accumulate), int(bool(use_trial)),
                                              L.dptr(e)))
        return float(e[0]), float(e[1]), float(e[2])

    # -- state --------------------------------------------------------------
    def upload(self, which: int, host: np.ndarray) -> None:
        a = L.as_f64(host)
        L.check(self._lib.ms_ctx_upload(self._h, which, L.dptr(a), 0, a.size))
        # the copy is asynchronous on the context stream; the source must stay valid
        L.check(self._lib.ms_ctx_sync(self._h))

    def set_positions(self, pos: np.ndarray) -> None:
        self.upload(L.ARR_POSITIONS, L.as_f64(pos, (self.nv, 3)))

    def set_tilts(self, tilts: np.ndarray) -> None:
        self.upload(L.ARR_TILTS, L.as_f64(tilts, (self.nv, 3)))

    def set_direction(self, d: np.ndarray) -> None:
        self.upload(L.ARR_DIRECTION, L.as_f64(d, (self.nv, 3)))

    def download(self, which: int) -> np.ndarray:
        n = int(self._lib.ms_ctx_array_len(self._h, which))
        out = np.empty(n, dtype=np.float64)
        L.check(self._lib.ms_ctx_get_array(self._h, which, L.dptr(out), 0, n))
        w = L.ARRAY_WIDTH[which]
        return out.reshape(-1, w) if w > 1 else out

    def device_view(self, which: int) -> _CudaArrayView:
        ptr = self._lib.ms_ctx_device_ptr(self._h, which)
        if not ptr:
            raise L.B200Error(f"array {which} is not available")
        n = int(self._lib.ms_ctx_array_len(self._h, which))
        w = L.ARRAY_WIDTH[which]
        return _CudaArrayView(ptr, (n // w, w) if w > 1 else (n,), self)

    # -- evaluation ---------------------------------------------------------
    @staticmethod
    def options(modules: int, *, flags: int = 0, want_grad: bool = True, constraint_mode: int = -1,
                k_vol: float = 0.0, v_target: float = 0.0, apply_fixed: bool = False,
                use_trial: bool = False, patch_begin: int = 0, patch_count: int = -1,
                diagnostics: bool = False, want_tilt_grad: bool = False) -> L.EvalOpts:
        return L.EvalOpts(modules=modules, flags=flags, want_grad=int(want_grad),
                          constraint_mode=constraint_mode, k_vol=k_vol, v_target=v_target,
                          apply_fixed=int(apply_fixed), use_trial=int(use_trial),
                          patch_begin=patch_begin, patch_count=patch_count,
                          diagnostics=int(diagnostics), want_tilt_grad=int(want_tilt_grad))

    def eval(self, opts: L.EvalOpts) -> EvalResult:
        """Evaluate with everything resident; only the 16 scalars come back."""
        sc = np.zeros(L.SC_COUNT)
        L.check(self._lib.ms_ctx_eval(self._h, ctypes.byref(opts), L.dptr(sc)))
        return EvalResult(sc)

    def eval_async(self, opts: L.EvalOpts) -> None:
        L.check(self._lib.ms_ctx_eval_async(self._h, ctypes.byref(opts)))

    def self_check(self) -> tuple[int, int, int]:
        """Violation counters of a self-check build (libms_b200_checked.so); raises on other builds."""
        out = (ctypes.c_int32 * 3)()
        L.check(self._lib.ms_ctx_self_check(self._h, out))
        return int(out[0]), int(out[1]), int(out[2])

    def eval_stage(self, opts: L.EvalOpts, stage: int) -> None:
        """Stage 0 = pass A, stage 1 = pass B + fused finalisation (ms_ctx_eval_async in two calls)."""
        L.check(self._lib.ms_ctx_eval_stage(self._h, ctypes.byref(opts), int(stage)))

    def eval_pass_a(self, opts: L.EvalOpts) -> None:
        L.check(self._lib.ms_ctx_eval_pass_a(self._h, ctypes.byref(opts)))

    def eval_pass_b(self, opts: L.EvalOpts) -> None:
        L.check(self._lib.ms_ctx_eval_pass_b(self._h, ctypes.byref(opts)))

    def eval_finish(self, opts: L.EvalOpts) -> None:
        L.check(self._lib.ms_ctx_eval_finish(self._h, ctypes.byref(opts)))

    def eval_reduce(self, opts: L.EvalOpts) -> None:
        L.check(self._lib.ms_ctx_eval_reduce(self._h, ctypes.byref(opts)))

    def eval_project(self, opts: L.EvalOpts) -> None:
        L.check(self._lib.ms_ctx_eval_project(self._h, ctypes.byref(opts)))

    # -- halo exchange helpers (multi-GPU partitions) -------------------------
    def set_send_rows(self, rows: np.ndarray) -> None:
        rows = np.ascontiguousarray(rows, dtype=np.int32)
        L.check(self._lib.ms_ctx_set_send_rows(self._h, L.iptr(rows), int(rows.size)))

    # -- halo exchange over NVLink peer memory (multi-GPU) -------------------
    def ipc_export(self, which: int) -> bytes:
        buf = (ctypes.c_uint8 * L.IPC_HANDLE_BYTES)()
        L.check(self._lib.ms_ctx_ipc_export(self._h, int(which), buf))
        return bytes(buf)

    def peer_close(self) -> None:
        L.check(self._lib.ms_ctx_peer_close(self._h))

    def peer_open(self, slot: int, which: int, handle: bytes) -> None:
        if len(handle) != L.IPC_HANDLE_BYTES:
            raise ValueError("IPC handles are 64 bytes")
        buf = (ctypes.c_uint8 * L.IPC_HANDLE_BYTES).from_buffer_copy(handle)
        L.check(self._lib.ms_ctx_peer_open(self._h, int(slot), int(which), buf))

    def peer_set_pointer(self, slot: int, which: int, device_ptr: int) -> None:
        L.check(self._lib.ms_ctx_peer_set_pointer(self._h, int(slot), int(which), ctypes.c_void_p(int(device_ptr))))

    def flag_words_ptr(self) -> int:
        p = self._lib.ms_ctx_flag_words_ptr(self._h)
        if not p:
            raise L.B200Error("flag words are not available")
        return int(p)

    def device_ptr(self, which: int) -> int:
        p = self._lib.ms_ctx_device_ptr(self._h, int(which))
        if not p:
            raise L.B200Error(f"array {which} is not available")
        return int(p)

    def set_ghost_sources(self, n_slots: int, owner_slot: np.ndarray, owner_row: np.ndarray) -> None:
        o = np.ascontiguousarray(owner_slot, dtype=np.int32)
        r = np.ascontiguousarray(owner_row, dtype=np.int32)
        if o.shape != (self.nv - self.n_owned,) or r.shape != o.shape:
            raise ValueError("one owner slot and one owner row per ghost row")
        L.check(self._lib.ms_ctx_set_ghost_sources(self._h, int(n_slots), L.iptr(o), L.iptr(r)))

    def halo_prepare(self) -> None:
        L.check(self._lib.ms_ctx_halo_prepare(self._h))

    def halo_signal(self, flag: int) -> None:
        L.check(self._lib.ms_ctx_halo_signal(self._h, int(flag)))

    def halo_pull(self, which: int, flag: int) -> None:
        L.check(self._lib.ms_ctx_halo_pull(self._h, int(which), int(flag)))

    def set_rank_slot(self, slot: int, n_slots: int) -> None:
        L.check(self._lib.ms_ctx_set_rank_slot(self._h, int(slot), int(n_slots)))

    def allreduce_scalars(self, count: int = 12) -> None:
        L.check(self._lib.ms_ctx_allreduce_scalars(self._h, int(count)))

    def set_push_targets(self, dst_slot, src_row, dst_row) -> None:
        a, b, c = (np.ascontiguousarray(x, dtype=np.int32) for x in (dst_slot, src_row, dst_row))
        if not (a.shape == b.shape == c.shape):
            raise ValueError("push target arrays must have the same length")
        L.check(self._lib.ms_ctx_set_push_targets(self._h, int(a.size), L.iptr(a), L.iptr(b), L.iptr(c)))

    def halo_push(self, which: int, flag: int) -> None:
        L.check(self._lib.ms_ctx_halo_push(self._h, int(which), int(flag)))

    def eval_partition(self, opts, exchange_positions: bool = True, in_kernel: bool = False) -> None:
        """One partitioned evaluation with the transport folded into the compute launches (5 launches), or, with
        ``in_kernel``, carried out inside the patch kernels behind the interior patches (2 launches: pass A and pass B, the
        last CTA of the last pass gathering the scalars; a pack of fewer than 64 threads falls back to the fused pull)."""
        flags = int(bool(exchange_positions)) | (2 if in_kernel else 0)
        L.check(self._lib.ms_ctx_eval_partition(self._h, ctypes.byref(opts), flags))

    def halo_error(self) -> bool:
        e = ctypes.c_int32(0)
        L.check(self._lib.ms_ctx_halo_error(self._h, ctypes.byref(e)))
        return bool(e.value)

    def pack_send(self, which: int, out_device_ptr: int) -> None:
        L.check(self._lib.ms_ctx_pack_send(self._h, int(which), ctypes.c_void_p(int(out_device_ptr))))

    def read_scalars(self) -> EvalResult:
        sc = np.zeros(L.SC_COUNT)
        L.check(self._lib.ms_ctx_read_scalars(self._h, L.dptr(sc)))
        return EvalResult(sc)

    def eval_host(self, opts: L.EvalOpts, pos: np.ndarray | None, *, grad: np.ndarray | None = None,
                  volgrad: np.ndarray | None = None, tilt_grad: np.ndarray | None = None) -> EvalResult:
        """End-to-end evaluation with HOST buffers: H2D positions, kernels, D2H results."""
        sc = np.zeros(L.SC_COUNT)
        for a in (grad, volgrad, tilt_grad):
            if a is not None and (a.dtype != np.float64 or not a.flags["C_CONTIGUOUS"] or a.shape != (self.nv, 3)):
                raise ValueError("output arrays must be C-contiguous float64 (nv,3)")
        p = None if pos is None else L.as_f64(pos, (self.nv, 3))
        L.check(self._lib.ms_ctx_eval_host(self._h, ctypes.byref(opts), L.dptr(p), L.dptr(sc),
                                           L.dptr(grad), L.dptr(volgrad), L.dptr(tilt_grad)))
        return EvalResult(sc)

    def make_trial(self, alpha: float) -> None:
        L.check(self._lib.ms_ctx_make_trial(self._h, float(alpha)))

    def accept_trial(self) -> None:
        L.check(self._lib.ms_ctx_accept_trial(self._h))

    def direction_from_gradient(self, scale: float = -1.0) -> None:
        L.check(self._lib.ms_ctx_direction_from_gradient(self._h, float(scale)))

    def axpy(self, dst: int, src: int, alpha: float, skip_fixed: bool = True) -> None:
        L.check(self._lib.ms_ctx_axpy(self._h, int(dst), int(src), float(alpha), int(bool(skip_fixed))))

    def vertex_average(self, rounds: int = 1, group=None) -> None:
        """Evolver-style vertex averaging of the resident positions, ``rounds`` times (``ms_ctx_vertex_average``):
        the device twin of ``geometry.vertex_average.vertex_average_arrays`` with the context's fixed mask as the
        immovable rows.  ``group``: (nv,) pin groups in the caller's vertex order, -1 = none.  Overwrites the trial
        positions."""
        g = None
        if group is not None:
            g = np.ascontiguousarray(group, dtype=np.int32)
            if g.shape != (self.nv,):
                raise ValueError(f"group must have shape ({self.nv},)")
        L.check(self._lib.ms_ctx_vertex_average(self._h, L.iptr(g), int(rounds)))

    def equiangulate(self, max_iterations: int = 100) -> int:
        """Delaunay edge flips of the resident triangle rows (``ms_ctx_equiangulate``), the device twin of
        ``geometry.equiangulate.equiangulate_triangles`` with the context's fixed mask; returns the number of flips.
        After a call that flipped, the leaflet selections must be set again (``set_leaflet``)."""
        flips, sweeps = ctypes.c_int64(0), ctypes.c_int32(0)
        L.check(self._lib.ms_ctx_equiangulate(self._h, int(max_iterations), ctypes.byref(flips), ctypes.byref(sweeps)))
        self.last_equiangulate_sweeps = int(sweeps.value)
        return int(flips.value)

    def equiangulate_stats(self) -> dict:
        """Sweeps run by the last ``equiangulate``, the selection rounds of each, and its times in ms: device time of
        the sweeps, row download, device packing of the new rows (CUDA events), commit of the new packing."""
        n = ctypes.c_int32(0)
        L.check(self._lib.ms_ctx_equiangulate_stats(self._h, None, None, 0, ctypes.byref(n)))
        ms = np.zeros(4)
        rounds = np.zeros(max(int(n.value), 1), dtype=np.int32)
        L.check(self._lib.ms_ctx_equiangulate_stats(self._h, L.dptr(ms), L.iptr(rounds), int(n.value), ctypes.byref(n)))
        return {"sweeps_run": int(n.value), "rounds": rounds[:int(n.value)].tolist(), "sweep_ms": float(ms[0]),
                "d2h_ms": float(ms[1]), "pack_ms": float(ms[2]), "upload_ms": float(ms[3])}

    def refine(self, levels: int = 1) -> np.ndarray:
        """1 -> 4 midpoint refinement of the resident mesh, ``levels`` times (``ms_ctx_refine``), the device twin of
        ``geometry.refine.refine_triangles`` with the context's fixed mask.  Updates ``nv`` / ``nf`` and returns the
        composed ``parent`` (refined facet -> original facet).  The leaflet selections must be set again."""
        nf0 = self.nf
        nv, nf = ctypes.c_int32(0), ctypes.c_int32(0)
        L.check(self._lib.ms_ctx_refine(self._h, int(levels), ctypes.byref(nv), ctypes.byref(nf)))
        self.nv = self.n_owned = int(nv.value)
        self.nf = int(nf.value)
        return np.arange(self.nf, dtype=np.int64) % max(nf0, 1)

    def refine_stats(self) -> dict:
        """Times of the last ``refine`` in ms: device time, download of rows and order, device packing of the refined
        rows (CUDA events), per-facet inheritance and commit."""
        ms = np.zeros(4)
        L.check(self._lib.ms_ctx_refine_stats(self._h, L.dptr(ms)))
        return {"device_ms": float(ms[0]), "d2h_ms": float(ms[1]), "pack_ms": float(ms[2]), "upload_ms": float(ms[3])}

    def triangles(self) -> np.ndarray:
        """The current (nf,3) triangle rows in the caller's vertex numbering."""
        out = np.empty((self.nf, 3), dtype=np.int32)
        L.check(self._lib.ms_ctx_get_triangles(self._h, L.iptr(out)))
        return out

    def cg_direction(self, restart: bool) -> None:
        L.check(self._lib.ms_ctx_cg_direction(self._h, int(bool(restart))))

    def cg_commit(self) -> None:
        L.check(self._lib.ms_ctx_cg_commit(self._h))

    def line_search_stats(self) -> tuple[float, float, float, float]:
        """(min edge length, max row norm of the direction, <g,d>, <g,g>) computed on the device."""
        out = np.zeros(4)
        L.check(self._lib.ms_ctx_line_search_stats(self._h, L.dptr(out)))
        return float(out[0]), float(out[1]), float(out[2]), float(out[3])

    def normal_change_ok(self, limit_radians: float = 0.5) -> bool:
        ok = ctypes.c_int32(0)
        L.check(self._lib.ms_ctx_normal_change_ok(self._h, float(limit_radians), ctypes.byref(ok)))
        return bool(ok.value)

    def minimize(self, opts: L.MinimizeOpts, n_steps: int, *, step_size: float, cg_iter: int = 0,
                 cg_have_history: bool = False) -> tuple[L.MinimizeResult, list]:
        """``n_steps`` steps of ``DeviceMinimizer.minimize`` under device control (``ms_ctx_minimize``): one CUDA graph,
        one host synchronisation.  Returns the result struct (step size and conjugate-gradient state after the call
        included) and the history rows ``(step, accepted energy, step size in, success)``."""
        res = L.MinimizeResult(step_size=float(step_size), cg_iter=int(cg_iter), cg_have_history=int(bool(cg_have_history)))
        cap = max(int(n_steps), 0)
        hist = np.zeros((max(cap, 1), 4))
        L.check(self._lib.ms_ctx_minimize(self._h, ctypes.byref(opts), int(n_steps), ctypes.byref(res), L.dptr(hist), cap))
        rows = [(int(h[0]), float(h[1]), float(h[2]), bool(h[3])) for h in hist[:min(res.n_history, cap)]]
        return res, rows

    def minimize_stats(self) -> dict:
        """The last ``minimize``: line searches, trials, evaluations, host synchronisations (blocking waits of the
        call), actions, normal-flip guards run and trials they rejected, the device time of its graph (CUDA events) and
        the host time spent building the graph, in ms."""
        n = np.zeros(7, dtype=np.int64)
        ms = np.zeros(2)
        L.check(self._lib.ms_ctx_minimize_stats(self._h, n.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), L.dptr(ms)))
        return {"steps": int(n[0]), "trials": int(n[1]), "evaluations": int(n[2]), "host_syncs": int(n[3]),
                "actions": int(n[4]), "guards": int(n[5]), "guard_rejects": int(n[6]), "device_ms": float(ms[0]),
                "build_ms": float(ms[1])}

    def dots(self) -> None:
        L.check(self._lib.ms_ctx_dots(self._h))

    # -- timing -------------------------------------------------------------
    def timer_start(self) -> None:
        L.check(self._lib.ms_ctx_timer_start(self._h))

    def timer_stop(self) -> float:
        ms = ctypes.c_float(0.0)
        L.check(self._lib.ms_ctx_timer_stop(self._h, ctypes.byref(ms)))
        return float(ms.value)

    def event_record(self, index: int) -> None:
        L.check(self._lib.ms_ctx_event_record(self._h, int(index)))

    def event_elapsed(self, i: int, j: int) -> float:
        ms = ctypes.c_float(0.0)
        L.check(self._lib.ms_ctx_event_elapsed(self._h, int(i), int(j), ctypes.byref(ms)))
        return float(ms.value)

    def flush_l2(self, nbytes: int = 256 << 20) -> None:
        L.check(self._lib.ms_ctx_flush_l2(self._h, int(nbytes)))

    def sync(self) -> None:
        L.check(self._lib.ms_ctx_sync(self._h))
