"""TEST-ONLY stand-in for ``membrane_solver_b200.context.DeviceMesh`` backed by the host emulator
(tests/emul): lets the CPU tier drive the plugin modules, the evaluation manager and the
residency logic end to end without a GPU.  The product never imports this."""

import numpy as np

import ms_test_helpers as H
from membrane_solver_b200 import _lib as L
from membrane_solver_b200.context import EvalResult


class FakeDeviceMesh:
    instances = []

    def __init__(self, device=0, **pack):
        self.pack = {k: v for k, v in pack.items() if v is not None and k in ("threads", "max_owned", "max_local")}
        self.nv = self.nf = 0
        self.gamma = 1.0
        self.kappa = self.c0 = 0.0
        self.k_tilt = 0.0
        self.tilts = None
        self.arrays = {}
        self.scalars = np.zeros(L.SC_COUNT)
        self._pg = self._pd = None
        self.topology_uploads = 0
        self.evals = 0
        FakeDeviceMesh.instances.append(self)

    # -- topology / parameters
    def set_topology(self, nv, tri, *, is_boundary=None, body_mask=None, fixed_mask=None, n_owned=None,
                     order_hint=None):
        self.nv, self.tri = int(nv), np.ascontiguousarray(tri, dtype=np.int32).reshape(-1, 3)
        self.nf = self.tri.shape[0]
        self.is_boundary, self.body_mask, self.fixed = is_boundary, body_mask, fixed_mask
        self.topology_uploads += 1
        # like the device: zeroed gradients, no trial positions, direction or conjugate-gradient history
        self.arrays.update({L.ARR_GRAD: np.zeros((self.nv, 3)), L.ARR_VOLGRAD: np.zeros((self.nv, 3))})
        self.arrays.pop(L.ARR_TRIAL, None)
        self.arrays.pop(L.ARR_DIRECTION, None)
        self._pg = self._pd = None

    def permutation(self):
        return np.arange(self.nv, dtype=np.int32)  # the emulator keeps the caller's vertex order

    def set_fixed_mask(self, fixed_mask):
        self.fixed = fixed_mask

    def set_surface_tension(self, gamma):
        self.gamma = gamma

    def set_bending_params(self, kappa, c0):
        self.kappa, self.c0 = kappa, c0

    def set_tilt_rigidity(self, k):
        self.k_tilt = float(k)

    def set_tilts(self, t):
        self.tilts = np.array(t, dtype=np.float64)

    options = staticmethod(lambda modules, **kw: dict(modules=modules, **kw))

    # -- evaluation
    def eval_host(self, opts, pos, *, grad=None, volgrad=None, tilt_grad=None):
        self.evals += 1
        kw = dict(self.pack)
        g, k, c = self.gamma, self.kappa, self.c0
        # a tilt-only evaluation runs pass B on the device, which leaves the RAW gradients of the modules
        tilt_only = (not opts.get("want_grad", True) and opts.get("want_tilt_grad", False)
                     and bool(opts["modules"] & L.MOD_TILT))
        out = H.emulate(pos, self.tri, modules=opts["modules"], flags=opts.get("flags", 0),
                        want_grad=opts.get("want_grad", True) or tilt_only, is_boundary=self.is_boundary,
                        body_mask=self.body_mask, tilts=self.tilts, gamma=g if np.ndim(g) else None, gamma_u=g if not np.ndim(g) else 1.0,
                        kappa=k if np.ndim(k) else None, kappa_u=0.0 if np.ndim(k) else float(k),
                        c0=c if np.ndim(c) else None, c0_u=0.0 if np.ndim(c) else float(c), k_tilt=self.k_tilt, **kw)
        sc = np.zeros(L.SC_COUNT)
        sc[L.SC_E_SURFACE], sc[L.SC_AREA], sc[L.SC_VOLUME] = out["E_surface"], out["area"], out["volume"]
        sc[L.SC_E_BENDING], sc[L.SC_E_TILT] = out["E_bending"], out["E_tilt"]
        sc[L.SC_E_BENDING_TILT] = out["E_bending_tilt"]
        g_out, gc = out["grad"], out["volgrad"]
        if opts.get("want_grad", True):
            # numpy restatement of k_dots / k_project (TEST ONLY)
            sc[L.SC_G_G], sc[L.SC_G_GC], sc[L.SC_GC_GC] = (g_out * g_out).sum(), (g_out * gc).sum(), (gc * gc).sum()
            mode = opts.get("constraint_mode", -1)
            if mode == 0 and (opts["modules"] & L.MOD_VOLUME) and sc[L.SC_GC_GC] > 1e-18:
                lam = sc[L.SC_G_GC] / sc[L.SC_GC_GC]
                g_out = g_out - lam * gc
                sc[L.SC_LAMBDA] = lam
            elif mode == 1 and (opts["modules"] & L.MOD_VOLUME):
                coef = opts.get("k_vol", 0.0) * (sc[L.SC_VOLUME] - opts.get("v_target", 0.0))
                g_out = g_out + coef * gc
                sc[L.SC_LAMBDA] = coef
            if opts.get("apply_fixed") and self.fixed is not None:
                g_out = np.where(np.asarray(self.fixed, bool)[:, None], 0.0, g_out)
        new = {L.ARR_E_VERTEX: out["e_vertex"], L.ARR_K_VECS: out["k_vecs"], L.ARR_A_VOR: out["a_vor"],
               L.ARR_A_EFF: out["a_eff"], L.ARR_TILT_GRAD: out["tilt_grad"]}
        if opts.get("want_grad", True) or tilt_only:  # an energy-only evaluation leaves the gradients alone
            new.update({L.ARR_GRAD: g_out, L.ARR_VOLGRAD: gc})
        self.arrays.update(new)
        self.scalars = sc.copy()
        if grad is not None:
            grad[:] = g_out
        if volgrad is not None:
            volgrad[:] = gc
        if tilt_grad is not None:
            tilt_grad[:] = out["tilt_grad"]
        return EvalResult(sc)

    def download(self, which):
        return np.array(self.arrays[which])

    def upload(self, which, host):
        self.arrays[which] = np.array(host, dtype=np.float64)

    def device_view(self, which):
        return self.arrays[which]  # writes land in the array, as through ms_ctx_device_ptr

    def read_scalars(self):
        return EvalResult(self.scalars.copy())

    def sync(self):
        pass

    # positions, trial positions and search direction live in ``arrays`` like the other named arrays
    pos = property(lambda self: self.arrays[L.ARR_POSITIONS],
                   lambda self, v: self.arrays.__setitem__(L.ARR_POSITIONS, v))
    trial = property(lambda self: self.arrays[L.ARR_TRIAL], lambda self, v: self.arrays.__setitem__(L.ARR_TRIAL, v))
    dir = property(lambda self: self.arrays[L.ARR_DIRECTION],
                   lambda self, v: self.arrays.__setitem__(L.ARR_DIRECTION, v))

    # -- leaflet modules (emulated ms_leaflet.cuh bodies) --
    def set_leaflet(self, leaflet, **desc):
        self.__dict__.setdefault("leaflets", {})[int(leaflet)] = desc
        self.leaflet_uploads = getattr(self, "leaflet_uploads", 0) + 1

    # -- tilt relaxation primitives: numpy restatements of the small kernels (TEST ONLY) --
    def set_leaflet_fixed(self, leaflet, fixed_rows):
        self.__dict__.setdefault("leaflet_fixed", {})[int(leaflet)] = (
            None if fixed_rows is None else np.asarray(fixed_rows, bool))

    def update_vertex_normals(self):
        p, t = self.pos, self.tri
        n = np.cross(p[t[:, 1]] - p[t[:, 0]], p[t[:, 2]] - p[t[:, 0]])
        out = np.zeros_like(p)
        for k in range(3):
            np.add.at(out, t[:, k], n)
        mag = np.linalg.norm(out, axis=1)
        ok = mag >= 1e-12
        out[ok] /= mag[ok][:, None]
        self.vnormals = out

    def _lf_arrays(self, leaflet):
        if leaflet == L.LEAFLET_IN:
            return L.ARR_TILTS_IN, L.ARR_TILT_GRAD_IN
        return L.ARR_TILTS_OUT, L.ARR_TILT_GRAD_OUT

    def leaflet_project_tilts(self, leaflet):
        a, _ = self._lf_arrays(leaflet)
        t = self.arrays[a]
        self.arrays[a] = t - (t * self.vnormals).sum(axis=1)[:, None] * self.vnormals

    def leaflet_gradient_norm2(self, leaflet, read=True):
        _, g = self._lf_arrays(leaflet)
        fx = getattr(self, "leaflet_fixed", {}).get(int(leaflet))
        if fx is not None:
            self.arrays[g][fx] = 0.0
        val = float((self.arrays[g] ** 2).sum())
        self.__dict__.setdefault("lf_results", np.zeros((3, 5)))[int(leaflet), 3] = val
        return val if read else None

    def leaflet_build_preconditioner(self, leaflet, k_smooth, kept_facets_only):
        from oracle import ref_leaflet as rl

        d = self.leaflets[int(leaflet)]
        keep = d.get("facet_keep")
        fx = getattr(self, "leaflet_fixed", {}).get(int(leaflet))
        fx = np.zeros(self.nv, bool) if fx is None else fx
        self.__dict__.setdefault("leaflet_minv", {})[int(leaflet)] = rl.leaflet_jacobi_inverse(
            self.pos, self.tri, area_facets=(np.asarray(keep, bool) if (kept_facets_only and keep is not None) else None),
            k_tilt=d.get("k_tilt", 0.0), k_smooth=k_smooth, fixed=fx)

    def _minv(self, leaflet, preconditioned):
        return self.leaflet_minv[int(leaflet)][:, None] if preconditioned else 1.0

    def leaflet_rz(self, leaflet, preconditioned, read=True):
        _, g = self._lf_arrays(leaflet)
        val = float((self.arrays[g] ** 2 * self._minv(leaflet, preconditioned)).sum())
        self.__dict__.setdefault("lf_results", np.zeros((3, 5)))[int(leaflet), 4] = val
        return val if read else None

    def leaflet_cg_direction(self, leaflet, beta, restart, preconditioned):
        _, g = self._lf_arrays(leaflet)
        z = -self.arrays[g] * self._minv(leaflet, preconditioned)
        dirs = self.__dict__.setdefault("leaflet_dir", {})
        dirs[int(leaflet)] = z if restart else z + beta * dirs[int(leaflet)]

    def leaflet_make_trial(self, leaflet, step, along_direction=False):
        a, g = self._lf_arrays(leaflet)
        t = self.arrays[a]
        y = t + step * self.leaflet_dir[int(leaflet)] if along_direction else t - step * self.arrays[g]
        y = y - (y * self.vnormals).sum(axis=1)[:, None] * self.vnormals
        fx = getattr(self, "leaflet_fixed", {}).get(int(leaflet))
        if fx is not None:
            y[fx] = t[fx]
        self.__dict__.setdefault("leaflet_trial", {})[int(leaflet)] = y

    def leaflet_swap_trial(self, leaflet):
        a, _ = self._lf_arrays(leaflet)
        self.arrays[a], self.leaflet_trial[int(leaflet)] = self.leaflet_trial[int(leaflet)], self.arrays[a]

    def eval_leaflet_pair(self, modules, *, want_grad=False, want_tilt_grad=True, accumulate=0, use_trial=False):
        self.eval_leaflet(L.LEAFLET_IN, modules, want_grad=want_grad, want_tilt_grad=want_tilt_grad, accumulate=accumulate,
                          use_trial=use_trial, read=False)
        self.eval_leaflet(L.LEAFLET_OUT, modules, want_grad=want_grad, want_tilt_grad=want_tilt_grad,
                          accumulate=accumulate | (L.ACC_GRAD if want_grad else 0), use_trial=use_trial, read=False)

    def leaflet_results(self):
        return np.array(self.__dict__.setdefault("lf_results", np.zeros((3, 5))))

    def eval_leaflet(self, leaflet, modules, *, want_grad=True, want_tilt_grad=True, accumulate=0, use_trial=False,
                     read=True):
        if int(leaflet) not in getattr(self, "leaflets", {}):
            raise L.B200Error("ms_ctx_set_leaflet has not been called for this leaflet")
        d = self.leaflets[int(leaflet)]
        arr_t = {L.LEAFLET_IN: L.ARR_TILTS_IN, L.LEAFLET_OUT: L.ARR_TILTS_OUT, L.LEAFLET_FIELD: L.ARR_TILTS_FIELD}[leaflet]
        arr_g = {L.LEAFLET_IN: L.ARR_TILT_GRAD_IN, L.LEAFLET_OUT: L.ARR_TILT_GRAD_OUT,
                 L.LEAFLET_FIELD: L.ARR_TILT_GRAD_FIELD}[leaflet]
        k, c = d.get("kappa", 0.0), d.get("c0", 0.0)
        r = H.emulate_leaflet(self.trial if use_trial else self.pos, self.tri, self.arrays[arr_t], sign=d["div_sign"],
                              keep=d.get("facet_keep"), is_boundary=self.is_boundary, interior=d.get("interior"),
                              base_zero=d.get("base_zero"), kappa=k if np.ndim(k) else None,
                              kappa_u=0.0 if np.ndim(k) else float(k), c0=c if np.ndim(c) else None,
                              c0_u=0.0 if np.ndim(c) else float(c), row_weight=d.get("tilt_row_weight"),
                              consistent=d.get("facet_consistent"), consistent_u=d.get("consistent", False),
                              k_tilt=d.get("k_tilt", 0.0), k_smooth=d.get("k_smooth", 0.0),
                              with_bt=bool(modules & L.MOD_BENDING_TILT), with_tilt=bool(modules & L.MOD_TILT),
                              with_smooth=bool(modules & L.MOD_TILT_SMOOTHNESS), want_grad=want_grad,
                              want_tilt_grad=want_tilt_grad)
        self.evals += 1
        if want_grad:
            self.arrays[L.ARR_GRAD] = r["grad"] + (self.arrays[L.ARR_GRAD] if accumulate & L.ACC_GRAD else 0.0)
        if want_tilt_grad:
            self.arrays[arr_g] = r["tilt_grad"] + (self.arrays[arr_g] if accumulate & L.ACC_TILT_GRAD else 0.0)
        self.__dict__.setdefault("lf_results", np.zeros((3, 5)))[int(leaflet), :3] = (r["E_bt"], r["E_tilt"], r["E_smooth"])
        return (r["E_bt"], r["E_tilt"], r["E_smooth"]) if read else None

    # -- device-resident loop (numpy restatement of the small kernels; TEST ONLY) --
    def set_positions(self, pos):
        self.pos = np.array(pos, dtype=np.float64)

    def set_direction(self, d):
        self.dir = np.array(d, dtype=np.float64)

    def eval(self, opts):
        p = self.trial if opts.get("use_trial") else self.pos
        return self.eval_host(opts, p)

    def direction_from_gradient(self, scale=-1.0):
        self.dir = scale * self.arrays[L.ARR_GRAD]

    def axpy(self, dst, src, alpha, skip_fixed=True):
        upd = alpha * self.arrays[src]
        if skip_fixed and self.fixed is not None:
            upd[np.asarray(self.fixed, bool)] = 0.0
        self.arrays[dst] = self.arrays[dst] + upd

    def dots(self):
        g, gc = self.arrays[L.ARR_GRAD], self.arrays[L.ARR_VOLGRAD]
        sc = self.scalars
        sc[L.SC_G_G], sc[L.SC_G_GC], sc[L.SC_GC_GC] = (g * g).sum(), (g * gc).sum(), (gc * gc).sum()

    def cg_direction(self, restart):
        g = self.arrays[L.ARR_GRAD]
        if restart or self._pg is None:
            self.dir = -g
            return
        beta = np.einsum("ij,ij->i", g, g - self._pg) / (np.einsum("ij,ij->i", self._pg, self._pg) + 1e-20)
        d = -g + beta[:, None] * self._pd
        d[beta < 0] = -g[beta < 0]
        if self.fixed is not None:
            d[np.asarray(self.fixed, bool)] = 0.0
        self.dir = d

    def cg_commit(self):
        self._pg, self._pd = self.arrays[L.ARR_GRAD].copy(), self.dir.copy()

    def make_trial(self, alpha):
        self.trial = self.pos + alpha * self.dir

    def accept_trial(self):
        self.pos = self.trial.copy()

    def line_search_stats(self):
        t, p = self.tri, self.pos
        e = np.concatenate([p[t[:, 2]] - p[t[:, 1]], p[t[:, 0]] - p[t[:, 2]], p[t[:, 1]] - p[t[:, 0]]])
        g = self.arrays[L.ARR_GRAD]
        min_edge = float(np.sqrt((e * e).sum(axis=1).min())) if self.nf else 0.0
        return (min_edge, float(np.sqrt((self.dir**2).sum(axis=1).max())),
                float((g * self.dir).sum()), float((g * g).sum()))

    def normal_change_ok(self, limit=0.5):
        # the rule of ms_ctx_normal_change_ok (include/ms_b200.h)
        if not (0.0 <= limit <= np.pi):
            raise L.B200Error("limit_radians must lie in [0, pi]")
        t = self.tri
        def normals(p):
            return np.cross(p[t[:, 1]] - p[t[:, 0]], p[t[:, 2]] - p[t[:, 0]])
        n0, n1 = normals(self.pos), normals(self.trial)
        m0, m1 = np.linalg.norm(n0, axis=1), np.linalg.norm(n1, axis=1)
        good = m0 > 1e-12
        with np.errstate(invalid="ignore", divide="ignore"):
            d = np.clip((n0[good] * n1[good]).sum(axis=1) / (m0[good] * m1[good]), -1.0, 1.0)  # NaN stays NaN
            bad = (m1[good] < 1e-12) | ~(d >= np.cos(limit))
        return not bool(bad.any())

    def close(self):
        pass
