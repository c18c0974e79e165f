"""The partitioned evaluation ``ms_ctx_eval_partition`` with several ranks on ONE GPU, against the whole-mesh float64
reference assembled from ``oracle/ref_modules.py``.

Every rank is a context of this process with its own stream; the contexts are wired to each other with device
pointers (``ms_ctx_peer_set_pointer``) instead of CUDA IPC handles, so the kernels are the ones the multi-process path
runs.  Each scenario runs on each rank layout in every launch form, on the same contexts and in one sequence, so the
flag epochs, the all-reduce slot parity and the host mirror of the in-kernel arrival counter carry across forms:

* ``unfused``: signal + pull, pass A, seed pull, pass B, reduce, all-reduce, project (10 launches);
* ``fused``: bit 0 -- the exchange folded into the compute launches (5 launches);
* ``in_kernel``: bits 0|1 -- the exchange inside the patch kernels (``ms::HaloPull``): interior patches first, the
  epilogue warps pull the ghost rows, the producer waits for every CTA's slice before its first patch that reads
  them, the last CTA of the last pass publishes and gathers the scalars;
* ``seeds_only``: bit 1 alone -- the caller places the ghost positions, the seeds travel inside the kernels;
* ``no_exchange``: no bit -- the caller places the ghost positions, the seeds travel with the fused pull;
* ``push``: ``ms_ctx_set_push_targets`` -- owners store into the neighbours' ghost slots, the receivers' patch kernels
  wait on local words (``attach_wait``), ``k_halo_push`` and ``k_allreduce_local_coef``;
* ``narrow``: a pack of 32-lane rounds with the in-kernel form requested, which falls back to the fused pull.

Before every evaluation the ghost rows of the positions and trial positions (owned rows stay valid) and every row of
the seeds, gradient, dV/dx and tilt gradient are filled with NaN, so a row an exchange misses shows up.

CPU tier: the same partitions and scenarios through the host emulator (pass A per rank, the ghost seed rows handed
over in NumPy, pass B per rank), summed over the ranks and compared with the whole-mesh reference; and the push
tables, which must cover every ghost row of every rank exactly once."""

import ctypes
import functools
from dataclasses import dataclass

import numpy as np
import pytest

import ms_test_helpers as H
from membrane_solver_b200 import _lib as L
from membrane_solver_b200.partition import ghost_sources, push_targets, send_lists, split_mesh, vertex_cuts
from membrane_solver_b200.synthetic import icosphere, open_sheet, tangent_tilts
from ms_test_helpers import rel_err, volgrad_close
from oracle import ref_modules as ref

S, V, B, T, BT = L.MOD_SURFACE, L.MOD_VOLUME, L.MOD_BENDING, L.MOD_TILT, L.MOD_BENDING_TILT
TOL = 1e-12
GAMMA_U, KAPPA_U, C0_U, K_TILT = 1.2, 1.3, 0.05, 0.7
K_VOL, ALPHA = 3.0, 0.37
NARROW = dict(threads=32, max_owned=64, max_local=200)
TINY_RANK = 40                   # owned vertices of the small rank of the uneven layout: fewer than one patch holds


# ---- meshes ------------------------------------------------------------------------------------------------------
@dataclass
class Mesh:
    pos: np.ndarray
    tri: np.ndarray
    is_b: np.ndarray | None      # boundary flags (None: closed)
    gamma: np.ndarray            # per-facet surface tension
    kappa: np.ndarray            # per-vertex bending parameters
    c0: np.ndarray
    tilts: np.ndarray
    body: np.ndarray             # partial body (facet mask)
    fixed: np.ndarray            # fixed vertices
    direction: np.ndarray        # search direction of the trial positions x + ALPHA d


@functools.lru_cache(maxsize=None)
def mesh(name, gpu):
    """``gpu``: the GPU tier's size; the emulator runs the icosphere at a third of it."""
    is_b, flat = None, False
    if name == "ico":             # 151 380 facets (50 000 in the CPU tier), closed, space-filling-curve order
        pos, tri = icosphere(87 if gpu else 50)
    elif name == "icoperm":       # 40 500 facets in random vertex order: contiguous cuts give ragged ranks
        pos0, tri0 = icosphere(45, reorder=False)
        old_of_new = np.random.default_rng(11).permutation(len(pos0))
        new_of_old = np.empty_like(old_of_new)
        new_of_old[old_of_new] = np.arange(len(pos0))
        pos, tri = np.ascontiguousarray(pos0[old_of_new]), new_of_old[tri0].astype(np.int32)
    elif name == "sheet":         # 30 000 facets with a boundary
        pos, tri = open_sheet(150, 100, jitter=0.05)
    elif name == "flat":          # 21 600 facets, z = 0: every interior vertex takes the |K| = 0 normal fallback
        pos, tri = open_sheet(120, 90)
        flat = True
    elif name == "small":         # 5 120 facets: the refusals
        pos, tri = icosphere(16)
    else:
        raise KeyError(name)
    if name in ("sheet", "flat"):
        is_b = ref.boundary_mask_from_triangles(tri, len(pos))
    nv, nf = len(pos), len(tri)
    rng = np.random.default_rng(nf)
    h = float(np.sqrt(ref.triangle_areas(pos, tri).mean()))
    direction = 0.05 * h * rng.normal(size=pos.shape)
    if flat:
        # the trial positions are the unit grid itself: moved in the plane, |K|^2 of an interior vertex is rounding noise
        # around the 1e-30 threshold of the normal fallback, and which branch a vertex takes would depend on the
        # summation order.  The trial array still has to come through the halo.
        direction[:] = 0.0
    return Mesh(pos=pos, tri=np.ascontiguousarray(tri, dtype=np.int32), is_b=is_b,
                gamma=1.0 + 0.3 * rng.random(nf), kappa=1.0 + 0.3 * rng.random(nv), c0=0.1 * rng.random(nv) - 0.05,
                tilts=tangent_tilts(pos, tri), body=(rng.random(nf) < 0.6).astype(np.uint8),
                fixed=(rng.random(nv) < 0.05).astype(np.uint8), direction=direction)


# ---- rank layouts ------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Layout:
    name: str
    mesh: str
    world: int
    uneven: bool = False

    def cuts(self, nv):
        if not self.uneven:
            return vertex_cuts(nv, self.world)
        # ranks 0 and 3 a seventh each, rank 1 TINY_RANK vertices (one patch, grid 1), rank 2 five times larger than
        # ranks 0 and 3; rank 1 is so thin that facets reach from rank 0 across it into rank 2
        a = nv // 7
        return np.array([0, a, a + TINY_RANK, nv - nv // 7, nv], dtype=np.int64)


LAYOUTS = {lay.name: lay for lay in [
    Layout("ico_w2", "ico", 2), Layout("ico_w3", "ico", 3), Layout("ico_w5", "ico", 5), Layout("ico_w8", "ico", 8),
    Layout("ico_uneven", "ico", 4, uneven=True),
    Layout("icoperm_w3", "icoperm", 3),          # every patch of every rank reads ghost rows
    Layout("sheet_w3", "sheet", 3),              # cut across the boundary
    Layout("flat_w3", "flat", 3),
]}


def parts_of(layout, gpu):
    m = mesh(layout.mesh, gpu)
    cuts = layout.cuts(len(m.pos))
    return [split_mesh(len(m.pos), m.tri, layout.world, r, cuts) for r in range(layout.world)]


def facets_over_three_ranks(layout, gpu):
    m = mesh(layout.mesh, gpu)
    cuts = layout.cuts(len(m.pos))
    owner = np.searchsorted(cuts, m.tri, side="right") - 1
    return int(np.count_nonzero((owner[:, 0] != owner[:, 1]) & (owner[:, 1] != owner[:, 2])
                                & (owner[:, 0] != owner[:, 2])))


# ---- scenarios ---------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Scenario:
    name: str
    modules: int
    flags: int = 0
    facet_gamma: bool = False
    vertex_bending: bool = False  # per-vertex kappa / c0 (else uniform, c0 = C0_U != 0)
    want_grad: bool = True
    constraint_mode: int = -1
    partial_body: bool = False
    fixed: bool = False           # fixed mask + apply_fixed

    @property
    def projected(self):
        return self.want_grad and (self.constraint_mode >= 0 or self.fixed)

    @property
    def bending(self):
        return bool(self.modules & B)

    @property
    def seeds_travel(self):
        return self.bending and self.want_grad


CLOSED = [
    Scenario("sbv", S | B | V),
    Scenario("sbv_energy", S | B | V, want_grad=False),
    Scenario("sbv_lagrange", S | B | V, constraint_mode=0),
    Scenario("sbv_penalty_fixed", S | B | V, constraint_mode=1, partial_body=True, fixed=True),
    Scenario("sv", S | V),                       # no bending: pass B is the first kernel and pulls the positions
    Scenario("s", S),
    Scenario("v", V),
    Scenario("sv_energy", S | V, want_grad=False),   # pass A alone publishes and gathers
    Scenario("k3_sbv_vertex_facet", S | B | V, facet_gamma=True, vertex_bending=True),
    Scenario("k0_svt_facet", S | V | T, facet_gamma=True),
]
BOUNDED = [
    Scenario("willmore", B, flags=L.FLAG_WILLMORE),
    Scenario("approx", B, flags=L.FLAG_APPROX),
    Scenario("sb", S | B),
    Scenario("s", S),
]
FLAT = [
    Scenario("sb", S | B),
    Scenario("b_vertex", B, vertex_bending=True),
]
SCENARIOS_OF = {"ico": CLOSED, "icoperm": CLOSED, "sheet": BOUNDED, "flat": FLAT}
CASES = {f"{lay.name}-{sc.name}": (lay, sc) for lay in LAYOUTS.values() for sc in SCENARIOS_OF[lay.mesh]}
CASE_IDS = list(CASES)


# ---- the float64 reference ---------------------------------------------------------------------------------------
def inputs(m, sc, trial):
    nv, nf = len(m.pos), len(m.tri)
    return dict(pos=m.pos + ALPHA * m.direction if trial else m.pos,
                is_b=m.is_b if m.is_b is not None else np.zeros(nv, bool),
                gamma=m.gamma if sc.facet_gamma else np.full(nf, GAMMA_U),
                kappa=m.kappa if sc.vertex_bending else KAPPA_U, c0=m.c0 if sc.vertex_bending else C0_U,
                body=m.body if sc.partial_body else np.ones(nf, np.uint8))


def v_target(m, sc):
    """Penalty target: 3 % below the body volume at the positions."""
    x = inputs(m, sc, False)
    return 0.97 * ref.body_volume(m.pos, m.tri[x["body"].astype(bool)])


@functools.lru_cache(maxsize=None)
def reference(mesh_name, gpu, sc, trial):
    m = mesh(mesh_name, gpu)
    x = inputs(m, sc, trial)
    pos, tri, is_b = x["pos"], m.tri, x["is_b"]
    g, tg = np.zeros_like(pos), np.zeros_like(pos)
    out = {}
    if sc.modules & S:
        out["E_surface"] = ref.surface_energy_and_gradient(pos, tri, x["gamma"], g)
        out["area"] = float(ref.triangle_areas(pos, tri).sum())
    if sc.modules & B:
        model = "willmore" if sc.flags & L.FLAG_WILLMORE else "helfrich"
        mode = "approx" if sc.flags & L.FLAG_APPROX else "analytic"
        out["E_bending"] = ref.bending_energy_and_gradient(pos, tri, x["kappa"], x["c0"], is_b, g, model, mode)
    if sc.modules & T:
        out["E_tilt"] = ref.tilt_energy_and_gradient(pos, tri, m.tilts, K_TILT, g, tg)
        out["tilt_grad"] = tg
    out["grad"] = g
    if sc.modules & V:
        tb = tri[x["body"].astype(bool)]
        out["volume"] = ref.body_volume(pos, tb)
        out["vol_grad"] = np.zeros_like(pos)
        ref.accumulate_volume_gradient(pos, tb, out["vol_grad"], 1.0)
    if sc.projected:
        p = g.copy()
        if sc.constraint_mode == 0:
            vg = out["vol_grad"]
            coef = -float(np.vdot(g, vg) / np.vdot(vg, vg))
            out["lambda"] = -coef
            out["lambda_scale"] = float(np.sqrt(np.vdot(g, g) / np.vdot(vg, vg)))
        elif sc.constraint_mode == 1:
            coef = K_VOL * (out["volume"] - v_target(m, sc))
            out["lambda"] = coef
            out["lambda_scale"] = K_VOL * out["volume"]
        if sc.constraint_mode >= 0:
            p += coef * out["vol_grad"]
        if sc.fixed:
            p[m.fixed.astype(bool)] = 0.0
        out["projected"] = p
    return out


SCALAR_NAMES = (("E_surface", L.SC_E_SURFACE), ("area", L.SC_AREA), ("volume", L.SC_VOLUME),
                ("E_bending", L.SC_E_BENDING), ("E_tilt", L.SC_E_TILT))


def grad_tol(sc):
    return 2e-12 if sc.bending else TOL


def check_against_reference(m, sc, trial, want, scalars, arrays, what):
    """``arrays``: the owned rows of every rank, concatenated (the cuts are contiguous: global row order)."""
    for name, slot in SCALAR_NAMES:
        if name in want:
            got = float(scalars[slot])
            assert abs(got - want[name]) <= TOL * max(1.0, abs(want[name])), (what, name, got, want[name])
    if not sc.want_grad:
        return
    grad = arrays["grad"].copy()
    if sc.flags & L.FLAG_APPROX:
        grad[m.is_b] = 0.0        # bending.py: the host module zeroes the boundary rows in approx mode
    assert rel_err(grad, want["grad"]) <= grad_tol(sc), (what, rel_err(grad, want["grad"]))
    if sc.modules & V:
        volgrad_close(arrays["vol_grad"], want["vol_grad"], inputs(m, sc, trial)["pos"])
    if sc.modules & T:
        assert rel_err(arrays["tilt_grad"], want["tilt_grad"]) <= TOL, what
    if "projected" in arrays:
        assert rel_err(arrays["projected"], want["projected"]) <= grad_tol(sc), (what, "projected")
        if "lambda" in want:
            got = float(scalars[L.SC_LAMBDA])
            assert abs(got - want["lambda"]) <= TOL * want["lambda_scale"], (what, "lambda", got, want["lambda"])


# ---- CPU tier ----------------------------------------------------------------------------------------------------
def test_layouts_have_their_edge_cases():
    """The uneven cut really has facets over three ranks and a rank several times larger than the others."""
    lay = LAYOUTS["ico_uneven"]
    assert facets_over_three_ranks(lay, True) > 0 and facets_over_three_ranks(lay, False) > 0
    for gpu in (False, True):
        owned = [p.n_owned for p in parts_of(lay, gpu)]
        assert owned[1] == TINY_RANK and owned[2] >= 4 * max(owned[0], owned[3]), owned
    assert facets_over_three_ranks(LAYOUTS["ico_w8"], True) > 0


@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_push_tables_cover_every_ghost_row_once(layout):
    """``push_targets`` (what ``PartitionedMesh`` hands to ``ms_ctx_set_push_targets``): over all sources, every ghost
    row of every rank is written exactly once, with the row of the vertex it stands for."""
    lay = LAYOUTS[layout]
    for gpu in (False, True):
        parts = parts_of(lay, gpu)
        table = [(p.n_owned, p.recv_blocks) for p in parts]
        ghosts = [p.ghost_ids for p in parts]
        written = [np.zeros(p.nv_local - p.n_owned, np.int64) for p in parts]
        for src in parts:
            slots, rows, dst_rows = push_targets(src, send_lists(src, ghosts), table)
            assert not np.any(slots == src.rank)
            assert np.all(rows < src.n_owned)
            for d in np.unique(slots):
                sel = slots == d
                dst = parts[int(d)]
                k = dst_rows[sel] - dst.n_owned
                assert np.all(k >= 0) and np.all(k < dst.ghost_ids.size)
                np.add.at(written[int(d)], k, 1)
                assert np.array_equal(dst.ghost_ids[k], src.lo + rows[sel])
        for w in written:
            assert np.all(w == 1)


def _emulate_rank(m, sc, loc, pos, phase, seeds=None, **pack):
    rows = loc.global_rows()
    x = inputs(m, sc, False)
    return H.emulate(pos[rows], loc.tri, modules=sc.modules, flags=sc.flags, want_grad=sc.want_grad,
                     is_boundary=None if m.is_b is None else m.is_b[rows], body_mask=x["body"][loc.facet_ids],
                     tilts=m.tilts[rows] if sc.modules & T else None,
                     gamma=m.gamma[loc.facet_ids] if sc.facet_gamma else None, gamma_u=GAMMA_U,
                     kappa=m.kappa[rows] if sc.vertex_bending else None, c0=m.c0[rows] if sc.vertex_bending else None,
                     kappa_u=KAPPA_U, c0_u=C0_U, k_tilt=K_TILT, n_owned=loc.n_owned, phase=phase, seeds=seeds, **pack)


@pytest.mark.parametrize("case", CASE_IDS)
def test_emulated_partition_matches_reference(case):
    lay, sc = CASES[case]
    m = mesh(lay.mesh, False)
    parts = parts_of(lay, False)
    for trial in (False, True):
        pos = inputs(m, sc, trial)["pos"]
        a_out = [None] * len(parts)
        if sc.bending or not sc.want_grad:                 # pass A per rank
            a_out = [_emulate_rank(m, sc, loc, pos, 1) for loc in parts]
        if lay.uneven:                                     # the small rank is a single patch
            assert _emulate_rank(m, sc, parts[1], pos, 1)["pack"]["n_patches"] == 1
        b_out = [None] * len(parts)
        if sc.want_grad:                                   # ghost seed rows from their owners, then pass B per rank
            for r, loc in enumerate(parts):
                seeds = None
                if sc.bending:
                    seeds = a_out[r]["seeds"].copy()
                    seeds[loc.n_owned:] = np.nan
                    owners, rows = ghost_sources(loc)
                    for o in np.unique(owners):
                        sel = owners == o
                        seeds[loc.n_owned + np.nonzero(sel)[0]] = a_out[int(o)]["seeds"][rows[sel]]
                b_out[r] = _emulate_rank(m, sc, loc, pos, 2, seeds=seeds)
        total = np.zeros(L.SC_COUNT)
        for r in range(len(parts)):                        # primary-facet sums, added in rank order
            src = b_out[r] if sc.want_grad and not sc.bending else a_out[r]
            for name, slot in SCALAR_NAMES:
                # with bending, pass A has every sum but the tilt energy, which pass B makes
                total[slot] += b_out[r][name] if name == "E_tilt" and sc.want_grad else src[name]
        arrays = {}
        if sc.want_grad:
            for key, out_key in (("grad", "grad"), ("vol_grad", "volgrad"), ("tilt_grad", "tilt_grad")):
                arrays[key] = np.concatenate([b[out_key][:loc.n_owned] for b, loc in zip(b_out, parts)])
                assert np.all(np.isfinite(arrays[key])), key
        want = reference(lay.mesh, False, sc, trial)
        check_against_reference(m, sc, trial, want, total, arrays, f"emulated trial={trial}")


# ---- GPU tier ----------------------------------------------------------------------------------------------------
FORM_FLAGS = {"fused": 1, "in_kernel": 3, "seeds_only": 2, "no_exchange": 0, "push": 1, "narrow": 3}
PULL_FORMS = ["unfused", "fused", "in_kernel", "seeds_only", "no_exchange"]


def _options(dm, m, sc, trial, raw=False):
    return dm.options(sc.modules, flags=sc.flags, want_grad=sc.want_grad, use_trial=trial,
                      constraint_mode=-1 if raw else sc.constraint_mode, k_vol=K_VOL,
                      v_target=v_target(m, sc) if sc.constraint_mode == 1 else 0.0, apply_fixed=sc.fixed and not raw)


def _sms():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


def cap_sets(world):
    """Grid caps 1, 2, 7 and SMs / W for every rank, then the four mixed over the ranks.  Every rank's persistent
    kernel must be resident at once (a rank waits inside its kernel for the others): the caps add up to <= SMs."""
    sms = _sms()
    caps = [1, 2, 7, sms // world]
    out = [[c] * world for c in caps] + [[caps[r % 4] for r in range(world)]]
    for cs in out:
        assert sum(cs) <= sms, (cs, sms)
    return out


class Rig:
    """W contexts of one partitioned mesh on GPU 0, each on its own stream, wired over device pointers."""

    def __init__(self, lay, sc, pack=None):
        import torch

        from membrane_solver_b200.context import DeviceMesh

        if L.device_count() < 1:
            pytest.fail("no CUDA device visible: the gpu tier must run on the B200 box")
        self.torch, self.lib, self.lay, self.sc = torch, L.lib(), lay, sc
        self.m = m = mesh(lay.mesh, True)
        self.parts = parts_of(lay, True)
        body = inputs(m, sc, False)["body"]
        self.dms, self.streams = [], []
        for loc in self.parts:
            rows = loc.global_rows()
            dm = DeviceMesh(0, **(pack or {}))
            self.dms.append(dm)
            dm.set_topology(loc.nv_local, loc.tri, n_owned=loc.n_owned,
                            is_boundary=None if m.is_b is None else m.is_b[rows], body_mask=body[loc.facet_ids],
                            fixed_mask=m.fixed[rows] if sc.fixed else None)
            dm.set_surface_tension(m.gamma[loc.facet_ids] if sc.facet_gamma else GAMMA_U)
            dm.set_bending_params(m.kappa[rows] if sc.vertex_bending else KAPPA_U,
                                  m.c0[rows] if sc.vertex_bending else C0_U)
            dm.set_tilt_rigidity(K_TILT)
            dm.set_positions(m.pos[rows])
            if sc.modules & T:
                dm.set_tilts(m.tilts[rows])        # the halo does not carry tilts: the ghost rows are uploaded
            dm.set_direction(m.direction[rows])
            dm.make_trial(ALPHA)
            dm.sync()
            stream = torch.cuda.Stream()
            L.check(self.lib.ms_ctx_set_stream(dm._h, stream.cuda_stream))
            self.streams.append(stream)
        torch.cuda.synchronize()
        # the owners' rows as the devices hold them: what a ghost row must equal after an exchange
        self.owned = {w: [dm.download(w)[:loc.n_owned].copy() for dm, loc in zip(self.dms, self.parts)]
                      for w in (L.ARR_POSITIONS, L.ARR_TRIAL)}
        world = lay.world
        for r, (loc, dm) in enumerate(zip(self.parts, self.dms)):
            owners, rows = ghost_sources(loc)
            for o in np.unique(owners):          # the owners of this rank's ghosts, as PartitionedMesh opens them
                for w in (L.ARR_POSITIONS, L.ARR_TRIAL, L.ARR_SEEDS):
                    dm.peer_set_pointer(int(o), w, self.dms[int(o)].device_ptr(w))
            for o in range(world):
                if o != r:
                    dm.peer_set_pointer(o, L.IPC_FLAGS, self.dms[o].flag_words_ptr())
            dm.set_rank_slot(r, world)
            dm.set_ghost_sources(world, owners, rows)
        for dm in self.dms:
            dm.halo_prepare()
        torch.cuda.synchronize()

    def close(self):
        self.torch.cuda.synchronize()
        for dm in self.dms:
            L.check(self.lib.ms_ctx_set_stream(dm._h, None))
            dm.close()

    def enable_push(self):
        """Every peer's arrays opened, the push tables built as ``PartitionedMesh`` builds them."""
        world = self.lay.world
        table = [(p.n_owned, p.recv_blocks) for p in self.parts]
        ghosts = [p.ghost_ids for p in self.parts]
        for r, (loc, dm) in enumerate(zip(self.parts, self.dms)):
            for o in range(world):
                if o != r:
                    for w in (L.ARR_POSITIONS, L.ARR_TRIAL, L.ARR_SEEDS):
                        dm.peer_set_pointer(o, w, self.dms[o].device_ptr(w))
            dm.set_push_targets(*push_targets(loc, send_lists(loc, ghosts), table))
        for dm in self.dms:
            dm.halo_prepare()
        self.torch.cuda.synchronize()

    def ghost_rows_of(self, r, which):
        owners, rows = ghost_sources(self.parts[r])
        src = self.owned[which]
        out = np.empty((rows.size, 3))
        for o in np.unique(owners):
            sel = owners == o
            out[sel] = src[int(o)][rows[sel]]
        return out

    def _upload_rows(self, dm, which, first_row, values):
        a = np.ascontiguousarray(values, dtype=np.float64).ravel()
        w = L.ARRAY_WIDTH[which]
        L.check(self.lib.ms_ctx_upload(dm._h, which, L.dptr(a), w * first_row, a.size))
        dm.sync()

    def _poison(self, caller_places):
        for r, (dm, loc) in enumerate(zip(self.dms, self.parts)):
            ng = loc.nv_local - loc.n_owned
            if ng:
                for w in (L.ARR_POSITIONS, L.ARR_TRIAL):
                    self._upload_rows(dm, w, loc.n_owned,
                                      self.ghost_rows_of(r, w) if caller_places else np.full((ng, 3), np.nan))
            for w in (L.ARR_SEEDS, L.ARR_GRAD, L.ARR_VOLGRAD, L.ARR_TILT_GRAD):
                n = int(self.lib.ms_ctx_array_len(dm._h, w))
                if n:
                    self._upload_rows(dm, w, 0, np.full(n, np.nan))

    def _issue(self, opts, form):
        """Every rank's calls of one evaluation, then every stream synchronised."""
        sc = self.sc
        for dm in self.dms:
            if form == "unfused":                  # PartitionedMesh.eval_async without the fused transport
                dm.halo_signal(L.FLAG_POSITIONS)
                dm.halo_pull(L.ARR_TRIAL if opts.use_trial else L.ARR_POSITIONS, L.FLAG_POSITIONS)
                dm.eval_pass_a(opts)
                if sc.seeds_travel:
                    dm.halo_signal(L.FLAG_SEEDS)
                    dm.halo_pull(L.ARR_SEEDS, L.FLAG_SEEDS)
                dm.eval_pass_b(opts)
                dm.eval_reduce(opts)
                dm.allreduce_scalars(12)
                dm.eval_project(opts)
            else:
                L.check(self.lib.ms_ctx_eval_partition(dm._h, ctypes.byref(opts), FORM_FLAGS[form]))
        self.torch.cuda.synchronize()

    def evaluate(self, form, caps, trial, raw=False):
        """One evaluation; returns the rank-0 scalars and the owned rows of the outputs, concatenated over the ranks."""
        sc, m = self.sc, self.m
        what = f"{form} caps={caps} trial={trial}{' raw' if raw else ''}"
        for dm, cap in zip(self.dms, caps):
            L.check(self.lib.ms_ctx_set_max_ctas(dm._h, int(cap)))
        self._poison(form in ("seeds_only", "no_exchange"))
        self._issue(_options(self.dms[0], m, sc, trial, raw), form)
        errors = [dm.halo_error() for dm in self.dms]
        assert not any(errors), (what, "halo_error", errors)
        scalars = [dm.read_scalars().scalars for dm in self.dms]
        for r, s in enumerate(scalars):            # rank-order sum: the same bits on every rank
            assert s.tobytes() == scalars[0].tobytes(), (what, r, s, scalars[0])
        out = {"scalars": scalars[0].copy()}
        names = []
        if sc.want_grad:
            names.append(("grad", L.ARR_GRAD))
            if sc.modules & V:
                names.append(("vol_grad", L.ARR_VOLGRAD))
            if sc.modules & T:
                names.append(("tilt_grad", L.ARR_TILT_GRAD))
        if sc.bending:
            names.append(("seeds", L.ARR_SEEDS))
        full = {}
        for key, which in names:
            full[key] = [dm.download(which) for dm in self.dms]
            out[key] = np.concatenate([a[:loc.n_owned] for a, loc in zip(full[key], self.parts)])
            assert np.all(np.isfinite(out[key])), (what, key)
        # ghost rows after the evaluation: bitwise the owners' rows
        moved = L.ARR_TRIAL if trial else L.ARR_POSITIONS
        for r, (dm, loc) in enumerate(zip(self.dms, self.parts)):
            if loc.nv_local == loc.n_owned:
                continue
            ghost = dm.download(moved)[loc.n_owned:]
            assert ghost.tobytes() == np.ascontiguousarray(self.ghost_rows_of(r, moved)).tobytes(), (what, r, "ghosts")
            if sc.seeds_travel:
                owners, rows = ghost_sources(loc)
                want = np.empty((rows.size, full["seeds"][r].shape[1]))
                for o in np.unique(owners):
                    want[owners == o] = full["seeds"][int(o)][rows[owners == o]]
                assert full["seeds"][r][loc.n_owned:].tobytes() == want.tobytes(), (what, r, "ghost seeds")
        return out

    def collect(self, form, caps, trial):
        """Raw outputs; with a projection also the projected gradient (a second evaluation)."""
        if not self.sc.projected:
            got = self.evaluate(form, caps, trial)
        else:
            raw = self.evaluate(form, caps, trial, raw=True)
            got = self.evaluate(form, caps, trial)
            got["projected"] = got.pop("grad")
            got["grad"] = raw["grad"]
        want = reference(self.lay.mesh, True, self.sc, trial)
        check_against_reference(self.m, self.sc, trial, want, got["scalars"], got, f"{form} caps={caps} trial={trial}")
        return got


def _scalar_slots(sc):
    return list(range(6)) + ([L.SC_G_G, L.SC_G_GC, L.SC_GC_GC, L.SC_LAMBDA, L.SC_COEF] if sc.want_grad else [])


def assert_equivalent(sc, base, got, what, bitwise_scalars=False):
    """Raw arrays bitwise (a patch's results do not depend on which CTA runs it); scalars within 1e-13 (the per-CTA
    rows are added in another grouping); the projected gradient, whose coefficient comes from them, at 1e-12."""
    for key in ("grad", "vol_grad", "tilt_grad", "seeds"):
        if key in base:
            assert base[key].tobytes() == got[key].tobytes(), (what, key, rel_err(got[key], base[key]))
    if "projected" in base:
        assert rel_err(got["projected"], base["projected"]) <= TOL, what
    s0, s1 = base["scalars"], got["scalars"]
    for k in _scalar_slots(sc):
        if bitwise_scalars:
            assert s0[k].tobytes() == s1[k].tobytes(), (what, k, s0[k], s1[k])
            continue
        scale = abs(s0[k])
        if k == L.SC_G_GC:
            scale = max(scale, float(np.sqrt(s0[L.SC_G_G] * s0[L.SC_GC_GC])))
        if k in (L.SC_LAMBDA, L.SC_COEF) and s0[L.SC_GC_GC] > 0:
            scale = max(scale, float(np.sqrt(s0[L.SC_G_G] / s0[L.SC_GC_GC])))
        assert abs(s1[k] - s0[k]) <= 1e-13 * scale, (what, k, s0[k], s1[k])


@pytest.mark.gpu
@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_layouts_reach_the_edge_cases_on_the_device(layout):
    """What the layouts are for, as the device packs them: the random-order icosphere gives ranks with no interior
    patch (every CTA waits before its first patch), the uneven cut a rank of a single patch."""
    from membrane_solver_b200.context import DeviceMesh

    lay = LAYOUTS[layout]
    for narrow in (False, True):
        for r, loc in enumerate(parts_of(lay, True)):
            dm = DeviceMesh(0, **(NARROW if narrow else {}))
            try:
                dm.set_topology(loc.nv_local, loc.tri, n_owned=loc.n_owned)
                n = len(dm.patch_ranges()) - 1
                interior = sum(dm.halo_rows(p, 1, 0, loc.n_owned).size == 0 for p in range(n))
                if lay.mesh == "icoperm":
                    assert interior == 0, (r, n, interior)
                elif not (lay.uneven and r == 1):
                    assert 0 < interior < n, (r, n, interior)
                if lay.uneven and r == 1:
                    assert n == 1, n
            finally:
                dm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASE_IDS)
def test_partitioned_evaluation_vs_reference_in_every_form(case):
    lay, sc = CASES[case]
    sets = cap_sets(lay.world)
    rig = Rig(lay, sc)
    try:
        base = {}
        for trial in (False, True):
            for form in PULL_FORMS:
                for caps in sets:
                    got = rig.collect(form, caps, trial)
                    if trial not in base:
                        base[trial] = got
                    else:
                        assert_equivalent(sc, base[trial], got, f"{form} caps={caps} trial={trial}")
            first = rig.collect("in_kernel", sets[-1], trial)      # repeats: the same bits, scalars included
            for _ in range(2):
                assert_equivalent(sc, first, rig.collect("in_kernel", sets[-1], trial), f"repeat trial={trial}",
                                  bitwise_scalars=True)
        rig.enable_push()
        for trial in (False, True):
            for caps in sets:
                assert_equivalent(sc, base[trial], rig.collect("push", caps, trial), f"push caps={caps} trial={trial}")
    finally:
        rig.close()
    # 32-lane rounds: the in-kernel form falls back to the fused pull (threads >= 64) and must still be right
    rig = Rig(lay, sc, pack=NARROW)
    try:
        for trial in (False, True):
            first = None
            for caps in sets:
                got = rig.collect("narrow", caps, trial)
                if first is None:
                    first = got
                else:
                    assert_equivalent(sc, first, got, f"narrow caps={caps} trial={trial}")
    finally:
        rig.close()


@pytest.mark.gpu
def test_partition_refusals_launch_nothing():
    """Each refused call returns an error before it launches or advances an epoch: the lock-step evaluation that
    follows on every rank is still clean and right."""
    from membrane_solver_b200.context import DeviceMesh

    lay = Layout("small_w2", "small", 2)
    sc = Scenario("sbv", S | B | V)
    rig = Rig(lay, sc)
    lib = L.lib()
    try:
        dm0, loc0 = rig.dms[0], rig.parts[0]

        def refused(opts):
            return lib.ms_ctx_eval_partition(dm0._h, ctypes.byref(opts), 3) != 0

        assert refused(dm0.options(S | BT))                                              # bending-tilt
        assert refused(dm0.options(T, want_grad=False, want_tilt_grad=True))            # tilt-only
        for count in (0, 1, L.PATCHES_INTERIOR, L.PATCHES_BOUNDARY):                    # whole partitions only
            assert refused(dm0.options(S | B | V, patch_count=count))
        n = loc0.n_owned
        for slot, src, dst in (([0], [0], [n]), ([2], [0], [n]), ([1], [n], [n]), ([1], [0], [-1]), ([-1], [0], [n])):
            assert lib.ms_ctx_set_push_targets(dm0._h, 1, L.iptr(np.array(slot, np.int32)),
                                               L.iptr(np.array(src, np.int32)), L.iptr(np.array(dst, np.int32))) != 0
        # the same partition wired for three ranks, the third never opened
        lone = DeviceMesh(0)
        try:
            lone.set_topology(loc0.nv_local, loc0.tri, n_owned=loc0.n_owned)
            lone.set_positions(rig.m.pos[loc0.global_rows()])
            owners, rows = ghost_sources(loc0)
            for w in (L.ARR_POSITIONS, L.ARR_TRIAL, L.ARR_SEEDS):
                lone.peer_set_pointer(1, w, rig.dms[1].device_ptr(w))
            lone.peer_set_pointer(1, L.IPC_FLAGS, rig.dms[1].flag_words_ptr())
            lone.set_rank_slot(0, 3)
            lone.set_ghost_sources(3, owners, rows)
            assert lib.ms_ctx_eval_partition(lone._h, ctypes.byref(lone.options(S | B | V)), 3) != 0
        finally:
            lone.close()
        # an empty partition (equal cuts): no row, no facet, no patch
        empty = DeviceMesh(0)
        try:
            empty.set_topology(0, np.zeros((0, 3), np.int32), n_owned=0)
            empty.set_rank_slot(0, 1)
            empty.set_ghost_sources(1, np.zeros(0, np.int32), np.zeros(0, np.int32))
            assert lib.ms_ctx_eval_partition(empty._h, ctypes.byref(empty.options(S)), 1) != 0
        finally:
            empty.close()
        sets = cap_sets(lay.world)
        for form in ("in_kernel", "fused"):
            rig.collect(form, sets[-1], False)
    finally:
        rig.close()
