"""Multi-GPU evaluation of one mesh: contiguous vertex partitions with one-ring ghosts.

SURVEY.md section 8(e).  The reference has no distributed path at all; this is the
B200-native extension BASELINE.json's north_star asks for.  The mesh is ordered along
a space-filling curve (``synthetic.sfc_order``), so a contiguous vertex range is a
compact surface region.  Rank ``r`` owns the vertex rows ``[cuts[r], cuts[r+1])`` and
lists every facet touching an owned vertex; the facet's other vertices that belong to
neighbouring ranks are *ghost* rows appended after the owned rows (sorted by global id,
hence grouped by owner rank, so receives land in place without a scatter).

One evaluation on every rank::

    halo(positions)  ->  pass A  ->  halo(seeds)  ->  pass B  ->  reduce
                     ->  all-reduce(12 scalars)  ->  project (KKT with the global lambda)

The two halo exchanges move ``24`` and ``40`` bytes per ghost vertex (O(sqrt(nv/P))
ghosts per rank); the all-reduce moves 96 bytes.  Two transports for the halo:

* ``peer`` (default on GPUs): each rank opens the owners' arrays through CUDA IPC and ONE kernel of this
  library waits for the owners' epoch flags and copies the ghost rows with NVLink peer loads
  (``ms_ctx_halo_signal`` / ``ms_ctx_halo_pull``) -- no staging buffer, no send/recv launches;
* ``nccl``: ``torch.distributed`` send/recv of rows gathered by ``ms_ctx_pack_send`` (also gloo in the
  CPU tests).

The scalar all-reduce is ``torch.distributed`` in both; it also orders the next overwrite of the exported
arrays after every rank's pulls.

Only numpy is needed to build the partition (``split_mesh``), so the plan is unit
tested on the CPU; ``PartitionedMesh`` needs a GPU per rank.
"""

from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np


@dataclass
class LocalMesh:
    """The part of the global mesh one rank holds (local row numbering)."""

    rank: int
    world: int
    cuts: np.ndarray            # (world+1,) global vertex cut points
    n_owned: int
    ghost_ids: np.ndarray       # (n_ghost,) global ids of the ghost rows, ascending
    tri: np.ndarray             # (nf_local,3) int32 local rows
    facet_ids: np.ndarray       # (nf_local,) global facet rows
    recv_blocks: list = field(default_factory=list)   # [(src_rank, first_ghost, count)]

    @property
    def nv_local(self) -> int:
        return self.n_owned + int(self.ghost_ids.size)

    @property
    def lo(self) -> int:
        return int(self.cuts[self.rank])

    def global_rows(self) -> np.ndarray:
        return np.concatenate([np.arange(self.lo, self.lo + self.n_owned, dtype=np.int64),
                               self.ghost_ids.astype(np.int64)])


def vertex_cuts(nv: int, world: int) -> np.ndarray:
    """Even contiguous split of the vertex rows."""
    return np.array([(nv * r) // world for r in range(world + 1)], dtype=np.int64)


def split_mesh(nv: int, tri: np.ndarray, world: int, rank: int, cuts: np.ndarray | None = None) -> LocalMesh:
    """Local mesh of ``rank``: owned range, ghosts, facets touching the owned range."""
    cuts = vertex_cuts(nv, world) if cuts is None else np.asarray(cuts, dtype=np.int64)
    lo, hi = int(cuts[rank]), int(cuts[rank + 1])
    tri = np.asarray(tri)
    inside = (tri >= lo) & (tri < hi)
    keep = inside.any(axis=1)
    facet_ids = np.nonzero(keep)[0]
    t = tri[facet_ids].astype(np.int64)
    ins = inside[facet_ids]
    ghost_ids = np.unique(t[~ins])
    local = np.where(ins, t - lo, 0)
    if ghost_ids.size:
        local = np.where(ins, local, (hi - lo) + np.searchsorted(ghost_ids, t))
    owners = np.searchsorted(cuts, ghost_ids, side="right") - 1
    blocks = []
    for src in np.unique(owners):
        idx = np.nonzero(owners == src)[0]
        blocks.append((int(src), int(idx[0]), int(idx.size)))  # ascending ids => contiguous block
    return LocalMesh(rank=rank, world=world, cuts=cuts, n_owned=hi - lo, ghost_ids=ghost_ids,
                     tri=np.ascontiguousarray(local, dtype=np.int32), facet_ids=facet_ids,
                     recv_blocks=blocks)


def send_lists(local: LocalMesh, all_ghost_ids: list[np.ndarray]) -> list[tuple[int, np.ndarray]]:
    """Rows of ``local`` (local numbering) that each other rank holds as ghosts.

    ``all_ghost_ids[r]`` is rank r's ``ghost_ids``.  Returned in destination-rank order;
    the rows for one destination are in ascending global id, which is the order of that
    destination's receive block.
    """
    out = []
    lo, hi = local.lo, local.lo + local.n_owned
    for dst, ghosts in enumerate(all_ghost_ids):
        if dst == local.rank:
            continue
        g = np.asarray(ghosts, dtype=np.int64)
        mine = g[(g >= lo) & (g < hi)]
        if mine.size:
            out.append((dst, (mine - lo).astype(np.int32)))
    return out


def ghost_sources(local: LocalMesh) -> tuple[np.ndarray, np.ndarray]:
    """For every ghost row of ``local`` (in ghost order): the rank that owns it and its row in the owner's local
    numbering (owned rows come first there, so it is the global id minus the owner's cut)."""
    owners = np.searchsorted(local.cuts, local.ghost_ids, side="right") - 1
    rows = local.ghost_ids - local.cuts[owners]
    return owners.astype(np.int32), rows.astype(np.int32)


def push_targets(local: LocalMesh, sends: list[tuple[int, np.ndarray]], table) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """For every row of ``local`` that another rank lists as a ghost: (that rank, the row here, the row THERE), the
    arguments of ``ms_ctx_set_push_targets``.  ``sends``: ``send_lists(local, ...)``; ``table[d]``: rank d's
    ``(n_owned, recv_blocks)``.  A destination's ghosts are ordered by global id and grouped by source rank
    (``LocalMesh.recv_blocks``), and ``send_lists`` gives this rank's rows for it in the same order."""
    from . import _lib as L

    slots, src, dst = [], [], []
    for d, rows in sends:
        n_owned_d, blocks_d = table[d]
        first = [b[1] for b in blocks_d if b[0] == local.rank]
        counts = [b[2] for b in blocks_d if b[0] == local.rank]
        if len(first) != 1 or counts[0] != rows.size:
            raise L.B200Error("send list and receive block of a neighbour disagree")
        slots.append(np.full(rows.size, d, dtype=np.int32))
        src.append(rows.astype(np.int32))
        dst.append((n_owned_d + first[0] + np.arange(rows.size)).astype(np.int32))
    cat = lambda xs: np.concatenate(xs) if xs else np.zeros(0, dtype=np.int32)  # noqa: E731
    return cat(slots), cat(src), cat(dst)


class HaloExchange:
    """Exchanges the ghost rows of per-vertex arrays between ranks (torch.distributed).

    ``tensor_of(which)`` must return a 2-D torch tensor view of the whole local array
    (owned rows then ghost rows); ``pack(which, out)`` must fill ``out`` (n_send, width)
    with the rows listed in ``send_rows`` (concatenated per destination).
    """

    def __init__(self, local: LocalMesh, sends: list[tuple[int, np.ndarray]], dist, torch, device):
        self.local = local
        self.dist = dist
        self.torch = torch
        self.device = device
        self.sends = sends
        self.send_rows = (np.concatenate([rows for _, rows in sends]) if sends
                          else np.zeros(0, dtype=np.int32)).astype(np.int32)
        self.send_offsets = np.concatenate([[0], np.cumsum([rows.size for _, rows in sends])]).astype(np.int64)
        self._buffers = {}

    def _buffer(self, width: int):
        buf = self._buffers.get(width)
        if buf is None:
            buf = self.torch.empty((max(1, int(self.send_rows.size)), width), dtype=self.torch.float64,
                                   device=self.device)
            self._buffers[width] = buf
        return buf

    def exchange(self, tensor, pack) -> None:
        """Fill the ghost rows of ``tensor`` from their owners."""
        dist, local = self.dist, self.local
        width = int(tensor.shape[1])
        buf = self._buffer(width)
        pack(buf)
        ops = []
        for k, (dst, rows) in enumerate(self.sends):
            a, b = int(self.send_offsets[k]), int(self.send_offsets[k + 1])
            ops.append(dist.P2POp(dist.isend, buf[a:b], dst))
        for src, first, count in local.recv_blocks:
            a = local.n_owned + first
            ops.append(dist.P2POp(dist.irecv, tensor[a:a + count], src))
        if ops:
            for req in dist.batch_isend_irecv(ops):
                req.wait()


class PartitionedMesh:
    """One rank's share of a mesh on its GPU plus the exchange plumbing."""

    def __init__(self, local: LocalMesh, device_index: int, *, body_mask=None, is_boundary=None,
                 fixed_mask=None, pack=None, reserve_sms: int = 0, transport: str | None = None,
                 fused: bool | None = None):
        import torch
        import torch.distributed as dist

        from . import _lib as L
        from .context import DeviceMesh

        self.L = L
        self.torch = torch
        self.dist = dist
        self.local = local
        self.device = torch.device("cuda", device_index)
        self.dm = DeviceMesh(device_index, **(pack or {}))
        self.dm.set_topology(local.nv_local, local.tri, n_owned=local.n_owned, body_mask=body_mask,
                             is_boundary=is_boundary, fixed_mask=fixed_mask)
        gathered = [None] * local.world
        dist.all_gather_object(gathered, local.ghost_ids)
        sends = send_lists(local, gathered)
        self.halo = HaloExchange(local, sends, dist, torch, self.device)
        self.dm.set_send_rows(self.halo.send_rows)
        import os as _os

        want = (transport or _os.environ.get("MS_HALO", "peer")).strip().lower()
        # MS_HALO_PUSH=1: owners STORE their rows into the neighbours' ghost slots and the receivers poll local words
        # (ms_ctx_set_push_targets).  Measured on 2 x B200: 0.624 ms per step against 0.619 ms for the default, in
        # which the neighbours pull -- remote polling was not the cost, the kernel boundaries are -- so it stays opt-in
        self._want_push = _os.environ.get("MS_HALO_PUSH", "0").strip() == "1"
        # exchange inside the patch kernels, hidden behind the interior patches (ms::HaloPull); MS_HALO_INKERNEL=0:
        # separate signal + pull launches between the passes
        self.in_kernel = _os.environ.get("MS_HALO_INKERNEL", "1").strip() != "0"
        self.push = False
        self.transport = "nccl"
        if want == "peer" and local.world > 1:
            self.transport = "peer" if self._open_peers(gathered) else "nccl"
        # transport folded into the compute launches (ms_ctx_eval_partition); MS_HALO_FUSED=0 keeps the ten-launch
        # sequence (the two must agree bit for bit: bench_multi_gpu's parity block runs on whichever is active)
        if fused is None:
            fused = _os.environ.get("MS_HALO_FUSED", "1").strip() != "0"
        self.fused = bool(fused) and self.transport == "peer"
        # the context launches on the legacy default stream; torch's current stream is the
        # same stream unless the caller changed it, so kernels and NCCL calls stay ordered
        if reserve_sms > 0:
            import ctypes as _ct

            n_sm = torch.cuda.get_device_properties(self.device).multi_processor_count
            L.check(L.lib().ms_ctx_set_max_ctas(self.dm._h, max(1, n_sm - int(reserve_sms))))
        self._views = {}
        self._side_stream = torch.cuda.Stream(device=self.device)
        self._compute_stream_handle = None  # the context's own stream (legacy default stream)

    def close(self) -> None:
        """Collective: every rank closes the peer arrays it opened, the ranks meet, then the contexts go."""
        self.torch.cuda.synchronize(self.device)
        self._views.clear()
        if self.transport == "peer":
            self.dm.peer_close()
        self.dist.barrier()
        self.dm.close()

    def view(self, which: int):
        t = self._views.get(which)
        if t is None:
            t = self.torch.as_tensor(self.dm.device_view(which), device=self.device)
            self._views[which] = t
        return t

    def _open_peers(self, all_ghost_ids) -> bool:
        """Exchange the IPC handles of the position / trial / seed arrays and of the flag words and open the
        owners of this rank's ghosts.  All ranks agree on the outcome (a failure anywhere -> NCCL for all)."""
        L, dm, dist, local = self.L, self.dm, self.dist, self.local
        whiches = (L.ARR_POSITIONS, L.ARR_TRIAL, L.ARR_SEEDS, L.IPC_FLAGS)
        ok, mine, err = 1, None, ""
        try:
            mine = [dm.ipc_export(w) for w in whiches]
        except L.B200Error as exc:
            ok, err = 0, str(exc)
        table = [None] * local.world
        dist.all_gather_object(table, mine)
        layout = [None] * local.world   # every rank's owned-row count and receive blocks (push targets)
        dist.all_gather_object(layout, (int(local.n_owned), [tuple(int(x) for x in b) for b in local.recv_blocks]))
        if ok and all(t is not None for t in table):
            owners, rows = ghost_sources(local)
            try:
                for o in np.unique(owners):
                    for w, handle in zip(whiches[:3], table[int(o)][:3]):
                        dm.peer_open(int(o), w, handle)
                for r in range(local.world):      # the flag / scalar words of every rank: all-reduce over peer memory
                    if r != local.rank:
                        dm.peer_open(r, L.IPC_FLAGS, table[r][3])
                dm.set_rank_slot(local.rank, local.world)
                dm.set_ghost_sources(local.world, owners, rows)
                if self._want_push and local.world <= 16:
                    dm.set_push_targets(*self._push_targets(layout))
                    self.push = True
                dm.halo_prepare()
            except L.B200Error as exc:
                ok, err = 0, str(exc)
        else:
            ok = 0
        flag = self.torch.tensor([ok], dtype=self.torch.int32, device=self.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0 and err:
            import sys

            print(f"[ms_b200] rank {local.rank}: peer-memory halo unavailable ({err}); using NCCL send/recv",
                  file=sys.stderr)
        return int(flag.item()) == 1

    def _push_targets(self, table):
        return push_targets(self.local, self.halo.sends, table)

    def exchange(self, which: int) -> None:
        if self.transport == "peer":
            flag = self.L.FLAG_SEEDS if which == self.L.ARR_SEEDS else self.L.FLAG_POSITIONS
            self.dm.halo_signal(flag)
            self.dm.halo_pull(which, flag)
            return
        self.halo.exchange(self.view(which), lambda buf: self.dm.pack_send(which, buf.data_ptr()))

    def _with_patches(self, opts, which: int):
        o = type(opts).from_buffer_copy(opts)
        o.patch_count = which
        return o

    def _exchange_on(self, stream, which: int) -> None:
        """Halo exchange of one array on a side stream (its row gather kernel runs there too)."""
        torch, lib, dm = self.torch, self.L.lib(), self.dm
        self.L.check(lib.ms_ctx_set_stream(dm._h, stream.cuda_stream))
        try:
            with torch.cuda.stream(stream):
                self.exchange(which)
        finally:
            self.L.check(lib.ms_ctx_set_stream(dm._h, self._compute_stream_handle))

    def eval_async(self, opts, *, exchange_positions: bool = True, overlap: bool = False) -> None:
        """One distributed evaluation; results stay on the devices (scalars are global).

        With ``overlap`` the halo exchanges run on a side stream while the INTERIOR patches (those whose
        halo lies entirely in the owned rows) are computed; only the patches that read ghost rows wait.
        Measured at 2 x 10 M facets the two extra persistent-kernel tails cost more (0.766 ms) than the
        hidden exchange latency saves (0.739 ms without), so it is off by default:

            side:  halo(positions) ............ | halo(seeds) ............
            main:  pass A interior | pass A boundary | pass B interior | pass B boundary | reduce | all-reduce | project
        """
        L, dm, torch = self.L, self.dm, self.torch
        bending = bool(opts.want_grad and (opts.modules & L.MOD_BENDING))
        if not overlap or self.local.world == 1 or opts.patch_count != L.PATCHES_ALL:
            if (self.fused and opts.patch_count == L.PATCHES_ALL and not (opts.modules & L.MOD_BENDING_TILT)
                    and (opts.want_grad or not opts.want_tilt_grad)):
                dm.eval_partition(opts, exchange_positions, in_kernel=self.in_kernel and not self.push)
                return
            if exchange_positions:
                self.exchange(L.ARR_TRIAL if opts.use_trial else L.ARR_POSITIONS)
            dm.eval_pass_a(opts)
            if bending:
                self.exchange(L.ARR_SEEDS)
            dm.eval_pass_b(opts)
            dm.eval_reduce(opts)
            self._allreduce_scalars()
            dm.eval_project(opts)
            return
        main = torch.cuda.current_stream(self.device)
        side = self._side_stream
        inner, outer = self._with_patches(opts, L.PATCHES_INTERIOR), self._with_patches(opts, L.PATCHES_BOUNDARY)
        if exchange_positions:
            side.wait_stream(main)  # the previous evaluation's readers of the ghost rows are done
            self._exchange_on(side, L.ARR_TRIAL if opts.use_trial else L.ARR_POSITIONS)
        dm.eval_pass_a(inner)
        if exchange_positions:
            main.wait_stream(side)
        dm.eval_pass_a(outer)
        if bending:
            side.wait_stream(main)  # seeds of the owned boundary rows are written
            self._exchange_on(side, L.ARR_SEEDS)
        dm.eval_pass_b(inner)
        if bending:
            main.wait_stream(side)
        dm.eval_pass_b(outer)
        dm.eval_reduce(outer)
        self._allreduce_scalars()
        dm.eval_project(opts)

    def _allreduce_scalars(self) -> None:
        """Global sums of the 12 evaluation scalars: one kernel pair over peer memory (rank-order sum, bitwise the
        same on every rank) with the peer transport, ``torch.distributed`` otherwise."""
        if self.transport == "peer":
            self.dm.allreduce_scalars(12)
            return
        sc = self.view(self.L.ARR_SCALARS)
        self.dist.all_reduce(sc[:12], op=self.dist.ReduceOp.SUM)

    def eval(self, opts, **kw):
        self.eval_async(opts, **kw)
        res = self.dm.read_scalars()
        if self.transport == "peer" and self.dm.halo_error():
            raise self.L.B200Error("a halo pull gave up waiting for a peer's flag (a rank left the lock-step sequence)")
        return res

    def eval_host(self, opts, pos_owned: np.ndarray, grad_owned: np.ndarray):
        """End-to-end evaluation with HOST buffers: this rank uploads the positions of its OWNED rows,
        the ghost rows arrive through the halo exchange, and the projected gradient of the owned rows
        is copied back together with the (global) scalars."""
        L, dm, n = self.L, self.dm, self.local.n_owned
        lib = L.lib()
        L.check(lib.ms_ctx_upload(dm._h, L.ARR_TRIAL if opts.use_trial else L.ARR_POSITIONS, L.dptr(pos_owned), 0,
                                  3 * n))
        self.eval_async(opts, exchange_positions=True)
        L.check(lib.ms_ctx_get_array(dm._h, L.ARR_GRAD, L.dptr(grad_owned), 0, 3 * n))
        return dm.read_scalars()


def _shared_mesh(n: int, rank: int, dist, tag: str):
    """Frequency-n icosphere on every rank: generated once (rank 0), shared through /dev/shm."""
    import os
    import time

    from .synthetic import icosphere

    shm = "/dev/shm" if os.path.isdir("/dev/shm") else "/tmp"
    path = os.path.join(shm, f"ms_b200_bench_{os.environ.get('MASTER_PORT', '0')}_{tag}_n{n}.npz")
    t0 = time.perf_counter()
    if rank == 0:
        pos, tri = icosphere(n)
        np.savez(path, pos=pos, tri=tri)
    dist.barrier()
    if rank != 0:
        with np.load(path) as z:
            pos, tri = z["pos"], z["tri"]
    dist.barrier()
    if rank == 0:
        os.remove(path)
    return pos, tri, time.perf_counter() - t0


def _parity_vs_single_gpu(pm, local, pos, tri, opts, rank, world, dist, torch, L, sample_rows: int = 4096):
    """Correctness of the partitioned evaluation against ONE GPU evaluating the same mesh (rank 0, its own
    context): the all-reduced scalars, and the projected gradient on a random sample of every rank's owned rows.
    Returns (dict, ok) on rank 0, (None, True) elsewhere."""
    from .context import DeviceMesh

    dm = pm.dm
    pm.eval_async(opts)
    torch.cuda.synchronize()
    sc = dm.read_scalars().scalars.copy()
    rng = np.random.default_rng(1234 + rank)
    rows = np.sort(rng.choice(local.n_owned, size=min(sample_rows, local.n_owned), replace=False))
    g_owned = dm.download(L.ARR_GRAD)[rows]
    payload = (local.lo + rows, g_owned)
    gathered = [None] * world if rank == 0 else None
    dist.gather_object(payload, gathered, dst=0)
    if rank != 0:
        return None, True
    nv, nf = pos.shape[0], tri.shape[0]
    one = DeviceMesh(pm.device.index)
    one.set_topology(nv, tri, body_mask=np.ones(nf, np.uint8))
    one.set_surface_tension(1.0)
    one.set_bending_params(1.0, 0.0)
    one.set_positions(pos)
    ref = one.eval(one.options(L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME, constraint_mode=0))
    g_ref = one.download(L.ARR_GRAD)
    one.close()
    names = {"E_surface": L.SC_E_SURFACE, "area": L.SC_AREA, "volume": L.SC_VOLUME, "E_bending": L.SC_E_BENDING,
             "lambda": L.SC_LAMBDA}
    err = {k: float(abs(sc[i] - ref.scalars[i]) / max(abs(ref.scalars[i]), 1e-300)) for k, i in names.items()}
    scale = float(np.abs(g_ref).max())
    g_err = 0.0
    n_rows = 0
    for ids, g in gathered:
        g_err = max(g_err, float(np.abs(g - g_ref[ids]).max()) / scale)
        n_rows += len(ids)
    tol = 1e-12
    ok = all(v <= 1e-11 if k == "lambda" else v <= tol for k, v in err.items()) and g_err <= tol
    return {"against": "one GPU evaluating the same mesh (rank 0)", "scalar_rel_err": err,
            "projected_grad_rel_err": g_err, "sampled_rows": n_rows, "tolerance": tol, "ok": bool(ok)}, bool(ok)


def _measure_partitioned(args, rank, world, local_rank, bench, total_facets: int, tag: str, *, with_e2e: bool,
                         with_parity: bool, steps: int):
    """Build, partition and time one mesh of ~total_facets facets on `world` GPUs.  Returns a dict on rank 0."""
    import os
    import time

    import torch
    import torch.distributed as dist

    from . import _lib as L
    from .synthetic import frequency_for_facets

    n = frequency_for_facets(total_facets)
    pos, tri, t_gen = _shared_mesh(n, rank, dist, tag)
    nv, nf = pos.shape[0], tri.shape[0]
    t0 = time.perf_counter()
    local = split_mesh(nv, tri, world, rank)
    pm = PartitionedMesh(local, local_rank, body_mask=np.ones(local.tri.shape[0], np.uint8),
                         reserve_sms=int(os.environ.get("MS_RESERVE_SMS", "0")),
                         pack=dict(threads=args.threads, max_owned=args.max_owned, max_local=args.max_local,
                                   fill_pct=args.fill, repair_sweeps=args.repair))
    dm = pm.dm
    dm.set_surface_tension(1.0)
    dm.set_bending_params(1.0, 0.0)
    pos_local = pos[local.global_rows()]
    dm.set_positions(pos_local)
    t_setup = time.perf_counter() - t0
    opts = dm.options(L.MOD_SURFACE | L.MOD_BENDING | L.MOD_VOLUME, constraint_mode=0)

    sampler = bench.ClockSampler(local_rank)
    overlap = os.environ.get("MS_OVERLAP", "0") != "0"
    for _ in range(max(3, args.warmup)):
        pm.eval_async(opts, overlap=overlap)
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.active.set()
    ev0.record()
    for _ in range(steps):
        pm.eval_async(opts, overlap=overlap)
    ev1.record()
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    sampler.active.clear()
    ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=pm.device)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_step = float(ms.item()) / steps
    res = dm.read_scalars()
    out = {"facets": nf, "vertices": nv, "frequency": n, "ms_per_step": ms_step, "steps": steps,
           "value": nf / (ms_step * 1e-3) / 1e9, "mesh_seconds": t_gen, "partition_pack_seconds": t_setup,
           "transport": pm.transport, "fused": bool(pm.fused), "push": bool(pm.push),
           "in_kernel": bool(pm.fused and pm.in_kernel and not pm.push),
           "energies": {"surface": res.e_surface, "bending": res.e_bending, "volume": res.volume}}
    phases = None
    if os.environ.get("MS_PHASES", "0") != "0":  # per-phase device times of this rank (diagnostic)
        names = ["halo(pos)", "pass A", "halo(seeds)", "pass B", "reduce", "all-reduce", "project"]
        acc = np.zeros(len(names))
        reps = 10
        for _ in range(reps):
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)]
            evs[0].record(); pm.exchange(L.ARR_POSITIONS)
            evs[1].record(); dm.eval_pass_a(opts)
            evs[2].record(); pm.exchange(L.ARR_SEEDS)
            evs[3].record(); dm.eval_pass_b(opts)
            evs[4].record(); dm.eval_reduce(opts)
            evs[5].record(); pm._allreduce_scalars()
            evs[6].record(); dm.eval_project(opts)
            evs[7].record(); torch.cuda.synchronize()
            acc += [evs[i].elapsed_time(evs[i + 1]) for i in range(len(names))]
        mine = torch.tensor(acc / reps, dtype=torch.float64, device=pm.device)
        allp = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allp, mine)
        info = dm.pack_info()
        stats = torch.tensor([info["n_listed"], info["n_patches"], local.tri.shape[0], local.nv_local],
                             dtype=torch.float64, device=pm.device)
        alls = [torch.zeros_like(stats) for _ in range(world)]
        dist.all_gather(alls, stats)
        phases = {"names": names, "ms_per_rank": [[round(float(x), 4) for x in t.tolist()] for t in allp],
                  "listed_patches_facets_rows_per_rank": [[int(x) for x in t.tolist()] for t in alls]}
        out["phases"] = phases
    if with_e2e:
        # ---- end to end: pinned host positions of the owned rows in, projected gradient out, every step ----
        lib = L.lib()
        pos_owned = np.ascontiguousarray(pos_local[:local.n_owned])
        grad_owned = np.empty_like(pos_owned)
        L.check(lib.ms_host_register(pos_owned.ctypes.data, pos_owned.nbytes))
        L.check(lib.ms_host_register(grad_owned.ctypes.data, grad_owned.nbytes))
        for _ in range(2):
            pm.eval_host(opts, pos_owned, grad_owned)
        e2e_steps = max(3, min(steps, 10))
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(e2e_steps):
            pm.eval_host(opts, pos_owned, grad_owned)
        ev1.record()
        torch.cuda.synchronize()
        dist.barrier()
        ms2 = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=pm.device)
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
        ms_e2e = float(ms2.item()) / e2e_steps
        L.check(lib.ms_host_unregister(pos_owned.ctypes.data))
        L.check(lib.ms_host_unregister(grad_owned.ctypes.data))
        io = torch.tensor([pos_owned.nbytes, grad_owned.nbytes + 8 * L.SC_COUNT], dtype=torch.float64, device=pm.device)
        dist.all_reduce(io, op=dist.ReduceOp.SUM)
        out["e2e"] = {"value": nf / (ms_e2e * 1e-3) / 1e9, "unit": bench.UNIT, "h2d_bytes_per_step": int(io[0].item()),
                      "d2h_bytes_per_step": int(io[1].item()), "ms_per_step": ms_e2e,
                      "api": "PartitionedMesh.eval_host per rank (pinned owned positions in, halo exchange, "
                             "projected gradient of the owned rows + scalars out)"}
    if pm.transport == "peer" and dm.halo_error():
        raise L.B200Error(f"rank {rank}: a peer-memory pull gave up waiting; the numbers of this run are void")
    ghosts = torch.tensor([local.ghost_ids.size, pm.halo.send_rows.size], dtype=torch.float64, device=pm.device)
    dist.all_reduce(ghosts, op=dist.ReduceOp.MAX)
    out["max_ghost_rows_per_rank"] = int(ghosts[0].item())
    if with_parity:
        parity, ok = _parity_vs_single_gpu(pm, local, pos, tri, opts, rank, world, dist, torch, L)
        flag = torch.tensor([1.0 if ok else 0.0], dtype=torch.float64, device=pm.device)
        dist.broadcast(flag, src=0)
        out["parity"] = parity
        if flag.item() == 0.0 and rank == 0:
            out["void"] = "the partitioned evaluation differs from the single-GPU evaluation: numbers of this run are void"
    sampler.close()
    out["clocks"] = sampler.summary()
    pm.close()
    del pm, dm
    torch.cuda.empty_cache()
    return out


def bench_multi_gpu(args, rank: int, world: int, local_rank: int, bench):
    """N>1 arm of bench.py.  Weak scaling (``args.facets`` facets per GPU) is the headline line the driver's
    scaling run reads; the same line carries ``strong``: the ``args.strong_facets``-facet mesh (BASELINE.json
    north_star: 100 M facets) cut over the N GPUs, and ``parity``: the partitioned result against one GPU
    evaluating the same mesh."""
    import json

    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    # host buffers (pinned positions / gradients of the e2e leg, pack scratch) next to this rank's GPU
    import os

    from .numa import bind_to_gpu

    numa = bind_to_gpu(local_rank) if os.environ.get("MS_NUMA_BIND", "1") != "0" else {"bound": False, "reason": "MS_NUMA_BIND=0"}
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    numa_all = [None] * world
    dist.all_gather_object(numa_all, numa)
    weak = _measure_partitioned(args, rank, world, local_rank, bench, args.facets * world, "weak", with_e2e=True,
                                with_parity=not args.no_parity, steps=args.steps)
    strong = None
    if args.strong_facets > 0:
        strong = _measure_partitioned(args, rank, world, local_rank, bench, args.strong_facets, "strong", with_e2e=False,
                                      with_parity=False, steps=max(3, min(args.steps, 10)))
    if rank == 0:
        peak, peak_kind = bench._peaks()
        value = weak["value"]
        peer = weak["transport"] == "peer"
        line = {
            "metric": bench.METRIC, "value": value, "unit": bench.UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": weak["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {**bench.workload_config(args, world), "parallelism": f"vertex-partition x{world}, 1-ring ghosts",
                       "max_ghost_rows_per_rank": weak["max_ghost_rows_per_rank"]},
            "roofline": {"bound": "hbm", "kernel": "whole step (all ranks)", "achieved": bench.B_STEP * value,
                         "peak": peak * world, "unit": "GB/s", "frac": bench.B_STEP * value / (peak * world),
                         "traffic": None, "peak_source": f"MEASURED_PEAKS.json ({peak_kind}) x {world} GPUs",
                         "bytes_per_facet": bench.B_STEP},
            "e2e": {**weak["e2e"], "numa": numa_all},
            "collectives_per_step": {"halo_exchanges": 2, "all_reduce": 1,
                                     "halo_transport": weak["transport"] + (" (push)" if weak.get("push") else
                                                                             " (inside the patch kernels)" if weak.get("in_kernel") else ""),
                                     "all_reduce_transport": "peer memory" if peer else "nccl",
                                     "halo_bytes_per_rank": weak["max_ghost_rows_per_rank"] * (24 + 40)},
            # in-kernel exchange: pass A and pass B only (halo pulls by the epilogue warps behind the interior patches,
            # scalars published and gathered by the last CTA).  Fused peer transport: signal+pull positions, pass A (raises the seed flag), seed
            # pull, pass B (reduces + publishes), gather + coefficient.  Unfused: pass A, pass B, reduce, coefficient
            # + per halo exchange flag signal + pull (peer) or the row gather (nccl) + the all-reduce's two kernels
            "gpu_launches": (2 if weak.get("in_kernel") else 5 if weak.get("fused") else 4 + (6 if peer else 2)) * args.steps,
            "launches_per_step": 2 if weak.get("in_kernel") else 5 if weak.get("fused") else 4 + (6 if peer else 2),
            "clocks": weak["clocks"],
            "energies": weak["energies"],
            "setup_seconds": weak["mesh_seconds"] + weak["partition_pack_seconds"],
            "parity": weak.get("parity"),
        }
        if "void" in weak:
            line["void"] = weak["void"]
        if "phases" in weak:
            line["phases"] = weak["phases"]
        if strong is not None:
            # strong scaling: total work fixed; the N = 1 run of bench.py reports the same mesh on one GPU
            line["strong"] = {"scaling": "strong", "facets": strong["facets"], "n_gpus": world,
                              "ms_per_step": strong["ms_per_step"], "value": strong["value"], "unit": bench.UNIT,
                              "steps": strong["steps"], "transport": strong["transport"],
                              "energies": strong["energies"],
                              "setup_seconds": strong["mesh_seconds"] + strong["partition_pack_seconds"],
                              "note": "speed-up over one GPU = strong.ms_per_step of the --gpus 1 line / this ms_per_step"}
        print(json.dumps(line))
    dist.destroy_process_group()
    return 0
