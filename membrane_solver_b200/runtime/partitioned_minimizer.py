"""Device-resident minimisation over a mesh partitioned across GPUs.

BASELINE.json north_star: "NCCL over NVLink handles the one-ring ghost-vertex halo exchange and the scalar
energy/volume allreduce for line search".  ``DeviceMinimizer`` (``runtime/device_minimizer.py``; the reference's
``Minimizer.minimize`` + ``backtracking_line_search_array``, ``runtime/minimizer.py:1189-1535``,
``runtime/steppers/line_search.py:267-541``) talks to ONE object with the ``DeviceMesh`` methods it needs.
``PartitionedDevice`` is that object for one rank of a ``PartitionedMesh``:

* evaluations go through ``PartitionedMesh.eval``: halo exchange of the (trial) positions and of the bending seeds,
  scalars summed over all ranks in rank order, KKT multiplier from the global sums -- so every rank reads the same
  energies and takes the same branch of the line search;
* per-row operations (direction, Polak-Ribiere update, trial positions, accept, Newton volume projection) act on the
  rank's own rows; ghost rows are refreshed by the exchange that precedes every evaluation;
* the line-search statistics are reduced across ranks: shortest edge (min), largest direction row (max),
  ``<g,d>`` and ``<g,g>`` over OWNED rows (sum);
* the normal-flip guard (``runtime/topology.py:13-48``) first brings the ghost rows of the trial positions, then
  every rank checks its facets and the verdicts are AND-ed.
* vertex averaging (the ``V`` command), equiangulation (``u``) and refinement (``r``) are refused: they run on a
  single GPU only.

All ranks call the same sequence (the loop control depends only on reduced values), which is what the peer-memory
transport's lock-step flags need.
"""

from __future__ import annotations

from .. import _lib as L
from .device_minimizer import DeviceMinimizer


class PartitionedDevice:
    """``DeviceMesh`` facade of one rank's partition (see the module docstring)."""

    def __init__(self, pm):
        self.pm = pm
        self.dm = pm.dm
        self.dist = pm.dist
        self.torch = pm.torch

    # -- evaluation --------------------------------------------------------------------------------------------
    def options(self, *args, **kwargs):
        return self.dm.options(*args, **kwargs)

    def eval(self, opts):
        return self.pm.eval(opts)

    # -- per-row operations on this rank's rows ----------------------------------------------------------------
    def direction_from_gradient(self, scale: float = -1.0) -> None:
        self.dm.direction_from_gradient(scale)

    def cg_direction(self, restart: bool) -> None:
        self.dm.cg_direction(restart)

    def cg_commit(self) -> None:
        self.dm.cg_commit()

    def axpy(self, dst: int, src: int, alpha: float, skip_fixed: bool = True) -> None:
        self.dm.axpy(dst, src, alpha, skip_fixed=skip_fixed)

    def vertex_average(self, rounds: int = 1, group=None) -> None:
        raise L.B200Error("vertex averaging (V) runs on a single GPU only: re-assemble the mesh on one device")

    def equiangulate(self, max_iterations: int = 100) -> int:
        raise L.B200Error("equiangulation (u) runs on a single GPU only: re-assemble the mesh on one device")

    def refine(self, levels: int = 1):
        raise L.B200Error("refinement (r) runs on a single GPU only: re-assemble the mesh on one device")

    def make_trial(self, alpha: float) -> None:
        self.dm.make_trial(alpha)

    def accept_trial(self) -> None:
        self.dm.accept_trial()

    # -- reductions across ranks -------------------------------------------------------------------------------
    def _all_reduce(self, values, op):
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device=self.pm.device)
        self.dist.all_reduce(t, op=op)
        return [float(x) for x in t.tolist()]

    def line_search_stats(self):
        min_edge, max_dir, g_dot_d, g_dot_g = self.dm.line_search_stats()
        # a rank without facets reports 0 for "no edge": keep it out of the minimum
        lo = self._all_reduce([-(min_edge if min_edge > 0.0 else float("inf")), max_dir], self.dist.ReduceOp.MAX)
        sums = self._all_reduce([g_dot_d, g_dot_g], self.dist.ReduceOp.SUM)
        edge = -lo[0]
        return (0.0 if edge == float("inf") else edge), lo[1], sums[0], sums[1]

    def normal_change_ok(self, limit: float = 0.5) -> bool:
        self.pm.exchange(L.ARR_TRIAL)          # ghost rows of the trial positions
        ok = 1.0 if self.dm.normal_change_ok(limit) else 0.0
        return self._all_reduce([ok], self.dist.ReduceOp.MIN)[0] > 0.5


def partitioned_minimizer(pm, **kwargs) -> DeviceMinimizer:
    """``DeviceMinimizer`` over a ``PartitionedMesh``; same keyword arguments.  Collective: every rank builds one
    and calls ``minimize`` with the same arguments."""
    return DeviceMinimizer(dm=PartitionedDevice(pm), **kwargs)


__all__ = ["PartitionedDevice", "partitioned_minimizer"]
