"""Slicing: the data-parallel mode the reference lists as future work
(book/src/future_work.md:9-11, book/src/parallelization.md:16-24).

Fixing the value of a leg that is summed over splits one contraction into dim(leg) independent
contractions of smaller networks whose results add up.  With S sliced legs of dimension 2 there are
2^S independent units: they bound the peak memory, and they shard over GPUs with a single
all-reduce at the end (`contract_sliced`).  The same replace-left path is used for every slice."""
from __future__ import annotations

import itertools
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

from ..tensornetwork.tensor import Tensor
from ..tensornetwork.tensordata import TensorData
from . import ContractionPath


def _flat(tn: Tensor) -> List[Tensor]:
    assert all(t.is_leaf() for t in tn.tensors), "slicing works on flat networks"
    return tn.tensors


def path_cost(tensors: Sequence[Tuple[Sequence[int], Sequence[int]]], path: ContractionPath, sliced: Iterable[int] = ()):
    """(flops 8MNK summed, peak intermediate elements, legs of the largest intermediate) with the
    `sliced` legs removed."""
    sl = set(sliced)
    ts: List[Optional[Dict[int, int]]] = [{l: d for l, d in zip(legs, dims) if l not in sl} for legs, dims in tensors]
    flops, peak, peak_legs = 0.0, 0.0, []
    for (i, j) in path.toplevel:
        a, b = ts[i], ts[j]
        out = {l: d for l, d in b.items() if l not in a}
        out.update({l: d for l, d in a.items() if l not in b})
        f = 8.0
        for l, d in a.items():
            f *= d
        for l, d in b.items():
            if l not in a:
                f *= d
        flops += f
        sz = 1.0
        for d in out.values():
            sz *= d
        if sz > peak:
            peak, peak_legs = sz, list(out)
        ts[i], ts[j] = out, None
    return flops, peak, peak_legs


def path_time(tensors: Sequence[Tuple[Sequence[int], Sequence[int]]], path: ContractionPath, sliced: Iterable[int] = ()) -> float:
    """Predicted device seconds of one slice (contraction_cost.gpu_time_tensors per pair): unlike the flop count it
    sees that halving K of the dominant pair costs the tcgen05 engine efficiency while halving M or N does not."""
    from ..tensornetwork.tensor import Tensor as _T
    from .contraction_cost import gpu_time_tensors
    sl = set(sliced)
    ts: List[Optional[_T]] = [_T([l for l in legs if l not in sl], [d for l, d in zip(legs, dims) if l not in sl]) for legs, dims in tensors]
    total = 0.0
    for (i, j) in path.toplevel:
        total += gpu_time_tensors(ts[i], ts[j])
        ts[i], ts[j] = ts[j] ^ ts[i], None
    return total


def find_slices(tn: Tensor, path: ContractionPath, min_slices: int = 1, max_peak_elements: Optional[float] = None,
                objective: str = "flops") -> List[int]:
    """Greedy slice finder: repeatedly slice the leg of the currently largest intermediate that
    minimises the total work (slices x flops, or slices x predicted device time with objective="time"), until there
    are at least `min_slices` slices and the largest intermediate has at most `max_peak_elements` elements.
    Output legs are never sliced."""
    leaves = _flat(tn)
    meta = [(t.legs, t.bond_dims) for t in leaves]
    count: Dict[int, int] = {}
    dim: Dict[int, int] = {}
    for legs, dims in meta:
        for l, d in zip(legs, dims):
            count[l] = count.get(l, 0) + 1
            dim[l] = d
    sliced: List[int] = []
    n_slices = 1
    while True:
        flops, peak, peak_legs = path_cost(meta, path, sliced)
        if n_slices >= min_slices and (max_peak_elements is None or peak <= max_peak_elements):
            return sliced
        cands = [l for l in peak_legs if count.get(l, 0) >= 2 and dim[l] > 1]
        if not cands:
            cands = [l for l in dim if count[l] >= 2 and dim[l] > 1 and l not in sliced]
        if not cands:
            return sliced
        best, best_cost = None, None
        for l in cands:
            f, p, _ = path_cost(meta, path, sliced + [l])
            if objective == "time":
                f = path_time(meta, path, sliced + [l])
            cost = (f * n_slices * dim[l], p)
            if best_cost is None or cost < best_cost:
                best, best_cost = l, cost
        sliced.append(best)
        n_slices *= dim[best]


def slice_assignments(tn: Tensor, legs: Sequence[int]) -> List[Tuple[int, ...]]:
    dim = {l: d for t in _flat(tn) for l, d in t.edges()}
    return list(itertools.product(*[range(dim[l]) for l in legs]))


def _leaf_array(t: Tensor) -> np.ndarray:
    td = t.tensordata
    if td.kind == "gate":
        from ..gates import load_gate, load_gate_adjoint
        name, angles, adj = td.gate
        return (load_gate_adjoint if adj else load_gate)(name, angles).reshape(t.bond_dims)
    if td.kind == "matrix":
        m = td.matrix
        return (m if isinstance(m, np.ndarray) else m.to_numpy()).reshape(t.bond_dims)
    raise RuntimeError("Cannot convert uncontracted tensor to data")


class SlicedNetwork:
    """Pre-extracts the leaves that contain sliced legs so that building slice number s is a few
    tiny numpy index operations; all other leaves are shared between slices."""

    def __init__(self, tn: Tensor, legs: Sequence[int]):
        self.tn, self.legs = tn, list(legs)
        self.leaves = list(_flat(tn))
        self.touched = {}
        for idx, t in enumerate(self.leaves):
            if any(l in t.legs for l in self.legs):
                self.touched[idx] = _leaf_array(t)
            elif t.tensordata.kind == "matrix" and not isinstance(t.tensordata.matrix, np.ndarray):
                # a device-resident leaf shared by every slice would be consumed by the first one:
                # download it once, every slice then uploads its own copy with the leaf block
                nt = Tensor(t.legs, t.bond_dims)
                nt.set_tensor_data(TensorData.Matrix(_leaf_array(t)))
                self.leaves[idx] = nt
        self.assignments = slice_assignments(tn, self.legs)

    def slice(self, assignment: Sequence[int]) -> Tensor:
        val = dict(zip(self.legs, assignment))
        out = []
        for idx, t in enumerate(self.leaves):
            if idx not in self.touched:
                out.append(t)
                continue
            arr = self.touched[idx]
            index = tuple(val[l] if l in val else slice(None) for l in t.legs)
            keep = [(l, d) for l, d in t.edges() if l not in val]
            nt = Tensor([l for l, _ in keep], [d for _, d in keep])
            nt.set_tensor_data(TensorData.Matrix(np.ascontiguousarray(arr[index])))
            out.append(nt)
        return Tensor.new_composite(out)


class SlicedPlan:
    """Compile + stage once, run many: the sliced contraction with every slice's leaf block resident on the device and
    the slice loop inside libtncb200 (tncb_plan_stage_slices / tncb_plan_run_slices)."""

    def __init__(self, tn: Tensor, path: ContractionPath, legs: Sequence[int], ctx=None, dtype=np.complex128):
        from .. import default_context, dtype_code
        from ..tensornetwork.contraction import NetworkPlan
        dtype_code(dtype)
        self.dtype = np.dtype(dtype)
        self.ctx = ctx or default_context()
        self.sn = SlicedNetwork(tn, legs)
        nets = [self.sn.slice(a) for a in self.sn.assignments]
        self.n_slices = len(nets)
        self.plan = NetworkPlan(nets[0], path, ctx=self.ctx, dtype=dtype)
        self.plan.stage_slices(nets)

    def run(self, rank: int = 0, world: int = 1, allreduce: bool = True) -> Tensor:
        from .._lib import check
        if world > 1 and self.dtype == np.complex64:
            raise ValueError("multi-rank sliced runs are complex128 only (the NCCL all-reduce has no complex64 path)")
        total = self.plan.run_slices(rank, world)
        if world > 1 and allreduce:
            check(self.ctx._l.tncb_comm_allreduce_sum(self.ctx.handle, total.tensordata.matrix.handle))
        return total


def contract_sliced(tn: Tensor, path: ContractionPath, legs: Sequence[int], ctx=None, rank: int = 0, world: int = 1,
                    allreduce: bool = True, dtype=np.complex128) -> Tensor:
    """Contracts every slice assigned to this rank (round-robin: slices rank, rank + world, ...), accumulates on the
    device and, with world > 1, sums over ranks with one NCCL all-reduce (`tncb_comm_allreduce_sum`; the communicator must
    have been set up with `dist.init_device_comm`).  One schedule is compiled, all slice payloads are uploaded once and
    the slice loop runs inside the library; `SlicedPlan` keeps that state for repeated runs.  dtype=np.complex64 runs
    the slices in complex64 (single rank only)."""
    from .. import TNCB_C64, dtype_code
    if world > 1 and dtype_code(dtype) == TNCB_C64:      # refused before any slice is staged
        raise ValueError("multi-rank sliced runs are complex128 only (the NCCL all-reduce has no complex64 path)")
    return SlicedPlan(tn, path, legs, ctx, dtype).run(rank, world, allreduce)
