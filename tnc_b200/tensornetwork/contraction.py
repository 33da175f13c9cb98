"""contract_tensor_network (tnc/src/tensornetwork/contraction.rs:30-52) over the C ABI.

The Python side only marshals the `Tensor` tree and the `ContractionPath` into the plain C
structs of include/tncb.h; schedule construction, leaf materialisation, the single host->device
upload and every pair kernel run inside libtncb200."""
from __future__ import annotations

import ctypes as C
import os
from itertools import chain
from typing import List, Optional

import numpy as np

from .. import Context, DeviceTensor, default_context, dtype_code
from .._lib import TncbError, TncbPath, TncbTn, check, u64_array
from ..contractionpath import ContractionPath
from .tensor import Tensor
from .tensordata import TensorData

_KIND = {"uncontracted": 0, "matrix": 1, "gate": 2, "device": 3}


# TncbTn as a numpy record (same layout as the ctypes Structure / the C struct): a composite's children are filled
# column-wise instead of one ctypes object per leaf (the 36-qubit bench network has 489 leaves per call)
_TN_DTYPE = np.dtype([("n_children", np.uint64), ("children", np.uint64), ("rank", np.int32), ("legs", np.uint64), ("dims", np.uint64),
                      ("kind", np.int32), ("host_re_im", np.uint64), ("gate_name", np.uint64), ("gate_angles", np.uint64),
                      ("n_gate_angles", np.int32), ("gate_adjoint", np.int32), ("device", np.uint64),
                      ("file_path", np.uint64), ("file_adjoint", np.int32)], align=True)
assert _TN_DTYPE.itemsize == C.sizeof(TncbTn), "TncbTn layout drifted"
_GATE_NAMES = {}


def _gate_name_ptr(name: str) -> int:
    hit = _GATE_NAMES.get(name)
    if hit is None:
        buf = C.create_string_buffer(name.encode())                         # interned: stays alive for the process
        hit = _GATE_NAMES[name] = (C.addressof(buf), buf)
    return hit[0]


class _Marshal:
    """Keeps every buffer the C tree points to alive for the duration of the call."""

    def __init__(self):
        self.keep: List[object] = []
        self.device_inputs: List[DeviceTensor] = []

    def _children(self, tensors) -> int:
        """array of TncbTn for `tensors`; returns its address"""
        n = len(tensors)
        rec = np.zeros(n, dtype=_TN_DTYPE)
        self.keep.append(rec)
        ranks = [len(t.legs) for t in tensors]
        tot = sum(ranks)
        legs = np.fromiter(chain.from_iterable(t.legs for t in tensors), dtype=np.uint64, count=tot)
        dims = np.fromiter(chain.from_iterable(t.bond_dims for t in tensors), dtype=np.uint64, count=tot)
        self.keep += [legs, dims]
        off = np.zeros(n, dtype=np.uint64)
        if n > 1:
            np.cumsum(np.asarray(ranks[:-1], dtype=np.uint64), out=off[1:])
        rec["legs"] = legs.ctypes.data + 8 * off
        rec["dims"] = dims.ctypes.data + 8 * off
        # one pass over the leaves into plain lists, one column assignment per field (a numpy record setitem or an
        # ndarray.ctypes access per leaf costs more than everything else in this function)
        kind, n_children, children = [0] * n, [0] * n, [0] * n
        host, device, gate_name, gate_adj, gate_ang, n_ang = [0] * n, [0] * n, [0] * n, [0] * n, [0] * n, [0] * n
        file_path, file_adj = [0] * n, [0] * n
        ang_vals: List[float] = []
        for i, t in enumerate(tensors):
            if t.tensors:
                n_children[i] = len(t.tensors)
                children[i] = self._children(t.tensors)
                ranks[i] = 0
                continue
            td = t.tensordata
            k = td.kind
            if k == "gate":
                name, ang, adj = td.gate
                kind[i] = 2
                gate_name[i] = _gate_name_ptr(name)
                gate_adj[i] = int(adj)
                gate_ang[i] = 8 * len(ang_vals)        # byte offset into `angles`, made absolute below
                if ang:
                    n_ang[i] = len(ang)
                    ang_vals.extend(ang)
            elif k == "matrix":
                m = td.matrix
                if isinstance(m, DeviceTensor):
                    if m.handle is None:   # consumed by an earlier call (the Rust move left TensorData::Uncontracted behind)
                        raise TncbError(-3, "Cannot convert uncontracted tensor to data (device tensor already consumed)")
                    kind[i] = 3
                    device[i] = m.handle.value or 0
                    self.device_inputs.append(m)
                else:
                    arr = np.asarray(m, dtype=np.complex128, order="C")
                    if list(arr.shape) != list(t.bond_dims):
                        arr = arr.reshape(t.bond_dims)
                    self.keep.append(arr)
                    kind[i] = 1
                    host[i] = arr.__array_interface__["data"][0]
            elif k == "file":   # TensorData::File((path, adjoint)): loaded by the library while it stages the leaves
                buf = C.create_string_buffer(os.fsencode(td.file[0]))
                self.keep.append(buf)
                kind[i] = 4
                file_path[i] = C.addressof(buf)
                file_adj[i] = int(bool(td.file[1]))
        angles = np.zeros(max(len(ang_vals), 1), dtype=np.float64)
        angles[:len(ang_vals)] = ang_vals
        self.keep.append(angles)
        abase = angles.__array_interface__["data"][0]
        rec["rank"] = ranks
        rec["kind"] = kind
        rec["n_children"] = n_children
        rec["children"] = children
        rec["host_re_im"] = host
        rec["device"] = device
        rec["gate_name"] = gate_name
        rec["gate_adjoint"] = gate_adj
        rec["n_gate_angles"] = n_ang
        rec["gate_angles"] = [abase + o if kd == 2 else 0 for o, kd in zip(gate_ang, kind)]
        rec["file_path"] = file_path
        rec["file_adjoint"] = file_adj
        return rec.ctypes.data

    def tn(self, t: Tensor) -> TncbTn:
        addr = self._children([t])
        return TncbTn.from_address(addr)

    def path(self, p: ContractionPath) -> TncbPath:
        out = TncbPath()
        flat = [x for pair in p.toplevel for x in pair]
        pairs = u64_array(flat)
        self.keep.append(pairs)
        out.n_pairs = len(p.toplevel)
        out.pairs = pairs
        idx = sorted(p.nested)
        if idx:
            ni = u64_array(idx)
            arr = (TncbPath * len(idx))(*[self.path(p.nested[i]) for i in idx])
            self.keep += [ni, arr]
            out.n_nested = len(idx)
            out.nested_index = ni
            out.nested = arr
        return out


def contract_tensor_network(tn: Tensor, contract_path: ContractionPath, ctx: Optional[Context] = None,
                            dtype=np.complex128) -> Tensor:
    """Fully contracts `tn` with the replace-left `contract_path`; returns the resulting
    leaf `Tensor` whose data stays on the device (`.to_numpy()` downloads it).
    dtype=np.complex64 runs every kernel in complex64 (f64 accumulation, one rounding per result; host payloads are
    narrowed while they are staged, device leaves must already be complex64); the result is complex64 then."""
    code = dtype_code(dtype)
    ctx = ctx or default_context()
    m = _Marshal()
    c_tn = m.tn(tn)
    c_path = m.path(contract_path)
    out = C.c_void_p()
    n_out = C.c_int()
    legs = u64_array([0] * 64)
    rc = ctx._l.tncb_contract_tensor_network_dt(ctx.handle, C.byref(c_tn), C.byref(c_path), code, C.byref(out), C.byref(n_out), legs)
    check(rc)
    for d in m.device_inputs:  # consumed by the call
        d.release()
    if not out.value:
        return Tensor()  # nothing left (empty network)
    dt = DeviceTensor.adopt(ctx, out)
    res = Tensor([legs[i] for i in range(n_out.value)], dt.shape)
    res.set_tensor_data(TensorData.Matrix(dt))
    return res


class NetworkPlan:
    """Compile once / execute many (tncb_plan_*): same structure, new payloads.  `dtype` (complex128 or complex64) is the
    element type of every run of the plan."""

    def __init__(self, tn: Tensor, contract_path: ContractionPath, ctx: Optional[Context] = None, dtype=np.complex128):
        self.handle = None
        code = dtype_code(dtype)
        self.dtype = np.dtype(dtype)
        self.ctx = ctx or default_context()
        m = _Marshal()
        c_tn, c_path = m.tn(tn), m.path(contract_path)
        h = C.c_void_p()
        check(self.ctx._l.tncb_plan_create_dt(self.ctx.handle, C.byref(c_tn), C.byref(c_path), code, C.byref(h)))
        self.handle = h

    def info(self) -> dict:
        n, k = C.c_uint64(), C.c_uint64()
        pk = C.c_uint64()
        fl, by = C.c_double(), C.c_double()
        check(self.ctx._l.tncb_plan_info(self.handle, C.byref(n), C.byref(fl), C.byref(by), C.byref(pk), C.byref(k)))
        return {"pairs": n.value, "flops": fl.value, "bytes": by.value, "peak_bytes": pk.value, "kernels": k.value}

    def stage(self, tn: Tensor) -> None:
        """Materialise + upload the leaves once (tncb_plan_stage); `run()` then needs no host data."""
        m = _Marshal()
        c_tn = m.tn(tn)
        check(self.ctx._l.tncb_plan_stage(self.ctx.handle, self.handle, C.byref(c_tn)))

    def run(self) -> Tensor:
        out, n_out, legs = C.c_void_p(), C.c_int(), u64_array([0] * 64)
        check(self.ctx._l.tncb_plan_run(self.ctx.handle, self.handle, C.byref(out), C.byref(n_out), legs))
        if not out.value:
            return Tensor()
        dt = DeviceTensor.adopt(self.ctx, out)
        res = Tensor([legs[i] for i in range(n_out.value)], dt.shape)
        res.set_tensor_data(TensorData.Matrix(dt))
        return res

    def stage_slices(self, slice_tns) -> None:
        """Materialise + upload the leaf blocks of every slice network once (tncb_plan_stage_slices)."""
        m = _Marshal()
        nodes = [m.tn(t) for t in slice_tns]
        ptrs = (C.POINTER(TncbTn) * len(nodes))(*[C.pointer(n) for n in nodes])
        check(self.ctx._l.tncb_plan_stage_slices(self.ctx.handle, self.handle, len(nodes), ptrs))

    def run_slices(self, first: int = 0, stride: int = 1) -> Tensor:
        """Sum of the slices first, first + stride, ... on the device, no host work per slice."""
        out, n_out, legs = C.c_void_p(), C.c_int(), u64_array([0] * 64)
        check(self.ctx._l.tncb_plan_run_slices(self.ctx.handle, self.handle, int(first), int(stride), C.byref(out), C.byref(n_out), legs))
        dt = DeviceTensor.adopt(self.ctx, out)
        res = Tensor([legs[i] for i in range(n_out.value)], dt.shape)
        res.set_tensor_data(TensorData.Matrix(dt))
        return res

    def execute(self, tn: Tensor) -> Tensor:
        m = _Marshal()
        c_tn = m.tn(tn)
        out, n_out, legs = C.c_void_p(), C.c_int(), u64_array([0] * 64)
        check(self.ctx._l.tncb_plan_execute(self.ctx.handle, self.handle, C.byref(c_tn), C.byref(out), C.byref(n_out), legs))
        for d in m.device_inputs:
            d.release()
        if not out.value:
            return Tensor()
        dt = DeviceTensor.adopt(self.ctx, out)
        res = Tensor([legs[i] for i in range(n_out.value)], dt.shape)
        res.set_tensor_data(TensorData.Matrix(dt))
        return res

    def __del__(self):
        try:
            if self.handle:
                self.ctx._l.tncb_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass
