"""tnc_b200 -- B200-native pairwise tensor-contraction hot path of qc-tum/TNC.

Host-side mirror (Python, over the C ABI in include/tncb.h) of the reference's interface for
this path: `tensornetwork.tensor.Tensor`, `tensornetwork.tensordata.TensorData`,
`contractionpath.ContractionPath`, `tensornetwork.contraction.contract_tensor_network`,
`builders.circuit_builder.Circuit` / `Permutor`, and `dist.communication` for the
partitioned fan-in (tnc::mpi::communication).  All numerics run in libtncb200 (CUDA, sm_100a);
nothing here computes on the CPU.
"""
from __future__ import annotations

import ctypes as C
from typing import Sequence

import numpy as np

from ._lib import TNCB_C64, TNCB_C128, TncbError, check, lib, u64_array

__all__ = ["Context", "DeviceTensor", "TncbError", "contract_pair", "contract_pair_into", "default_context", "dtype_code", "lib"]

_DTYPE_CODES = {np.dtype(np.complex128): TNCB_C128, np.dtype(np.complex64): TNCB_C64}
_CODE_DTYPES = {v: k for k, v in _DTYPE_CODES.items()}


def dtype_code(dtype) -> int:
    """tncb_dtype of numpy.complex128 / numpy.complex64; any other dtype raises ValueError (before any library call)."""
    try:
        return _DTYPE_CODES[np.dtype(dtype)]
    except (TypeError, KeyError):
        raise ValueError(f"dtype must be numpy.complex128 or numpy.complex64, got {dtype!r}") from None


class Context:
    """One device + stream + arena (tncb_ctx)."""

    def __init__(self, device: int = 0, arena_bytes: int = 0):
        self._l = lib()
        h = C.c_void_p()
        check(self._l.tncb_ctx_create(device, arena_bytes, C.byref(h)))
        self.handle = h
        self.device = device

    def synchronize(self) -> None:
        check(self._l.tncb_ctx_synchronize(self.handle))

    @property
    def stream(self) -> int:
        return int(self._l.tncb_ctx_stream(self.handle) or 0)

    def stats(self) -> dict:
        a, b, c = C.c_uint64(), C.c_uint64(), C.c_uint64()
        check(self._l.tncb_ctx_stats(self.handle, C.byref(a), C.byref(b), C.byref(c)))
        return {"kernel_launches": a.value, "arena_peak_bytes": b.value, "arena_live_bytes": c.value}

    def set_tcgen05_slices(self, slices: int) -> None:
        """0: FP64 tensor pipe (DMMA).  2..8: tcgen05 int8 digit slicing (K1') for large pairs."""
        check(self._l.tncb_ctx_set_tcgen05_slices(self.handle, int(slices)))

    def set_tcgen05_engine(self, engine: int) -> None:
        """0: modular (CRT) int8 engine (default).  1: the 7-bit digit-slicing engine of round 1."""
        check(self._l.tncb_ctx_set_tcgen05_engine(self.handle, int(engine)))

    def set_tolerance(self, rel: float) -> None:
        """Normwise tolerance of K1' (0 = full FP64 mantissa), see tncb.h."""
        check(self._l.tncb_ctx_set_tolerance(self.handle, float(rel)))

    def set_tcgen05_moduli(self, n: int) -> None:
        check(self._l.tncb_ctx_set_tcgen05_moduli(self.handle, int(n)))

    def trim(self) -> dict:
        """Give unused arena slabs back to the driver (tncb_ctx_trim)."""
        f, r = C.c_uint64(), C.c_uint64()
        check(self._l.tncb_ctx_trim(self.handle, C.byref(f), C.byref(r)))
        return {"freed_bytes": f.value, "reserved_bytes": r.value}

    def set_tcgen05_products(self, products: int = 0, min_k3: int = 0) -> None:
        """3 / 4 real int8 products per complex product (0 = by K), see tncb.h; both forms give identical bits."""
        check(self._l.tncb_ctx_set_tcgen05_products(self.handle, int(products), int(min_k3)))

    def set_tcgen05_workspace(self, nbytes: int) -> None:
        check(self._l.tncb_ctx_set_tcgen05_workspace(self.handle, int(nbytes)))

    def engine_counts(self) -> dict:
        arr = (C.c_uint64 * 8)()
        check(self._l.tncb_ctx_engine_counts(self.handle, arr))
        names = ["k0", "k0_splitk", "k1_dmma", "k1_dmma_splitk", "k1_tcgen05", "k2", "permute", "reserved"]
        return {n: int(arr[i]) for i, n in enumerate(names)}

    def last_tcgen05_info(self) -> dict:
        ops, n = C.c_double(), C.c_int()
        check(self._l.tncb_ctx_last_tcgen05_info(self.handle, C.byref(ops), C.byref(n)))
        pr = C.c_int()
        check(self._l.tncb_ctx_last_tcgen05_products(self.handle, C.byref(pr)))
        return {"int8_ops": ops.value, "n_moduli": n.value, "products": pr.value}

    def set_tcgen05_threshold(self, min_tiles: int, min_k: int) -> None:
        check(self._l.tncb_ctx_set_tcgen05_threshold(self.handle, int(min_tiles), int(min_k)))

    def time_gemm(self, enable=True) -> None:
        """False/0 off, True/1 last launch of the dominant GEMM kernel, 2 accumulate every tcgen05 GEMM launch."""
        check(self._l.tncb_ctx_time_gemm(self.handle, int(enable)))

    def gemm_totals(self) -> dict:
        ms, ops, n = C.c_double(), C.c_double(), C.c_uint64()
        check(self._l.tncb_ctx_gemm_totals(self.handle, C.byref(ms), C.byref(ops), C.byref(n)))
        return {"ms": ms.value, "int8_ops": ops.value, "launches": n.value}

    def last_gemm_ms(self) -> float:
        ms = C.c_float()
        check(self._l.tncb_ctx_last_gemm_ms(self.handle, C.byref(ms)))
        return float(ms.value)

    def reset_stats(self) -> None:
        check(self._l.tncb_ctx_reset_stats(self.handle))

    def close(self) -> None:
        if getattr(self, "handle", None):
            self._l.tncb_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx = None


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


class DeviceTensor:
    """A device-resident complex128 or complex64 tensor (tncb_tensor), row-major."""

    def __init__(self, ctx: Context, handle, shape: Sequence[int], dtype=np.complex128):
        self.ctx = ctx
        self.handle = handle
        self.shape = tuple(int(s) for s in shape)
        self.dtype = np.dtype(dtype)

    @classmethod
    def from_numpy(cls, ctx: Context, arr: np.ndarray, dtype=np.complex128) -> "DeviceTensor":
        """Upload `arr` converted to `dtype` (complex128 unless complex64 is asked for explicitly)."""
        code = dtype_code(dtype)
        a = np.asarray(arr, dtype=dtype, order="C")  # (ascontiguousarray would promote 0-d to 1-d)
        h = C.c_void_p()
        check(ctx._l.tncb_tensor_upload_dt(ctx.handle, a.ndim, u64_array(a.shape), code, a.ctypes.data_as(C.c_void_p), C.byref(h)))
        return cls(ctx, h, a.shape, dtype)

    @classmethod
    def empty(cls, ctx: Context, shape: Sequence[int], dtype=np.complex128) -> "DeviceTensor":
        code = dtype_code(dtype)
        h = C.c_void_p()
        check(ctx._l.tncb_tensor_alloc_dt(ctx.handle, len(shape), u64_array(shape), code, C.byref(h)))
        return cls(ctx, h, shape, dtype)

    @classmethod
    def adopt(cls, ctx: Context, handle) -> "DeviceTensor":
        l = ctx._l
        r = l.tncb_tensor_rank(handle)
        dims = u64_array([0] * max(r, 1))
        check(l.tncb_tensor_dims(handle, dims))
        return cls(ctx, handle, [dims[i] for i in range(r)], _CODE_DTYPES[l.tncb_tensor_dtype(handle)])

    def to_numpy(self) -> np.ndarray:
        """A host copy in the tensor's own dtype."""
        if self.handle is None:
            raise TncbError(-3, "Cannot convert uncontracted tensor to data")
        out = np.empty(self.shape, dtype=self.dtype)
        check(self.ctx._l.tncb_tensor_download(self.ctx.handle, self.handle, out.ctypes.data_as(C.c_void_p)))
        return out

    def device_ptr(self) -> int:
        return int(self.ctx._l.tncb_tensor_device_ptr(self.handle) or 0)

    def release(self):
        """Give up ownership (the C side consumed the handle)."""
        h, self.handle = self.handle, None
        return h

    def free(self) -> None:
        if self.handle is not None and self.ctx.handle is not None:
            self.ctx._l.tncb_tensor_free(self.ctx.handle, self.handle)
        self.handle = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def tcgen05_bound(k: int, rel: float = 0.0, n_moduli: int = 0) -> dict:
    """Host-only: what K1' does for contraction length k (tncb_tcgen05_bound)."""
    n, a, b, bd = C.c_int(), C.c_int(), C.c_int(), C.c_double()
    check(lib().tncb_tcgen05_bound(int(k), float(rel), int(n_moduli), C.byref(n), C.byref(a), C.byref(b), C.byref(bd)))
    return {"n_moduli": n.value, "bits_a": a.value, "bits_b": b.value, "bound": bd.value}


def tcgen05_tables(n_moduli: int) -> dict:
    """Host-only: moduli and split CRT weights of K1' (tncb_tcgen05_tables)."""
    m = (C.c_int * n_moduli)()
    r1, r2 = (C.c_double * n_moduli)(), (C.c_double * n_moduli)()
    lp = C.c_double()
    check(lib().tncb_tcgen05_tables(int(n_moduli), m, r1, r2, C.byref(lp)))
    return {"moduli": list(m), "rho1": list(r1), "rho2": list(r2), "log2_product": lp.value}


def contract_pair(ctx: Context, a_legs, a, b_legs, b):
    """tetra::contract equivalent for host arrays: returns (out_legs, ndarray).
    out legs = (b \\ a) ++ (a \\ b) (contraction.rs:64, tensor.rs:463-479)."""
    da = a if isinstance(a, DeviceTensor) else DeviceTensor.from_numpy(ctx, np.asarray(a))
    db = b if isinstance(b, DeviceTensor) else DeviceTensor.from_numpy(ctx, np.asarray(b))
    out_legs = [l for l in b_legs if l not in a_legs] + [l for l in a_legs if l not in b_legs]
    h = C.c_void_p()
    check(ctx._l.tncb_contract_pair(ctx.handle, len(out_legs), u64_array(out_legs),
                                    len(a_legs), u64_array(a_legs), da.handle,
                                    len(b_legs), u64_array(b_legs), db.handle, C.byref(h)))
    da.release(); db.release()
    out = DeviceTensor.adopt(ctx, h)
    return out_legs, out.to_numpy()


def contract_pair_into(ctx: Context, a_legs, da: DeviceTensor, b_legs, db: DeviceTensor, dc: DeviceTensor) -> None:
    """Device-resident pair into a pre-allocated output (operands stay alive); asynchronous on
    the context stream."""
    check(ctx._l.tncb_contract_pair_into(ctx.handle, len(a_legs), u64_array(a_legs), da.handle,
                                         len(b_legs), u64_array(b_legs), db.handle, dc.handle))


def contract_pair_host(ctx: Context, a_legs, a: np.ndarray, b_legs, b: np.ndarray, out: np.ndarray) -> None:
    """Pipelined host-buffer pair (tncb_contract_pair_host): asynchronous; `out` (C-contiguous complex128 with
    prod(out dims) elements, ideally pinned like a and b) is valid after ctx.synchronize()."""
    check(ctx._l.tncb_contract_pair_host(ctx.handle, len(a_legs), u64_array(a_legs), u64_array(a.shape), a.ctypes.data_as(C.c_void_p),
                                         len(b_legs), u64_array(b_legs), u64_array(b.shape), b.ctypes.data_as(C.c_void_p),
                                         out.ctypes.data_as(C.c_void_p)))


def upload_into(ctx: Context, host: np.ndarray, dst: DeviceTensor) -> None:
    """Asynchronous H2D of a (pinned) host array into an existing device tensor."""
    check(ctx._l.tncb_tensor_write(ctx.handle, dst.handle, host.ctypes.data_as(C.c_void_p)))


def download_into(ctx: Context, src: DeviceTensor, host: np.ndarray) -> None:
    """Asynchronous D2H into a (pinned) host array; synchronise the context before reading."""
    check(ctx._l.tncb_tensor_read(ctx.handle, src.handle, host.ctypes.data_as(C.c_void_p)))
