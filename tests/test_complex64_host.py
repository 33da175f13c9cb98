"""complex64 element type, host side (no GPU): the new C ABI symbols, their argument checks, the Python dtype checks, the
marshalled tree (identical for both dtypes), the complex64 operand-bit default of K1' and the C++ mirror overloads."""
import ctypes as C
import math
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW_SYMBOLS = ["tncb_tensor_upload_dt", "tncb_tensor_alloc_dt", "tncb_tensor_dtype", "tncb_contract_tensor_network_dt",
               "tncb_plan_create_dt"]


def test_new_symbols_exported(built_lib):
    from tnc_b200._lib import SIGNATURES, TNCB_C64, TNCB_C128
    hdr = open(os.path.join(ROOT, "include", "tncb.h")).read()
    assert "TNCB_C128 = 0" in hdr and "TNCB_C64 = 1" in hdr
    assert (TNCB_C128, TNCB_C64) == (0, 1)
    for name in NEW_SYMBOLS:
        assert hasattr(built_lib, name) and name in SIGNATURES, name


def test_new_entry_points_return_statuses():
    """NULL / zero / out-of-range arguments give a status, never a crash (one child process, like the sweep over every
    symbol).  A plan can be compiled without a device (ctx = NULL): its byte counts follow the dtype."""
    code = r"""
import sys, ctypes as C
sys.path.insert(0, %r)
from tnc_b200._lib import lib, TncbTn, TncbPath, u64_array
l = lib()
out = C.c_void_p()
assert l.tncb_tensor_dtype(None) == -1
assert l.tncb_tensor_upload_dt(None, 0, None, 1, None, C.byref(out)) == -1
assert l.tncb_tensor_alloc_dt(None, 0, None, 1, C.byref(out)) == -1
assert l.tncb_tensor_alloc_dt(None, 0, None, 7, None) == -1
assert l.tncb_contract_tensor_network_dt(None, None, None, 1, None, None, None) == -1
assert l.tncb_plan_create_dt(None, None, None, 1, None) == -1
# a two-leaf network, compiled host-only in both dtypes and with a bad one
legs_a, legs_b, dims = u64_array([0, 1]), u64_array([1, 2]), u64_array([8, 8])
data = (C.c_double * 128)()
leaves = (TncbTn * 2)()
for lf, lg in zip(leaves, (legs_a, legs_b)):
    lf.rank = 2; lf.legs = lg; lf.dims = dims; lf.kind = 1; lf.host_re_im = data
tn = TncbTn(); tn.n_children = 2; tn.children = leaves
p = TncbPath(); p.n_pairs = 1; p.pairs = u64_array([0, 1])
assert l.tncb_plan_create_dt(None, C.byref(tn), C.byref(p), 2, C.byref(out)) == -1
assert l.tncb_plan_create_dt(None, C.byref(tn), C.byref(p), -1, C.byref(out)) == -1
res = {}
for dt in (0, 1):
    h = C.c_void_p()
    assert l.tncb_plan_create_dt(None, C.byref(tn), C.byref(p), dt, C.byref(h)) == 0
    n, k, pk = C.c_uint64(), C.c_uint64(), C.c_uint64(); fl, by = C.c_double(), C.c_double()
    assert l.tncb_plan_info(h, C.byref(n), C.byref(fl), C.byref(by), C.byref(pk), C.byref(k)) == 0
    res[dt] = (n.value, fl.value, by.value, pk.value)
    l.tncb_plan_destroy(h)
assert res[0][:2] == res[1][:2], res
assert res[0][2] == 2 * res[1][2] == 16 * 3 * 64, res
assert res[1][3] < res[0][3], res
print("DT_OK")
""" % ROOT
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "DT_OK" in r.stdout, (r.returncode, r.stdout[-500:], r.stderr[-1500:])


class _NoLib:
    """A context whose library must never be reached."""
    handle = None

    class _L:
        def __getattr__(self, name):
            raise AssertionError(f"{name} was called")
    _l = _L()


def _net():
    from tnc_b200.builders import random_circuit_builder
    from tnc_b200.tensornetwork import Tensor, TensorData
    tn, _ = random_circuit_builder(6, 3, 0.5, 0.5, np.random.default_rng(5)).into_amplitude_network("010101")
    extra = Tensor([10_000], [2])
    extra.set_tensor_data(TensorData.new_from_data([2], np.array([1.0 + 0.5j, -0.25j])))
    tn.push_tensor(extra)
    return tn


@pytest.mark.parametrize("bad", [np.float64, np.float32, np.complex256 if hasattr(np, "complex256") else "c32", "int8", None, "x"])
def test_other_dtypes_rejected_before_the_library(built_lib, bad):
    import tnc_b200 as tb
    from tnc_b200.contractionpath import ContractionPath
    from tnc_b200.contractionpath.slicing import SlicedPlan, contract_sliced
    from tnc_b200.tensornetwork import NetworkPlan, contract_tensor_network
    tn = _net()
    p = ContractionPath.simple([(0, i) for i in range(1, len(tn.tensors))])
    ctx = _NoLib()
    with pytest.raises(ValueError):
        contract_tensor_network(tn, p, ctx=ctx, dtype=bad)
    with pytest.raises(ValueError):
        NetworkPlan(tn, p, ctx=ctx, dtype=bad)
    with pytest.raises(ValueError):
        SlicedPlan(tn, p, [], ctx=ctx, dtype=bad)
    with pytest.raises(ValueError):
        contract_sliced(tn, p, [], ctx=ctx, dtype=bad)
    with pytest.raises(ValueError):
        tb.DeviceTensor.from_numpy(ctx, np.zeros(2), dtype=bad)
    with pytest.raises(ValueError):
        tb.DeviceTensor.empty(ctx, [2], dtype=bad)
    assert tb.dtype_code(np.complex128) == 0 and tb.dtype_code(np.complex64) == 1 and tb.dtype_code("complex64") == 1


def test_multi_rank_sliced_complex64_refused(built_lib):
    from tnc_b200.contractionpath import ContractionPath
    from tnc_b200.contractionpath.slicing import contract_sliced
    tn = _net()
    p = ContractionPath.simple([(0, i) for i in range(1, len(tn.tensors))])
    with pytest.raises(ValueError, match="complex128 only"):
        contract_sliced(tn, p, [], ctx=_NoLib(), world=2, dtype=np.complex64)


def _dump(tn_ptr):
    """Everything the C side can read from a marshalled tncb_tn tree, payload bytes included."""
    t = tn_ptr
    if t.n_children:
        return ("composite", [_dump(t.children[i]) for i in range(t.n_children)])
    legs = [t.legs[i] for i in range(t.rank)]
    dims = [t.dims[i] for i in range(t.rank)]
    payload = None
    if t.kind == 1:
        payload = C.string_at(C.cast(t.host_re_im, C.c_void_p), 16 * int(np.prod(dims, dtype=np.int64)))
    elif t.kind == 2:
        payload = (t.gate_name, [t.gate_angles[i] for i in range(t.n_gate_angles)], t.gate_adjoint)
    return (t.kind, t.rank, legs, dims, payload)


class _Capture:
    """A context whose library records the tree it is handed and reports an error (the call goes no further)."""
    handle = None

    def __init__(self):
        self.seen = []
        cap = self

        class _L:
            def tncb_contract_tensor_network_dt(self, h, tn, path, dtype, *rest):
                cap.seen.append((dtype, _dump(tn._obj)))
                return -1

            def tncb_plan_create_dt(self, h, tn, path, dtype, *rest):
                cap.seen.append((dtype, _dump(tn._obj)))
                return -1

            def __getattr__(self, name):
                from tnc_b200._lib import lib
                return getattr(lib(), name)
        self._l = _L()


def test_marshalled_tree_is_identical_for_both_dtypes(built_lib):
    import tnc_b200 as tb
    from tnc_b200.contractionpath import ContractionPath
    from tnc_b200.tensornetwork import NetworkPlan, contract_tensor_network
    tn = _net()
    p = ContractionPath.simple([(0, i) for i in range(1, len(tn.tensors))])
    cap = _Capture()
    for dt in (np.complex128, np.complex64):
        with pytest.raises(tb.TncbError):
            contract_tensor_network(tn, p, ctx=cap, dtype=dt)
        with pytest.raises(tb.TncbError):
            NetworkPlan(tn, p, ctx=cap, dtype=dt)
    assert [s[0] for s in cap.seen] == [0, 0, 1, 1]
    assert cap.seen[0][1] == cap.seen[1][1] == cap.seen[2][1] == cap.seen[3][1]
    kinds = {c[0] for c in cap.seen[0][1][1]}
    assert kinds == {1, 2}, kinds                      # gates and a host matrix travel


@pytest.mark.parametrize("log2k", range(0, 14))
def test_complex64_operand_bits(built_lib, log2k):
    """tncb_tcgen05_bound(K, K 2^-24) is what K1' does for a complex64 pair without a tolerance: a = 28 bits, bound
    2^(4-a) K = 2^-24 K, at most 10 moduli for K <= 2^13 (9 at K = 4096)."""
    import tnc_b200 as tb
    k = 2 ** log2k
    r = tb.tcgen05_bound(k, k * 2.0 ** -24)
    assert r["bits_a"] == 28 and r["bits_b"] >= 28, r
    assert r["n_moduli"] <= 10, r
    assert r["bound"] <= k * 2.0 ** -24 * (1 + 1e-12), r
    if k == 4096:
        assert r["n_moduli"] == 9, r
    assert tb.tcgen05_bound(k)["n_moduli"] > r["n_moduli"]


def test_cpp_mirror_dtype_overloads_compile(tmp_path):
    src = tmp_path / "use_dtype.cpp"
    src.write_text(r"""
#include "tnc.hpp"
void use(tnc::Context& ctx, tnc::Tensor tn, const tnc::ContractionPath& p) {
  tnc::Tensor a = tnc::contract_tensor_network(ctx, tn, p);                  // complex128, as before
  tnc::Tensor b = tnc::contract_tensor_network(ctx, tn, p, TNCB_C64);
  tnc::NetworkPlan p128(ctx, tn, p);
  tnc::NetworkPlan p64(ctx, tn, p, TNCB_C64);
  std::vector<tnc::Complex64> e = b.elements();
  (void)a; (void)e;
}
""")
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-Wall", "-I", os.path.join(ROOT, "include"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
