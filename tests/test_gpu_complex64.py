"""complex64 on the device: f32 in, f64 inside, one rounding out.

Bit-exactness: K0, K0 split-K, K0-batch, K1 (DMMA), K1 split-K and K2 pick their configuration from the pair alone, so
their complex64 result equals complex64(complex128 kernel on the widened operands) bit for bit.
K1' (CRT): a = 28 operand bits -> |C - C_exact| <= 2^-24 K max|b[n,:]| max|a[m,:]|, plus the final rounding 2^-24 |C|.
Networks: every pair adds at most one complex64 rounding (2^-24 relative) on top of errors that the contraction
propagates with the gain of the network; for the amplitudes below the derived allowance is rel 1e-4 (single amplitude)
and 1e-5 normwise (statevector).  Observed errors are printed (run with -s)."""
import ctypes as C
import json
import os
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = 2.0 ** -24


def rand64(rng, shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)


def bits_equal(x, y):
    x, y = np.ascontiguousarray(x), np.ascontiguousarray(y)
    return x.dtype == y.dtype and x.shape == y.shape and np.array_equal(x.view(np.uint32), y.view(np.uint32))


def pair(ctx, a_legs, a, b_legs, b, dtype):
    import tnc_b200 as tb
    da = tb.DeviceTensor.from_numpy(ctx, a, dtype=dtype)
    db = tb.DeviceTensor.from_numpy(ctx, b, dtype=dtype)
    legs, out = tb.contract_pair(ctx, a_legs, da, b_legs, db)
    return legs, out


# (name, a legs, a dims, b legs, b dims, engine counter): permuted and interleaved legs, ragged tiles
PAIRS = [
    ("k0", [0, 1, 2], [3, 5, 7], [2, 3, 1], [7, 4, 5], "k0"),
    ("k0_splitk", [0, 1, 2], [2, 64, 64], [1, 2, 3], [64, 64, 3], "k0_splitk"),
    ("k1_dmma", [0, 1, 2, 3], [8, 12, 10, 6], [3, 4, 1, 5], [6, 9, 12, 7], "k1_dmma"),
    ("k1_splitk", [0, 1, 2], [32, 64, 64], [2, 3, 1], [64, 48, 64], "k1_dmma_splitk"),
    ("k2_big_a", [0, 1, 2, 3], [16, 16, 16, 4], [3, 4], [4, 3], "k2"),
    ("k2_big_b", [5, 3], [4, 4], [3, 0, 1, 2], [4, 16, 8, 33], "k2"),
]


@pytest.mark.parametrize("name,al,ad,bl,bd,engine", PAIRS, ids=[p[0] for p in PAIRS])
def test_pair_bit_exact(ctx, name, al, ad, bl, bd, engine):
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    a, b = rand64(rng, ad), rand64(rng, bd)
    ctx.reset_stats()
    legs64, got = pair(ctx, al, a, bl, b, np.complex64)
    ec = ctx.engine_counts()
    assert ec[engine] == 1 and sum(ec.values()) == 1, ec
    legs128, ref = pair(ctx, al, a.astype(np.complex128), bl, b.astype(np.complex128), np.complex128)
    assert legs64 == legs128 and got.dtype == np.complex64 and ref.dtype == np.complex128
    assert bits_equal(got, ref.astype(np.complex64)), (name, np.abs(got - ref).max())


def test_k0_batch_bit_exact_through_a_plan(ctx):
    """A complex64 plan batches the tiny pairs of each tree level into one k0_batch_kernel launch; its result equals the
    pair-by-pair executor (the first, uncached call of contract_tensor_network) bit for bit, and that executor runs the
    single-pair K0 kernel checked above."""
    from tnc_b200.builders import random_circuit_builder
    from tnc_b200.tensornetwork import NetworkPlan, contract_tensor_network
    from test_gpu_networks import greedy
    tn, _ = random_circuit_builder(12, 6, 0.5, 0.5, np.random.default_rng(9)).into_amplitude_network("0" * 12)
    path = greedy(tn)
    plan = NetworkPlan(tn, path, ctx=ctx, dtype=np.complex64)
    info = plan.info()
    assert info["kernels"] < info["pairs"], info           # batched
    got = plan.execute(tn).to_numpy()
    eager = contract_tensor_network(tn, path, ctx=ctx, dtype=np.complex64).to_numpy()
    assert got.dtype == np.complex64 and bits_equal(got, eager), (got, eager)
    ref = complex(contract_tensor_network(tn, path, ctx=ctx).to_numpy())
    print(f"12q amplitude: complex64 {complex(got)} complex128 {ref} rel {abs(complex(got) - ref) / abs(ref):.2e}")
    assert abs(complex(got) - ref) <= 1e-4 * abs(ref)


def _crt_check(ctx, al, a, bl, b, k, expect_moduli):
    import torch
    ctx.reset_stats()
    legs, got = pair(ctx, al, a, bl, b, np.complex64)
    ec = ctx.engine_counts()
    info = ctx.last_tcgen05_info()
    assert ec["k1_tcgen05"] == 1, ec
    assert info["n_moduli"] == expect_moduli, info
    # oracle: complex128 GEMM of the widened operands on the device (torch), C[N..., M...]
    at = torch.from_numpy(a.astype(np.complex128)).cuda()
    bt = torch.from_numpy(b.astype(np.complex128)).cuda()
    letters = {l: chr(97 + i) for i, l in enumerate(sorted(set(al) | set(bl)))}
    eq = "".join(letters[l] for l in al) + "," + "".join(letters[l] for l in bl) + "->" + "".join(letters[l] for l in legs)
    ref = torch.einsum(eq, at, bt).cpu().numpy()
    # row maxima (max over re / im) of Bt[n, :] and At[m, :]
    shared = [l for l in al if l in bl]
    amax = np.maximum(np.abs(a.real), np.abs(a.imag)).astype(np.float64).max(axis=tuple(al.index(l) for l in shared))
    bmax = np.maximum(np.abs(b.real), np.abs(b.imag)).astype(np.float64).max(axis=tuple(bl.index(l) for l in shared))
    amax, bmax = amax.reshape(-1), bmax.reshape(-1)      # (free legs keep their operand order: M and N of the GEMM view)
    bound = EPS * k * np.outer(bmax, amax).reshape(got.shape)
    bound_re = bound + EPS * np.abs(ref.real)
    bound_im = bound + EPS * np.abs(ref.imag)
    d = got.astype(np.complex128) - ref
    ratio = max((np.abs(d.real) / bound_re).max(), (np.abs(d.imag) / bound_im).max())
    print(f"K1' complex64 K={k}: {info['n_moduli']} moduli, max |err| / bound = {ratio:.3f}")
    assert ratio <= 1.0, ratio
    return info


def test_k1prime_c2_pair(ctx):
    """The C2 pair (4^6 x 4^6 x 4^6, both operands permuted) on the CRT engine with its complex64 default."""
    import tnc_b200 as tb
    from bench import c2_problem
    al, ad, bl, bd = c2_problem()
    rng = np.random.default_rng(2)
    a, b = rand64(rng, ad), rand64(rng, bd)
    k = 4 ** 6
    _crt_check(ctx, al, a, bl, b, k, tb.tcgen05_bound(k, k * EPS)["n_moduli"])


@pytest.mark.parametrize("log2k", [14, 15, 16])
def test_k1prime_long_k_with_engine_1(ctx, log2k):
    """Engine 1 (digit slicing) has no complex64 path: complex64 pairs still take the CRT engine."""
    import tnc_b200 as tb
    k = 2 ** log2k
    rng = np.random.default_rng(log2k)
    a = rand64(rng, [k, 256])            # legs (k, m): K first
    b = rand64(rng, [256, k])            # legs (n, k)
    try:
        ctx.set_tcgen05_engine(1)
        _crt_check(ctx, [1, 0], a, [2, 1], b, k, tb.tcgen05_bound(k, k * EPS)["n_moduli"])
    finally:
        ctx.set_tcgen05_engine(0)


def test_exact_kernels(ctx):
    import tnc_b200 as tb
    from tnc_b200._lib import check
    rng = np.random.default_rng(11)
    x = rand64(rng, [8, 33, 16, 9])
    for perm in ([3, 1, 0, 2], [2, 3, 0, 1], [1, 0, 2, 3]):
        d = tb.DeviceTensor.from_numpy(ctx, x, dtype=np.complex64)
        out = C.c_void_p()
        parr = (C.c_int * 4)(*perm)
        ctx.reset_stats()
        check(ctx._l.tncb_permute(ctx.handle, d.handle, parr, C.byref(out)))
        d.release()
        assert ctx.engine_counts()["permute"] == 1
        got = tb.DeviceTensor.adopt(ctx, out).to_numpy()
        assert bits_equal(got, np.transpose(x, perm)), perm
    d = tb.DeviceTensor.from_numpy(ctx, x, dtype=np.complex64)
    check(ctx._l.tncb_conjugate(ctx.handle, d.handle))
    assert bits_equal(d.to_numpy(), np.conj(x))
    y = rand64(rng, x.shape)
    dy = tb.DeviceTensor.from_numpy(ctx, y, dtype=np.complex64)
    check(ctx._l.tncb_tensor_add(ctx.handle, d.handle, dy.handle))
    assert bits_equal(d.to_numpy(), np.conj(x) + y)


def test_reference_kats_in_complex64(ctx, kat):
    for x, y, xy in (("A", "B", "AxB"), ("B", "C", "BxC")):
        a, b = np.asarray(kat[x]["data"]), np.asarray(kat[y]["data"])
        legs, got = pair(ctx, kat[x]["legs"], a, kat[y]["legs"], b, np.complex64)
        assert legs == kat[xy]["legs"] and got.dtype == np.complex64
        k = int(np.prod([d for l, d in zip(kat[x]["legs"], a.shape) if l in kat[y]["legs"]]))
        tol = 4 * EPS * (k + 1) * np.abs(a).max() * np.abs(b).max()
        err = np.abs(got - np.asarray(kat[xy]["data"])).max()
        print(f"KAT {xy} complex64: err {err:.2e} tol {tol:.2e}")
        assert err <= tol


def _amp_pair(ctx, tn, path, label):
    from tnc_b200.tensornetwork import contract_tensor_network
    ctx.reset_stats()
    a64 = contract_tensor_network(tn, path, ctx=ctx, dtype=np.complex64).to_numpy()
    ec = ctx.engine_counts()
    a128 = contract_tensor_network(tn, path, ctx=ctx).to_numpy()
    rel = abs(complex(a64) - complex(a128)) / abs(complex(a128))
    print(f"{label}: complex64 {complex(a64)} complex128 {complex(a128)} rel {rel:.3e} engines {ec}")
    assert a64.dtype == np.complex64
    return rel


def test_config3_network(ctx):
    from tnc_b200.builders import random_circuit
    from test_gpu_networks import greedy
    tn = random_circuit(24, 12, 0.5, 0.5, np.random.default_rng(1))
    assert _amp_pair(ctx, tn, greedy(tn), "config 3 (24q)") <= 1e-4


def test_bench_network(ctx):
    from bench import build_network, greedy_path
    tn = build_network()
    assert _amp_pair(ctx, tn, greedy_path(tn), "36q bench network") <= 1e-4


def test_sycamore53_d10(ctx):
    from tnc_b200.builders import sycamore_circuit
    from tnc_b200.contractionpath import ContractionPath
    d = json.load(open(os.path.join(ROOT, "bench_inputs", "sycamore53_d10.json")))
    assert not d["sliced_legs"]
    tn = sycamore_circuit(53, 10, np.random.default_rng(1)).into_amplitude_network("0" * 53)[0]
    path = ContractionPath.simple([tuple(x) for x in d["toplevel"]])
    assert _amp_pair(ctx, tn, path, "Sycamore-53 depth 10") <= 1e-4


def test_statevector_normwise(ctx):
    from tnc_b200.builders import random_circuit_builder
    from tnc_b200.tensornetwork import contract_tensor_network
    from test_gpu_networks import greedy
    tn, _ = random_circuit_builder(10, 8, 0.5, 0.5, np.random.default_rng(12)).into_statevector_network()
    path = greedy(tn)
    s64 = contract_tensor_network(tn, path, ctx=ctx, dtype=np.complex64).to_numpy()
    s128 = contract_tensor_network(tn, path, ctx=ctx).to_numpy()
    rel = np.linalg.norm((s64 - s128).ravel()) / np.linalg.norm(s128.ravel())
    print(f"10q statevector: normwise rel {rel:.3e}")
    assert s64.dtype == np.complex64 and rel <= 1e-5


def test_plan_replay_and_sliced(ctx):
    from tnc_b200.builders import random_circuit, random_circuit_builder
    from tnc_b200.contractionpath.slicing import SlicedPlan, find_slices
    from tnc_b200.tensornetwork import NetworkPlan, contract_tensor_network
    from test_gpu_networks import greedy
    c = random_circuit_builder(14, 8, 0.5, 0.5, np.random.default_rng(21))
    tn, _ = c.into_amplitude_network("0" * 14)
    path = greedy(tn)
    plan = NetworkPlan(tn, path, ctx=ctx, dtype=np.complex64)
    for bits in ["0" * 14, "1" * 14, "01" * 7]:
        t2, _ = random_circuit_builder(14, 8, 0.5, 0.5, np.random.default_rng(21)).into_amplitude_network(bits)
        replay = plan.execute(t2).to_numpy()
        eager = contract_tensor_network(t2, path, ctx=ctx, dtype=np.complex64).to_numpy()
        assert bits_equal(replay, eager), (bits, replay, eager)
    plan.stage(tn)
    assert bits_equal(plan.run().to_numpy(), plan.execute(tn).to_numpy())
    tn = random_circuit(16, 8, 0.5, 0.5, np.random.default_rng(3))
    p = greedy(tn)
    flat = complex(contract_tensor_network(tn, p, ctx=ctx, dtype=np.complex64).to_numpy())
    legs = find_slices(tn, p, min_slices=8)
    sp = SlicedPlan(tn, p, legs, ctx=ctx, dtype=np.complex64)
    got = sp.run().to_numpy()
    assert got.dtype == np.complex64
    rel = abs(complex(got) - flat) / abs(flat)
    print(f"sliced ({sp.n_slices} slices) vs flat, complex64: rel {rel:.3e}")
    assert rel <= 1e-5


def test_refusals(ctx):
    import tnc_b200 as tb
    from tnc_b200.tensornetwork import Tensor, TensorData, contract_tensor_network
    from tnc_b200.contractionpath import ContractionPath
    l = ctx._l
    rng = np.random.default_rng(0)
    a64 = tb.DeviceTensor.from_numpy(ctx, rand64(rng, [4, 4]), dtype=np.complex64)
    b128 = tb.DeviceTensor.from_numpy(ctx, rand64(rng, [4, 4]))
    out = C.c_void_p()
    from tnc_b200._lib import u64_array
    assert l.tncb_contract_pair_keep(ctx.handle, 2, u64_array([0, 1]), a64.handle, 2, u64_array([1, 2]), b128.handle, C.byref(out)) == -1
    c64 = tb.DeviceTensor.empty(ctx, [4, 4], dtype=np.complex64)
    assert l.tncb_contract_pair_into(ctx.handle, 2, u64_array([0, 1]), b128.handle, 2, u64_array([1, 2]), b128.handle, c64.handle) == -1
    assert l.tncb_tensor_add(ctx.handle, a64.handle, b128.handle) == -1
    # a device leaf of the wrong dtype: refused, and still owned by the caller
    x, y = Tensor([0, 1], [4, 4]), Tensor([1, 2], [4, 4])
    x.set_tensor_data(TensorData.Matrix(a64))
    y.set_tensor_data(TensorData.new_from_data([4, 4], rand64(rng, [4, 4]).astype(np.complex128).reshape(-1)))
    with pytest.raises(tb.TncbError) as e:
        contract_tensor_network(Tensor.new_composite([x, y]), ContractionPath.single(0, 1), ctx=ctx)
    assert e.value.status == -1 and a64.handle is not None
    res = contract_tensor_network(Tensor.new_composite([x, y]), ContractionPath.single(0, 1), ctx=ctx, dtype=np.complex64)
    assert res.to_numpy().dtype == np.complex64
    assert l.tncb_comm_send(ctx.handle, c64.handle, 0) == -9
    assert l.tncb_comm_allreduce_sum(ctx.handle, c64.handle) == -9


def test_default_dtype_unchanged(ctx):
    """The complex128 network through tncb_contract_tensor_network_dt(..., TNCB_C128) equals the existing call bit for bit."""
    from tnc_b200.builders import random_circuit
    from tnc_b200.tensornetwork.contraction import _Marshal
    from tnc_b200._lib import check, u64_array
    import tnc_b200 as tb
    from test_gpu_networks import greedy
    tn = random_circuit(16, 8, 0.5, 0.5, np.random.default_rng(8))
    p = greedy(tn)
    res = []
    for dt in (None, 0):
        m = _Marshal()
        c_tn, c_path = m.tn(tn), m.path(p)
        out, n_out, legs = C.c_void_p(), C.c_int(), u64_array([0] * 64)
        if dt is None:
            check(ctx._l.tncb_contract_tensor_network(ctx.handle, C.byref(c_tn), C.byref(c_path), C.byref(out), C.byref(n_out), legs))
        else:
            check(ctx._l.tncb_contract_tensor_network_dt(ctx.handle, C.byref(c_tn), C.byref(c_path), dt, C.byref(out), C.byref(n_out), legs))
        res.append(tb.DeviceTensor.adopt(ctx, out).to_numpy())
    assert res[0].dtype == np.complex128 and bits_equal(res[0], res[1])
