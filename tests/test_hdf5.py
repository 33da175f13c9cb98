"""HDF5 tensor files (tnc/src/io/hdf5.rs) through the C ABI (tncb_hdf5_*, csrc/hdf5io.cpp) -- host only, no GPU.

Pinning, since neither libhdf5 nor a byte-level fixture of the reference exists here:
  * a file written by libhdf5 itself (tests/golden/testhdf5_7.4_GLNX86.mat, SciPy 1.18.1's BSD-licensed MATLAB-7.3 test
    fixture scipy/io/matlab/tests/data/testhdf5_7.4_GLNX86.mat, stored verbatim) is read correctly;
  * the writer's output is walked by an independent pure-Python restatement of the format (tests/h5check.py::parse_v0),
    which asserts what libhdf5 relies on when it opens such a file;
  * files emitted by a second independent builder in the encodings of newer libhdf5 objects (h5check.LatestFile) are read
    correctly;
  * the reference's own three tests (hdf5.rs:196-257) are replayed through writer + reader."""
import ctypes as C
import os
import struct
import subprocess
import sys

import numpy as np
import pytest

import h5check

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBHDF5_FIXTURE = os.path.join(ROOT, "tests", "golden", "testhdf5_7.4_GLNX86.mat")


@pytest.fixture(scope="module")
def h5(built_lib):
    from tnc_b200.io import hdf5
    return hdf5


def cplx(rng, shape):
    return rng.uniform(-1, 1, shape) + 1j * rng.uniform(-1, 1, shape)


# ---------------------------------------------------------------- a file libhdf5 wrote
def test_reads_a_file_written_by_libhdf5(h5):
    """512-byte user block, superblock 0 with a base address, symbol-table root group, version-1 object header with a
    version-1 fill value, version-2 data layout, IEEE f64 dataset 0:pi/4:2pi of shape (9, 1)."""
    with h5.Hdf5File(LIBHDF5_FIXTURE, "/") as f:
        assert f.member_names() == ["testdouble"]
        assert f.shape(0) == [9, 1]
        got = f.read(0)
    assert got.dtype == np.complex128
    np.testing.assert_array_equal(got.imag, 0)
    np.testing.assert_allclose(got.real.ravel(), np.arange(9) * np.pi / 4, rtol=0, atol=1e-15)
    # the same file has no /tensors group
    from tnc_b200 import TncbError
    with pytest.raises(TncbError) as e:
        h5.load_data(LIBHDF5_FIXTURE)
    assert e.value.status == -10 and "tensors" in str(e.value)


# ---------------------------------------------------------------- the reference's tests (hdf5.rs:196-257)
REF_DATA = np.array([[1.0 + 0j, 2j], [3.0 + 0j, 1j]])


def test_load_data(h5, tmp_path):
    """hdf5.rs:196-212 (create_hdf5_data: /tensors/-1 = [[1, 2i], [3, i]])."""
    p = tmp_path / "data.h5"
    h5.store_tensor(p, [], [])          # an empty network first: only the output tensor
    assert h5.Hdf5File(p).member_names() == ["-1"]
    h5.store_data(p, REF_DATA)
    got = h5.load_data(p)
    assert got.shape == (2, 2)
    np.testing.assert_array_equal(got, REF_DATA)


def test_load_tensor(h5, tmp_path):
    """hdf5.rs:214-236 (create_hdf5_tensor: "-1" without data, bids [0, 1]; "0" = the matrix, bids [0, 1])."""
    p = tmp_path / "tensor.h5"
    h5.store_tensor(p, [("0", [0, 1], REF_DATA)], [0, 1])
    tn = h5.load_tensor(p)
    assert tn.legs == [0, 1]
    assert len(tn.tensors) == 1
    t = tn.tensors[0]
    assert t.legs == [0, 1] and t.bond_dims == [2, 2] and t.tensordata.kind == "matrix"
    np.testing.assert_array_equal(t.tensordata.matrix, REF_DATA)


def test_write_read(h5, tmp_path):
    """hdf5.rs:238-257."""
    data = np.array([1.0, -2j, -3.0, -2 - 1j, 0, 0.5 + 2j]).reshape(2, 3)
    h5.store_data(tmp_path / "wr.h5", data)
    np.testing.assert_array_equal(h5.load_data(tmp_path / "wr.h5"), data)


# ---------------------------------------------------------------- writer output under an independent parser
@pytest.mark.parametrize("n", [0, 1, 8, 9, 100, 257, 1053, 2100])
def test_writer_output_is_well_formed(h5, tmp_path, n):
    """1053 = the leaves of the Sycamore-53 depth-12 network; 2100 members need a three-level B-tree (8 per symbol node,
    32 per B-tree node)."""
    rng = np.random.default_rng(n)
    tensors = []
    for i in range(n):
        rank = int(rng.integers(0, 5))
        shape = [int(rng.integers(1, 4)) for _ in range(rank)]
        tensors.append((str(i), [int(x) for x in rng.integers(0, 1 << 40, rank)], cplx(rng, shape)))
    out_legs = [int(x) for x in rng.integers(0, 1 << 40, 3)]
    p = tmp_path / "net.h5"
    h5.store_tensor(p, tensors, out_legs)
    raw = open(p, "rb").read()
    info = h5check.parse_v0(raw)
    assert sorted(info) == sorted([t[0] for t in tensors] + ["-1"])
    assert info["-1"]["bids"] == out_legs and info["-1"]["data_addr"] == h5check.UNDEF
    for name, bids, arr in tensors:
        i = info[name]
        assert i["shape"] == list(arr.shape) and i["bids"] == bids
        got = np.frombuffer(raw, dtype=np.complex128, count=arr.size, offset=i["data_addr"]).reshape(arr.shape)
        np.testing.assert_array_equal(got, arr)
    # and back through the reader: members come in strcmp order (Group::member_names), not numeric order
    tn = h5.load_tensor(p)
    order = sorted((t[0] for t in tensors), key=lambda s: s.encode())
    assert tn.legs == out_legs and len(tn.tensors) == n
    by_name = {t[0]: t for t in tensors}
    for got, name in zip(tn.tensors, order):
        _, bids, arr = by_name[name]
        assert got.legs == bids and got.bond_dims == list(arr.shape)
        np.testing.assert_array_equal(got.tensordata.matrix, arr)


def test_writer_rejects_bad_names(h5, tmp_path):
    from tnc_b200 import TncbError
    with pytest.raises(TncbError):
        h5.store_tensor(tmp_path / "x.h5", [("a/b", [0], np.zeros(2))], [])
    with pytest.raises(TncbError):
        h5.store_tensor(tmp_path / "x.h5", [("a", [0], np.zeros(2)), ("a", [1], np.zeros(2))], [])
    with pytest.raises(TncbError) as e:
        h5.store_data(tmp_path / "no_such_dir" / "x.h5", np.zeros(2))
    assert e.value.status == -10


# ---------------------------------------------------------------- reader on the encodings of newer libhdf5 objects
def _latest_file(rng, userblock=0):
    """/tensors with: "-1" (null dataspace, i32 bids, as `empty::<Complex64>()` + `array![0, 1]` give, hdf5.rs:146-152),
    "a" contiguous {r, i} f64, "b" compact big-endian f32 compound with an i16 big-endian attribute, "c" chunked 5 x 7 in
    2 x 4 chunks with shuffle + deflate (edge chunks clipped), header split by a continuation block,
    "d" chunked without filters, one chunk missing (reads as zeros)."""
    F = h5check.LatestFile(userblock)
    a = cplx(rng, (3, 4))
    b = cplx(rng, (2, 2, 2)).astype(np.complex64)
    c = cplx(rng, (5, 7))
    d = cplx(rng, (4, 4))
    ty = h5check._complex_type_v3()
    ds = {}
    ds["-1"] = F.dataset(None, ty, bytes([3, 1]) + struct.pack("<QQ", h5check.UNDEF, 0), attrs=[h5check._attr_v3("bids", [0, 1], 4, True)])
    ds["a"] = F.dataset(a.shape, ty, F.contiguous(a.tobytes()), attrs=[h5check._attr_v3("bids", [7, 1 << 33, 2, 5][:2], 8, False),
                                                                       h5check._attr_v3("tids", [-1], 8, True)])
    b_be = b.astype(">c8").tobytes()
    ds["b"] = F.dataset(b.shape, h5check._complex_type_v3(("re", "im"), 4, big=True), F.compact(b_be),
                        attrs=[h5check._attr_v3("bids", [300, 2, 1], 2, True, big=True)])
    chunks = []
    for i in range(0, 5, 2):
        for j in range(0, 7, 4):
            blk = np.zeros((2, 4), dtype=np.complex128)
            sub = c[i:i + 2, j:j + 4]
            blk[:sub.shape[0], :sub.shape[1]] = sub
            chunks.append(((i, j), h5check.deflate(h5check.shuffle(blk.tobytes(), 16)), 0))
    ds["c"] = F.dataset(c.shape, ty, F.chunked(c.shape, (2, 4), 16, chunks), attrs=[h5check._attr_v3("bids", [4, 9], 1, False)],
                        filters=h5check.filters_v2(True, 16), split=True)
    d_expect = d.copy()
    d_expect[2:, :2] = 0
    chunks = [((i, j), np.ascontiguousarray(d[i:i + 2, j:j + 2]).tobytes(), 0) for i in (0, 2) for j in (0, 2) if (i, j) != (2, 0)]
    ds["d"] = F.dataset(d.shape, ty, F.chunked(d.shape, (2, 2), 16, chunks), attrs=[h5check._attr_v3("bids", [1, 2], 8, False)])
    tensors = F.group(sorted(ds.items(), reverse=True))          # link order in the header is not name order
    root = F.group([("tensors", tensors)])
    return F.finish(root), {"a": a, "b": b.astype(np.complex128), "c": c, "d": d_expect}


@pytest.mark.parametrize("userblock", [0, 1024])
def test_reader_handles_newer_encodings(h5, tmp_path, userblock):
    raw, expect = _latest_file(np.random.default_rng(5), userblock)
    p = tmp_path / "latest.h5"
    p.write_bytes(raw)
    with h5.Hdf5File(p) as f:
        assert f.member_names() == ["-1", "a", "b", "c", "d"]
        assert f.attr(0, "bids") == [0, 1]
        assert f.attr(1, "bids") == [7, 1 << 33] and f.attr(1, "tids") == [-1]
        assert f.attr(2, "bids") == [300, 2, 1]
        assert f.attr(3, "bids") == [4, 9]
        for i, k in enumerate("abcd", start=1):
            assert f.shape(i) == list(expect[k].shape)
            np.testing.assert_array_equal(f.read(i), expect[k])
    tn = h5.load_tensor(p)
    assert tn.legs == [0, 1] and [t.legs for t in tn.tensors] == [[7, 1 << 33], [300, 2, 1], [4, 9], [1, 2]]
    assert h5.load_data(p).size == 0                                   # first member is "-1": null dataspace, no data


def test_foreign_attributes_are_skipped(h5, tmp_path):
    """an attribute of a type outside the subset (here a variable-length string, as h5py writes for str attributes) next
    to `bids` does not make the dataset unreadable"""
    F = h5check.LatestFile()
    a = (np.arange(6) + 1j).reshape(2, 3)
    vlen = bytes([0x19, 0x01, 0, 0]) + struct.pack("<I", 16) + bytes([0x13, 0, 0, 0]) + struct.pack("<I", 1)
    nm, sp = b"note\0", h5check._space_v2([])
    attr = bytes([3, 0]) + struct.pack("<HHH", len(nm), len(vlen), len(sp)) + b"\0" + nm + vlen + sp + b"\0" * 16
    ds = F.dataset(a.shape, h5check._complex_type_v3(), F.contiguous(a.tobytes()), attrs=[attr, h5check._attr_v3("bids", [3, 4], 8, False)])
    p = tmp_path / "vlen.h5"
    p.write_bytes(F.finish(F.group([("tensors", F.group([("0", ds)]))])))
    with h5.Hdf5File(p) as f:
        assert f.member_names() == ["0"] and f.attr(0, "bids") == [3, 4]
        np.testing.assert_array_equal(f.read(0), a)
        from tnc_b200 import TncbError
        with pytest.raises(TncbError):
            f.attr(0, "note")                       # skipped, hence absent


def test_unsupported_features_are_named(h5, tmp_path):
    """dense link storage (fractal heap address defined) -> TNCB_ERR_UNSUPPORTED, not a wrong answer"""
    from tnc_b200 import TncbError
    F = h5check.LatestFile()
    dense = F.object_header([h5check._msg_v2(0x02, bytes([0, 0]) + struct.pack("<QQ", 4096, 8192))])
    root = F.group([("tensors", dense)])
    p = tmp_path / "dense.h5"
    p.write_bytes(F.finish(root))
    with pytest.raises(TncbError) as e:
        h5.Hdf5File(p)
    assert e.value.status == -9 and "dense link storage" in str(e.value)


def test_cyclic_btree_is_an_error(h5, tmp_path):
    """a B-tree child pointer bent back to its parent (300 members: a two-level tree) is reported, not followed forever"""
    from tnc_b200 import TncbError
    p = tmp_path / "cyc.h5"
    h5.store_tensor(p, [(str(i), [i], np.zeros(1)) for i in range(300)], [])
    raw = bytearray(p.read_bytes())
    roots = [i for i in range(0, len(raw) - 8, 8) if raw[i:i + 4] == b"TREE" and raw[i + 4] == 0 and raw[i + 5] == 1]
    assert len(roots) == 1                                           # the level-1 root of /tensors
    r = roots[0]
    raw[r + 24 + 8:r + 24 + 16] = struct.pack("<Q", r)               # child 0 := the root itself
    p.write_bytes(bytes(raw))
    with pytest.raises(TncbError) as e:
        h5.Hdf5File(p)
    assert e.value.status == -10 and "B-tree" in str(e.value)


def test_not_hdf5_and_missing(h5, tmp_path):
    from tnc_b200 import TncbError
    p = tmp_path / "junk.h5"
    p.write_bytes(b"not an hdf5 file at all" * 100)
    for path in (p, tmp_path / "missing.h5"):
        with pytest.raises(TncbError) as e:
            h5.load_data(path)
        assert e.value.status == -10


# ---------------------------------------------------------------- TensorData::File.into_data (tensordata.rs:43-49)
def _load_leaf(lib, path, adjoint, dims):
    from tnc_b200._lib import check, u64_array
    out = np.empty(dims, dtype=np.complex128)
    check(lib.tncb_hdf5_load_leaf(os.fsencode(path), int(adjoint), len(dims), u64_array(dims), out.ctypes.data))
    return out


def test_file_leaf_into_data(h5, built_lib, tmp_path):
    from oracle import tnc_oracle as orc
    from tnc_b200 import TncbError
    rng = np.random.default_rng(11)
    for shape in [(), (4, 4), (2, 2, 2, 2), (2, 3, 3, 2), (2, 2, 2, 2, 2, 2, 2, 2)]:
        a = cplx(rng, shape)
        p = tmp_path / "leaf.h5"
        h5.store_data(p, a)
        np.testing.assert_array_equal(_load_leaf(built_lib, p, False, list(shape)), a)
        r = len(shape)
        adj = np.conj(np.transpose(a, list(range(r // 2, r)) + list(range(r // 2)))) if r else np.conj(a)
        np.testing.assert_array_equal(_load_leaf(built_lib, p, True, list(adj.shape)), adj)
        if r:   # the oracle's adjoint rule (gates.rs:82-99), pinned by the reference's adjoint identity KAT
            np.testing.assert_array_equal(adj, orc.matrix_adjoint(a))
    # adjoint of a rank that is no power of two: `assert!(data.ndim().is_power_of_two())` (gates.rs:84)
    h5.store_data(tmp_path / "r3.h5", cplx(rng, (2, 2, 2)))
    with pytest.raises(TncbError) as e:
        _load_leaf(built_lib, tmp_path / "r3.h5", True, [2, 2, 2])
    assert e.value.status == -2
    # the file's shape must be the leaf's bond dimensions
    h5.store_data(tmp_path / "m.h5", cplx(rng, (2, 8)))
    with pytest.raises(TncbError) as e:
        _load_leaf(built_lib, tmp_path / "m.h5", False, [4, 4])
    assert e.value.status == -2
    np.testing.assert_array_equal(_load_leaf(built_lib, tmp_path / "m.h5", True, [8, 2]).shape, (8, 2))


def test_oracle_reader_agrees(h5, tmp_path):
    """the oracle's own File-leaf reader (oracle.load_data_hdf5, shares no code with csrc/hdf5io.cpp) returns what the
    library returns, also behind a three-level group B-tree, and the oracle's File payload applies the adjoint rule"""
    from oracle import tnc_oracle as orc
    rng = np.random.default_rng(8)
    a = cplx(rng, (2, 3, 2, 3))
    h5.store_data(tmp_path / "a.h5", a)
    np.testing.assert_array_equal(orc.load_data_hdf5(tmp_path / "a.h5"), a)
    np.testing.assert_array_equal(orc.load_data_hdf5(tmp_path / "a.h5"), h5.load_data(tmp_path / "a.h5"))
    t = orc.OTensor([0, 1, 2, 3], [2, 3, 2, 3], ("file", str(tmp_path / "a.h5"), True))
    np.testing.assert_array_equal(t.materialise(), np.conj(np.transpose(a, [2, 3, 0, 1])))
    many = [(str(i), [i], cplx(rng, (2,))) for i in range(2100)]
    h5.store_tensor(tmp_path / "many.h5", many, [0])
    assert orc.load_data_hdf5(tmp_path / "many.h5").shape == ()              # "-1" sorts first: declared, never written
    h5.store_tensor(tmp_path / "many.h5", many[5:], [0])                      # now "-1" ... still first
    with h5.Hdf5File(tmp_path / "many.h5") as f:
        first_with_data = f.member_names()[1]
    assert first_with_data == "10"


def test_file_tensordata_mirror(h5):
    from tnc_b200.tensornetwork.tensordata import TensorData
    td = TensorData.File("x.h5", False)
    assert td.adjoint().file == ("x.h5", True) and td.adjoint().adjoint().file == ("x.h5", False)   # tensordata.rs:65


# ---------------------------------------------------------------- malformed input never leaves the mapping
FUZZ = r"""
import sys, numpy as np
sys.path.insert(0, %r)
from tnc_b200.io import hdf5
from tnc_b200 import TncbError
rng = np.random.default_rng(int(sys.argv[2]))
raw = bytearray(open(sys.argv[1], 'rb').read())
ok = bad = 0
for trial in range(int(sys.argv[3])):
    b = bytearray(raw)
    mode = trial %% 3
    if mode == 0:
        for _ in range(int(rng.integers(1, 6))):
            b[int(rng.integers(0, min(len(b), 6000)))] = int(rng.integers(0, 256))
    elif mode == 1:
        b = b[:int(rng.integers(0, len(b)))]
    else:
        i = int(rng.integers(0, min(len(b), 6000) - 8)); b[i:i + 8] = int(rng.integers(0, 1 << 63)).to_bytes(8, 'little')
    open(sys.argv[1] + '.fz', 'wb').write(b)
    try:
        with hdf5.Hdf5File(sys.argv[1] + '.fz') as f:
            for i in range(len(f.member_names())):
                if np.prod(f.shape(i), dtype=np.float64) < 1e6:
                    f.read(i)
                try:
                    f.attr(i, 'bids')
                except TncbError:
                    pass
        ok += 1
    except TncbError as e:
        assert e.status in (-1, -9, -10), e
        bad += 1
print(ok, bad)
"""


@pytest.mark.parametrize("kind", ["earliest", "latest"])
def test_corrupted_files_are_rejected_not_followed(h5, tmp_path, kind):
    """bit flips, truncations and wild addresses: every outcome is a clean status (or a successful read of garbage
    values), never a crash -- run in a child process so that a crash would be seen as one."""
    rng = np.random.default_rng(3)
    p = tmp_path / "fz.h5"
    if kind == "earliest":
        h5.store_tensor(p, [(str(i), [i], cplx(rng, (3,))) for i in range(40)], [0])
    else:
        p.write_bytes(_latest_file(rng)[0])
    r = subprocess.run([sys.executable, "-c", FUZZ % (ROOT,), str(p), "7", "600"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    ok, bad = map(int, r.stdout.split())
    assert ok + bad == 600 and bad > 50


def test_network_file_round_trip_contracts_to_the_same_amplitude(h5, tmp_path):
    """a circuit network written as /tensors/<i>{bids} (gates materialised), read back with load_tensor -- members arrive in
    name order "0", "1", "10", "11", ..., not in circuit order -- and contracted by the oracle along a path found on the
    LOADED network gives the amplitude of the original network"""
    from oracle import tnc_oracle as orc
    from tnc_b200.builders import random_circuit
    from tnc_b200.contractionpath.paths import Cotengrust
    from tnc_b200.gates import load_gate, load_gate_adjoint
    tn = random_circuit(10, 6, 0.6, 0.6, np.random.default_rng(12))

    def payload(t):
        td = t.tensordata
        if td.kind == "gate":
            return (load_gate_adjoint if td.gate[2] else load_gate)(td.gate[0], td.gate[1]).reshape(t.bond_dims)
        return np.asarray(td.matrix, dtype=np.complex128).reshape(t.bond_dims)

    h5.store_tensor(tmp_path / "net.h5", [(str(i), t.legs, payload(t)) for i, t in enumerate(tn.tensors)], [])
    loaded = h5.load_tensor(tmp_path / "net.h5")
    assert loaded.legs == [] and len(loaded.tensors) == len(tn.tensors)
    order = sorted(range(len(tn.tensors)), key=lambda i: str(i).encode())
    assert [t.legs for t in loaded.tensors] == [tn.tensors[i].legs for i in order]

    def amplitude(net):
        opt = Cotengrust(net); opt.find_path()
        path = opt.get_best_replace_path()
        def to_o(t):
            if t.is_composite():
                return orc.OTensor(children=[to_o(c) for c in t.tensors])
            td = t.tensordata
            return orc.OTensor(list(t.legs), list(t.bond_dims), ("gate", td.gate[0], td.gate[1], td.gate[2]) if td.kind == "gate" else np.asarray(td.matrix))
        return complex(orc.contract_tensor_network(to_o(net), orc.OPath(list(path.toplevel), {})).data)

    a, b = amplitude(tn), amplitude(loaded)
    assert abs(a - b) <= 1e-13 * abs(a)
