"""N>1 path.  CPU: world_size-2/3 gloo tests of the host-side logic (broadcast, mapping, scatter,
fan-in schedule agree on all ranks) -- the counterpart of the reference's #[mpi_test]s
(tnc/tests/integration_tests.rs:85-164).  GPU: NCCL fan-in == flat when >= 2 devices exist."""
import os
import socket
import subprocess
import sys

import pytest
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))


def free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


@pytest.mark.parametrize("world", [2, 3])
def test_gloo_host_logic(built_lib, world):
    import dist_worker
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = free_port()
    procs = [ctx.Process(target=dist_worker.cpu_logic, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    res = dict(q.get(timeout=5) for _ in range(world))
    assert len(res) == world
    # mapping and fan-in schedule are identical on every rank
    assert all(res[r][0] == res[0][0] and res[r][1] == res[0][1] for r in range(world))
    assert sorted(r for _, r in res[0][0]) == list(range(world))


@pytest.mark.parametrize("world", [2, 3, 4])
def test_gloo_full_fanin_with_the_oracle_as_engine(built_lib, world):
    """contract_partitioned and PartitionedPlan end to end on CPU ranks: the amplitude after scatter + local contraction +
    fan-in equals the flat one (see dist_worker.cpu_fanin)."""
    import dist_worker
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = free_port()
    procs = [ctx.Process(target=dist_worker.cpu_fanin, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=180)
        assert p.exitcode == 0
    res = dict(q.get(timeout=5) for _ in range(world))
    assert all(res[r] == ("ok", world - 1) for r in range(world))


def test_partition_packing_round_trips(built_lib):
    """the compact form partitions travel in (dist.communication._pack_tensor) loses nothing: nested composites, gate,
    matrix, file and empty leaves"""
    import pickle
    import numpy as np
    from tnc_b200.builders import random_circuit
    from tnc_b200.dist.communication import _pack_tensor, _unpack_tensor
    from tnc_b200.tensornetwork import Tensor, TensorData
    rc = random_circuit(8, 5, 0.5, 0.5, np.random.default_rng(2))
    m = Tensor.new([0, 1], [2, 4]); m.set_tensor_data(TensorData.Matrix(np.arange(8, dtype=np.complex128).reshape(2, 4)))
    f = Tensor.new([1, 2], [4, 3]); f.set_tensor_data(TensorData.File("x.h5", True))
    tn = Tensor.new_composite([Tensor.new_composite(rc.tensors[:7]), Tensor.new_composite(rc.tensors[7:]), Tensor.new_composite([m, f, Tensor.new([], [])])])

    def same(a, b):
        assert a.legs == b.legs and a.bond_dims == b.bond_dims and len(a.tensors) == len(b.tensors)
        ta, tb = a.tensordata, b.tensordata
        assert ta.kind == tb.kind and ta.gate == tb.gate and ta.file == tb.file
        if ta.kind == "matrix":
            np.testing.assert_array_equal(ta.matrix, tb.matrix)
        for x, y in zip(a.tensors, b.tensors):
            same(x, y)

    same(tn, _unpack_tensor(pickle.loads(pickle.dumps(_pack_tensor(tn), protocol=pickle.HIGHEST_PROTOCOL))))


@pytest.mark.gpu
def test_nccl_fanin_equals_flat():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 2
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(free_port()), os.path.join(ROOT, "tests", "dist_worker.py")]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0 and "DIST_OK" in r.stdout and "SLICED_OK" in r.stdout, r.stdout[-3000:]
