#!/usr/bin/env python
"""bench.py -- the driver's measurement contract for the pairwise-contraction hot path.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json: "pairwise contractions/sec + effective ZGEMM TFLOP/s on random-circuit network"; north star:
the 36-qubit random-circuit amplitude network): `random_circuit(36 qubits, 10 rounds, p1 = p2 = 0.5, Sycamore coupling,
seed 1)` closed with <0| bras -> 489 leaves, 488 pairwise contractions.  A "step" is ONE full contraction of that network
through `contract_tensor_network`; K steps are timed in each of the two forms below (value and e2e).

--dump-outputs DIR writes, after the timed steps, what the last step of each form returned on rank 0: DIR/amplitude.npy
(value) and DIR/amplitude_e2e.npy (e2e), each the complex amplitude as float64 [re, im]; --impl reference writes its
own DIR/amplitude.npy.  The network and path are fixed by the seed, so two builds run with the same arguments can be
compared output for output.

  N = 1   greedy (Cotengrust) path, 6.7e12 flop.
          value = pairs/s with the leaves resident in HBM (tncb_plan_stage + tncb_plan_run),
          e2e   = the public call `contract_tensor_network(tn, path)` from HOST leaves: schedule construction, gate
                  materialisation, one H2D of the leaf block, every pair kernel, D2H of the amplitude -- exactly the
                  timed region of benchmark/src/main.rs:355-360.
  N > 1   BASELINE config 4: the same network partitioned into N parts (planned outside the timer,
          tools/plan_partitions.py -> bench_inputs/c4_partitions.json), one partition per GPU, boundary tensors fanned
          in over NCCL p2p (mpi/communication.rs:125-249, timed like main.rs:369-399).  scaling = "strong".
          value = pairs/s with the partitions scattered and their leaves staged beforehand (local contraction + fan-in),
          e2e   = `dist.contract_partitioned` from rank 0's host network (broadcast + scatter + leaf upload inside).
          "parity_n" compares the N-GPU amplitudes (fan-in and sliced) with the flat 1-GPU amplitude on rank 0.
  --impl reference: the reference's CPU path for the same network / path: the oracle port of contract_tensor_network
          (oracle/tnc_oracle.py; TTGT with torch-CPU MKL zgemm, all host threads) -- the Rust crate cannot be built
          here (no cargo, un-vendored git dependencies), so kind = "port".

Extra objects: "roofline" (the dominant kernel crt_gemm_kernel: int8 tensor pipe, timed live with CUDA events on every
launch inside the timed region), "pair_c2" (BASELINE configs[1], the single 4096^3 pair: engines side by side, host
pipeline), "cpu_baseline", "clocks", "gpu_launches".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "pairwise contractions/sec (effective ZGEMM TFLOP/s in zgemm_tflops)"
NET = {"qubits": 36, "rounds": 10, "p1": 0.5, "p2": 0.5, "seed": 1}
WORKLOAD = ("36-qubit random-circuit amplitude network (10 rounds, p1=p2=0.5, Sycamore coupling, seed 1; 489 leaves, "
            "488 pairs) through contract_tensor_network")
# Measured on this pool's B200 with tools/fp64_peak.cu (profiles/r01_fp64_peak_microbench.txt):
# DMMA m8n8k4 sustained, = 148 SM x 64 FMA/clk x 2 x 1.965 GHz.  tcgen05 has no f64 kind.
FP64_TENSOR_PEAK_TFLOPS = 37.2
INT8_NOMINAL_TOPS = 4500.0   # dense int8 tcgen05 (kind::i8), 2 x the nominal bf16 figure
# Measured on this pool's B200 with tools/i8_peak.cu (profiles/r02_i8_peak.txt): back-to-back UMMA kind::i8 cta_group::2 from
# resident shared memory, 4533 TOP/s sustained over 274 ms (4592 over 54 ms) -- the int8 tensor pipe at ~1.88 GHz.
INT8_MEASURED_TOPS = 4533.0


# ------------------------------------------------------------------------------------------------ inputs
def build_network():
    from tnc_b200.builders import random_circuit
    return random_circuit(NET["qubits"], NET["rounds"], NET["p1"], NET["p2"], np.random.default_rng(NET["seed"]))


def greedy_path(tn):
    from tnc_b200.contractionpath.paths import Cotengrust
    opt = Cotengrust(tn)
    opt.find_path()
    return opt.get_best_replace_path()


def partition_plan(tn, n):
    """(partitioned network, nested path, facts): committed plan if it matches the network, else planned now."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import plan_partitions as pp
    got = pp.load(tn, n)
    if got is None:
        d = pp.plan(tn, (n,))
        from tnc_b200.contractionpath import ContractionPath
        from tnc_b200.tensornetwork.partitioning import partition_tensor_network
        p = d["plans"][str(n)]
        path = ContractionPath({int(k): ContractionPath.simple([tuple(x) for x in v]) for k, v in p["nested"].items()},
                               [tuple(x) for x in p["toplevel"]])
        got = (partition_tensor_network(tn, p["partitioning"]), path,
               {k: p[k] for k in ("critical_path_flops", "total_flops", "partition_sizes", "predicted_critical_path_ms", "chosen")})
    return got


def path_flops(tn, path) -> float:
    """sum of 8MNK over the executed pairs (SURVEY 8d) == contract_cost_tensors + 2 per output element"""
    def walk(inputs, p):
        tot = 0.0
        inputs = list(inputs)
        for i in sorted(p.nested):
            tot += walk(inputs[i].tensors, p.nested[i])
            inputs[i] = inputs[i].external_tensor()
        for (i, j) in p.toplevel:
            a, b = inputs[i], inputs[j]
            tot += 8.0 * (a | b).size()
            inputs[i] = b ^ a
        return tot
    return walk(tn.tensors, path)


def count_pairs(path) -> int:
    return len(path.toplevel) + sum(count_pairs(p) for p in path.nested.values())


def leaf_bytes(tn) -> int:
    if tn.is_composite():
        return sum(leaf_bytes(c) for c in tn.tensors)
    return 16 * int(np.prod(tn.bond_dims)) if tn.bond_dims else 16


def to_oracle(t):
    from oracle import tnc_oracle as orc
    if t.is_composite():
        return orc.OTensor(children=[to_oracle(c) for c in t.tensors])
    td = t.tensordata
    d = ("gate", td.gate[0], td.gate[1], td.gate[2]) if td.kind == "gate" else (np.asarray(td.matrix) if td.kind == "matrix" else None)
    return orc.OTensor(list(t.legs), list(t.bond_dims), d)


def to_opath(p):
    from oracle import tnc_oracle as orc
    return orc.OPath(list(p.toplevel), {i: to_opath(q) for i, q in p.nested.items()})


def c2_problem():
    """SURVEY 8(d) C2: A legs [0..11]; shared legs at A's odd positions; in B they sit at the
    even positions in reversed order (different relative order -> both need a permute)."""
    a_legs = list(range(12))
    shared = [11, 9, 7, 5, 3, 1]
    b_legs = [x for p in zip(shared, range(12, 18)) for x in p]
    dims = [4] * 12
    return a_legs, dims, b_legs, dims


def pinned_complex(shape, rng):
    import torch
    n = int(np.prod(shape))
    t = torch.empty(n, dtype=torch.complex128, pin_memory=torch.cuda.is_available())
    a = t.numpy()
    a.real[:] = rng.random(n) * 2 - 1
    a.imag[:] = rng.random(n) * 2 - 1
    return t, a.reshape(shape)


# ------------------------------------------------------------------------------------------------ helpers
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.06] or [r for (_, r) in self.rows]
        for r in rows:
            p = [x.strip() for x in r.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1])); pw.append(float(p[2]))
            except ValueError:
                continue
            for nm, v in zip(names, p[3:7]):
                if v == "Active":
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def effective_cpus() -> int:
    """Host cores this process may actually use: min(affinity, cgroup CPU quota).  The GPU boxes
    expose 128 logical CPUs but cap the container at 16 (cpu.max = 1600000 100000); running MKL
    with 128 threads there is 16x *slower* than with 16, so the baseline uses the quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return n


def _peak(key, fallback):
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)[key])
    except Exception:
        return fallback  # B200_PROFILING.md fallback


def _captured_traffic():
    """DRAM bytes per launch of the dominant kernel on C2 from the committed ncu summary of this round (a capture of the
    same command, never measured under the timer); None if no r02 capture is committed."""
    import re
    for name in ("r02_ncu_crt_gemm_summary.txt",):
        try:
            txt = open(os.path.join(ROOT, "profiles", name)).read()
            rd = re.search(r"^dram__bytes_read\.sum\s+([0-9.]+)\s+(\w+)", txt, re.M)
            wr = re.search(r"^dram__bytes_write\.sum\s+([0-9.]+)\s+(\w+)", txt, re.M)
            scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
            return float(rd.group(1)) * scale[rd.group(2)] + float(wr.group(1)) * scale[wr.group(2)], name
        except Exception:
            continue
    return None, None


def dump_outputs(directory, outputs):
    """Each complex output as DIR/<name>.npy, float64 with a trailing [re, im] axis."""
    os.makedirs(directory, exist_ok=True)
    for name, z in outputs.items():
        z = np.asarray(z, dtype=np.complex128)
        np.save(os.path.join(directory, name + ".npy"), np.stack([z.real, z.imag], axis=-1))


def oracle_network_seconds(tn, path, repeats, warm=1):
    import torch
    from oracle import tnc_oracle as orc
    otn, op = to_oracle(tn), to_opath(path)
    amp = None
    for _ in range(warm):
        amp = complex(orc.contract_tensor_network(otn, op, backend="torch").data)
    ts = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        amp = complex(orc.contract_tensor_network(otn, op, backend="torch").data)
        ts.append(time.perf_counter() - t0)
    return ts, amp


# ------------------------------------------------------------------------------------------------ reference arm
def run_reference(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    cores = effective_cpus()
    torch.set_num_threads(cores)
    tn = build_network()
    if world == 1:
        net, path, mode = tn, greedy_path(tn), "flat, greedy Cotengrust path"
    else:
        net, path, facts = partition_plan(tn, world)
        mode = f"partitioned into {world} parts (tools/plan_partitions.py), local paths then the fan-in pairs, sequentially on the host"
    pairs, flops = count_pairs(path), path_flops(net, path)
    ts, amp = oracle_network_seconds(net, path, args.steps, warm=max(1, args.warmup))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"amplitude": amp})
    sec = float(np.mean(ts))
    val = pairs / sec
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "contractions/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": max(1, args.warmup), "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "zgemm_tflops": flops / sec * 1e-12,
        "config": {"workload": WORKLOAD, "path": mode, "pairs": pairs, "flops_8mnk": flops},
        "cpu_baseline": {"value": val, "unit": "contractions/s", "cores": cores, "kind": "port",
                         "sample": f"{args.steps} full contractions of the network after {max(1, args.warmup)} warm-up "
                                   f"(oracle port of contract_tensor_network: permute+contiguous+MKL zgemm via torch-CPU, {torch.get_num_threads()} threads)",
                         "zgemm_tflops": flops / sec * 1e-12, "ms_per_network": sec * 1e3},
        "e2e": {"value": val, "unit": "contractions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "amplitude": [amp.real, amp.imag],
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ our arm
def pair_c2(tb, ctx, torch, stream, steps):
    """BASELINE configs[1]: the single 4096^3 pair, device-resident, engines side by side + host-buffer end to end."""
    a_legs, a_dims, b_legs, b_dims = c2_problem()
    M = N = K = 4096
    flops = 8.0 * M * N * K
    rng = np.random.default_rng(20240612)
    _, a = pinned_complex(a_dims, rng)
    _, b = pinned_complex(b_dims, rng)
    _, c_host = pinned_complex([4] * 12, np.random.default_rng(0))
    dA, dB = tb.DeviceTensor.from_numpy(ctx, a), tb.DeviceTensor.from_numpy(ctx, b)
    dC = tb.DeviceTensor.empty(ctx, [4] * 12)

    def timed(n):
        for _ in range(3):
            tb.contract_pair_into(ctx, a_legs, dA, b_legs, dB, dC)
        ctx.synchronize()
        ctx.time_gemm(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(n):
            tb.contract_pair_into(ctx, a_legs, dA, b_legs, dB, dC)
        e1.record(stream)
        ctx.synchronize(); torch.cuda.synchronize()
        g = ctx.last_gemm_ms()
        ctx.time_gemm(0)
        return e0.elapsed_time(e1) / n, g
    out = {"workload": "C2: single pairwise contraction, rank-12 dim-4 operands, M=N=K=4096, interleaved shared legs", "flops_8mnk": flops,
           "algorithmic_bytes": 16.0 * 3 * M * N, "engines": {}}
    ms, g = timed(steps)
    info = ctx.last_tcgen05_info()
    out["engines"]["tcgen05_modular"] = {"ms_per_pair": ms, "gemm_kernel_ms": g, "zgemm_tflops": flops / ms * 1e-9, "n_moduli": info["n_moduli"],
                                         "int8_tops_gemm_kernel": info["int8_ops"] / g * 1e-9}
    out["default_int8_ops"], out["default_gemm_ms"] = info["int8_ops"], g
    ctx.set_tcgen05_moduli(13)
    ms, g = timed(5)
    out["engines"]["tcgen05_modular_13_moduli"] = {"ms_per_pair": ms, "gemm_kernel_ms": g, "zgemm_tflops": flops / ms * 1e-9,
                                                    "note": "fewer moduli = fewer operand bits: measured error ~1e-12 of max|C|, see tncb_tcgen05_bound"}
    ctx.set_tcgen05_moduli(0)
    ctx.set_tcgen05_engine(1)
    ms, g = timed(5)
    out["engines"]["tcgen05_digit_slicing_s8"] = {"ms_per_pair": ms, "gemm_kernel_ms": g, "zgemm_tflops": flops / ms * 1e-9, "note": "round-1 engine"}
    ctx.set_tcgen05_engine(0)
    ctx.set_tcgen05_slices(0)
    ms, g = timed(5)
    out["engines"]["dmma_fp64"] = {"ms_per_pair": ms, "gemm_kernel_ms": g, "zgemm_tflops": flops / ms * 1e-9,
                                   "frac_of_measured_fp64_peak": flops / g * 1e-9 / FP64_TENSOR_PEAK_TFLOPS}
    ctx.set_tcgen05_slices(8)
    # end to end with host buffers: H2D of both operands, the pair, D2H of the result
    def e2e_step():
        tb.upload_into(ctx, a, dA); tb.upload_into(ctx, b, dB)
        tb.contract_pair_into(ctx, a_legs, dA, b_legs, dB, dC)
        tb.download_into(ctx, dC, c_host)
    e2e_step(); ctx.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(5):
        e2e_step()
    e1.record(stream)
    ctx.synchronize(); torch.cuda.synchronize()
    out["e2e_host_buffers"] = {"ms_per_pair": e0.elapsed_time(e1) / 5, "h2d_bytes": int(2 * 16 * 4 ** 12), "d2h_bytes": int(16 * 4 ** 12),
                               "how": "serial on the ctx stream: H2D(a), H2D(b), pair, D2H(result)"}
    # pipelined host API: H2D of pair j+1, kernels of pair j and D2H of pair j-1 overlap (tncb_contract_pair_host)
    outs = [pinned_complex([4] * 12, np.random.default_rng(1))[1] for _ in range(3)]
    for j in range(3):
        tb.contract_pair_host(ctx, a_legs, a, b_legs, b, outs[j % 3])
    ctx.synchronize()
    t0 = time.perf_counter()
    n_pipe = 12
    for j in range(n_pipe):
        tb.contract_pair_host(ctx, a_legs, a, b_legs, b, outs[j % 3])
    ctx.synchronize()
    ms = (time.perf_counter() - t0) * 1e3 / n_pipe
    same = bool(np.array_equal(outs[0], c_host.reshape(outs[0].shape)))
    out["e2e_host_buffers_pipelined"] = {"ms_per_pair": ms, "pairs": n_pipe, "equals_serial_result": same,
                                         "how": "tncb_contract_pair_host, 12 back-to-back pairs from pinned buffers, wall clock incl. the final synchronize"}
    dA.free(); dB.free(); dC.free()
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    import tnc_b200 as tb
    from tnc_b200.tensornetwork import NetworkPlan, contract_tensor_network

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: tnc_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    meta_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        meta_group = dist.new_group(backend="gloo")     # metadata (paths, legs, pickled leaf descriptions) travels over CPU sockets
    ctx = tb.Context(local)
    stream = torch.cuda.ExternalStream(ctx.stream, device=local)
    warmup = max(args.warmup, 3)

    def barrier():
        if world > 1:
            dist.barrier()
        ctx.synchronize()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], device=f"cuda:{local}", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_ranks_ok(ok: bool) -> bool:
        """True only if every rank says so: a leg that failed on ONE rank must be abandoned by ALL ranks together, or the
        others would wait for it inside the next collective until the driver's clock runs out."""
        return max_over_ranks(0.0 if ok else 1.0) == 0.0

    tn = build_network()                                  # same seed on every rank -> same network
    fpath = greedy_path(tn)
    if world == 1:
        net, path, facts = tn, fpath, {}
        mode = "flat, greedy Cotengrust path"
    else:
        net, path, facts = partition_plan(tn, world)
        mode = f"{world} partitions (one per GPU) + NCCL p2p fan-in"
    pairs, flops = count_pairs(path), path_flops(net, path)

    # ---- the step, in its two forms -------------------------------------------------------------------------
    if world == 1:
        plan = NetworkPlan(net, path, ctx=ctx)
        plan.stage(net)
        step_resident = lambda: plan.run()
        step_e2e = lambda: contract_tensor_network(net, path, ctx=ctx)
    else:
        from tnc_b200.dist import PartitionedPlan, contract_partitioned, init_device_comm
        init_device_comm(ctx, meta_group)
        pplan = PartitionedPlan(net if rank == 0 else None, path if rank == 0 else None, ctx, meta_group)
        step_resident = lambda: pplan.run()
        step_e2e = lambda: contract_partitioned(net if rank == 0 else None, path if rank == 0 else None, ctx, meta_group)

    def read_amp(res):
        return complex(res.to_numpy()) if rank == 0 else None

    # ---- value: leaves resident in HBM, K steps timed with CUDA events on the ctx stream ---------------------
    for _ in range(warmup):
        amp = read_amp(step_resident())
    ctx.synchronize()
    ctx.reset_stats()
    ctx.time_gemm(2)
    barrier()
    sampler = ClockSampler(local)
    time.sleep(0.15)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    ev0.record(stream)
    for _ in range(args.steps):
        res = step_resident()
    ev1.record(stream)
    ctx.synchronize(); torch.cuda.synchronize()
    t1 = time.time()
    barrier()
    clocks = sampler.stop(t0, t1)
    amp = read_amp(res)
    total_ms = max_over_ranks(ev0.elapsed_time(ev1))
    st = ctx.stats()
    gt = ctx.gemm_totals()
    ctx.time_gemm(0)
    ec = ctx.engine_counts()
    launches = int(st["kernel_launches"])
    if world > 1:
        lt = torch.tensor([float(launches)], device=f"cuda:{local}", dtype=torch.float64)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
        launches = int(lt.item())
    ms_per_step = total_ms / args.steps
    value = pairs / (ms_per_step * 1e-3)

    # ---- e2e: the public call from host leaves, device->host read of the amplitude inside -----------------
    e2e_steps = args.steps
    for _ in range(warmup):       # W >= 3 like the resident form: the library compiles its plan on the SECOND sighting of a structure
        read_amp(step_e2e())
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    ev0.record(stream)
    for _ in range(e2e_steps):
        amp_e2e = read_amp(step_e2e())
    ev1.record(stream)
    ctx.synchronize(); torch.cuda.synchronize()
    w1 = time.perf_counter()
    e2e_ms = max_over_ranks(ev0.elapsed_time(ev1)) / e2e_steps
    e2e_wall_ms = max_over_ranks((w1 - w0) * 1e3) / e2e_steps
    e2e_val = pairs / (e2e_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"amplitude": amp, "amplitude_e2e": amp_e2e})

    line = None
    if rank == 0:
        bf16_meas = _peak("bf16_tflops", 1590.0)
        line = {
            "metric": METRIC, "value": value, "unit": "contractions/s", "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "dtype_note": "complex128 in, complex128 out; GEMM-like pairs run as 16-17 exact int8 modular GEMMs on tcgen05 + CRT "
                                          "(guaranteed normwise bound 2^-49 K max|b| max|a|, measured 1e-15: FP64-GEMM-equivalent), all other pairs in FP64",
            "data": "synthetic", "zgemm_tflops": flops / (ms_per_step * 1e-3) * 1e-12,
            "config": {"workload": WORKLOAD, "path": mode, "pairs": pairs, "flops_8mnk": flops,
                       "l2": "every step re-reads its operands from HBM: the dominant pairs move 0.3-6 GB each (> 126 MB L2)",
                       "engines_per_step": {k: v // max(1, args.steps) for k, v in ec.items() if v}},
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": "contractions/s", "h2d_bytes_per_step": leaf_bytes(net), "d2h_bytes_per_step": 16,
                    "ms_per_step": e2e_ms, "wall_ms_per_step": e2e_wall_ms, "steps": e2e_steps,
                    "amplitude": [amp_e2e.real, amp_e2e.imag]},
            "gpu_launches": launches,
            "amplitude": [amp.real, amp.imag],
        }
        if facts:
            line["config"]["partitioning"] = facts
        if gt["launches"]:
            ach = gt["int8_ops"] / (gt["ms"] * 1e-3) * 1e-12
            traffic, tfile = _captured_traffic()
            line["roofline"] = {
                "bound": "tensor", "kernel": "crt_gemm_kernel (tcgen05.mma.cta_group::2.kind::i8, TMA, TMEM; one int8 GEMM per modulus)",
                "achieved": ach, "peak": INT8_MEASURED_TOPS, "unit": "int8 TOP/s", "frac": ach / INT8_MEASURED_TOPS,
                "peak_source": "int8 tensor-pipe peak measured on this pool with tools/i8_peak.cu (profiles/r02_i8_peak.txt, sustained); MEASURED_PEAKS.json "
                               f"has no int8 entry: against its bf16 burst x 2 = {2.0 * bf16_meas:.0f} the fraction is {ach / (2.0 * bf16_meas):.3f}, against nominal 4500 "
                               f"{ach / INT8_NOMINAL_TOPS:.3f}; ncu on the C2 launch: 96 % of the per-cycle pipe peak at a power-capped 1.50 GHz (profiles/r02_ncu_crt_gemm_summary.txt)",
                "how": f"CUDA events around every one of the {gt['launches']} launches of the kernel inside the timed region (sum of durations "
                       f"{gt['ms']:.3f} ms = {gt['ms'] / total_ms:.2f} of it); executed int8 ops = 2 x (4, or 3 from K >= 4096) x moduli x Np x Mp x Kp (padded tiles)",
                "kernel_ms_per_step": gt["ms"] / args.steps, "launches_per_step": gt["launches"] / args.steps,
                "executed_int8_ops_per_step": gt["int8_ops"] / args.steps,
                "traffic": traffic, "traffic_note": (f"dram read+write of ONE launch on the C2 pair from profiles/{tfile} (ncu --set full of this kernel; not a "
                                                     "measurement of the timed run)") if traffic else "no ncu capture committed yet",
                "algorithmic_flops_per_step": flops,
            }
    # ---- extra objects (never fatal) ------------------------------------------------------------------------
    extras = {}
    try:
        if world == 1 and not args.no_pair:
            extras["pair_c2"] = pair_c2(tb, ctx, torch, stream, 10)
        if world == 1 and not args.no_extras:
            # the same network on the FP64 pipe only, and with a better tree (random-greedy, 64 trials)
            ctx.set_tcgen05_slices(0)
            plan.run(); ctx.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(3):
                plan.run()
            e1.record(stream); ctx.synchronize(); torch.cuda.synchronize()
            extras["dmma_only"] = {"ms_per_step": e0.elapsed_time(e1) / 3, "zgemm_tflops": flops / (e0.elapsed_time(e1) / 3) * 1e-9}
            ctx.set_tcgen05_slices(8)
            # the same network as 8 slices on this one GPU (slice loop inside the library): the overhead of slicing itself
            from tnc_b200.contractionpath.slicing import SlicedPlan, find_slices
            legs = find_slices(tn, fpath, min_slices=8)
            sp = SlicedPlan(tn, fpath, legs, ctx=ctx)
            samp = complex(sp.run().to_numpy())
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(3):
                r8 = sp.run()
            e1.record(stream); ctx.synchronize(); torch.cuda.synchronize()
            extras["sliced8_on_1gpu"] = {"ms_per_step": e0.elapsed_time(e1) / 3, "vs_flat": e0.elapsed_time(e1) / 3 / ms_per_step,
                                         "rel_diff_vs_flat": abs(samp - amp) / abs(amp), "sliced_legs": [int(l) for l in legs]}
        if world > 1:
            extras["parity_n"] = parity_and_modes(tb, ctx, dist, torch, stream, tn, fpath, net, path, amp, rank, world, local, meta_group, max_over_ranks,
                                                  all_ranks_ok)
    except Exception as e:  # keep the headline line even if an extra leg fails
        extras["extras_error"] = f"{type(e).__name__}: {e}"
    if not args.no_config5:
        try:
            plan = pplan = step_resident = step_e2e = sp = res = r8 = None      # drop the headline workload's device state first
            import gc
            gc.collect()
            ctx.trim()
            extras["config5_sycamore53_d12"] = config5_sycamore(tb, ctx, dist, rank, world, max_over_ranks, all_ranks_ok)
        except Exception as e:
            extras["config5_error"] = f"{type(e).__name__}: {e}"
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cores = effective_cpus()
            torch.set_num_threads(cores)
            ts, amp_cpu = oracle_network_seconds(net, path, 2, warm=1)
            sec = float(np.mean(ts))
            cpu = {"value": pairs / sec, "unit": "contractions/s", "cores": cores, "kind": "port",
                   "sample": f"2 full contractions of the same network and path after 1 warm-up (oracle port: permute+contiguous+MKL zgemm via torch-CPU, "
                             f"{cores} threads = cgroup quota of {os.cpu_count()} logical CPUs)",
                   "zgemm_tflops": flops / sec * 1e-12, "ms_per_network": sec * 1e3,
                   "rel_diff_gpu_vs_cpu": abs(amp - amp_cpu) / abs(amp_cpu)}
            line["cpu_baseline"] = cpu
        line.update(extras)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0 and world > 1 and not extras.get("parity_n", {}).get("ok", False):
        raise SystemExit("multi-GPU parity check failed: " + json.dumps(extras))


CONFIG5_PATH = os.path.join("bench_inputs", "sycamore53_d12.json")
# amplitude <0^53| C |0^53> of the Sycamore-53 depth-12 circuit (seed 1), measured with two independent paths / slicings on
# a B200 (profiles/r02_config5_sycamore53_d12.jsonl: they agree to 2e-15); regression reference of the config5 object
CONFIG5_AMPLITUDE = complex(-6.148484459425177e-09, -5.130555022162778e-09)


def config5_sycamore(tb, ctx, dist, rank, world, max_over_ranks, all_ranks_ok, steps=2):
    """BASELINE config 5: Sycamore-53 depth-12 single amplitude as 2^s slices of one replace-left path (found offline by
    tools/search_path.py: random-greedy + subtree reconfiguration + slicing under the device-time model), slices round-robin
    over the ranks, one ncclAllReduce.  Timed: every slice through the compiled plan (leaves resident) + all-reduce + D2H of
    the amplitude, wall clock between barriers, max over ranks."""
    from tnc_b200.builders import sycamore_circuit
    from tnc_b200.contractionpath import ContractionPath
    from tnc_b200.contractionpath.slicing import SlicedPlan, path_cost
    d = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), CONFIG5_PATH)))
    w = d["network"].split()
    tn5 = sycamore_circuit(int(w[1][:-1]), int(w[3]), np.random.default_rng(int(w[5]))).into_amplitude_network("0" * int(w[1][:-1]))[0]
    path5 = ContractionPath.simple([tuple(x) for x in d["toplevel"]])
    legs = d["sliced_legs"]
    flops_slice, peak, _ = path_cost([(t.legs, t.bond_dims) for t in tn5.tensors], path5, legs)
    t0 = time.perf_counter()
    sp, err = None, None
    try:
        sp = SlicedPlan(tn5, path5, legs, ctx=ctx)
    except Exception as e:      # e.g. no room for the 64 GiB workspace on ONE rank: every rank must skip the leg together
        err = e
    if not all_ranks_ok(err is None):
        sp = None
        raise RuntimeError(f"setup failed on a rank (this rank: {err!r})")
    setup = time.perf_counter() - t0
    ts, amp5 = [], None
    for it in range(1 + steps):
        if world > 1:
            dist.barrier()
        ctx.synchronize()
        t0 = time.perf_counter()
        amp5 = complex(sp.run(rank, world).to_numpy())
        dt = max_over_ranks(time.perf_counter() - t0)
        if it:
            ts.append(dt)
    n_slices = sp.n_slices
    del sp                      # frees the plan's workspace and staged leaves
    sec = float(np.median(ts))
    pairs5 = len(path5.toplevel) * n_slices
    return {"workload": "Sycamore-53 depth-12 single-amplitude network (sycamore_circuit(53, 12), seed 1, bitstring 0^53): 1053 tensors",
            "path": f"{CONFIG5_PATH}: {d.get('finder', '')}", "mode": f"{n_slices} slices round-robin over {world} rank(s) + 1 ncclAllReduce",
            "n_gpus": world, "slices": n_slices, "pairs": pairs5, "flops_8mnk": flops_slice * n_slices, "peak_tensor_GiB": peak * 16 / 2 ** 30,
            "seconds": sec, "seconds_all": [round(t, 4) for t in ts], "setup_seconds_untimed": setup,
            "contractions_per_s": pairs5 / sec, "zgemm_tflops": flops_slice * n_slices / sec * 1e-12,
            "amplitude": [amp5.real, amp5.imag], "rel_diff_vs_committed_amplitude": abs(amp5 - CONFIG5_AMPLITUDE) / abs(CONFIG5_AMPLITUDE),
            "cpu_baseline": "oracle port, 1 of 64 slices of the same path: 87.3 s on 16 cores -> 5586 s extrapolated (tools/bench_sliced.py --cpu-slices 1, "
                            "profiles/r02_config5_sycamore53_d12.jsonl)"}


def parity_and_modes(tb, ctx, dist, torch, stream, tn, fpath, net, path, amp_fanin, rank, world, local, meta_group, max_over_ranks, all_ranks_ok):
    """Rank 0: flat 1-GPU amplitude of the same network (greedy path) and the partitioned path executed on ONE GPU;
    all ranks: the sliced mode (2^s slices round-robin + one ncclAllReduce).  Asserts |amp_N - amp_flat| <= 1e-9 |amp_flat|."""
    from tnc_b200.contractionpath.slicing import SlicedPlan, find_slices
    from tnc_b200.tensornetwork import contract_tensor_network
    out = {}
    flat = None
    err = None
    try:
        if rank == 0:
            flat = complex(contract_tensor_network(tn, fpath, ctx=ctx).to_numpy())
            ctx.synchronize()
            ts = []
            for _ in range(3):
                t0 = time.perf_counter()
                one = complex(contract_tensor_network(net, path, ctx=ctx).to_numpy())
                ts.append(time.perf_counter() - t0)
            out["same_partitioned_path_on_1gpu_ms"] = float(np.median(ts)) * 1e3
            out["fanin"] = {"amplitude": [amp_fanin.real, amp_fanin.imag], "rel_diff_vs_flat": abs(amp_fanin - flat) / abs(flat),
                            "rel_diff_vs_same_path_1gpu": abs(amp_fanin - one) / abs(one)}
        legs = find_slices(tn, fpath, min_slices=max(8, world))
        t0 = time.perf_counter()
        sp = SlicedPlan(tn, fpath, legs, ctx=ctx)          # compile once + stage every slice's leaves (planning, untimed)
        setup_ms = (time.perf_counter() - t0) * 1e3
    except Exception as e:      # a failure on ONE rank (rank 0's reference legs, a plan that does not fit) ends the leg on ALL ranks
        err = e
    if not all_ranks_ok(err is None):
        raise RuntimeError(f"parity leg failed on a rank before its collectives (this rank: {err!r})")
    ts = []
    for _ in range(4):
        dist.barrier(); ctx.synchronize()
        t0 = time.perf_counter()
        samp = complex(sp.run(rank, world).to_numpy())
        ts.append(max_over_ranks(time.perf_counter() - t0))
    if rank == 0:
        n_sl = 2 ** len(legs)
        out["sliced"] = {"mode": f"greedy path, {n_sl} slices round-robin over {world} ranks (slice loop inside the library) + 1 ncclAllReduce",
                         "ms": float(np.median(ts[1:])) * 1e3, "setup_ms_untimed": setup_ms,
                         "amplitude": [samp.real, samp.imag], "rel_diff_vs_flat": abs(samp - flat) / abs(flat)}
        out["flat_amplitude"] = [flat.real, flat.imag]
        out["tolerance"] = 1e-9
        out["ok"] = bool(out["fanin"]["rel_diff_vs_flat"] <= 1e-9 and out["sliced"]["rel_diff_vs_flat"] <= 1e-9)
    return out


def main():
    ap = argparse.ArgumentParser()
    def positive(s):
        n = int(s)
        if n < 1:
            raise argparse.ArgumentTypeError(f"must be >= 1, got {n}")
        return n
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive, default=20, help="timed full contractions of the headline network, in each form")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pair", action="store_true", help="skip the pair_c2 object")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra objects")
    ap.add_argument("--no-config5", action="store_true", help="skip the Sycamore-53 depth-12 object (about 30 s at N = 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float64 [re, im])")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
