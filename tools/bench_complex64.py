"""complex64 vs complex128 on the same seeded inputs, alternating the two dtypes within one process.

  python tools/bench_complex64.py --out profiles/r03_complex64.jsonl            # one GPU
  python tools/bench_complex64.py --dry-run                                     # inputs and paths only, no device

Workloads: the C2 pair (4^6 x 4^6 x 4^6; DMMA only and with K1'), the 36-qubit bench network (resident leaves and end
to end), BASELINE config 3 (24 qubits), Sycamore-53 depth 10 and config 5 (Sycamore-53 depth 12, sliced, one GPU).
Each JSON line holds, per dtype: seconds per run over the repeats, engine counts, K1' moduli, peak arena bytes, and the
max relative difference of the complex64 result against complex128 (normwise: max |c64 - c128| / max |c128|), with the
card name and power limit read in the same process."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
DTYPES = (np.complex128, np.complex64)


def card() -> dict:
    import torch
    out = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        out["power_limit_and_max_sm_clock"] = q[0] if q else None
    except (OSError, subprocess.SubprocessError):
        out["power_limit_and_max_sm_clock"] = None
    return out


def rel_diff(x64, x128) -> float:
    x64, x128 = np.asarray(x64).astype(np.complex128), np.asarray(x128)
    return float(np.abs(x64 - x128).max() / max(np.abs(x128).max(), 1e-300))


def timed(ctx, fn, repeats):
    """fn() once per dtype per repeat, the two dtypes alternating; returns per dtype: seconds, last result, counters."""
    res = {np.dtype(d).name: {"seconds": []} for d in DTYPES}
    for _ in range(repeats):
        for d in DTYPES:
            r = res[np.dtype(d).name]
            ctx.synchronize()
            ctx.reset_stats()
            t0 = time.perf_counter()
            out = fn(d)
            ctx.synchronize()
            r["seconds"].append(time.perf_counter() - t0)
            st = ctx.stats()
            r["engine_counts"] = ctx.engine_counts()
            r["k1prime_moduli"] = ctx.last_tcgen05_info()["n_moduli"] if r["engine_counts"]["k1_tcgen05"] else None
            r["arena_peak_bytes"] = st["arena_peak_bytes"]
            r["result"] = out
    for r in res.values():
        s = r["seconds"]
        r["median_s"] = float(np.median(s))
        r["spread_s"] = [float(min(s)), float(max(s))]
    out64, out128 = res["complex64"].pop("result"), res["complex128"].pop("result")
    return res, rel_diff(out64, out128)


def sycamore(depth_file):
    from tnc_b200.builders import sycamore_circuit
    from tnc_b200.contractionpath import ContractionPath
    d = json.load(open(os.path.join(ROOT, "bench_inputs", depth_file)))
    w = d["network"].split()
    q, depth, seed = int(w[1][:-1]), int(w[3]), int(w[5])
    tn = sycamore_circuit(q, depth, np.random.default_rng(seed)).into_amplitude_network("0" * q)[0]
    return d, tn, ContractionPath.simple([tuple(x) for x in d["toplevel"]])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_complex64.jsonl"))
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--no-config5", action="store_true")
    ap.add_argument("--dry-run", action="store_true", help="build every input and path, stop before the device")
    a = ap.parse_args()
    from bench import NET, build_network, c2_problem, greedy_path
    from tnc_b200.builders import random_circuit
    al, ad, bl, bd = c2_problem()
    rng = np.random.default_rng(2)
    ca = (rng.standard_normal(ad) + 1j * rng.standard_normal(ad)).astype(np.complex64)
    cb = (rng.standard_normal(bd) + 1j * rng.standard_normal(bd)).astype(np.complex64)
    net36 = build_network()
    path36 = greedy_path(net36)
    c3 = random_circuit(24, 12, 0.5, 0.5, np.random.default_rng(1))
    path3 = greedy_path(c3)
    _, d10, path10 = sycamore("sycamore53_d10.json")
    inputs = {"c2": (len(al), len(bl)), "net36": len(path36.toplevel), "config3": len(path3.toplevel), "sycamore_d10": len(path10.toplevel)}
    if a.dry_run:
        print(json.dumps({"dry_run": True, "pairs": inputs}))
        return
    import torch
    import tnc_b200 as tb
    from tnc_b200.contractionpath.slicing import SlicedPlan
    from tnc_b200.tensornetwork import NetworkPlan, contract_tensor_network
    info = card()
    ctx = tb.Context(0)
    lines = []

    def emit(name, workload, res, rel, extra=None):
        rec = {"object": name, "workload": workload, **info, "repeats": a.repeats, "rel_diff_c64_vs_c128": rel,
               "speedup_c64": res["complex128"]["median_s"] / res["complex64"]["median_s"], **res, **(extra or {})}
        print(json.dumps(rec), flush=True)
        lines.append(rec)

    # ---- the C2 pair: DMMA only, then with K1' (default engine) ----
    ops = {}
    for d in DTYPES:
        k = np.dtype(d).name
        ops[k] = (tb.DeviceTensor.from_numpy(ctx, ca, dtype=d), tb.DeviceTensor.from_numpy(ctx, cb, dtype=d),
                  tb.DeviceTensor.empty(ctx, [4] * 12, dtype=d))

    def c2(d):   # five pairs, then one download of the 4096 x 4096 result (268 MB complex128, 134 MB complex64)
        x, y, z = ops[np.dtype(d).name]
        for _ in range(5):
            tb.contract_pair_into(ctx, al, x, bl, y, z)
        ctx.synchronize()
        return z.to_numpy()
    for label, slices in (("dmma", 0), ("k1prime", 8)):
        ctx.set_tcgen05_slices(slices)
        c2(np.complex128), c2(np.complex64)          # warm-up
        res, rel = timed(ctx, c2, a.repeats)
        for r in res.values():
            r["seconds_per_pair"] = r["median_s"] / 5
        emit(f"c2_pair_{label}", "C2 pair 4^6 x 4^6 x 4^6, both operands permuted, 5 pairs per timed run", res, rel)
    ctx.set_tcgen05_slices(8)
    del ops

    # ---- networks: resident leaves through a plan (and end to end for the bench network) ----
    def resident(tn, path):
        plans = {np.dtype(d).name: NetworkPlan(tn, path, ctx=ctx, dtype=d) for d in DTYPES}
        for p in plans.values():
            p.stage(tn)
            p.run()                                    # warm-up
        res, rel = timed(ctx, lambda d: plans[np.dtype(d).name].run().to_numpy(), a.repeats)
        return res, rel, {k: p.info() for k, p in plans.items()}

    for name, work, tn, path in (
            ("net36_resident", f"bench.py network: random_circuit({NET['qubits']}, {NET['rounds']}), greedy path, leaves resident", net36, path36),
            ("config3_resident", "BASELINE config 3: random_circuit(24, 12), seed 1, greedy path, leaves resident", c3, path3),
            ("sycamore53_d10_resident", "Sycamore-53 depth 10, bench_inputs/sycamore53_d10.json path, leaves resident", d10, path10)):
        res, rel, pinfo = resident(tn, path)
        emit(name, work, res, rel, {"plan_info": pinfo})
        ctx.trim()
    for d in DTYPES:
        contract_tensor_network(net36, path36, ctx=ctx, dtype=d)
        contract_tensor_network(net36, path36, ctx=ctx, dtype=d)    # second sighting compiles the cached plan
    res, rel = timed(ctx, lambda d: contract_tensor_network(net36, path36, ctx=ctx, dtype=d).to_numpy(), a.repeats)
    emit("net36_end_to_end", "bench.py network, contract_tensor_network per run (leaf upload included)", res, rel)
    ctx.trim()

    # ---- config 5: Sycamore-53 depth 12, sliced, one GPU ----
    if not a.no_config5:
        d12, tn12, path12 = sycamore("sycamore53_d12.json")
        plans = {}
        setup = {}
        for d in DTYPES:
            t0 = time.perf_counter()
            plans[np.dtype(d).name] = SlicedPlan(tn12, path12, d12["sliced_legs"], ctx=ctx, dtype=d)
            setup[np.dtype(d).name] = time.perf_counter() - t0
        res, rel = timed(ctx, lambda d: plans[np.dtype(d).name].run().to_numpy(), max(1, a.repeats - 1))
        emit("config5_sycamore53_d12_sliced", f"Sycamore-53 depth 12, {plans['complex128'].n_slices} slices on one GPU", res, rel,
             {"setup_seconds_untimed": setup, "plan_info": {k: p.plan.info() for k, p in plans.items()}})
        del plans
        ctx.trim()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
