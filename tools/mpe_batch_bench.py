#!/usr/bin/env python
"""Batched MPE against batched PR on config 5 (500-variable BN, W=6 K=3 seed=11, 20 observed ids), one JSON line.

    python tools/mpe_batch_bench.py [--iters 10] [--out FILE]

For 65 536 and 2^20 evidence sets (resident on the device), in one process:
1. device time per batch of BN.partition_batch (PR) and BN.mpe_batch (MPE), CUDA events on the context's stream, the
   two alternating, on the default engine (K9: ve_fused / ve_fused_max) and with one launch per bucket forced (K8);
2. the kernels of one MPE and one PR batch from torch.profiler (CUDA activities, runs of their own): the decode launch
   on its own, the max-mode interpreter, the evidence check;
3. the argmax rows per set (R), the sets per slice and the scratch bytes;
4. a sample of sets of every batch against single BN.mpe queries (value bits and assignment).
The card's name, power limit and SM clocks are read in the same process."""
import argparse
import json
import os
import random
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from bnpp_b200 import capi, model, synth  # noqa: E402
from plan_emulator import describe  # noqa: E402

SCRATCH_BUDGET = 1 << 30        # bytes of argmax rows per slice (ve.cu, batch_slice)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    return {"gpu": torch.cuda.get_device_name(0), "power_limit_max_sm_clock_current_sm_clock": q.stdout.strip().splitlines()[0]
            if q.returncode == 0 and q.stdout.strip() else "unavailable"}


def timed(ctx, fns, iters):
    """-> {name: [ms per call]}, the calls alternating"""
    s = ctx.torch_stream
    for _ in range(3):
        for fn in fns.values():
            fn()
    ctx.sync()
    t = {k: [] for k in fns}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(iters):
        for k, fn in fns.items():
            e0.record(s)
            fn()
            e1.record(s)
            e1.synchronize()
            t[k].append(e0.elapsed_time(e1))
    return t


def kernels(ctx, fn, reps=3):
    """device time per kernel name over `reps` calls -> {name: {"us_per_call", "launches_per_call"}}"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    ctx.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        ctx.sync()
    out = {}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", None) or 0.0
        if us <= 0:
            continue
        name = e.key.split("(")[0].replace("void ", "")[:60]
        out[name] = {"us_per_call": round(us / reps, 1), "launches_per_call": e.count / reps}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--sizes", default="65536,1048576")
    ap.add_argument("--sample", type=int, default=64)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mpe_batch_bench: needs a CUDA device")
    info = gpu_info()
    ctx = capi.Context(0)
    N, W, K, seed, nobs = 500, 6, 3, 11, 20
    _, bn = model.from_uai_text(ctx, synth.random_bn_uai(N, W, K, seed))
    evs = synth.evidence_batch(N, nobs, 1 << 16, seed=5, fixed_ids=True)       # the sets of tools/batch_bench.py
    observed = sorted(evs[0])
    base = np.array([[e[v] for v in observed] for e in evs], dtype=np.uint8)
    rng = np.random.default_rng(7)
    order = bn.order([v for v in range(N) if v not in set(observed)], observed, "mf")[0]
    mpe_plan = bn._cached_plan(("mpe", tuple(observed), tuple(order)), model.MPEPlan, observed, order)
    desc = describe(mpe_plan.h)
    rows = sum(int(np.prod([c for _, c in st["scope"]], dtype=np.int64)) for st in desc["steps"] if st["elim"] >= 0)
    n_elim = sum(1 for st in desc["steps"] if st["elim"] >= 0)
    out = dict(info, config="config 5: 500-variable BN (W=6 K=3 seed=11), 20 observed ids fixed, evidence resident on the device",
               argmax_rows_per_set=rows, eliminating_steps=n_elim, plan_steps=len(desc["steps"]), sizes={})
    for nb in [int(x) for x in a.sizes.split(",")]:
        if nb <= base.shape[0]:
            ev = base[:nb]
        else:
            ev = np.concatenate([base, np.stack([rng.integers(0, bn.cards[v], nb - base.shape[0]) for v in observed],
                                                axis=1).astype(np.uint8)])
        dev = torch.from_numpy(np.ascontiguousarray(ev)).to("cuda:%d" % ctx.device)
        torch.cuda.synchronize()
        slice_ = min(nb, max(1, SCRATCH_BUDGET // rows))
        res = {"sets": nb, "sets_per_slice_k9": slice_, "slices_k9": -(-nb // slice_), "scratch_bytes_k9": rows * slice_}
        for engine, fused in (("k9", True), ("k8", False)):
            mpe_plan.set_fused(fused)
            pr_plan = bn.plan(observed, order)
            pr_plan.set_fused(fused)
            g = mpe_plan.fused_info(nb)[0] if fused else 0
            t = timed(ctx, {"pr": lambda: bn.partition_batch(observed, dev, "mf"),
                            "mpe": lambda: bn.mpe_batch(observed, dev, "mf")}, a.iters if fused else max(3, a.iters // 2))
            e = {"lanes_per_set": g, "pr_ms_median": statistics.median(t["pr"]), "mpe_ms_median": statistics.median(t["mpe"]),
                 "pr_ms_min": min(t["pr"]), "mpe_ms_min": min(t["mpe"]), "iters": len(t["pr"])}
            e["mpe_over_pr"] = e["mpe_ms_median"] / e["pr_ms_median"]
            e["pr_queries_per_s"] = nb / e["pr_ms_median"] * 1e3
            e["mpe_queries_per_s"] = nb / e["mpe_ms_median"] * 1e3
            e["mpe_kernels"] = kernels(ctx, lambda: bn.mpe_batch(observed, dev, "mf"))
            e["pr_kernels"] = kernels(ctx, lambda: bn.partition_batch(observed, dev, "mf"))
            # a sample against single queries: every slice boundary and random sets
            value, assign = bn.mpe_batch(observed, dev, "mf")
            ctx.sync()
            value, assign = value.cpu().numpy().copy(), assign.cpu().numpy().copy()
            pick = {0, nb - 1} | {b for k in range(1, -(-nb // slice_)) for b in (k * slice_ - 1, k * slice_)}
            pick = sorted(pick | set(random.Random(nb).sample(range(nb), a.sample)))
            bad = 0
            for b in pick:
                v, asg, _ = bn.mpe({u: int(x) for u, x in zip(observed, ev[b])}, "mf")
                bad += int(np.float64(v).view(np.uint64) != value[b:b + 1].view(np.uint64)[0] or list(assign[:, b]) != asg)
            e["sample_sets_checked"], e["sample_sets_differing"] = len(pick), bad
            res[engine] = e
            pr_plan.set_fused(True)
        mpe_plan.set_fused(True)
        out["sizes"][str(nb)] = res
        del dev
    s = json.dumps(out)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    bn.close()
    ctx.close()


if __name__ == "__main__":
    main()
