#!/usr/bin/env python
"""Batched marginal MAP against batched MPE and PR on config 5, and single MAP queries against MPE, one JSON line.

    python tools/map_bench.py [--iters 10] [--out FILE]

Config 5: the 500-variable BN of tools/mpe_batch_bench.py (W=6 K=3 seed=11, its 20 observed ids).  The MAP set M:
20 unobserved ids drawn by random.Random(9), if K9 accepts the constrained order (a dry plan's fused_info); otherwise
the last 20 unobserved ids.  Both candidates' constrained widths are recorded.  In one process:
1. device time per batch of BN.map_batch (MAP), BN.mpe_batch (MPE) and BN.partition_batch (PR) for 65 536 and 2^20
   sets resident on the device, CUDA events on the context's stream, the three alternating, on the default engine
   (K9) and with one launch per bucket forced (K8);
2. the kernels of one MAP batch from torch.profiler (runs of their own): the mixed interpreter against the decode;
3. a sample of sets of every MAP batch against single BN.map queries (value bits, MAP assignment, summed rows 0xFF);
4. end-to-end time of a single BN.map query against BN.mpe on asia, alarm, hepar2, network and andes (plans cached,
   host clock around calls that end in a device synchronise).
The card's name, power limit and SM clocks are read in the same process."""
import argparse
import gzip
import json
import os
import random
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from bnpp_b200 import capi, model, synth  # noqa: E402
from map_emulator import DryMAPPlan, rows as map_rows  # noqa: E402
from mpe_batch_bench import gpu_info, kernels, timed  # noqa: E402
from mpe_fused_interp import fused_info  # noqa: E402
from plan_emulator import describe  # noqa: E402

SCRATCH_BUDGET = 1 << 30        # bytes of argmax rows per slice (ve.cu, batch_slice)
SINGLE_NETS = ("asia", "alarm", "hepar2", "network", "andes")


def constrained(cards, scopes, observed, m):
    """-> (order, width, K9 lanes per set for 65 536 sets) of the constrained mf order, from a dry plan"""
    summed = [v for v in range(len(cards)) if v not in set(observed) and v not in set(m)]
    order, width = model.elim_order_constrained(cards, scopes, summed, m, "mf", observed=observed)
    p = DryMAPPlan(cards, scopes, observed, m, order)
    try:
        assert p.rc == 0, p.rc
        return order, width, fused_info(p.h, 1 << 16)[0]
    finally:
        p.close()


def single_queries(ctx, reps):
    """end-to-end ms of BN.map (3 MAP variables) and BN.mpe on the golden networks, the calls alternating"""
    from fused_interp import parse_uai
    models = json.load(gzip.open(os.path.join(ROOT, "tests", "golden", "models.json.gz"), "rt"))
    out = {}
    for name in SINGLE_NETS:
        m = models[name]
        cards, scopes, tables = parse_uai(m["uai"])
        bn = model.BN(ctx, cards, list(zip(scopes, tables)))
        ev = {int(k): v for k, v in next((c["evidence"] for c in m["pr"] if c["evidence"]), {}).items()}
        free = [v for v in range(len(cards)) if v not in ev]
        mv = sorted(random.Random("map-" + name).sample(free, min(3, len(free))))
        t = {"map": [], "mpe": []}
        for i in range(reps + 2):
            for k, fn in (("map", lambda: bn.map(mv, ev, "mf")), ("mpe", lambda: bn.mpe(ev, "mf"))):
                t0 = time.perf_counter()
                fn()
                dt = (time.perf_counter() - t0) * 1e3
                if i >= 2:
                    t[k].append(dt)
        out[name] = {"nvars": len(cards), "map_vars": mv, "observed": len(ev),
                     "map_ms_median": statistics.median(t["map"]), "mpe_ms_median": statistics.median(t["mpe"]),
                     "map_ms_min": min(t["map"]), "mpe_ms_min": min(t["mpe"]), "reps": reps}
        bn.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--sizes", default="65536,1048576")
    ap.add_argument("--sample", type=int, default=64)
    ap.add_argument("--single-reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("map_bench: needs a CUDA device")
    info = gpu_info()
    ctx = capi.Context(0)
    N, W, K, seed, nobs = 500, 6, 3, 11, 20
    uai = synth.random_bn_uai(N, W, K, seed)
    _, bn = model.from_uai_text(ctx, uai)
    evs = synth.evidence_batch(N, nobs, 1 << 16, seed=5, fixed_ids=True)       # the sets of tools/mpe_batch_bench.py
    observed = sorted(evs[0])
    free = [v for v in range(N) if v not in set(observed)]
    drawn = sorted(random.Random(9).sample(free, 20))
    _, w_drawn, g_drawn = constrained(bn.cards, bn.scopes, observed, drawn)
    block = free[-20:]
    _, w_block, g_block = constrained(bn.cards, bn.scopes, observed, block)
    mv, why = (drawn, "20 unobserved ids drawn by random.Random(9)") if g_drawn > 0 else \
        (block, "the last 20 unobserved ids: K9 refuses the constrained order of the 20 drawn ids (width %d)" % w_drawn)
    base = np.array([[e[v] for v in observed] for e in evs], dtype=np.uint8)
    rng = np.random.default_rng(7)
    mpe_order = bn.order(free, observed, "mf")[0]
    map_plan = bn._map_plan(mv, observed, "mf")
    mpe_plan = bn._cached_plan(("mpe", tuple(observed), tuple(mpe_order)), model.MPEPlan, observed, mpe_order)
    pr_plan = bn.plan(observed, mpe_order)
    desc = describe(map_plan.h)
    rows = sum(n for _, _, n in map_rows(desc, set(mv)))
    n_max = len(map_rows(desc, set(mv)))
    out = dict(info, config="config 5: 500-variable BN (W=6 K=3 seed=11), 20 observed ids fixed, evidence resident on the device",
               map_vars=mv, map_vars_choice=why, drawn_map_vars=drawn, drawn_constrained_width=w_drawn,
               drawn_k9_lanes=g_drawn, block_constrained_width=w_block, block_k9_lanes=g_block,
               map_argmax_rows_per_set=rows, max_steps=n_max,
               sum_steps=sum(1 for st in desc["steps"] if st["elim"] >= 0) - n_max, plan_steps=len(desc["steps"]), sizes={})
    for nb in [int(x) for x in a.sizes.split(",")]:
        if nb <= base.shape[0]:
            ev = base[:nb]
        else:
            ev = np.concatenate([base, np.stack([rng.integers(0, bn.cards[v], nb - base.shape[0]) for v in observed],
                                                axis=1).astype(np.uint8)])
        dev = torch.from_numpy(np.ascontiguousarray(ev)).to("cuda:%d" % ctx.device)
        torch.cuda.synchronize()
        slice_ = min(nb, max(1, SCRATCH_BUDGET // max(1, rows)))
        res = {"sets": nb, "map_sets_per_slice_k9": slice_, "map_slices_k9": -(-nb // slice_)}
        for engine, fused in (("k9", True), ("k8", False)):
            for p in (map_plan, mpe_plan, pr_plan):
                p.set_fused(fused)
            g = map_plan.fused_info(nb)[0] if fused else 0
            t = timed(ctx, {"pr": lambda: bn.partition_batch(observed, dev, "mf"),
                            "mpe": lambda: bn.mpe_batch(observed, dev, "mf"),
                            "map": lambda: bn.map_batch(mv, observed, dev, "mf")}, a.iters if fused else max(3, a.iters // 2))
            e = {"map_lanes_per_set": g, "iters": len(t["pr"])}
            for k in ("map", "mpe", "pr"):
                e[k + "_ms_median"] = statistics.median(t[k])
                e[k + "_ms_min"] = min(t[k])
                e[k + "_queries_per_s"] = nb / e[k + "_ms_median"] * 1e3
            e["map_over_mpe"] = e["map_ms_median"] / e["mpe_ms_median"]
            e["map_over_pr"] = e["map_ms_median"] / e["pr_ms_median"]
            e["map_kernels"] = kernels(ctx, lambda: bn.map_batch(mv, observed, dev, "mf"))
            value, assign = bn.map_batch(mv, observed, dev, "mf")
            ctx.sync()
            value, assign = value.cpu().numpy().copy(), assign.cpu().numpy().copy()
            pick = {0, nb - 1} | {b for k in range(1, -(-nb // slice_)) for b in (k * slice_ - 1, k * slice_)}
            pick = sorted(pick | set(random.Random(nb).sample(range(nb), a.sample)))
            summed = [v for v in free if v not in set(mv)]
            bad = 0
            for b in pick:
                v, xm, _ = bn.map(mv, {u: int(x) for u, x in zip(observed, ev[b])}, "mf")
                bad += int(np.float64(v).view(np.uint64) != value[b:b + 1].view(np.uint64)[0]
                           or any(int(assign[u, b]) != x for u, x in xm.items()) or (assign[summed, b] != 0xFF).any())
            e["sample_sets_checked"], e["sample_sets_differing"] = len(pick), bad
            res[engine] = e
        for p in (map_plan, mpe_plan, pr_plan):
            p.set_fused(True)
        out["sizes"][str(nb)] = res
        del dev
    bn.close()
    out["single_query_end_to_end"] = single_queries(ctx, a.single_reps)
    s = json.dumps(out)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
