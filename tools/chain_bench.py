"""Windows on / off in one process (bnpp_tuning_set "chain_depth"): config 4 (bench.py's `value` network) and the
width-30 network (`strong`, unsharded), the two plans of a network timed alternately, every query a graph replay
timed by CUDA events, median of --reps; Z of the two plans compared bit for bit.  Prints one JSON line per network
with the card's name, power limit and SM clocks read in the same call.

    python tools/chain_bench.py [--reps 30] [--depths 4,1] [--nets 1,strong]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), [s.strip() for s in out.split(",")]))
    except Exception as e:
        return {"error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--depths", default="4,1", help="chain_depth values (4 = the default, 1 = no windows)")
    ap.add_argument("--nets", default="1,strong")
    args = ap.parse_args()
    import torch
    from bnpp_b200 import capi, model, synth
    ctx = capi.Context(0)
    s = ctx.torch_stream
    depths = [int(d) for d in args.depths.split(",")]
    for key in args.nets.split(","):
        key = key if key == "strong" else int(key)
        N, W, K, seed, ev = synth.wide_bn(key)
        _, bn = model.from_uai_text(ctx, synth.random_bn_uai(N, W, K, seed))
        obs = sorted(ev)
        order, width = bn.order([v for v in range(N) if v not in ev], ev, "mf")
        vals = [ev[v] for v in obs]
        plans = {}
        for d in depths:
            old = capi.tuning_set("chain_depth", d)
            plans[d] = model.VEPlan(ctx, bn.cards, bn.scopes, obs, order)
            capi.tuning_set("chain_depth", old)
        res = {d: torch.zeros(2, dtype=torch.float64, device="cuda") for d in depths}
        for d in depths:                       # first run, graph capture, warm replays
            for _ in range(4):
                plans[d].run(bn.table_ptrs, vals, res[d].data_ptr() + 8, res[d].data_ptr())
        ctx.sync()
        times = {d: [] for d in depths}
        for _ in range(args.reps):
            for d in depths:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(s)
                plans[d].run(bn.table_ptrs, vals, res[d].data_ptr() + 8, res[d].data_ptr())
                e1.record(s)
                e1.synchronize()
                times[d].append(e0.elapsed_time(e1))
        z = {d: res[d][0].item() for d in depths}
        zb = {d: res[d][0].cpu().numpy().tobytes().hex() for d in depths}
        rows = {}
        for d in depths:
            p = plans[d]
            med = statistics.median(times[d])
            rows["chain_depth=%d" % d] = {"median_ms": med, "min_ms": min(times[d]), "max_ms": max(times[d]),
                                          "launches": p.n_launches, "algorithmic_GB": p.bytes / 1e9, "Z": z[d],
                                          "union_entries_per_s": p.union_entries / med * 1e3}
        # per-launch profile of the first plan (CUDA events around every launch, graph replay off): the windows' rows
        prof = plans[depths[0]]
        prof.set_profiling(True)
        acc = None
        for _ in range(3):
            prof.run(bn.table_ptrs, vals, res[depths[0]].data_ptr() + 8, res[depths[0]].data_ptr())
            st = prof.step_stats()
            acc = st if acc is None else [dict(a, ms=a["ms"] + b["ms"]) for a, b in zip(acc, st)]
        prof.set_profiling(False)
        wide = [dict(r, ms=r["ms"] / 3, GBs=r["bytes"] / (r["ms"] / 3) / 1e6) for r in acc if r["bytes"] >= 1e8]
        out = {"profiled_chain_depth": depths[0], "wide_launches": wide,
               "network": "config 4 key=%s (N=%d W=%d K=%d seed=%d, min-fill width %d)" % (key, N, W, K, seed, width),
               "reps": args.reps, "Z_same_bits": len(set(zb.values())) == 1, "plans": rows, "card": card()}
        print(json.dumps(out), flush=True)
        for p in plans.values():
            p.close()
        bn.close()
    ctx.close()


if __name__ == "__main__":
    main()
