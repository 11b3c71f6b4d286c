#!/usr/bin/env python
"""MPE against PR on the GPU, one JSON line.   python tools/mpe_bench.py [--queries 30] [--out FILE]

1. config 4 (synth.wide_bn(1) with its evidence, min-fill): device time per query of PR (VEPlan.run) and MPE
   (MPEPlan.run_mpe), both replayed from their CUDA graphs, CUDA events on the context's stream, queries alternating;
2. the widest max-product step, event-timed with set_profiling: its bytes 8 * (sum #F_k + #out) + #out (the argmax
   table) over its time, against a device-to-device copy of 4 GiB measured in the same process (read + write bytes);
   the decode kernel on its own from torch.profiler (CUDA activities, a run of its own);
3. the golden networks end to end: BN.mpe against BN.partition (host clock around a query that ends in a sync).
The card's name, power limit and maximum SM clock are read in the same process."""
import argparse
import gzip
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from bnpp_b200 import capi, model, synth  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    return {"gpu": torch.cuda.get_device_name(0), "power_limit_and_max_sm_clock": q.stdout.strip().splitlines()[0]
            if q.returncode == 0 and q.stdout.strip() else "unavailable"}


def copy_peak(stream, nbytes=4 << 30, reps=10):
    """device-to-device copy bandwidth, read + write bytes per second"""
    with torch.cuda.stream(stream):
        a = torch.ones(nbytes // 8, dtype=torch.float64, device="cuda")
        b = torch.empty_like(a)
        b.copy_(a)
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        best = None
        for _ in range(reps):
            t0.record(stream)
            b.copy_(a)
            t1.record(stream)
            t1.synchronize()
            ms = t0.elapsed_time(t1)
            best = ms if best is None else min(best, ms)
    del a, b
    torch.cuda.empty_cache()
    return 2 * nbytes / (best * 1e-3)


def config4(ctx, queries):
    N, W, K, seed, ev = synth.wide_bn(1)
    _, bn = model.from_uai_text(ctx, synth.random_bn_uai(N, W, K, seed))
    assert all(c == 2 for c in bn.cards)
    observed = sorted(ev)
    obs_val = [ev[v] for v in observed]
    order, width = bn.order([v for v in range(N) if v not in ev], ev, "mf")
    pr = bn.plan(observed, order)
    mpe = model.MPEPlan(ctx, bn.cards, bn.scopes, observed, order)
    s = ctx.torch_stream
    with torch.cuda.stream(s):
        res = torch.zeros(2, dtype=torch.float64, device="cuda")
        buf = torch.zeros(2 + N, dtype=torch.int32, device="cuda")
    run_pr = lambda: pr.run(bn.table_ptrs, obs_val, res.data_ptr(), res.data_ptr() + 8)  # noqa: E731
    run_mpe = lambda: mpe.run_mpe(bn.table_ptrs, obs_val, buf.data_ptr(), buf.data_ptr() + 8)  # noqa: E731
    for _ in range(3):              # run 1 resolves the launches, run 2 builds the replay graph
        run_pr()
        run_mpe()
    ctx.sync()
    t = {"pr": [], "mpe": []}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(queries):
        for name, fn in (("pr", run_pr), ("mpe", run_mpe)):
            ev0.record(s)
            fn()
            ev1.record(s)
            ev1.synchronize()
            t[name].append(ev0.elapsed_time(ev1))
    value = float(buf[:2].cpu().view(torch.float64).item())
    out = {"N": N, "width": width, "observed": len(ev), "launches_pr": pr.n_launches, "launches_mpe": mpe.n_launches + 1,
           "pr_ms_median": statistics.median(t["pr"]), "mpe_ms_median": statistics.median(t["mpe"]),
           "pr_ms_min": min(t["pr"]), "mpe_ms_min": min(t["mpe"]), "queries_each": queries,
           "pr_peak_bytes": pr.peak_bytes, "mpe_peak_bytes": mpe.peak_bytes,
           "argmax_arena_bytes": mpe.peak_bytes - pr.peak_bytes, "Z": float(res[1].item()), "mpe_value": value}
    out["mpe_over_pr"] = out["mpe_ms_median"] / out["pr_ms_median"]
    return bn, mpe, run_mpe, out


def widest_step(ctx, mpe, run_mpe, peak, reps=5):
    mpe.set_profiling(True)
    runs = []
    for _ in range(reps):
        run_mpe()
        runs.append(mpe.step_stats())
    mpe.set_profiling(False)
    elim = [i for i, st in enumerate(runs[0]) if "_max<" in st["kernel"]]
    i = max(elim, key=lambda j: runs[0][j]["entries"])
    st = runs[0][i]
    ms = statistics.median(r[i]["ms"] for r in runs)
    n_out = st["entries"] // 2                      # binary network: the output has half the union's entries
    nbytes = st["bytes"] + n_out                    # 8 * (sum #F_k + #out) + the argmax byte per output entry
    rate = nbytes / (ms * 1e-3)
    return {"step": i, "kernel": st["kernel"], "k": st["k"], "union_entries": st["entries"], "bytes": nbytes,
            "ms_median": ms, "bytes_per_s": rate, "share_of_copy_peak": rate / peak}


def decode_time(ctx, run_mpe, reps=20):
    from torch.profiler import ProfilerActivity, profile
    run_mpe()
    ctx.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            run_mpe()
        ctx.sync()
    for e in prof.key_averages():
        if "mpe_decode" in e.key:
            us = getattr(e, "device_time", None) or getattr(e, "cuda_time", None)
            return {"decode_us": us, "decode_count": e.count}
    return {"decode_us": None, "decode_count": 0}


def small_networks(ctx, reps=30):
    models = json.load(gzip.open(os.path.join(ROOT, "tests", "golden", "models.json.gz"), "rt"))
    out = {}
    for name, m in models.items():
        _, bn = model.from_uai_text(ctx, m["uai"])
        for _ in range(3):
            bn.partition({}, "mf")
            bn.mpe({}, "mf")
        tp, tm = [], []
        for _ in range(reps):
            t0 = time.perf_counter()
            bn.partition({}, "mf")
            t1 = time.perf_counter()
            bn.mpe({}, "mf")
            tm.append((time.perf_counter() - t1) * 1e3)
            tp.append((t1 - t0) * 1e3)
        pr_plan = bn.plan([], bn._order_cache[((), "mf")])
        out[name] = {"pr_ms": round(statistics.median(tp), 4), "mpe_ms": round(statistics.median(tm), 4),
                     "pr_launches": 1 if pr_plan.fused_info(1)[0] else pr_plan.n_launches,
                     "mpe_launches": [p for k, p in bn._plans.items() if k[0] == "mpe"][0].n_launches + 1}
        bn.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=30)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mpe_bench: needs a CUDA device")
    info = gpu_info()
    ctx = capi.Context(0)
    peak = copy_peak(ctx.torch_stream)
    bn, mpe, run_mpe, c4 = config4(ctx, a.queries)
    wide = widest_step(ctx, mpe, run_mpe, peak)
    dec = decode_time(ctx, run_mpe)
    mpe.close()
    bn.close()
    small = small_networks(ctx)
    line = dict(info, copy_peak_bytes_per_s=peak, config4=c4, widest_max_step=wide, decode=dec, small_networks=small,
                targets={"mpe_over_pr_max": 1.25, "widest_step_share_min": 0.80})
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
