#!/usr/bin/env python
"""Sharded MPE against sharded PR on the strong-scaling network, one JSON line.
    python tools/mpe_shard_bench.py [--queries 20] [--out FILE]                      (one GPU)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node G --master-addr 127.0.0.1 --master-port 29512 \\
        tools/mpe_shard_bench.py [--queries 20] [--out FILE]                          (G GPUs)

The network is synth.STRONG (N=76 W=44 K=4 seed=3, 8 observed leaves, min-fill width 30), sharded over the ranks as
`BN.partition` / `BN.mpe` shard it.  Every rank runs its slab through the product-level sharded entry points --
bnpp_ve_plan_run_sharded (PR: the rank's plan, then the all-reduce of the partition) and bnpp_mpe_plan_run_sharded
(MPE: the rank's plan, the all-gather of the records and the max-loc) -- with PR and MPE queries alternating, each
timed by CUDA events on the context's stream after a barrier, warm (plans resolved, graphs captured); a query's time is
the largest over the ranks, and the median over the queries is reported.  Also: every rank's peak bytes of
intermediates + argmax tables and its widest step (bnpp_ve_plan_info), the same from dry plans on the host for 1, 2, 4
and 8 ranks, and the sharded MPE value against the unsharded MPE query on rank 0.  The card's name and power limit are
read in the same process."""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from bnpp_b200 import capi, model, sharding, synth  # noqa: E402


class _Rank:
    def __init__(self, rank, world):
        self.rank, self.world = rank, world


class _DryCtx:
    """what a plan needs of a context to be created without a device (a dry plan)"""
    h = None

    def __init__(self):
        self.L = capi.lib()

    def check(self, rc):
        if rc != 0:
            raise capi.BnppError(rc, "dry plan")


def host_peaks(cards, scopes, ev):
    """-> {world: (largest per-rank peak bytes, largest per-rank widest step)} of dry MPE plans"""
    out = {}
    N = len(cards)
    dry = _DryCtx()
    free = [v for v in range(N) if v not in ev]
    full_order, _ = model.elim_order(cards, scopes, free, "mf", observed=sorted(ev))
    live = [[v for v in sc if v not in ev] for sc in scopes]
    for world in (1, 2, 4, 8):
        g = world.bit_length() - 1
        shard = sharding.pick_shard_vars(live, full_order, g)
        peak = step = 0
        for r in range(world):
            e = {**ev, **sharding.shard_evidence(shard, r)}
            order, _ = model.elim_order(cards, scopes, [v for v in range(N) if v not in e], "mf", observed=sorted(e))
            p = model.MPEPlan(dry, cards, scopes, sorted(e), order)
            peak, step = max(peak, p.peak_bytes), max(step, p.max_step_entries)
            p.close()
        out[world] = (peak, step)
    return out


def gpu_info(device):
    q = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    return {"gpu": torch.cuda.get_device_name(device), "power_limit_and_max_sm_clock": q.stdout.strip().splitlines()[0]
            if q.returncode == 0 and q.stdout.strip() else "unavailable"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from bnpp_b200.nccl import ShardComm
    ctx = capi.Context(local)
    comm = ShardComm(ctx, rank, world)
    N, W, K, seed, ev = synth.wide_bn("strong")
    bn = model.from_uai_text(ctx, synth.random_bn_uai(N, W, K, seed))[1]
    full, shard = bn.shard(ev, "mf", _Rank(rank, world)) if world > 1 else (dict(ev), [])
    observed = sorted(full)
    obs_val = [full[v] for v in observed]
    order, width = bn.order([v for v in range(N) if v not in full], full, "mf")
    p_pr = bn.plan(observed, order)
    p_mpe = model.MPEPlan(ctx, bn.cards, bn.scopes, observed, order)
    s = ctx.torch_stream
    with torch.cuda.stream(s):
        res = torch.empty(2, dtype=torch.float64, device="cuda")
        mbuf = torch.empty(2 + N, dtype=torch.int32, device="cuda")

    def pr():
        comm.run_sharded(p_pr, bn.table_ptrs, obs_val, res.data_ptr(), res.data_ptr() + 8)

    def mpe():
        comm.run_mpe_sharded(p_mpe, bn.table_ptrs, obs_val, mbuf.data_ptr(), mbuf.data_ptr() + 8)

    def barrier():
        if world > 1:
            dist.barrier()

    for _ in range(3):                      # plans resolved, graphs captured (from the second run on), pool warm
        pr()
        mpe()
    ctx.sync()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = {"pr": [], "mpe": []}
    for _ in range(args.queries):
        for name, fn in (("pr", pr), ("mpe", mpe)):
            ctx.sync()
            barrier()
            t0.record(s)
            fn()
            t1.record(s)
            t1.synchronize()
            t = torch.tensor([t0.elapsed_time(t1)], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms[name].append(float(t.item()))
    ctx.sync()
    z = float(res[1].item())
    host = mbuf.cpu().numpy()
    value = float(host[:2].view("float64")[0])
    assignment = [int(x) for x in host[2:].view("uint32")]
    peaks = torch.tensor([p_pr.peak_bytes, p_mpe.peak_bytes, p_mpe.max_step_entries], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(peaks, op=dist.ReduceOp.MAX)
    out = None
    if rank == 0:
        p_pr.close()
        p_mpe.close()
        bn.drop_plans()
        v1, a1, _ = bn.mpe(ev, "mf")              # the unsharded query on this GPU
        bn.drop_plans()
        hp = host_peaks(bn.cards, bn.scopes, ev)
        med_pr, med_mpe = statistics.median(ms["pr"]), statistics.median(ms["mpe"])
        out = {
            "metric": "sharded MPE vs sharded PR, strong-scaling network (synth.STRONG, min-fill width 30)",
            "gpus": world, **gpu_info(local), "queries": args.queries, "rank_width": width, "shard_vars": shard,
            "pr_ms_median": med_pr, "mpe_ms_median": med_mpe, "mpe_over_pr": med_mpe / med_pr,
            "pr_ms": ms["pr"], "mpe_ms": ms["mpe"],
            "rank_peak_bytes_pr": int(peaks[0].item()), "rank_peak_bytes_mpe": int(peaks[1].item()),
            "rank_max_step_entries_mpe": int(peaks[2].item()),
            "host_mpe_peak_bytes_by_gpus": {str(k): v[0] for k, v in hp.items()},
            "host_mpe_max_step_entries_by_gpus": {str(k): v[1] for k, v in hp.items()},
            "allgather_words": world * ((2 + N + 1) // 2 * 2),
            "pr_sharded": z, "mpe_sharded": value, "mpe_one_gpu": v1,
            "mpe_value_rel_diff": abs(value - v1) / v1, "assignment_equal": assignment == a1,
        }
        line = json.dumps(out)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")
    comm.close()
    if world > 1:
        dist.destroy_process_group()
    if out is not None and not math.isclose(out["mpe_sharded"], out["mpe_one_gpu"], rel_tol=1e-12):
        sys.exit(1)


if __name__ == "__main__":
    main()
