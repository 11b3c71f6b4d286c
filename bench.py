#!/usr/bin/env python
"""bench.py -- headline benchmark of the bn-pp factor-algebra hot path on B200.

Metric (BASELINE.json): factor entries/sec of fused product+sum-out, measured on config 4: exact PR by variable
elimination (min-fill) on the synthetic "wide" Bayesian network whose largest elimination step is a 2^28-entry fp64
union table, with observed leaves (so the result is a non-trivial P(e) that the unmodified reference computed too:
tests/golden/wide.json).  One step = one full PR query: every bucket of the elimination order is one fused
product+sum-out launch, intermediates stay in HBM.  "entries" = sum over the elimination steps of the union-table size
(SURVEY 8d).

  value    : device-timed, CPTs already resident, plan prebuilt (graph replay).
  e2e      : BN.partition(evidence, "mf", comm=...) from HOST buffers each step: pinned CPTs -> H2D, min-fill ordering on
             the host, planning, the launches, (N > 1: the NCCL sum-out), scalar -> D2H.  Nothing cached.
  roofline : the widest fused launch, algorithmic bytes 8 * (sum #operands + #out) over its CUDA-event duration inside
             a timed pass, against MEASURED_PEAKS.json.
  golden   : Z (and at N > 1 every rank's partial) against the reference's own numbers; a mismatch > 1e-9 exits 1.

N > 1 (torchrun), two series on the same line:
  weak   (`value`)  : the network is too wide for one GPU by log2(N) variables (width 27 + log2 N); each rank eliminates
                      the slab selected by fixing those variables to its rank's bits; the cross-shard sum-out is one
                      NCCL all-reduce of the partition (bnpp_ve_plan_run_sharded).  Per-GPU work stays fixed.
  strong (`strong`) : ONE fixed network (width 30, the N = 8 weak network) at every N.
  pr_queries        : config 5 -- 65 536 (and 2^20) evidence sets on the 500-variable network split over the ranks.

N = 1 adds the legs that pin every other number quoted in DESIGN.md: `shapes` (SURVEY 8d headline shapes, mixed
cardinalities, multi-valued elimination), `configs_1_3` (latency-bound configs), `multivalued` (Munin1's widest
step), `same_sample` (this GPU on the reference arm's own sample network) and `cpu_baseline`.

--impl reference: the UNMODIFIED reference (oracle/_ref/ref_harness) on the host cores, on a bounded sample of the
config-4 generator chosen so that K + W steps end within a few minutes; nothing of bnpp_b200's native code is loaded.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "factor entries/sec (fused product+sum-out), VE PR on 2^28-entry tables"
UNIT = "entries/s"

# bounded CPU samples of the config-4 generator (N, W, K, seed), largest first; min-fill width / union entries per
# query (from the reference's own order): 21 / 1.49e7, 19 / 3.19e6, 16 / 1.27e6.  The reference needs ~0.5 us per entry.
CPU_SAMPLES = [(48, 26, 4, 3), (42, 20, 4, 3), (44, 20, 4, 5)]
CPU_SAMPLE_ENTRIES = [1.486e7, 3.188e6, 1.269e6]
CPU_RATE = 2.0e6            # entries/s per reference process, for choosing the sample only
CPU_BUDGET_S = 150.0        # whole --impl reference run


def pick_cpu_sample(steps, warmup):
    for s, e in zip(CPU_SAMPLES, CPU_SAMPLE_ENTRIES):
        if e / CPU_RATE * (steps + warmup) <= CPU_BUDGET_S:
            return s
    return CPU_SAMPLES[-1]


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons, sampled back to back from just before the timed regions until after
    them (B200_PROFILING.md recipe; in-process NVML when available: a sample every millisecond)."""
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.stop_flag = False
        self.max_mhz = None

    def run(self):
        try:
            self._run_nvml()
        except Exception:
            self._run_smi()

    def _run_nvml(self):
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        bits = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self.stop_flag:
            self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            for nm, b in bits.items():
                if r & b:
                    self.reasons.add(nm)
            time.sleep(0.001)

    def _run_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for nm, v in zip(self.NAMES, f[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(nm)
            except Exception:
                pass

    def summary(self):
        self.stop_flag = True
        self.join(timeout=6)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def union_entries(scopes, order):
    """sum over elimination steps of the union-table size (binary variables), bucket elimination"""
    rank = {v: i for i, v in enumerate(order)}
    buckets = {v: [] for v in order}
    for sc in scopes:
        live = [v for v in sc if v in rank]
        if live:
            buckets[min(live, key=rank.get)].append(set(live))
    total = 0
    for v in order:
        if not buckets[v]:
            continue
        u = set().union(*buckets[v])
        total += 2 ** len(u)
        u.discard(v)
        if u:
            buckets[min(u, key=rank.get)].append(u)
    return total


# ------------------------------------------------------------------------------------------------------------
# the reference arm (and the cpu_baseline of the GPU arm): oracle/_ref only
# ------------------------------------------------------------------------------------------------------------
def cpu_reference_leg(sample, steps=1, warmup=0, procs=None):
    """times the unmodified reference (oracle/_ref/ref_harness, BN::partition with -mf) on `sample`.  The reference
    is single-threaded per query, so all host cores are used the only way it can use them: `procs` independent
    queries side by side (one process each); value = all their entries / wall time.  The entry count comes from the
    order the reference itself prints.  Nothing of bnpp_b200's native library is loaded here."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import concurrent.futures
    import oracle as orc
    from bnpp_b200 import synth          # pure-Python generator
    N, W, K, seed = sample
    text = synth.random_bn_uai(N, W, K, seed)
    scopes, _ = synth.random_bn_scopes(N, W, K, seed)
    path = "/tmp/bnpp_cpu_sample_%d.uai" % os.getpid()
    with open(path, "w") as f:
        f.write(text)
    if procs is None:
        procs = max(1, min(os.cpu_count() or 1, 32))
    if orc.have_ref():
        kind = "reference"
        rows = orc.RefHarness().run(["model " + path, "opt mf", "order"])
        o = [r for r in rows if r[0] == "ORDER"][0]
        width, order = int(o[1]), [int(x) for x in o[3:]]

        def one(_):
            rows = orc.RefHarness().run(["model " + path, "opt mf", "pr"], timeout=3000)
            pr = [r for r in rows if r[0] == "PR"][0]
            return float(pr[1]), float(pr[2])
    else:
        kind = "port"
        procs = 1
        m = orc.read_uai(path)
        order, width = list(range(N)), -1

        def one(_):
            t0 = time.perf_counter()
            z = orc.partition(m, {}, order)
            return z, (time.perf_counter() - t0) * 1e3
    entries = union_entries(scopes, order)
    walls, z, per_query_ms = [], None, []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        with concurrent.futures.ThreadPoolExecutor(procs) as ex:     # each task is its own OS process (the harness)
            res = list(ex.map(one, range(procs)))
        if it >= warmup:
            walls.append(time.perf_counter() - t0)
            per_query_ms += [r[1] for r in res]
        z = res[0][0]
    os.unlink(path)
    wall = sum(walls) / len(walls)
    return {"value": entries * procs / wall, "unit": UNIT, "cores": procs, "kind": kind,
            "sample": "config-4 generator N=%d W=%d K=%d seed=%d, no evidence (min-fill width %d, %d union entries per query); "
                      "%d concurrent single-threaded queries per step (the reference has no threading), %d timed step(s) after "
                      "%d warm-up, %.2f s wall each, %.2f s per query inside the reference; Z=%.12g"
                      % (N, W, K, seed, width, entries, procs, len(walls), warmup, wall,
                         sum(per_query_ms) / len(per_query_ms) / 1e3, z),
            "sample_network": list(sample), "sample_entries": entries, "sample_width": width,
            "steps_run": len(walls), "Z": z}, wall * 1e3


def config5_cpu_leg(text, evs, procs=None, per_proc=2):
    """the reference's BN::partition (-mf) on the first evidence sets of config 5: `procs` harness processes side by
    side (the reference is single-threaded), `per_proc` queries each -> (queries/s, cores, kind, Z of set 0)"""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import concurrent.futures
    import oracle as orc
    if not orc.have_ref():
        return None
    if procs is None:
        procs = max(1, min(os.cpu_count() or 1, 32))
    path = "/tmp/bnpp_cpu_config5_%d.uai" % os.getpid()
    with open(path, "w") as f:
        f.write(text)

    def one(i):
        script = ["model " + path]
        for ev in evs[i * per_proc:(i + 1) * per_proc]:
            script += ["evidset %d %s" % (len(ev), " ".join("%d %d" % kv for kv in sorted(ev.items()))), "opt mf", "pr"]
        rows = orc.RefHarness().run(script, timeout=600)
        return [float(r[1]) for r in rows if r[0] == "PR"]
    t0 = time.perf_counter()
    with concurrent.futures.ThreadPoolExecutor(procs) as ex:
        res = list(ex.map(one, range(procs)))
    wall = time.perf_counter() - t0
    os.unlink(path)
    n = sum(len(r) for r in res)
    return {"value": n / wall, "unit": "queries/s", "cores": procs, "kind": "reference",
            "sample": "%d evidence sets of the same batch, %d concurrent single-threaded reference processes x %d queries "
                      "(model load included), %.2f s wall" % (n, procs, per_proc, wall)}, res[0][0]


# ------------------------------------------------------------------------------------------------------------
# GPU legs
# ------------------------------------------------------------------------------------------------------------
class Dist:
    """rank / world and the two communicators: torch.distributed (plumbing: rendezvous, timing barriers, max over
    ranks) and the product's own NCCL communicator for the one collective of the path"""

    def __init__(self):
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.shard_comm = None

    def init(self, ctx):
        import torch
        if self.world > 1:
            from bnpp_b200.nccl import ShardComm
            self.shard_comm = ShardComm(ctx, self.rank, self.world)
            with torch.cuda.stream(ctx.torch_stream):
                warm = torch.zeros(1, dtype=torch.float64, device="cuda")
            for _ in range(3):                           # NCCL builds its channels on the first collective: not part of a step
                self.shard_comm.allreduce_sum(warm.data_ptr(), 1)
            ctx.sync()

    def barrier(self):
        import torch
        import torch.distributed as dist
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max(self, x):
        import torch
        import torch.distributed as dist
        if self.world == 1:
            return float(x)
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum(self, x):
        import torch
        import torch.distributed as dist
        if self.world == 1:
            return float(x)
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t)
        return float(t.item())

    def gather(self, obj):
        import torch.distributed as dist
        if self.world == 1:
            return [obj]
        out = [None] * self.world
        dist.all_gather_object(out, obj)
        return out


def load_wide_golden():
    p = os.path.join(ROOT, "tests", "golden", "wide.json")
    return json.load(open(p))["networks"] if os.path.exists(p) else {}


def wide_leg(ctx, D, key, steps, warmup, profile, e2e, sampler=None):
    """exact PR on one config-4 network (`key`: a GPU count of synth.WIDE, or "strong"), sharded over D.world ranks.
    -> dict with device-timed entries/s, e2e, golden comparison, per-launch stats (profile=True)"""
    import torch
    from bnpp_b200 import model, sharding, synth
    N, W, K, seed, base_ev = synth.wide_bn(key)
    text = synth.random_bn_uai(N, W, K, seed)
    _, bn = model.from_uai_text(ctx, text)
    stream = ctx.torch_stream
    comm = D.shard_comm
    variables0 = [v for v in range(N) if v not in base_ev]
    full_order, full_width = bn.order(variables0, base_ev, "mf")
    full_entries = union_entries(bn.conditioned_scopes(set(base_ev)), full_order)
    evidence, shard_vars = bn.shard(base_ev, "mf", comm)
    variables = [v for v in range(N) if v not in evidence]
    order, width = bn.order(variables, evidence, "mf")
    plan = bn.plan(sorted(evidence), order)
    obs_val = [evidence[v] for v in sorted(evidence)]
    with torch.cuda.stream(stream):
        res = torch.zeros(4, dtype=torch.float64, device="cuda")

    def one_query():
        if comm is not None:
            comm.run_sharded(plan, bn.table_ptrs, obs_val, res.data_ptr(), res.data_ptr() + 8)
        else:
            plan.run(bn.table_ptrs, obs_val, res.data_ptr(), res.data_ptr() + 8)

    # this rank's slab on its own first (no collective): compared with the reference's value for that slab
    plan.run(bn.table_ptrs, obs_val, res.data_ptr() + 16, res.data_ptr() + 24)
    ctx.sync()
    z_local = float(res[3].item())
    for _ in range(max(0, warmup - 1)):
        one_query()
    ctx.sync()
    if sampler is not None:
        sampler.start()
    D.barrier()
    launches0 = ctx.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        one_query()                 # the plan replays as one CUDA graph (+ one all-reduce at N > 1); no host sync inside
    e1.record(stream)
    D.barrier()
    dev_ms = D.max(e0.elapsed_time(e1))
    gpu_launches = ctx.launches - launches0
    last = res[:2].cpu().numpy()        # what the last timed step returned, before the passes below overwrite `res`
    z_total = float(res[1].item())
    entries_rank = plan.union_entries
    entries_all = D.sum(entries_rank)
    out = {"network": [N, W, K, seed], "evidence": {str(k): v for k, v in base_ev.items()}, "width": full_width,
           "width_per_rank": width, "shard_vars": shard_vars, "n_launches": plan.n_launches,
           "entries_per_rank": entries_rank, "entries_all_ranks": entries_all, "entries_unsharded": full_entries,
           "redundant_work": entries_all / full_entries if full_entries else None,
           "steps": steps, "ms_per_step": dev_ms / steps, "value": entries_all * steps / (dev_ms / 1e3),
           "useful_value": full_entries * steps / (dev_ms / 1e3),
           "gpu_launches": gpu_launches, "Z": z_total, "Z_rank": z_local, "bytes_per_step": plan.bytes,
           "peak_intermediate_GB": plan.peak_bytes / 1e9, "max_step_entries": plan.max_step_entries,
           "outputs": {"result": last[:1], "partition": last[1:]}}

    # golden: the reference's own numbers (oracle/make_wide_golden.py), total and per slab
    gold = load_wide_golden().get("8" if key == "strong" else str(key))
    chk = {"available": False}
    if gold and gold.get("partials"):
        def pr_of(assign):
            want = 0.0
            hit = 0
            for k_, p_ in gold["partials"].items():
                kv = dict((int(a.split("=")[0]), int(a.split("=")[1])) for a in k_.split(",") if a)
                if all(kv.get(v) == val for v, val in assign.items()):
                    want += p_["pr"]
                    hit += 1
            return want, hit
        want_total, n_total = pr_of({})
        mine = {v: evidence[v] for v in shard_vars}
        want_rank, n_rank = pr_of(mine)
        complete = n_total == len(gold["partials"]) == (8 if key == "strong" else int(key))
        ok_vars = set(shard_vars) <= set(gold.get("shard_vars", []))
        if complete and ok_vars and n_rank * D.world == n_total:
            errs = D.gather(abs(z_local - want_rank) / want_rank)
            chk = {"available": True, "Z_reference": want_total, "rel_err": abs(z_total - want_total) / want_total,
                   "rank_partial_rel_err_max": max(errs), "reference_runs": n_total,
                   "source": "tests/golden/wide.json (oracle/_ref, BN::partition -mf, one run per slab)"}
            chk["ok"] = chk["rel_err"] <= 1e-9 and chk["rank_partial_rel_err_max"] <= 1e-9
    out["golden"] = chk

    if profile:
        # second timed pass, same K steps, with a CUDA event pair around EVERY launch on the launching stream
        # (graph replay off): this is where the roofline's per-launch durations come from
        plan.set_profiling(True)
        plan.run(bn.table_ptrs, obs_val, res.data_ptr(), res.data_ptr() + 8)      # untimed: the events are created here
        plan.step_stats()
        per_launch = None
        # The launches of a step are enqueued one by one from the host; while the GPU is faster than the host (the small
        # steps at the start of a query) a kernel's start event fires before the kernel itself is in the queue, and the
        # gap lands in its measured duration (0.33-0.40 ms run to run for the widest launch).  So every step is enqueued
        # BEHIND a gate -- the stream waits for an event recorded after a fixed delay on a side stream -- and then runs
        # back to back on the device.
        side = torch.cuda.Stream()
        for _ in range(steps):
            with torch.cuda.stream(side):
                torch.cuda._sleep(6_000_000)        # ~3 ms at 1.9 GHz: more than the host needs to enqueue a query
                gate = torch.cuda.Event()
                gate.record(side)
            stream.wait_event(gate)
            plan.run(bn.table_ptrs, obs_val, res.data_ptr(), res.data_ptr() + 8)
            st = plan.step_stats()
            per_launch = st if per_launch is None else [dict(a, ms=a["ms"] + b["ms"]) for a, b in zip(per_launch, st)]
        torch.cuda.synchronize()
        out["per_launch"] = [dict(a, ms=a["ms"] / steps) for a in per_launch]
        out["profiled_ms"] = sum(a["ms"] for a in out["per_launch"])
        plan.set_profiling(False)

    if e2e:
        for _ in range(2):
            bn.drop_plans()
            bn.reupload()
            bn.partition(base_ev, "mf", comm=comm)
        D.barrier()
        t0 = time.perf_counter()
        parts = {}
        for _ in range(steps):
            bn.drop_plans()               # nothing cached: ordering + planning are paid every step
            bn.reupload()                 # pinned host CPTs -> HBM
            z_e2e, _ = bn.partition(base_ev, "mf", comm=comm)     # ... launches ... (all-reduce) ... scalar -> host
            for kk, vv in bn.last_timing.items():
                parts[kk] = parts.get(kk, 0.0) + vv / steps
        e2e_s = D.max(time.perf_counter() - t0)
        out["e2e"] = {"value": entries_all * steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": bn.h2d_bytes,
                      "d2h_bytes_per_step": 16, "ms_per_step": e2e_s / steps * 1e3, "host_breakdown_ms": parts, "Z": z_e2e,
                      "what": "nothing cached: pinned host CPTs -> HBM, host min-fill ordering, planning, launches, scalar D2H, every step"}
        # steady state of the same call: the API keeps the plan of an observed-id set (as it does for config 5);
        # a step still uploads the CPTs from pinned host memory, runs the query and reads the scalar back
        for _ in range(2):
            bn.reupload()
            bn.partition(base_ev, "mf", comm=comm)
        D.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            bn.reupload()
            z_st, _ = bn.partition(base_ev, "mf", comm=comm)
        st_s = D.max(time.perf_counter() - t0)
        out["e2e"]["steady"] = {"value": entries_all * steps / st_s, "unit": UNIT, "ms_per_step": st_s / steps * 1e3, "Z": z_st,
                                "what": "plan of the observed-id set kept by the API; H2D CPTs, launches, scalar D2H every step"}
    bn.close()
    return out


def config5_leg(ctx, D, nsets, steps, warmup, cpu_arm):
    """The other half of BASELINE.json's metric -- VE PR queries/sec -- on config 5: `nsets` evidence sets on the
    500-variable BN, PR per set, the sets split contiguously over the ranks (no collective on the path)."""
    import numpy as np
    import torch
    from bnpp_b200 import model, sharding, synth
    N, W, K, seed, nobs = 500, 6, 3, 11, 20
    text = synth.random_bn_uai(N, W, K, seed)
    _, bn = model.from_uai_text(ctx, text)
    if nsets <= 65536:
        evs = synth.evidence_batch(N, nobs, nsets, seed=5, fixed_ids=True)
        observed = sorted(evs[0])
        allv = np.array([[ev[v] for v in observed] for ev in evs], dtype=np.uint8)
        how = "random.Random(5)"
    else:
        evs = synth.evidence_batch(N, nobs, 4, seed=5, fixed_ids=True)
        observed = sorted(evs[0])
        allv = np.random.default_rng(5).integers(0, 2, (nsets, nobs), dtype=np.uint8)
        how = "numpy default_rng(5)"
    lo, hi = sharding.batch_slice(D.rank, D.world, nsets)
    host = torch.from_numpy(allv[lo:hi].copy()).pin_memory()
    dev = host.cuda()
    s = ctx.torch_stream
    for _ in range(max(3, warmup)):
        z = bn.partition_batch(observed, dev, "mf")
    ctx.sync()
    D.barrier()
    l0 = ctx.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    for _ in range(steps):
        z = bn.partition_batch(observed, dev, "mf")
    e1.record(s)
    D.barrier()
    z_last = z.cpu().numpy()            # `z` is the model's result buffer: the calls below write it again
    ms = D.max(e0.elapsed_time(e1)) / steps
    launches = (ctx.launches - l0) // steps
    plan = [p for k_, p in bn._plans.items()][0]
    lanes, arena, n_steps = plan.fused_info(hi - lo)
    # end to end, steady state: the API keeps the plan of an observed-id set (order, program) -- every call pays
    # the H2D of its evidence slice, the launch and the D2H of every Z
    zh = torch.empty(hi - lo, dtype=torch.float64).pin_memory()

    def call():
        zz = bn.partition_batch(observed, None, "mf", host_values=host)
        with torch.cuda.stream(s):
            zh.copy_(zz, non_blocking=True)
        ctx.sync()
    call()
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        call()
    e2e_ms = D.max((time.perf_counter() - t0) * 1e3) / steps
    # ... and cold: ordering, planning and the program upload paid by the call as well
    t0 = time.perf_counter()
    for _ in range(min(steps, 3)):
        bn.drop_plans()
        call()
    cold_ms = D.max((time.perf_counter() - t0) * 1e3) / min(steps, 3)
    z0 = D.gather(float(zh[0]))[0]
    bn.close()
    cpu = None
    if cpu_arm and D.rank == 0 and nsets <= 65536:
        try:
            got = config5_cpu_leg(text, evs)
            if got:
                cpu, z_ref = got
                cpu["Z_set0_reference"], cpu["Z_set0_gpu"] = z_ref, z0
        except Exception as e:
            cpu = {"error": "%s: %s" % (type(e).__name__, e)}
    return {"metric": "VE PR queries/sec", "value": nsets / ms * 1e3, "unit": "queries/s", "ms_per_batch": ms, "n_sets": nsets,
            "sets_per_rank": hi - lo,
            "config": {"workload": "config 5: %d evidence sets (%s), synthetic BN N=%d W=%d K=%d seed=%d, %d observed ids fixed, "
                                   "PR per set via VE (min-fill), contiguous slices over %d rank(s), no collective"
                                   % (nsets, how, N, W, K, seed, nobs, D.world),
                       "l2_flush": "none: the launch reads its evidence slice, 64 KB of CPTs and its program and writes 8 B per "
                                   "set; the intermediates stay in shared memory, so this leg is instruction-bound, not HBM-bound"},
            "e2e": {"value": nsets / e2e_ms * 1e3, "unit": "queries/s", "ms_per_batch": e2e_ms,
                    "h2d_bytes_per_step": int(host.numel()), "d2h_bytes_per_step": 8 * (hi - lo),
                    "what": "steady state: plan of the observed-id set kept by the API; H2D evidence, launch, D2H of every Z"},
            "e2e_cold": {"value": nsets / cold_ms * 1e3, "unit": "queries/s", "ms_per_batch": cold_ms,
                         "what": "nothing cached: host min-fill ordering, planning and program upload inside the call"},
            "gpu_launches_per_batch": launches, "union_entries_per_s": plan.union_entries * nsets / ms * 1e3,
            "kernel": ("ve_fused: one launch, %d lanes per evidence set, %d doubles of shared memory per set, %d steps"
                       % (lanes, arena, n_steps)) if lanes else "contract_batched: one launch per bucket",
            "sample_Z": z0, "cpu_baseline": cpu, "outputs": {"z": z_last}}


def same_sample_leg(ctx, sample, steps):
    """this GPU on the very network the reference arm times (same generator parameters, no evidence, -mf)"""
    import torch
    from bnpp_b200 import model, synth
    N, W, K, seed = sample
    _, bn = model.from_uai_text(ctx, synth.random_bn_uai(N, W, K, seed))
    order, width = bn.order(list(range(N)), {}, "mf")
    plan = bn.plan([], order)
    res = torch.zeros(2, dtype=torch.float64, device="cuda")
    s = ctx.torch_stream
    for _ in range(3):
        plan.run(bn.table_ptrs, [], res.data_ptr(), res.data_ptr() + 8)
    ctx.sync()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    for _ in range(steps):
        plan.run(bn.table_ptrs, [], res.data_ptr(), res.data_ptr() + 8)
    e1.record(s)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    t0 = time.perf_counter()
    for _ in range(steps):
        bn.drop_plans()
        bn.reupload()
        z, _ = bn.partition({}, "mf")
    e2e_ms = (time.perf_counter() - t0) * 1e3 / steps
    ent = plan_entries = union_entries(bn.scopes, order)
    bn.close()
    return {"sample_network": list(sample), "width": width, "entries": ent, "steps": steps, "ms_per_query": ms, "value": plan_entries / ms * 1e3,
            "unit": UNIT, "e2e": {"value": ent / e2e_ms * 1e3, "ms_per_query": e2e_ms}, "Z": z,
            "note": "L2-resident at this size (the tables are MBs): a same-config ratio against the reference arm, not a roofline number"}


def multivalued_leg(ctx):
    """PR (-mf) on Munin1 (cardinalities up to 21): per-launch profile, the widest multi-valued step"""
    import torch
    from bnpp_b200 import model
    path = os.path.join(ROOT, "oracle", "_ref", "models", "bayesnets", "Munin1.uai")
    if not os.path.exists(path):
        return {"unavailable": "oracle/_ref/models not present"}
    _, bn = model.from_uai_text(ctx, open(path).read())
    z, _ = bn.partition({}, "mf")
    t0 = time.perf_counter()
    z, _ = bn.partition({}, "mf")
    replay_ms = (time.perf_counter() - t0) * 1e3
    order, width = bn.order(list(range(bn.nvars)), {}, "mf")
    plan = bn.plan([], order)
    res = torch.zeros(2, dtype=torch.float64, device="cuda")
    plan.set_profiling(True)
    acc = None
    for _ in range(3):
        plan.run(bn.table_ptrs, [], res.data_ptr(), res.data_ptr() + 8)
        st = plan.step_stats()
        acc = st if acc is None else [dict(a, ms=a["ms"] + b["ms"]) for a, b in zip(acc, st)]
    plan.set_profiling(False)
    peak, _ = peaks()
    top = sorted(acc, key=lambda s: -s["ms"])[:3]
    rows = [{"ms": s["ms"] / 3, "k": s["k"], "entries": s["entries"], "bytes": s["bytes"], "GBs": s["bytes"] / (s["ms"] / 3) / 1e6,
             "frac": s["bytes"] / (s["ms"] / 3) / 1e6 / peak, "entries_per_s": s["entries"] / (s["ms"] / 3) * 1e3, "kernel": s["kernel"]}
            for s in top]
    bn.close()
    return {"network": "Munin1.uai (189 variables, min-fill width %d)" % width, "Z": z, "query_ms_replay": replay_ms,
            "launches": len(acc), "sum_launch_ms": sum(s["ms"] for s in acc) / 3, "top_launches": rows,
            "note": "the widest step writes 3.9e7 entries from operands of 4.3e6 and 5.6e6 entries (both broadcast over most of "
                    "the output): 2.7e8 union entries for 0.39 GB of algorithmic traffic -- bound by shared-memory reads and "
                    "issue slots per union entry, not by HBM (DESIGN.md 4.1)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config5", action="store_true", help="skip the PR-queries/sec legs (config 5)")
    ap.add_argument("--no-extra", action="store_true", help="skip the N = 1 legs shapes / configs_1_3 / multivalued / same_sample")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling leg (width-30 network)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of each leg returned as DIR/<name>.npy (float64; at N > 1, rank "
                         "0's): the inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    D = Dist()
    sample = pick_cpu_sample(args.steps, args.warmup)

    if args.impl == "reference":
        if D.rank != 0:
            return 0
        cb, t_ms = cpu_reference_leg(sample, steps=max(1, args.steps), warmup=min(args.warmup, 1))
        line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
                "steps": cb["steps_run"], "warmup": min(args.warmup, 1), "ms_per_step": t_ms, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": "config 4 generator, bounded CPU sample: " + cb["sample"], "same_config": False,
                           "same_config_note": "the GPU arm's workload is the width-27 network (2.2e9 entries per query: ~50 min in "
                                               "the reference, tests/golden/wide.json); the GPU arm reports its own throughput on THIS "
                                               "sample under `same_sample`"},
                "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    import numpy as np
    import torch
    import torch.distributed as dist
    from bnpp_b200 import capi

    if D.world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", D.local))
    torch.cuda.set_device(D.local)
    ctx = capi.Context(D.local)
    D.init(ctx)
    n_gpus = D.world
    if n_gpus not in (1, 2, 4, 8):
        raise SystemExit("bench.py supports 1, 2, 4 or 8 GPUs")

    sampler = ClockSampler(D.local) if D.rank == 0 else None
    weak = wide_leg(ctx, D, n_gpus, args.steps, args.warmup, profile=True, e2e=True, sampler=sampler)
    clocks = sampler.summary() if sampler is not None else None

    strong = None
    if not args.no_strong:
        try:
            strong = wide_leg(ctx, D, "strong", args.steps, 2, profile=False, e2e=False)
            strong.pop("per_launch", None)
        except Exception as e:
            strong = {"error": "%s: %s" % (type(e).__name__, e)}

    config5 = None
    if not args.no_config5:
        config5 = {}
        for nsets in (65536, 1 << 20):
            try:
                config5[str(nsets)] = config5_leg(ctx, D, nsets, args.steps, args.warmup,
                                                  cpu_arm=not args.no_cpu_baseline and n_gpus == 1)
            except Exception as e:      # the headline line must not depend on an auxiliary leg
                config5[str(nsets)] = {"error": "%s: %s" % (type(e).__name__, e)}

    if D.rank != 0:
        if D.world > 1:
            dist.destroy_process_group()
        return 0

    outputs = {"wide_" + k: v for k, v in weak.pop("outputs").items()}
    outputs.update({"strong_" + k: v for k, v in (strong or {}).pop("outputs", {}).items()})
    for nsets, leg in (config5 or {}).items():
        outputs.update({"pr_queries_%s_%s" % (nsets, k): v for k, v in leg.pop("outputs", {}).items()})
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), np.asarray(arr, dtype=np.float64))

    # ---- roofline of the dominant kernel: the widest fused launch ---------------------------------
    peak, peak_kind = peaks()
    per_launch = weak.pop("per_launch")
    widest = max(range(len(per_launch)), key=lambda i: per_launch[i]["bytes"])
    wl = per_launch[widest]
    w_ms = wl["ms"]
    achieved = wl["bytes"] / w_ms / 1e6
    big = [s for s in per_launch if s["entries"] >= (1 << 24)]
    big_bytes = sum(s["bytes"] for s in big)
    big_ms = sum(s["ms"] for s in big)
    all_ms = sum(s["ms"] for s in per_launch)
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if n_gpus == 1 and os.path.exists(tp):
        tj = json.load(open(tp))      # dram__bytes_read.sum + dram__bytes_write.sum of this launch, one `ncu --set full` capture
        if tj.get("kernel_variant") and tj["kernel_variant"] in wl.get("kernel", "") and tj.get("algorithmic_bytes") == wl["bytes"]:
            traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
            traffic_src = "profiles/r2_traffic.json (one ncu --set full capture of the same launch, profiles/r2_canon_full.md: same kernel variant, same algorithmic bytes)"
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes": wl["bytes"], "peak_kind": peak_kind,
                "measured_in": "second timed pass of the same K steps with a CUDA event pair around every launch, each step "
                               "enqueued behind a gate so that it runs back to back on the device "
                               "(launch durations sum to %.3f ms per step vs %.3f ms in the graph-replayed pass `value` is taken from)"
                               % (weak["profiled_ms"], weak["ms_per_step"]),
                "kernel": "%s, widest launch: k=%d operands, %d union entries, %.3f GB algorithmic, %.3f ms"
                          % (wl.get("kernel", "contract"), wl["k"], wl["entries"], wl["bytes"] / 1e9, w_ms),
                "launches_ge_2p24_entries": {"n": len(big), "GBs": big_bytes / big_ms / 1e6 if big_ms else None,
                                             "frac": big_bytes / big_ms / 1e6 / peak if big_ms else None,
                                             "share_of_step_ms": big_ms / all_ms if all_ms else None},
                "whole_step": {"GBs": weak["bytes_per_step"] / weak["ms_per_step"] / 1e6,
                               "frac": weak["bytes_per_step"] / weak["ms_per_step"] / 1e6 / peak}}

    extra = {}
    if n_gpus == 1 and not args.no_extra:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        for name, fn in (("same_sample", lambda: same_sample_leg(ctx, sample, args.steps)),
                         ("multivalued", lambda: multivalued_leg(ctx)),
                         ("configs_1_3", lambda: dict(__import__("config_bench").run(ctx, reps=30), reps=30)),
                         ("shapes", lambda: shapes_leg(ctx, peak))):
            try:
                extra[name] = fn()
            except Exception as e:
                extra[name] = {"error": "%s: %s" % (type(e).__name__, e)}

    cb = None
    if not args.no_cpu_baseline and n_gpus == 1:
        cb, _ = cpu_reference_leg(sample, steps=1)

    N, W, K, seed = weak["network"]
    e2e = weak.pop("e2e")
    gold = weak["golden"]
    line = {"metric": METRIC, "value": weak["value"], "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": weak["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "config 4: synthetic random BN N=%d W=%d K=%d seed=%d, %d observed leaves, exact PR via VE (min-fill "
                                   "width %d%s); %d fused launches per query, %d union entries per rank, largest union table 2^%d entries"
                                   % (N, W, K, seed, len(weak["evidence"]), weak["width"],
                                      (", sharded on variables %s -> width %d per rank" % (weak["shard_vars"], weak["width_per_rank"]))
                                      if weak["shard_vars"] else "",
                                      weak["n_launches"], weak["entries_per_rank"], weak["max_step_entries"].bit_length() - 1),
                       "l2_flush": "inputs larger than L2: every step streams %.1f GB of tables through a 126 MB L2"
                                   % (weak["bytes_per_step"] / 1e9),
                       "partition": weak["Z"], "partition_e2e": e2e["Z"], "partition_reference": gold.get("Z_reference"),
                       "peak_intermediate_GB": weak["peak_intermediate_GB"]},
            "e2e": e2e, "gpu_launches": weak["gpu_launches"], "clocks": clocks, "roofline": roofline, "cpu_baseline": cb,
            "golden": gold, "weak": {k: weak[k] for k in ("entries_per_rank", "entries_all_ranks", "entries_unsharded",
                                                          "redundant_work", "useful_value", "Z_rank")},
            "strong": strong, "pr_queries": config5}
    line.update(extra)
    print(json.dumps(line))
    if D.world > 1:
        dist.destroy_process_group()
    bad = [g for g in (gold, (strong or {}).get("golden", {})) if g.get("available") and not g.get("ok")]
    if bad or (e2e["Z"] and gold.get("available") and abs(e2e["Z"] - gold["Z_reference"]) > 1e-9 * gold["Z_reference"]):
        print("bench.py: PARTITION DIFFERS FROM THE REFERENCE'S: %s" % bad, file=sys.stderr)
        return 1
    return 0


def shapes_leg(ctx, peak):
    """SURVEY 8d headline shapes (F-elem / F-bcast / F-small x sum-out position x B order, 2^28 union entries), the
    mixed-cardinality case and multi-valued elimination (cardinalities 3, 4, 5, 7, 8), each with its roofline fraction"""
    import shapes_bench as sb
    rows = sb.run_binary(ctx, 28, 3, verbose=False, peak=peak)
    rows += sb.run_mixed(ctx, 3, verbose=False, peak=peak)
    rows += sb.run_mv(ctx, [3, 4, 5, 7, 8], 3, verbose=False, peak=peak)
    return {"peak_GBs": peak, "iters_per_row": 3, "rows": rows, "min_frac": min(r["frac"] for r in rows),
            "rows_below_0.70": [dict(kind=r["kind"], k=r["k"], frac=r["frac"], kernel=r["kernel"]) for r in rows if r["frac"] < 0.70]}


if __name__ == "__main__":
    sys.exit(main())
