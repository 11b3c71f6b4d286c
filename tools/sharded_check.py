#!/usr/bin/env python
"""Multi-GPU check of the sharded public API (run under torchrun, one rank per GPU): BN.partition(..., comm=),
BN.marginals_fast(..., comm=), BN.mpe(..., comm=) and BN.map(..., comm=) on a network sharded over the ranks against the
same queries on one GPU (every rank runs the unsharded query too), and against the reference's golden PR where one
exists.  The MAP set is the later two thirds of the unobserved variables; a set whose widest clique holds too few MAP
variables to shard on is reported and skipped.
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 tools/sharded_check.py"""
import gzip
import json
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from bnpp_b200 import capi, model, synth  # noqa: E402
from bnpp_b200.nccl import ShardComm  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
torch.cuda.set_device(local)
ctx = capi.Context(local)
comm = ShardComm(ctx, rank, world)
G = json.load(gzip.open(os.path.join(ROOT, "tests", "golden", "synthetic.json.gz"), "rt"))
ok = True
for rec in G["bn"]:
    if rec["N"] > 48:
        continue
    ev = {int(k): v for k, v in rec["evidence"].items()}
    bn = model.from_uai_text(ctx, synth.random_bn_uai(rec["N"], rec["W"], rec["K"], rec["seed"]))[1]
    z_sh, _ = bn.partition(ev, "mf", comm=comm)
    z_1, _ = bn.partition(ev, "mf")
    want = [c for c in rec["cases"] if c["flag"] == "mf"][0].get("pr")
    good = math.isclose(z_sh, z_1, rel_tol=1e-12) and (want is None or math.isclose(z_sh, want, rel_tol=1e-9))
    mar_sh = bn.marginals_fast(ev, "mf", comm=comm)
    mar_1 = bn.marginals_fast(ev, "mf")
    worst = max(float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))) for a, b in zip(mar_sh, mar_1))
    good = good and worst <= 1e-9
    v_sh, a_sh, _ = bn.mpe(ev, "mf", comm=comm)
    v_1, a_1, _ = bn.mpe(ev, "mf")
    good_mpe = math.isclose(v_sh, v_1, rel_tol=1e-12) and a_sh == a_1
    free = [v for v in range(bn.nvars) if v not in ev]
    m = free[len(free) // 3:]
    try:
        mv_sh, mx_sh, _ = bn.map(m, ev, "mf", comm=comm)
        mv_1, mx_1, _ = bn.map(m, ev, "mf")
        good_map = math.isclose(mv_sh, mv_1, rel_tol=1e-12) and mx_sh == mx_1
        map_line = "MAP sharded %.17g  one GPU %.17g" % (mv_sh, mv_1)
    except ValueError as e:             # the same on every rank: the choice is host work on the same inputs
        good_map, map_line = True, "MAP not sharded (%s)" % e
    ok = ok and good and good_mpe and good_map
    if rank == 0:
        print("N=%d world=%d  PR sharded %.17g  one GPU %.17g  reference %s  marginals max rel diff %.2e  %s"
              % (rec["N"], world, z_sh, z_1, want, worst, "ok" if good else "MISMATCH"), flush=True)
        print("      MPE sharded %.17g  one GPU %.17g  assignment %s  %s  %s"
              % (v_sh, v_1, "same" if a_sh == a_1 else "DIFFERENT", map_line,
                 "ok" if good_mpe and good_map else "MISMATCH"), flush=True)
    bn.close()
flag = torch.tensor([0 if ok else 1], device="cuda")
dist.all_reduce(flag)
comm.close()
dist.destroy_process_group()
sys.exit(1 if flag.item() else 0)
