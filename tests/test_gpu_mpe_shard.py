"""Sharded MPE and marginal MAP on the GPU: the max-loc kernel (bnpp_mpe_shard_select) against the reference of
tests/shard_select.py bit for bit; virtual ranks on one GPU (each rank's query is the single `BN.mpe` / `BN.map` with its
shard values observed, the records are packed and selected on the device) against the unsharded query; the sharded run
(bnpp_mpe_plan_run_sharded) on a one-rank communicator against bnpp_mpe_plan_run bit for bit, graph replays included;
its argument checks; and, with two or more GPUs, `BN.mpe` / `BN.map(..., comm=)` over NCCL ranks."""
import ctypes
import gzip
import json
import math
import os
import sys

import numpy as np
import pytest

import oracle as orc
import shard_select
from bnpp_b200 import sharding, synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EINVAL = -1
RANDOM = [(30, 10, 3, 1), (30, 10, 3, 2), (40, 12, 3, 3)]


@pytest.fixture(scope="module")
def ctx():
    from bnpp_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


class _Rank:
    """what BN.shard / BN.map_shard read of a communicator"""

    def __init__(self, rank, world):
        self.rank, self.world = rank, world


def _lib(ctx):
    L = ctx.L
    L.bnpp_mpe_shard_select.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p,
                                        ctypes.c_void_p]
    return L


def _select_dev(ctx, records, nranks, nvars):
    """-> (value as uint64 bits, assignment uint32 array, kernel name) of bnpp_mpe_shard_select on the device"""
    import torch
    L = _lib(ctx)
    with torch.cuda.stream(ctx.torch_stream):
        rec = torch.from_numpy(np.ascontiguousarray(records, dtype=np.uint32).view(np.int32)).to("cuda", non_blocking=False)
        out = torch.full((2 + nvars,), -1, dtype=torch.int32, device="cuda")
    ctx.check(L.bnpp_mpe_shard_select(ctx.h, nranks, nvars, rec.data_ptr(), out.data_ptr(), out.data_ptr() + 8))
    name = ctx.last_launch()[0]
    ctx.sync()
    host = out.cpu().numpy()
    return int(host[:2].view(np.uint64)[0]), host[2:].view(np.uint32).copy(), name


def _values(rng, nranks, kind):
    if kind == "random":
        return rng.uniform(0.0, 1.0, nranks)
    if kind == "ties":                          # few distinct values: the maximum repeats
        return rng.choice([0.0, 0.125, 0.25, 0.5], nranks)
    if kind == "nan":
        v = rng.choice([0.25, 0.5, np.nan], nranks)
        return v
    if kind == "nan_first":
        v = rng.uniform(0.0, 1.0, nranks)
        v[0] = np.nan
        return v
    if kind == "nan_last":
        v = rng.uniform(0.0, 1.0, nranks)
        v[-1] = np.nan
        return v
    if kind == "all_nan":
        return np.full(nranks, np.nan)
    return np.zeros(nranks)                     # "zero"


@pytest.mark.parametrize("nranks", [1, 2, 3, 8, 64, 1024])
@pytest.mark.parametrize("nvars", [1, 2, 7, 1041])
def test_select_kernel_against_reference(ctx, nranks, nvars):
    rng = np.random.default_rng(nranks * 7919 + nvars)
    for kind in ("random", "ties", "nan", "nan_first", "nan_last", "all_nan", "zero"):
        values = _values(rng, nranks, kind)
        assign = rng.integers(0, 2 ** 32, (nranks, nvars), dtype=np.uint64).astype(np.uint32)
        rec = shard_select.pack(values, assign)
        win, value, want_a = shard_select.select(rec, nranks, nvars)
        bits, got_a, name = _select_dev(ctx, rec, nranks, nvars)
        what = (nranks, nvars, kind, win)
        assert name == "mpe_shard_select", name
        assert bits == int(np.float64(value).view(np.uint64)), what
        assert np.array_equal(got_a, want_a), what


def test_select_kernel_errors(ctx):
    import torch
    L = _lib(ctx)
    with torch.cuda.stream(ctx.torch_stream):
        buf = torch.zeros(16, dtype=torch.int32, device="cuda")
    p = buf.data_ptr()
    assert L.bnpp_mpe_shard_select(ctx.h, 0, 2, p, p, p + 8) == EINVAL
    assert L.bnpp_mpe_shard_select(ctx.h, 2, 0, p, p, p + 8) == EINVAL
    assert L.bnpp_mpe_shard_select(ctx.h, 2, 2, None, p, p + 8) == EINVAL
    assert L.bnpp_mpe_shard_select(ctx.h, 2, 2, p, None, p + 8) == EINVAL
    assert L.bnpp_mpe_shard_select(ctx.h, 2, 2, p, p, None) == EINVAL
    assert L.bnpp_mpe_shard_select(None, 2, 2, p, p, p + 8) == EINVAL
    ctx.sync()


# --- virtual ranks on one GPU -------------------------------------------------------------------------------------------

def _networks():
    with gzip.open(os.path.join(ROOT, "tests", "golden", "models.json.gz"), "rt") as f:
        g = json.load(f)
    out = []
    for name, m in g.items():
        ev = next(({int(k): v for k, v in c["evidence"].items()} for c in m["pr"] if c["evidence"] and c["flag"] == "mf"), {})
        out.append((name, m["uai"], ev))
    for n, w, k, seed in RANDOM:
        out.append(("random_bn_%d_%d" % (n, seed), synth.random_bn_uai(n, w, k, seed), {n - 1: 1, n - 3: 0}))
    return out


def _cpt_product(om, assignment):
    p = 1.0
    for f in om.factors:
        idx = int(np.ravel_multi_index([assignment[v] for v in f.scope], [int(om.card[v]) for v in f.scope])) if f.scope else 0
        p *= float(f.values[idx])
    return p


def _map_vars(bn, ev):
    free = [v for v in range(bn.nvars) if v not in ev]
    return free[len(free) // 3:]


def test_virtual_ranks_mpe(ctx):
    from bnpp_b200 import model
    n_cases = n_skip = 0
    for name, text, ev in _networks():
        bn = model.from_uai_text(ctx, text)[1]
        om = orc.parse_uai(text)
        one_v, one_a, _ = bn.mpe(ev, "mf")
        for world in (2, 4, 8):
            try:
                _, shard = bn.shard(ev, "mf", _Rank(0, world))
            except ValueError:
                n_skip += 1
                continue
            vals, assigns = [], []
            for r in range(world):
                v, a, _ = bn.mpe({**ev, **sharding.shard_evidence(shard, r)}, "mf")
                vals.append(v)
                assigns.append(a)
            win, want_v, want_a = shard_select.select(shard_select.pack(vals, assigns), world, bn.nvars)
            bits, got_a, _ = _select_dev(ctx, shard_select.pack(vals, assigns), world, bn.nvars)
            value = float(np.uint64(bits).view(np.float64))
            got_a = [int(x) for x in got_a]
            what = (name, world, shard, win)
            assert bits == int(np.float64(want_v).view(np.uint64)) and got_a == [int(x) for x in want_a], what
            assert math.isclose(value, one_v, rel_tol=1e-12), (what, value, one_v)
            assert math.isclose(_cpt_product(om, got_a), value, rel_tol=1e-12), what
            assert all(got_a[v] == x for v, x in ev.items()), what
            # the same assignment as one GPU unless the two are (near-)tied maxima
            assert got_a == one_a or math.isclose(_cpt_product(om, one_a), _cpt_product(om, got_a), rel_tol=1e-9), what
            n_cases += 1
        bn.close()
    assert n_cases >= 20, (n_cases, n_skip)


def test_virtual_ranks_map(ctx):
    from bnpp_b200 import model
    n_cases = n_skip = 0
    for name, text, ev in _networks():
        bn = model.from_uai_text(ctx, text)[1]
        m = _map_vars(bn, ev)
        summed = [v for v in range(bn.nvars) if v not in ev and v not in m]
        if model.elim_order_constrained(bn.cards, bn.scopes, summed, m, "mf", observed=sorted(ev))[1] > 20:
            bn.close()                          # the constrained order of this MAP set is too wide for a test
            continue
        one_v, one_x, _ = bn.map(m, ev, "mf")
        for world in (2, 4, 8):
            try:
                _, shard = bn.map_shard(m, ev, "mf", _Rank(0, world))
            except ValueError:
                n_skip += 1
                continue
            assert set(shard) <= set(m)
            rest = [v for v in m if v not in shard]
            vals, assigns = [], []
            for r in range(world):
                ev_r = {**ev, **sharding.shard_evidence(shard, r)}
                v, x, _ = bn.map(rest, ev_r, "mf")
                a = [ev_r.get(u, x.get(u, 0xFFFFFFFF)) for u in range(bn.nvars)]
                vals.append(v)
                assigns.append(a)
            bits, got_a, _ = _select_dev(ctx, shard_select.pack(vals, assigns), world, bn.nvars)
            value = float(np.uint64(bits).view(np.float64))
            got_x = {v: int(got_a[v]) for v in m}
            what = (name, world, shard)
            assert math.isclose(value, one_v, rel_tol=1e-12), (what, value, one_v)
            if got_x != one_x:                  # only between (near-)tied maxima: P(x_M, e) of both
                p_one, _ = bn.partition({**ev, **one_x}, "mf")
                p_got, _ = bn.partition({**ev, **got_x}, "mf")
                assert math.isclose(p_one, p_got, rel_tol=1e-9), what
            n_cases += 1
        bn.close()
    assert n_cases >= 10, (n_cases, n_skip)


# --- the sharded run on one rank ----------------------------------------------------------------------------------------

def _plans(ctx, bn, ev):
    from bnpp_b200 import model
    observed = sorted(ev)
    free = [v for v in range(bn.nvars) if v not in ev]
    order, _ = bn.order(free, ev, "mf")
    m = _map_vars(bn, ev)
    summed = [v for v in free if v not in m]
    map_order, _ = model.elim_order_constrained(bn.cards, bn.scopes, summed, m, "mf", observed=observed)
    return [lambda: model.MPEPlan(ctx, bn.cards, bn.scopes, observed, order),
            lambda: model.MAPPlan(ctx, bn.cards, bn.scopes, observed, map_order, map_vars=m)]


def test_one_rank_sharded_run_equals_plan_run(ctx):
    import torch
    from bnpp_b200 import model
    from bnpp_b200.nccl import ShardComm
    comm = ShardComm(ctx, 0, 1)
    n, w, k, seed = RANDOM[2]
    ev = {n - 1: 1, n - 3: 0}
    bn = model.from_uai_text(ctx, synth.random_bn_uai(n, w, k, seed))[1]
    observed = sorted(ev)
    for make in _plans(ctx, bn, ev):
        direct, sharded = make(), make()
        for run in range(3):                    # the second and third runs replay the plan's graph
            with torch.cuda.stream(ctx.torch_stream):
                a = torch.full((2 + bn.nvars,), -7, dtype=torch.int32, device="cuda")
                b = torch.full((2 + bn.nvars,), -7, dtype=torch.int32, device="cuda")
            direct.run_mpe(bn.table_ptrs, [ev[v] for v in observed], a.data_ptr(), a.data_ptr() + 8)
            comm.run_mpe_sharded(sharded, bn.table_ptrs, [ev[v] for v in observed], b.data_ptr(), b.data_ptr() + 8)
            assert ctx.last_launch()[0] == "mpe_shard_select"
            ctx.sync()
            assert torch.equal(a.cpu(), b.cpu()), (type(direct).__name__, run)
        direct.close()
        sharded.close()
    bn.close()
    comm.close()


def test_sharded_run_errors(ctx):
    import torch
    from bnpp_b200 import model
    from bnpp_b200.nccl import ShardComm
    comm = ShardComm(ctx, 0, 1)
    n, w, k, seed = RANDOM[0]
    ev = {n - 1: 1}
    bn = model.from_uai_text(ctx, synth.random_bn_uai(n, w, k, seed))[1]
    observed = sorted(ev)
    free = [v for v in range(bn.nvars) if v not in ev]
    order, _ = bn.order(free, ev, "mf")
    pr = model.VEPlan(ctx, bn.cards, bn.scopes, observed, order)
    mar = model.MarPlan(ctx, bn.cards, bn.scopes, observed, order)
    mpe = model.MPEPlan(ctx, bn.cards, bn.scopes, observed, order)
    L = comm.lib
    L.bnpp_mpe_plan_run_sharded.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p),
                                            ctypes.POINTER(ctypes.c_uint32), ctypes.c_void_p, ctypes.c_void_p]
    with torch.cuda.stream(ctx.torch_stream):
        buf = torch.zeros(2 + bn.nvars, dtype=torch.int32, device="cuda")
    tp = (ctypes.c_void_p * len(bn.table_ptrs))(*bn.table_ptrs)
    ov = (ctypes.c_uint32 * 1)(ev[n - 1])
    v, a = buf.data_ptr(), buf.data_ptr() + 8
    assert L.bnpp_mpe_plan_run_sharded(ctx.h, pr.h, comm.comm, tp, ov, v, a) == EINVAL
    assert L.bnpp_mpe_plan_run_sharded(ctx.h, mar.h, comm.comm, tp, ov, v, a) == EINVAL
    assert L.bnpp_mpe_plan_run_sharded(ctx.h, mpe.h, comm.comm, tp, ov, None, a) == EINVAL
    assert L.bnpp_mpe_plan_run_sharded(ctx.h, mpe.h, comm.comm, tp, ov, v, None) == EINVAL
    assert L.bnpp_mpe_plan_run_sharded(ctx.h, None, comm.comm, tp, ov, v, a) == EINVAL
    assert L.bnpp_mpe_plan_run_sharded(ctx.h, mpe.h, None, tp, ov, v, a) == EINVAL
    assert L.bnpp_mpe_plan_run_sharded(ctx.h, mpe.h, comm.comm, tp, ov, v, a) == 0
    ctx.sync()
    for p in (pr, mar, mpe):
        p.close()
    bn.close()
    comm.close()


# --- NCCL ranks (two or more GPUs) --------------------------------------------------------------------------------------

def _nccl_worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)      # carries the NCCL unique id only
    torch.cuda.set_device(rank)
    from bnpp_b200 import capi, model
    from bnpp_b200.nccl import ShardComm
    ctx = capi.Context(rank)
    comm = ShardComm(ctx, rank, world)
    out = []
    for n, w, k, seed in RANDOM:
        ev = {n - 1: 1, n - 3: 0}
        bn = model.from_uai_text(ctx, synth.random_bn_uai(n, w, k, seed))[1]
        v_sh, a_sh, _ = bn.mpe(ev, "mf", comm=comm)
        v_1, a_1, _ = bn.mpe(ev, "mf")
        m = [v for v in range(n) if v not in ev][(n - 2) // 3:]
        mv_sh, mx_sh, _ = bn.map(m, ev, "mf", comm=comm)
        mv_1, mx_1, _ = bn.map(m, ev, "mf")
        out.append((seed, v_sh, a_sh, v_1, a_1, mv_sh, mx_sh, mv_1, mx_1))
        bn.close()
    q.put((rank, out))
    comm.close()
    ctx.close()
    dist.destroy_process_group()


def _device_count():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("world", [2, 4])
def test_nccl_ranks(world):
    if _device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    import torch.multiprocessing as mp
    mpc = mp.get_context("spawn")
    q = mpc.Queue()
    port = 29800 + world + (os.getpid() % 100)
    procs = [mpc.Process(target=_nccl_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = {}
    for _ in range(world):
        r, out = q.get(timeout=600)
        results[r] = out
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for r in range(1, world):
        assert results[r] == results[0], r          # every rank returns the same answer
    for seed, v_sh, a_sh, v_1, a_1, mv_sh, mx_sh, mv_1, mx_1 in results[0]:
        assert math.isclose(v_sh, v_1, rel_tol=1e-12), (seed, v_sh, v_1)
        assert a_sh == a_1, seed
        assert math.isclose(mv_sh, mv_1, rel_tol=1e-12), (seed, mv_sh, mv_1)
        assert mx_sh == mx_1, seed
