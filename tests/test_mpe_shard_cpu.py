"""Sharded MPE and marginal MAP without a GPU: the max-loc rule over the ranks' records (tests/shard_select.py) on
crafted records; `gloo` ranks at world 2 and 4 that each emulate their dry MPE / MAP plan (tests/mpe_emulator.py,
tests/map_emulator.py) with the shard variables observed at their values, gather the records and select -- against
enumeration of the whole network; and the choice of shard variables for a maximising query
(sharding.pick_max_shard_vars) against the MPE / PR choice."""
import math
import os
import sys

import numpy as np
import pytest
import torch.multiprocessing as mp

import oracle as orc
import shard_select
from bnpp_b200 import model, sharding
from fused_interp import parse_uai
from map_emulator import ASSIGN_SUMMED
from mpe_oracle import max_last_axis

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAN = float("nan")


def _records(values, nvars, seed=0):
    rng = np.random.default_rng(seed)
    return shard_select.pack(values, rng.integers(0, 2 ** 32, (len(values), nvars), dtype=np.uint64).astype(np.uint32))


@pytest.mark.parametrize("nvars", [1, 2, 7, 8])
def test_select_rule(nvars):
    cases = [
        ([0.1, 0.5, 0.3], 1),                 # unique max
        ([0.5, 0.2, 0.5, 0.5], 0),            # ties: the lowest rank
        ([0.1, 0.4, 0.2, 0.4], 1),
        ([NAN, 0.3, 0.9], 0),                 # NaN first: rank 0 is kept (nothing is strictly greater than a NaN)
        ([0.3, 0.9, NAN], 1),                 # NaN last: never replaces a number
        ([0.3, NAN, 0.2, 0.7], 3),
        ([NAN, NAN, NAN], 0),                 # all NaN
        ([0.0, 0.0, 0.0, 0.0], 0),            # all zero (impossible evidence on every rank)
        ([0.0, -0.0, 0.0], 0),
        ([0.25], 0),
    ]
    for values, want in cases:
        rec = _records(values, nvars)
        assert rec.size == len(values) * shard_select.stride(nvars)
        win, value, assignment = shard_select.select(rec, len(values), nvars)
        assert win == want, (values, win)
        assert np.float64(value).view(np.uint64) == np.float64(values[want]).view(np.uint64)
        assert np.array_equal(assignment, rec.reshape(len(values), -1)[want, 2:2 + nvars])
        # the rule is the one of the max kernels over an axis
        assert int(max_last_axis(np.asarray(values, dtype=np.float64).reshape(1, -1))[1][0]) == want


def test_record_stride_is_even():
    for nvars in range(1, 12):
        s = shard_select.stride(nvars)
        assert s % 2 == 0 and 2 + nvars <= s <= 3 + nvars
    rec = _records([0.5, 0.75, 0.25], 3)            # odd nvars: the values stay at even words (8-byte aligned)
    assert [rec[r * 6:r * 6 + 2].view(np.float64)[0] for r in range(3)] == [0.5, 0.75, 0.25]


# --- shard variables of a maximising query -----------------------------------------------------------------------------

def test_pick_max_shard_vars_rules():
    scopes = [[0, 1, 2], [2, 3], [3, 4]]
    order = [0, 1, 2, 3, 4]
    cards = [2] * 5
    assert sharding.widest_clique(scopes, order) == [0, 1, 2]
    assert sharding.pick_max_shard_vars(scopes, order, 2, cards, [0, 1, 2, 3, 4]) == [1, 2]
    assert sharding.pick_max_shard_vars(scopes, order, 2, cards, [0, 2, 4]) == [0, 2]     # MAP variables only
    assert sharding.pick_max_shard_vars(scopes, order, 1, cards, [1, 3]) == [1]
    with pytest.raises(ValueError, match="no 2 binary MAP shard variables"):
        sharding.pick_max_shard_vars(scopes, order, 2, cards, [3, 4])             # MAP set outside the widest clique
    with pytest.raises(ValueError):
        sharding.pick_max_shard_vars(scopes, order, 2, cards, [1, 3, 4])          # only one of them in it
    with pytest.raises(ValueError):
        sharding.pick_max_shard_vars(scopes, order, 1, [2, 2, 3, 2, 2], [0, 1, 2])  # the candidate has 3 values
    assert sharding.pick_max_shard_vars(scopes, order, 0, cards, []) == []


def test_pick_max_shard_vars_equals_mpe_choice(golden_models):
    n_same = n_raise = 0
    for name, m in golden_models.items():
        cards, scopes, _ = parse_uai(m["uai"])
        for case in m["pr"]:
            if case["flag"] != "mf":
                continue
            ev = {int(k): v for k, v in case["evidence"].items()}
            free = [v for v in range(len(cards)) if v not in ev]
            order, _ = model.elim_order(cards, scopes, free, "mf", observed=sorted(ev))
            live = [[v for v in sc if v not in ev] for sc in scopes]
            for g in (1, 2, 3):
                want = sharding.pick_shard_vars(live, order, g)
                if len(want) == g and all(cards[v] == 2 for v in want):
                    assert sharding.pick_max_shard_vars(live, order, g, cards, free) == want, (name, g)
                    n_same += 1
                else:
                    with pytest.raises(ValueError):
                        sharding.pick_max_shard_vars(live, order, g, cards, free)
                    n_raise += 1
    assert n_same >= 20 and n_raise >= 1, (n_same, n_raise)


# --- gloo ranks: every rank emulates its slab, the records are gathered and the best one selected -----------------------

N, W, K = 16, 8, 3


def _network(seed):
    from bnpp_b200 import synth
    text = synth.random_bn_uai(N, W, K, seed)
    cards, scopes, tables = parse_uai(text)
    return text, cards, scopes, [np.asarray(t, dtype=np.float64) for t in tables]


def _map_vars(cards, ev):
    free = [v for v in range(len(cards)) if v not in ev]
    return free[len(free) // 3:]            # the later two thirds: they fill the widest clique of the constrained order


def _gather_select(dist, torch, value, assignment, world):
    rec = torch.from_numpy(shard_select.pack([value], [assignment]).view(np.int32).copy())
    parts = [torch.empty_like(rec) for _ in range(world)]
    dist.all_gather(parts, rec)
    records = np.concatenate([p.numpy() for p in parts]).view(np.uint32)
    return shard_select.select(records, world, len(assignment))


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import map_emulator
    import mpe_emulator
    g = world.bit_length() - 1
    out = []
    for seed in (3, 4, 7):
        text, cards, scopes, tables = _network(seed)
        ev = {N - 1: seed % 2}
        free = [v for v in range(N) if v not in ev]
        live = [[v for v in sc if v not in ev] for sc in scopes]
        # MPE: the shard variables of `BN.shard` (every unobserved variable is maximised)
        order, _ = model.elim_order(cards, scopes, free, "mf", observed=sorted(ev))
        shard = sharding.pick_max_shard_vars(live, order, g, cards, free)
        assert shard == sharding.pick_shard_vars(live, order, g)
        ev_r = {**ev, **sharding.shard_evidence(shard, rank)}
        obs_r = sorted(ev_r)
        order_r, _ = model.elim_order(cards, scopes, [v for v in range(N) if v not in ev_r], "mf", observed=obs_r)
        p = mpe_emulator.DryMPEPlan(cards, scopes, obs_r, order_r)
        assert p.rc == 0
        value, assignment = mpe_emulator.emulate(p.h, tables, obs_r, [ev_r[v] for v in obs_r], N)
        p.close()
        win, v_sel, a_sel = _gather_select(dist, torch, value, assignment, world)
        out.append(("mpe", seed, ev, shard, win, float(v_sel), [int(x) for x in a_sel]))
        # MAP: shard variables among the MAP variables of the widest clique of the constrained order
        m = _map_vars(cards, ev)
        summed = [v for v in free if v not in m]
        order, _ = model.elim_order_constrained(cards, scopes, summed, m, "mf", observed=sorted(ev))
        shard = sharding.pick_max_shard_vars(live, order, g, cards, m)
        ev_r = {**ev, **sharding.shard_evidence(shard, rank)}
        obs_r = sorted(ev_r)
        m_r = [v for v in m if v not in shard]
        order_r, _ = model.elim_order_constrained(cards, scopes, summed, m_r, "mf", observed=obs_r)
        p = map_emulator.DryMAPPlan(cards, scopes, obs_r, m_r, order_r)
        assert p.rc == 0
        value, assignment = map_emulator.emulate(p.h, tables, obs_r, [ev_r[v] for v in obs_r], N, m_r)
        p.close()
        win, v_sel, a_sel = _gather_select(dist, torch, value, assignment, world)
        out.append(("map", seed, ev, shard, win, float(v_sel), [int(x) for x in a_sel]))
    if rank == 0:
        q.put(out)
    dist.destroy_process_group()


def _cpt_product(om, assignment):
    p = 1.0
    for f in om.factors:
        idx = int(np.ravel_multi_index([assignment[v] for v in f.scope], [int(om.card[v]) for v in f.scope])) if f.scope else 0
        p *= float(f.values[idx])
    return p


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_mpe_map_gloo(world):
    import map_oracle
    import mpe_oracle
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29700 + world + (os.getpid() % 200)
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=300)
        assert p.exitcode == 0
    out = q.get(timeout=10)
    assert len(out) == 6
    for kind, seed, ev, shard, win, value, assignment in out:
        text, cards, scopes, tables = _network(seed)
        ev = {int(k): v for k, v in ev.items()}
        what = (kind, seed, world, shard, win)
        assert len(shard) == world.bit_length() - 1, what
        assert all(assignment[v] == x for v, x in ev.items()), what
        assert sharding.shard_evidence(shard, win) == {v: assignment[v] for v in shard}, what
        if kind == "mpe":
            om = orc.parse_uai(text)
            want, want_a, second = mpe_oracle.mpe_brute_force(om, ev)
            assert math.isclose(value, want, rel_tol=1e-12), what
            assert math.isclose(_cpt_product(om, assignment), value, rel_tol=1e-12), what
            if want - second > 1e-9 * want:
                assert assignment == want_a, what
        else:
            m = _map_vars(cards, ev)
            assert set(shard) <= set(m), what
            want, want_a, second = map_oracle.map_brute_force(cards, scopes, tables, ev, m)
            assert math.isclose(value, want, rel_tol=1e-12), what
            if want - second > 1e-9 * want:
                assert {v: assignment[v] for v in m} == want_a, what
            assert all(assignment[v] == ASSIGN_SUMMED for v in range(N) if v not in m and v not in ev), what
