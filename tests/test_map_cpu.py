"""Marginal MAP without a GPU: the constrained elimination order (bnpp_elim_order_constrained) against the plain
order, the reference-container path and the width of the order; dry MAP plans (bnpp_map_plan_create) emulated in mixed
mode against enumeration of max_{x_M} sum_{x_S}, against the PR emulation (M empty) and the MPE emulation (M = every
unobserved variable); the batched step program of MAP plans (kFusedMax exactly on the max steps, R_s the prefix sum of
n_out over them) interpreted on the CPU; and the creation errors."""
import math
import random

import numpy as np
import pytest

import batch_networks as bnet
import map_emulator as me
import map_oracle
import mpe_emulator
import mpe_fused_interp as mfi
from bnpp_b200 import model
from fused_interp import DryPlan, parse_uai
from plan_emulator import describe, run as pr_run

SMALL = ["asia", "asia_positive", "cancer", "earthquake", "grid3x3"]
RANDOM = ["random_%d" % s for s in range(bnet.N_RANDOM)]
HEURISTICS = ["mf", "wmf", "md"]
NB = 5
OK, EINVAL = 0, -1          # BNPP_OK, BNPP_EINVAL


def _network(name, golden_models):
    """-> (cards, scopes, tables, observed)"""
    if name in golden_models:
        cards, scopes, tables = parse_uai(golden_models[name]["uai"])
        obs = sorted(int(v) for v in next((c["evidence"] for c in golden_models[name]["pr"] if c["evidence"]), {}))
        if not obs:
            obs = sorted(random.Random(name).sample(range(len(cards)), max(1, len(cards) // 5)))
        return cards, scopes, tables, obs
    return bnet.mixed_bn(int(name.split("_")[1]))


def _map_sets(name, cards, observed):
    """seeded MAP sets of 1, 2 and about a third of the unobserved variables"""
    free = [v for v in range(len(cards)) if v not in set(observed)]
    rng = random.Random("map-" + name)
    sizes = sorted({min(len(free), k) for k in (1, 2, max(1, len(free) // 3))})
    return [sorted(rng.sample(free, k)) for k in sizes]


def _order(cards, scopes, observed, m, heuristic):
    summed = [v for v in range(len(cards)) if v not in set(observed) and v not in set(m)]
    if heuristic is None:
        return summed + list(m)
    return model.elim_order_constrained(cards, scopes, summed, m, heuristic, observed=observed)[0]


def _bits(x):
    return np.float64(x).view(np.uint64)


@pytest.mark.parametrize("heuristic", HEURISTICS)
def test_constrained_order(golden_models, heuristic):
    for name in golden_models:
        cards, scopes, _, ev_obs = _network(name, golden_models)
        for observed in ([], ev_obs):
            for m in _map_sets(name, cards, observed):
                summed = [v for v in range(len(cards)) if v not in set(observed) and v not in set(m)]
                order, width = model.elim_order_constrained(cards, scopes, summed, m, heuristic, observed=observed)
                ref, ref_w = model.elim_order_constrained(cards, scopes, summed, m, heuristic, observed=observed,
                                                          reference_containers=True)
                first, _ = model.elim_order(cards, scopes, summed, heuristic, observed=observed)
                what = (name, heuristic, observed, m)
                assert order[:len(summed)] == first, what
                assert order == ref and width == ref_w, what
                assert sorted(order[:len(summed)]) == sorted(summed) and sorted(order[len(summed):]) == m, what
                live = [[v for v in sc if v not in set(observed)] for sc in scopes]
                assert width == model.order_width(cards, live, order), what


def _cases():
    return [(n, k) for n in SMALL + RANDOM for k in range(3)]


def _case(golden_models, name, k):
    cards, scopes, tables, observed = _network(name, golden_models)
    sets = _map_sets(name, cards, observed)
    m = sets[k % len(sets)]
    heuristic = [None, "mf", "wmf"][k]
    return cards, scopes, [np.asarray(t, dtype=np.float64) for t in tables], observed, m, _order(cards, scopes, observed, m, heuristic)


@pytest.mark.parametrize("name,k", _cases())
def test_dry_map_plans_against_enumeration(golden_models, name, k):
    cards, scopes, tables, observed, m, order = _case(golden_models, name, k)
    p = me.DryMAPPlan(cards, scopes, observed, m, order)
    assert p.rc == 0, p.rc
    try:
        ev = bnet.evidence_sets([cards[v] for v in observed], NB, seed=k + len(name))
        for e in ev:
            e = [int(x) for x in e]
            value, assignment = me.emulate(p.h, tables, observed, e, len(cards), m)
            best, best_a, second = map_oracle.map_brute_force(cards, scopes, tables, dict(zip(observed, e)), m)
            assert math.isclose(value, best, rel_tol=1e-12, abs_tol=0.0), (name, m, value, best)
            if best > 0 and best - second > 1e-9 * best:
                assert {v: assignment[v] for v in m} == best_a, (name, m, e)
            for v in range(len(cards)):
                if v in dict(zip(observed, e)):
                    assert assignment[v] == dict(zip(observed, e))[v]
                elif v not in m:
                    assert assignment[v] == me.ASSIGN_SUMMED
    finally:
        p.close()


@pytest.mark.parametrize("name", SMALL + RANDOM[:8] + ["alarm", "hepar2"])
def test_empty_and_full_map_sets_are_pr_and_mpe(golden_models, name):
    cards, scopes, tables, observed = _network(name, golden_models)
    tables = [np.asarray(t, dtype=np.float64) for t in tables]
    free = [v for v in range(len(cards)) if v not in set(observed)]
    order = bnet.mf_order(cards, scopes, observed)
    ev = [int(x) for x in bnet.evidence_sets([cards[v] for v in observed], 2, seed=3)[1]]
    # M empty: the PR emulation of the same order, every unobserved variable summed
    p, pr = me.DryMAPPlan(cards, scopes, observed, [], order), DryPlan(cards, scopes, observed, order)
    try:
        assert p.rc == 0
        d = describe(pr.h)
        assert describe(p.h) == d
        value, assignment = me.emulate(p.h, tables, observed, ev, len(cards), [])
        result, _ = pr_run(d, tables, ev)
        want = float(result[0]) if any(st["out"] < 0 for st in d["steps"]) else 1.0
        assert _bits(value) == _bits(want), (name, value, want)
        assert all(assignment[v] == me.ASSIGN_SUMMED for v in free)
    finally:
        p.close()
        pr.close()
    # M = every unobserved variable: the MPE plan and its emulation
    p, mp = me.DryMAPPlan(cards, scopes, observed, free, order), mpe_emulator.DryMPEPlan(cards, scopes, observed, order)
    try:
        assert p.rc == 0 and mp.rc == 0
        assert describe(p.h) == describe(mp.h)
        got = me.emulate(p.h, tables, observed, ev, len(cards), free)
        want = mpe_emulator.emulate(mp.h, tables, observed, ev, len(cards))
        assert _bits(got[0]) == _bits(want[0]) and got[1] == want[1], name
        assert mfi.program(p.h, NB)[0].tolist() == mfi.program(mp.h, NB)[0].tolist()
    finally:
        p.close()
        mp.close()


@pytest.mark.parametrize("name,k", _cases())
def test_mixed_program_layout_and_interpreter(golden_models, name, k):
    cards, scopes, tables, observed, m, order = _case(golden_models, name, k)
    p = me.DryMAPPlan(cards, scopes, observed, m, order)
    assert p.rc == 0
    try:
        desc = describe(p.h)
        g, arena, n_steps = mfi.fused_info(p.h, NB)
        prog, tab = mfi.program(p.h, NB)
        assert g > 0 and prog.size > 0, name
        rows = me.rows(desc, set(m))
        heads = mfi.headers(prog, n_steps)
        # kFusedMax exactly on the max steps, each with its own R_s: the prefix sum of n_out over the max steps
        assert sorted((row, n_out) for n_out, cx, kk, flags, row in heads if flags & mfi.MAX) == sorted((r, n) for _, r, n in rows)
        assert all(row == 0 for n_out, cx, kk, flags, row in heads if not flags & mfi.MAX)
        n_elim = sum(1 for st in desc["steps"] if st["elim"] >= 0)
        assert sum(1 for h in heads if h[1] > 1 or h[3] & mfi.MAX) <= n_elim
        for (_, r0, n0), (_, r1, _) in zip(rows, rows[1:]):
            assert r1 == r0 + n0
        R = sum(n for _, _, n in rows)
        ev = bnet.evidence_sets([cards[v] for v in observed], NB, seed=k)
        scratch = np.full(max(1, R * NB), 0xAB, dtype=np.uint8)
        for b in range(NB):
            e = [int(x) for x in ev[b]]
            value = me.interpret_mixed(prog, tab, n_steps, arena, tables, e, scratch, b, NB)
            assignment = me.decode(desc, scratch, b, NB, observed, e, len(cards), m)
            want_v, want_a = me.emulate(p.h, tables, observed, e, len(cards), m)
            assert _bits(value) == _bits(want_v), (name, b, value, want_v)
            assert assignment == [x & 0xFF for x in want_a], (name, b)
    finally:
        p.close()


def test_map_plan_creation_errors(golden_models):
    cards, scopes, _ = parse_uai(golden_models["asia"]["uai"])
    observed = [7]
    free = [v for v in range(8) if v != 7]

    def rc(m, order, obs=observed, cards_=cards, scopes_=scopes):
        p = me.DryMAPPlan(cards_, scopes_, obs, m, order)
        p.close()
        return p.rc

    assert rc([0, 2], [v for v in free if v not in (0, 2)] + [0, 2]) == OK
    assert rc([7], free) == EINVAL                                     # observed
    assert rc([0, 0], [v for v in free if v] + [0]) == EINVAL         # repeated
    assert rc([8], free) == EINVAL                                     # >= nvars
    assert rc([0], [v for v in free if v not in (0, 3)] + [0]) == EINVAL   # the order misses variable 3
    assert rc([0], [0] + [v for v in free if v]) == EINVAL             # a MAP variable before a summed one
    assert rc([0, 2], [v for v in free if v not in (0, 2)] + [0, 2, 8]) == EINVAL   # order entry >= nvars
    # more than 255 values: refused for a MAP variable, accepted for a summed one
    big = list(cards)
    big[1] = 300
    big_scopes = [[1]] + [sc for sc in scopes if 1 not in sc]
    rest = [v for v in free if v != 1 and any(v in sc for sc in big_scopes)]
    assert rc([1], rest + [1], cards_=big, scopes_=big_scopes) == EINVAL
    assert rc([rest[-1]], [1] + rest, cards_=big, scopes_=big_scopes) == OK
