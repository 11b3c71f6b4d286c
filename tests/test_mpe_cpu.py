"""MPE plans without a GPU: the schedule of a dry MPE plan (bnpp_mpe_plan_create with ctx = NULL) is executed in max
mode by the CPU emulator of tests/mpe_emulator.py and must give the most probable explanation -- against enumeration
on the small networks and on seeded random networks of mixed cardinalities, against max-product VE in the reference's
bucket order on the others -- and creation must reject what the uint8 argmax tables and the decode cannot serve."""
import math

import numpy as np

import mpe_oracle
import oracle as orc
from bnpp_b200 import model
from fused_interp import parse_uai
from mpe_emulator import DryMPEPlan, emulate

SMALL = ["asia", "asia_positive", "cancer", "earthquake", "grid3x3"]
FLAGS = ["", "mf", "wmf", "md"]


def _order(cards, scopes, ev, flag):
    free = [v for v in range(len(cards)) if v not in ev]
    if not flag:
        return free
    return model.elim_order(cards, scopes, free, flag, observed=sorted(ev))[0]


def _evidence_sets(m):
    seen = []
    for case in m["pr"]:
        ev = {int(k): v for k, v in case["evidence"].items()}
        if ev not in seen:
            seen.append(ev)
    return seen


def _cpt_product(om, assignment):
    p = 1.0
    for f in om.factors:
        idx = int(np.ravel_multi_index([assignment[v] for v in f.scope], [int(om.card[v]) for v in f.scope])) if f.scope else 0
        p *= float(f.values[idx])
    return p


def _check_brute(om, cards, scopes, tables, ev, flag, what):
    observed = sorted(ev)
    p = DryMPEPlan(cards, scopes, observed, _order(cards, scopes, ev, flag))
    assert p.rc == 0, (what, p.rc)
    value, assignment = emulate(p.h, tables, observed, [ev[v] for v in observed], len(cards))
    p.close()
    want, want_a, second = mpe_oracle.mpe_brute_force(om, ev)
    assert math.isclose(value, want, rel_tol=1e-14, abs_tol=0.0), (what, flag, value, want)
    if want > 0 and want - second > 1e-12 * want:
        assert assignment == want_a, (what, flag)


def test_mpe_plans_small_models_against_enumeration(golden_models):
    n = 0
    for name in SMALL:
        m = golden_models[name]
        cards, scopes, tables = parse_uai(m["uai"])
        om = orc.parse_uai(m["uai"])
        for ev in _evidence_sets(m):
            for flag in FLAGS:
                _check_brute(om, cards, scopes, tables, ev, flag, name)
                n += 1
    assert n >= 40


def test_mpe_plans_other_models_against_max_product_ve(golden_models):
    n = 0
    for name, m in golden_models.items():
        if name in SMALL:
            continue
        cards, scopes, tables = parse_uai(m["uai"])
        om = orc.parse_uai(m["uai"])
        # the (heuristic, evidence) pairs the golden PR cases cover: variables in id order is not a usable order on
        # every one of these networks
        for case in m["pr"]:
            ev, flag = {int(k): v for k, v in case["evidence"].items()}, case["flag"]
            observed = sorted(ev)
            order = _order(cards, scopes, ev, flag)
            p = DryMPEPlan(cards, scopes, observed, order)
            assert p.rc == 0, (name, flag, p.rc)
            value, assignment = emulate(p.h, tables, observed, [ev[v] for v in observed], len(cards))
            p.close()
            want, _ = mpe_oracle.mpe_ve(om, ev, order)
            assert math.isclose(value, want, rel_tol=1e-12), (name, flag, value, want)
            assert math.isclose(_cpt_product(om, assignment), value, rel_tol=1e-12), (name, flag)
            assert all(assignment[v] == x for v, x in ev.items())
            n += 1
    assert n >= 40


def random_network(seed, nvars=14, max_parents=3):
    """a seeded Bayesian network with cardinalities 2..5 and a joint of at most 2^20 entries -> UAI text"""
    rng = np.random.default_rng(seed)
    while True:
        cards = [int(c) for c in rng.integers(2, 6, nvars)]
        if np.prod(cards, dtype=np.float64) <= 2 ** 20:
            break
        nvars -= 1
    lines = ["BAYES", str(nvars), " ".join(map(str, cards)), str(nvars)]
    scopes, tables = [], []
    for v in range(nvars):
        k = int(rng.integers(0, min(v, max_parents) + 1))
        parents = sorted(rng.choice(v, size=k, replace=False).tolist()) if k else []
        scopes.append(parents + [v])
        t = rng.uniform(0.05, 1.0, [cards[u] for u in parents] + [cards[v]])
        t[rng.random(t.shape) < 0.1] = 0.0            # some impossible entries
        t += (t.sum(-1, keepdims=True) == 0)          # ... never a whole row
        t /= t.sum(-1, keepdims=True)
        if seed % 4 == 0:
            t = np.round(t, 1)                        # coarse tables: ties between assignments
        tables.append(t.reshape(-1))
    lines += ["%d %s" % (len(s), " ".join(map(str, s))) for s in scopes]
    for t in tables:
        lines += [str(t.size), " ".join(repr(float(x)) for x in t)]
    return "\n".join(lines) + "\n"


def test_mpe_plans_random_mixed_cardinality_networks_against_enumeration():
    for seed in range(20):
        text = random_network(seed)
        cards, scopes, tables = parse_uai(text)
        om = orc.parse_uai(text)
        rng = np.random.default_rng(1000 + seed)
        obs = sorted(rng.choice(len(cards), size=int(rng.integers(0, 4)), replace=False).tolist())
        ev = {v: int(rng.integers(0, cards[v])) for v in obs}
        for flag in FLAGS:
            _check_brute(om, cards, scopes, tables, ev, flag, "random-%d" % seed)


def test_mpe_plan_creation_errors():
    # a variable with 300 values: the argmax tables are uint8
    cards, scopes = [300, 2], [[0], [0, 1]]
    p = DryMPEPlan(cards, scopes, [], [0, 1])
    assert p.rc == -1
    p.close()
    # ... observed, it is fine
    p = DryMPEPlan(cards, scopes, [0], [1])
    assert p.rc == 0
    p.close()
    # an order that misses an unobserved variable some scope mentions
    p = DryMPEPlan([2, 2, 2], [[0], [0, 1], [1, 2]], [], [0, 1])
    assert p.rc == -1
    p.close()
    # ... a variable no factor mentions may be left out (its value is 0)
    p = DryMPEPlan([2, 2, 2], [[0], [0, 1]], [], [0, 1])
    assert p.rc == 0
    p.close()
