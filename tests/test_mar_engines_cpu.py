"""All-marginals plans (bnpp_mar_plan_create) without a GPU: where the result steps of the two-pass bucket-tree plan
write, and the step programs of its one-launch engine (K9, `ve_fused`) and of its task engine (K10, `ve_tasks`),
executed by the CPU interpreter of tests/fused_interp.py against the reference's one VE pass per variable
(tests/mar_reference.py).

A marginals plan is not a tree of steps: in its downward pass the product a bucket holds feeds the message to every
child and its own marginal, so one intermediate has several readers.  K10 cuts such a plan into tasks that hand
intermediates to later tasks through the plan's global arena; the interpreted task programs, run in sequence and
sharing that arena and the result buffer, must give every marginal.  The device half is tests/test_gpu_mar_engines.py."""
import math

import numpy as np
import pytest

import batch_networks as bnet
from fused_interp import DryPlan, interpret, parse_uai
from mar_reference import enum_marginals, oracle_marginals, result_steps

REL = 1e-13
TASK_NETWORKS = ["alarm", "win95pts", "hailfinder", "hepar2", "network"]
K9_MULTIVALUED = ["win95pts", "hailfinder", "hepar2"]
RANDOM = ["random_%d" % s for s in range(bnet.N_RANDOM)]

_refs = {}


def _golden_cases(golden_models, name):
    """-> [(cards, scopes, tables, ev)] for every mf evidence case of a golden network"""
    m = golden_models[name]
    cards, scopes, tables = parse_uai(m["uai"])
    return [(cards, scopes, tables, {int(k): int(v) for k, v in c["evidence"].items()}) for c in m["pr"] if c["flag"] == "mf"]


def _random_cases(name):
    """-> [(cards, scopes, tables, ev)]: no evidence, and two evidence sets over the network's observed ids (the second
    observes card - 1 everywhere)"""
    cards, scopes, tables, observed = bnet.network(name, None)
    ev = bnet.evidence_sets([cards[v] for v in observed], 2, 7)
    return [(cards, scopes, tables, {})] + [(cards, scopes, tables, {v: int(x) for v, x in zip(observed, row)}) for row in ev]


def _reference(key, cards, scopes, tables, ev):
    if key not in _refs:
        _refs[key] = oracle_marginals(cards, scopes, tables, ev)
    return _refs[key]


def _dry(cards, scopes, ev):
    observed = sorted(ev)
    return DryPlan(cards, scopes, observed, bnet.mf_order(cards, scopes, observed), marginals=True)


def _normalized(seg):
    """normalize_segments (elementwise.cu): the sum in index order, then a true division"""
    z = 0.0
    for x in seg:
        z += float(x)
    return seg / z


def _check(what, result, layout, want):
    off, size, _ = layout
    for v, w in want.items():
        got = _normalized(result[off[v]:off[v] + size[v]])
        assert got.shape == w.shape, (what, v)
        assert np.all(np.abs(got - w) <= REL * np.abs(w)), (what, v, got, w)      # a zero of the reference is exact


def test_mar_plan_layout(golden_models):
    """every unobserved variable that a factor mentions has exactly one result step, which writes its card(v) entries
    over [v] at its layout offset; observed and unmentioned variables have one-entry slices that no step writes; no
    two result steps overlap and the slices tile the result in id order"""
    cases = []
    for name in golden_models:
        cards, scopes, tables = parse_uai(golden_models[name]["uai"])
        evs = {tuple(sorted(e.items())) for *_, e in _golden_cases(golden_models, name)} | {()}
        cases += [(name, cards, scopes, dict(e)) for e in sorted(evs)]
    for name in RANDOM + ["unmentioned"]:
        cards, scopes, _, observed = bnet.unmentioned_bn() if name == "unmentioned" else bnet.network(name, None)
        cases += [(name, cards, scopes, {}), (name, cards, scopes, {v: 0 for v in observed})]
    n_unmentioned = 0
    for name, cards, scopes, ev in cases:
        p = _dry(cards, scopes, ev)
        try:
            off, size, total = p.layout
            desc, steps = result_steps(p.h)
        finally:
            p.close()
        assert desc["result_size"] == total
        assert off == [sum(size[:v]) for v in range(len(cards))] and total == sum(size), name
        mentioned = {v for sc in scopes for v in sc}
        writers = {}
        for s, roff, ovars, ocards in steps:
            assert len(ovars) == 1, (name, s, ovars)
            writers.setdefault(ovars[0], []).append((s, roff, ocards))
        for v in range(len(cards)):
            if v in ev or v not in mentioned:
                n_unmentioned += v not in mentioned
                assert size[v] == 1 and v not in writers, (name, ev, v)
                continue
            assert size[v] == cards[v], (name, v)
            assert len(writers.get(v, [])) == 1, (name, ev, v, writers.get(v))
            _, roff, ocards = writers[v][0]
            assert roff == off[v] and ocards == [cards[v]], (name, ev, v, roff, off[v], ocards)
        spans = sorted((roff, roff + math.prod(oc)) for _, roff, _, oc in steps)
        assert all(a[1] <= b[0] for a, b in zip(spans, spans[1:])), (name, ev, "result steps overlap")
    assert n_unmentioned >= 2


def _task_cases(golden_models):
    for name in TASK_NETWORKS:
        for i, (cards, scopes, tables, ev) in enumerate(_golden_cases(golden_models, name)):
            yield "%s/%d" % (name, i), cards, scopes, tables, ev
    for name in RANDOM:
        for i, (cards, scopes, tables, ev) in enumerate(_random_cases(name)):
            yield "%s/%d" % (name, i), cards, scopes, tables, ev


def test_mar_task_programs(golden_models):
    """K10: the task programs of a marginals plan cut at most 0 (no limit), 1 and 7 steps per task, interpreted in
    sequence over one global arena and one result buffer, give every marginal of the reference (1e-13)"""
    n = 0
    for key, cards, scopes, tables, ev in _task_cases(golden_models):
        want = _reference(key, cards, scopes, tables, ev)
        observed = sorted(ev)
        p = _dry(cards, scopes, ev)
        try:
            total = p.layout[2]
            for cut in (0, 1, 7):
                segs = p.segments(cut)
                assert segs and segs[0][0] == 0 and segs[-1][1] == p.n_steps(), (key, cut, "tasks cover every step")
                assert all(a[1] == b[0] for a, b in zip(segs, segs[1:])), (key, cut)
                glob, result = {}, np.full(total, np.nan)
                for first, end, lanes, arena, prog, tab in segs:
                    assert cut == 0 or end - first <= cut
                    interpret(prog, tab, end - first, arena, tables, [ev[v] for v in observed], total, glob=glob, result=result)
                _check("%s cut=%d" % (key, cut), result, p.layout, want)
                n += 1
        finally:
            p.close()
    assert n == 3 * (len(RANDOM) * 3 + 9)


def test_mar_fused_program_multivalued(golden_models):
    """K9: the one-launch program of a marginals plan on the multi-valued networks it accepts, every mf evidence case"""
    n = 0
    for name in K9_MULTIVALUED:
        for i, (cards, scopes, tables, ev) in enumerate(_golden_cases(golden_models, name)):
            p = _dry(cards, scopes, ev)
            try:
                G, arena, n_steps = p.fused_info(1)
                assert G > 0, (name, ev, "K9 refuses the plan")
                prog, tab = p.program(1)
                total = p.layout[2]
                result, _ = interpret(prog, tab, n_steps, arena, tables, [ev[v] for v in sorted(ev)], total)
                _check("%s/%d K9" % (name, i), result, p.layout, _reference("%s/%d" % (name, i), cards, scopes, tables, ev))
                n += 1
            finally:
                p.close()
    assert n == 6


@pytest.mark.parametrize("name", ["random_0", "random_3", "random_7", "random_13", "edges"])
def test_oracle_marginals_match_enumeration(name):
    """the two references agree (1e-13) where enumeration is possible"""
    cards, scopes, tables, observed = bnet.unmentioned_bn() if name == "unmentioned" else bnet.network(name, None)
    for row in bnet.evidence_sets([cards[v] for v in observed], 3, 1):
        ev = {v: int(x) for v, x in zip(observed, row)}
        a, b = oracle_marginals(cards, scopes, tables, ev), enum_marginals(cards, scopes, tables, ev)
        assert sorted(a) == sorted(b)
        for v in a:
            assert np.allclose(a[v], b[v], rtol=REL, atol=0.0), (name, ev, v, a[v], b[v])
