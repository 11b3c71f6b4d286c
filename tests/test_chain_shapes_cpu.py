"""Every window shape without a GPU: contract_chain has an instantiation for each (m, add) that chain_shape_ok allows,
and a network of tests/chain_nets.py must make the planner form exactly that window -- its levels, their side counts,
one launch for it -- including sides that are raw input views in file order or with an observed variable.  Windows
the tile cap, a third added variable, an added variable eliminated inside the window or chain_depth must cut come out
shorter, and the emulated schedule of a window plan gives the per-step plan's numbers."""
import json
import math
import os

import numpy as np
import pytest

from bnpp_b200 import model, synth
from chain_nets import chain_net, chain_shapes, shape_cases
from fused_interp import DryPlan, parse_uai
from plan_emulator import describe, run
from test_chain_plan_cpu import (check_windows, depth, n_launches, synthetic_cases, three_operand_net, tile_cap_net,
                                 windows)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = shape_cases()


def window_shape(d, a, m):
    """(m, add, k, sides) of the window of m levels starting at step a: the head is the intermediate whose innermost
    axis the first level eliminates, its m fastest axes the tile; a level adds the variables of its sides that are in
    neither the head nor an earlier level's sides"""
    F, steps = d["factors"], d["steps"]
    producer = {st["out"]: i for i, st in enumerate(steps) if st["out"] >= 0}
    first = steps[a]
    head = max((f for f in first["ops"] if F[f]["src"] < 0 and producer.get(f, a) < a and F[f]["axes"][-1][0] == first["elim"]),
               key=lambda f: F[f]["size"])
    hv = [v for v, _, _ in F[head]["axes"]]
    known = set(hv)
    add, k, sides, cur = [], [], [], head
    for j in range(m):
        st = steps[a + j]
        s = [f for f in st["ops"] if f != cur]
        new = {v for f in s for v, _, _ in F[f]["axes"]} - known
        known |= new
        add.append(len(new))
        k.append(len(s))
        sides.append(s)
        cur = st["out"]
    return m, tuple(add), tuple(k), sides


def dry(cards, scopes, obs, order, chain=None):
    if chain is None:
        return DryPlan(cards, scopes, obs, order)
    with depth(chain):
        return DryPlan(cards, scopes, obs, order)


def formed(p):
    d = describe(p.h)
    wins = windows(p.h)
    check_windows(d, wins)
    assert n_launches(p.h) == len(d["steps"]) - sum(m - 1 for _, m in wins)
    return d, wins, [window_shape(d, a, m)[:3] for a, m in wins]


def test_there_are_66_shapes():
    shapes = chain_shapes()
    assert len(shapes) == len(set(shapes)) == 66
    assert sum(m == 2 for m, _ in shapes) == 9 and (4, (0, 0, 0, 2)) in shapes and (4, (2, 0, 0, 0)) not in shapes


@pytest.mark.parametrize("name,m,add,k,opts", CASES, ids=[c[0] for c in CASES])
def test_shape_forms_its_window(name, m, add, k, opts):
    """one window, of exactly that shape and those side counts, following the link rules, one launch"""
    cards, scopes, _, order, obs = chain_net(m, add, k, **opts)
    p = dry(cards, scopes, obs, order)
    _, wins, shapes = formed(p)
    assert shapes == [(m, add, k)], (wins, shapes)
    p.close()


def suite_shapes():
    """the (m, add) of the windows the networks of tests/test_gpu_chain.py form"""
    wide = json.load(open(os.path.join(ROOT, "tests", "golden", "wide.json")))["networks"]
    nets = []
    for key in [1, 2, "strong"]:
        N, W, K, seed, ev = synth.wide_bn(key)
        slabs = [""] if key != "strong" else list(wide["8"]["partials"])
        for slab in slabs:
            e = dict(ev)
            e.update((int(a.split("=")[0]), int(a.split("=")[1])) for a in slab.split(",") if a)
            nets.append((N, W, K, seed, e))
    nets += [(N, W, 4, seed, ev) for seed, N, W, ev in synthetic_cases()]
    out = set()
    for net in nets + ["k3", "cap"]:
        if net == "k3" or net == "cap":
            cards, scopes, _, order = three_operand_net() if net == "k3" else tile_cap_net()
            obs = []
        else:
            N, W, K, seed, ev = net
            cards, scopes, _ = parse_uai(synth.random_bn_uai(N, W, K, seed))
            obs = sorted(ev)
            order, _ = model.elim_order(cards, scopes, [v for v in range(N) if v not in ev], "mf", observed=obs)
        p = DryPlan(cards, scopes, obs, order)
        out |= {s[:2] for s in formed(p)[2]}
        p.close()
    return out


def test_every_shape_and_side_count_is_covered():
    """the cases form all 66 shapes, and every level index sees 0, 1 and 2 side tables"""
    shapes, ks = set(), {}
    for name, m, add, k, opts in CASES:
        shapes.add((m, add))
        for j, kj in enumerate(k):
            ks.setdefault(j, set()).add(kj)
    assert shapes == set(chain_shapes())
    assert all(ks[j] == {0, 1, 2} for j in range(4)), ks
    before = suite_shapes()
    print("window shapes formed: %d by the networks of test_gpu_chain.py, %d with chain_nets (of %d)"
          % (len(before), len(before | shapes), len(chain_shapes())))
    assert before <= shapes


def canonical(axes, order):
    """the dense strides of the axes in canonical order: the earliest eliminated innermost, kept variables outside
    them with the largest id innermost"""
    rank = {v: i for i, v in enumerate(order)}
    st, dense = {}, 1
    for v, c, _ in sorted(axes, key=lambda a: (0, rank[a[0]]) if a[0] in rank else (1, -a[0])):
        st[v] = dense
        dense *= c
    return [st[v] for v, _, _ in axes]


@pytest.mark.parametrize("name,m,add,k,opts", [c for c in CASES if "raw" in c[4]], ids=[c[0] for c in CASES if "raw" in c[4]])
def test_raw_sides_reach_the_window(name, m, add, k, opts):
    """the raw case's side is an input view of 2^16 entries read in place: file-order strides, not the canonical
    ones, and for "ev" an observed axis folded into its base"""
    cards, scopes, tables, order, obs = chain_net(m, add, k, **opts)
    p = DryPlan(cards, scopes, obs, order)
    d, wins, _ = formed(p)
    raw = [f for s in window_shape(d, *wins[0])[3] for f in s if d["factors"][f]["src"] >= 0]
    assert raw, "no side of the window is an input view"
    F = d["factors"]
    for f in raw:
        assert F[f]["size"] == 1 << 16
        assert [s for _, _, s in F[f]["axes"]] != canonical(F[f]["axes"], order)
        assert bool(F[f]["obs"]) == (opts["raw"] == "ev")
        if F[f]["obs"]:
            assert len(scopes[F[f]["src"]]) == 17 and max(s for _, _, s in F[f]["axes"]) == 1 << 16
    p.close()


CUTS = [
    # a level that would add three variables: the window ends before it
    ("add3", (3, (1, 0, 3), (1, 0, 1), {}), None, [(2, (1, 0), (1, 0))]),
    # a tile above 16 doubles: the first level of four would output 2^5
    ("tile4", (4, (2, 0, 0, 0), (1, 0, 0, 0), {}), None, [(3, (2, 0, 0), (1, 0, 0))]),
    # ... the second level of three would output 2^5
    ("tile3", (3, (2, 2, 0), (1, 1, 0), {}), None, [(2, (2, 2), (1, 1))]),
    # the variable level 0 adds is eliminated right after t1: a third level would not eliminate t2, and the step that
    # eliminates it and t2's level form no window of their own (t2's union is 2^19 entries)
    ("inside", (3, (1, 0, 0), (1, 0, 0), {}), None, [(2, (1, 0), (1, 0))]),
    # chain_depth cuts a chain of four: two windows of two, or one of three and a level on its own
    ("depth2", (4, (0, 1, 1, 1), (1, 1, 2, 1), {}), 2, [(2, (0, 1), (1, 1)), (2, (1, 1), (2, 1))]),
    ("depth3", (4, (0, 1, 1, 1), (1, 1, 2, 1), {}), 3, [(3, (0, 1, 1), (1, 1, 2))]),
    ("depth1", (4, (0, 1, 1, 1), (1, 1, 2, 1), {}), 1, []),
]


@pytest.mark.parametrize("name,net,chain,want", CUTS, ids=[c[0] for c in CUTS])
def test_cut_and_fallback(name, net, chain, want):
    m, add, k, opts = net
    cards, scopes, tables, order, obs = chain_net(m, add, k, **opts)
    if name == "inside":
        order.insert(order.index(2) + 1, m + 1)     # the variable level 0 adds, eliminated right after t1
    p = dry(cards, scopes, obs, order, chain)
    _, wins, shapes = formed(p)
    assert shapes == want, (wins, shapes)
    p.close()


EMULATED = [c for c in CASES if c[0] in ("2-22-k21", "3-012-k121", "4-0000-k1201", "3-101-k121-ev", "4-0002-k1022-ev")]


@pytest.mark.parametrize("name,m,add,k,opts", EMULATED, ids=[c[0] for c in EMULATED])
def test_emulated_window_plan_matches_per_step(name, m, add, k, opts):
    """the windowed plan's re-ordered schedule, executed step by step on the CPU, gives the per-step plan's result
    table and Z, for both values of the observed variable"""
    cards, scopes, tables, order, obs = chain_net(m, add, k, **opts)
    p, p0 = dry(cards, scopes, obs, order), dry(cards, scopes, obs, order, 1)
    assert windows(p.h)
    for vals in ([[0], [1]] if obs else [[]]):
        got, z = run(describe(p.h), tables, vals)
        want, z0 = run(describe(p0.h), tables, vals)
        assert got.size >= 1 << 19 and np.isfinite(got).all()
        assert np.allclose(got, want, rtol=1e-12, atol=0) and math.isclose(z, z0, rel_tol=1e-12), (vals, z, z0)
    p.close()
    p0.close()
