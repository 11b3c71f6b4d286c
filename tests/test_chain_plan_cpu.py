"""Windows of VE plans without a GPU (ve.cu form_windows, contract_chain.cu): runs of wide binary eliminations that a
single-query run executes as one contract_chain launch.  Dry plans must form windows only where every link rule
holds, count one launch per window, and keep a schedule that the step-by-step CPU emulator still executes to the
same numbers as the plan without windows."""
import ctypes
import math

import numpy as np
import pytest

from bnpp_b200 import capi, model, synth
from fused_interp import DryPlan, parse_uai
from map_emulator import DryMAPPlan
from mpe_emulator import DryMPEPlan
from plan_emulator import describe, run

MIN_UNION = 1 << 20
MAX_SIDE = 1 << 16
MAX_DEPTH = 4


def windows(h):
    L = capi.lib()
    L.bnpp_ve_plan_windows.argtypes = [ctypes.c_void_p, ctypes.c_uint32, capi.c_u32p, capi.c_u32p, capi.c_u32p]
    n = ctypes.c_uint32()
    assert L.bnpp_ve_plan_windows(h, 0, ctypes.byref(n), None, None) == 0
    a, m = (ctypes.c_uint32 * max(1, n.value))(), (ctypes.c_uint32 * max(1, n.value))()
    assert L.bnpp_ve_plan_windows(h, n.value, ctypes.byref(n), ctypes.cast(a, capi.c_u32p), ctypes.cast(m, capi.c_u32p)) == 0
    return list(zip(a[:n.value], m[:n.value]))


def n_launches(h):
    vals = [ctypes.c_uint64() for _ in range(5)]
    assert capi.lib().bnpp_ve_plan_info(h, None, None, None, *[ctypes.byref(v) for v in vals]) == 0
    return vals[0].value


class depth:
    """bnpp_tuning_set("chain_depth") for the plans created inside"""

    def __init__(self, d):
        self.d = d

    def __enter__(self):
        self.old = capi.tuning_set("chain_depth", self.d)

    def __exit__(self, *a):
        capi.tuning_set("chain_depth", self.old)


def union(d, st):
    n = int(np.prod([c for _, c in st["scope"]], dtype=np.uint64)) if st["scope"] else 1
    return n * (2 if st["elim"] >= 0 else 1)


def check_windows(d, wins):
    """every level of every window satisfies the link rules of form_windows"""
    F, steps = d["factors"], d["steps"]
    readers = {}
    for i, st in enumerate(steps):
        for f in set(st["ops"]):
            readers.setdefault(f, []).append(i)
    producer = {st["out"]: i for i, st in enumerate(steps) if st["out"] >= 0}
    for a, m in wins:
        assert 2 <= m <= MAX_DEPTH
        t1 = steps[a]
        heads = [f for f in t1["ops"] if f in producer and producer[f] < a]
        assert heads, "the first level reads no intermediate"
        prev = None
        for j in range(m):
            st = steps[a + j]
            head = heads[0] if j == 0 else steps[a + j - 1]["out"]
            if j == 0:
                for h in heads:      # the head is the operand whose innermost axis this level eliminates
                    if F[h]["axes"] and F[h]["axes"][-1][0] == st["elim"] and readers[h] == [a]:
                        head = h
            assert st["out"] >= 0 and not st["want_z"] and st["elim"] >= 0
            assert readers[head] == [a + j], "the head / a level's output has another reader"
            assert F[head]["axes"][-1][0] == st["elim"], "a level does not eliminate the innermost axis of its input"
            assert union(d, st) >= MIN_UNION
            for f in st["ops"]:
                assert all(c == 2 for _, c, _ in F[f]["axes"]), "a non-binary variable"
                if f != head:
                    assert F[f]["size"] <= MAX_SIDE, "a side operand above 2^16 entries"
                    assert f not in producer or producer[f] < a, "a side table produced inside the window"
            assert len(st["ops"]) <= 3
            prev = st
        assert prev is not None
        # one launch reads the head and the side tables while it writes the last level's output: disjoint arena slots
        inner = {steps[a + j]["out"] for j in range(m - 1)}
        out = F[prev["out"]]
        for j in range(m):
            for f in steps[a + j]["ops"]:
                if F[f]["src"] < 0 and f not in inner:
                    lo, hi = F[f]["off"], F[f]["off"] + F[f]["size"]
                    assert hi <= out["off"] or out["off"] + out["size"] <= lo, "a window writes over what it reads"


def three_operand_net(seed=7):
    """a wide bucket with two side tables too large to be multiplied together first (fold_small keeps all three): the
    head H(t0, t1, r0..r18) of 2^21 entries, S_a(t0, r0..r13) and S_b(t0, r5..r18) of 2^15 each, then S_c(t1, r0..r3)
    -> (cards, scopes, tables, order); the order eliminates h0 (making H), t0 (three operands), t1, then the rest"""
    rng = np.random.default_rng(seed)
    h0, t0, t1 = 0, 1, 2
    r = list(range(3, 22))
    scopes = [[h0, t0, t1] + r, [t0] + r[:14], [t0] + r[5:], [t1] + r[:4]]
    tables = [rng.uniform(0.5, 1.5, 1 << len(sc)) for sc in scopes]
    return [2] * 22, scopes, tables, [h0, t0, t1] + r


def tile_cap_net(seed=11):
    """levels that add two variables each: H(t0, t1, t2, r0..r17), S0(t0, n0, n1, r0..r2), S1(t1, n2, n3, r0..r2),
    S2(t2, r0); n0..n3 are eliminated last.  Three levels would need a 32-double tile at the second one, so the window
    is cut to two -> (cards, scopes, tables, order)"""
    rng = np.random.default_rng(seed)
    h0, t, r, n = 0, [1, 2, 3], list(range(4, 22)), list(range(22, 26))
    scopes = [[h0] + t + r, [t[0], n[0], n[1]] + r[:3], [t[1], n[2], n[3]] + r[:3], [t[2], r[0]]]
    tables = [rng.uniform(0.5, 1.5, 1 << len(sc)) for sc in scopes]
    return [2] * 26, scopes, tables, [h0] + t + r + n


def level_ops(d, wins):
    """operand counts of every level of every window"""
    return [len(d["steps"][a + j]["ops"]) for a, m in wins for j in range(m)]


def tile_cut_windows(d, wins):
    """windows whose next step would be a link and a level within the depth, but whose tile would then exceed 16
    doubles (some level's input or output above 4 bits): the cut the tile cap makes"""
    F, steps = d["factors"], d["steps"]
    readers = {}
    for i, st in enumerate(steps):
        for f in set(st["ops"]):
            readers.setdefault(f, []).append(i)
    producer = {st["out"]: i for i, st in enumerate(steps) if st["out"] >= 0}
    out = []
    for a, m in wins:
        if m >= MAX_DEPTH:
            continue
        last = steps[a + m - 1]["out"]
        nxt = readers.get(last, [])
        if len(nxt) != 1 or steps[nxt[0]]["out"] < 0 or steps[nxt[0]]["elim"] < 0:
            continue
        t = steps[nxt[0]]
        if F[last]["axes"][-1][0] != t["elim"] or union(d, t) < MIN_UNION or len(t["ops"]) > 3:
            continue
        if any(F[f]["size"] > MAX_SIDE for f in t["ops"] if f != last):
            continue
        levels = [steps[a + j] for j in range(m)] + [t]
        head = max((f for f in levels[0]["ops"] if f in producer and F[f]["axes"][-1][0] == levels[0]["elim"]),
                   key=lambda f: F[f]["size"])
        hv = [v for v, _, _ in F[head]["axes"]]
        if len(hv) < m + 1 or hv[-(m + 1)] != t["elim"]:
            continue
        rest, tile, added, nb, over = set(hv[:-(m + 1)]), hv[::-1][:m + 1], [], 0, False
        cur = head
        for j, st in enumerate(levels):
            new = []
            for f in st["ops"]:
                if f != cur:
                    new += [v for v, _, _ in F[f]["axes"] if v not in tile and v not in rest and v not in added + new]
            inb = (m + 1 - j) + nb
            over |= inb > 4 or inb - 1 + len(new) > 4
            added += new
            nb += len(new)
            cur = st["out"]
        if over:
            out.append((a, m))
    return out


def wide_plan(key, chain=None):
    N, W, K, seed, ev = synth.wide_bn(key)
    cards, scopes, tables = parse_uai(synth.random_bn_uai(N, W, K, seed))
    obs = sorted(ev)
    order, _ = model.elim_order(cards, scopes, [v for v in range(N) if v not in ev], "mf", observed=obs)
    if chain is None:
        return DryPlan(cards, scopes, obs, order)
    with depth(chain):
        return DryPlan(cards, scopes, obs, order)


def test_config4_windows_cut_launches():
    p0 = wide_plan(1, 1)
    assert windows(p0.h) == [] and n_launches(p0.h) == len(describe(p0.h)["steps"])
    p = wide_plan(1)
    d = describe(p.h)
    wins = windows(p.h)
    assert wins, "config 4 forms no window"
    check_windows(d, wins)
    want = len(d["steps"]) - sum(m - 1 for _, m in wins)
    assert n_launches(p.h) == want < n_launches(p0.h) == 87
    # the steps and their union entries stay the same
    d0 = describe(p0.h)
    assert sorted(union(d0, s) for s in d0["steps"]) == sorted(union(d, s) for s in d["steps"])
    p.close()
    p0.close()


@pytest.mark.parametrize("key", ["strong", 2])
def test_wide_networks_windows_follow_the_rules(key):
    p = wide_plan(key)
    wins = windows(p.h)
    assert wins
    check_windows(describe(p.h), wins)
    assert n_launches(p.h) == len(describe(p.h)["steps"]) - sum(m - 1 for _, m in wins)
    p.close()


def synthetic_cases():
    """seeded networks of min-fill width 18-24, without evidence and with leaves observed (evidence on side tables)"""
    out = []
    for seed in range(40):
        N, W = 44 + seed % 5 * 3, 24 + seed % 4 * 2
        cards, scopes, tables = parse_uai(synth.random_bn_uai(N, W, 4, seed))
        order, width = model.elim_order(cards, scopes, list(range(N)), "mf")
        if not 18 <= width <= 24:
            continue
        out.append((seed, N, W, {}))
        parents = set(v for sc in scopes for v in sc[:-1])
        leaves = [v for v in range(N) if v not in parents]
        if leaves:
            out.append((seed, N, W, {v: (v + seed) % 2 for v in leaves[:3]}))
        if len(out) >= 12:
            break
    return out


def test_synthetic_networks_windows_and_emulated_results():
    cases = synthetic_cases()
    assert len(cases) >= 10
    with_windows = emulated = 0
    for seed, N, W, ev in cases:
        cards, scopes, tables = parse_uai(synth.random_bn_uai(N, W, 4, seed))
        obs = sorted(ev)
        order, width = model.elim_order(cards, scopes, [v for v in range(N) if v not in ev], "mf", observed=obs)
        p = DryPlan(cards, scopes, obs, order)
        d = describe(p.h)
        wins = windows(p.h)
        check_windows(d, wins)
        assert n_launches(p.h) == len(d["steps"]) - sum(m - 1 for _, m in wins)
        with_windows += bool(wins)
        if wins and width <= 21 and emulated < 3:
            # the re-ordered schedule, executed step by step, gives what the schedule without windows gives
            with depth(1):
                p0 = DryPlan(cards, scopes, obs, order)
            vals = [ev[v] for v in obs]
            got, _ = run(d, tables, vals)
            want, _ = run(describe(p0.h), tables, vals)
            assert math.isclose(got[0], want[0], rel_tol=1e-12), (seed, got[0], want[0])
            if not ev:
                assert math.isclose(got[0], 1.0, rel_tol=1e-9)
            p0.close()
            emulated += 1
        p.close()
    assert with_windows >= 4 and emulated >= 1


def test_three_operand_level_forms_a_window():
    """a level whose step multiplies the head by two side tables ((s0 * s1) * h, the step's own order) is fused, and
    the re-ordered schedule still emulates to the per-step plan's numbers"""
    cards, scopes, tables, order = three_operand_net()
    p = DryPlan(cards, scopes, [], order)
    d = describe(p.h)
    wins = windows(p.h)
    check_windows(d, wins)
    assert 3 in level_ops(d, wins), (wins, level_ops(d, wins))
    with depth(1):
        p0 = DryPlan(cards, scopes, [], order)
    got, _ = run(d, tables, [])
    want, _ = run(describe(p0.h), tables, [])
    assert math.isclose(got[0], want[0], rel_tol=1e-12), (got[0], want[0])
    p.close()
    p0.close()


def test_tile_cap_cuts_windows():
    """the 16-double tile cuts a window: the next step links, but its level would need a larger tile"""
    cards, scopes, tables, order = tile_cap_net()
    p = DryPlan(cards, scopes, [], order)
    d = describe(p.h)
    wins = windows(p.h)
    check_windows(d, wins)
    assert tile_cut_windows(d, wins), wins
    p.close()


def test_windows_keep_the_arena_and_the_peak():
    """a window's head and side tables live until its last level; the inner levels' outputs keep their per-step
    lifetimes, so the arena and the reported peak stay near those of the plan without windows"""
    for key in [1, 2, "strong"]:
        p, p0 = wide_plan(key), wide_plan(key, 1)
        d, d0 = describe(p.h), describe(p0.h)
        extent = lambda dd: max(f["off"] + f["size"] for f in dd["factors"] if f["src"] < 0)
        assert extent(d) <= 1.25 * extent(d0), (key, extent(d), extent(d0))
        peak = lambda h: [ctypes.c_uint64() for _ in range(5)]
        v, v0 = peak(p.h), peak(p0.h)
        capi.lib().bnpp_ve_plan_info(p.h, None, None, None, *[ctypes.byref(x) for x in v])
        capi.lib().bnpp_ve_plan_info(p0.h, None, None, None, *[ctypes.byref(x) for x in v0])
        assert v[3].value <= 1.25 * v0[3].value, (key, v[3].value, v0[3].value)
        p.close()
        p0.close()


def test_mpe_and_map_plans_form_no_windows():
    """the argmax rows of max steps follow the step order: MPE and MAP plans keep one launch per step"""
    for seed, N, W, ev in synthetic_cases():
        if ev:
            continue
        cards, scopes, _ = parse_uai(synth.random_bn_uai(N, W, 4, seed))
        order, width = model.elim_order(cards, scopes, list(range(N)), "mf")
        pr = DryPlan(cards, scopes, [], order)
        if not windows(pr.h):
            pr.close()
            continue
        mpe = DryMPEPlan(cards, scopes, [], order)
        assert mpe.rc == 0 and windows(mpe.h) == []
        map_vars = order[-4:]          # the order ends with the MAP variables
        mp = DryMAPPlan(cards, scopes, [], map_vars, order)
        assert mp.rc == 0 and windows(mp.h) == []
        for p in (pr, mpe, mp):
            p.close()
        return
    pytest.fail("no synthetic network with windows")
