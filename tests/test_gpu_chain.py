"""Windows of VE plans on the GPU (contract_chain.cu): a run of wide binary eliminations as one launch with its
intermediates in registers must give the SAME BITS as the per-step launches (chain_depth = 1) -- Z and the result --
on the config-4 network (against tests/golden/wide.json), every slab of the width-30 network, seeded synthetic
networks, a level of three operands and a window the tile cap cuts, in the first run, in graph replays and with new
evidence values after the graph was captured.  Profiled
rows are one per launch: their union entries add up to those of the per-step rows and none reports 0 ms."""
import json
import math
import os

import pytest

pytestmark = pytest.mark.gpu

from bnpp_b200 import capi, synth  # noqa: E402
from plan_emulator import describe  # noqa: E402
from test_chain_plan_cpu import level_ops, synthetic_cases, three_operand_net, tile_cap_net, tile_cut_windows, windows  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def wide():
    return json.load(open(os.path.join(ROOT, "tests", "golden", "wide.json")))["networks"]


def make_plan(bn, observed, order, depth):
    from bnpp_b200 import model
    old = capi.tuning_set("chain_depth", depth)
    try:
        return model.VEPlan(bn.ctx, bn.cards, bn.scopes, observed, order)
    finally:
        capi.tuning_set("chain_depth", old)


def run(bn, plan, obs_val):
    import torch
    res = torch.zeros(2 + plan.result_size, dtype=torch.float64, device="cuda")
    with torch.cuda.stream(bn.ctx.torch_stream):
        res.zero_()
    plan.run(bn.table_ptrs, obs_val, res.data_ptr() + 16, res.data_ptr())
    bn.ctx.sync()
    r = res.cpu().numpy()
    return r[0], r[2:]


def same_bits(bn, observed, order, values_list, want_windows=True):
    """fused (default depth) and per-step plans, three runs each per evidence value set (first run, graph capture,
    replay) -> the Zs of the fused plan; the same bits everywhere"""
    fused, plain = make_plan(bn, observed, order, 4), make_plan(bn, observed, order, 1)
    assert not want_windows or windows(fused.h), "no window formed"
    assert windows(plain.h) == []
    zs = []
    for vals in values_list:
        for _ in range(3):
            zf, rf = run(bn, fused, vals)
            zp, rp = run(bn, plain, vals)
            assert zf.tobytes() == zp.tobytes(), (vals, zf, zp)
            assert rf.tobytes() == rp.tobytes()
        zs.append(float(zf))
    fused.close()
    plain.close()
    return zs


def test_config4_same_bits_and_golden(ctx, wide):
    from bnpp_b200 import model
    N, W, K, seed, ev = synth.wide_bn(1)
    _, bn = model.from_uai_text(ctx, synth.random_bn_uai(N, W, K, seed))
    obs = sorted(ev)
    order, _ = bn.order([v for v in range(N) if v not in ev], ev, "mf")
    vals = [ev[v] for v in obs]
    other = [1 - v for v in vals]             # new evidence values after the replay graph was captured
    z = same_bits(bn, obs, order, [vals, other, vals])
    want = wide["1"]["pr"]
    assert math.isclose(z[0], want, rel_tol=1e-9) and z[2] == z[0], (z, want)
    bn.close()


def test_width30_every_slab_same_bits(ctx, wide):
    from bnpp_b200 import model
    g = wide["8"]
    N, W, K, seed, ev = synth.wide_bn("strong")
    _, bn = model.from_uai_text(ctx, synth.random_bn_uai(N, W, K, seed))
    total, slabs = 0.0, 0
    for key, part in g["partials"].items():
        e = dict(ev)
        e.update((int(a.split("=")[0]), int(a.split("=")[1])) for a in key.split(",") if a)
        obs = sorted(e)
        order, _ = bn.order([v for v in range(N) if v not in e], e, "mf")
        z = same_bits(bn, obs, order, [[e[v] for v in obs]])[0]
        assert math.isclose(z, part["pr"], rel_tol=1e-9), (key, z, part["pr"])
        total += z
        slabs += 1
    assert slabs == 8 and math.isclose(total, g["pr"], rel_tol=1e-9)
    bn.close()


def test_synthetic_networks_same_bits(ctx):
    from bnpp_b200 import model
    done = 0
    for seed, N, W, ev in synthetic_cases():
        _, bn = model.from_uai_text(ctx, synth.random_bn_uai(N, W, 4, seed))
        obs = sorted(ev)
        order, _ = bn.order([v for v in range(N) if v not in ev], ev, "mf")
        vals = [ev[v] for v in obs]
        probe = make_plan(bn, obs, order, 4)
        has = bool(windows(probe.h))
        probe.close()
        if has:
            sets = [vals, [1 - v for v in vals]] if vals else [vals]
            same_bits(bn, obs, order, sets)
            done += 1
        bn.close()
    assert done >= 4


def three_operand_bn(ctx):
    from bnpp_b200 import model
    cards, scopes, tables, order = three_operand_net()
    return model.BN(ctx, cards, list(zip(scopes, tables))), order


def test_three_operand_level_same_bits(ctx):
    """a level multiplying the head by two side tables, (s0 * s1) * h as the step itself does"""
    bn, order = three_operand_bn(ctx)
    probe = make_plan(bn, [], order, 4)
    assert 3 in level_ops(describe(probe.h), windows(probe.h))
    probe.close()
    same_bits(bn, [], order, [[]])
    bn.close()


def test_window_cut_by_the_tile_cap_same_bits(ctx):
    from bnpp_b200 import model
    cards, scopes, tables, order = tile_cap_net()
    bn = model.BN(ctx, cards, list(zip(scopes, tables)))
    probe = make_plan(bn, [], order, 4)
    assert tile_cut_windows(describe(probe.h), windows(probe.h))
    probe.close()
    same_bits(bn, [], order, [[]])
    bn.close()


def test_profiled_rows_are_launches(ctx):
    """one row per launch: union entries add up to those of the per-step plan's rows, no row of moved bytes at 0 ms,
    the windows' rows named contract_chain; over the networks the windows cover levels adding two variables and a
    first level of three operands"""
    from bnpp_b200 import model
    names, k3 = set(), 0
    nets = [("c4",) + tuple(synth.wide_bn(1))] + [(s, N, W, 4, s, ev) for s, N, W, ev in synthetic_cases()] + [("k3",)]
    for net in nets:
        if net[0] == "k3":
            bn, order = three_operand_bn(ctx)
            ev, obs = {}, []
        else:
            tag, N, W, K, seed, ev = net
            _, bn = model.from_uai_text(ctx, synth.random_bn_uai(N, W, K, seed))
            obs = sorted(ev)
            order, _ = bn.order([v for v in range(N) if v not in ev], ev, "mf")
        p = make_plan(bn, obs, order, 4)
        if not windows(p.h):
            p.close()
            bn.close()
            continue
        p.set_profiling(True)
        run(bn, p, [ev[v] for v in obs])
        rows = p.step_stats()
        plain = make_plan(bn, obs, order, 1)          # one row per step: the same steps, the same union entries
        assert sum(r["entries"] for r in rows) == sum(r["entries"] for r in plain.step_stats())
        plain.close()
        assert len(rows) == p.n_launches
        assert sum(r["bytes"] for r in rows) == p.bytes
        assert all(r["ms"] > 0 for r in rows if r["bytes"]), [r for r in rows if r["bytes"] and not r["ms"]]
        chain = [r for r in rows if r["kernel"].startswith("contract_chain")]
        assert len(chain) == len(windows(p.h))
        names.update(r["kernel"] for r in chain)
        k3 += sum(r["k"] == 3 for r in chain)
        p.close()
        bn.close()
    assert any("2" in n.split("add=")[1] for n in names), names
    assert k3 > 0, "no window starts with a three-operand level"
