"""Marginal MAP on the GPU (bnpp_map_plan_create; BN.map, BN.map_batch; `bn` prompt command `map`).

Single runs (launch per bucket, the decode as the last node of the replay graph) must equal the CPU emulation of the
dry plan in mixed mode (tests/map_emulator.py) bit for bit -- value bits and the assignment of every variable, the
summed-variable sentinel included -- on the first run, with other evidence and on graph replay.  M = every unobserved
variable must give bnpp_mpe_plan_run's answer and M empty bnpp_ve_plan_run's value, bit for bit.

Batches go through `ve_fused_mixed` (K9 with sum and max steps in one program, the default and every forced lane
width) and K8 (`contract_batched*` for sum steps, their max variants for max steps: plain, captured, and replayed after
the evidence changed in place); every set must equal its single bnpp_mpe_plan_run on the same MAP plan bit for bit."""
import math
import os
import random
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import batch_networks as bnet  # noqa: E402
import map_emulator as me  # noqa: E402
import map_oracle  # noqa: E402
from fused_interp import parse_uai  # noqa: E402
from plan_emulator import describe  # noqa: E402
from test_gpu_mpe_batch import BAD_EVIDENCE, BATCHES, EINVAL, LANES, SMALL, _same, _vals, _zero_bn  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "bnpp_b200", "bin")
NETWORKS = SMALL + list(bnet.MV_GOLDEN) + ["random_%d" % s for s in range(bnet.N_RANDOM)] + ["many_parents", "unmentioned"]
SUMMED8 = 0xFF


@pytest.fixture(scope="module")
def ctx():
    from bnpp_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


def _network(name, golden_models):
    if name in SMALL:
        cards, scopes, tables = parse_uai(golden_models[name]["uai"])
        obs = sorted(int(v) for v in next((c["evidence"] for c in golden_models[name]["pr"] if c["evidence"]), {}))
        return cards, scopes, tables, obs
    if name == "unmentioned":
        return bnet.unmentioned_bn()
    return bnet.network(name, golden_models)


def _map_set(name, cards, observed):
    """a seeded MAP set of about a third of the unobserved variables, at most three (at least one, never all of two or
    more): wider MAP sets make the constrained order of the golden networks too wide for K9"""
    free = [v for v in range(len(cards)) if v not in set(observed)]
    k = max(1, min(len(free) - 1, len(free) // 3, 3)) if len(free) > 1 else len(free)
    return sorted(random.Random("map-gpu-" + name).sample(free, k))


class MapNet:
    """a network on the device, the MAP plan of (M, its observed ids, heuristic) that BN.map and BN.map_batch share,
    and single-run references of its evidence sets (bnpp_mpe_plan_run on that plan, every variable's assignment)"""

    def __init__(self, ctx, name, cards, scopes, tables, observed, m, heuristic="mf", nsets=max(BATCHES), seed=0):
        import torch
        from bnpp_b200 import model
        self.ctx, self.name, self.cards, self.scopes, self.observed, self.m = ctx, name, cards, scopes, list(observed), list(m)
        self.tables = [np.asarray(t, dtype=np.float64) for t in tables]
        self.heuristic = heuristic
        self.bn = model.BN(ctx, cards, list(zip(scopes, tables)))
        self.plan = self.bn._map_plan(self.m, self.observed, heuristic)
        self.order = self.bn._order_cache[("map", tuple(self.observed), tuple(sorted(self.m)), heuristic)]
        self.ev = bnet.evidence_sets([cards[v] for v in self.observed], nsets, seed)
        with torch.cuda.stream(ctx.torch_stream):
            self.buf = torch.empty(2 + len(cards), dtype=torch.int32, device="cuda:%d" % ctx.device)
        self._ref = {}

    def run_single(self, row):
        """-> (value, assignment as uint32 list) of one bnpp_mpe_plan_run on the MAP plan"""
        self.plan.run_mpe(self.bn.table_ptrs, [int(x) for x in row], self.buf.data_ptr(), self.buf.data_ptr() + 8)
        self.ctx.sync()
        host = self.buf.cpu().numpy()
        return float(host[:2].view(np.float64)[0]), [int(x) for x in host[2:].view(np.uint32)]

    def single(self, row):
        key = bytes(np.asarray(row, dtype=np.uint8))
        if key not in self._ref:
            self._ref[key] = self.run_single(row)
        return self._ref[key]

    def refs(self, rows):
        r = [self.single(row) for row in rows]
        return (np.array([v for v, _ in r], dtype=np.float64),
                np.array([[x & 0xFF for x in a] for _, a in r], dtype=np.uint8).T.reshape(len(self.cards), -1))

    def emulate(self, row):
        p = me.DryMAPPlan(self.cards, self.scopes, self.observed, self.m, self.order)
        try:
            assert p.rc == 0
            return me.emulate(p.h, self.tables, self.observed, [int(x) for x in row], len(self.cards), self.m)
        finally:
            p.close()

    def close(self):
        self.bn.close()


def _check_single(net, rows):
    """single runs against the emulation: the first run, other evidence, and the replay graph with the first evidence
    again; value bits and every variable's assignment"""
    for i, row in enumerate(list(rows) + [rows[0], rows[0]]):
        got = net.run_single(row)
        want = net.emulate(row)
        assert np.float64(got[0]).view(np.uint64) == np.float64(want[0]).view(np.uint64), (net.name, i, got[0], want[0])
        assert got[1] == want[1], (net.name, i)


@pytest.mark.parametrize("name", SMALL + ["alarm", "hepar2", "child"] + ["random_%d" % s for s in range(6)])
@pytest.mark.parametrize("heuristic", [None, "mf"])
def test_single_runs_equal_emulation(ctx, golden_models, name, heuristic):
    cards, scopes, tables, observed = _network(name, golden_models)
    net = MapNet(ctx, name, cards, scopes, tables, observed, _map_set(name, cards, observed), heuristic, nsets=4, seed=2)
    try:
        _check_single(net, net.ev)
        value, xm, _ = net.bn.map(net.m, dict(zip(observed, (int(x) for x in net.ev[2]))), heuristic)
        want = net.emulate(net.ev[2])
        assert np.float64(value).view(np.uint64) == np.float64(want[0]).view(np.uint64)
        assert xm == {v: want[1][v] for v in net.m}
    finally:
        net.close()


def _wide_summed_bn(seed=3):
    """a summed root of 300 values above a MAP pair: summed variables may have any cardinality"""
    rng = random.Random(seed)
    cards = [300, 3, 2, 2, 4]
    scopes = [[0], [1, 0], [2, 1, 0], [3, 2], [4, 1]]
    tables = [bnet._cpt(rng, cards, sc[0], sc[1:]) for sc in scopes]
    return cards, scopes, tables, [3]


def test_summed_variable_of_300_values(ctx):
    cards, scopes, tables, observed = _wide_summed_bn()
    net = MapNet(ctx, "wide", cards, scopes, tables, observed, [1, 2], "mf", nsets=3, seed=1)
    try:
        _check_single(net, net.ev)
        for row in net.ev:
            e = {3: int(row[0])}
            value, assignment = net.run_single(row)
            best, best_a, second = map_oracle.map_brute_force(cards, scopes, tables, e, [1, 2])
            assert math.isclose(value, best, rel_tol=1e-12)
            if best - second > 1e-9 * best:
                assert {v: assignment[v] for v in (1, 2)} == best_a
            assert assignment[0] == assignment[4] == me.ASSIGN_SUMMED
        for nb in (2, 257):
            ev = bnet.evidence_sets([2], nb, seed=nb)
            _check_batches(net, ev)
    finally:
        net.close()


@pytest.mark.parametrize("name", ["asia", "alarm", "random_3", "many_parents"])
def test_all_and_no_map_variables(ctx, golden_models, name):
    """M = every unobserved variable: bnpp_mpe_plan_run's value and assignment; M empty: bnpp_ve_plan_run's value"""
    cards, scopes, tables, observed = _network(name, golden_models)
    free = [v for v in range(len(cards)) if v not in set(observed)]
    from bnpp_b200 import model
    bn = model.BN(ctx, cards, list(zip(scopes, tables)))
    try:
        for row in bnet.evidence_sets([cards[v] for v in observed], 3, seed=4):
            ev = {v: int(x) for v, x in zip(observed, row)}
            for h in (None, "mf"):
                mv, ma, _ = bn.mpe(ev, h)
                v, xm, _ = bn.map(free, ev, h)
                assert np.float64(v).view(np.uint64) == np.float64(mv).view(np.uint64), (name, h)
                assert xm == {u: ma[u] for u in free}, (name, h)
                z, _ = bn.partition(ev, h)
                v0, x0, _ = bn.map([], ev, h)
                assert np.float64(v0).view(np.uint64) == np.float64(z).view(np.uint64), (name, h, v0, z)
                assert x0 == {}
        # the batches of both extremes equal their single runs as well
        for m in (free, []):
            net = MapNet(ctx, name, cards, scopes, tables, observed, m, "mf", nsets=257, seed=5)
            try:
                _check_batches(net, net.ev[:257])
            finally:
                net.close()
    finally:
        bn.close()


def _batch(net, vals, fused=True, lanes=None):
    """-> (values, assignment [nvars][nb], status bits, lanes per set (0: K8), name of the last kernel launch)"""
    net.ctx.status()
    net.plan.set_fused(fused)
    if lanes:
        os.environ["BNPP_FUSED_G"] = str(lanes)
    try:
        g = net.plan.fused_info(vals.shape[0])[0] if fused and vals.shape[0] > 1 else 0
        value, assignment = net.bn.map_batch(net.m, net.observed, vals, net.heuristic)
        net.ctx.sync()
        return value.cpu().numpy().copy(), assignment.cpu().numpy().copy(), net.ctx.status(), g, net.ctx.last_launch()[0]
    finally:
        os.environ.pop("BNPP_FUSED_G", None)
        net.plan.set_fused(True)


def _mixed(net):
    """the plan has both summing and max steps"""
    d = describe(net.plan.h)
    elims = [st["elim"] for st in d["steps"] if st["elim"] >= 0]
    return any(e in net.m for e in elims) and any(e not in net.m for e in elims)


def _check_batches(net, ev, expect_k9=True, used_lanes=None):
    import torch
    nb = ev.shape[0]
    want = net.refs(ev)
    vals = _vals(ev)
    mixed = _mixed(net)
    v, a, st, g, kern = _batch(net, vals)
    assert st == 0, (net.name, nb, st)
    if nb > 1 and expect_k9:
        assert g > 0, (net.name, nb)
        assert kern.startswith("ve_fused_mixed<") == mixed, (net.name, kern)
    _same((v, a), want, "%s nb=%d default (lanes %d, %s)" % (net.name, nb, g, kern))
    for lanes in LANES:
        vl, al, st, g, kern = _batch(net, vals, lanes=lanes)
        assert st == 0
        if g and mixed:
            assert kern == "ve_fused_mixed<G=%d>" % g, (net.name, kern, g)
        if used_lanes is not None and g:
            used_lanes.add(g)
        _same((vl, al), want, "%s nb=%d BNPP_FUSED_G=%d (lanes %d)" % (net.name, nb, lanes, g))
    for rep in range(2):
        vk, ak, st, _, _ = _batch(net, vals, fused=False)
        assert st == 0
        _same((vk, ak), want, "%s nb=%d K8 run %d" % (net.name, nb, rep + 1))
    new = np.roll(ev, 1, axis=0) if nb > 1 else next((r for r in net.ev if not np.array_equal(r, ev[0])), ev[0])[None]
    with torch.cuda.stream(net.ctx.torch_stream):
        vals.copy_(torch.from_numpy(np.ascontiguousarray(new)).to(vals.device))
    net.ctx.sync()
    vk, ak, st, _, _ = _batch(net, vals, fused=False)
    assert st == 0
    _same((vk, ak), net.refs(new), "%s nb=%d K8 replay after new evidence" % (net.name, nb))
    return v, a


@pytest.mark.parametrize("name", NETWORKS)
def test_batch_equals_single_runs(ctx, golden_models, name):
    cards, scopes, tables, observed = _network(name, golden_models)
    m = _map_set(name, cards, observed)
    net = MapNet(ctx, name, cards, scopes, tables, observed, m, "mf", seed=len(name))
    expect_k9 = name not in ("insurance", "Water")      # their constrained orders have buckets too wide for K9
    if not expect_k9:
        assert net.plan.fused_info(2)[0] == 0
    try:
        assert _mixed(net) or name in ("cancer", "earthquake"), name
        for nb in BATCHES:
            _, a = _check_batches(net, net.ev[:nb], expect_k9)
            summed = [v for v in range(len(cards)) if v not in set(observed) and v not in set(m)]
            assert (a[summed] == SUMMED8).all()
            assert np.array_equal(a[observed], net.ev[:nb].T) or not observed
    finally:
        net.close()


def test_every_lane_width_runs_the_mixed_interpreter(ctx):
    used = set()
    for seed in range(4):
        cards, scopes, tables, observed = bnet.mixed_bn(seed)
        net = MapNet(ctx, "random_%d" % seed, cards, scopes, tables, observed, _map_set("r%d" % seed, cards, observed),
                     seed=seed)
        try:
            assert _mixed(net)
            _check_batches(net, net.ev[:257], True, used_lanes=used)
        finally:
            net.close()
    assert used >= {8, 16, 32, 128}, used


def test_sliced_batch_odd_slices_ragged_tail(ctx):
    """K8 slices a batch (odd slice size, a short last slice, slice + 1); the argmax rows of the max steps only"""
    cards, scopes, tables, observed = bnet.sliced_bn()
    m = [v for v in range(len(cards) - 12, len(cards)) if v not in observed]
    net = MapNet(ctx, "sliced", cards, scopes, tables, observed, m, "mf", nsets=8)
    try:
        desc = describe(net.plan.h)
        R = sum(n for _, _, n in me.rows(desc, set(m)))
        s = min(bnet.slice_of(desc, 1 << 30), (1 << 30) // max(1, R))
        assert s % 2 == 1 and s > 2, s
        assert net.plan.fused_info(2)[0] == 0
        rng = random.Random(7)
        for nb in (s + 1, 2 * s + s // 3):
            ev = bnet.evidence_sets([cards[v] for v in observed], nb, seed=nb)
            vals = _vals(ev)
            bounds = {0, 1, s - 2, s - 1, s, nb - 1} | ({s + 1, 2 * s - 1, 2 * s, 2 * s + 1} if nb > 2 * s else set())
            sample = sorted(bounds | set(rng.sample(range(nb), 24)))
            want = net.refs(ev[sample])
            for rep in range(3):
                v, a, st, _, _ = _batch(net, vals, fused=rep == 0)
                assert st == 0
                _same((v[sample], a[:, sample]), want, "sliced nb=%d run %d" % (nb, rep + 1))
    finally:
        net.close()


def test_zero_probability_sets_in_a_batch(ctx):
    cards, scopes, tables, observed = _zero_bn()
    net = MapNet(ctx, "zero", cards, scopes, tables, observed, [2], "mf", nsets=257, seed=1)
    try:
        for nb in (2, 3, 257):
            ev = net.ev[:nb].copy()
            ev[::2, 0] = 1
            ev[1::2, 0] = 0
            v, a = _check_batches(net, ev)
            assert (v[::2] == 0).all() and (v[1::2] > 0).all()
            assert (a[2, ::2] == 0).all() and (a[0] == SUMMED8).all()
    finally:
        net.close()


@pytest.mark.parametrize("fused", [True, False])
def test_out_of_range_evidence(ctx, fused):
    cards, scopes, tables, observed = bnet.edge_bn()
    net = MapNet(ctx, "edges", cards, scopes, tables, observed, [4, 6], "mf", nsets=6, seed=6)
    try:
        bad = net.ev.copy()
        bad[3, 2] = 2
        v, a, st, g, _ = _batch(net, _vals(bad), fused=fused)
        assert (g > 0) == fused
        assert st & BAD_EVIDENCE
        read_as = bad.copy()
        read_as[3, 2] = 0
        _same((v, a), net.refs(read_as), "illegal value 2 of a card-2 column (fused=%s)" % fused)
        assert a[observed[2], 3] == 0
    finally:
        net.close()


def config5():
    """config 5 (500 variables, W=6 K=3 seed=11, 20 fixed observed ids) and the MAP set of tools/map_bench.py: the last
    20 unobserved ids (20 ids drawn at random give a constrained width of 22, too wide for K9)"""
    from bnpp_b200 import synth
    N, W, K, seed, nobs = 500, 6, 3, 11, 20
    cards, scopes, tables = parse_uai(synth.random_bn_uai(N, W, K, seed))
    evs = synth.evidence_batch(N, nobs, 1 << 16, seed=5, fixed_ids=True)
    observed = sorted(evs[0])
    free = [v for v in range(N) if v not in set(observed)]
    m = free[-20:]
    return cards, scopes, tables, observed, m, evs


def test_config5_sample_against_single_runs(ctx):
    cards, scopes, tables, observed, m, evs = config5()
    net = MapNet(ctx, "config5", cards, scopes, tables, observed, m, "mf", nsets=2)
    try:
        ev = np.array([[e[v] for v in observed] for e in evs], dtype=np.uint8)
        sample = sorted(random.Random(5).sample(range(ev.shape[0]), 512))
        want = net.refs(ev[sample])
        vals = _vals(ev)
        v, a, st, g, kern = _batch(net, vals)
        assert st == 0 and g > 0 and kern.startswith("ve_fused_mixed<"), kern
        _same((v[sample], a[:, sample]), want, "config 5 K9")
        vk, ak, st, _, _ = _batch(net, vals, fused=False)
        assert st == 0
        _same((vk[sample], ak[:, sample]), want, "config 5 K8")
        assert np.array_equal(v.view(np.uint64), vk.view(np.uint64)) and np.array_equal(a, ak)
    finally:
        net.close()


def test_api_errors(ctx):
    import ctypes
    import torch
    from bnpp_b200 import capi
    cards, scopes, tables, observed = bnet.mixed_bn(1)
    net = MapNet(ctx, "errors", cards, scopes, tables, observed, _map_set("errors", cards, observed), nsets=4)
    dev = torch.device("cuda:%d" % ctx.device)
    ev = _vals(net.ev)
    value = torch.empty(4, dtype=torch.float64, device=dev)
    assign = torch.empty((len(cards), 4), dtype=torch.uint8, device=dev)
    tp = (ctypes.c_void_p * len(net.bn.table_ptrs))(*net.bn.table_ptrs)
    try:
        assert ctx.L.bnpp_mpe_plan_run_batched(net.plan.h, tp, 4, len(observed), ctypes.c_void_p(ev.data_ptr()),
                                               ctypes.c_void_p(value.data_ptr()), ctypes.c_void_p(assign.data_ptr())) == 0
        ctx.sync()
        assert ctx.L.bnpp_mpe_plan_run_batched(net.plan.h, tp, 4, len(observed) + 1, ctypes.c_void_p(ev.data_ptr()),
                                               ctypes.c_void_p(value.data_ptr()), ctypes.c_void_p(assign.data_ptr())) == EINVAL
        for call in (lambda: net.plan.run_batched(net.bn.table_ptrs, 4, ev.data_ptr(), value.data_ptr()),
                     lambda: net.plan.run(net.bn.table_ptrs, [int(x) for x in net.ev[0]], value.data_ptr())):
            with pytest.raises(capi.BnppError) as e:       # the sum-product entries refuse MAP plans
                call()
            assert e.value.code == EINVAL
        free = [v for v in range(len(cards)) if v not in observed]
        for bad in ([observed[0]], [free[0], free[0]], [len(cards)]):
            with pytest.raises(capi.BnppError) as e:
                net.bn.map(bad, {v: 0 for v in observed})
            assert e.value.code == EINVAL, bad
    finally:
        net.close()


def test_bn_cli_map(tmp_path, golden_models):
    """`map 0, 2` at the bn prompt prints what BN.map returns for the file's evidence"""
    from bnpp_b200 import capi, model
    uai = tmp_path / "asia.uai"
    uai.write_text(golden_models["asia"]["uai"])
    evid = tmp_path / "asia.uai.evid"
    evid.write_text("1\n2 6 0 7 1")
    c = capi.Context(0)
    try:
        _, bn = model.from_uai_text(c, golden_models["asia"]["uai"])
        for extra, h in [([], None), (["-mf"], "mf")]:
            want, want_x, _ = bn.map([0, 2], {6: 0, 7: 1}, h)
            p = subprocess.run([os.path.join(BIN, "bn"), str(uai), str(evid)] + extra, input="map 0, 2\nquit\n",
                               capture_output=True, text=True, timeout=300)
            assert p.returncode == 0, p.stderr
            lines = [ln.split("? ")[-1] for ln in p.stdout.splitlines()]
            i = next(k for k, ln in enumerate(lines) if ln.startswith(">> MAP = "))
            assert math.isclose(float(lines[i].split("=")[1]), want, rel_tol=1e-5), (lines[i], want)
            assert lines[i + 1] == ">> Assignment = 0=%d 2=%d" % (want_x[0], want_x[2]), lines[i + 1]
            assert lines[i + 2].startswith(">> Executed in ")
        bn.close()
    finally:
        c.close()
