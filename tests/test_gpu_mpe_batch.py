"""Batched MPE (bnpp_mpe_plan_run_batched, BN.mpe_batch) through both batch engines: `ve_fused_max` (K9 in max mode, the
whole plan in one launch per slice, every lane width) and the max-product variants of `contract_batched*` (K8, one
launch per bucket: first run, captured run, and the replayed graph after the evidence changed in place), each followed
by the per-set decode.

Every set of every batch must equal its own single query (`BN.mpe`, i.e. bnpp_mpe_plan_run through the same plan):
the value bit for bit and the whole assignment.  The networks: the small and the multi-valued golden networks, 20
seeded mixed-cardinality networks, a CPT with ten observed axes (K8's evidence digits), an observed variable no factor
mentions, a network whose K8 slices are odd with a short last one, uniform CPTs (every assignment ties), a batch mixing
zero-probability sets with normal ones, and config 5 (65 536 sets)."""
import ctypes
import os
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import batch_networks as bnet  # noqa: E402
from fused_interp import parse_uai  # noqa: E402

BATCHES = (1, 2, 3, 257, 1027)
LANES = (2, 4, 8, 16, 32, 128)      # every width fused_valid_g accepts
SMALL = ["asia", "asia_positive", "cancer", "earthquake", "grid3x3"]
NETWORKS = SMALL + list(bnet.MV_GOLDEN) + ["random_%d" % s for s in range(bnet.N_RANDOM)] + ["many_parents", "unmentioned"]
BAD_EVIDENCE = 2        # BNPP_STATUS_BAD_EVIDENCE
EINVAL = -1


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


class Net:
    """a network on the device, the MPE plan of its observed ids (the one BN.mpe and BN.mpe_batch share) and the
    single-query references of its evidence sets"""

    def __init__(self, ctx, name, cards, scopes, tables, observed, nsets=max(BATCHES), seed=0):
        from bnpp_b200 import model
        self.ctx, self.name, self.cards, self.observed = ctx, name, cards, list(observed)
        self.bn = model.BN(ctx, cards, list(zip(scopes, tables)))
        self.order = bnet.mf_order(cards, scopes, self.observed)
        self.plan = self.bn._cached_plan(("mpe", tuple(self.observed), tuple(self.order)), model.MPEPlan, self.observed,
                                         self.order)
        self.ev = bnet.evidence_sets([cards[v] for v in self.observed], nsets, seed)
        self._ref = {}

    def single(self, row):
        key = bytes(np.asarray(row, dtype=np.uint8))
        if key not in self._ref:
            value, assignment, _ = self.bn.mpe({v: int(x) for v, x in zip(self.observed, row)}, "mf")
            self._ref[key] = (value, assignment)
        return self._ref[key]

    def refs(self, rows):
        r = [self.single(row) for row in rows]
        return np.array([v for v, _ in r], dtype=np.float64), np.array([a for _, a in r], dtype=np.uint8).T.reshape(len(self.cards), -1)

    def close(self):
        self.bn.close()


def _vals(ev):
    import torch
    t = torch.tensor(np.ascontiguousarray(ev), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    return t


def _batch(net, vals, fused=True, lanes=None):
    """-> (values, assignment [nvars][nb], BNPP status bits of the run, lanes per set the run used (0: K8))"""
    net.ctx.status()            # clear
    net.plan.set_fused(fused)
    if lanes:
        os.environ["BNPP_FUSED_G"] = str(lanes)
    try:
        g = net.plan.fused_info(vals.shape[0])[0] if fused and vals.shape[0] > 1 else 0
        value, assignment = net.bn.mpe_batch(net.observed, vals, "mf")
        net.ctx.sync()
        return value.cpu().numpy().copy(), assignment.cpu().numpy().copy(), net.ctx.status(), g
    finally:
        os.environ.pop("BNPP_FUSED_G", None)
        net.plan.set_fused(True)


def _same(got, want, what):
    gv, ga = got
    wv, wa = want
    bad = np.flatnonzero(gv.view(np.uint64) != wv.view(np.uint64))
    if bad.size:
        i = bad[0]
        pytest.fail("%s: %d of %d values differ from the single queries, first set %d: %r != %r" % (what, bad.size, gv.size, i, gv[i], wv[i]))
    assert ga.shape == wa.shape, (what, ga.shape, wa.shape)
    bad = np.argwhere(ga != wa)
    if bad.size:
        v, b = bad[0]
        pytest.fail("%s: %d assignment entries differ, first variable %d of set %d: %d != %d" % (what, len(bad), v, b, ga[v, b], wa[v, b]))


def check_engines(net, ev, expect_k9, used_lanes=None):
    """every engine on one batch against the single queries -> (values, assignment) of the batch"""
    import torch
    nb = ev.shape[0]
    want = net.refs(ev)
    vals = _vals(ev)
    v, a, st, g = _batch(net, vals)
    assert st == 0, (net.name, nb, st)
    if nb > 1 and expect_k9:
        assert g > 0, (net.name, nb)
    _same((v, a), want, "%s nb=%d default (lanes %d)" % (net.name, nb, g))
    for lanes in LANES:
        vl, al, st, g = _batch(net, vals, lanes=lanes)
        assert st == 0
        if used_lanes is not None and g:
            used_lanes.add(g)
        _same((vl, al), want, "%s nb=%d BNPP_FUSED_G=%d (lanes %d)" % (net.name, nb, lanes, g))
    # K8: plain run, captured run, then the replayed graph after the evidence changed in place
    for rep in range(2):
        vk, ak, st, _ = _batch(net, vals, fused=False)
        assert st == 0
        _same((vk, ak), want, "%s nb=%d K8 run %d" % (net.name, nb, rep + 1))
    new = np.roll(ev, 1, axis=0) if nb > 1 else next((r for r in net.ev if not np.array_equal(r, ev[0])), ev[0])[None]
    if net.observed and nb == 1:
        assert not np.array_equal(new, ev)
    with torch.cuda.stream(net.ctx.torch_stream):
        vals.copy_(torch.from_numpy(np.ascontiguousarray(new)).to(vals.device))
    net.ctx.sync()
    vk, ak, st, _ = _batch(net, vals, fused=False)
    assert st == 0
    _same((vk, ak), net.refs(new), "%s nb=%d K8 replay after new evidence" % (net.name, nb))
    return v, a


@pytest.mark.parametrize("name", NETWORKS)
def test_batch_equals_single_queries(ctx, golden_models, name):
    net = Net(ctx, name, *_network(name, golden_models), seed=len(name))
    expect_k9 = name != "Water"          # Water's widest buckets run one launch each
    if not expect_k9:
        assert net.plan.fused_info(2)[0] == 0
    try:
        for nb in BATCHES:
            check_engines(net, net.ev[:nb], expect_k9)
        if name == "many_parents":
            from plan_emulator import describe
            assert bnet.max_observed_axes(describe(net.plan.h)) > 8
    finally:
        net.close()


def test_every_lane_width_is_exercised(ctx):
    """BNPP_FUSED_G reaches every K9 group width in max mode (fused_pick may widen a forced one)"""
    used = set()
    for seed in range(4):
        net = Net(ctx, "random_%d" % seed, *bnet.mixed_bn(seed), seed=seed)
        try:
            check_engines(net, net.ev[:257], True, used_lanes=used)
        finally:
            net.close()
    assert used >= {8, 16, 32, 128}, used


def test_sliced_batch_odd_slices_ragged_tail(ctx):
    """K8 slices a batch: an odd slice size, three slices with a short last one, and slice + 1 (a last slice of one
    set); the argmax rows of every slice are strided by that slice's own size"""
    import torch
    from plan_emulator import describe
    net = Net(ctx, "sliced", *bnet.sliced_bn(), nsets=8)
    try:
        desc = describe(net.plan.h)
        R = sum(int(np.prod([c for _, c in st["scope"]], dtype=np.int64)) for st in desc["steps"] if st["elim"] >= 0)
        s = min(bnet.slice_of(desc, 1 << 30), (1 << 30) // R)
        n3 = 2 * s + s // 3
        assert s % 2 == 1 and s > 2, s
        assert net.plan.fused_info(2)[0] == 0          # one launch per bucket by default
        rng = random.Random(7)
        for nb in (s + 1, n3):
            ev = bnet.evidence_sets([net.cards[v] for v in net.observed], nb, seed=nb)
            vals = _vals(ev)
            bounds = {0, 1, s - 2, s - 1, s, nb - 1} | ({s + 1, 2 * s - 1, 2 * s, 2 * s + 1} if nb > 2 * s else set())
            sample = sorted(bounds | set(rng.sample(range(nb), 24)))
            want = net.refs(ev[sample])
            runs = []
            for rep in range(3):
                v, a, st, _ = _batch(net, vals, fused=rep == 0)
                assert st == 0
                _same((v[sample], a[:, sample]), want, "sliced nb=%d run %d" % (nb, rep + 1))
                runs.append((v, a))
            assert all(np.array_equal(r[0].view(np.uint64), runs[0][0].view(np.uint64)) and np.array_equal(r[1], runs[0][1])
                       for r in runs)
            with torch.cuda.stream(ctx.torch_stream):
                vals.copy_(torch.roll(vals, 1, 0))
            ctx.sync()
            v, a, st, _ = _batch(net, vals, fused=False)
            assert st == 0
            assert np.array_equal(v, np.roll(runs[0][0], 1)) and np.array_equal(a, np.roll(runs[0][1], 1, axis=1)), nb
    finally:
        net.close()


def _uniform_bn(seed=4):
    cards, scopes, _, observed = bnet.mixed_bn(seed)
    tables = [[1.0 / cards[sc[0]]] * int(np.prod([cards[v] for v in sc])) for sc in scopes]
    return cards, scopes, tables, observed


def test_ties_lowest_values_win(ctx):
    """uniform CPTs: every assignment of the free variables ties, each one takes value 0"""
    cards, scopes, tables, observed = _uniform_bn()
    net = Net(ctx, "uniform", cards, scopes, tables, observed, nsets=257, seed=3)
    try:
        for nb in (3, 257):
            v, a = check_engines(net, net.ev[:nb], True)
            free = [u for u in range(len(cards)) if u not in observed]
            assert (a[free] == 0).all()
            assert np.array_equal(a[observed], net.ev[:nb].T)
    finally:
        net.close()


def _zero_bn():
    """x1 = 1 is impossible whatever x0; x2 and x3 hang below"""
    cards = [3, 2, 3, 2]
    scopes = [[0], [1, 0], [2, 1], [3, 0, 2]]
    rng = random.Random(2)
    tables = [bnet._cpt(rng, cards, sc[0], sc[1:]) for sc in scopes]
    tables[1] = [1.0] * 3 + [0.0] * 3           # P(x1 | x0): child most significant
    return cards, scopes, tables, [1, 3]


def test_zero_probability_sets_in_a_batch(ctx):
    """sets whose evidence has probability 0 give value 0, as their single queries do, and x0 -- whose bucket holds the
    impossible entry, every product there is 0 -- takes its lowest value; their neighbours are unaffected"""
    cards, scopes, tables, observed = _zero_bn()
    net = Net(ctx, "zero", cards, scopes, tables, observed, nsets=257, seed=1)
    try:
        for nb in (2, 3, 257):
            ev = net.ev[:nb].copy()
            ev[::2, 0] = 1
            ev[1::2, 0] = 0
            v, a = check_engines(net, ev, True)
            assert (v[::2] == 0).all() and (v[1::2] > 0).all()
            assert (a[0, ::2] == 0).all()
    finally:
        net.close()


def test_config5_sample_against_single_runs(ctx):
    """65 536 sets of config 5 through K9 (max mode) and K8, 512 of them against single runs"""
    from bnpp_b200 import synth
    N, W, K, seed, nobs = 500, 6, 3, 11, 20
    cards, scopes, tables = parse_uai(synth.random_bn_uai(N, W, K, seed))
    evs = synth.evidence_batch(N, nobs, 1 << 16, seed=5, fixed_ids=True)
    observed = sorted(evs[0])
    net = Net(ctx, "config5", cards, scopes, tables, observed, nsets=2)
    try:
        ev = np.array([[e[v] for v in observed] for e in evs], dtype=np.uint8)
        sample = sorted(random.Random(5).sample(range(ev.shape[0]), 512))
        want = net.refs(ev[sample])
        vals = _vals(ev)
        v, a, st, g = _batch(net, vals)
        assert st == 0 and g > 0
        _same((v[sample], a[:, sample]), want, "config 5 K9")
        vk, ak, st, _ = _batch(net, vals, fused=False)
        assert st == 0
        _same((vk[sample], ak[:, sample]), want, "config 5 K8")
        assert np.array_equal(v.view(np.uint64), vk.view(np.uint64)) and np.array_equal(a, ak)
    finally:
        net.close()


@pytest.mark.parametrize("fused", [True, False])
def test_out_of_range_evidence(ctx, fused):
    """an illegal value raises the status bit; that set equals its single run with the value read as 0, and reports 0"""
    net = Net(ctx, "edges", *bnet.edge_bn(), nsets=6, seed=6)
    try:
        assert [net.cards[v] for v in net.observed] == [2, 3, 2, bnet.BIG_CARD]
        bad = net.ev.copy()
        bad[3, 2] = 2
        v, a, st, g = _batch(net, _vals(bad), fused=fused)
        assert (g > 0) == fused
        assert st & BAD_EVIDENCE
        read_as = bad.copy()
        read_as[3, 2] = 0
        _same((v, a), net.refs(read_as), "illegal value 2 of a card-2 column (fused=%s)" % fused)
        assert a[net.observed[2], 3] == 0
    finally:
        net.close()


def test_api_errors(ctx):
    from bnpp_b200 import capi, model
    import torch
    cards, scopes, tables, observed = bnet.mixed_bn(1)
    net = Net(ctx, "errors", cards, scopes, tables, observed, nsets=4)
    L = ctx.L
    dev = torch.device("cuda:%d" % ctx.device)
    ev = _vals(net.ev)
    value = torch.empty(4, dtype=torch.float64, device=dev)
    assign = torch.empty((len(cards), 4), dtype=torch.uint8, device=dev)
    tp = (ctypes.c_void_p * len(net.bn.table_ptrs))(*net.bn.table_ptrs)

    def run(plan, nb=4, n_obs=len(observed), e=ev.data_ptr(), v=value.data_ptr(), a=assign.data_ptr()):
        return L.bnpp_mpe_plan_run_batched(plan.h, tp, nb, n_obs, ctypes.c_void_p(e), ctypes.c_void_p(v), ctypes.c_void_p(a))

    try:
        assert run(net.plan) == 0
        ctx.sync()
        assert run(net.plan, nb=0) == EINVAL
        assert run(net.plan, n_obs=len(observed) + 1) == EINVAL
        assert run(net.plan, e=None) == EINVAL
        assert run(net.plan, v=None) == EINVAL
        assert run(net.plan, a=None) == EINVAL
        pr = net.bn.plan(observed, net.order)         # a sum-product plan
        assert run(pr) == EINVAL
        with pytest.raises(capi.BnppError) as e:       # ... and the sum-product batch entry keeps refusing MPE plans
            net.plan.run_batched(net.bn.table_ptrs, 4, ev.data_ptr(), value.data_ptr())
        assert e.value.code == EINVAL
        net.plan.set_fused(True)                       # accepted: it selects the batch engine
        assert isinstance(net.plan, model.MPEPlan)
    finally:
        net.close()


def test_mpe_batch_host_values(ctx):
    """BN.mpe_batch from pinned host evidence equals BN.mpe set by set; the result buffers are reused per batch size"""
    import torch
    cards, scopes, tables, observed = bnet.mixed_bn(2)
    net = Net(ctx, "host", cards, scopes, tables, observed, nsets=33, seed=2)
    try:
        host = torch.from_numpy(np.ascontiguousarray(net.ev)).pin_memory()
        v, a = net.bn.mpe_batch(observed, None, "mf", host_values=host)
        ctx.sync()
        assert v.shape == (33,) and a.shape == (len(cards), 33) and a.dtype == torch.uint8
        _same((v.cpu().numpy(), a.cpu().numpy()), net.refs(net.ev), "host values")
        v2, a2 = net.bn.mpe_batch(observed, None, "mf", host_values=host)
        assert v2.data_ptr() == v.data_ptr() and a2.data_ptr() == a.data_ptr()
    finally:
        net.close()
