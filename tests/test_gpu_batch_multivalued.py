"""Batched evidence (config 5) on multi-valued networks, through both batch engines: `ve_fused` (K9, the whole batch in
one launch, every lane width) and `contract_batched*` (K8, one launch per bucket: first run, captured run, and the
replayed graph after the evidence changed in place).

Every set of every batch of up to 1027 sets equals the per-set single query through the same plan bit for bit (the
same products in the same order), a seeded sample equals the CPU oracle's bucket elimination with the plan's order
(1e-12), and on the random networks an exhaustive float64 enumeration (`math.fsum` over every joint assignment, 1e-12).
The networks reach what binary networks cannot: eliminated variables of 3 to 19 values for every operand count K8's
generic kernel is instantiated for, evidence bytes above 15, odd and single-set batches (K8's one-set-per-thread
variants), a ragged last slice, a CPT with ten observed axes, an observed variable that no factor mentions, and
out-of-range values in the transposed (K8) and in-place (K9) evidence check."""
import math
import os
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import batch_networks as bnet  # noqa: E402
import oracle as orc  # noqa: E402

BATCHES = (1, 2, 3, 257, 1027)
LANES = (8, 16, 32, 128)
ORACLE_SAMPLE = 8
ENUM_SAMPLE = 48
REL = 1e-12
BAD_EVIDENCE = 2        # BNPP_STATUS_BAD_EVIDENCE


@pytest.fixture(scope="module")
def ctx():
    from bnpp_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


class Net:
    """a network on the device with one plan for its observed ids, and the per-set references of its evidence sets"""

    def __init__(self, ctx, name, cards, scopes, tables, observed, nsets=max(BATCHES), seed=0):
        from bnpp_b200 import model
        self.ctx, self.name, self.cards, self.observed = ctx, name, cards, list(observed)
        self.bn = model.BN(ctx, cards, list(zip(scopes, tables)))
        self.order = bnet.mf_order(cards, scopes, self.observed)
        assert self.bn.order([v for v in range(len(cards)) if v not in set(observed)], self.observed, "mf")[0] == self.order
        self.plan = self.bn.plan(self.observed, self.order)
        self.desc = bnet.dry_describe(cards, scopes, self.observed, self.order)
        self.omodel = orc.OModel("BAYES", cards, [orc.OFactor(sc, t) for sc, t in zip(scopes, tables)])
        self.joint = bnet.joint_table(cards, scopes, tables) if math.prod(cards) <= bnet.MAX_JOINT else None
        self.ev = bnet.evidence_sets([cards[v] for v in self.observed], nsets, seed)
        self._ref = {}

    def evidence(self, row):
        return {v: int(x) for v, x in zip(self.observed, row)}

    def single(self, row):
        key = bytes(np.asarray(row, dtype=np.uint8))
        if key not in self._ref:
            self._ref[key] = self.bn.partition(self.evidence(row), "mf")[0]
        return self._ref[key]

    def refs(self, rows):
        return np.array([self.single(r) for r in rows])

    def close(self):
        self.bn.close()


def _vals(ev):
    import torch
    t = torch.tensor(np.ascontiguousarray(ev), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    return t


def _batch(net, vals, fused=True, lanes=None):
    """-> (Z of every set, BNPP status bits of the run, lanes per set the run used (0: K8))"""
    net.ctx.status()            # clear
    net.plan.set_fused(fused)
    if lanes:
        os.environ["BNPP_FUSED_G"] = str(lanes)
    try:
        g = net.plan.fused_info(vals.shape[0])[0] if fused and vals.shape[0] > 1 else 0
        z = net.bn.partition_batch(net.observed, vals, "mf")
        net.ctx.sync()
        return z.cpu().numpy().copy(), net.ctx.status(), g
    finally:
        os.environ.pop("BNPP_FUSED_G", None)
        net.plan.set_fused(True)


def _same(got, want, what):
    bad = np.flatnonzero(got != want)
    if bad.size:
        i = bad[0]
        rel = float(np.max(np.abs(got[bad] - want[bad]) / np.abs(want[bad])))
        pytest.fail("%s: %d of %d sets differ from the per-set queries, first set %d: %r != %r, max rel %.3g"
                    % (what, bad.size, got.size, i, got[i], want[i], rel))


def check_engines(net, ev, expect_k9, used_lanes=None):
    """every engine on one batch against the per-set queries, bit for bit -> Z of the batch"""
    import torch
    nb = ev.shape[0]
    want = net.refs(ev)
    vals = _vals(ev)
    z, st, g = _batch(net, vals)
    assert st == 0, (net.name, nb, st)
    if nb > 1 and expect_k9:
        assert g > 0, (net.name, nb)
    _same(z, want, "%s nb=%d default (lanes %d)" % (net.name, nb, g))
    for lanes in LANES:
        zl, st, g = _batch(net, vals, lanes=lanes)
        assert st == 0
        if used_lanes is not None and g:
            used_lanes.add(g)
        _same(zl, want, "%s nb=%d BNPP_FUSED_G=%d (lanes %d)" % (net.name, nb, lanes, g))
    # K8: plain run, captured run, then the replayed graph after the evidence changed in place
    for rep in range(2):
        zk, st, _ = _batch(net, vals, fused=False)
        assert st == 0
        _same(zk, want, "%s nb=%d K8 run %d" % (net.name, nb, rep + 1))
    new = np.roll(ev, 1, axis=0) if nb > 1 else net.ev[1:2]        # other values for every set
    assert not np.array_equal(new, ev)
    with torch.cuda.stream(net.ctx.torch_stream):
        vals.copy_(torch.from_numpy(new).to(vals.device))
    net.ctx.sync()
    zk, st, _ = _batch(net, vals, fused=False)
    assert st == 0
    _same(zk, net.refs(new), "%s nb=%d K8 replay after new evidence" % (net.name, nb))
    return z


def check_references(net, ev, z, rng):
    """a sample of the batch against the oracle (plan's order) and, on small networks, against enumeration"""
    nb = ev.shape[0]
    for i in rng.sample(range(nb), min(nb, ORACLE_SAMPLE)):
        want = orc.partition(net.omodel, net.evidence(ev[i]), net.order)
        assert abs(z[i] - want) <= REL * abs(want), (net.name, i, z[i], want)
    if net.joint is not None:
        for i in sorted(set(rng.sample(range(nb), min(nb, ENUM_SAMPLE)) + [min(1, nb - 1)])):
            want = bnet.enumerate_z(net.joint, net.observed, ev[i])
            assert abs(z[i] - want) <= REL * abs(want), (net.name, i, z[i], want)


@pytest.mark.parametrize("name", bnet.NETWORKS)
def test_batch_equals_single_queries(ctx, golden_models, name):
    net = Net(ctx, name, *bnet.network(name, golden_models), seed=len(name))
    # K9 takes every batch of these networks but Water's, whose widest buckets run one launch each
    expect_k9 = name != "Water"
    if not expect_k9:
        assert net.plan.fused_info(2)[0] == 0
    rng = random.Random(name)
    try:
        for nb in BATCHES:
            ev = net.ev[:nb]
            z = check_engines(net, ev, expect_k9)
            check_references(net, ev, z, rng)
        if name == "many_parents":
            assert bnet.max_observed_axes(net.desc) > 8
    finally:
        net.close()


def test_every_lane_width_is_exercised(ctx):
    """BNPP_FUSED_G reaches every K9 group width on these networks (fused_pick may widen a forced one)"""
    used = set()
    for seed in range(4):
        net = Net(ctx, "random_%d" % seed, *bnet.mixed_bn(seed), seed=seed)
        try:
            check_engines(net, net.ev[:257], True, used_lanes=used)
        finally:
            net.close()
    assert used >= set(LANES), used


def test_sliced_batch_odd_slices_ragged_tail(ctx):
    """K8 slices a batch that would make an intermediate over ~1 GiB: odd slice size, a ragged last slice, three
    slices, and a batch of slice + 1 (a last slice of one set, misaligned in the result)"""
    import torch
    net = Net(ctx, "sliced", *bnet.sliced_bn(), nsets=8)
    try:
        s = bnet.slice_of(net.desc, 1 << 30)
        n3 = 2 * s + s // 3
        assert s % 2 == 1 and s > 2, s
        assert -(-n3 // s) >= 3 and n3 - 2 * s < s
        rng = random.Random(7)
        for nb in (s + 1, n3):
            assert bnet.slice_of(net.desc, nb) == s
            ev = bnet.evidence_sets([net.cards[v] for v in net.observed], nb, seed=nb)
            vals = _vals(ev)
            bounds = {0, 1, s - 2, s - 1, s, nb - 1} | ({s + 1, 2 * s - 1, 2 * s, 2 * s + 1} if nb > 2 * s else set())
            sample = sorted(bounds | set(rng.sample(range(nb), 24)))
            want = net.refs(ev[sample])
            z, st, _ = _batch(net, vals)
            assert st == 0
            _same(z[sample], want, "sliced nb=%d default" % nb)
            zk = []
            for rep in range(2):
                zr, st, _ = _batch(net, vals, fused=False)
                assert st == 0
                _same(zr[sample], want, "sliced nb=%d K8 run %d" % (nb, rep + 1))
                zk.append(zr)
            assert np.array_equal(zk[0], zk[1]) and np.array_equal(zk[0], z)
            with torch.cuda.stream(ctx.torch_stream):
                vals.copy_(torch.roll(vals, 1, 0))
            ctx.sync()
            zr, st, _ = _batch(net, vals, fused=False)
            assert st == 0
            assert np.array_equal(zr, np.roll(zk[0], 1)), "sliced nb=%d K8 replay after new evidence" % nb
            for i in rng.sample(sample, 4):
                want_o = orc.partition(net.omodel, net.evidence(ev[i]), net.order)
                assert abs(z[i] - want_o) <= REL * abs(want_o), (nb, i)
    finally:
        net.close()


@pytest.mark.parametrize("nb", [5, 6])
@pytest.mark.parametrize("fused", [True, False])
def test_evidence_range_per_column(ctx, nb, fused):
    """value 2 is legal for the card-3 column (no flag, its own Z) and illegal for a card-2 column: the flag is raised
    and that set's Z is the one of value 0, every other set unaffected; K9 checks the matrix in place, K8 transposed"""
    net = Net(ctx, "edges", *bnet.edge_bn(), nsets=nb, seed=nb)
    try:
        assert [net.cards[v] for v in net.observed] == [2, 3, 2, bnet.BIG_CARD]
        ev = net.ev.copy()
        ev[2, 1] = 2
        ev[2, 3] = bnet.BIG_CARD - 1
        z, st, g = _batch(net, _vals(ev), fused=fused)
        assert (g > 0) == fused
        assert st == 0, st
        _same(z, net.refs(ev), "legal value 2 of a card-3 column (fused=%s)" % fused)
        bad = ev.copy()
        bad[3, 2] = 2
        z, st, _ = _batch(net, _vals(bad), fused=fused)
        assert st & BAD_EVIDENCE
        read_as = bad.copy()
        read_as[3, 2] = 0
        _same(z, net.refs(read_as), "illegal value 2 of a card-2 column (fused=%s)" % fused)
    finally:
        net.close()


@pytest.mark.parametrize("fused", [True, False])
def test_observed_variable_no_factor_mentions(ctx, fused):
    """every byte 0..255 for the observed variable outside every scope: the Z of the rest, no flag"""
    cards, scopes, tables, observed = bnet.unmentioned_bn()
    net = Net(ctx, "unmentioned", cards, scopes, tables, observed, nsets=256, seed=9)
    try:
        ev = net.ev.copy()
        ev[:, -1] = np.arange(256, dtype=np.uint8)
        z, st, g = _batch(net, _vals(ev), fused=fused)
        assert (g > 0) == fused
        assert st == 0, st
        zero = ev.copy()
        zero[:, -1] = 0
        _same(z, net.refs(zero), "unmentioned variable (fused=%s)" % fused)
        rest = orc.OModel("BAYES", cards[:-1], net.omodel.factors)
        for i in (0, 17, 255):
            want = orc.partition(rest, {v: int(x) for v, x in zip(observed[:-1], ev[i, :-1])}, net.order)
            assert abs(z[i] - want) <= REL * abs(want), i
    finally:
        net.close()
