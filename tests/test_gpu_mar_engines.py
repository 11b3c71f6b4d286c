"""All-marginals plans (bnpp_mar_plan_create: two passes over the bucket tree, every marginal in one run) on every
engine that runs them, against plain references of P(v | e) (tests/mar_reference.py).

Single runs: the first run of a plan with one launch per bucket is checked against the reference; every other engine
must give the same bits -- the one-launch kernel (K9, `ve_fused`), the task engine (K10, `ve_tasks`, which cuts the
plan's DAG into tasks: in the downward pass one product feeds several later steps), the replayed CUDA graph after the
evidence values changed, and the dynamic path that plans every step at run time (tables not 32-byte aligned).

Batches (bnpp_ve_plan_run_batched, result [result_size][nb]): every set's column equals its single run bit for bit --
normalised, with NaN where P(e) = 0 and 1.0 in one-entry slices -- and, with normalisation off, the single run's
unnormalised values in every slice of more than one entry.  Engines: K9 at every lane width it accepts, and K8 (one
launch per bucket) as first run, captured run and graph replay after the evidence changed in place.  Also: a
one-rank sharded run."""
import os
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import batch_networks as bnet  # noqa: E402
from fused_interp import parse_uai  # noqa: E402
from mar_reference import SLOW, oracle_marginals, slow_golden  # noqa: E402

GOLDEN = ["asia", "child", "alarm", "grid3x3", "network", "insurance", "win95pts", "hailfinder", "hepar2", "andes", "Water"]
RANDOM = ["random_%d" % s for s in range(bnet.N_RANDOM)]
NETWORKS = GOLDEN + RANDOM + ["many_parents", "edges", "unmentioned", "wide"]
BATCHES = (1, 2, 3, 257, 1027)
LANES = (2, 4, 8, 16, 32, 128)      # every width fused_valid_g accepts
REL, GOLDEN_REL = 1e-12, 1e-9
SENTINEL = -7.0                     # no marginal takes it: a slice a run should write and did not keeps it
BAD_EVIDENCE = 2                    # BNPP_STATUS_BAD_EVIDENCE

_refs = {}


@pytest.fixture(scope="module")
def ctx():
    from bnpp_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def stored():
    return slow_golden()


def _network(name, golden_models):
    """-> (cards, scopes, tables, single-run evidence cases, observed ids of the batches)"""
    if name in GOLDEN:
        m = golden_models[name]
        cards, scopes, tables = parse_uai(m["uai"])
        cases = []
        for c in m["pr"]:
            ev = {int(k): int(v) for k, v in c["evidence"].items()}
            if c["flag"] == "mf" and ev not in cases:
                cases.append(ev)
        observed = sorted(max(cases, key=len))
        if not observed:
            observed = sorted(random.Random(name).sample(range(len(cards)), 3))
        return cards, scopes, tables, cases, observed
    if name == "wide":
        from bnpp_b200 import synth
        cards, scopes, tables = parse_uai(synth.random_bn_uai(40, 24, 3, 3))      # min-fill width 15: streaming kernels
        return cards, scopes, tables, [{}, {5: 1, 17: 0, 33: 1}], [5, 17, 33]
    cards, scopes, tables, observed = bnet.unmentioned_bn() if name == "unmentioned" else bnet.network(name, None)
    row = bnet.evidence_sets([cards[v] for v in observed], 2, 3)[1]
    return cards, scopes, tables, [{}, {v: int(x) for v, x in zip(observed, row)}], observed


def _reference(name, cards, scopes, tables, ev, stored):
    key = (name, tuple(sorted(ev.items())))
    if key not in _refs:
        if name in SLOW:
            _refs[key] = next(m for e, m in stored[name] if e == ev)
        else:
            _refs[key] = oracle_marginals(cards, scopes, tables, ev)
    return _refs[key]


class Net:
    """a network on the device and the fresh marginals plans made for it (closed with it)"""

    def __init__(self, ctx, cards, scopes, tables, observed):
        from bnpp_b200 import model
        self.ctx, self.cards, self.scopes, self.tables = ctx, cards, scopes, tables
        self.bn = model.BN(ctx, cards, list(zip(scopes, tables)))
        self.observed = list(observed)
        self.order = bnet.mf_order(cards, scopes, self.observed)
        self._plans = []

    def plan(self, observed=None, fused=True, segments=None, cut=0):
        """a FRESH marginals plan (tasks can only be cut before a plan's first run)"""
        from bnpp_b200 import model
        obs = self.observed if observed is None else sorted(observed)
        order = self.order if observed is None else bnet.mf_order(self.cards, self.scopes, obs)
        p = model.MarPlan(self.ctx, self.cards, self.scopes, obs, order)
        p.set_fused(fused)
        if segments is not None:
            p.set_segments(segments, cut)
        self._plans.append(p)
        return p

    def close(self):
        for p in self._plans:
            p.close()
        self.bn.close()


def _set_normalize(p, on):
    p.ctx.check(p.ctx.L.bnpp_ve_plan_set_normalize(p.h, int(on)))


def _device(ctx, a, dtype=None):
    import torch
    with torch.cuda.stream(ctx.torch_stream):
        t = torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).to("cuda:%d" % ctx.device)
    ctx.sync()
    return t


def _single(p, ptrs, ev):
    """one run of a plan -> (result, launches)"""
    import torch
    ctx = p.ctx
    with torch.cuda.stream(ctx.torch_stream):
        res = torch.full((max(1, p.result_size),), SENTINEL, dtype=torch.float64, device="cuda:%d" % ctx.device)
    ctx.sync()
    l0 = ctx.launches
    p.run(ptrs, [ev[v] for v in p.observed], res.data_ptr(), None)
    ctx.sync()
    return res.cpu().numpy(), ctx.launches - l0


def _same(got, want, what, rows=None):
    g, w = got.view(np.uint64), want.view(np.uint64)
    if rows is not None:
        g, w = g[rows], w[rows]
    bad = np.argwhere(g != w)
    if bad.size:
        i = tuple(bad[0])
        pytest.fail("%s: %d entries differ, first %s: %r != %r" % (what, len(bad), i, got[rows][i] if rows is not None else got[i],
                                                                   want[rows][i] if rows is not None else want[i]))


def _check_reference(res, p, want, golden_mar, what):
    for v in range(len(p.off)):
        seg = res[p.off[v]:p.off[v] + p.size[v]]
        if v not in want:
            assert p.size[v] == 1 and seg[0] == 1.0, (what, v, seg)
            continue
        assert np.all(np.abs(seg - want[v]) <= REL * np.abs(want[v])), (what, v, seg, want[v])
        if golden_mar is not None:
            assert np.allclose(seg, golden_mar[v], rtol=GOLDEN_REL, atol=0.0), (what, v, seg, golden_mar[v])


@pytest.mark.parametrize("name", NETWORKS)
def test_single_run_engines(ctx, golden_models, stored, name):
    """one launch per bucket == the reference; K9, K10 (tasks of at most 0 / 1 / 5 steps), graph replay with other
    evidence values in between, and the dynamic path == that first run, bit for bit"""
    import torch
    cards, scopes, tables, cases, _ = _network(name, golden_models)
    net = Net(ctx, cards, scopes, tables, [])
    ptrs = net.bn.table_ptrs
    try:
        # tables one double past a 32-byte boundary: the dynamic path
        offs, total = [], 0
        for t in tables:
            offs.append(total + 1)
            total += (len(t) + 1 + 3) // 4 * 4
        host = np.zeros(total)
        for t, o in zip(tables, offs):
            host[o:o + len(t)] = t
        dev = _device(ctx, host)
        unaligned = [dev.data_ptr() + 8 * o for o in offs]
        for ev in cases:
            what = "%s ev=%s" % (name, ev)
            p = net.plan(ev, fused=False, segments=False)
            base, per_bucket = _single(p, ptrs, ev)
            gm = golden_models[name]["mar"] if name in GOLDEN else []
            golden_mar = next((c["mar"] for c in gm if {int(k): v for k, v in c["evidence"].items()} == ev), None)
            _check_reference(base, p, _reference(name, cards, scopes, tables, ev, stored), golden_mar, what)

            p = net.plan(ev)
            if p.fused_info(1)[0] > 0:
                _same(_single(p, ptrs, ev)[0], base, what + " K9")
            for cut in (0, 1, 5):
                got, launches = _single(net.plan(ev, fused=False, segments=True, cut=cut), ptrs, ev)
                _same(got, base, what + " K10 cut=%d" % cut)
                if cut == 0:
                    assert launches < per_bucket, (what, launches, per_bucket)
            # runs 2 and 3 replay the plan's graph; run 2 with other evidence values
            other = {v: (x + 1) % cards[v] for v, x in ev.items()}
            base_other = _single(net.plan(ev, fused=False, segments=False), ptrs, other)[0]
            for segments in (False, True):
                p = net.plan(ev, fused=False, segments=segments)
                for run, e, want in [(1, ev, base), (2, other, base_other), (3, ev, base)]:
                    _same(_single(p, ptrs, e)[0], want, what + " segments=%s run %d" % (segments, run))
            _same(_single(net.plan(ev, fused=False), unaligned, ev)[0], base, what + " dynamic path")
        del dev
        torch.cuda.synchronize()
    finally:
        net.close()


class Batch:
    """the batch plan of a network, its single-run plan and the single runs of the evidence rows seen so far"""

    def __init__(self, ctx, net, nsets=max(BATCHES), seed=0):
        self.ctx, self.net = ctx, net
        self.bplan = net.plan()
        self.splan = net.plan()
        self.ev = bnet.evidence_sets([net.cards[v] for v in net.observed], nsets, seed)
        self._ref = {}
        self.out = {}

    def singles(self, rows, normalize):
        """-> [result_size][len(rows)] of single runs of the single-run plan"""
        import torch
        todo = []
        for r in rows:
            k = (bytes(np.asarray(r, dtype=np.uint8)), normalize)
            if k not in self._ref and k not in todo:
                todo.append(k)
        if todo:
            p, n = self.splan, max(1, self.splan.result_size)
            _set_normalize(p, normalize)
            with torch.cuda.stream(self.ctx.torch_stream):
                buf = torch.full((len(todo), n), SENTINEL, dtype=torch.float64, device="cuda:%d" % self.ctx.device)
            for i, (k, _) in enumerate(todo):
                p.run(self.net.bn.table_ptrs, list(k), buf[i].data_ptr(), None)
            self.ctx.sync()
            _set_normalize(p, True)
            host = buf.cpu().numpy()
            for i, k in enumerate(todo):
                self._ref[k] = host[i]
        return np.stack([self._ref[(bytes(np.asarray(r, dtype=np.uint8)), normalize)] for r in rows], axis=1)

    def run(self, vals, fused, lanes=None, normalize=True):
        """one batched run into the batch's result buffer (same pointer for every run of nb sets) -> (result
        [result_size][nb], status bits, lanes per set (0: K8), launches)"""
        import torch
        nb = vals.shape[0]
        p = self.bplan
        out = self.out.get(nb)
        if out is None:
            with torch.cuda.stream(self.ctx.torch_stream):
                out = self.out[nb] = torch.empty((max(1, p.result_size), nb), dtype=torch.float64, device=vals.device)
        with torch.cuda.stream(self.ctx.torch_stream):
            out.fill_(SENTINEL)
        self.ctx.sync()
        self.ctx.status()           # clear
        p.set_fused(fused)
        _set_normalize(p, normalize)
        if lanes:
            os.environ["BNPP_FUSED_G"] = str(lanes)
        try:
            g = p.fused_info(nb)[0] if fused and nb > 1 else 0
            l0 = self.ctx.launches
            p.run_batched(self.net.bn.table_ptrs, nb, vals.data_ptr(), out.data_ptr())
            self.ctx.sync()
            return out.cpu().numpy().copy(), self.ctx.status(), g, self.ctx.launches - l0
        finally:
            os.environ.pop("BNPP_FUSED_G", None)
            p.set_fused(True)
            _set_normalize(p, True)

    def check(self, got, rows, normalize, what):
        want = self.singles(rows, normalize)
        multi = None if normalize else np.repeat(np.array(self.bplan.size) > 1, self.bplan.size)
        _same(got, want, what, rows=multi)


def check_batch(b, ev, engine, name=""):
    """one engine ("k9": the default, then every lane width; "k8": first, captured and replayed run) in both
    normalisation modes on one batch against the single runs of its sets"""
    import torch
    nb = ev.shape[0]
    vals = _device(b.ctx, ev, torch.uint8)
    for normalize in (True, False):
        tag = "%s nb=%d normalize=%d" % (name, nb, normalize)
        if engine == "k9":
            got, st, g, _ = b.run(vals, True, normalize=normalize)
            assert st == 0 and g > 0, (tag, st, g)
            b.check(got, ev, normalize, tag + " K9 default (lanes %d)" % g)
            for lanes in LANES:
                got, st, gl, _ = b.run(vals, True, lanes=lanes, normalize=normalize)
                assert st == 0
                b.check(got, ev, normalize, tag + " BNPP_FUSED_G=%d (lanes %d)" % (lanes, gl))
            continue
        # K8: plain run, captured run, then the replayed graph after the evidence changed in place
        counts = []
        for rep in range(2):
            got, st, _, n = b.run(vals, False, normalize=normalize)
            assert st == 0
            b.check(got, ev, normalize, tag + " K8 run %d" % (rep + 1))
            counts.append(n)
        new = np.roll(ev, 1, axis=0) if nb > 1 else next((r for r in b.ev if not np.array_equal(r, ev[0])), ev[0])[None]
        with torch.cuda.stream(b.ctx.torch_stream):
            vals.copy_(_device(b.ctx, new, torch.uint8))
        b.ctx.sync()
        got, st, _, n = b.run(vals, False, normalize=normalize)
        assert st == 0
        b.check(got, new, normalize, tag + " K8 replay")
        counts.append(n)
        if ev.shape[1] and name != "many_parents":      # many_parents: extra launches for its evidence digits
            assert counts[2] == counts[0], (tag, "launches of the plain and the replayed run", counts)
        with torch.cuda.stream(b.ctx.torch_stream):
            vals.copy_(_device(b.ctx, ev, torch.uint8))
        b.ctx.sync()


K9_BATCH = [n for n in NETWORKS if n not in ("insurance", "win95pts", "hailfinder", "andes", "Water", "wide")]


@pytest.mark.parametrize("name", K9_BATCH)
def test_batched_marginals_k9(ctx, golden_models, name):
    """batches of 2, 3, 257 and 1027 sets through K9 (one launch for the batch), default and every lane width: every
    set's column equals its single run, normalised and not"""
    cards, scopes, tables, _, observed = _network(name, golden_models)
    net = Net(ctx, cards, scopes, tables, observed)
    try:
        b = Batch(ctx, net)
        for nb in BATCHES[1:]:          # a batch of one set runs K8
            check_batch(b, b.ev[:nb], "k9", name)
    finally:
        net.close()


@pytest.mark.parametrize("name", NETWORKS)
def test_batched_marginals_k8(ctx, golden_models, name):
    """batches of 1, 2, 3, 257 and 1027 sets through K8 (one launch per bucket for the batch): first run, captured run,
    replay after the evidence changed in place; every set's column equals its single run, normalised and not"""
    cards, scopes, tables, _, observed = _network(name, golden_models)
    net = Net(ctx, cards, scopes, tables, observed)
    try:
        b = Batch(ctx, net)
        for nb in BATCHES:
            check_batch(b, b.ev[:nb], "k8", name)
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


def test_zero_probability_sets(ctx):
    """sets whose evidence has probability 0: NaN in every slice of more than one entry, as 0/0 in their single runs,
    1.0 in the observed ones; the sets around them are unaffected"""
    import torch
    cards, scopes, tables, observed = _zero_bn()
    net = Net(ctx, cards, scopes, tables, observed)
    try:
        b = Batch(ctx, net, nsets=257, seed=1)
        for nb in (2, 3, 257):
            ev = b.ev[:nb].copy()
            ev[::2, 0] = 1
            ev[1::2, 0] = 0
            check_batch(b, ev, "k9", "zero")
            check_batch(b, ev, "k8", "zero")
            got = b.run(_device(ctx, ev, torch.uint8), True)[0]
            multi = np.repeat(np.array(b.bplan.size) > 1, b.bplan.size)
            assert np.isnan(got[multi][:, ::2]).all() and not np.isnan(got[:, 1::2]).any()
            assert (got[~multi] == 1.0).all()
    finally:
        net.close()


@pytest.mark.parametrize("fused", [True, False])
def test_out_of_range_evidence(ctx, fused):
    """value 2 in a card-2 column is read as 0 and raises BNPP_STATUS_BAD_EVIDENCE; the set's column is the single run
    of value 0, every other set unaffected"""
    import torch
    net = Net(ctx, *bnet.edge_bn())
    try:
        assert [net.cards[v] for v in net.observed] == [2, 3, 2, bnet.BIG_CARD]
        b = Batch(ctx, net, nsets=6, seed=6)
        bad = b.ev.copy()
        bad[3, 2] = 2
        got, st, g, _ = b.run(_device(ctx, bad, torch.uint8), fused)
        assert (g > 0) == fused
        assert st & BAD_EVIDENCE
        read_as = bad.copy()
        read_as[3, 2] = 0
        b.check(got, read_as, True, "out-of-range value (fused=%s)" % fused)
    finally:
        net.close()


@pytest.mark.parametrize("fused", [True, False])
def test_unmentioned_variable(ctx, fused):
    """every byte 0..255 for the observed variable no factor mentions: 1.0 in its slice of every set, no flag"""
    import torch
    net = Net(ctx, *bnet.unmentioned_bn())
    try:
        b = Batch(ctx, net, nsets=256, seed=9)
        ev = b.ev.copy()
        ev[:, -1] = np.arange(256, dtype=np.uint8)
        got, st, g, _ = b.run(_device(ctx, ev, torch.uint8), fused)
        assert st == 0 and (g > 0) == fused
        last = len(net.cards) - 1
        assert b.bplan.size[last] == 1 and (got[b.bplan.off[last]] == 1.0).all()
        b.check(got, ev, True, "unmentioned (fused=%s)" % fused)
    finally:
        net.close()


@pytest.mark.parametrize("name", ["alarm", "hepar2", "wide"])
def test_sharded_single_rank(ctx, golden_models, name):
    """bnpp_ve_plan_run_sharded of a marginals plan over a one-rank communicator: the slices times this rank's
    partition, summed over the ranks, divided by the summed partitions -- the single run within 2 ulp"""
    import torch
    from bnpp_b200.nccl import ShardComm
    cards, scopes, tables, cases, _ = _network(name, golden_models)
    ev = max(cases, key=len)
    net = Net(ctx, cards, scopes, tables, [])
    comm = ShardComm(ctx, 0, 1)
    try:
        p = net.plan(ev)
        want = _single(p, net.bn.table_ptrs, ev)[0]
        z, _ = net.bn.partition(ev, "mf")
        n = p.result_size
        with torch.cuda.stream(ctx.torch_stream):
            res = torch.full((n + 1,), SENTINEL, dtype=torch.float64, device="cuda:%d" % ctx.device)
            res[n] = z
        comm.run_sharded(p, net.bn.table_ptrs, [ev[v] for v in p.observed], res.data_ptr(), res.data_ptr() + 8 * n)
        ctx.sync()
        got = res.cpu().numpy()[:n]
        assert np.all(np.abs(got - want) <= 2 * np.spacing(np.abs(want))), (name, np.max(np.abs(got - want) / np.spacing(np.abs(want))))
    finally:
        comm.close()
        net.close()
