"""GPU parity tests proper: the CUDA path, called through the C ABI, against
(1) per-op dumps of the unmodified reference (tests/golden/ops_*.json.gz) and
(2) the CPU oracle on seeded inputs.  Values are BIT-EXACT (same multiplication and
summation order as the reference); partitions (tree-reduced on the GPU, sequential in
the reference) agree to 1e-12 relative."""
import math
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import oracle as orc  # noqa: E402

ZREL = 1e-12


@pytest.fixture(scope="module")
def ctx():
    import torch
    from bnpp_b200 import capi
    assert torch.cuda.is_available(), "GPU tests need a CUDA device; there is no CPU fallback"
    c = capi.Context(0)
    yield c
    c.close()


def dev(ctx, rec, cards):
    from bnpp_b200.factor import DeviceFactor
    return DeviceFactor.from_host(ctx, rec["scope"], [cards[v] for v in rec["scope"]], rec["values"], rec["partition"])


def zclose(a, b):
    return a == b or math.isclose(a, b, rel_tol=ZREL, abs_tol=1e-300)


def test_reference_op_dumps(ctx, golden_ops):
    """product / divide / sum_out / conditioning / normalize / max / min, code/factor.cpp:97-255"""
    for c in golden_ops:
        cards = c["cards"]
        a, b = dev(ctx, c["a"], cards), dev(ctx, c["b"], cards)
        p = a.product(b)
        assert p.scope == c["p"]["scope"]
        assert np.array_equal(p.values(), np.array(c["p"]["values"]))
        assert zclose(p.partition, c["p"]["partition"])
        q = a.divide(b)
        assert q.scope == c["q"]["scope"] and np.array_equal(q.values(), np.array(c["q"]["values"]))
        assert zclose(q.partition, c["q"]["partition"])
        assert ctx.status() == 0
        s = p.sum_out(c["sum_var"])
        assert s.scope == c["s"]["scope"] and np.array_equal(s.values(), np.array(c["s"]["values"]))
        assert zclose(s.partition, c["s"]["partition"])
        ev = {int(k): v for k, v in c["evidence"].items()}
        cf = p.condition(ev)
        assert cf.scope == c["c"]["scope"] and np.array_equal(cf.values(), np.array(c["c"]["values"]))
        assert zclose(cf.partition, c["c"]["partition"])
        # the reference normalises with ITS sequential partition; feed the same Z for a bit-exact check
        pref = dev(ctx, c["p"], cards)
        n = pref.normalize()
        assert np.array_equal(n.values(), np.array(c["n"]["values"])) and n.partition == 1.0
        assert pref.max() == c["max_p"] and pref.min() == c["min_p"]
        qref = dev(ctx, c["q"], cards)
        assert qref.max() == c["max_q"] and qref.min() == c["min_q"]


def test_zero_divisor_flag(ctx):
    from bnpp_b200.factor import DeviceFactor
    a = DeviceFactor.from_host(ctx, [0, 1], [2, 2], [1, 2, 3, 4])
    b = DeviceFactor.from_host(ctx, [1], [2], [0.0, 2.0])
    a.divide(b)
    assert ctx.status() & 1          # the reference asserts here (code/factor.cpp:169)
    assert ctx.status() == 0         # cleared


def rand_factor(ctx, rng, scope, cards):
    from bnpp_b200.factor import DeviceFactor
    n = int(np.prod([cards[v] for v in scope])) if scope else 1
    vals = np.random.default_rng(rng.randrange(1 << 30)).uniform(0.1, 1.0, n)
    of = orc.OFactor(scope, vals)
    return of, DeviceFactor.from_host(ctx, scope, [cards[v] for v in scope], vals, of.partition)


@pytest.mark.parametrize("binary", [True, False])
def test_fused_step_random(ctx, binary):
    """k-ary product -> sum_out in one kernel (code/model.cpp:414-418) on random scopes,
    random output axis orders, with and without an eliminated variable: bit-exact vs the oracle."""
    from bnpp_b200.factor import fused_product_sum_out
    rng = random.Random(7 if binary else 11)
    for case in range(120):
        nvars = rng.randint(1, 12 if binary else 7)
        cards = [2] * nvars if binary else [rng.choice([2, 2, 3, 4, 5]) for _ in range(nvars)]
        k = rng.randint(1, 6)
        ofs, dfs = [], []
        for _ in range(k):
            w = rng.randint(0, nvars)
            sc = rng.sample(range(nvars), w)
            o, d = rand_factor(ctx, rng, sc, cards)
            ofs.append(o); dfs.append(d)
        union = []
        for o in ofs:
            union += [v for v in o.scope if v not in union]
        elim = rng.choice(union) if union and rng.random() < 0.8 else None
        out_scope = [v for v in union if v != elim]
        rng.shuffle(out_scope)
        want = orc.product_sum_out(ofs, out_scope, elim, cards)
        got = fused_product_sum_out(ctx, dfs, out_scope, elim)
        assert np.array_equal(got.values(), want.values), (case, ctx.last_launch())
        assert zclose(got.partition, want.partition)


def headline_case(kind, nbits, k, reverse_b):
    """SURVEY §8d headline shapes at `nbits` union bits: returns (scopeA, scopeB, elim var)"""
    allv = list(range(nbits))
    if kind == "elem":
        a, b = allv, list(allv)
    elif kind == "bcast":
        a, b = allv[:-1], allv[1:]
    else:  # small: B over 10 scattered variables
        step = max(1, nbits // 10)
        a, b = allv, allv[::step][:10]
        if k not in b:
            b = sorted(set(b[:-1] + [k]))
    if reverse_b:
        b = b[::-1]
    return a, b, k


@pytest.mark.parametrize("kind", ["elem", "bcast", "small"])
@pytest.mark.parametrize("reverse_b", [False, True])
def test_headline_shapes_reduced(ctx, kind, reverse_b):
    """F-elem / F-bcast / F-small x sum-out position {leading, middle, trailing}, 2^20 union entries,
    entry-wise against the oracle"""
    from bnpp_b200.factor import fused_product_sum_out
    nbits = 20
    rng = random.Random(3)
    cards = [2] * nbits
    for k in (0, nbits // 2, nbits - 1):
        sa, sb, elim = headline_case(kind, nbits, k, reverse_b)
        if elim not in sa and elim not in sb:
            continue
        oa, da = rand_factor(ctx, rng, sa, cards)
        ob, db = rand_factor(ctx, rng, sb, cards)
        union = sa + [v for v in sb if v not in sa]
        out_scope = [v for v in union if v != elim]
        want = orc.product_sum_out([oa, ob], out_scope, elim, cards)
        got = fused_product_sum_out(ctx, [da, db], out_scope, elim)
        assert np.array_equal(got.values(), want.values), (kind, k, reverse_b, ctx.last_launch())
        assert zclose(got.partition, want.partition)


def test_mixed_cardinality_large(ctx):
    from bnpp_b200.factor import fused_product_sum_out
    rng = random.Random(5)
    cards = [3, 4, 5, 2, 3, 4, 2, 5, 3, 2, 4]      # 1.7M union entries
    sa = [0, 1, 2, 3, 4, 5, 6, 7]
    sb = [10, 9, 8, 7, 2, 0]
    oa, da = rand_factor(ctx, rng, sa, cards)
    ob, db = rand_factor(ctx, rng, sb, cards)
    for elim in (0, 7, 10, 2):
        union = sa + [v for v in sb if v not in sa]
        out_scope = [v for v in union if v != elim]
        want = orc.product_sum_out([oa, ob], out_scope, elim, cards)
        got = fused_product_sum_out(ctx, [da, db], out_scope, elim)
        assert np.array_equal(got.values(), want.values)
        assert zclose(got.partition, want.partition)


def test_edge_cases(ctx):
    """width-0 operands, size-1 outputs, variable not in scope, everything observed"""
    from bnpp_b200.factor import DeviceFactor
    s = DeviceFactor.from_host(ctx, [], [], [2.5])
    a = DeviceFactor.from_host(ctx, [4, 2], [3, 2], [1, 2, 3, 4, 5, 6])
    p = s.product(a)
    assert p.scope == [4, 2] and np.array_equal(p.values(), 2.5 * np.arange(1, 7)) and p.partition == 52.5
    p2 = a.product(s)
    assert np.array_equal(p2.values(), p.values())
    ss = s.product(s)
    assert ss.scope == [] and ss.values()[0] == 6.25 and ss.partition == 6.25
    c = a.sum_out(9)                       # not in scope: deep copy (code/factor.cpp:185-188)
    assert c.scope == [4, 2] and np.array_equal(c.values(), a.values()) and c.partition == a.partition
    t = a.sum_out(4).sum_out(2)
    assert t.scope == [] and t.values()[0] == 21.0 and t.partition == 21.0
    e = a.condition({4: 2, 2: 1, 7: 0})     # all observed -> width-0 scalar
    assert e.scope == [] and e.values()[0] == 6.0 and e.partition == 6.0
    e2 = a.condition({})
    assert np.array_equal(e2.values(), a.values())
    n = DeviceFactor.from_host(ctx, [1], [2], [0.0, 0.0]).normalize()
    assert np.all(np.isnan(n.values()))    # 0/0, true division as in code/factor.cpp:250


def test_errors(ctx):
    from bnpp_b200 import capi
    from bnpp_b200.factor import DeviceFactor
    a = DeviceFactor.from_host(ctx, [0, 1], [2, 2], [1, 2, 3, 4])
    out = DeviceFactor.empty(ctx, [0], [2])
    with pytest.raises(capi.BnppError) as ei:   # variable 1 neither kept nor eliminated
        ctx.product_sum_out([(a.ptr, a.scope, a.cards, None)], [0], [2], None, out.ptr)
    assert ei.value.code == -1
    with pytest.raises(capi.BnppError):          # cardinality mismatch
        ctx.product_sum_out([(a.ptr, a.scope, a.cards, None)], [0], [3], 1, out.ptr)


def test_sum_out_commutes_and_partition_invariant_2p26(ctx):
    """size-independent properties on a table too big to check entry-wise against the CPU oracle"""
    import torch
    from bnpp_b200.factor import DeviceFactor, fused_product_sum_out
    nbits = 26
    g = torch.Generator(device="cuda").manual_seed(1)
    scope = list(range(nbits))
    a = DeviceFactor.empty(ctx, scope, [2] * nbits)
    b = DeviceFactor.empty(ctx, scope[1:], [2] * (nbits - 1))
    a.buf[:-1] = torch.rand(a.size, generator=g, device="cuda", dtype=torch.float64) * 0.9 + 0.1
    b.buf[:-1] = torch.rand(b.size, generator=g, device="cuda", dtype=torch.float64) * 0.9 + 0.1
    torch.cuda.synchronize()
    zs = []
    for k in (0, 13, 25):
        out = fused_product_sum_out(ctx, [a, b], [v for v in scope if v != k], k)
        zs.append(out.partition)
        assert zclose(out.sum(), out.partition)
    assert all(math.isclose(z, zs[0], rel_tol=1e-12) for z in zs)     # Z(sum_out) = Z(product), any variable
    want = float((a.buf[:-1].view(2, -1) * b.buf[:-1]).sum().item())
    assert math.isclose(zs[0], want, rel_tol=1e-11)
    s1 = a.sum_out(3).sum_out(20)
    s2 = a.sum_out(20).sum_out(3)
    assert torch.allclose(s1.buf[:-1], s2.buf[:-1], rtol=1e-14, atol=0.0)   # (p+q)+(r+s) vs (p+r)+(q+s)


def test_transposed_operands_through_shared_memory(ctx):
    """operands whose fastest axes are the output's slowest go through the shared-memory tile
    (`staged` variant): pure products and fused steps, K = 1..3, entry-wise against the oracle"""
    from bnpp_b200.factor import fused_product_sum_out
    rng = random.Random(21)
    nbits = 18
    cards = [2] * nbits
    allv = list(range(nbits))
    seen = set()
    cases = [
        ([allv[::-1]], None),                                   # K=1: a full bit-reversal copy
        ([allv, allv[::-1]], None),                             # product, B reversed
        ([allv, allv[::-1]], 7),                                # fused, B reversed
        ([allv[:-1], allv[::-1], [3, 9]], 17),                  # K=3, the big reversed one in the middle
        ([allv[::-1], allv[2:]], 0),                            # the reversed operand first
    ]
    from bnpp_b200 import capi
    # operands whose contiguous runs inside a tile are short (8 doubles) or cut by the eliminated variable
    mixed = allv[9:] + allv[:9]
    cases += [
        ([allv, mixed[::-1]], 4),
        ([allv[6:] + allv[:6], allv], 12),
        ([allv[3:][::-1] + allv[:3], allv], None),
        ([allv[:17], allv[::-1]], 3),                           # A lacks the innermost output axis: scalar loads along x
        ([allv[::-1], allv[1:17] + [0]], 0),                    # ... and x is its stride-1 axis
        ([allv[:17], allv[::-1], allv[5:]], 2),                 # K=3: two riders with different micro-tiles
        ([allv[::-1], [17, 4, 11]], None),                      # a small table whose fastest axis is not the output's
    ]
    try:
        for scopes, elim in cases:
            ofs, dfs = [], []
            for sc in scopes:
                o, d = rand_factor(ctx, rng, sc, cards)
                ofs.append(o); dfs.append(d)
            out_scope = [v for v in allv if v != elim]
            want = orc.product_sum_out(ofs, out_scope, elim, cards)
            for tma, rider in ((1, 1), (1, 0), (0, 0)):     # tile by TMA bulk copies (other operands prefetched or not) / cp.async
                capi.tuning_set("staged_tma", tma)
                capi.tuning_set("staged_async", rider)
                got = fused_product_sum_out(ctx, dfs, out_scope, elim)
                seen.add(ctx.last_launch()[0].split(",")[0])
                assert np.array_equal(got.values(), want.values), (scopes, elim, tma, rider, ctx.last_launch())
                assert zclose(got.partition, want.partition)
    finally:
        capi.tuning_set("staged_tma", 1)
        capi.tuning_set("staged_async", 1)
    # LDGSTS tiles, the transposed operand alone by TMA, and other operands riding along
    variants = {s.split("<")[1] for s in seen}
    assert any(v.startswith("staged") for v in variants), variants
    assert any(v.startswith("tma/") and len(v) == 5 for v in variants), variants
    assert any(v.startswith("tma/") and len(v) >= 6 for v in variants), variants


def test_transposed_operands_many_chunks_per_cta(ctx):
    """the staged kernels as persistent loops: 2^22 output entries = 2048 chunks over ~300 CTAs, so every CTA walks
    several chunks -- the stage ring wraps, the mbarrier parities flip, the chunk bases of later chunks are used -- in
    the TMA variant with the other operand riding along (F-bcast shape: B reversed and without x0, A without the
    innermost axis), with the transposed operand alone, and in the element-wise variant; entry-wise against the oracle"""
    from bnpp_b200 import capi
    from bnpp_b200.factor import fused_product_sum_out
    rng = random.Random(33)
    nbits = 23
    cards = [2] * nbits
    allv = list(range(nbits))
    cases = [
        ([allv[:-1], allv[1:][::-1]], 0),                       # F-bcast, leading variable summed out
        ([allv[:-1], allv[1:][::-1]], 11),                      # ... a middle one (both operands hold it)
        ([allv[:-1], allv[1:][::-1]], nbits - 1),               # ... the trailing one
        ([allv, allv[::-1]], 11),                               # F-elem reversed
        ([allv[::-1]], None),                                   # K = 1: a full bit-reversal copy
    ]
    seen = set()
    try:
        for scopes, elim in cases:
            ofs, dfs = [], []
            for sc in scopes:
                o, d = rand_factor(ctx, rng, sc, cards)
                ofs.append(o); dfs.append(d)
            out_scope = [v for v in allv if v != elim]
            want = orc.product_sum_out(ofs, out_scope, elim, cards)
            for tma, rider in ((1, 1), (1, 0), (0, 0)):
                capi.tuning_set("staged_tma", tma)
                capi.tuning_set("staged_async", rider)
                got = fused_product_sum_out(ctx, dfs, out_scope, elim)
                name, grid, _ = ctx.last_launch()
                seen.add(name.split(",")[0].split("<")[1])
                assert grid * 2 < (1 << (len(out_scope) - 1)) // 1024, (name, grid)        # more than two chunks per CTA
                assert np.array_equal(got.values(), want.values), (scopes, elim, tma, rider, name)
                assert zclose(got.partition, want.partition)
                del got
            del ofs, dfs, want
    finally:
        capi.tuning_set("staged_tma", 1)
        capi.tuning_set("staged_async", 1)
    assert any(v.startswith("staged") for v in seen) and any(v.startswith("tma/") and len(v) >= 6 for v in seen), seen


def test_bcast_2p30_partition_invariant(ctx):
    """largest single-GPU shapes: 2^30 union entries (4 GiB operands); Z(sum_out) must not depend on
    which variable is summed out, and must equal the direct reduction of a product slice"""
    import torch
    from bnpp_b200.factor import DeviceFactor, fused_product_sum_out
    nbits = 30
    g = torch.Generator(device="cuda").manual_seed(3)
    a = DeviceFactor.empty(ctx, list(range(nbits - 1)), [2] * (nbits - 1))
    b = DeviceFactor.empty(ctx, list(range(1, nbits)), [2] * (nbits - 1))
    a.buf[:-1] = torch.rand(a.size, generator=g, device="cuda", dtype=torch.float64) * 0.9 + 0.1
    b.buf[:-1] = torch.rand(b.size, generator=g, device="cuda", dtype=torch.float64) * 0.9 + 0.1
    torch.cuda.synchronize()
    zs = []
    for k in (0, 15, 29):
        out = fused_product_sum_out(ctx, [a, b], [v for v in range(nbits) if v != k], k)
        zs.append(out.partition)
        del out
    assert all(math.isclose(z, zs[0], rel_tol=1e-12) for z in zs)
    # Z = sum_{x0} sum_{x29} sum_rest A[x0,rest] B[rest,x29] = <sum_x0 A, sum_x29 B>
    sa = a.buf[:-1].view(2, -1).sum(0)
    sb = b.buf[:-1].view(-1, 2).sum(1)
    want = float(torch.dot(sa, sb).item())
    assert math.isclose(zs[0], want, rel_tol=1e-11)


def test_too_big_and_too_many_operands(ctx):
    """limits are refused with the documented codes before anything is launched or allocated"""
    from bnpp_b200 import capi
    fake = 0x10000000          # never dereferenced: planning fails first
    wide = list(range(33))
    with pytest.raises(capi.BnppError) as e:      # 2^33-entry output: the reference's `unsigned` sizes cannot hold it either
        ctx.product_sum_out([(fake, wide, [2] * 33, None)], wide, [2] * 33, None, fake)
    assert e.value.code == -4
    ops = [(fake, [0], [2], None)] * 7
    with pytest.raises(capi.BnppError) as e:      # more than BNPP_MAX_OPERANDS tables in one launch
        ctx.product_sum_out(ops, [0], [2], None, fake)
    assert e.value.code == -3
    with pytest.raises(capi.BnppError) as e:      # divide needs exactly two operands
        ctx.product_sum_out(ops[:3], [0], [2], None, fake, divide=True)
    assert e.value.code == -1
