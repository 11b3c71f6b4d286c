"""MPE on the GPU: the max-product step (bnpp_product_max_out) bit for bit against the oracle, MPE plans
(bnpp_mpe_plan_*, BN.mpe) against the CPU emulation of the same plan on the first run, on the replay graph and
with other evidence, config 4, the edge cases of the semantics, and the `bn -mpe` / `mn mpe` CLIs."""
import math
import os
import random
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import mpe_oracle  # noqa: E402
import oracle as orc  # noqa: E402
from bnpp_b200 import capi, model, synth  # noqa: E402
from fused_interp import parse_uai  # noqa: E402
from mpe_emulator import DryMPEPlan, emulate  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "bnpp_b200", "bin")
SMALL = ["asia", "asia_positive", "cancer", "earthquake", "grid3x3"]


@pytest.fixture(scope="module")
def ctx():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device; there is no CPU fallback"
    c = capi.Context(0)
    yield c
    c.close()


# ---- the op -------------------------------------------------------------------------------------------------------
def _dev(ctx, values):
    import torch
    with torch.cuda.stream(ctx.torch_stream):
        t = torch.from_numpy(np.ascontiguousarray(values, dtype=np.float64)).to("cuda:%d" % ctx.device)
    return t


def _max_out(ctx, operands, out_scope, cards, elim):
    """operands: (OFactor as the kernel sees it, device tensor, element offset, strides or None) -> (values, argmax)"""
    import torch
    n = int(np.prod([cards[v] for v in out_scope], dtype=np.int64)) if out_scope else 1
    with torch.cuda.stream(ctx.torch_stream):
        out = torch.empty(max(1, n), dtype=torch.float64, device="cuda:%d" % ctx.device)
        arg = torch.empty(max(1, n), dtype=torch.uint8, device=out.device)
    ops = [(t.data_ptr() + 8 * off, f.scope, [cards[v] for v in f.scope], st) for f, t, off, st in operands]
    ctx.product_max_out(ops, out_scope, [cards[v] for v in out_scope], elim, out.data_ptr(), arg.data_ptr())
    ctx.sync()
    return out[:n].cpu().numpy(), arg[:n].cpu().numpy()


def _check_op(ctx, operands, out_scope, cards, elim, what):
    got, garg = _max_out(ctx, operands, out_scope, cards, elim)
    want, warg = mpe_oracle.product_max_out([o[0] for o in operands], out_scope, elim, cards)
    kernel = ctx.last_launch()[0]
    assert np.array_equal(got, want.values, equal_nan=True), (what, kernel)
    finite = ~np.isnan(want.values)
    assert np.array_equal(got[finite].view(np.uint64), want.values[finite].view(np.uint64)), (what, kernel)
    assert np.array_equal(garg, warg), (what, kernel)
    return kernel


def _rand_values(rng, n, ties, nan):
    v = rng.uniform(0.0, 1.0, n)
    if ties:
        v = np.round(v * 4) / 4                    # few distinct values: many ties
    if nan and n > 1:
        v[rng.integers(0, n)] = np.nan
    return v


def test_product_max_out_generic_random_layouts(ctx):
    """K = 1..6, cardinalities 2..7, operands in file order, some of them strided evidence views"""
    rng = np.random.default_rng(3)
    pyr = random.Random(3)
    kernels = set()
    for case in range(150):
        nvars = pyr.randint(1, 7)
        cards = [pyr.randint(2, 7) for _ in range(nvars)]
        elim = pyr.randrange(nvars)
        operands = []
        for _ in range(pyr.randint(1, 6)):
            sc = pyr.sample(range(nvars), pyr.randint(0, nvars))
            if elim not in sc and pyr.random() < 0.7:
                sc.insert(pyr.randrange(len(sc) + 1), elim)
            ties, nan = case % 3 == 0, case % 7 == 0
            if pyr.random() < 0.3:
                # a view of a table with one more (observed) axis, fixed at a value: base offset + strides
                obs_card, pos = pyr.randint(2, 4), pyr.randint(0, len(sc))
                full_cards = [cards[v] for v in sc[:pos]] + [obs_card] + [cards[v] for v in sc[pos:]]
                full = _rand_values(rng, int(np.prod(full_cards)), ties, nan).reshape(full_cards)
                val = pyr.randrange(obs_card)
                strides = [int(s) // 8 for s in full.strides]
                view = np.take(full, val, axis=pos)
                operands.append((orc.OFactor(sc, view.reshape(-1), 0.0), _dev(ctx, full.reshape(-1)), val * strides[pos],
                                 strides[:pos] + strides[pos + 1:]))
            else:
                vals = _rand_values(rng, int(np.prod([cards[v] for v in sc])) if sc else 1, ties, nan)
                operands.append((orc.OFactor(sc, vals, 0.0), _dev(ctx, vals), 0, None))
        union = []
        for f, _, _, _ in operands:
            union += [v for v in f.scope if v not in union]
        if elim not in union:
            continue
        out_scope = [v for v in union if v != elim]
        pyr.shuffle(out_scope)
        kernels.add(_check_op(ctx, operands, out_scope, cards, elim, case).split("<")[0])
    assert "contract_generic_max" in kernels, kernels


@pytest.mark.parametrize("k", [1, 2, 3])
def test_product_max_out_canonical_binary_layouts(ctx, k):
    """every operand with the eliminated variable as its stride-1 axis, the output's fastest axis next or absent:
    the layout VE plans give a wide bucket -- contract_canon_max"""
    rng = np.random.default_rng(10 + k)
    nout = 13
    cards = [2] * (nout + 1)
    elim = nout
    out_scope = list(range(nout))
    for case in range(6):
        operands = []
        for q in range(k):
            if q == 0:
                sc = out_scope + [elim]                                      # LC_V4: 32-byte loads
            else:
                keep = sorted(rng.choice(nout - 1, size=int(rng.integers(0, nout - 1)), replace=False).tolist())
                sc = keep + ([nout - 1] if case % 2 else []) + [elim]        # with or without the output's fastest axis
            vals = _rand_values(rng, 2 ** len(sc), case % 2 == 0, case == 3)
            operands.append((orc.OFactor(sc, vals, 0.0), _dev(ctx, vals), 0, None))
        kernel = _check_op(ctx, operands, out_scope, cards, elim, (k, case))
        assert kernel.startswith("contract_canon_max"), kernel


def test_product_max_out_errors(ctx):
    import torch
    t = torch.ones(600, dtype=torch.float64, device="cuda:%d" % ctx.device)
    a = torch.empty(600, dtype=torch.uint8, device=t.device)
    with pytest.raises(capi.BnppError) as e:
        ctx.product_max_out([(t.data_ptr(), [0, 1], [2, 2], None)], [0, 1], [2, 2], -1, t.data_ptr(), a.data_ptr())
    assert e.value.code == -1
    with pytest.raises(capi.BnppError) as e:       # 300 values do not fit the uint8 argmax
        ctx.product_max_out([(t.data_ptr(), [0, 1], [2, 300], None)], [0], [2], 1, t.data_ptr(), a.data_ptr())
    assert e.value.code == -1


def test_fused_product_max_out_helper(ctx):
    from bnpp_b200.factor import DeviceFactor, fused_product_max_out
    rng = np.random.default_rng(5)
    cards = [3, 2, 4]
    fs = [orc.OFactor([0, 1], rng.uniform(size=6), 0.0), orc.OFactor([2, 1], rng.uniform(size=8), 0.0)]
    dfs = [DeviceFactor.from_host(ctx, f.scope, [cards[v] for v in f.scope], f.values) for f in fs]
    out, arg = fused_product_max_out(ctx, dfs, [2, 0], 1)
    want, warg = mpe_oracle.product_max_out(fs, [2, 0], 1, cards)
    assert np.array_equal(out.values(), want.values) and np.array_equal(arg.cpu().numpy(), warg)


# ---- plans --------------------------------------------------------------------------------------------------------
def _order(bn, ev, flag):
    return bn.order([v for v in range(bn.nvars) if v not in ev], ev, flag or None)[0]


def _other(ev, cards):
    return {v: (x + 1) % cards[v] for v, x in ev.items()}


def _check_plan(bn, text, ev, flag, what):
    cards, scopes, tables = parse_uai(text)
    observed = sorted(ev)
    order = _order(bn, ev, flag)
    p = DryMPEPlan(cards, scopes, observed, order)
    assert p.rc == 0
    want = emulate(p.h, tables, observed, [ev[v] for v in observed], len(cards))
    other = _other(ev, cards)
    want_other = emulate(p.h, tables, observed, [other[v] for v in observed], len(cards))
    p.close()
    first = bn.mpe(ev, flag or None)
    assert first[0] == want[0] and first[1] == want[1], (what, flag, first[:2], want)
    if ev:
        got = bn.mpe(other, flag or None)                  # the same plan, other evidence values
        assert got[0] == want_other[0] and got[1] == want_other[1], (what, flag, "other evidence")
    for _ in range(2):                                     # replay graph with the first evidence again
        again = bn.mpe(ev, flag or None)
        assert again[:2] == first[:2], (what, flag, "replay")


def test_mpe_plans_golden_models_against_emulator(ctx, golden_models):
    n = 0
    for name, m in golden_models.items():
        _, bn = model.from_uai_text(ctx, m["uai"])
        cases = [(c["flag"], {int(k): v for k, v in c["evidence"].items()}) for c in m["pr"]]
        if name in SMALL:
            evs = []
            for _, ev in cases:
                if ev not in evs:
                    evs.append(ev)
            cases = [(f, ev) for ev in evs for f in ["", "mf", "wmf", "md"]]
        for flag, ev in cases:
            _check_plan(bn, m["uai"], ev, flag, name)
            n += 1
        bn.close()
    assert n >= 80


def test_mpe_width22_network_canon_and_generic_max(ctx):
    text = synth.random_bn_uai(50, 30, 4, 3)
    _, bn = model.from_uai_text(ctx, text)
    ev = {49: 1, 47: 0}
    _check_plan(bn, text, ev, "mf", "width-22")
    order, width = bn.order([v for v in range(bn.nvars) if v not in ev], ev, "mf")
    assert 20 <= width <= 23, width
    p = model.MPEPlan(ctx, bn.cards, bn.scopes, sorted(ev), order)
    import torch
    buf = torch.empty(2 + bn.nvars, dtype=torch.int32, device="cuda:%d" % ctx.device)
    p.set_profiling(True)
    p.run_mpe(bn.table_ptrs, [ev[v] for v in sorted(ev)], buf.data_ptr(), buf.data_ptr() + 8)
    kernels = [s["kernel"] for s in p.step_stats()]
    assert any(k.startswith("contract_canon_max") for k in kernels), kernels
    assert any(k.startswith("contract_generic_max") for k in kernels), kernels
    ctx.sync()
    host = buf.cpu().numpy()
    assert [int(x) for x in host[2:].view(np.uint32)] == bn.mpe(ev, "mf")[1]
    p.close()
    bn.close()


def test_mpe_unaligned_tables_take_the_dynamic_path(ctx, golden_models):
    """tables that are not 32-byte aligned: every step is planned at run time (run_dynamic), still max-product"""
    import torch
    for name, text, flag, ev in [("alarm", golden_models["alarm"]["uai"], "mf", {}),
                                 ("width-22", synth.random_bn_uai(50, 30, 4, 3), "mf", {49: 1, 47: 0})]:
        cards, scopes, tables = parse_uai(text)
        _, bn = model.from_uai_text(ctx, text)
        want = bn.mpe(ev, flag)
        offs, total = [], 0
        for t in tables:
            offs.append(total + 1)                     # one double past a 32-byte boundary
            total += (t.size + 1 + 3) // 4 * 4
        host = np.zeros(total)
        for t, o in zip(tables, offs):
            host[o:o + t.size] = t
        with torch.cuda.stream(ctx.torch_stream):
            dev = torch.from_numpy(host).to("cuda:%d" % ctx.device)
            buf = torch.zeros(2 + len(cards), dtype=torch.int32, device=dev.device)
        observed = sorted(ev)
        p = model.MPEPlan(ctx, cards, scopes, observed, _order(bn, ev, flag))
        for _ in range(2):
            p.run_mpe([dev.data_ptr() + 8 * o for o in offs], [ev[v] for v in observed], buf.data_ptr(), buf.data_ptr() + 8)
            ctx.sync()
            got = buf.cpu().numpy()
            assert float(got[:2].view(np.float64)[0]) == want[0], name
            assert [int(x) for x in got[2:].view(np.uint32)] == want[1], name
        p.close()
        bn.close()


def _cpt_product(cards, scopes, tables, a):
    p = 1.0
    for sc, t in zip(scopes, tables):
        p *= float(t[int(np.ravel_multi_index([a[v] for v in sc], [cards[v] for v in sc]))])
    return p


def test_mpe_config4(ctx):
    N, W, K, seed, ev = synth.wide_bn(1)
    text = synth.random_bn_uai(N, W, K, seed)
    cards, scopes, tables = parse_uai(text)
    _, bn = model.from_uai_text(ctx, text)
    value, a, _ = bn.mpe(ev, "mf")
    assert all(a[v] == x for v, x in ev.items())
    assert math.isclose(_cpt_product(cards, scopes, tables, a), value, rel_tol=1e-12)
    z, _ = bn.partition(ev, "mf")
    assert 0 < value <= z
    for v in range(N):
        if v in ev:
            continue
        b = list(a)
        b[v] ^= 1
        assert _cpt_product(cards, scopes, tables, b) <= value * (1 + 1e-12), v
    again = bn.mpe(ev, "mf")
    assert again[:2] == (value, a)
    bn.close()


# ---- edge cases ---------------------------------------------------------------------------------------------------
def _bn(ctx, cards, factors):
    return model.BN(ctx, cards, [(sc, np.asarray(v, dtype=np.float64)) for sc, v in factors])


def test_mpe_edge_cases(ctx):
    # uniform CPTs: every assignment ties, the lowest values win
    bn = _bn(ctx, [3, 2, 4], [([0], [1 / 3] * 3), ([1, 0], [0.5] * 6), ([2, 1], [0.25] * 8)])
    for flag in [None, "mf"]:
        value, a, _ = bn.mpe({}, flag)
        assert a == [0, 0, 0] and math.isclose(value, 1 / 3 * 0.5 * 0.25, rel_tol=1e-15)
    # zero-probability evidence: value 0, not an error
    value, a, _ = bn.mpe({0: 1}, None)
    assert value > 0
    bn.close()
    bn = _bn(ctx, [2, 2], [([0], [0.4, 0.6]), ([1, 0], [1.0, 1.0, 0.0, 0.0])])   # P(x1 = 1 | x0) = 0
    value, a, _ = bn.mpe({1: 1}, None)
    assert value == 0.0 and a == [0, 1]
    # an evidence value out of range
    with pytest.raises(capi.BnppError):
        bn.mpe({1: 2}, None)
    # all variables observed: the product of the evidence entries
    value, a, _ = bn.mpe({0: 1, 1: 0}, None)
    assert value == 0.6 * 1.0 and a == [1, 0]
    # the sum-product run entry points refuse an MPE plan
    p = model.MPEPlan(ctx, bn.cards, bn.scopes, [], [0, 1])
    import torch
    buf = torch.empty(4, dtype=torch.float64, device="cuda:%d" % ctx.device)
    with pytest.raises(capi.BnppError) as e:
        p.run(bn.table_ptrs, [], buf.data_ptr(), buf.data_ptr() + 8)
    assert e.value.code == -1
    with pytest.raises(capi.BnppError) as e:
        p.run_batched(bn.table_ptrs, 2, buf.data_ptr(), buf.data_ptr())
    assert e.value.code == -1
    p.close()
    bn.close()


# ---- CLIs ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def files(tmp_path_factory, golden_models):
    d = tmp_path_factory.mktemp("uai_mpe")
    out = {}
    for name in ["asia", "grid3x3"]:
        p = d / (name + ".uai")
        p.write_text(golden_models[name]["uai"])
        out[name] = str(p)
    out["dir"] = d
    return out


def test_bn_cli_mpe(files, golden_models):
    evid = files["dir"] / "asia.uai.evid"
    evid.write_text("1\n2 0 1 2 1")
    om = orc.parse_uai(golden_models["asia"]["uai"])
    want, want_a, _ = mpe_oracle.mpe_brute_force(om, {0: 1, 2: 1})
    for extra in [[], ["-mf"]]:
        p = subprocess.run([os.path.join(BIN, "bn"), files["asia"], str(evid), "-mpe"] + extra, capture_output=True,
                           text=True, timeout=300)
        assert p.returncode == 0, p.stderr
        lines = p.stdout.splitlines()
        assert lines[0].startswith(">> MPE = ") and lines[1].startswith(">> Assignment = ")
        assert lines[2].startswith(">> Executed in ") and lines[3] == ""
        assert math.isclose(float(lines[0].split("=")[1]), want, rel_tol=1e-5)
        assert [int(x) for x in lines[1].split("=")[1].split()] == want_a


def test_mn_cli_mpe_writes_solution_file(files, golden_models):
    g = golden_models["grid3x3"]
    gev = files["dir"] / "g.evid"
    gev.write_text(g["shipped"]["PR_evid"])
    prefix = str(files["dir"] / "g")
    p = subprocess.run([os.path.join(BIN, "mn"), files["grid3x3"], str(gev), "-ve", "-mf", "-o", prefix],
                       input="mpe\nquit\n", capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    ev = orc.parse_evidence(g["shipped"]["PR_evid"])
    want, want_a, _ = mpe_oracle.mpe_brute_force(orc.parse_uai(g["uai"]), ev)
    assert "MPE = " in p.stdout and "Assignment = " + " ".join(map(str, want_a)) in p.stdout
    mpe_line = [ln for ln in p.stdout.splitlines() if "MPE = " in ln][0]         # after the "? " prompt
    assert math.isclose(float(mpe_line.split("MPE = ")[1]), math.log10(want), rel_tol=1e-5)
    toks = open(prefix + ".MPE").read().split()
    assert toks[0] == "MPE" and toks[1] == "1" and int(toks[2]) == len(want_a)
    assert [int(x) for x in toks[3:]] == want_a
