"""Pins the CPU oracle (oracle/factor_oracle.c + oracle/oracle.py) against outputs of the
UNMODIFIED reference (tests/golden/*.json.gz, made by oracle/make_golden.py) and against
the reference's own shipped goldens.  CPU only."""
import math

import numpy as np
import pytest

import oracle as orc
from bnpp_b200 import synth

REL = 1e-12   # restatement vs reference: same arithmetic, at most a different multiplication order


def close(a, b, rel=REL):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    return a.shape == b.shape and np.allclose(a, b, rtol=rel, atol=0.0, equal_nan=True)


def F(rec):
    return orc.OFactor(rec["scope"], rec["values"], rec["partition"])


def test_ops_bit_exact(golden_ops):
    """per-op dumps of code/factor.cpp:97-255 on randomised scopes: BIT-exact values and scopes"""
    for c in golden_ops:
        card = c["cards"]
        a, b = F(c["a"]), F(c["b"])
        p = orc.product(a, b, card)
        assert p.scope == c["p"]["scope"]
        assert np.array_equal(p.values, np.array(c["p"]["values"]))
        assert p.partition == c["p"]["partition"]
        q = orc.divide(a, b, card)
        assert q.scope == c["q"]["scope"] and np.array_equal(q.values, np.array(c["q"]["values"]))
        assert q.partition == c["q"]["partition"]
        s = orc.sum_out(p, c["sum_var"], card)
        assert s.scope == c["s"]["scope"] and np.array_equal(s.values, np.array(c["s"]["values"]))
        assert s.partition == c["s"]["partition"]
        ev = {int(k): v for k, v in c["evidence"].items()}
        cf = orc.condition(p, ev, card)
        assert cf.scope == c["c"]["scope"] and np.array_equal(cf.values, np.array(c["c"]["values"]))
        assert cf.partition == c["c"]["partition"]
        n = orc.normalize(p)
        assert np.array_equal(n.values, np.array(c["n"]["values"])) and n.partition == 1.0
        assert orc.fmax(p) == c["max_p"] and orc.fmin(p) == c["min_p"]
        assert orc.fmax(q) == c["max_q"] and orc.fmin(q) == c["min_q"]
        # the fused step restatement equals product followed by sum_out
        if c["sum_var"] in p.scope:
            fs = orc.product_sum_out([a, b], s.scope, c["sum_var"], card)
            assert close(fs.values, s.values, 1e-14)


def test_partition_all_models(golden_models):
    for name, m in golden_models.items():
        model = orc.parse_uai(m["uai"])
        for case in m["pr"]:
            ev = {int(k): v for k, v in case["evidence"].items()}
            z = orc.partition(model, ev, case.get("order"))
            assert math.isclose(z, case["pr"], rel_tol=1e-11), (name, case["flag"], z, case["pr"])


def test_marginals(golden_models):
    for name in ["asia", "cancer", "earthquake", "child", "grid3x3"]:
        m = golden_models[name]
        model = orc.parse_uai(m["uai"])
        for case in m["mar"]:
            if case["flag"]:
                continue
            ev = {int(k): v for k, v in case["evidence"].items()}
            got = orc.marginals(model, ev)
            for g, want in zip(got, case["mar"]):
                assert close(g.values, want, 1e-11), name


def test_shipped_goldens(golden_models):
    """the reference's own fixtures: grid3x3.uai.PR/.MAR, network.uai.PR (6 significant digits)"""
    g = golden_models["grid3x3"]
    model = orc.parse_uai(g["uai"])
    want_pr = float(g["shipped"]["PR"].split()[-1])
    ev = orc.parse_evidence(g["shipped"]["PR_evid"])
    z = orc.joint(model, ev).partition            # what `mn` runs, code/model.cpp:51-67
    assert abs(math.log10(z) - want_pr) < 5e-5
    ev = orc.parse_evidence(g["shipped"]["MAR_evid"])
    toks = g["shipped"]["MAR"].split()
    assert toks[0] == "MAR"
    vals = [float(t) for t in toks[3:]]
    got = orc.joint_marginals(model, ev)
    i = 0
    for v in range(model.nvars):
        k = int(vals[i]); want = vals[i + 1:i + 1 + k]; i += 1 + k
        have = got[v].values if got[v].size == k else (np.array([0.0, 1.0]) if ev[v] == 1 else np.array([1.0, 0.0]))
        assert np.allclose(have, want, rtol=2e-5, atol=1e-9)
    n = golden_models["network"]
    model = orc.parse_uai(n["uai"])
    case = [c for c in n["pr"] if c["flag"] == "mf"][0]
    z = orc.partition(model, {}, case["order"])
    assert abs(math.log10(z) - float(n["shipped"]["PR"].split()[-1])) < 5e-4
    toks = n["shipped"]["MAR"].split()
    vals = [float(t) for t in toks[3:]]
    mar = [c for c in n["mar"] if c["flag"] == "mf"][0]["mar"]
    for v in range(model.nvars):
        assert np.allclose(mar[v], vals[3 * v + 1:3 * v + 3], rtol=2e-5, atol=1e-9)


def test_bp(golden_models, golden_synth):
    for name in ["asia", "alarm", "child", "grid3x3", "insurance"]:
        m = golden_models[name]
        model = orc.parse_uai(m["uai"])
        for case in m["bp"]:
            ev = {int(k): v for k, v in case["evidence"].items()}
            factors = [orc.condition(f, ev, model.card) for f in model.factors] if case["cond"] else model.factors
            fg = orc.OFactorGraph(model.card, factors)
            assert fg.update() == case["sweeps"], name
            for v in range(model.nvars):
                if case["cond"] and v in ev:
                    continue
                assert close(fg.marginal(v), case["mar"][v], 1e-10), (name, v)
    for rec in golden_synth["ising"]:
        if rec["n"] > 8:
            continue
        model = orc.parse_uai(synth.ising_uai(rec["n"], rec["h"], rec["J"], rec["seed"]))
        fg = orc.OFactorGraph(model.card, model.factors)
        assert fg.update() == rec["sweeps"]
        p0 = [fg.marginal(v)[0] for v in range(model.nvars)]
        assert close(p0, rec["p0"], 1e-10)


def test_ising40_bp(golden_synth):
    rec = [r for r in golden_synth["ising"] if r["n"] == 40 and r["J"] == 0.5][0]
    model = orc.parse_uai(synth.ising_uai(40, rec["h"], rec["J"], rec["seed"]))
    fg = orc.OFactorGraph(model.card, model.factors)
    assert fg.update() == rec["sweeps"]
    p0 = [fg.marginal(v)[0] for v in range(model.nvars)]
    assert close(p0, rec["p0"], 1e-10)


def test_synthetic_generators_pinned(golden_synth):
    import hashlib
    for rec in golden_synth["ising"]:
        t = synth.ising_uai(rec["n"], rec["h"], rec["J"], rec["seed"])
        assert hashlib.sha256(t.encode()).hexdigest() == rec["sha256"]
    for rec in golden_synth["bn"] + golden_synth["batch"]:
        t = synth.random_bn_uai(rec["N"], rec["W"], rec["K"], rec["seed"])
        assert hashlib.sha256(t.encode()).hexdigest() == rec["sha256"]


def test_synthetic_bn_partition(golden_synth):
    for rec in golden_synth["bn"]:
        model = orc.parse_uai(synth.random_bn_uai(rec["N"], rec["W"], rec["K"], rec["seed"]))
        ev = {int(k): v for k, v in rec["evidence"].items()}
        for case in rec["cases"]:
            if "pr" not in case or case["width"] > 12:
                continue
            z = orc.partition(model, ev, case["order"])
            assert math.isclose(z, case["pr"], rel_tol=1e-11)


@pytest.mark.skipif(not orc.have_ref(), reason="oracle/_ref not built (needs the reference's sources: make -C oracle ref REF=...)")
def test_ref_harness_matches_fixture(golden_models):
    """the travelling binary still answers as when the fixtures were made"""
    import os, tempfile
    m = golden_models["asia"]
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "asia.uai")
        open(p, "w").write(m["uai"])
        rows = orc.RefHarness().run(["model " + p, "evidset 2 0 1 2 1", "opt mf", "pr"])
    z = float([r for r in rows if r[0] == "PR"][0][1])
    assert z == [c for c in m["pr"] if c["flag"] == "mf" and c["evidence"]][0]["pr"]
