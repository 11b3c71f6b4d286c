"""Test infrastructure for all-marginals plans (tests/test_mar_engines_cpu.py and tests/test_gpu_mar_engines.py):
plain references of every variable's marginal P(v | e) and what a marginals plan's describe dump says about where its
result steps write.

References, both float64 and both independent of the bucket-tree plan:
- `oracle_marginals`: the reference's N variable-elimination passes (oracle.marginals, code/model.cpp:320-339), the
  pass of v eliminating the other unobserved variables in min-fill order -- what `bn -mar -mf` does -- with the
  observed ones appended.  File order is not an option: on andes its intermediates do not fit in memory.
- `enum_marginals`: exhaustive enumeration of the joint, every entry summed exactly (math.fsum), for networks of at
  most batch_networks.MAX_JOINT joint states.

Both return {v: array} for the unobserved variables that some factor mentions only: the marginal of any other
variable is the constant [1.0] of a one-entry slice."""
import json
import math
import os

import numpy as np

if __name__ == "__main__":
    import conftest  # noqa: F401  (run as a script: the import paths the suite has)
import batch_networks as bnet
import oracle as orc
from bnpp_b200 import model
from plan_emulator import describe


def oracle_marginals(cards, scopes, tables, ev):
    """ev: {variable: value} -> {v: P(v | ev)} for every unobserved v a factor mentions, by one VE pass per variable"""
    om = orc.OModel("BAYES", cards, [orc.OFactor(sc, t) for sc, t in zip(scopes, tables)])
    observed = sorted(ev)
    n = len(cards)

    def order_for(v):
        rest = [u for u in range(n) if u != v and u not in ev]
        return model.elim_order(cards, scopes, rest, "mf", observed=observed)[0] + observed

    # oracle.marginals, less the passes whose result is the constant [1.0]
    out = {}
    factors = [orc.condition(f, ev, om.card) for f in om.factors]
    mentioned = {v for sc in scopes for v in sc}
    for v in range(n):
        if v in ev or v not in mentioned:
            continue
        f = orc.normalize(orc.variable_elimination(order_for(v), factors, om.card))
        assert f.scope == [v]
        out[v] = np.array(f.values, dtype=np.float64)
    return out


def enum_marginals(cards, scopes, tables, ev):
    """ev: {variable: value} -> {v: P(v | ev)} for every unobserved v a factor mentions, by enumeration (math.fsum per
    entry)"""
    joint = bnet.joint_table(cards, scopes, tables)
    idx = [slice(None)] * joint.ndim
    for v, x in ev.items():
        idx[v] = slice(int(x), int(x) + 1)
    sub = joint[tuple(idx)]
    z = math.fsum(np.ravel(sub).tolist())
    out = {}
    mentioned = {v for sc in scopes for v in sc}
    for v in range(len(cards)):
        if v in ev or v not in mentioned:
            continue
        moved = np.moveaxis(sub, v, 0).reshape(cards[v], -1)
        out[v] = np.array([math.fsum(row.tolist()) for row in moved]) / z
    return out


def result_steps(plan_handle):
    """-> (describe dump, [(step index, roff, output variables, output cards)] of the steps that write the result)"""
    desc = describe(plan_handle)
    out = []
    for s, st in enumerate(desc["steps"]):
        if st["out"] == -1:         # bnpp_ve_plan_describe writes 0 for a result step, read back minus one
            out.append((s, st["roff"], [v for v, _ in st["scope"]], [c for _, c in st["scope"]]))
    return desc, out


# networks whose oracle passes take tens of seconds (andes: 27 s, Water: 12 s on one CPU core): their references are
# stored in tests/golden/mar_oracle.json, written by `python tests/mar_reference.py` from `oracle_marginals`
SLOW = ("andes", "Water")
SLOW_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mar_oracle.json")


def slow_golden():
    """-> {name: [(evidence, {v: array})]} of the stored references"""
    with open(SLOW_GOLDEN) as f:
        data = json.load(f)
    return {name: [({int(k): int(x) for k, x in c["evidence"].items()}, {int(v): np.array(m) for v, m in c["mar"].items()})
                   for c in cases] for name, cases in data.items()}


if __name__ == "__main__":
    from conftest import load_golden
    from fused_interp import parse_uai
    gm = load_golden("models")
    out = {}
    for name in SLOW:
        cards, scopes, tables = parse_uai(gm[name]["uai"])
        out[name] = []
        for c in gm[name]["pr"]:
            if c["flag"] != "mf":
                continue
            ev = {int(k): int(x) for k, x in c["evidence"].items()}
            mar = oracle_marginals(cards, scopes, tables, ev)
            out[name].append({"evidence": {str(k): x for k, x in ev.items()}, "mar": {str(v): m.tolist() for v, m in mar.items()}})
    with open(SLOW_GOLDEN, "w") as f:
        json.dump(out, f, separators=(",", ":"))
        f.write("\n")
