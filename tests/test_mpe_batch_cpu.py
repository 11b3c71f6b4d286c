"""Batched MPE without a GPU: the max-mode program a dry MPE plan compiles itself into for a batch (`ve_fused_max`) is
interpreted on the CPU for several evidence sets (tests/mpe_fused_interp.py), writing argmax bytes at the rows its
headers name; every row offset R_s must equal the layout recomputed from `bnpp_ve_plan_describe`, and the batched
decode must give the value and assignment of the plan's own max-mode emulation bit for bit -- and on the small
networks the enumerated MPE (value to 1e-14, assignment wherever the best beats the runner-up)."""
import math

import numpy as np
import pytest

import batch_networks as bnet
import mpe_fused_interp as mfi
import mpe_oracle
import oracle as orc
from fused_interp import parse_uai
from mpe_emulator import DryMPEPlan, emulate
from plan_emulator import describe

SMALL = ["asia", "asia_positive", "cancer", "earthquake", "grid3x3"]
NETWORKS = SMALL + list(bnet.MV_GOLDEN) + ["random_%d" % s for s in range(bnet.N_RANDOM)]
NB = 6


def _network(name, golden_models):
    if name in SMALL:
        cards, scopes, tables = parse_uai(golden_models[name]["uai"])
        obs = sorted(int(v) for v in next((c["evidence"] for c in golden_models[name]["pr"] if c["evidence"]), {}))
        return cards, scopes, tables, obs
    return bnet.network(name, golden_models)


def _check_layout(desc, prog, n_steps):
    """the program's kFusedMax steps are the plan's eliminating steps, each with its own R_s and n_out"""
    want = sorted((r, n) for _, r, n in mfi.rows(desc))
    got = sorted((row, n_out) for n_out, cx, k, flags, row in mfi.headers(prog, n_steps) if flags & mfi.MAX)
    assert got == want
    # no padding: the rows of consecutive eliminating steps are contiguous
    rows = mfi.rows(desc)
    for (_, r0, n0), (_, r1, _) in zip(rows, rows[1:]):
        assert r1 == r0 + n0
    return sum(n for _, _, n in rows)


@pytest.mark.parametrize("name", NETWORKS)
def test_max_program_and_batched_decode_equal_emulation(golden_models, name):
    cards, scopes, tables, observed = _network(name, golden_models)
    order = bnet.mf_order(cards, scopes, observed)
    p = DryMPEPlan(cards, scopes, observed, order)
    assert p.rc == 0, p.rc
    try:
        desc = describe(p.h)
        g, arena, n_steps = mfi.fused_info(p.h, NB)
        prog, tab = mfi.program(p.h, NB)
        if name == "Water":         # its widest buckets run one launch each: K8 serves its batches
            assert g == 0 and prog.size == 0
            return
        assert g > 0 and prog.size > 0, name
        assert mfi.fused_info(p.h, 1)[0] > 0      # the program exists for single sets too (they stay launch-per-bucket)
        R = _check_layout(desc, prog, n_steps)
        ev = bnet.evidence_sets([cards[v] for v in observed], NB, seed=len(name))
        scratch = np.full(max(1, R * NB), 0xAB, dtype=np.uint8)
        tabs = [np.asarray(t, dtype=np.float64) for t in tables]
        om = orc.OModel("BAYES", cards, [orc.OFactor(sc, t) for sc, t in zip(scopes, tables)]) \
            if name in SMALL or name.startswith("random") else None
        for b in range(NB):
            value = mfi.interpret_max(prog, tab, n_steps, arena, tabs, ev[b], scratch, b, NB)
            assignment = mfi.decode(desc, scratch, b, NB, observed, ev[b], len(cards))
            want_v, want_a = emulate(p.h, tabs, observed, [int(x) for x in ev[b]], len(cards))
            assert np.float64(value).view(np.uint64) == np.float64(want_v).view(np.uint64), (name, b, value, want_v)
            assert assignment == want_a, (name, b)
            if om is not None and math.prod(cards[v] for v in range(len(cards)) if v not in observed) <= 1 << 22:
                e = {v: int(x) for v, x in zip(observed, ev[b])}
                best, best_a, second = mpe_oracle.mpe_brute_force(om, e)
                assert math.isclose(value, best, rel_tol=1e-14, abs_tol=0.0), (name, b, value, best)
                if best > 0 and best - second > 1e-12 * best:
                    assert assignment == best_a, (name, b)
        assert not (scratch == 0xAB).all() or R == 0
    finally:
        p.close()


def test_mpe_plan_fused_switch_on_dry_plans():
    """set_fused(mpe_plan, 1) is accepted (it selects the batch engine); 0 turns the program off"""
    cards, scopes, tables, observed = bnet.mixed_bn(0)
    p = DryMPEPlan(cards, scopes, observed, bnet.mf_order(cards, scopes, observed))
    try:
        L = p.L
        assert L.bnpp_ve_plan_set_fused(p.h, 0) == 0
        assert mfi.fused_info(p.h, 4)[0] == 0 and mfi.program(p.h, 4)[0].size == 0
        assert L.bnpp_ve_plan_set_fused(p.h, 1) == 0
        assert mfi.fused_info(p.h, 4)[0] > 0
    finally:
        p.close()
