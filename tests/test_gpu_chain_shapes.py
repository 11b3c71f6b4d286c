"""Every window shape on the GPU (contract_chain.cu): for each network of tests/chain_nets.py -- all 66 (m, add)
instantiations, sides 0 / 1 / 2 per level, sides that are raw input views in file order or with an observed variable
-- the windowed plan and the per-step plan (chain_depth = 1) give the SAME BITS for Z and the result in the first run,
the graph capture and its replays, also after the evidence value moved a side's base.  The result is the window's
output table itself (chain_nets keeps the variables the window does not eliminate), so every entry the window wrote is
compared.  The profiled window row names the instantiation of that shape; the result and Z match a float64 CPU
emulation of the plan; and a windowed plan whose tables are not 32-byte aligned (the dynamic path, one launch per
step) gives the windowed run's bits."""
import math
import types

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from bnpp_b200 import capi, model  # noqa: E402
from chain_nets import chain_net, shape_cases  # noqa: E402
from plan_emulator import describe, run as emulate  # noqa: E402
from test_chain_plan_cpu import windows  # noqa: E402
from test_gpu_chain import make_plan, run, same_bits  # noqa: E402

CASES = shape_cases()
# one case per m, and the cases with an evidence-view side: the result and Z against the CPU emulation
EMULATED = {"2-22-k21", "3-012-k121", "4-0000-k1201", "2-01-k11-ev", "3-101-k121-ev", "4-0002-k1022-ev", "4-1111-k1212-ev"}


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def kernel_name(m, add):
    return "contract_chain<D=%d,add=%s>" % (m, "".join(map(str, add)))


@pytest.mark.parametrize("name,m,add,k,opts", CASES, ids=[c[0] for c in CASES])
def test_shape_same_bits(ctx, name, m, add, k, opts):
    cards, scopes, tables, order, obs = chain_net(m, add, k, **opts)
    bn = model.BN(ctx, cards, list(zip(scopes, tables)))
    vals = [0] * len(obs)
    # with an observed variable: runs 4-6 replay the graph with the other value (the side's base moved), 7-9 go back
    sets = [vals, [1] * len(obs), vals] if obs else [vals]
    zs = same_bits(bn, obs, order, sets)
    if obs:
        assert zs[0] != zs[1] and zs[2] == zs[0], zs
    p = make_plan(bn, obs, order, 4)
    assert len(windows(p.h)) == 1
    p.set_profiling(True)
    z, res = run(bn, p, vals)
    chain = [r["kernel"] for r in p.step_stats() if r["kernel"].startswith("contract_chain")]
    assert chain == [kernel_name(m, add)], chain
    assert z.tobytes() == np.float64(zs[0]).tobytes()
    if name in EMULATED:
        d = describe(p.h)
        for i, v in enumerate(sets[:2]):
            want, wz = emulate(d, tables, v)
            got = res if i == 0 else run(bn, p, v)[1]
            assert math.isclose(zs[i], wz, rel_tol=1e-12), (v, zs[i], wz)
            assert np.allclose(got, want, rtol=1e-12, atol=0), (v, np.max(np.abs(got / want - 1)))
    p.close()
    bn.close()


def test_unaligned_tables_take_the_dynamic_path(ctx):
    """tables one double past a 32-byte boundary: run_dynamic executes the windowed plan's re-ordered steps one launch
    each, to the bits of the windowed run"""
    import torch
    cards, scopes, tables, order, obs = chain_net(4, (0, 0, 0, 2), (1, 0, 2, 2), raw="ev", added="middle")
    bn = model.BN(ctx, cards, list(zip(scopes, tables)))
    offs, total = [], 0
    for t in tables:
        offs.append(total + 1)
        total += (len(t) + 1 + 3) // 4 * 4
    host = np.zeros(total)
    for t, o in zip(tables, offs):
        host[o:o + len(t)] = t
    with torch.cuda.stream(ctx.torch_stream):
        dev = torch.from_numpy(host).to("cuda")
    ctx.sync()
    unaligned = types.SimpleNamespace(ctx=ctx, table_ptrs=[dev.data_ptr() + 8 * o for o in offs])
    p = make_plan(bn, obs, order, 4)
    assert windows(p.h) and p.n_launches < len(describe(p.h)["steps"])
    for vals in ([0], [1]):
        want = run(bn, p, vals)
        before = ctx.launches
        got = run(unaligned, p, vals)
        assert ctx.launches - before >= len(describe(p.h)["steps"])
        assert got[0].tobytes() == want[0].tobytes() and got[1].tobytes() == want[1].tobytes(), (vals, got, want)
    p.close()
    del dev
    bn.close()
