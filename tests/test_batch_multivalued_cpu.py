"""The networks of tests/test_gpu_batch_multivalued.py without a GPU: the mixed-cardinality generator is seeded, the
CPU oracle (the GPU test's second reference) equals exhaustive enumeration on them, and their dry plans contain the
steps the GPU test claims to reach -- so a change of generator that loses coverage fails here."""
import math

import numpy as np

import batch_networks as bnet
import oracle as orc
from fused_interp import parse_uai

REL = 1e-12


def test_generator_is_deterministic():
    for seed in range(bnet.N_RANDOM):
        a, b = bnet.mixed_bn(seed), bnet.mixed_bn(seed)
        assert a == b
        cards, scopes, tables, observed = a
        assert bnet.BIG_CARD in cards and cards.index(bnet.BIG_CARD) in observed
        assert set(cards) <= set(bnet.CARDS) | {bnet.BIG_CARD} and math.prod(cards) <= bnet.MAX_JOINT
        for sc, t in zip(scopes, tables):
            rows = np.asarray(t).reshape(cards[sc[0]], -1)          # child digit most significant
            assert np.allclose(rows.sum(axis=0), 1.0, rtol=0, atol=1e-15)
    assert bnet.mixed_bn(0) != bnet.mixed_bn(1)
    ev = bnet.evidence_sets([2, 3, bnet.BIG_CARD], 300, seed=4)
    assert np.array_equal(ev, bnet.evidence_sets([2, 3, bnet.BIG_CARD], 300, seed=4))
    assert ev.max(axis=0).tolist() == [1, 2, bnet.BIG_CARD - 1] and ev[1].tolist() == [1, 2, bnet.BIG_CARD - 1]


def test_oracle_equals_enumeration():
    nets = [bnet.mixed_bn(s) for s in range(bnet.N_RANDOM)] + [bnet.edge_bn()]
    for i, (cards, scopes, tables, observed) in enumerate(nets):
        m = orc.OModel("BAYES", cards, [orc.OFactor(sc, t) for sc, t in zip(scopes, tables)])
        order = bnet.mf_order(cards, scopes, observed)
        joint = bnet.joint_table(cards, scopes, tables)
        assert math.isclose(math.fsum(joint.ravel().tolist()), 1.0, rel_tol=1e-14)
        for row in bnet.evidence_sets([cards[v] for v in observed], 6, seed=i):
            ev = {v: int(x) for v, x in zip(observed, row)}
            want = bnet.enumerate_z(joint, observed, row)
            got = orc.partition(m, ev, order)
            assert abs(got - want) <= REL * want, (i, ev, got, want)


def test_batch_networks_reach_the_kernels(golden_models):
    mv = [n for n, m in golden_models.items() if max(parse_uai(m["uai"])[0]) > 2]
    assert len(mv) >= 4 and set(bnet.MV_GOLDEN) <= set(mv), mv
    descs = []
    for name in bnet.NETWORKS:
        cards, scopes, _, observed = bnet.network(name, golden_models)
        descs.append(bnet.dry_describe(cards, scopes, observed, bnet.mf_order(cards, scopes, observed)))
    cov = bnet.coverage(descs)
    assert all(cov.values()), cov


def test_sliced_network_slices_oddly():
    """the K8 slice of the sliced network is odd, and the GPU test's batch of 2 slice + slice // 3 sets has three
    slices with a shorter last one"""
    cards, scopes, _, observed = bnet.sliced_bn()
    desc = bnet.dry_describe(cards, scopes, observed, bnet.mf_order(cards, scopes, observed))
    s = bnet.slice_of(desc, 1 << 30)
    n3 = 2 * s + s // 3
    assert s % 2 == 1 and -(-n3 // s) == 3 and 0 < n3 - 2 * s < s, s
