"""Test infrastructure for batched evidence on multi-valued networks (tests/test_gpu_batch_multivalued.py and
tests/test_batch_multivalued_cpu.py): seeded Bayesian networks with mixed cardinalities, an exhaustive float64
reference, evidence sets with their edge values, and what a plan's describe dump says about the steps a batch runs.

Networks are (cards, scopes, tables) in the reference's layout: scope = [child, parents...], last variable fastest,
so a CPT holds P(child | parents) with the child as its most significant digit."""
import math
import random

import numpy as np

from bnpp_b200 import model
from fused_interp import DryPlan, parse_uai
from plan_emulator import describe

CARDS = (2, 3, 4, 5, 7)
BIG_CARD = 19           # evidence bytes above 15: a value that no longer fits a nibble
MAX_JOINT = 1 << 16     # networks up to this many joint states are also checked by enumeration
SLICE_BUDGET = 1 << 27  # K8 processes the batch in slices of (SLICE_BUDGET / widest intermediate) sets
# the golden networks with variables of more than two values, and the batch networks of the tests
MV_GOLDEN = ("child", "alarm", "insurance", "hailfinder", "hepar2", "Water")
N_RANDOM = 20
NETWORKS = list(MV_GOLDEN) + ["random_%d" % s for s in range(N_RANDOM)] + ["many_parents", "edges"]


def _cpt(rng, cards, child, parents):
    """P(child | parents), normalised over the child for every parent assignment"""
    npa = math.prod(cards[p] for p in parents)
    rows = []
    for _ in range(npa):
        w = [rng.uniform(0.05, 1.0) for _ in range(cards[child])]
        s = math.fsum(w)
        rows.append([x / s for x in w])
    return [rows[p][c] for c in range(cards[child]) for p in range(npa)]


def mixed_bn(seed, n=7, max_parents=3):
    """-> (cards, scopes, tables, observed): n variables with cards from CARDS and one with BIG_CARD, at most MAX_JOINT
    joint states, up to max_parents parents each.  observed: about half the variables, always the BIG_CARD one."""
    rng = random.Random(seed)
    while True:
        big = rng.randrange(n)
        cards = [BIG_CARD if v == big else rng.choice(CARDS) for v in range(n)]
        if math.prod(cards) <= MAX_JOINT:
            break
    scopes, tables = [], []
    for v in range(n):
        parents = sorted(rng.sample(range(v), min(v, rng.randint(1, max_parents))))
        scopes.append([v] + parents)
        tables.append(_cpt(rng, cards, v, parents))
    observed = sorted(set(rng.sample(range(n), n // 2)) | {big})
    return cards, scopes, tables, observed


def many_parents_bn(seed=3, n_parents=10):
    """a child with n_parents parents, all of them observed (more observed axes in one CPT than K8's parameter block
    holds), the child and two descendants free"""
    rng = random.Random(seed)
    cards = [rng.choice((2, 3)) for _ in range(n_parents)] + [3, 4, 2]
    c = n_parents
    scopes = [[v] for v in range(n_parents)] + [[c] + list(range(n_parents)), [c + 1, c], [c + 2, 0, c + 1]]
    tables = [_cpt(rng, cards, sc[0], sc[1:]) for sc in scopes]
    return cards, scopes, tables, list(range(n_parents))


def unmentioned_bn(seed=11):
    """a mixed network plus one more variable (the last id) that no factor mentions; it is observed"""
    cards, scopes, tables, observed = mixed_bn(seed, n=6)
    return cards + [2], scopes, tables, observed + [len(cards)]


def edge_bn(seed=5):
    """observed columns with cards 2, 3, 2, BIG_CARD (in that order): value 2 is legal in column 1 only"""
    rng = random.Random(seed)
    cards = [2, 3, 4, 2, 5, BIG_CARD, 3]
    scopes = [[0], [1, 0], [2, 0, 1], [3, 2], [4, 2, 3], [5, 4], [6, 5, 4, 1]]
    tables = [_cpt(rng, cards, sc[0], sc[1:]) for sc in scopes]
    return cards, scopes, tables, [0, 1, 3, 5]


def sliced_bn(seed=1, n=40, window=18):
    """binary network with ternary variables whose widest mf intermediate (9216 entries) makes K8 slice a batch into
    slices of an odd number of sets (checked by the tests through `slice_of`)"""
    rng = random.Random(seed)
    cards = [3 if v % 9 == 4 else 2 for v in range(n)]
    scopes, tables = [], []
    for v in range(n):
        parents = sorted(rng.sample(range(max(0, v - window), v), min(v, 3)))
        scopes.append([v] + parents)
        tables.append(_cpt(rng, cards, v, parents))
    return cards, scopes, tables, [n - 1, n - 5, n - 9]


def network(name, golden_models):
    """-> (cards, scopes, tables, observed) of one of NETWORKS; a golden network observes a seeded quarter of its
    variables"""
    if name in MV_GOLDEN:
        cards, scopes, tables = parse_uai(golden_models[name]["uai"])
        rng = random.Random(name)
        return cards, scopes, tables, sorted(rng.sample(range(len(cards)), max(2, len(cards) // 4)))
    if name == "many_parents":
        return many_parents_bn()
    if name == "edges":
        return edge_bn()
    return mixed_bn(int(name.split("_")[1]))


def to_uai(cards, scopes, tables):
    out = ["BAYES", str(len(cards)), " ".join(map(str, cards)), str(len(scopes))]
    out += ["%d %s" % (len(sc), " ".join(map(str, sc))) for sc in scopes]
    out += ["%d %s" % (len(t), " ".join("%.17g" % x for x in t)) for t in tables]
    return "\n".join(out) + "\n"


def mf_order(cards, scopes, observed):
    """the order BN.partition(ev, "mf") and BN.partition_batch(..., "mf") use"""
    variables = [v for v in range(len(cards)) if v not in set(observed)]
    return model.elim_order(cards, scopes, variables, "mf", observed=sorted(observed))[0]


def joint_table(cards, scopes, tables):
    """every joint assignment's probability (float64, shape = cards); only for networks of at most MAX_JOINT states"""
    n = len(cards)
    assert math.prod(cards) <= MAX_JOINT
    joint = np.ones(cards, dtype=np.float64)
    for sc, t in zip(scopes, tables):
        a = np.asarray(t, dtype=np.float64).reshape([cards[v] for v in sc])
        order = sorted(range(len(sc)), key=lambda i: sc[i])
        a = np.transpose(a, order).reshape([cards[v] if v in sc else 1 for v in range(n)])
        joint = joint * a
    return joint


def enumerate_z(joint, observed, values):
    """sum over every assignment of the free variables, exactly rounded (math.fsum)"""
    idx = [slice(None)] * joint.ndim
    for v, x in zip(observed, values):
        idx[v] = int(x)
    return math.fsum(np.ravel(joint[tuple(idx)]).tolist())


def evidence_sets(obs_cards, nsets, seed):
    """[nsets][len(obs_cards)] uint8 values in range, seeded; set 1 and every 97th set observe card - 1 everywhere"""
    rng = np.random.default_rng(seed)
    ev = np.stack([rng.integers(0, c, nsets) for c in obs_cards], axis=1).astype(np.uint8) if obs_cards else \
        np.zeros((nsets, 0), dtype=np.uint8)
    for i in [1] + list(range(97, nsets, 97)):
        if i < nsets:
            ev[i] = [c - 1 for c in obs_cards]
    return ev


def dry_describe(cards, scopes, observed, order):
    p = DryPlan(cards, scopes, observed, order)
    try:
        return describe(p.h)
    finally:
        p.close()


def slice_of(desc, nb):
    """the sets per K8 slice for a batch of nb (run_batched_once in ve.cu): the widest intermediate at most ~1 GiB"""
    widest = max([1, desc["result_size"]] + [f["size"] for f in desc["factors"] if f["src"] < 0])
    return min(nb, max(1, SLICE_BUDGET // widest))


def step_kinds(desc):
    """-> set of (operands K, values of the eliminated variable) over the plan's eliminating steps"""
    out = set()
    for st in desc["steps"]:
        if st["elim"] < 0:
            continue
        cx = [c for fid in st["ops"] for v, c, _ in desc["factors"][fid]["axes"] if v == st["elim"]]
        out.add((len(st["ops"]), cx[0]))
    return out


def max_observed_axes(desc):
    """most observed axes of one resident CPT that a step reads"""
    used = {fid for st in desc["steps"] for fid in st["ops"]}
    return max([len(f["obs"]) for i, f in enumerate(desc["factors"]) if f["src"] >= 0 and i in used] + [0])


def coverage(descs):
    """what the batch networks' plans together make K8 and K9 run -> dict of named booleans"""
    kinds = set().union(*[step_kinds(d) for d in descs])
    return {
        **{"cx>=3 K=%d" % k: any(kk == k and cx >= 3 for kk, cx in kinds) for k in (1, 2, 3, 4)},
        "binary K>=5": any(kk >= 5 and cx == 2 for kk, cx in kinds),
        "CPT with >=3 observed axes": max(max_observed_axes(d) for d in descs) >= 3,
        "CPT with >8 observed axes": max(max_observed_axes(d) for d in descs) > 8,
    }
