"""Test infrastructure: the reference computation for marginal MAP (no counterpart in the reference implementation).

Enumeration of  max_{x_M} sum_{x_S} prod_f f(x, e)  over the joint table of a small network (at most
batch_networks.MAX_JOINT states): for every assignment of the MAP variables the summed variables are added with
math.fsum (exactly rounded), then the best assignment is kept."""
import math

import numpy as np

import batch_networks as bnet


def map_brute_force(cards, scopes, tables, evidence, map_vars):
    """-> (value, {v: x_v} of the best MAP assignment, runner-up value); evidence: {var: value}.  Ties keep the first
    assignment in id order (the MAP variable with the largest id fastest)."""
    joint = bnet.joint_table(cards, scopes, tables)
    idx = tuple(int(evidence[v]) if v in evidence else slice(None) for v in range(len(cards)))
    free = [v for v in range(len(cards)) if v not in evidence]
    j = joint[idx]                                          # axes: free variables in id order
    m = sorted(map_vars)
    pos = [free.index(v) for v in m]
    rest = [i for i in range(len(free)) if i not in pos]
    j = np.transpose(j, pos + rest).reshape(math.prod(cards[v] for v in m), -1)
    sums = [math.fsum(row.tolist()) for row in j]
    best = int(np.argmax(sums))
    second = max(sums[:best] + sums[best + 1:]) if len(sums) > 1 else -math.inf
    x = np.unravel_index(best, [cards[v] for v in m]) if m else ()
    return sums[best], {v: int(xi) for v, xi in zip(m, x)}, second
