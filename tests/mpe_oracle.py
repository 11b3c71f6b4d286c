"""Test infrastructure: the reference computations for MPE (no counterpart in the reference implementation).

Max-product in numpy on top of the oracle's factors (oracle/oracle.py): a max-product step by the library's rule
(the maximum starts at x = 0, a later x replaces it only if its product is strictly greater -- ties keep the lowest x,
a NaN never replaces a number), MPE by enumeration, and max-product variable elimination in the reference's bucket
order with the decode backwards through the remembered choices."""
import numpy as np

import oracle as orc


def _over(values, scope, union, card):
    """a table over `scope` (last fastest) as an array over `union`, size-1 axes where it does not depend"""
    shape = [int(card[v]) for v in scope]
    a = np.asarray(values, dtype=np.float64).reshape(shape if shape else [1])
    if not scope:
        return a.reshape([1] * len(union))
    order = sorted(range(len(scope)), key=lambda i: union.index(scope[i]))
    a = np.transpose(a, order)
    have = [scope[i] for i in order]
    return a.reshape([int(card[v]) if v in have else 1 for v in union])


def max_last_axis(acc):
    """-> (max over the last axis, uint8 first index attaining it): best starts at x = 0 and x replaces it only if
    strictly greater, so ties keep the lowest x and a NaN never replaces a number"""
    best = np.array(acc[..., 0], dtype=np.float64)
    arg = np.zeros(best.shape, dtype=np.uint8)
    for x in range(1, acc.shape[-1]):
        m = acc[..., x] > best
        best = np.where(m, acc[..., x], best)
        arg = np.where(m, np.uint8(x), arg)
    return best, arg


def product_max_out(operands, out_scope, var, card):
    """max-product step: out[o] = max_x prod_k F_k(o, x), products in operand order -> (OFactor over out_scope,
    uint8 argmax array laid out like it)"""
    union = list(out_scope) + [var]
    acc = None
    for f in operands:
        a = _over(f.values, f.scope, union, card)
        acc = a.copy() if acc is None else acc * a
    acc = np.broadcast_to(acc, [int(card[v]) for v in union])
    best, arg = max_last_axis(acc)
    best = best.reshape(-1)
    return orc.OFactor(out_scope, best, float(best.sum())), arg.reshape(-1)


def _conditioned(f, evidence, card):
    shape = [int(card[v]) for v in f.scope]
    a = f.values.reshape(shape if shape else [1])
    if not f.scope:
        return [], a.reshape(-1)
    idx = tuple(evidence[v] if v in evidence else slice(None) for v in f.scope)
    return [v for v in f.scope if v not in evidence], np.ascontiguousarray(a[idx]).reshape(-1)


def mpe_brute_force(model, evidence):
    """enumeration over the unobserved variables (joints of at most 2^22 entries)
    -> (value, assignment, second-best value)"""
    card = [int(c) for c in model.card]
    free = [v for v in range(model.nvars) if v not in evidence]
    n = int(np.prod([card[v] for v in free], dtype=np.uint64)) if free else 1
    assert n <= 1 << 22, "joint too large for enumeration"
    joint = np.ones([card[v] for v in free] or [1])
    for f in model.factors:
        scope, vals = _conditioned(f, evidence, card)
        a = _over(vals, scope, free, card) if free else vals.reshape([1])
        joint = joint * a
    flat = joint.reshape(-1)
    i = int(np.argmax(flat))
    second = float(np.max(np.delete(flat, i))) if flat.size > 1 else -np.inf
    assignment = [0] * model.nvars
    for v, x in evidence.items():
        assignment[v] = int(x)
    for v, x in zip(free, np.unravel_index(i, [card[v] for v in free]) if free else []):
        assignment[v] = int(x)
    return float(flat[i]), assignment, second


def mpe_ve(model, evidence, order):
    """max-product variable elimination in the reference's bucket order (mirrors variable_elimination), then the
    decode backwards through the remembered choices -> (value, assignment)"""
    card = model.card
    factors = [orc.condition(f, evidence, card) for f in model.factors]
    value = 1.0
    buckets = {v: [] for v in order}
    remaining = list(order)

    def place(f):
        nonlocal value
        for v in remaining:
            if v in f.scope:
                buckets[v].append(f)
                return
        assert f.size == 1, "the order misses a variable"
        value = value * float(f.values[0])

    for f in factors:
        place(f)
    records = []
    while remaining:
        var = remaining.pop(0)
        if not buckets[var]:
            continue
        out_scope = []
        for f in buckets[var]:
            out_scope += [v for v in f.scope if v != var and v not in out_scope]
        newf, arg = product_max_out(buckets[var], out_scope, var, card)
        records.append((var, out_scope, arg))
        place(newf)
    assignment = [0] * model.nvars
    for v, x in evidence.items():
        assignment[v] = int(x)
    for var, scope, arg in reversed(records):
        idx = np.ravel_multi_index([assignment[v] for v in scope], [int(card[v]) for v in scope]) if scope else 0
        assignment[var] = int(arg[idx])
    return value, assignment
