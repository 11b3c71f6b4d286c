"""Host-side multi-GPU partitioning of the path (SURVEY §8e).  Pure Python, no device needed.

* evidence / query batches: contiguous slices, no communication;
* one wide factor: the log2(G) variables of the widest elimination clique that the order
  eliminates LAST become shard variables.  With the canonical VE layout they are the
  leading axes of every wide table, so fixing them to the bits of a rank selects that
  rank's slab; summing them out across shards is one all-reduce of the partition.  For MPE and
  marginal MAP they must be maximised variables, and maximising them out is one all-gather of every
  rank's (value, assignment) and a max-loc.
"""


def batch_slice(rank, world, n):
    """contiguous [lo, hi) of n independent units for `rank`"""
    return rank * n // world, (rank + 1) * n // world


def pick_shard_vars(scopes, order, g):
    """the g variables of the widest elimination clique that `order` eliminates last"""
    if g <= 0:
        return []
    return widest_clique(scopes, order)[-g:]


def pick_max_shard_vars(scopes, order, g, cards, max_vars):
    """shard variables of a query that maximises over `max_vars` (MPE: every unobserved variable; marginal MAP: the MAP
    variables): the g variables of `max_vars` in the widest elimination clique of `order` that it eliminates last.
    Taking the max over the ranks of each rank's max over the other MAP variables of a sum over the summed ones is
    exact only when the shard variables are maximised, so a summed variable is never one.  ValueError when the widest
    clique holds fewer than g of them or one of the g is not binary."""
    if g <= 0:
        return []
    mx = set(max_vars)
    picked = [v for v in widest_clique(scopes, order) if v in mx][-g:]
    if len(picked) != g or any(int(cards[v]) != 2 for v in picked):
        raise ValueError("no %d binary MAP shard variables in the widest clique" % g)
    return picked


def widest_clique(scopes, order):
    """the variables of the widest elimination clique of `order` (the first one found), in elimination order"""
    rank = {v: i for i, v in enumerate(order)}
    buckets = {v: [] for v in order}
    for sc in scopes:
        live = [v for v in sc if v in rank]
        if live:
            buckets[min(live, key=rank.get)].append(set(live))
    best, best_u = -1, set()
    for v in order:
        if not buckets[v]:
            continue
        u = set().union(*buckets[v])
        if len(u) > best:
            best, best_u = len(u), set(u)
        u.discard(v)
        if u:
            buckets[min(u, key=rank.get)].append(u)
    return sorted(best_u, key=rank.get)


def shard_evidence(shard_vars, rank, cards=None):
    """value of every shard variable on `rank` (mixed radix over their cardinalities, first variable fastest)"""
    ev, r = {}, rank
    for v in shard_vars:
        c = 2 if cards is None else int(cards[v])
        ev[v] = r % c
        r //= c
    return ev


def shard_count(shard_vars, cards=None):
    n = 1
    for v in shard_vars:
        n *= 2 if cards is None else int(cards[v])
    return n


def pick_shard_vars_c(scopes, cards, order, g):
    """the same choice through the C ABI (bnpp_pick_shard_vars), for C / C++ callers"""
    import ctypes
    from . import capi, model
    L = capi.lib()
    arr, keep = model._scopes(scopes, cards)
    od = capi._u32(order)
    out = (ctypes.c_uint32 * max(1, g))()
    L.bnpp_pick_shard_vars.argtypes = [ctypes.c_int, ctypes.POINTER(capi.Scope), ctypes.c_int, capi.c_u32p, ctypes.c_int, capi.c_u32p]
    n = L.bnpp_pick_shard_vars(len(scopes), arr, len(order), ctypes.cast(od, capi.c_u32p), g, ctypes.cast(out, capi.c_u32p))
    return list(out[:n])
