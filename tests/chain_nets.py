"""Test infrastructure: networks whose VE plan forms one window (chain.hpp) of a chosen shape.

A window runs m binary eliminations t0 .. t{m-1} as one contract_chain launch; level j multiplies its input by k[j]
side tables (0 .. 2) that add add[j] new variables (0 .. 2).  chain_net builds, for a shape (m, add) and side counts
k, a network whose plan forms exactly that window:

  F0(h0, t0 .. t{m-1}, rest)      eliminating h0 first makes the head H(t0 .. t{m-1}, rest), t0 innermost
  level j's sides                 t_j, level j's new variables, a few rest variables and, as the layout options say,
                                  a later tile variable or a variable an earlier level added

The order eliminates h0, t0 .. t{m-1} only: the rest and the new variables are kept, so the window's output table is
copied into the query's result as it is, and a test comparing results bit for bit compares every entry the window
wrote (a sum over it would hide a wrong entry in its rounding, or a swap of two variables nothing else tells apart).
The result step eliminates nothing, so it never links and the window ends at its m-th level.

R rest variables make the narrowest level's union exactly 2^20 entries (the least a link takes); the head is at most
2^23 doubles.  Two sides of one level cover all of the rest between them, so their joint table is above the cap of
ve.cu fold_small and they stay two operands.  The raw options put a side at a level of 2^20 entries (fold_small's cap
2^15), where an input view of 2^16 entries is read in place with its file-order strides: `raw="cpt"` a CPT of 16
variables, `raw="ev"` a CPT of 17 variables with an observed one in the middle (a view whose base moves with the
evidence value)."""
import numpy as np

MAX_LEVELS, MAX_ADD, TILE_BITS = 4, 2, 4


def shape_ok(m, add):
    """contract_chain.cu chain_shape_ok: every level's input and output tile within 16 doubles"""
    nb = 0
    for j in range(m):
        inb = m - j + nb
        if inb > TILE_BITS or inb - 1 + add[j] > TILE_BITS:
            return False
        nb += add[j]
    return True


def chain_shapes():
    """every (m, add) with a contract_chain instantiation"""
    out = []
    for m in range(2, MAX_LEVELS + 1):
        for code in range((MAX_ADD + 1) ** m):
            add = tuple(code // (MAX_ADD + 1) ** j % (MAX_ADD + 1) for j in range(m))
            if shape_ok(m, add):
                out.append((m, add))
    return out


def level_bits(m, add):
    """log2 of level j's union entries, less the rest variables"""
    return [m - j + sum(add[:j]) + add[j] for j in range(m)]


def chain_net(m, add, k, scatter=False, later=False, earlier=True, added="outer", raw=None, seed=0):
    """-> (cards, scopes, tables, order, observed): a network whose dry plan forms one window of m levels, level j
    adding add[j] variables with k[j] side tables (k[j] >= 1 where add[j] > 0).

    scatter: side rest variables at scattered rest bits (several Fields per side); later: the first side of every level
    but the last also holds the next tile variable; earlier: the last side of a level holds the variable added last by
    the levels before it; added: the new variables "outer", "middle" or "inner" to the rest in the window output's
    layout (kept variables are laid out by id, the largest innermost); raw: None, "cpt" or "ev" (see the module).
    add[j] may exceed 2 to build a window the planner must cut."""
    assert len(add) == len(k) == m and all(kj >= (aj > 0) for aj, kj in zip(add, k)) and max(k) <= 2
    rng = np.random.default_rng(seed)
    bits = level_bits(m, add)
    R = 20 - min(bits)
    nt = sum(add)
    h0, t = 0, list(range(1, m + 1))
    kept = list(range(m + 1, m + 1 + nt + R))
    cut = {"outer": 0, "middle": R // 2, "inner": R}[added]
    new = kept[cut:cut + nt]
    rest = kept[:cut] + kept[cut + nt:]
    nv = kept[-1] + 1
    o = None
    if raw == "ev":
        o, nv = nv, nv + 1
    order = [h0] + t
    cards = [2] * nv

    f0 = [h0] + t + rest
    scopes = [[f0[i] for i in rng.permutation(len(f0))]]
    raw_at = None
    if raw:
        raw_at = next(j for j in range(m) if bits[j] == min(bits) and k[j] > 0)
    for j in range(m):
        news = new[sum(add[:j]):sum(add[:j + 1])]
        sides = [[t[j]] for _ in range(k[j])]
        for i, v in enumerate(news):
            sides[(i + j) % k[j]].append(v)
        if k[j] and later and j + 1 < m:
            sides[0].append(t[j + 1])
        if k[j] and earlier and sum(add[:j]):
            sides[-1].append(new[sum(add[:j]) - 1])
        for q, sc in enumerate(sides):
            if j == raw_at and q == 0:
                # an input view of exactly 2^16 entries, t_j slowest (file order is not the canonical order)
                sc += rest[:16 - len(sc)]
                if raw == "ev":
                    sc.insert(len(sc) // 2, o)
                continue
            room = 16 - len(sc)
            if k[j] == 2:
                pick = rest[q::2] if scatter else (rest[:11] if q == 0 else rest[R - 11:])
                sc += pick[:min(11, room)]
            elif scatter:
                sc += [rest[(b + j) % R] for b in (1, 3, 6, 7, 10)]
            else:
                sc += rest[2 * j:2 * j + 4]
        scopes += sides
    tables = [rng.uniform(0.5, 1.5, int(np.prod([cards[v] for v in sc]))) for sc in scopes]
    return cards, scopes, tables, order, ([o] if o is not None else [])


def shape_cases():
    """(name, m, add, k, options) for every shape: side counts and layout options in rotation, so that every level
    index sees k = 0, 1 and 2, and the raw sides at every m"""
    cases = []
    placements = ["outer", "middle", "inner"]
    for i, (m, add) in enumerate(chain_shapes()):
        k = tuple((0 if a == 0 else 1) if (i + j) % 3 == 0 else (1 if (i + j) % 3 == 1 else 2) for j, a in enumerate(add))
        opts = {"scatter": i % 2 == 1, "later": i % 4 in (1, 2), "earlier": i % 5 != 3, "added": placements[i % 3]}
        cases.append(("%d-%s-k%s" % (m, "".join(map(str, add)), "".join(map(str, k))), m, add, k, opts))
    for m, add, k, raw in [(2, (1, 1), (1, 2), "cpt"), (3, (0, 1, 1), (1, 1, 1), "cpt"), (4, (0, 1, 1, 1), (0, 1, 2, 1), "cpt"),
                           (2, (0, 1), (1, 1), "ev"), (3, (1, 0, 1), (1, 2, 1), "ev"), (4, (0, 0, 0, 2), (1, 0, 2, 2), "ev"),
                           (4, (1, 1, 1, 1), (1, 2, 1, 2), "ev")]:
        cases.append(("%d-%s-k%s-%s" % (m, "".join(map(str, add)), "".join(map(str, k)), raw), m, add, k,
                      {"raw": raw, "scatter": m == 3, "added": "middle"}))
    return cases
