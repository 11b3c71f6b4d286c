"""Test infrastructure: CPU emulators of a marginal-MAP plan (bnpp_map_plan_*).

* `emulate` runs the schedule of a dry MAP plan (`plan_emulator.describe`) with numpy: operand products in operand order
  like the kernels, the maximum over the eliminated variable by the library's rule (start at x = 0, a later x replaces
  it only if strictly greater) on steps whose variable is a MAP variable, the sum in index order on every other step;
  the argmax tables of the max steps are kept and the decode walks them backwards as the device's decode does.
* `interpret_mixed` runs the step program of a batched MAP run (`ve_fused_mixed`, fused.hpp) for one evidence set: a
  kFusedMax step takes the maximum and writes its argmax bytes at (R_s + o) * slice + b, every other step sums as
  `ve_fused` does.  `decode` is the batched decode with R_s recomputed from `describe` over the max steps only.
A summed variable reports ASSIGN_SUMMED (0xFFFFFFFF; 0xFF in a batch)."""
import ctypes

import numpy as np

import mpe_oracle
from bnpp_b200 import capi, model
from fused_interp import GLOBAL, HEADER_WORDS, OPERAND_WORDS, TABLE, TO_GLOBAL, TO_RESULT, WANT_Z
from mpe_fused_interp import MAX
from plan_emulator import describe

ASSIGN_SUMMED = 0xFFFFFFFF


class DryMAPPlan:
    """bnpp_map_plan created without a context; rc is the creation's return code"""

    def __init__(self, cards, scopes, observed, map_vars, order):
        L = capi.lib()
        model._declare(L)
        self.L = L
        arr, self._keep = model._scopes(scopes, cards)
        c, ov, mv, od = capi._u32(cards), capi._u32(observed), capi._u32(map_vars), capi._u32(order)
        h = ctypes.c_void_p()
        self.rc = L.bnpp_map_plan_create(None, len(cards), ctypes.cast(c, capi.c_u32p), len(scopes), arr, len(observed),
                                         ctypes.cast(ov, capi.c_u32p), len(map_vars), ctypes.cast(mv, capi.c_u32p),
                                         len(order), ctypes.cast(od, capi.c_u32p), ctypes.byref(h))
        self.h = h

    def close(self):
        if self.h:
            self.L.bnpp_ve_plan_destroy(self.h)
            self.h = None


def run(desc, tables, ev, map_set):
    """-> (value, argmax tables (elim var, output scope, its cards, table) of the max steps in step order)"""
    slots = {}
    args = []
    value = 1.0

    def operand(fid):
        f = desc["factors"][fid]
        shape = [c for _, c, _ in f["axes"]]
        if f["src"] >= 0:
            mem = tables[f["src"]][sum(st * ev[col] for st, col in f["obs"]):]
            if not shape:
                return [], np.asarray(mem[0])
            return [v for v, _, _ in f["axes"]], np.lib.stride_tricks.as_strided(
                mem, shape=shape, strides=[8 * s for _, _, s in f["axes"]])
        return slots[fid]

    for st in desc["steps"]:
        out_vars = [v for v, _ in st["scope"]]
        union = out_vars + ([st["elim"]] if st["elim"] >= 0 else [])
        card = dict(st["scope"])
        acc = None
        for fid in st["ops"]:
            vars_, a = operand(fid)
            for v, c, _ in desc["factors"][fid]["axes"]:
                card[v] = c
            if vars_:
                order = sorted(range(len(vars_)), key=lambda i: union.index(vars_[i]))
                a = np.transpose(a, order)
                have = [vars_[i] for i in order]
                a = a.reshape([card[v] if v in have else 1 for v in union])
            else:
                a = np.asarray(a).reshape([1] * len(union))
            acc = a.astype(np.float64) if acc is None else acc * a
        acc = np.broadcast_to(acc, [card[v] for v in union])
        if st["elim"] in map_set:
            acc, arg = mpe_oracle.max_last_axis(acc)
            args.append((st["elim"], out_vars, [card[v] for v in out_vars], arg.reshape(-1)))
        elif st["elim"] >= 0:
            tot = acc[..., 0].copy()
            for x in range(1, card[st["elim"]]):
                tot = tot + acc[..., x]
            acc = tot
        if st["out"] < 0:
            value = float(np.asarray(acc).reshape(-1)[0])
        else:
            slots[st["out"]] = (out_vars, np.ascontiguousarray(acc))
    return value, args


def emulate(plan_h, tables, observed, ev_values, nvars, map_vars):
    """-> (value, assignment of every variable id): the dry plan's schedule in mixed mode and the backward decode"""
    map_set = set(map_vars)
    value, args = run(describe(plan_h), tables, ev_values, map_set)
    assignment = [0 if v in map_set else ASSIGN_SUMMED for v in range(nvars)]
    for v, x in zip(observed, ev_values):
        assignment[v] = int(x)
    for elim, scope, cards, arg in reversed(args):
        idx = int(np.ravel_multi_index([assignment[v] for v in scope], cards)) if scope else 0
        assignment[elim] = int(arg[idx])
    return value, assignment


def rows(desc, map_set):
    """the argmax row layout of a MAP plan: [(step index, R_s, n_out)] over its max steps in plan order"""
    out, r = [], 0
    for s, st in enumerate(desc["steps"]):
        if st["elim"] < 0 or st["elim"] not in map_set:
            continue
        n_out = int(np.prod([c for _, c in st["scope"]], dtype=np.int64))
        out.append((s, r, n_out))
        r += n_out
    return out


def interpret_mixed(prog, tab, n_steps, arena_doubles, tables, ev, scratch, b, slice_):
    """one evidence set (set b of a slice of slice_ sets) of a MAP program -> value; argmax bytes into scratch"""
    arena = np.full(max(1, arena_doubles), np.nan)
    value = None
    pc = 0
    prog = [int(w) for w in prog]
    for _ in range(n_steps):
        n_out, cx, kf, out_off, tab_off, _, _, row = prog[pc:pc + HEADER_WORDS]
        pc += HEADER_WORDS
        k, flags = kf & 0xff, kf >> 8
        assert not flags & (WANT_Z | TO_GLOBAL), "a MAP program asks for a partition or a global output"
        vals = None
        for q in range(k):
            w0, w1, sx, w3 = prog[pc:pc + OPERAND_WORDS]
            pc += OPERAND_WORDS
            kind, nobs = w0 & 0xff, w0 >> 8
            offs = tab[tab_off + q * n_out:tab_off + (q + 1) * n_out].astype(np.int64)
            if kind == 0:
                mem, base = arena, w1
            else:
                assert w3 == TABLE and w3 != GLOBAL
                base = 0
                for j in range(0, nobs, 2):
                    s0, i0, s1, i1 = prog[pc:pc + 4]
                    pc += 4
                    base += s0 * int(ev[i0])
                    if j + 1 < nobs:
                        base += s1 * int(ev[i1])
                mem = tables[w1]
            t = np.stack([mem[base + offs + x * sx] for x in range(cx)])       # [cx][n_out]
            vals = t if vals is None else vals * t                          # operand order, as the kernel multiplies
        if flags & MAX:
            best = vals[0].copy()
            arg = np.zeros(n_out, dtype=np.uint8)
            for x in range(1, cx):
                m = vals[x] > best
                best = np.where(m, vals[x], best)
                arg[m] = x
            scratch[(row + np.arange(n_out)) * slice_ + b] = arg
        else:
            assert row == 0
            best = vals[0].copy()
            for x in range(1, cx):
                best = best + vals[x]                                       # index order, as the kernel adds
        assert not np.isnan(best).any(), "a step read an entry nobody wrote"
        if flags & TO_RESULT:
            assert n_out == 1 and out_off == 0
            value = float(best[0])
        else:
            assert out_off + n_out <= arena_doubles
            arena[out_off:out_off + n_out] = best
    assert pc == len(prog)
    return 1.0 if value is None else value


def decode(desc, scratch, b, slice_, observed, ev, nvars, map_vars):
    """the batched decode of set b: max steps backwards, argmax at (R_s + o) * slice_ + b; summed variables 0xFF"""
    map_set = set(map_vars)
    assignment = [0 if v in map_set else 0xFF for v in range(nvars)]
    for v, x in zip(observed, ev):
        assignment[v] = int(x)
    for s, r, _ in reversed(rows(desc, map_set)):
        st = desc["steps"][s]
        scope = [v for v, _ in st["scope"]]
        idx = int(np.ravel_multi_index([assignment[v] for v in scope], [c for _, c in st["scope"]])) if scope else 0
        assignment[st["elim"]] = int(scratch[(r + idx) * slice_ + b])
    return assignment
