"""Test infrastructure: a CPU emulator of an MPE plan (bnpp_mpe_plan_*).

The schedule of a dry MPE plan (`plan_emulator.describe`) is executed with numpy in max mode: operand products in
operand order like the kernels, the maximum over the eliminated variable by the library's rule (start at x = 0, a
later x replaces it only if strictly greater), every eliminating step's argmax table kept, then the decode walks the
eliminating steps backwards exactly as the device's one-thread decode does."""
import ctypes

import numpy as np

import mpe_oracle
from bnpp_b200 import capi, model
from plan_emulator import describe


class DryMPEPlan:
    """bnpp_mpe_plan created without a context"""

    def __init__(self, cards, scopes, observed, order):
        L = capi.lib()
        model._declare(L)
        self.L = L
        arr, self._keep = model._scopes(scopes, cards)
        c, ov, od = capi._u32(cards), capi._u32(observed), capi._u32(order)
        h = ctypes.c_void_p()
        self.rc = L.bnpp_mpe_plan_create(None, len(cards), ctypes.cast(c, capi.c_u32p), len(scopes), arr, len(observed),
                                         ctypes.cast(ov, capi.c_u32p), len(order), ctypes.cast(od, capi.c_u32p),
                                         ctypes.byref(h))
        self.h = h

    def close(self):
        if self.h:
            self.L.bnpp_ve_plan_destroy(self.h)
            self.h = None


def run(desc, tables, ev):
    """-> (value, argmax tables (elim var, output scope, its cards, table) of the eliminating steps in step order) of the
    plan `desc` for evidence values `ev` (one per observed id, in plan order)"""
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
        vars_, arr = slots[fid]
        return vars_, arr

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
        if st["elim"] >= 0:
            acc, arg = mpe_oracle.max_last_axis(acc)
            args.append((st["elim"], out_vars, [card[v] for v in out_vars], arg.reshape(-1)))
        if st["out"] < 0:
            value = float(np.asarray(acc).reshape(-1)[0])
        else:
            slots[st["out"]] = (out_vars, np.ascontiguousarray(acc))
    return value, args


def emulate(plan_h, tables, observed, ev_values, nvars):
    """-> (value, assignment): the dry plan's schedule in max mode and the backward decode"""
    d = describe(plan_h)
    value, args = run(d, tables, ev_values)
    assignment = [0] * nvars
    for v, x in zip(observed, ev_values):
        assignment[v] = int(x)
    for elim, scope, cards, arg in reversed(args):
        idx = int(np.ravel_multi_index([assignment[v] for v in scope], cards)) if scope else 0
        assignment[elim] = int(arg[idx])
    return value, assignment
