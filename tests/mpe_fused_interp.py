"""Test infrastructure: a CPU interpreter of the max-mode step program of an MPE plan (`ve_fused_max`, fused.hpp) and
of the batched decode (`mpe_decode_batched`).

The max-mode counterpart of `fused_interp.interpret`: the same step sequence, arena offsets and operand-offset tables,
the products of every entry in operand order, then the maximum over the eliminated variable by the library's rule
(start at x = 0, a later x replaces it only if its product is strictly greater).  A kFusedMax step writes the argmax
byte of output entry o for set b at (R_s + o) * slice + b of a byte scratch, R_s taken from header word 7; the decode
walks the plan's eliminating steps backwards with R_s recomputed from `bnpp_ve_plan_describe`, so the row layout both
batch engines share is pinned without a GPU.  Entries are vectorised with numpy (IEEE float64, the kernels' rounding)."""
import ctypes

import numpy as np

from bnpp_b200 import capi
from fused_interp import GLOBAL, HEADER_WORDS, OPERAND_WORDS, TABLE, TO_GLOBAL, TO_RESULT, WANT_Z

MAX = 16            # kFusedMax


def program(plan_h, nb):
    """-> (prog words, offset-table words) of the fused program a batched run over nb sets executes; empty when the
    plan does not run fused"""
    L = capi.lib()
    L.bnpp_ve_plan_fused_program.argtypes = [ctypes.c_void_p, ctypes.c_uint32, capi.c_u32p, ctypes.c_uint64, capi.c_u64p,
                                             capi.c_u32p, ctypes.c_uint64, capi.c_u64p]
    np_, nt = ctypes.c_uint64(), ctypes.c_uint64()
    assert L.bnpp_ve_plan_fused_program(plan_h, nb, None, 0, ctypes.byref(np_), None, 0, ctypes.byref(nt)) == 0
    prog = np.zeros(max(1, np_.value), dtype=np.uint32)
    tab = np.zeros(max(1, nt.value), dtype=np.uint32)
    assert L.bnpp_ve_plan_fused_program(plan_h, nb, prog.ctypes.data_as(capi.c_u32p), prog.size, ctypes.byref(np_),
                                        tab.ctypes.data_as(capi.c_u32p), tab.size, ctypes.byref(nt)) == 0
    return prog[:np_.value], tab[:nt.value]


def fused_info(plan_h, nb):
    L = capi.lib()
    g, a, n = ctypes.c_int32(), ctypes.c_uint32(), ctypes.c_uint32()
    assert L.bnpp_ve_plan_fused_info(plan_h, nb, ctypes.byref(g), ctypes.byref(a), ctypes.byref(n)) == 0
    return g.value, a.value, n.value


def rows(desc):
    """the argmax row layout of a plan: [(step index, R_s, n_out)] over its eliminating steps in plan order"""
    out, r = [], 0
    for s, st in enumerate(desc["steps"]):
        if st["elim"] < 0:
            continue
        n_out = int(np.prod([c for _, c in st["scope"]], dtype=np.int64))
        out.append((s, r, n_out))
        r += n_out
    return out


def headers(prog, n_steps):
    """-> [(n_out, cx, k, flags, word 7)] of the program's steps"""
    out, pc = [], 0
    prog = [int(w) for w in prog]
    for _ in range(n_steps):
        n_out, cx, kf = prog[pc:pc + 3]
        out.append((n_out, cx, kf & 0xff, kf >> 8, prog[pc + 7]))
        pc += HEADER_WORDS
        for _ in range(kf & 0xff):
            w0 = prog[pc]
            pc += OPERAND_WORDS
            if w0 & 0xff:
                pc += 4 * (((w0 >> 8) + 1) // 2)
    assert pc == len(prog)
    return out


def interpret_max(prog, tab, n_steps, arena_doubles, tables, ev, scratch, b, slice_):
    """one evidence set (set b of a slice of slice_ sets) -> value; argmax bytes into scratch"""
    arena = np.full(max(1, arena_doubles), np.nan)
    value = None
    pc = 0
    prog = [int(w) for w in prog]
    for _ in range(n_steps):
        n_out, cx, kf, out_off, tab_off, _, _, row = prog[pc:pc + HEADER_WORDS]
        pc += HEADER_WORDS
        k, flags = kf & 0xff, kf >> 8
        assert not flags & (WANT_Z | TO_GLOBAL), "a max-mode program asks for a partition or a global output"
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
        best = vals[0].copy()
        arg = np.zeros(n_out, dtype=np.uint8)
        for x in range(1, cx):
            m = vals[x] > best
            best = np.where(m, vals[x], best)
            arg[m] = x
        assert not np.isnan(best).any(), "a step read an entry nobody wrote"
        if flags & MAX:
            scratch[(row + np.arange(n_out)) * slice_ + b] = arg
        else:
            assert cx == 1 and row == 0
        if flags & TO_RESULT:
            assert n_out == 1 and out_off == 0
            value = float(best[0])
        else:
            assert out_off + n_out <= arena_doubles
            arena[out_off:out_off + n_out] = best
    assert pc == len(prog)
    return 1.0 if value is None else value


def decode(desc, scratch, b, slice_, observed, ev, nvars):
    """the batched decode of set b: eliminating steps backwards, argmax at (R_s + o) * slice_ + b"""
    assignment = [0] * nvars
    for v, x in zip(observed, ev):
        assignment[v] = int(x)
    for s, r, _ in reversed(rows(desc)):
        st = desc["steps"][s]
        scope = [v for v, _ in st["scope"]]
        idx = int(np.ravel_multi_index([assignment[v] for v in scope], [c for _, c in st["scope"]])) if scope else 0
        assignment[st["elim"]] = int(scratch[(r + idx) * slice_ + b])
    return assignment
