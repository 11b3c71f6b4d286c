"""Python mirror of `bn::BN` inference entry points (reference code/model.hh:49-120) over the C ABI.

The CPTs are uploaded to HBM once (`BN(...)`) and stay resident; `partition` /
`marginals` are BN::partition / BN::marginals (code/model.cpp:250-346): ordering on the
host with the reference's heuristics and tie-breaks (bnpp_elim_order), then one
device-resident variable-elimination plan (bnpp_ve_plan_*).  Only the result returns.
"""
import ctypes
import time

import numpy as np
import torch

from . import capi

HEUR = {"min-fill": 0, "mf": 0, "weighted-min-fill": 1, "wmf": 1, "min-degree": 2, "md": 2}


def _declare(L):
    if getattr(L, "_ve_declared", False):
        return
    P = ctypes.POINTER
    L.bnpp_elim_order.argtypes = [ctypes.c_int, capi.c_u32p, ctypes.c_int, P(capi.Scope), ctypes.c_int, capi.c_u32p,
                                  ctypes.c_int, capi.c_u32p, ctypes.c_int, capi.c_u32p, capi.c_u32p, capi.c_u32p]
    L.bnpp_order_width.argtypes = [ctypes.c_int, capi.c_u32p, ctypes.c_int, P(capi.Scope), ctypes.c_int, capi.c_u32p,
                                   capi.c_u32p]
    L.bnpp_ve_plan_create.argtypes = [ctypes.c_void_p, ctypes.c_int, P(capi.Scope), ctypes.c_int, capi.c_u32p,
                                      ctypes.c_int, capi.c_u32p, P(ctypes.c_void_p)]
    L.bnpp_ve_plan_destroy.argtypes = [ctypes.c_void_p]
    L.bnpp_ve_plan_info.argtypes = [ctypes.c_void_p, P(ctypes.c_int32), capi.c_u32p, capi.c_u32p, capi.c_u64p,
                                    capi.c_u64p, capi.c_u64p, capi.c_u64p, capi.c_u64p]
    L.bnpp_ve_plan_run.argtypes = [ctypes.c_void_p, P(ctypes.c_void_p), capi.c_u32p, ctypes.c_void_p, ctypes.c_void_p]
    L.bnpp_ve_plan_run_batched.argtypes = [ctypes.c_void_p, P(ctypes.c_void_p), ctypes.c_uint32, ctypes.c_uint32,
                                           ctypes.c_void_p, ctypes.c_void_p]
    L.bnpp_mar_plan_create.argtypes = [ctypes.c_void_p, ctypes.c_int, capi.c_u32p, ctypes.c_int, P(capi.Scope), ctypes.c_int,
                                       capi.c_u32p, ctypes.c_int, capi.c_u32p, P(ctypes.c_void_p)]
    L.bnpp_mar_plan_layout.argtypes = [ctypes.c_void_p, ctypes.c_int, capi.c_u32p, capi.c_u32p, capi.c_u64p]
    L.bnpp_ve_plan_set_profiling.argtypes = [ctypes.c_void_p, ctypes.c_int]
    L.bnpp_ve_plan_set_normalize.argtypes = [ctypes.c_void_p, ctypes.c_int]
    L.bnpp_mar_plan_normalize.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    L.bnpp_ve_plan_result_size.argtypes = [ctypes.c_void_p, capi.c_u64p]
    L.bnpp_ve_plan_set_fused.argtypes = [ctypes.c_void_p, ctypes.c_int]
    L.bnpp_ve_plan_fused_info.argtypes = [ctypes.c_void_p, ctypes.c_uint32, P(ctypes.c_int32), capi.c_u32p, capi.c_u32p]
    L.bnpp_ve_plan_set_segments.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_uint32]
    L.bnpp_ve_plan_step_stats.argtypes = [ctypes.c_void_p, ctypes.c_uint64, P(ctypes.c_float), capi.c_u64p, capi.c_u64p,
                                          P(ctypes.c_int32)]
    L.bnpp_ve_plan_step_kernel.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_char_p, ctypes.c_size_t]
    L.bnpp_mpe_plan_create.argtypes = [ctypes.c_void_p, ctypes.c_int, capi.c_u32p, ctypes.c_int, P(capi.Scope), ctypes.c_int,
                                       capi.c_u32p, ctypes.c_int, capi.c_u32p, P(ctypes.c_void_p)]
    L.bnpp_mpe_plan_run.argtypes = [ctypes.c_void_p, P(ctypes.c_void_p), capi.c_u32p, ctypes.c_void_p, ctypes.c_void_p]
    L.bnpp_mpe_plan_run_batched.argtypes = [ctypes.c_void_p, P(ctypes.c_void_p), ctypes.c_uint32, ctypes.c_uint32,
                                            ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    L.bnpp_elim_order_constrained.argtypes = [ctypes.c_int, capi.c_u32p, ctypes.c_int, P(capi.Scope), ctypes.c_int,
                                              capi.c_u32p, ctypes.c_int, capi.c_u32p, ctypes.c_int, capi.c_u32p, ctypes.c_int,
                                              capi.c_u32p, capi.c_u32p, capi.c_u32p]
    L.bnpp_map_plan_create.argtypes = [ctypes.c_void_p, ctypes.c_int, capi.c_u32p, ctypes.c_int, P(capi.Scope), ctypes.c_int,
                                       capi.c_u32p, ctypes.c_int, capi.c_u32p, ctypes.c_int, capi.c_u32p, P(ctypes.c_void_p)]
    L._ve_declared = True


def _scopes(scope_list, cards):
    n = len(scope_list)
    arr = (capi.Scope * max(1, n))()
    keep = []
    for i, sc in enumerate(scope_list):
        s, ka = capi.make_scope(sc, [cards[v] for v in sc])
        arr[i] = s
        keep.append(ka)
    return arr, keep


def elim_order(cards, scopes, variables, heuristic, reference_containers=False, observed=(), _arr=None, _cards=None):
    """Graph(...).ordering(variables) of code/graph.cpp:41-101 -> (order, width).  Host only.
    `scopes` are ORIGINAL factor scopes; `observed` variables are removed from them (and from
    `variables`) inside the library, as BN::partition does by conditioning (code/model.cpp:283-287).
    reference_containers=True runs the slow path on std::unordered_set adjacency (cross-check)."""
    L = capi.lib()
    _declare(L)
    arr = _arr if _arr is not None else _scopes(scopes, cards)[0]
    c = _cards if _cards is not None else capi._u32(cards)
    v = capi._u32(variables)
    ob = capi._u32(list(observed))
    out = (ctypes.c_uint32 * max(1, len(variables)))()
    width, n = ctypes.c_uint32(), ctypes.c_uint32()
    rc = L.bnpp_elim_order(len(cards), ctypes.cast(c, capi.c_u32p), len(scopes), arr, len(observed),
                           ctypes.cast(ob, capi.c_u32p), len(variables), ctypes.cast(v, capi.c_u32p),
                           HEUR[heuristic] | (0x100 if reference_containers else 0), ctypes.cast(out, capi.c_u32p),
                           ctypes.byref(n), ctypes.byref(width))
    if rc != 0:
        raise capi.BnppError(rc, "bnpp_elim_order")
    return list(out[:n.value]), width.value


def elim_order_constrained(cards, scopes, first, last, heuristic, reference_containers=False, observed=(), _arr=None,
                           _cards=None):
    """the constrained order of marginal MAP -> (order, width): `first` (the summed variables) exactly as `elim_order`
    orders them, then `last` (the MAP variables) by the same heuristic on the same graph, the fill edges of the first
    phase in place; width over both phases.  Host only."""
    L = capi.lib()
    _declare(L)
    arr = _arr if _arr is not None else _scopes(scopes, cards)[0]
    c = _cards if _cards is not None else capi._u32(cards)
    f, la, ob = capi._u32(first), capi._u32(last), capi._u32(list(observed))
    out = (ctypes.c_uint32 * max(1, len(first) + len(last)))()
    width, n = ctypes.c_uint32(), ctypes.c_uint32()
    rc = L.bnpp_elim_order_constrained(len(cards), ctypes.cast(c, capi.c_u32p), len(scopes), arr, len(observed),
                                       ctypes.cast(ob, capi.c_u32p), len(first), ctypes.cast(f, capi.c_u32p), len(last),
                                       ctypes.cast(la, capi.c_u32p), HEUR[heuristic] | (0x100 if reference_containers else 0),
                                       ctypes.cast(out, capi.c_u32p), ctypes.byref(n), ctypes.byref(width))
    if rc != 0:
        raise capi.BnppError(rc, "bnpp_elim_order_constrained")
    return list(out[:n.value]), width.value


def order_width(cards, scopes, order):
    """Graph::order_width, code/graph.cpp:197-237"""
    L = capi.lib()
    _declare(L)
    arr, keep = _scopes(scopes, cards)
    c, o = capi._u32(cards), capi._u32(order)
    width = ctypes.c_uint32()
    rc = L.bnpp_order_width(len(cards), ctypes.cast(c, capi.c_u32p), len(scopes), arr, len(order),
                            ctypes.cast(o, capi.c_u32p), ctypes.byref(width))
    if rc != 0:
        raise capi.BnppError(rc, "bnpp_order_width")
    return width.value


class VEPlan:
    """bnpp_ve_plan: the schedule of fused elimination launches for (scopes, observed ids, order)."""

    def __init__(self, ctx, cards, scopes, observed, order, _arr=None):
        self.ctx = ctx
        L = ctx.L
        _declare(L)
        arr, self._keep = (_arr, None) if _arr is not None else _scopes(scopes, cards)
        self.observed = list(observed)
        ov, od = capi._u32(self.observed), capi._u32(order)
        h = ctypes.c_void_p()
        ctx.check(L.bnpp_ve_plan_create(ctx.h, len(scopes), arr, len(self.observed), ctypes.cast(ov, capi.c_u32p),
                                        len(order), ctypes.cast(od, capi.c_u32p), ctypes.byref(h)))
        self.h = h
        rank = ctypes.c_int32()
        rv = (ctypes.c_uint32 * capi_max_rank())()
        rc_ = (ctypes.c_uint32 * capi_max_rank())()
        vals = [ctypes.c_uint64() for _ in range(5)]
        ctx.check(L.bnpp_ve_plan_info(h, ctypes.byref(rank), ctypes.cast(rv, capi.c_u32p), ctypes.cast(rc_, capi.c_u32p),
                                      *[ctypes.byref(v) for v in vals]))
        self.result_scope = list(rv[:rank.value])
        self.result_cards = list(rc_[:rank.value])
        self.result_size = int(np.prod(self.result_cards, dtype=np.uint64)) if rank.value else 1
        self.n_launches, self.union_entries, self.bytes, self.peak_bytes, self.max_step_entries = [v.value for v in vals]

    def run(self, table_ptrs, obs_val, result_ptr, z_ptr=None):
        n = len(table_ptrs)
        tp = (ctypes.c_void_p * max(1, n))(*table_ptrs)
        ov = capi._u32(obs_val)
        self.ctx.check(self.ctx.L.bnpp_ve_plan_run(self.h, tp, ctypes.cast(ov, capi.c_u32p), ctypes.c_void_p(result_ptr),
                                                   ctypes.c_void_p(z_ptr) if z_ptr else None))

    def run_batched(self, table_ptrs, nb, ev_ptr, result_ptr):
        """ev_ptr: device uint8 [nb][len(observed)]; result_ptr: device double [result_size][nb]"""
        n = len(table_ptrs)
        tp = (ctypes.c_void_p * max(1, n))(*table_ptrs)
        self.ctx.check(self.ctx.L.bnpp_ve_plan_run_batched(self.h, tp, int(nb), len(self.observed),
                                                           ctypes.c_void_p(ev_ptr), ctypes.c_void_p(result_ptr)))

    def set_profiling(self, on=True):
        self.ctx.check(self.ctx.L.bnpp_ve_plan_set_profiling(self.h, int(on)))

    def set_fused(self, on=True):
        """one launch for the whole plan when every step is small (default), or one launch per bucket"""
        self.ctx.check(self.ctx.L.bnpp_ve_plan_set_fused(self.h, int(on)))

    def set_segments(self, on=True, max_steps=0):
        """EXPERIMENTAL: inside a launch-per-bucket plan, every run of consecutive small steps as one ve_fused launch"""
        self.ctx.check(self.ctx.L.bnpp_ve_plan_set_segments(self.h, int(on), int(max_steps)))

    def fused_info(self, nb=1):
        """-> (lanes per evidence set, 0 = a run over nb sets is not fused; shared-memory doubles per set; steps)"""
        g, a, n = ctypes.c_int32(), ctypes.c_uint32(), ctypes.c_uint32()
        self.ctx.check(self.ctx.L.bnpp_ve_plan_fused_info(self.h, int(nb), ctypes.byref(g), ctypes.byref(a), ctypes.byref(n)))
        return g.value, a.value, n.value

    def step_stats(self):
        n = self.n_launches
        ms = (ctypes.c_float * max(1, n))()
        by = (ctypes.c_uint64 * max(1, n))()
        en = (ctypes.c_uint64 * max(1, n))()
        k = (ctypes.c_int32 * max(1, n))()
        self.ctx.check(self.ctx.L.bnpp_ve_plan_step_stats(self.h, n, ms, ctypes.cast(by, capi.c_u64p),
                                                          ctypes.cast(en, capi.c_u64p), k))
        out = []
        buf = ctypes.create_string_buffer(160)
        for i in range(n):
            self.ctx.L.bnpp_ve_plan_step_kernel(self.h, i, buf, 160)
            out.append({"ms": ms[i], "bytes": by[i], "entries": en[i], "k": k[i], "kernel": buf.value.decode()})
        return out

    def close(self):
        if self.h:
            self.ctx.L.bnpp_ve_plan_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            if self.h and self.ctx.h:      # the plan owns a device arena: never leak it
                self.close()
        except Exception:
            pass


def capi_max_rank():
    return 64


class MarPlan(VEPlan):
    """bnpp_mar_plan: every marginal in one two-pass bucket-tree plan (SURVEY 8f row 2)."""

    def __init__(self, ctx, cards, scopes, observed, order, _arr=None):
        self.ctx = ctx
        L = ctx.L
        _declare(L)
        arr, self._keep = (_arr, None) if _arr is not None else _scopes(scopes, cards)
        self.observed = list(observed)
        c, ov, od = capi._u32(cards), capi._u32(self.observed), capi._u32(order)
        h = ctypes.c_void_p()
        ctx.check(L.bnpp_mar_plan_create(ctx.h, len(cards), ctypes.cast(c, capi.c_u32p), len(scopes), arr,
                                         len(self.observed), ctypes.cast(ov, capi.c_u32p), len(order),
                                         ctypes.cast(od, capi.c_u32p), ctypes.byref(h)))
        self.h = h
        n = len(cards)
        off, size = (ctypes.c_uint32 * max(1, n))(), (ctypes.c_uint32 * max(1, n))()
        total = ctypes.c_uint64()
        ctx.check(L.bnpp_mar_plan_layout(h, n, ctypes.cast(off, capi.c_u32p), ctypes.cast(size, capi.c_u32p),
                                         ctypes.byref(total)))
        self.off, self.size, self.result_size = list(off[:n]), list(size[:n]), total.value
        vals = [ctypes.c_uint64() for _ in range(5)]
        ctx.check(L.bnpp_ve_plan_info(h, None, None, None, *[ctypes.byref(v) for v in vals]))
        self.n_launches, self.union_entries, self.bytes, self.peak_bytes, self.max_step_entries = [v.value for v in vals]


class MPEPlan(VEPlan):
    """bnpp_mpe_plan: max-product variable elimination over the schedule of a VEPlan, then an on-device decode of the
    most probable assignment.  `order` must cover every unobserved variable.  ctx.h may be None: a dry plan."""

    def __init__(self, ctx, cards, scopes, observed, order, _arr=None):
        self.ctx = ctx
        L = ctx.L
        _declare(L)
        arr, self._keep = (_arr, None) if _arr is not None else _scopes(scopes, cards)
        self.observed = list(observed)
        self.nvars = len(cards)
        c, ov, od = capi._u32(cards), capi._u32(self.observed), capi._u32(order)
        h = ctypes.c_void_p()
        ctx.check(L.bnpp_mpe_plan_create(ctx.h, len(cards), ctypes.cast(c, capi.c_u32p), len(scopes), arr,
                                         len(self.observed), ctypes.cast(ov, capi.c_u32p), len(order),
                                         ctypes.cast(od, capi.c_u32p), ctypes.byref(h)))
        self.h = h
        self.result_size = 1
        vals = [ctypes.c_uint64() for _ in range(5)]
        ctx.check(L.bnpp_ve_plan_info(h, None, None, None, *[ctypes.byref(v) for v in vals]))
        self.n_launches, self.union_entries, self.bytes, self.peak_bytes, self.max_step_entries = [v.value for v in vals]

    def run_mpe(self, table_ptrs, obs_val, value_ptr, assignment_ptr):
        """value_ptr: device double; assignment_ptr: device uint32 [nvars].  Asynchronous."""
        tp = (ctypes.c_void_p * max(1, len(table_ptrs)))(*table_ptrs)
        ov = capi._u32(obs_val)
        self.ctx.check(self.ctx.L.bnpp_mpe_plan_run(self.h, tp, ctypes.cast(ov, capi.c_u32p), ctypes.c_void_p(value_ptr),
                                                    ctypes.c_void_p(assignment_ptr)))

    def run_mpe_batched(self, table_ptrs, nb, ev_ptr, value_ptr, assignment_ptr):
        """ev_ptr: device uint8 [nb][len(observed)]; value_ptr: device double [nb]; assignment_ptr: device uint8
        [nvars][nb].  Asynchronous."""
        tp = (ctypes.c_void_p * max(1, len(table_ptrs)))(*table_ptrs)
        self.ctx.check(self.ctx.L.bnpp_mpe_plan_run_batched(self.h, tp, int(nb), len(self.observed), ctypes.c_void_p(ev_ptr),
                                                            ctypes.c_void_p(value_ptr), ctypes.c_void_p(assignment_ptr)))

    def set_fused(self, on=True):
        """the engine of batched runs: the whole plan in one launch per slice when every step is small (default), or one
        launch per bucket; single runs are always one launch per bucket"""
        super().set_fused(on)


class MAPPlan(MPEPlan):
    """bnpp_map_plan: marginal MAP over the schedule of a VEPlan -- steps eliminating a MAP variable take the maximum
    (and keep their argmax tables for the decode), every other eliminating step sums.  `order` must eliminate every
    summed variable before any MAP variable.  Runs as an MPEPlan (run_mpe, run_mpe_batched); a summed variable reports
    ASSIGN_SUMMED (0xFFFFFFFF; 0xFF in a batch).  ctx.h may be None: a dry plan."""

    def __init__(self, ctx, cards, scopes, observed, order, map_vars=(), _arr=None):
        self.ctx = ctx
        L = ctx.L
        _declare(L)
        arr, self._keep = (_arr, None) if _arr is not None else _scopes(scopes, cards)
        self.observed = list(observed)
        self.map_vars = list(map_vars)
        self.nvars = len(cards)
        c, ov, mv, od = capi._u32(cards), capi._u32(self.observed), capi._u32(self.map_vars), capi._u32(order)
        h = ctypes.c_void_p()
        ctx.check(L.bnpp_map_plan_create(ctx.h, len(cards), ctypes.cast(c, capi.c_u32p), len(scopes), arr,
                                         len(self.observed), ctypes.cast(ov, capi.c_u32p), len(self.map_vars),
                                         ctypes.cast(mv, capi.c_u32p), len(order), ctypes.cast(od, capi.c_u32p),
                                         ctypes.byref(h)))
        self.h = h
        self.result_size = 1
        vals = [ctypes.c_uint64() for _ in range(5)]
        ctx.check(L.bnpp_ve_plan_info(h, None, None, None, *[ctypes.byref(v) for v in vals]))
        self.n_launches, self.union_entries, self.bytes, self.peak_bytes, self.max_step_entries = [v.value for v in vals]


ASSIGN_SUMMED = 0xFFFFFFFF


class BN:
    """Model(name, variables, factors) with the factors resident in HBM (code/model.cpp:14-19)."""

    def __init__(self, ctx, cards, factors):
        """factors: list of (scope ids, host values) in the reference's layout (last variable fastest)"""
        self.ctx = ctx
        self.cards = [int(c) for c in cards]
        self.scopes = [[int(v) for v in sc] for sc, _ in factors]
        sizes = [int(np.asarray(v).size) for _, v in factors]
        self._sizes, self._offs = sizes, None
        # one pinned staging buffer, one H2D copy, tables 32-byte aligned inside one allocation
        offs, total = [], 0
        for n in sizes:
            offs.append(total)
            total += (n + 3) // 4 * 4
        self._host = torch.empty(max(1, total), dtype=torch.float64).pin_memory() if torch.cuda.is_available() \
            else torch.empty(max(1, total), dtype=torch.float64)
        hv = self._host.numpy()
        for (sc, v), o, n in zip(factors, offs, sizes):
            hv[o:o + n] = np.asarray(v, dtype=np.float64).reshape(-1)
        self._offs = offs
        self.h2d_bytes = 8 * total
        with torch.cuda.stream(ctx.torch_stream):
            self._dev = torch.empty(max(1, total), dtype=torch.float64, device="cuda:%d" % ctx.device)
            self._dev.copy_(self._host, non_blocking=True)
        self.table_ptrs = [self._dev.data_ptr() + 8 * o for o in offs]
        self._plans = {}
        self._shard_cache = {}
        self._batch_plans = {}
        self._order_cache = {}      # (observed ids, heuristic) -> elimination order: a function of the model's structure only
        self._res2 = None
        self._batch_out = {}
        self.last_timing = {}
        self._scope_arr, self._scope_keep = _scopes(self.scopes, self.cards)   # the model's structure never changes
        self._cards_arr = capi._u32(self.cards)

    @property
    def nvars(self):
        return len(self.cards)

    def reupload(self):
        """host -> device copy of every table (what an end-to-end query pays once per model)"""
        with torch.cuda.stream(self.ctx.torch_stream):
            self._dev.copy_(self._host, non_blocking=True)

    def conditioned_scopes(self, observed):
        return [[v for v in sc if v not in observed] for sc in self.scopes]

    def order(self, variables, observed, heuristic=None):
        """the order BN::variable_elimination uses (code/model.cpp:358-369)"""
        if heuristic is None:
            return [v for v in variables if v not in observed], None
        return elim_order(self.cards, self.scopes, variables, heuristic, observed=sorted(observed), _arr=self._scope_arr,
                          _cards=self._cards_arr)

    MAX_PLANS = 64      # every plan keeps its device arena, offset tables and replay graph: the cache is bounded (oldest out)

    def plan(self, observed, order):
        return self._cached_plan((tuple(observed), tuple(order)), VEPlan, observed, order)

    def _cached_plan(self, key, cls, observed, order):
        p = self._plans.get(key)
        if p is None:
            while len(self._plans) >= self.MAX_PLANS:
                old_key = next(iter(self._plans))
                old = self._plans.pop(old_key)
                self._batch_plans = {k: v for k, v in self._batch_plans.items() if v is not old}
                old.close()
            p = cls(self.ctx, self.cards, self.scopes, observed, order, _arr=self._scope_arr)
            self._plans[key] = p
        return p

    def variable_elimination(self, evidence, order):
        """-> (result scope, result cards, device tensor of size+1 doubles, partition last)"""
        observed = sorted(evidence)
        p = self.plan(observed, order)
        with torch.cuda.stream(self.ctx.torch_stream):
            res = torch.empty(p.result_size + 1, dtype=torch.float64, device=self._dev.device)
        p.run(self.table_ptrs, [evidence[v] for v in observed], res.data_ptr(), res.data_ptr() + 8 * p.result_size)
        return p.result_scope, p.result_cards, res

    def shard(self, evidence, heuristic, comm):
        """wide-factor sharding (SURVEY 8e): the log2(world) variables of the widest elimination clique that the order
        of the UNSHARDED query eliminates last, observed at this rank's values -> (evidence incl. shard values, shard vars)"""
        from . import sharding
        g = (comm.world - 1).bit_length() if comm is not None else 0
        if g == 0:
            return dict(evidence), []
        if (1 << g) != comm.world:
            raise ValueError("wide-factor sharding needs a power-of-two number of ranks")
        key = (tuple(sorted(evidence)), heuristic, g)
        shard_vars = self._shard_cache.get(key)
        if shard_vars is None:
            variables = [v for v in range(self.nvars) if v not in evidence]
            full_order, _ = self.order(variables, evidence, heuristic)
            live = self.conditioned_scopes(set(evidence))
            shard_vars = [v for v in sharding.pick_shard_vars(live, full_order, g)]
            if len(shard_vars) != g or any(self.cards[v] != 2 for v in shard_vars):
                raise ValueError("no %d binary shard variables in the widest clique" % g)
            self._shard_cache[key] = shard_vars
        full = dict(evidence)
        full.update(sharding.shard_evidence(shard_vars, comm.rank))
        return full, shard_vars

    def partition(self, evidence=None, heuristic=None, comm=None):
        """BN::partition, VE branch (code/model.cpp:275-294) -> (Z, uptime_ms).
        comm (a nccl.ShardComm over all ranks): the network is sharded over the ranks by the leading variables of its
        widest clique, every rank eliminates its slab and the partition is summed over NVLink (bnpp_ve_plan_run_sharded);
        every rank returns the same Z."""
        t0 = time.perf_counter()
        evidence = dict(evidence or {})
        if comm is not None and comm.world > 1:
            evidence, _ = self.shard(evidence, heuristic, comm)
        observed = sorted(evidence)
        okey = (tuple(observed), heuristic)
        order = self._order_cache.get(okey)
        if order is None:
            variables = [v for v in range(self.nvars) if v not in evidence]
            order, _ = self.order(variables, evidence, heuristic)
            if len(self._order_cache) >= self.MAX_PLANS:
                self._order_cache.pop(next(iter(self._order_cache)))
            self._order_cache[okey] = order
        t1 = time.perf_counter()
        p = self.plan(observed, order)
        t2 = time.perf_counter()
        if self._res2 is None:
            with torch.cuda.stream(self.ctx.torch_stream):
                self._res2 = torch.empty(2, dtype=torch.float64, device=self._dev.device)
                self._res2_host = torch.empty(2, dtype=torch.float64).pin_memory()
        assert p.result_size == 1
        if comm is not None and comm.world > 1:
            comm.run_sharded(p, self.table_ptrs, [evidence[v] for v in observed], self._res2.data_ptr(), self._res2.data_ptr() + 8)
        else:
            p.run(self.table_ptrs, [evidence[v] for v in observed], self._res2.data_ptr(), self._res2.data_ptr() + 8)
        with torch.cuda.stream(self.ctx.torch_stream):
            self._res2_host.copy_(self._res2, non_blocking=True)
        self.ctx.sync()
        t3 = time.perf_counter()
        z0, z1 = self._res2_host.tolist()
        assert z0 == z1 or (comm is not None and abs(z0 - z1) <= 1e-12 * abs(z1))     # code/model.cpp:288
        self.last_timing = {"order_ms": (t1 - t0) * 1e3, "plan_ms": (t2 - t1) * 1e3, "run_ms": (t3 - t2) * 1e3}
        return z1, (time.perf_counter() - t0) * 1e3

    def mpe(self, evidence=None, heuristic=None, comm=None):
        """Most probable explanation (no reference counterpart) -> (value, assignment list, uptime_ms).
        value = max over the unobserved variables of the product of every CPT conditioned on the evidence, i.e.
        P(x*, e), not normalised; assignment[v] is the evidence value of an observed v.  Ties go to the lowest values.
        The order is the one `partition` uses (heuristic None: variables in id order).
        comm (a nccl.ShardComm over all ranks): the network is sharded over the ranks exactly as `partition` shards it,
        every rank maximises over its slab, and the ranks' values and assignments are all-gathered and the best one kept
        on the device (bnpp_mpe_plan_run_sharded); every rank returns the same answer, the shard variables at the
        winning rank's values.  The ranks form their products in another order than one GPU does, so the value agrees
        with the unsharded query to rounding, and under exactly tied maxima the lowest rank wins, which can give another
        assignment than one GPU.  Batches (`mpe_batch`) are sharded by contiguous slices and need no collective."""
        t0 = time.perf_counter()
        evidence = dict(evidence or {})
        sharded = comm is not None and comm.world > 1
        if sharded:
            evidence, _ = self.shard(evidence, heuristic, comm)
        observed = sorted(evidence)
        okey = (tuple(observed), heuristic)
        order = self._order_cache.get(okey)
        if order is None:
            variables = [v for v in range(self.nvars) if v not in evidence]
            order, _ = self.order(variables, evidence, heuristic)
            if len(self._order_cache) >= self.MAX_PLANS:
                self._order_cache.pop(next(iter(self._order_cache)))
            self._order_cache[okey] = order
        t1 = time.perf_counter()
        p = self._cached_plan(("mpe", tuple(observed), tuple(order)), MPEPlan, observed, order)
        t2 = time.perf_counter()
        n = self.nvars
        if getattr(self, "_mpe_buf", None) is None or self._mpe_buf.numel() != 2 + n:
            # [value (two uint32 words), assignment[nvars]]: one device-to-host copy of 1 + nvars words
            with torch.cuda.stream(self.ctx.torch_stream):
                self._mpe_buf = torch.empty(2 + n, dtype=torch.int32, device=self._dev.device)
                self._mpe_host = torch.empty(2 + n, dtype=torch.int32).pin_memory()
        if sharded:
            comm.run_mpe_sharded(p, self.table_ptrs, [evidence[v] for v in observed], self._mpe_buf.data_ptr(),
                                 self._mpe_buf.data_ptr() + 8)
        else:
            p.run_mpe(self.table_ptrs, [evidence[v] for v in observed], self._mpe_buf.data_ptr(), self._mpe_buf.data_ptr() + 8)
        with torch.cuda.stream(self.ctx.torch_stream):
            self._mpe_host.copy_(self._mpe_buf, non_blocking=True)
        self.ctx.sync()
        t3 = time.perf_counter()
        host = self._mpe_host.numpy()
        value = float(host[:2].view(np.float64)[0])
        assignment = [int(x) for x in host[2:].view(np.uint32)]
        self.last_timing = {"order_ms": (t1 - t0) * 1e3, "plan_ms": (t2 - t1) * 1e3, "run_ms": (t3 - t2) * 1e3}
        return value, assignment, (time.perf_counter() - t0) * 1e3

    def _map_order(self, m, observed, heuristic):
        """the elimination order of a MAP query (m: sorted MAP variables): heuristic None orders the summed variables,
        then the MAP variables, each in id order; else the constrained heuristic order"""
        okey = ("map", tuple(observed), tuple(m), heuristic)
        order = self._order_cache.get(okey)
        if order is None:
            obs, ms = set(observed), set(m)
            summed = [v for v in range(self.nvars) if v not in obs and v not in ms]
            if heuristic is None:
                order = summed + [v for v in m if v not in obs]
            else:
                order, _ = elim_order_constrained(self.cards, self.scopes, summed, m, heuristic, observed=sorted(observed),
                                                  _arr=self._scope_arr, _cards=self._cards_arr)
            if len(self._order_cache) >= self.MAX_PLANS:
                self._order_cache.pop(next(iter(self._order_cache)))
            self._order_cache[okey] = order
        return order

    def _map_plan(self, map_vars, observed, heuristic):
        """the MAP plan of (MAP variables, observed ids, heuristic), over the order of `_map_order`"""
        m = sorted(int(v) for v in map_vars)        # a repeated, observed or unknown id: BNPP_EINVAL from the library
        order = self._map_order(m, observed, heuristic)

        def make(ctx, cards, scopes, obs_, order_, _arr=None):
            return MAPPlan(ctx, cards, scopes, obs_, order_, map_vars=m, _arr=_arr)
        return self._cached_plan(("map", tuple(observed), tuple(m), tuple(order)), make, observed, order)

    def map_shard(self, map_vars, evidence, heuristic, comm):
        """wide-factor sharding of a marginal MAP query: the log2(world) MAP variables of the widest elimination clique
        of the UNSHARDED query's constrained order that it eliminates last (sharding.pick_max_shard_vars: ValueError
        unless there are that many and they are binary), observed at this rank's values
        -> (evidence incl. shard values, shard vars)"""
        from . import sharding
        g = (comm.world - 1).bit_length()
        if (1 << g) != comm.world:
            raise ValueError("wide-factor sharding needs a power-of-two number of ranks")
        m = sorted(int(v) for v in map_vars)
        observed = sorted(evidence)
        key = ("map", tuple(observed), tuple(m), heuristic, g)
        shard_vars = self._shard_cache.get(key)
        if shard_vars is None:
            order = self._map_order(m, observed, heuristic)
            live = self.conditioned_scopes(set(evidence))
            shard_vars = self._shard_cache[key] = sharding.pick_max_shard_vars(live, order, g, self.cards, m)
        full = dict(evidence)
        full.update(sharding.shard_evidence(shard_vars, comm.rank))
        return full, shard_vars

    def map(self, map_vars, evidence=None, heuristic=None, comm=None):
        """Marginal MAP (no reference counterpart) -> (value, {v: x_v for v in map_vars}, uptime_ms).
        value = max over the MAP variables of the sum over every other unobserved variable of the product of every CPT
        conditioned on the evidence, i.e. P(x_M*, e), not normalised.  Ties go to the lowest values in decode order.
        The order eliminates the summed variables first (heuristic None: each group in id order; else the constrained
        heuristic order of `elim_order_constrained`).
        comm (a nccl.ShardComm over all ranks): sharded like `mpe`, but the shard variables are MAP variables of the
        widest clique of the constrained order (`map_shard`): maximising a rank's max-of-sums over the ranks is exact
        only for maximised shard variables.  Every rank runs the MAP plan over the other MAP variables with the shard
        variables observed, and returns the same answer; the shard variables report the winning rank's values.  Ties
        and rounding as for `mpe`.  Batches (`map_batch`) are sharded by contiguous slices and need no collective."""
        t0 = time.perf_counter()
        evidence = dict(evidence or {})
        map_vars = [int(v) for v in map_vars]
        sharded = comm is not None and comm.world > 1
        rank_vars = map_vars
        if sharded:
            evidence, shard_vars = self.map_shard(map_vars, evidence, heuristic, comm)
            rank_vars = [v for v in map_vars if v not in shard_vars]
        observed = sorted(evidence)
        p = self._map_plan(rank_vars, observed, heuristic)
        t1 = time.perf_counter()
        n = self.nvars
        if getattr(self, "_mpe_buf", None) is None or self._mpe_buf.numel() != 2 + n:
            with torch.cuda.stream(self.ctx.torch_stream):
                self._mpe_buf = torch.empty(2 + n, dtype=torch.int32, device=self._dev.device)
                self._mpe_host = torch.empty(2 + n, dtype=torch.int32).pin_memory()
        if sharded:
            comm.run_mpe_sharded(p, self.table_ptrs, [evidence[v] for v in observed], self._mpe_buf.data_ptr(),
                                 self._mpe_buf.data_ptr() + 8)
        else:
            p.run_mpe(self.table_ptrs, [evidence[v] for v in observed], self._mpe_buf.data_ptr(), self._mpe_buf.data_ptr() + 8)
        with torch.cuda.stream(self.ctx.torch_stream):
            self._mpe_host.copy_(self._mpe_buf, non_blocking=True)
        self.ctx.sync()
        t2 = time.perf_counter()
        host = self._mpe_host.numpy()
        value = float(host[:2].view(np.float64)[0])
        assignment = host[2:].view(np.uint32)
        self.last_timing = {"plan_ms": (t1 - t0) * 1e3, "run_ms": (t2 - t1) * 1e3}
        return value, {v: int(assignment[v]) for v in map_vars}, (time.perf_counter() - t0) * 1e3

    def map_batch(self, map_vars, observed, values, heuristic="mf", host_values=None):
        """Marginal MAP for a batch of evidence sets sharing the observed ids, the batched counterpart of `map`.
        observed: sorted variable ids; values: torch.uint8 CUDA tensor [nb][len(observed)] (or host_values, a pinned
        uint8 tensor, to include the H2D copy).  -> (value [nb] float64, assignment [nvars][nb] uint8), device tensors:
        a MAP variable's row holds its decoded values, an observed variable's the evidence, a summed variable's 0xFF.
        Every set equals its single run of the same plan bit for bit.  The tensors are the model's result buffers
        for MAP batches of nb sets (see `mpe_batch`: synchronise before reading them elsewhere, clone to keep them)."""
        observed = list(observed)
        p = self._map_plan([int(v) for v in map_vars], observed, heuristic)
        with torch.cuda.stream(self.ctx.torch_stream):
            if host_values is not None:
                values = host_values.to(self._dev.device, non_blocking=True)
            nb = values.shape[0]
            out = self._batch_out.get(("map", nb))
            if out is None:
                out = self._batch_out[("map", nb)] = (torch.empty(nb, dtype=torch.float64, device=self._dev.device),
                                                       torch.empty((self.nvars, nb), dtype=torch.uint8, device=self._dev.device))
        p.run_mpe_batched(self.table_ptrs, nb, values.data_ptr(), out[0].data_ptr(), out[1].data_ptr())
        self._keep_alive = values
        return out

    def partition_batch(self, observed, values, heuristic="mf", host_values=None):
        """PR for a batch of evidence sets sharing the observed ids (config 5).
        observed: sorted variable ids; values: torch.uint8 CUDA tensor [nb][len(observed)] (or pass
        host_values, a pinned uint8 tensor, to include the H2D copy).  -> device tensor [nb] of Z.
        The returned tensor is the model's result buffer for batches of nb sets, written on the context's stream:
        synchronise (`ctx.sync()`) before reading it on another stream, and clone it if it must survive the next call
        with the same nb (stable pointers are what lets the library replay the run as a graph)."""
        observed = list(observed)
        # one plan per (observed ids, heuristic): the order depends on the ids only, so repeated batches over the same
        # ids pay neither the host ordering nor the planning again (drop_plans() forgets it)
        bkey = (tuple(observed), heuristic)
        p = self._batch_plans.get(bkey)
        if p is None:
            variables = [v for v in range(self.nvars) if v not in set(observed)]
            order, _ = self.order(variables, observed, heuristic)
            p = self._batch_plans[bkey] = self.plan(observed, order)
        assert p.result_size == 1
        with torch.cuda.stream(self.ctx.torch_stream):
            if host_values is not None:
                values = host_values.to(self._dev.device, non_blocking=True)
            nb = values.shape[0]
            # one result buffer per batch size, reused: stable pointers let the library replay the run as a graph
            out = self._batch_out.get(nb)
            if out is None:
                out = self._batch_out[nb] = torch.empty(nb, dtype=torch.float64, device=self._dev.device)
        p.run_batched(self.table_ptrs, nb, values.data_ptr(), out.data_ptr())
        self._keep_alive = values
        return out

    def mpe_batch(self, observed, values, heuristic="mf", host_values=None):
        """MPE for a batch of evidence sets sharing the observed ids, the batched counterpart of `mpe`.
        observed: sorted variable ids; values: torch.uint8 CUDA tensor [nb][len(observed)] (or pass host_values, a pinned
        uint8 tensor, to include the H2D copy).  -> (value [nb] float64, assignment [nvars][nb] uint8), device tensors;
        every set's value and assignment equal `mpe` for its evidence (an out-of-range value is read as 0 and raises
        BNPP_STATUS_BAD_EVIDENCE, see ctx.status()).
        The returned tensors are the model's result buffers for batches of nb sets, written on the context's stream:
        synchronise (`ctx.sync()`) before reading them on another stream, and clone them if they must survive the next
        call with the same nb (stable pointers are what lets the library replay the run as a graph)."""
        observed = list(observed)
        bkey = ("mpe", tuple(observed), heuristic)
        p = self._batch_plans.get(bkey)
        if p is None:
            variables = [v for v in range(self.nvars) if v not in set(observed)]
            order, _ = self.order(variables, observed, heuristic)
            p = self._batch_plans[bkey] = self._cached_plan(("mpe", tuple(observed), tuple(order)), MPEPlan, observed, order)
        with torch.cuda.stream(self.ctx.torch_stream):
            if host_values is not None:
                values = host_values.to(self._dev.device, non_blocking=True)
            nb = values.shape[0]
            out = self._batch_out.get(("mpe", nb))
            if out is None:
                out = self._batch_out[("mpe", nb)] = (torch.empty(nb, dtype=torch.float64, device=self._dev.device),
                                                       torch.empty((self.nvars, nb), dtype=torch.uint8, device=self._dev.device))
        p.run_mpe_batched(self.table_ptrs, nb, values.data_ptr(), out[0].data_ptr(), out[1].data_ptr())
        self._keep_alive = values
        return out

    def marginals_fast(self, evidence=None, heuristic="mf", comm=None):
        """every marginal from ONE bucket-tree plan (two passes) instead of one VE pass per variable;
        same tables as `marginals` up to rounding.  -> list of arrays ([1.0] for observed variables).
        comm: the network sharded over the ranks (see `partition`): unnormalised slices P(v, e, shard = rank's values)
        are summed over NVLink, then normalised; the shard variables' own marginals come from the ranks' partitions."""
        evidence = dict(evidence or {})
        if comm is not None and comm.world > 1:
            return self._marginals_sharded(evidence, heuristic, comm)
        observed = sorted(evidence)
        variables = [v for v in range(self.nvars) if v not in evidence]
        order, _ = self.order(variables, evidence, heuristic)
        key = ("mar", tuple(observed), tuple(order))
        p = self._plans.get(key)
        if p is None:
            p = MarPlan(self.ctx, self.cards, self.scopes, observed, order, _arr=self._scope_arr)
            self._plans[key] = p
        with torch.cuda.stream(self.ctx.torch_stream):
            res = torch.empty(max(1, p.result_size), dtype=torch.float64, device=self._dev.device)
        p.run(self.table_ptrs, [evidence[v] for v in observed], res.data_ptr(), None)
        self.ctx.sync()
        host = res.cpu().numpy()
        return [host[o:o + n] for o, n in zip(p.off, p.size)]

    def _marginals_sharded(self, evidence, heuristic, comm):
        from . import sharding
        full, shard_vars = self.shard(evidence, heuristic, comm)
        observed = sorted(full)
        variables = [v for v in range(self.nvars) if v not in full]
        order, _ = self.order(variables, full, heuristic)
        key = ("mar", tuple(observed), tuple(order))
        p = self._plans.get(key)
        if p is None:
            p = MarPlan(self.ctx, self.cards, self.scopes, observed, order, _arr=self._scope_arr)
            self._plans[key] = p
        n = max(1, p.result_size)
        z_rank, _ = self.partition(full, heuristic)            # this rank's slab: P(evidence, shard variables = its values)
        with torch.cuda.stream(self.ctx.torch_stream):
            res = torch.zeros(n + 1 + comm.world, dtype=torch.float64, device=self._dev.device)
            res[n] = z_rank
            res[n + 1 + comm.rank] = z_rank
        # slices weighted by the rank's partition, summed over NVLink, divided by the total (bnpp_ve_plan_run_sharded)
        comm.run_sharded(p, self.table_ptrs, [full[v] for v in observed], res.data_ptr(), res.data_ptr() + 8 * n)
        comm.allreduce_sum(res.data_ptr() + 8 * (n + 1), comm.world)      # every rank's Z, for the shard variables' own marginals
        self.ctx.sync()
        host = res.cpu().numpy()
        out = [host[o:o + s_].copy() for o, s_ in zip(p.off, p.size)]
        zr = host[n + 1:n + 1 + comm.world]
        for v in shard_vars:
            m = np.zeros(self.cards[v])
            for r in range(comm.world):
                m[sharding.shard_evidence(shard_vars, r)[v]] += zr[r]
            out[v] = m / zr.sum()
        return out

    def marginals(self, evidence=None, heuristic=None):
        """BN::marginals, VE branch (code/model.cpp:320-339): one VE pass per variable, normalised.
        Observed variables are dropped from the ordering input (the reference crashes there, SURVEY A.2 i)."""
        evidence = dict(evidence or {})
        out = []
        for v in range(self.nvars):
            variables = [u for u in range(self.nvars) if u != v and u not in evidence]
            order, _ = self.order(variables, evidence, heuristic)
            scope, cards, res = self.variable_elimination(evidence, order)
            n = res.numel() - 1
            with torch.cuda.stream(self.ctx.torch_stream):
                nrm = torch.empty(n, dtype=torch.float64, device=res.device)
            self.ctx.normalize(n, res.data_ptr(), nrm.data_ptr(), z_ptr=res.data_ptr() + 8 * n)
            out.append(nrm)
        self.ctx.sync()
        return [t.cpu().numpy() for t in out]

    def sum_product(self, max_sweeps=10000, epsilon=0.001):
        """BN::sum_product (code/model.cpp:736-753): evidence is ignored, as in the reference"""
        from .sumproduct import FactorGraph
        hv = self._host.numpy()
        facs = [(sc, hv[o:o + n]) for sc, o, n in zip(self.scopes, self._offs, self._sizes)]
        fg = FactorGraph(self.ctx, self.cards, facs)
        sweeps = fg.update(max_sweeps, epsilon)
        return fg, sweeps

    def drop_plans(self):
        """forget every cached plan (and free its arena): the next query orders and plans from scratch"""
        for p in self._plans.values():
            p.close()
        self._plans = {}
        self._batch_plans = {}
        self._order_cache = {}

    def close(self):
        self.drop_plans()


def from_uai_text(ctx, text):
    """read_uai_model for tests/bench (the parser itself is the reference's host glue, code/io.cpp:43-100)"""
    toks = []
    for line in text.splitlines():
        for t in line.split():
            if t.startswith("#"):
                break
            toks.append(t)
    it = iter(toks)
    kind = next(it)
    n = int(next(it))
    cards = [int(next(it)) for _ in range(n)]
    m = int(next(it))
    scopes = []
    for _ in range(m):
        w = int(next(it))
        scopes.append([int(next(it)) for _ in range(w)])
    factors = []
    for sc in scopes:
        sz = int(next(it))
        factors.append((sc, np.array([float(next(it)) for _ in range(sz)])))
    return kind, BN(ctx, cards, factors)


class Sampler:
    """bnpp_sampler: forward sampling of a Bayesian network on the GPU (BN::logical_sampling / BN::likelihood_weighting,
    code/model.cpp:540-690).  Factor i must be the CPT of variable i with the child first in its scope."""

    def __init__(self, bn):
        self.bn, self.ctx = bn, bn.ctx
        L = self.ctx.L
        P = ctypes.POINTER
        L.bnpp_sampler_create.argtypes = [ctypes.c_void_p, ctypes.c_int, capi.c_u32p, P(capi.Scope), capi.c_u32p,
                                          P(ctypes.c_void_p), P(ctypes.c_void_p)]
        L.bnpp_sampler_destroy.argtypes = [ctypes.c_void_p]
        L.bnpp_sampler_logical.argtypes = [ctypes.c_void_p, ctypes.c_int, capi.c_u32p, capi.c_u32p, ctypes.c_uint64,
                                           ctypes.c_uint64, capi.c_u64p]
        L.bnpp_sampler_likelihood.argtypes = [ctypes.c_void_p, ctypes.c_int, capi.c_u32p, capi.c_u32p, ctypes.c_double,
                                              ctypes.c_double, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64,
                                              ctypes.POINTER(ctypes.c_double), capi.c_u64p]
        n = bn.nvars
        assert len(bn.scopes) == n and all(sc[0] == v for v, sc in enumerate(bn.scopes)), "factor i must be the CPT of variable i"
        # topological order: parents before children (any such order samples the same distribution)
        order, done = [], set()
        while len(order) < n:
            before = len(order)
            for v in range(n):
                if v not in done and all(p in done for p in bn.scopes[v][1:]):
                    order.append(v)
                    done.add(v)
            assert len(order) > before, "cyclic network"
        od = capi._u32(order)
        tp = (ctypes.c_void_p * n)(*bn.table_ptrs)
        h = ctypes.c_void_p()
        self.ctx.check(L.bnpp_sampler_create(self.ctx.h, n, ctypes.cast(bn._cards_arr, capi.c_u32p), bn._scope_arr,
                                             ctypes.cast(od, capi.c_u32p), tp, ctypes.byref(h)))
        self.h = h

    def _ev(self, evidence):
        ev = sorted(evidence.items())
        return len(ev), capi._u32([e[0] for e in ev]), capi._u32([e[1] for e in ev])

    def logical(self, evidence, n_samples, seed=1):
        """-> estimate of P(evidence) = hits / n_samples"""
        k, a, b = self._ev(evidence)
        hits = ctypes.c_uint64()
        self.ctx.check(self.ctx.L.bnpp_sampler_logical(self.h, k, ctypes.cast(a, capi.c_u32p), ctypes.cast(b, capi.c_u32p),
                                                       int(n_samples), int(seed), ctypes.byref(hits)))
        return hits.value / n_samples

    def likelihood(self, evidence, u_bound, n_star, seed=1, batch=1 << 14, max_samples=1 << 30):
        """-> (estimate of P(evidence) = U * N / M, samples used M)"""
        k, a, b = self._ev(evidence)
        n, m = ctypes.c_double(), ctypes.c_uint64()
        self.ctx.check(self.ctx.L.bnpp_sampler_likelihood(self.h, k, ctypes.cast(a, capi.c_u32p), ctypes.cast(b, capi.c_u32p),
                                                          float(u_bound), float(n_star), int(batch), int(max_samples), int(seed),
                                                          ctypes.byref(n), ctypes.byref(m)))
        return u_bound * n.value / m.value, m.value

    def close(self):
        if self.h:
            self.ctx.L.bnpp_sampler_destroy(self.h)
            self.h = None
