"""ctypes binding of the C ABI in include/bnpp_b200.h (libbnpp_b200.so).

PyTorch is used only as plumbing: device memory (`torch.empty(..., device="cuda")`),
the current CUDA stream and events.  All arithmetic happens in the hand-written
sm_100a kernels behind the ABI.  There is no fallback: if the shared library is
missing or no CUDA device is usable, the calls raise.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbnpp_b200.so")

c_u32p = ctypes.POINTER(ctypes.c_uint32)
c_i32p = ctypes.POINTER(ctypes.c_int32)
c_i64p = ctypes.POINTER(ctypes.c_int64)
c_u64p = ctypes.POINTER(ctypes.c_uint64)
c_f64p = ctypes.POINTER(ctypes.c_double)

EXPORTS = [
    "bnpp_version", "bnpp_ctx_create", "bnpp_ctx_destroy", "bnpp_ctx_sync", "bnpp_ctx_status", "bnpp_last_error",
    "bnpp_launch_count", "bnpp_last_launch", "bnpp_alloc", "bnpp_free", "bnpp_upload", "bnpp_download", "bnpp_fill",
    "bnpp_union_scope", "bnpp_scope_size", "bnpp_product_sum_out", "bnpp_product", "bnpp_sum_out", "bnpp_condition",
    "bnpp_normalize", "bnpp_reduce", "bnpp_fg_create", "bnpp_fg_destroy", "bnpp_fg_sweep", "bnpp_fg_update",
    "bnpp_fg_marginals", "bnpp_elim_order", "bnpp_order_width", "bnpp_ve_plan_create", "bnpp_ve_plan_destroy",
    "bnpp_ve_plan_info", "bnpp_ve_plan_run", "bnpp_ve_plan_run_batched", "bnpp_ve_plan_set_profiling",
    "bnpp_ve_plan_step_stats", "bnpp_ve_plan_step_kernel", "bnpp_ve_plan_set_fused", "bnpp_ve_plan_fused_info", "bnpp_ve_plan_fused_program", "bnpp_ve_plan_describe", "bnpp_ve_plan_set_segments", "bnpp_ve_plan_segments", "bnpp_ve_plan_segment_program", "bnpp_mar_plan_create", "bnpp_mar_plan_layout", "bnpp_pick_shard_vars",
    "bnpp_tuning_set", "bnpp_tuning_get", "bnpp_ve_plan_result_size", "bnpp_ve_plan_set_normalize",
    "bnpp_mar_plan_normalize", "bnpp_fg_reset", "bnpp_ve_plan_launches",
    "bnpp_sampler_create", "bnpp_sampler_destroy", "bnpp_sampler_logical", "bnpp_sampler_likelihood",
    "bnpp_product_max_out", "bnpp_mpe_plan_create", "bnpp_mpe_plan_run", "bnpp_mpe_plan_run_batched",
    "bnpp_elim_order_constrained", "bnpp_map_plan_create", "bnpp_mpe_plan_nvars", "bnpp_mpe_shard_select",
    "bnpp_ve_plan_windows",
]


def tuning_set(key, value):
    """process-wide kernel-selection knob (bnpp_tuning_set); returns the previous value"""
    L = lib()
    L.bnpp_tuning_set.argtypes = [ctypes.c_char_p, ctypes.c_uint64]
    L.bnpp_tuning_get.argtypes = [ctypes.c_char_p, c_u64p]
    old = ctypes.c_uint64()
    if L.bnpp_tuning_get(key.encode(), ctypes.byref(old)) != 0 or L.bnpp_tuning_set(key.encode(), int(value)) != 0:
        raise BnppError(-1, "unknown tuning key %r" % key)
    return old.value


class Scope(ctypes.Structure):
    _fields_ = [("rank", ctypes.c_int32), ("var_id", c_u32p), ("card", c_u32p)]


class Operand(ctypes.Structure):
    _fields_ = [("data", ctypes.c_void_p), ("scope", Scope), ("stride", c_i64p)]


class BnppError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("bnpp_b200 error %d: %s" % (code, msg))
        self.code = code


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("bnpp_b200: %s is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); "
                               "there is no CPU fallback" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        L.bnpp_last_error.restype = ctypes.c_char_p
        L.bnpp_last_error.argtypes = [ctypes.c_void_p]
        L.bnpp_launch_count.restype = ctypes.c_uint64
        L.bnpp_launch_count.argtypes = [ctypes.c_void_p]
        L.bnpp_scope_size.restype = ctypes.c_uint64
        L.bnpp_ctx_create.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p)]
        L.bnpp_ctx_destroy.argtypes = [ctypes.c_void_p]
        L.bnpp_ctx_sync.argtypes = [ctypes.c_void_p]
        L.bnpp_ctx_status.argtypes = [ctypes.c_void_p, c_u32p, ctypes.c_int]
        L.bnpp_last_launch.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_size_t, c_u32p, c_u32p]
        L.bnpp_alloc.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.POINTER(ctypes.c_void_p)]
        L.bnpp_free.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.bnpp_upload.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64]
        L.bnpp_download.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64]
        L.bnpp_fill.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_double]
        L.bnpp_union_scope.argtypes = [ctypes.POINTER(Scope), ctypes.POINTER(Scope), c_u32p, c_u32p]
        L.bnpp_scope_size.argtypes = [ctypes.POINTER(Scope)]
        L.bnpp_product_sum_out.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(Operand), ctypes.POINTER(Scope),
                                           ctypes.c_int64, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
        L.bnpp_product_max_out.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(Operand), ctypes.POINTER(Scope),
                                           ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p]
        L.bnpp_product.argtypes = [ctypes.c_void_p, ctypes.POINTER(Scope), ctypes.c_void_p, ctypes.POINTER(Scope),
                                   ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
        L.bnpp_sum_out.argtypes = [ctypes.c_void_p, ctypes.POINTER(Scope), ctypes.c_void_p, ctypes.c_uint32,
                                   ctypes.c_void_p, ctypes.c_void_p]
        L.bnpp_condition.argtypes = [ctypes.c_void_p, ctypes.POINTER(Scope), ctypes.c_void_p, ctypes.c_int, c_u32p, c_u32p,
                                     ctypes.c_void_p, ctypes.c_void_p]
        L.bnpp_normalize.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_double,
                                     ctypes.c_void_p]
        L.bnpp_reduce.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_double,
                                  ctypes.c_void_p]
        L.bnpp_fg_create.argtypes = [ctypes.c_void_p, ctypes.c_int, c_u32p, ctypes.c_int, c_i32p, c_u32p, c_u64p, c_f64p,
                                     ctypes.POINTER(ctypes.c_void_p)]
        L.bnpp_fg_destroy.argtypes = [ctypes.c_void_p]
        L.bnpp_fg_sweep.argtypes = [ctypes.c_void_p, c_f64p]
        L.bnpp_fg_update.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_double, c_u32p]
        L.bnpp_fg_marginals.argtypes = [ctypes.c_void_p, c_f64p]
        _lib = L
    return _lib


def _u32(seq):
    arr = (ctypes.c_uint32 * max(1, len(seq)))(*[int(x) for x in seq])
    return arr


def make_scope(var_ids, cards):
    """-> (Scope, keepalive)"""
    v, c = _u32(var_ids), _u32(cards)
    return Scope(len(var_ids), ctypes.cast(v, c_u32p), ctypes.cast(c, c_u32p)), (v, c)


class Context:
    """One per device.  Kernels run on `self.torch_stream` (a torch.cuda.Stream created here, or the
    one passed in); record torch.cuda.Events on that stream to time them."""

    def __init__(self, device=0, stream=None):
        import torch
        self.L = lib()
        self.device = device
        handle = ctypes.c_void_p()
        if not torch.cuda.is_available():
            rc = self.L.bnpp_ctx_create(device, None, ctypes.byref(handle))   # fails loudly: no CPU fallback
            raise BnppError(rc, self.L.bnpp_last_error(None).decode())
        torch.cuda.set_device(device)
        self.torch_stream = stream if stream is not None else torch.cuda.Stream(device)
        stream = ctypes.c_void_p(self.torch_stream.cuda_stream)
        rc = self.L.bnpp_ctx_create(device, stream, ctypes.byref(handle))
        if rc != 0:
            raise BnppError(rc, self.L.bnpp_last_error(None).decode())
        self.h = handle

    def check(self, rc):
        if rc != 0:
            raise BnppError(rc, self.L.bnpp_last_error(self.h).decode())

    def close(self):
        if self.h:
            self.L.bnpp_ctx_destroy(self.h)
            self.h = None

    def sync(self):
        self.check(self.L.bnpp_ctx_sync(self.h))

    def status(self, clear=True):
        bits = ctypes.c_uint32()
        self.check(self.L.bnpp_ctx_status(self.h, ctypes.byref(bits), int(clear)))
        return bits.value

    @property
    def launches(self):
        return int(self.L.bnpp_launch_count(self.h))

    def last_launch(self):
        buf = ctypes.create_string_buffer(160)
        g, b = ctypes.c_uint32(), ctypes.c_uint32()
        self.L.bnpp_last_launch(self.h, buf, 160, ctypes.byref(g), ctypes.byref(b))
        return buf.value.decode(), g.value, b.value

    # ---- ops on raw device pointers (ints) ---------------------------------
    @staticmethod
    def _operands(operands, keep):
        ops = (Operand * len(operands))()
        for i, (ptr, ids, cards, strides) in enumerate(operands):
            sc, ka = make_scope(ids, cards)
            keep.append(ka)
            st = None
            if strides is not None:
                sa = (ctypes.c_int64 * max(1, len(strides)))(*[int(s) for s in strides])
                keep.append(sa)
                st = ctypes.cast(sa, c_i64p)
            ops[i] = Operand(ctypes.c_void_p(ptr), sc, st)
        return ops

    def product_sum_out(self, operands, out_ids, out_cards, elim_var, out_ptr, z_ptr=None, divide=False):
        """operands: list of (ptr, var_ids, cards, strides-or-None)"""
        k = len(operands)
        keep = []
        ops = self._operands(operands, keep)
        osc, ka = make_scope(out_ids, out_cards)
        self.check(self.L.bnpp_product_sum_out(self.h, k, ops, ctypes.byref(osc), -1 if elim_var is None else int(elim_var),
                                               int(divide), ctypes.c_void_p(out_ptr),
                                               ctypes.c_void_p(z_ptr) if z_ptr else None))

    def product_max_out(self, operands, out_ids, out_cards, elim_var, out_ptr, arg_ptr):
        """max-product step: out = max over elim_var of the product, arg (device uint8) = the first maximising value"""
        keep = []
        ops = self._operands(operands, keep)
        osc, ka = make_scope(out_ids, out_cards)
        self.check(self.L.bnpp_product_max_out(self.h, len(operands), ops, ctypes.byref(osc), int(elim_var),
                                               ctypes.c_void_p(out_ptr), ctypes.c_void_p(arg_ptr)))

    def product(self, a_ptr, a_ids, a_cards, b_ptr, b_ids, b_cards, out_ptr, z_ptr=None, divide=False):
        sa, k1 = make_scope(a_ids, a_cards)
        sb, k2 = make_scope(b_ids, b_cards)
        self.check(self.L.bnpp_product(self.h, ctypes.byref(sa), ctypes.c_void_p(a_ptr), ctypes.byref(sb),
                                       ctypes.c_void_p(b_ptr), int(divide), ctypes.c_void_p(out_ptr),
                                       ctypes.c_void_p(z_ptr) if z_ptr else None))

    def sum_out(self, ptr, ids, cards, var, out_ptr, z_ptr=None):
        s, k = make_scope(ids, cards)
        self.check(self.L.bnpp_sum_out(self.h, ctypes.byref(s), ctypes.c_void_p(ptr), int(var), ctypes.c_void_p(out_ptr),
                                       ctypes.c_void_p(z_ptr) if z_ptr else None))

    def condition(self, ptr, ids, cards, evidence, out_ptr, z_ptr=None):
        s, k = make_scope(ids, cards)
        ev = sorted(evidence.items())
        vs, vals = _u32([e[0] for e in ev]), _u32([e[1] for e in ev])
        self.check(self.L.bnpp_condition(self.h, ctypes.byref(s), ctypes.c_void_p(ptr), len(ev),
                                         ctypes.cast(vs, c_u32p), ctypes.cast(vals, c_u32p), ctypes.c_void_p(out_ptr),
                                         ctypes.c_void_p(z_ptr) if z_ptr else None))

    def normalize(self, n, in_ptr, out_ptr, z_ptr=None, z_host=1.0):
        self.check(self.L.bnpp_normalize(self.h, int(n), ctypes.c_void_p(in_ptr),
                                         ctypes.c_void_p(z_ptr) if z_ptr else None, float(z_host),
                                         ctypes.c_void_p(out_ptr)))

    def reduce(self, op, n, in_ptr, result_ptr, init=0.0):
        self.check(self.L.bnpp_reduce(self.h, {"sum": 0, "max": 1, "min": 2}[op], int(n), ctypes.c_void_p(in_ptr),
                                      float(init), ctypes.c_void_p(result_ptr)))

    def fill(self, ptr, n, value):
        self.check(self.L.bnpp_fill(self.h, ctypes.c_void_p(ptr), int(n), float(value)))


def union_scope(a_ids, a_cards, b_ids, b_cards):
    """code/domain.cpp:32-52 through the ABI (host only)"""
    sa, k1 = make_scope(a_ids, a_cards)
    sb, k2 = make_scope(b_ids, b_cards)
    n = len(a_ids) + len(b_ids)
    ids, cards = (ctypes.c_uint32 * max(1, n))(), (ctypes.c_uint32 * max(1, n))()
    w = lib().bnpp_union_scope(ctypes.byref(sa), ctypes.byref(sb), ctypes.cast(ids, c_u32p), ctypes.cast(cards, c_u32p))
    return list(ids[:w]), list(cards[:w])
