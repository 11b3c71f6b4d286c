"""Python mirror of `bn::Factor` (reference code/factor.hh:10-48) over the C ABI.

Used by the tests and bench.py to drive the CUDA path with the reference's own
vocabulary: a factor is a scope (variable ids, last fastest) plus a dense fp64 table
resident in HBM; every operation returns a new factor and its partition
(code/factor.cpp:117-255).  The table and its partition live in ONE device
allocation of size+1 doubles (partition last), so nothing returns to the host until
`values()` / `partition` is asked for.
"""
import numpy as np
import torch

from . import capi


class DeviceFactor:
    def __init__(self, ctx, scope, cards, buf):
        self.ctx = ctx
        self.scope = [int(v) for v in scope]
        self.cards = [int(c) for c in cards]
        self.buf = buf                    # torch.float64 cuda tensor, size + 1 entries
        self.size = int(np.prod(self.cards, dtype=np.uint64)) if self.cards else 1
        assert buf.numel() == self.size + 1

    # ---- construction --------------------------------------------------------
    @staticmethod
    def empty(ctx, scope, cards):
        n = int(np.prod([int(c) for c in cards], dtype=np.uint64)) if len(cards) else 1
        with torch.cuda.stream(ctx.torch_stream):
            buf = torch.empty(n + 1, dtype=torch.float64, device="cuda:%d" % ctx.device)
        return DeviceFactor(ctx, scope, cards, buf)

    @staticmethod
    def from_host(ctx, scope, cards, values, partition=None):
        """Factor(domain, values, partition), code/factor.cpp:12-16"""
        values = np.ascontiguousarray(values, dtype=np.float64).reshape(-1)
        f = DeviceFactor.empty(ctx, scope, cards)
        assert values.size == f.size
        host = np.empty(f.size + 1)
        host[:-1] = values
        host[-1] = float(np.sum(values)) if partition is None else partition
        with torch.cuda.stream(ctx.torch_stream):
            f.buf.copy_(torch.from_numpy(host), non_blocking=False)
        return f

    @property
    def ptr(self):
        return self.buf.data_ptr()

    @property
    def zptr(self):
        return self.buf.data_ptr() + 8 * self.size

    @property
    def width(self):
        return len(self.scope)

    # ---- host reads (synchronise) ---------------------------------------------
    def values(self):
        self.ctx.sync()
        return self.buf[:-1].cpu().numpy()

    @property
    def partition(self):
        self.ctx.sync()
        return float(self.buf[-1].item())

    def _card_of(self, other):
        m = dict(zip(self.scope, self.cards))
        m.update(zip(other.scope, other.cards))
        return m

    # ---- ops, code/factor.cpp:117-255 ------------------------------------------
    def product(self, other, divide=False):
        ids, cards = capi.union_scope(self.scope, self.cards, other.scope, other.cards)
        out = DeviceFactor.empty(self.ctx, ids, cards)
        self.ctx.product(self.ptr, self.scope, self.cards, other.ptr, other.scope, other.cards, out.ptr, out.zptr,
                         divide=divide)
        return out

    def divide(self, other):
        return self.product(other, divide=True)

    def sum_out(self, var):
        if var in self.scope:
            keep = [(v, c) for v, c in zip(self.scope, self.cards) if v != var]
        else:
            keep = list(zip(self.scope, self.cards))
        out = DeviceFactor.empty(self.ctx, [k[0] for k in keep], [k[1] for k in keep])
        self.ctx.sum_out(self.ptr, self.scope, self.cards, var, out.ptr, out.zptr)
        if var not in self.scope:
            # the reference deep-copies, partition included (code/factor.cpp:185-188)
            with torch.cuda.stream(self.ctx.torch_stream):
                out.buf[-1:].copy_(self.buf[-1:])
        return out

    def condition(self, evidence):
        keep = [(v, c) for v, c in zip(self.scope, self.cards) if v not in evidence]
        out = DeviceFactor.empty(self.ctx, [k[0] for k in keep], [k[1] for k in keep])
        self.ctx.condition(self.ptr, self.scope, self.cards, evidence, out.ptr, out.zptr)
        return out

    def normalize(self):
        out = DeviceFactor.empty(self.ctx, self.scope, self.cards)
        self.ctx.normalize(self.size, self.ptr, out.ptr, z_ptr=self.zptr)
        self.ctx.fill(out.zptr, 1, 1.0)     # code/factor.cpp:252
        return out

    def _reduce(self, op, init=0.0):
        with torch.cuda.stream(self.ctx.torch_stream):
            r = torch.empty(1, dtype=torch.float64, device=self.buf.device)
        self.ctx.reduce(op, self.size, self.ptr, r.data_ptr(), init)
        self.ctx.sync()
        return float(r.item())

    def max(self):
        return self._reduce("max")

    def min(self):
        return self._reduce("min", self.partition)

    def sum(self):
        return self._reduce("sum")


def fused_product_sum_out(ctx, factors, out_scope, elim_var):
    """One elimination step (code/model.cpp:414-418) in one kernel; `out_scope` fixes the output layout."""
    cards = {}
    for f in factors:
        cards.update(zip(f.scope, f.cards))
    out = DeviceFactor.empty(ctx, out_scope, [cards[v] for v in out_scope])
    ctx.product_sum_out([(f.ptr, f.scope, f.cards, None) for f in factors], out.scope, out.cards, elim_var,
                        out.ptr, out.zptr)
    return out


def fused_product_max_out(ctx, factors, out_scope, elim_var):
    """One max-product step (MPE) in one kernel -> (factor over `out_scope` holding max_x of the product, device uint8
    tensor of the first maximising x per entry).  The factor's partition slot is not written."""
    cards = {}
    for f in factors:
        cards.update(zip(f.scope, f.cards))
    out = DeviceFactor.empty(ctx, out_scope, [cards[v] for v in out_scope])
    with torch.cuda.stream(ctx.torch_stream):
        arg = torch.empty(max(1, out.size), dtype=torch.uint8, device=out.buf.device)
    ctx.product_max_out([(f.ptr, f.scope, f.cards, None) for f in factors], out.scope, out.cards, elim_var,
                        out.ptr, arg.data_ptr())
    return out, arg[:out.size]
