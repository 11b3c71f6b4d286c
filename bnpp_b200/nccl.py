"""The path's one collective through the product's own C ABI (include/bnpp_b200_nccl.h).

`ShardComm` owns an ncclComm_t (one rank per GPU) and sums a device buffer over all ranks with
bnpp_shard_allreduce_sum -- the cross-shard sum-out of wide-factor sharding -- or, for MPE and marginal MAP, gathers
every rank's value and assignment and keeps the best (bnpp_mpe_plan_run_sharded).  The unique id
travels over torch.distributed (plumbing); the reduction itself does not go through torch.
"""
import ctypes
import os

from . import capi

_HERE = os.path.dirname(os.path.abspath(__file__))


class _UniqueId(ctypes.Structure):
    _fields_ = [("internal", ctypes.c_char * 128)]


class ShardComm:
    def __init__(self, ctx, rank=0, world=1):
        import torch.distributed as dist
        self.ctx = ctx
        self.rank, self.world = rank, world
        self.nccl = ctypes.CDLL("libnccl.so.2")
        self.lib = ctypes.CDLL(os.path.join(_HERE, "libbnpp_b200_nccl.so"))
        self.lib.bnpp_shard_allreduce_sum.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64]
        uid = _UniqueId()
        if rank == 0:
            rc = self.nccl.ncclGetUniqueId(ctypes.byref(uid))
            assert rc == 0, "ncclGetUniqueId failed (%d)" % rc
        if world > 1:
            # all 128 bytes: a c_char array field would stop at the first NUL
            box = [ctypes.string_at(ctypes.byref(uid), 128) if rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            ctypes.memmove(ctypes.byref(uid), box[0], 128)
        self.comm = ctypes.c_void_p()
        self.nccl.ncclCommInitRank.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int, _UniqueId, ctypes.c_int]
        rc = self.nccl.ncclCommInitRank(ctypes.byref(self.comm), world, uid, rank)
        assert rc == 0, "ncclCommInitRank failed (%d)" % rc

    def run_sharded(self, plan, table_ptrs, obs_val, result_ptr, z_ptr=None):
        """bnpp_ve_plan_run_sharded: this rank's slab of the plan, then the cross-shard sum-out of result and partition"""
        n = len(table_ptrs)
        tp = (ctypes.c_void_p * max(1, n))(*table_ptrs)
        ov = capi._u32(obs_val)
        self.lib.bnpp_ve_plan_run_sharded.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p),
                                                      capi.c_u32p, ctypes.c_void_p, ctypes.c_void_p]
        self.ctx.check(self.lib.bnpp_ve_plan_run_sharded(self.ctx.h, plan.h, self.comm, tp, ctypes.cast(ov, capi.c_u32p),
                                                         ctypes.c_void_p(result_ptr), ctypes.c_void_p(z_ptr) if z_ptr else None))

    def run_mpe_sharded(self, plan, table_ptrs, obs_val, value_ptr, assignment_ptr):
        """bnpp_mpe_plan_run_sharded: this rank's slab of an MPE or MAP plan, then the all-gather of every rank's value
        and assignment and the max-loc over them; every rank receives the winner's (value_ptr: device double,
        assignment_ptr: device uint32 [nvars]).  Asynchronous."""
        tp = (ctypes.c_void_p * max(1, len(table_ptrs)))(*table_ptrs)
        ov = capi._u32(obs_val)
        self.lib.bnpp_mpe_plan_run_sharded.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                                       ctypes.POINTER(ctypes.c_void_p), capi.c_u32p, ctypes.c_void_p,
                                                       ctypes.c_void_p]
        self.ctx.check(self.lib.bnpp_mpe_plan_run_sharded(self.ctx.h, plan.h, self.comm, tp, ctypes.cast(ov, capi.c_u32p),
                                                          ctypes.c_void_p(value_ptr), ctypes.c_void_p(assignment_ptr)))

    def allreduce_sum(self, ptr, n):
        """in place, on the context's stream"""
        self.ctx.check(self.lib.bnpp_shard_allreduce_sum(self.ctx.h, self.comm, ctypes.c_void_p(ptr), int(n)))

    def close(self):
        if self.comm:
            self.nccl.ncclCommDestroy.argtypes = [ctypes.c_void_p]
            self.nccl.ncclCommDestroy(self.comm)
            self.comm = None
