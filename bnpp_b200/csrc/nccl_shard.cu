// The cross-shard steps of wide-factor sharding: one NCCL all-reduce (fp64 sum) of the ranks' results over NVLink /
// NVSwitch, or for MPE / MAP one all-gather of their (value, assignment) records.  See include/bnpp_b200_nccl.h.
#include <nccl.h>

#include "../../include/bnpp_b200_nccl.h"
#include "common.cuh"

extern "C" int bnpp_shard_allreduce_sum(bnpp_ctx *ctx, void *nccl_comm, double *buf_dev, uint64_t n)
{
    if (!ctx || !nccl_comm || !buf_dev) return BNPP_EINVAL;
    const ncclResult_t r = ncclAllReduce(buf_dev, buf_dev, n, ncclDouble, ncclSum, static_cast<ncclComm_t>(nccl_comm), ctx->stream);
    if (r != ncclSuccess) {
        ctx->last_error = std::string("ncclAllReduce: ") + ncclGetErrorString(r);
        return BNPP_ECUDA;
    }
    return BNPP_OK;
}

// One network sharded over the ranks of `nccl_comm` (wide-factor sharding, SURVEY 8e): the plan was created with
// the shard variables among its observed ids; every rank runs it with its own values for them, then the ranks'
// result tables -- P(kept variables, evidence, shard variables = this rank's values) -- are summed over NVLink:
// the cross-shard sum-out.
// A marginals plan hands back NORMALISED slices (each bucket's product is normalised on its own, so a slice does
// not carry the weight of the other connected components): the slices of rank r are therefore weighted by that
// rank's partition Z_r = P(evidence, shard variables = r's values), which the caller passes in *z_dev (from the
// rank's partition plan), summed over the ranks together with the Z_r, and divided by the total.
extern "C" int bnpp_ve_plan_run_sharded(bnpp_ctx *ctx, bnpp_ve_plan *plan, void *nccl_comm, const double *const *tables_dev,
                                        const uint32_t *obs_val, double *result_dev, double *z_dev)
{
    if (!ctx || !plan || !nccl_comm || !result_dev) return BNPP_EINVAL;
    uint64_t n = 0, total = 0;
    int rc = bnpp_ve_plan_result_size(plan, &n);
    if (rc != BNPP_OK) return rc;
    const bool is_mar = bnpp_mar_plan_layout(plan, 0, nullptr, nullptr, &total) == BNPP_OK;
    if (is_mar && !z_dev) {
        ctx->last_error = "sharded marginals: z_dev must hold this rank's partition on entry";
        return BNPP_EINVAL;
    }
    rc = bnpp_ve_plan_run(plan, tables_dev, obs_val, result_dev, is_mar ? nullptr : z_dev);
    if (rc != BNPP_OK) return rc;
    if (is_mar) {
        // result[i] *= Z_r : a product with the width-0 factor [Z_r] (Factor::product, code/factor.cpp:117-147)
        if (n >= (1ull << 32)) return BNPP_ETOOBIG;
        uint32_t id = 0, card = (uint32_t)n;
        bnpp_operand ops[2];
        ops[0].data = result_dev;
        ops[0].scope.rank = 1;
        ops[0].scope.var_id = &id;
        ops[0].scope.card = &card;
        ops[0].stride = nullptr;
        ops[1].data = z_dev;
        ops[1].scope.rank = 0;
        ops[1].scope.var_id = nullptr;
        ops[1].scope.card = nullptr;
        ops[1].stride = nullptr;
        rc = bnpp_product_sum_out(ctx, 2, ops, &ops[0].scope, -1, 0, result_dev, nullptr);
        if (rc != BNPP_OK) return rc;
    }
    ncclComm_t comm = static_cast<ncclComm_t>(nccl_comm);
    ncclResult_t r = ncclGroupStart();
    if (r == ncclSuccess) r = ncclAllReduce(result_dev, result_dev, n, ncclDouble, ncclSum, comm, ctx->stream);
    if (r == ncclSuccess && z_dev && !(z_dev >= result_dev && z_dev < result_dev + n))
        r = ncclAllReduce(z_dev, z_dev, 1, ncclDouble, ncclSum, comm, ctx->stream);
    const ncclResult_t r2 = ncclGroupEnd();
    if (r == ncclSuccess) r = r2;
    if (r != ncclSuccess) {
        ctx->last_error = std::string("ncclAllReduce: ") + ncclGetErrorString(r);
        return BNPP_ECUDA;
    }
    if (is_mar) return bnpp_normalize(ctx, n, result_dev, z_dev, 0.0, result_dev);     // / sum of the Z_r: true division
    return BNPP_OK;
}

// MPE / MAP of one sharded network: the cross-shard step of a max is a max, and the winner's assignment must travel
// with its value.  NCCL has no max-loc, so every rank gathers every rank's (value, assignment) record and one small
// kernel of the core library picks the winner -- the same on every rank, since all of them see the same records.
extern "C" int bnpp_mpe_plan_run_sharded(bnpp_ctx *ctx, bnpp_ve_plan *plan, void *nccl_comm, const double *const *tables_dev,
                                         const uint32_t *obs_val, double *value_dev, uint32_t *assignment_dev)
{
    if (!ctx || !plan || !nccl_comm || !value_dev || !assignment_dev) return BNPP_EINVAL;
    uint32_t nvars = 0;
    if (bnpp_mpe_plan_nvars(plan, &nvars) != BNPP_OK) {
        ctx->last_error = "bnpp_mpe_plan_run_sharded: not an MPE or MAP plan";
        return BNPP_EINVAL;
    }
    ncclComm_t comm = static_cast<ncclComm_t>(nccl_comm);
    int rank = 0, world = 0;
    ncclResult_t r = ncclCommUserRank(comm, &rank);
    if (r == ncclSuccess) r = ncclCommCount(comm, &world);
    if (r != ncclSuccess) {
        ctx->last_error = std::string("ncclCommUserRank / ncclCommCount: ") + ncclGetErrorString(r);
        return BNPP_ECUDA;
    }
    const uint64_t stride = (2ull + nvars + 1) & ~1ull;       // even: every record's value stays 8-byte aligned
    double *buf = nullptr;
    int rc = bnpp_alloc(ctx, (uint64_t)world * stride / 2, &buf);
    if (rc != BNPP_OK) return rc;
    uint32_t *records = reinterpret_cast<uint32_t *>(buf);
    uint32_t *mine = records + (uint64_t)rank * stride;
    rc = bnpp_mpe_plan_run(plan, tables_dev, obs_val, reinterpret_cast<double *>(mine), mine + 2);
    if (rc == BNPP_OK) {
        r = ncclAllGather(mine, records, stride, ncclUint32, comm, ctx->stream);
        if (r != ncclSuccess) {
            ctx->last_error = std::string("ncclAllGather: ") + ncclGetErrorString(r);
            rc = BNPP_ECUDA;
        }
    }
    if (rc == BNPP_OK) rc = bnpp_mpe_shard_select(ctx, (uint32_t)world, nvars, records, value_dev, assignment_dev);
    const int rc_free = bnpp_free(ctx, buf);
    return rc != BNPP_OK ? rc : rc_free;
}
