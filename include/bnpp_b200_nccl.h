/* bnpp_b200_nccl.h -- the one collective of the path (SURVEY.md §8e), in its own library
 * (libbnpp_b200_nccl.so) so that the core library has no NCCL dependency.
 *
 * A factor too wide for one GPU is sharded by the variables of its widest clique that the
 * order eliminates last (bnpp_pick_shard_vars in bnpp_b200.h); every rank eliminates its own
 * slab with the ordinary plan, treating the shard variables as observed at its rank's
 * values.  Summing the shard variables out is then the ONLY cross-GPU step of the query:
 * an all-reduce (fp64 sum) of each rank's result over NVLink.  Maximising them out (MPE,
 * marginal MAP) is an all-gather of every rank's value and assignment and a max-loc on the
 * device.  The reference has no counterpart (single process, single thread).
 */
#ifndef BNPP_B200_NCCL_H_
#define BNPP_B200_NCCL_H_

#include "bnpp_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* In-place sum over all ranks of buf_dev[0..n) (doubles), enqueued on the context's stream.
 * nccl_comm is an ncclComm_t created by the caller (one rank per GPU). */
int bnpp_shard_allreduce_sum(bnpp_ctx *ctx, void *nccl_comm, double *buf_dev, uint64_t n);

/* BN::partition / variable_elimination / marginals of ONE network sharded over the ranks of nccl_comm
 * (code/model.cpp:275-294, 320-339, 348-446; the reference has no multi-process form).  `plan` is this rank's
 * bnpp_ve_plan (or marginals plan) created with the shard variables (bnpp_pick_shard_vars) among its
 * observed ids, obs_val holds the evidence values and THIS RANK's values of the shard variables.  Every
 * rank runs its slab, then the result tables (bnpp_ve_plan_result_size doubles: the scalar P(e) for a
 * partition plan, a table over the kept variables otherwise) and *z_dev are summed over all ranks in place
 * -- the cross-shard sum-out -- so every rank ends with the result of the unsharded query.
 * A marginals plan returns normalised slices, so for it *z_dev must hold THIS RANK's partition
 * P(evidence, shard variables = its values) on entry (run the rank's partition plan first): the slices are weighted
 * by it, summed over the ranks and divided by the sum of the partitions (*z_dev on return).  The slices of the shard
 * variables themselves hold 1 (each rank sees them observed): their marginals follow from the ranks' partitions.
 * Asynchronous on the context's stream. */
int bnpp_ve_plan_run_sharded(bnpp_ctx *ctx, bnpp_ve_plan *plan, void *nccl_comm, const double *const *tables_dev,
                             const uint32_t *obs_val, double *result_dev, double *z_dev);

/* MPE or marginal MAP of ONE network sharded over the ranks of nccl_comm.  `plan` is this rank's MPE or MAP plan
 * (bnpp_mpe_plan_create / bnpp_map_plan_create; ctx must be its context) created with the shard variables among its
 * observed ids -- for MAP they must be MAP variables: a rank's value max_{M \ shard} sum_S is maximised over the ranks,
 * which is exact only for maximised shard variables -- and obs_val holds the evidence and THIS RANK's shard values.
 * Every rank runs bnpp_mpe_plan_run into its record (stride = 2 + nvars words rounded up to even, in a buffer of
 * world * stride words from the context's pool), the records are all-gathered in place (ncclAllGather), and
 * bnpp_mpe_shard_select (bnpp_b200.h) picks the largest value -- the lowest rank on ties, never a NaN over a number --
 * and writes its value and assignment to value_dev / assignment_dev[nvars] on every rank.  The shard variables report
 * the winning rank's values.  Asynchronous on the context's stream.  A PR or marginals plan or a NULL argument returns
 * BNPP_EINVAL. */
int bnpp_mpe_plan_run_sharded(bnpp_ctx *ctx, bnpp_ve_plan *plan, void *nccl_comm, const double *const *tables_dev,
                              const uint32_t *obs_val, double *value_dev, uint32_t *assignment_dev);

#ifdef __cplusplus
}
#endif
#endif
