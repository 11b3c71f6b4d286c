/* bnpp_b200.h -- C ABI of the B200-native factor-algebra hot path of bn-pp.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  bn-pp has no FFI of its own: the
 * boundary is what sits UNDER its public C++ classes `bn::Factor` / `bn::Domain`
 * (code/factor.hh:10-48, code/domain.hh:11-45) and under the inner loops of
 * `BN::variable_elimination` (code/model.cpp:348-446) and `FactorGraph::update`
 * (code/graph.cpp:298-403).  Every entry point below names the reference code it
 * replaces.  Plain pointers and sizes only; no C++ or torch types.
 *
 * Conventions
 *   - All tables are dense fp64, row-major with the LAST scope variable fastest
 *     (code/domain.cpp:20-24).  A scope is (rank, var_id[], card[]).
 *   - `double *` table arguments are DEVICE pointers (from bnpp_alloc or any CUDA
 *     allocation on the context's device, e.g. a torch tensor's data_ptr()).
 *   - `z_dev`, when non-NULL, is a DEVICE pointer to one double that receives the
 *     result's partition  Z = sum of its entries  (code/factor.cpp:139,172,204,234),
 *     reduced in a fixed order (bit-stable across runs).
 *   - Calls are asynchronous on the context's stream; bnpp_download and
 *     bnpp_ctx_sync synchronise.  One host thread per context (SURVEY §8b threading).
 *   - Every function returns 0 on success or a negative BNPP_E* code; no exceptions
 *     cross the ABI.  bnpp_last_error gives the message.  There is NO CPU fallback:
 *     without a usable CUDA device every compute call fails with BNPP_ECUDA.
 */
#ifndef BNPP_B200_H_
#define BNPP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BNPP_OK        0
#define BNPP_EINVAL   -1   /* malformed scope / operand (variable in neither output nor eliminated, ...) */
#define BNPP_ECUDA    -2   /* CUDA runtime error (message in bnpp_last_error) */
#define BNPP_ERANK    -3   /* more than BNPP_MAX_AXES non-mergeable axes or BNPP_MAX_OPERANDS operands */
#define BNPP_ETOOBIG  -4   /* a table has >= 2^32 entries (the reference's `unsigned` limit, code/domain.hh:41-42) */
#define BNPP_ENOMEM   -5

#define BNPP_MAX_RANK      64   /* scope width accepted at the ABI */
#define BNPP_MAX_AXES      32   /* iteration axes left after merging contiguous ones */
#define BNPP_MAX_OPERANDS   6   /* operands of one fused elimination step */

/* status bits accumulated on the device, read with bnpp_ctx_status */
#define BNPP_STATUS_ZERO_DIVISOR 1u   /* code/factor.cpp:169 asserts on this */
#define BNPP_STATUS_BAD_EVIDENCE 2u   /* a batched evidence value >= its variable's cardinality (replaced by 0); code/factor.cpp:83-95 throws */

typedef struct bnpp_ctx bnpp_ctx;

/* Layout of a dense table: the reference's Domain (code/domain.cpp:15-26). */
typedef struct {
    int32_t rank;
    const uint32_t *var_id;   /* [rank] scope order, last fastest */
    const uint32_t *card;     /* [rank] */
} bnpp_scope;

/* One operand of a contraction: a (possibly strided / sliced / permuted) view of a
 * device table.  stride == NULL means dense row-major over `scope`.  Evidence
 * reduction (code/factor.cpp:214-242) is expressed as a view: observed axes are
 * dropped from the scope and their offset folded into `data`. */
typedef struct {
    const double *data;
    bnpp_scope scope;
    const int64_t *stride;    /* [rank] in elements, or NULL */
} bnpp_operand;

/* ---- context, memory -------------------------------------------------------- */
/* stream: a cudaStream_t to launch on (e.g. torch's current stream), or NULL to
 * create a private non-blocking stream. */
int bnpp_ctx_create(int device, void *stream, bnpp_ctx **out);
int bnpp_ctx_destroy(bnpp_ctx *ctx);
int bnpp_ctx_sync(bnpp_ctx *ctx);
int bnpp_ctx_status(bnpp_ctx *ctx, uint32_t *status_bits, int clear);   /* synchronises */
const char *bnpp_last_error(const bnpp_ctx *ctx);
int bnpp_version(void);
/* number of kernels this context has launched (bench.py's gpu_launches) */
uint64_t bnpp_launch_count(const bnpp_ctx *ctx);
/* name, grid and block of the most recent contraction launch (diagnostics / tests) */
int bnpp_last_launch(const bnpp_ctx *ctx, char *name, size_t name_len, uint32_t *grid, uint32_t *block);

/* Kernel-selection knobs, process wide (tests and profiling; the defaults are the product):
 *   "mv_min_entries" : union entries from which an elimination of a variable with > 2 values takes the tiled
 *                      multi-valued kernel (contract_mv; default 2^15, 0 = always)
 *   "mv_emax"        : union entries per tile of the gather variant of that kernel (64..2048; 0 = default)
 *   "mv_staged"      : 1 (default) = operands whose tile footprint is a compact range are staged in shared memory
 *                      by bulk copies (contract_mvt); 0 = always the gather variant (contract_mv)
 *   "staged_tma"     : 1 (default) = the tile of a transposed operand of a binary elimination comes in by bulk copies
 *                      of its contiguous runs (contract_staged_bulk); 0 = element-wise cp.async (contract_staged)
 *   "staged_async"   : 1 (default) = in that kernel the other operands are prefetched too (cp.async, a ring of stages)
 *                      when their micro-tiles are at most two values; 0 = loaded into registers chunk by chunk
 *   "chain_depth"    : levels of a window of a VE plan (runs of wide binary eliminations as one contract_chain launch,
 *                      intermediates in registers), read when a plan is created; default 4; 0 or 1 = no windows
 * Unknown keys return BNPP_EINVAL.  Environment BNPP_MV_MIN_ENTRIES / BNPP_MV_EMAX / BNPP_STAGED_TMA / BNPP_STAGED_ASYNC /
 * BNPP_CHAIN_DEPTH seed the defaults. */
int bnpp_tuning_set(const char *key, uint64_t value);
int bnpp_tuning_get(const char *key, uint64_t *value);

int bnpp_alloc(bnpp_ctx *ctx, uint64_t n_doubles, double **dptr);     /* stream-ordered pool */
int bnpp_free(bnpp_ctx *ctx, double *dptr);
int bnpp_upload(bnpp_ctx *ctx, double *dst_dev, const double *src_host, uint64_t n);   /* async if src is pinned */
int bnpp_download(bnpp_ctx *ctx, double *dst_host, const double *src_dev, uint64_t n); /* synchronises */
int bnpp_fill(bnpp_ctx *ctx, double *dst_dev, uint64_t n, double value);   /* Factor(domain, value), code/factor.cpp:18-23 */

/* ---- scope helpers (host only; no device needed) ------------------------------ */
/* code/domain.cpp:32-52: d1 in order, then d2-only variables in d2 order.
 * out arrays must hold a.rank + b.rank entries; returns the union rank. */
int bnpp_union_scope(const bnpp_scope *a, const bnpp_scope *b, uint32_t *out_var_id, uint32_t *out_card);
/* code/domain.cpp:15-26: product of the cardinalities; 0 on overflow of 2^64 */
uint64_t bnpp_scope_size(const bnpp_scope *s);

/* ---- the fused elimination step (K3; also the engine under every op below) ---- */
/* out[o] = sum_{x < card(elim_var)}  prod_k  operand_k[ pi_k(o, x) ]
 * Replaces `prod *= *pf` over a bucket followed by `prod.sum_out(var)`
 * (code/model.cpp:414-418) without materialising the product.
 *   elim_var  < 0 : no variable is summed out (pure k-ary product).
 *   divide != 0   : k must be 2; computes operand_0 / operand_1 (code/factor.cpp:149-180);
 *                   a zero divisor sets BNPP_STATUS_ZERO_DIVISOR.
 * Every operand variable must be in `out` or be elim_var.  `out` is dense over
 * out_scope, in ANY axis order the caller chooses. */
int bnpp_product_sum_out(bnpp_ctx *ctx, int k, const bnpp_operand *operands,
                         const bnpp_scope *out_scope, int64_t elim_var, int divide,
                         double *out_dev, double *z_dev);

/* Max-product step (MPE; no reference counterpart):
 *   out[o] = max_x prod_k operand_k[pi_k(o, x)],  arg[o] = the first x attaining it (uint8)
 * Products are formed as in bnpp_product_sum_out.  The maximum starts at x = 0 and x replaces it
 * only if its product is strictly greater: ties keep the lowest x and a NaN never replaces a
 * number.  argmax_dev is dense over out_scope like out_dev.  elim_var < 0 or an eliminated
 * variable with more than 255 values returns BNPP_EINVAL.  No partition is computed. */
int bnpp_product_max_out(bnpp_ctx *ctx, int k, const bnpp_operand *operands, const bnpp_scope *out_scope,
                         int64_t elim_var, double *out_dev, uint8_t *argmax_dev);

/* ---- reference-shaped single ops ---------------------------------------------- */
/* Factor::product / Factor::divide, code/factor.cpp:117-180. out is dense over
 * bnpp_union_scope(a, b). */
int bnpp_product(bnpp_ctx *ctx, const bnpp_scope *sa, const double *a_dev,
                 const bnpp_scope *sb, const double *b_dev, int divide,
                 double *out_dev, double *z_dev);
/* Factor::sum_out, code/factor.cpp:182-212. out is dense over `s` minus var (order
 * kept); if var is not in scope the table is copied (code/factor.cpp:185-188). */
int bnpp_sum_out(bnpp_ctx *ctx, const bnpp_scope *s, const double *in_dev, uint32_t var,
                 double *out_dev, double *z_dev);
/* Factor::conditioning, code/factor.cpp:214-242. Observed variables (ev_var/ev_val
 * pairs; ids not in scope are ignored) are pinned, free axes keep their order. */
int bnpp_condition(bnpp_ctx *ctx, const bnpp_scope *s, const double *in_dev,
                   int n_ev, const uint32_t *ev_var, const uint32_t *ev_val,
                   double *out_dev, double *z_dev);
/* Factor::normalize, code/factor.cpp:244-255: out[i] = in[i] / Z with TRUE division.
 * Z is *z_dev when z_dev != NULL (device-resident, no sync) else z_host. */
int bnpp_normalize(bnpp_ctx *ctx, uint64_t n, const double *in_dev, const double *z_dev, double z_host,
                   double *out_dev);
/* Factor::max (starts from 0.0), Factor::min (starts from the partition),
 * code/factor.cpp:97-115, and the plain sum (`partition +=` lines).
 * op: 0 = sum, 1 = max, 2 = min.  init is the min's start value. result_dev: device double. */
int bnpp_reduce(bnpp_ctx *ctx, int op, uint64_t n, const double *in_dev, double init, double *result_dev);

/* ---- device-resident variable elimination -------------------------------------- */
/* Graph::ordering / min_fill / weighted_min_fill / min_degree (code/graph.cpp:41-195) on
 * the HOST with the reference's tie-breaks (libstdc++ unordered_set iteration order).
 *   scopes  : ORIGINAL factor scopes; obs_var[n_obs] are removed from them first, which
 *             is the graph BN::partition builds from its conditioned factors
 *             (code/model.cpp:283-287, 362);
 *   vars    : the variables to order, in the caller's order (observed ones are dropped:
 *             the reference crashes on them, SURVEY A.2 i);
 *   heuristic: 0 = min-fill, 1 = weighted min-fill, 2 = min-degree; | 0x100 selects the
 *             slow implementation on the reference's own containers (cross-check).
 * order_out must hold n_vars_to_order ids; *n_order_out receives the count.  Needs no device. */
int bnpp_elim_order(int nvars, const uint32_t *card, int nfac, const bnpp_scope *scopes, int n_obs,
                    const uint32_t *obs_var, int n_vars_to_order, const uint32_t *vars, int heuristic,
                    uint32_t *order_out, uint32_t *n_order_out, uint32_t *width_out);
/* Constrained elimination order for marginal MAP (no reference counterpart): `first` (the summed
 * variables) ordered exactly as bnpp_elim_order orders them, then `last` (the MAP variables) ordered
 * by the same heuristic on the same conditioned graph with the fill edges of the first phase in
 * place.  heuristic | 0x100 as for bnpp_elim_order.  order_out must hold n_first + n_last ids;
 * *width_out receives the width over both phases.  Needs no device. */
int bnpp_elim_order_constrained(int nvars, const uint32_t *card, int nfac, const bnpp_scope *scopes, int n_obs,
                                const uint32_t *obs_var, int n_first, const uint32_t *first, int n_last,
                                const uint32_t *last, int heuristic, uint32_t *order_out, uint32_t *n_order_out,
                                uint32_t *width_out);
/* Wide-factor sharding over G = 2^g GPUs (SURVEY §8e; no reference counterpart): the g variables of
 * the widest elimination clique that `order` eliminates last.  Every rank then runs the ordinary
 * plan with these variables observed at its rank's values; bnpp_shard_allreduce_sum
 * (bnpp_b200_nccl.h) sums them out across ranks.  Host only; returns how many were written. */
int bnpp_pick_shard_vars(int nfac, const bnpp_scope *scopes, int n_order, const uint32_t *order, int g, uint32_t *out);
/* Graph::order_width, code/graph.cpp:197-237 (host). */
int bnpp_order_width(int nvars, const uint32_t *card, int nfac, const bnpp_scope *scopes, int n_order,
                     const uint32_t *order, uint32_t *width_out);

/* BN::variable_elimination (code/model.cpp:348-446) over resident tables, preceded by
 * the conditioning of every factor (code/model.cpp:283-286) expressed as views.
 *   scopes[nfac]  : ORIGINAL scopes of the dense input tables;
 *   obs_var[n_obs]: observed variables -- their VALUES are given per run;
 *   order[n_order]: elimination order over unobserved variables.  Unobserved variables
 *                   not in `order` are kept: the result is a table over them, ascending
 *                   variable id, last fastest (the reference leaves this order to a
 *                   pointer-keyed hash set, SURVEY A.4).
 * One plan serves any number of runs (other evidence values, other table contents).
 * ctx may be NULL: a DRY plan -- planning is host work -- that can be inspected (info, layout,
 * fused_info, fused_program) but not run (the run entry points return BNPP_EINVAL). */
typedef struct bnpp_ve_plan bnpp_ve_plan;
int bnpp_ve_plan_create(bnpp_ctx *ctx, int nfac, const bnpp_scope *scopes, int n_obs, const uint32_t *obs_var,
                        int n_order, const uint32_t *order, bnpp_ve_plan **out);
int bnpp_ve_plan_destroy(bnpp_ve_plan *plan);
/* result scope (arrays of BNPP_MAX_RANK), kernel launches per run, sum over elimination
 * steps of the union-table entries (the "factor entries" of BASELINE.json's metric), the
 * algorithmic bytes 8*(sum #operands + #out) over all launches, peak bytes of live
 * intermediates, and the largest step.  Any pointer may be NULL. */
int bnpp_ve_plan_info(const bnpp_ve_plan *plan, int32_t *result_rank, uint32_t *result_var, uint32_t *result_card,
                      uint64_t *n_launches, uint64_t *union_entries, uint64_t *algorithmic_bytes,
                      uint64_t *peak_bytes, uint64_t *max_step_entries);
/* tables_dev[nfac]: device tables; obs_val[n_obs]: evidence values; result_dev: device
 * buffer of the result's size; z_dev: optional device double for its partition.  Asynchronous.
 * An evidence value >= its variable's cardinality returns BNPP_EINVAL (the reference throws from
 * Factor::operator[], code/factor.cpp:83-95). */
int bnpp_ve_plan_run(bnpp_ve_plan *plan, const double *const *tables_dev, const uint32_t *obs_val,
                     double *result_dev, double *z_dev);
/* MPE (no reference counterpart): the most probable assignment of every unobserved variable given
 * the evidence, and its value  max_x prod_f f(x, e)  -- P(x*, e) for a Bayesian network, not
 * normalised.  The steps are those bnpp_ve_plan_create builds for the same inputs with every sum
 * replaced by a max (rule of bnpp_product_max_out); each eliminating step keeps its argmax table
 * (one byte per output entry, counted in peak_bytes) and a one-thread decode walks them backwards.
 * `order` must cover every unobserved variable that some scope mentions, and an eliminated
 * variable may have at most 255 values; else BNPP_EINVAL.  ctx may be NULL (a dry plan).
 * Single runs are launch-per-bucket (never the K9 / K10 paths); from the second run on a run is one
 * replay of a CUDA graph that includes the decode.  Batches: bnpp_mpe_plan_run_batched.
 * run: assignment_dev[nvars] receives one uint32 per variable id: the evidence value for an
 * observed variable, 0 for a variable no factor mentions; value_dev one double.  Zero-probability
 * evidence gives value 0 and the lowest values.  An evidence value out of range returns
 * BNPP_EINVAL.  bnpp_ve_plan_run / _run_batched / _run_sharded return BNPP_EINVAL on an MPE plan; one network sharded
 * over several GPUs runs with bnpp_mpe_plan_run_sharded of bnpp_b200_nccl.h. */
int bnpp_mpe_plan_create(bnpp_ctx *ctx, int nvars, const uint32_t *card, int nfac, const bnpp_scope *scopes,
                         int n_obs, const uint32_t *obs_var, int n_order, const uint32_t *order, bnpp_ve_plan **out);
/* Marginal MAP (no reference counterpart): the jointly most probable assignment of the MAP variables
 * map_var[n_map] given the evidence, every other unobserved variable summed out, and its value
 * max_{x_M} sum_{x_S} prod_f f(x, e)  -- P(x_M*, e) for a Bayesian network, not normalised.  The steps
 * are those of bnpp_ve_plan_create for the same order; a step eliminating a MAP variable is a max step
 * (rule and argmax table of bnpp_product_max_out), every other eliminating step sums.  The argmax
 * arena, the argmax rows of batches (R_s: the sum of n_out over the MAX steps before s) and the decode
 * cover the max steps only.  The order must eliminate every summed variable before any MAP variable
 * (constrained elimination: bnpp_elim_order_constrained), which makes the result exact.  M = every
 * unobserved variable gives the MPE plan of bnpp_mpe_plan_create; M empty gives the value of
 * bnpp_ve_plan_run for the same order.  BNPP_EINVAL when a MAP variable is observed, repeated,
 * >= nvars or has more than 255 values (summed variables may have any), when the order misses an
 * unobserved variable that some scope mentions, or when it names a MAP variable before a summed one.
 * ctx may be NULL (a dry plan).  Run it with bnpp_mpe_plan_run / bnpp_mpe_plan_run_batched: a MAP
 * variable reports its decoded value (0 if no factor mentions it), an observed variable its evidence
 * value, a summed variable BNPP_ASSIGN_SUMMED in the element type (uint32 0xFFFFFFFF, batch uint8 0xFF). */
#define BNPP_ASSIGN_SUMMED 0xFFFFFFFFu
int bnpp_map_plan_create(bnpp_ctx *ctx, int nvars, const uint32_t *card, int nfac, const bnpp_scope *scopes,
                         int n_obs, const uint32_t *obs_var, int n_map, const uint32_t *map_var, int n_order,
                         const uint32_t *order, bnpp_ve_plan **out);
/* run an MPE or MAP plan for one evidence set (see above) */
int bnpp_mpe_plan_run(bnpp_ve_plan *plan, const double *const *tables_dev, const uint32_t *obs_val,
                      double *value_dev, uint32_t *assignment_dev);
/* the nvars an MPE or MAP plan was created with (the length of its assignment); BNPP_EINVAL for any other plan */
int bnpp_mpe_plan_nvars(const bnpp_ve_plan *plan, uint32_t *nvars);
/* Max-loc over the ranks of a sharded MPE or MAP query (bnpp_mpe_plan_run_sharded, bnpp_b200_nccl.h), one block of one
 * launch (kernel mpe_shard_select).  records_dev holds nranks records of stride = 2 + nvars rounded up to an even number
 * of uint32 words; rank r's starts at word r * stride: its value (a double, words 0-1, 8-byte aligned) and its assignment
 * (nvars uint32, words 2..) -- what bnpp_mpe_plan_run writes.  The winner is the largest value; equal values keep the
 * lowest rank and a NaN never replaces a number (the rule of bnpp_product_max_out over the ranks: rank 0 first, a later
 * rank replaces it only if strictly greater).  Its value goes to value_dev, its assignment to assignment_dev[nvars].
 * Asynchronous on the context's stream.  nranks == 0, nvars == 0 or a NULL pointer returns BNPP_EINVAL. */
int bnpp_mpe_shard_select(bnpp_ctx *ctx, uint32_t nranks, uint32_t nvars, const uint32_t *records_dev, double *value_dev,
                          uint32_t *assignment_dev);
/* MPE or MAP for a BATCH of evidence sets over one MPE or MAP plan: ev_dev [nb][n_obs] uint8 as for
 * bnpp_ve_plan_run_batched; value_dev receives [nb] doubles, assignment_dev [nvars][nb] uint8 (batch
 * fastest).  Every set's value and assignment equal, bit for bit, what bnpp_mpe_plan_run returns for its
 * evidence: the observed variables report the values the set was computed with, a variable no factor
 * mentions reports 0.  A value >= its variable's cardinality is read as 0 (and reported as 0) and raises
 * BNPP_STATUS_BAD_EVIDENCE.  Engines as for batched PR: the whole plan in one launch per slice (K9,
 * ve_fused_max; a MAP plan with both max and summing steps ve_fused_mixed) when fused_info accepts the
 * plan for nb > 1 sets, else one launch per bucket (K8's max-product variants for max steps, its sum
 * kernels for the others, replayed as a captured graph from the third run with the same buffers on);
 * bnpp_ve_plan_set_fused(plan, 0) forces K8.  A decode launch per slice, one thread per set, follows.
 * A MAP plan's summed variables report 0xFF.
 * Argmax layout, shared by both engines: max step s (plan order, bnpp_ve_plan_describe; every eliminating
 * step of an MPE plan) owns the rows [R_s, R_s + n_out_s) of a plan-owned byte scratch, R_s = the sum of
 * n_out over the max steps before it; the argmax of its output entry o for set b of a slice of `slice` sets is at byte
 * (R_s + o) * slice + b.  Batches are cut into slices so that the scratch stays within 1 GiB (K8: also its
 * widest intermediate).  A plan that is neither MPE nor MAP, an n_obs other than the plan's, a NULL buffer or nb == 0 returns
 * BNPP_EINVAL. */
int bnpp_mpe_plan_run_batched(bnpp_ve_plan *plan, const double *const *tables_dev, uint32_t nb, uint32_t n_obs,
                              const uint8_t *ev_dev, double *value_dev, uint8_t *assignment_dev);
/* entries of the result table a run writes (PR: 1; marginals plan: the layout's total) */
int bnpp_ve_plan_result_size(const bnpp_ve_plan *plan, uint64_t *n);
/* BN::marginals (code/model.cpp:320-339) for EVERY variable in one plan: two passes over the
 * bucket tree of `order` (which must cover all unobserved variables) instead of one VE pass
 * per variable.  Run it with bnpp_ve_plan_run: result_dev receives, per variable id
 * ascending, card(v) normalised doubles -- or a single 1.0 for an observed variable or one no
 * factor mentions (the reference returns the width-0 factor [1] there).  bnpp_mar_plan_layout
 * gives each variable's offset and size and the total. */
int bnpp_mar_plan_create(bnpp_ctx *ctx, int nvars, const uint32_t *card, int nfac, const bnpp_scope *scopes, int n_obs,
                         const uint32_t *obs_var, int n_order, const uint32_t *order, bnpp_ve_plan **out);
int bnpp_mar_plan_layout(const bnpp_ve_plan *plan, int nvars, uint32_t *off, uint32_t *size, uint64_t *total);
/* A marginals plan normalises every slice at the end of a run, single or batched.  set_normalize(plan, 0)
 * leaves the slices unnormalised (P(v, evidence) -- what a sharded run sums over the ranks before it
 * normalises, bnpp_b200_nccl.h); bnpp_mar_plan_normalize then normalises the result buffer of a SINGLE
 * run in place (it does not know a batch's [result_size][nb] layout). */
int bnpp_ve_plan_set_normalize(bnpp_ve_plan *plan, int on);
int bnpp_mar_plan_normalize(bnpp_ve_plan *plan, double *result_dev);

/* K8 -- the same plan for a BATCH of evidence sets (BASELINE config 5): ev_dev is a device
 * matrix [nb][n_obs] of evidence values (uint8, column j = obs_var[j] of the plan);
 * result_dev receives [result_size][nb] doubles, batch fastest (PR: one double per set).
 * One launch per bucket for the whole batch; CPTs are shared, never copied per set.
 * n_obs must equal the plan's; a value >= its variable's cardinality is treated as 0 and raises
 * BNPP_STATUS_BAD_EVIDENCE (bnpp_ctx_status).
 * A marginals plan: entry i of the layout (bnpp_mar_plan_layout) for set b at result_dev[i * nb + b], and
 * each set's column equals, bit for bit, what bnpp_ve_plan_run returns for its evidence -- normalised
 * slices (NaN where P(evidence) = 0, as 0/0 in the single run), 1.0 in the one-entry slices.  With
 * set_normalize(plan, 0) the slices of more than one entry hold the single run's unnormalised values
 * and the one-entry slices are not written. */
int bnpp_ve_plan_run_batched(bnpp_ve_plan *plan, const double *const *tables_dev, uint32_t nb, uint32_t n_obs,
                             const uint8_t *ev_dev, double *result_dev);
/* K9 -- a plan whose elimination steps are all small (every union table <= 2^14 entries: the
 * shipped toy networks, config 1/2 queries, config 5 batches) runs as ONE launch: a group of
 * lanes owns an evidence set and walks the bucket loop of code/model.cpp:409-439 with the
 * intermediates of the set in shared memory; results are bit-identical to the launch-per-bucket
 * path.  On by default (environment BNPP_FUSED=0 turns it off for new plans); set_fused(plan, 0)
 * forces one launch per bucket.  On an MPE or MAP plan it selects the engine of bnpp_mpe_plan_run_batched
 * only (single MPE / MAP runs are always launch-per-bucket), and fused_info / fused_program describe the
 * max-mode program (fused.hpp: kFusedMax steps carry their first argmax row R_s in header word 7; in a MAP
 * program exactly the max steps carry the flag).  fused_info: lanes per evidence set a run over nb sets would use
 * (0 = not fused), shared-memory doubles per set, steps in the launch. */
int bnpp_ve_plan_set_fused(bnpp_ve_plan *plan, int on);
int bnpp_ve_plan_fused_info(bnpp_ve_plan *plan, uint32_t nb, int32_t *lanes_per_set, uint32_t *arena_doubles,
                            uint32_t *n_steps);
/* the step program of a fused run (format: bnpp_b200/csrc/fused.hpp) for inspection; CPT operand
 * records carry the input-table index (word 1) and 0xffffffff (word 3) instead of an address.
 * Pass NULL buffers to query the sizes.  Works on dry plans (created with ctx == NULL). */
int bnpp_ve_plan_fused_program(bnpp_ve_plan *plan, uint32_t nb, uint32_t *prog, uint64_t prog_cap, uint64_t *prog_words,
                               uint32_t *offtab, uint64_t tab_cap, uint64_t *tab_words);
/* The whole schedule as numbers (every launch's operands and output, where each intermediate lives in the plan's
 * arena), for inspection and for CPU emulation of the HOST logic (bucket schedule, small-table folding, arena
 * lifetimes) on dry plans; the word stream is documented at the definition in bnpp_b200/csrc/ve.cu.  Pass buf = NULL
 * to query the size. */
int bnpp_ve_plan_describe(const bnpp_ve_plan *plan, uint64_t *buf, uint64_t cap, uint64_t *words);
/* K10 -- TASKS, on by default (environment BNPP_FUSED_SEGMENTS=0 turns it off for new plans): a plan that is not one
 * launch altogether (K9) is cut into tasks -- subtrees of the bucket tree whose steps are all small, each run by one
 * CTA with its intermediates in shared memory -- and all tasks of one dependency level form ONE launch (ve_tasks);
 * wide steps stay their own launches, and every launch is a node of the replay graph.  Replaces the loop of
 * code/model.cpp:409-439 for mixed plans (Munin*, Link, Pigs, andes: ~1000 tiny buckets -> a few dozen launches).
 * set_segments(plan, on, max_steps): max_steps > 0 limits the steps per task (tests); only before the first run can
 * the tasks be re-cut.  _segments lists the tasks (a contiguous step range each), _segment_program dumps one task's
 * program like _fused_program (0xfffffffe in an address's high word: the intermediate with that index in the plan's
 * global arena), _launches counts the kernel launches of a single-query run. */
int bnpp_ve_plan_set_segments(bnpp_ve_plan *plan, int on, uint32_t max_steps);
int bnpp_ve_plan_segments(bnpp_ve_plan *plan, uint32_t cap, uint32_t *n, uint32_t *first_step, uint32_t *end_step,
                          int32_t *lanes, uint32_t *arena_doubles);
int bnpp_ve_plan_launches(bnpp_ve_plan *plan, uint64_t *launches, uint32_t *groups, uint32_t *levels);
/* windows of a VE plan (one contract_chain launch each): the first step and the number of steps of each */
int bnpp_ve_plan_windows(const bnpp_ve_plan *plan, uint32_t cap, uint32_t *n, uint32_t *first_step, uint32_t *n_steps);
int bnpp_ve_plan_segment_program(bnpp_ve_plan *plan, uint32_t segment, uint32_t *prog, uint64_t prog_cap, uint64_t *prog_words,
                                 uint32_t *offtab, uint64_t tab_cap, uint64_t *tab_words);
/* per-launch CUDA-event timing for roofline reports: enable, run, then read
 * ms / algorithmic bytes / union entries / operand count per launch (synchronises). */
int bnpp_ve_plan_set_profiling(bnpp_ve_plan *plan, int on);
int bnpp_ve_plan_step_stats(bnpp_ve_plan *plan, uint64_t n, float *ms, uint64_t *bytes, uint64_t *entries, int32_t *k);
/* kernel variant the last profiled run used for launch `step` (diagnostics) */
int bnpp_ve_plan_step_kernel(const bnpp_ve_plan *plan, uint64_t step, char *name, size_t name_len);

/* ---- factor-graph sum-product (K7), code/graph.cpp:256-403 --------------------- */
typedef struct bnpp_fg bnpp_fg;
/* Builds the device edge tables once.  Factor f has scope
 * fscope[foff[f] .. foff[f+1]) and a dense table of host doubles at ftab + toff[f].
 * Messages start uniform 1/card (code/graph.cpp:261-274). */
int bnpp_fg_create(bnpp_ctx *ctx, int nvars, const uint32_t *card, int nfac,
                   const int32_t *foff, const uint32_t *fscope,
                   const uint64_t *toff, const double *ftab_host, bnpp_fg **out);
int bnpp_fg_destroy(bnpp_fg *fg);
/* One sweep = all variable->factor updates, then all factor->variable updates
 * (code/graph.cpp:298-326); *maxerror_host receives the sweep's max relative change
 * (NaN ignored, inf kept, code/graph.cpp:349-356).  Synchronises. */
int bnpp_fg_sweep(bnpp_fg *fg, double *maxerror_host);
/* FactorGraph::update(max, epsilon), code/graph.cpp:298-332: *sweeps receives the
 * 0-based index of the converging sweep, or max_sweeps.  The whole loop is ONE cooperative launch (both
 * phases of every sweep separated by grid barriers, convergence test and sweep counter on the device); the
 * host reads the count once.  Synchronises. */
int bnpp_fg_update(bnpp_fg *fg, uint32_t max_sweeps, double epsilon, uint32_t *sweeps);
/* messages back to the uniform start (code/graph.cpp:261-274), e.g. before a second update() */
int bnpp_fg_reset(bnpp_fg *fg);
/* FactorGraph::marginal for every variable (code/graph.cpp:393-403):
 * out_host[moff_var[v] .. +card[v]) with moff_var the exclusive prefix sum of card. */
int bnpp_fg_marginals(bnpp_fg *fg, double *out_host);

/* ---- forward sampling (SURVEY 8f row 4), code/model.cpp:540-690 over code/factor.cpp:257-288 ------------ */
/* One thread per sample walks the variables in the reference's topological order (`order`, variable ids) and draws
 * each from its CPT given the sampled parents -- Factor::sampling -- with a counter-based generator keyed by
 * (seed, sample index): reproducible where the reference (std::random_device per draw) is not.
 *   scopes[nvars]    : factor i is the CPT of variable i, scope[0] the child, then its parents (code/model.cpp:111-119)
 *   tables_dev[nvars]: the resident CPT of every variable (at most 2048 variables of at most 255 values) */
typedef struct bnpp_sampler bnpp_sampler;
int bnpp_sampler_create(bnpp_ctx *ctx, int nvars, const uint32_t *card, const bnpp_scope *scopes, const uint32_t *order,
                        const double *const *tables_dev, bnpp_sampler **out);
int bnpp_sampler_destroy(bnpp_sampler *s);
/* BN::logical_sampling, code/model.cpp:540-560: *hits of n_samples forward samples agree with the evidence. */
int bnpp_sampler_logical(bnpp_sampler *s, int n_ev, const uint32_t *ev_var, const uint32_t *ev_val, uint64_t n_samples,
                         uint64_t seed, uint64_t *hits);
/* BN::likelihood_weighting, code/model.cpp:620-690 (bounded variance): evidence variables are clamped, a sample
 * weighs W = the product of their CPT entries; samples are consumed IN ORDER until the sum of W / u_bound reaches
 * n_star (or max_samples).  *n_sum = that sum, *m = samples used; the estimate is u_bound * n_sum / m.  `batch`
 * samples are drawn per launch; the answer does not depend on it. */
int bnpp_sampler_likelihood(bnpp_sampler *s, int n_ev, const uint32_t *ev_var, const uint32_t *ev_val, double u_bound,
                            double n_star, uint64_t batch, uint64_t max_samples, uint64_t seed, double *n_sum, uint64_t *m);

#ifdef __cplusplus
}
#endif
#endif /* BNPP_B200_H_ */
