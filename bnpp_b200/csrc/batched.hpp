// Interface between the VE plan (ve.cu) and the batched-evidence kernel (batched.cu).
#pragma once
#include <cstdint>
#include <utility>
#include <vector>

struct bnpp_ctx;

namespace bnpp {

constexpr int kMaxObsPerOperand = 8;    // observed axes one K8 operand reads its evidence base through

// One operand of a batched elimination step: an intermediate [entries][batch] or a resident
// CPT view read through a per-evidence-set base offset.
struct BatchedOperandDesc {
    const double *ptr;
    bool batched;
    const std::vector<uint32_t> *var, *card;
    const std::vector<int64_t> *stride;              // empty => dense
    const std::vector<std::pair<int64_t, int>> *obs; // (stride, evidence column) of observed axes
};

int contract_batched_step(bnpp_ctx *ctx, int k, const BatchedOperandDesc *ops, const std::vector<uint32_t> &out_var,
                          const std::vector<uint32_t> &out_card, int64_t elim, uint32_t nb, const uint8_t *ev_dev,
                          uint32_t ev_stride, uint32_t n_obs, double *out_dev, std::vector<uint32_t> *offtab_host,
                          uint32_t **offtab_dev, uint8_t *arg_dev = nullptr);
// arg_dev != nullptr and elim >= 0: a max-product step (MPE), the first maximising value of the eliminated variable for
// output entry o and set b at arg_dev[o * nb + b]
// ev_dev above is COLUMN-major ([n_obs][ev_stride], first set of the slice at ev_dev[0]); this turns the
// caller's row-major [nb][n_obs] matrix into it (transpose) or copies it, replacing values outside their
// variable's cardinality (card_dev[n_obs]) by 0 and raising BNPP_STATUS_BAD_EVIDENCE
int sanitize_evidence_launch(bnpp_ctx *ctx, const uint8_t *in, uint8_t *out, uint32_t nb, uint32_t n_obs, const uint32_t *card_dev,
                             bool transpose);
// a CPT with more than kMaxObsPerOperand observed axes: its evidence base per set, sum of stride * value over `obs`
// (stride, column), written as `digits` base-256 digits into columns digit_col.. of the column-major [cols][nb]
// matrix ev_dev, so that K8 reads the CPT through those columns with strides 1, 256, ...
int evidence_digits_launch(bnpp_ctx *ctx, const std::vector<std::pair<int64_t, int>> &obs, uint8_t *ev_dev, uint32_t nb,
                           uint32_t digit_col, uint32_t digits);

}  // namespace bnpp
