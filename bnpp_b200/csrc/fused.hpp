// K9 -- a whole variable-elimination plan in ONE launch (fused.cu), and the program format the
// plan compiles itself into (ve.cu).
//
// Networks whose elimination steps are all small (config 1/2 single queries, config 5 batches:
// every union table <= a few thousand entries) are launch- and round-trip-bound when each bucket
// is its own kernel: every intermediate goes out to HBM/L2 and comes back, every step pays a
// launch.  Here a group of G lanes owns one evidence set and interprets the plan's step list
// from start to finish; the intermediates of a set never leave shared memory.
#pragma once
#include <cstddef>
#include <cstdint>

struct bnpp_ctx;

namespace bnpp {

constexpr int kFusedThreads = 128;      // CTA size; a CTA holds kFusedThreads / G evidence sets
constexpr int kFusedInlineEv = 256;     // single query: evidence values travel in the kernel parameters

// ---- program: uint32 words, every record a multiple of 4 words (fetched with 128-bit loads) ----
// step header, 8 words
//   [0] n_out     output entries
//   [1] cx        cardinality of the eliminated variable (1 = pure product)
//   [2] k | flags << 8
//   [3] out_off   arena offset of the output, or offset into the result buffer (kFusedToResult)
//   [4] tab_off   first word of this step's operand-offset table [k][n_out] in `offtab`
//   [5..6] device address of the output (kFusedToGlobal: a later launch of the plan reads it)
//   [7] kFusedMax: R_s, the first argmax row of the step (MPE / MAP plans; 0 otherwise)
// then k operand records, 4 words each
//   [0] kind | nobs << 8     kind 0: intermediate in the arena, 1: resident CPT view
//   [1] arena offset         | low  32 bits of the CPT's device address
//   [2] sx                   stride of the eliminated variable (0: the operand lacks it)
//   [3] 0                    | high 32 bits of the CPT's device address
// each CPT operand followed by its observed axes, (stride, evidence column) pairs padded to 4 words
constexpr uint32_t kFusedToResult = 1u;     // flags
constexpr uint32_t kFusedWantZ = 2u;
constexpr uint32_t kFusedToGlobal = 8u;     // the output goes to the device address in header words 5 (low) and 6 (high), dense
constexpr uint32_t kFusedPairs = 4u;        // cx == 2 and every arena operand holds the eliminated variable at stride 1 on even offsets
constexpr uint32_t kFusedMax = 16u;         // a max step of an MPE / MAP program: the argmax of output entry o for set b
                                            // goes to byte (R_s + o) * nb + b of the launch's argmax rows (ve_fused_max,
                                            // ve_fused_mixed: there the steps without this flag sum)
constexpr uint32_t kFusedHeaderWords = 8;
constexpr uint32_t kFusedOperandWords = 4;

struct FusedLaunch {
    const uint32_t *prog;
    const uint32_t *offtab;
    const uint8_t *ev;          // [nb][n_obs] evidence values, one row per set; nullptr: ev_inline (nb == 1)
    double *result;             // [result_size][nb], batch fastest
    double *z;                  // nb == 1: partition of the result step (may be nullptr)
    uint32_t nb, n_obs, n_steps;
    uint32_t arena;             // doubles of shared memory per evidence set (even)
    uint8_t ev_inline[kFusedInlineEv];
};

// ve_fused_max: the launch of an MPE program -- every step takes the maximum over its eliminated variable (products
// as in the sum path; the maximum starts at x = 0, a later x replaces it only if strictly greater) and a kFusedMax
// step writes its argmax bytes to `arg` ([rows][nb], rows of header word 7); result = the value of every set.
// ve_fused_mixed (a MAP program that also sums) takes the same launch: only kFusedMax steps take the maximum.
struct FusedMaxLaunch {
    FusedLaunch f;
    uint8_t *arg;
};

// K10: many independent programs of ONE query in one launch, a CTA (128 lanes) per program ("task")
struct TaskRecord {
    uint32_t prog_off;          // first word of the task's program in `prog`
    uint32_t tab_base;          // first word of its operand-offset tables in `offtab`
    uint32_t n_steps;
    uint32_t arena;             // doubles of shared memory the task needs
};
struct TaskLaunch {
    const uint32_t *prog;
    const uint32_t *offtab;
    const TaskRecord *tasks;    // device, 16-byte records
    double *result;
    double *z;
    uint32_t n_tasks, n_obs;
    uint8_t ev_inline[kFusedInlineEv];
};
const void *tasks_kernel();
int tasks_geometry(bnpp_ctx *ctx, uint32_t n_tasks, uint32_t arena, unsigned *grid, unsigned *smem);
int tasks_launch(bnpp_ctx *ctx, const TaskLaunch &p, unsigned grid, unsigned smem);

// G = lanes per evidence set: 8, 16, 32 (a warp) or 128 (the CTA)
bool fused_valid_g(int G);
size_t fused_smem_bytes(int G, uint32_t arena);
int fused_launch(bnpp_ctx *ctx, int G, const FusedLaunch &p);
int fused_max_launch(bnpp_ctx *ctx, int G, const FusedMaxLaunch &p);
int fused_mixed_launch(bnpp_ctx *ctx, int G, const FusedMaxLaunch &p);

}  // namespace bnpp
