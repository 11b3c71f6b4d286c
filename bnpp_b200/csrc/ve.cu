// Device-resident variable elimination: plan + executor.
//
// Replaces the bucket-elimination loop of BN::variable_elimination (reference
// code/model.cpp:382-445) together with the up-front conditioning of every CPT
// (code/model.cpp:283-286, 321-324):
//   * evidence is never materialised -- a conditioned CPT is a strided VIEW of the
//     resident table whose base offset is computed from the evidence values at run
//     time (code/factor.cpp:214-242 reduced to pointer arithmetic);
//   * each bucket is ONE fused kernel launch (product of the bucket, sum out the
//     variable), never writing the product table (code/model.cpp:414-418);
//   * intermediates stay in HBM from the first bucket to the final scalar; only the
//     result crosses back to the host.
// The reference leaves the axis order of intermediates to the iteration order of an
// address-keyed hash set (SURVEY A.4); here it is CANONICAL: axes sorted by
// elimination time, the next variable to be eliminated innermost.  Every operand of a
// bucket then has the eliminated variable as its fastest axis (32-byte loads) and
// scopes are mutually order-compatible (pure broadcasts, no transposes).
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <thread>
#include <vector>

#include "batched.hpp"
#include "chain.hpp"
#include "common.cuh"
#include "contract.hpp"
#include "elim_order.hpp"
#include "fused.hpp"

namespace bnpp {
int contract(bnpp_ctx *ctx, int k, const bnpp_operand *ops, const bnpp_scope *out_scope, int64_t elim_var, int divide,
             double *out_dev, double *z_dev, bool max_mode = false, uint8_t *arg_dev = nullptr);
int fill(bnpp_ctx *ctx, double *out, uint64_t n, double value);
int normalize_segments(bnpp_ctx *ctx, double *buf, const uint32_t *off_dev, const uint32_t *size_dev, int n);
int normalize_segments_batched(bnpp_ctx *ctx, double *buf, const uint32_t *off_dev, const uint32_t *size_dev, int n, uint32_t nb);
uint32_t chain_depth_knob();

struct PlanFactor {
    std::vector<uint32_t> var, card;
    std::vector<int64_t> stride;            // empty = dense over (var, card)
    int src = -1;                           // >= 0: view of input table `src`; -1: intermediate
    std::vector<std::pair<int64_t, int>> obs;   // (stride, index into obs_val) folded into the base at run time
    uint64_t size = 1;                      // entries addressed
    int last_use = -1;                      // step index after which an intermediate is freed
};

struct PlanStep {
    std::vector<int> operands;
    int out = -1;                           // PlanFactor index, or -2 = the caller's result buffer
    std::vector<uint32_t> rvar, rcard;      // out == -2: scope written there ...
    uint64_t roff = 0;                      // ... at this offset (doubles)
    bool want_z = false;                    // out == -2: also write the partition (the VE result)
    int64_t elim = -1;
    bool max = false;                       // MPE / MAP plans: a max step (its eliminated variable is a MAP variable)
    uint64_t union_entries = 0, bytes = 0;
};

// variable id -> elimination time.  Ids are dense small integers in every UAI model: a flat
// table (planning a 1000-variable network does ~10^5 lookups); stray large ids fall back to a map.
class RankMap {
public:
    bool count(uint32_t v) const { return v < kDense ? (v < has_.size() && has_[v]) : sparse_.count(v) != 0; }
    uint64_t at(uint32_t v) const { return v < kDense ? (v < val_.size() ? val_[v] : UINT64_MAX) : sparse_.at(v); }
    void set(uint32_t v, uint64_t r)
    {
        if (v >= kDense) {
            sparse_[v] = r;
            return;
        }
        if (v >= has_.size()) {
            has_.resize((size_t)v + 64, 0);
            val_.resize((size_t)v + 64, 0);
        }
        has_[v] = 1;
        val_[v] = r;
    }

private:
    static constexpr uint32_t kDense = 1u << 22;
    std::vector<char> has_;
    std::vector<uint64_t> val_;
    std::map<uint32_t, uint64_t> sparse_;
};

// K9: the plan compiled into the step program of fused.hpp (one launch for the whole plan)
struct FusedProgram {
    bool built = false, ok = false;
    std::vector<uint32_t> prog, offtab;
    // 64-bit device addresses inside `prog`, written at run time: (word of the low half, word of the high half,
    // what it points to: input table `index` (kind 0) or the plan-arena slot of intermediate `index` (kind 1))
    struct Slot { uint32_t lo, hi; int kind, index; };
    std::vector<Slot> ptr_slots;
    std::vector<uint64_t> slot_addr;                    // the addresses `prog` holds right now
    uint32_t n_steps = 0, arena = 0, max_out = 0;
    uint64_t total_union = 0;                           // union entries of all steps, per evidence set
    uint32_t *prog_dev = nullptr, *offtab_dev = nullptr;
    bool offtab_uploaded = false;
};
// MPE / MAP decode (bnpp_mpe_plan_run): one thread walks the max steps in reverse.  rec: the n_obs observed ids, the
// n_sum summed ids (MAP plans; they report BNPP_ASSIGN_SUMMED), then per max step, last first: elim var, argmax table
// offset (bytes, lo, hi), rank, rank x (var, stride) over the step's output scope -- every variable there is
// eliminated later (a MAP variable: the order puts them last), so it is already decoded.  The evidence values travel
// in the parameters (a replay re-parameterises the node), in device memory beyond kDecodeInlineObs.
constexpr uint32_t kDecodeInlineObs = 896;
struct MpeDecodeParams {
    const uint32_t *rec;
    const uint8_t *arg;
    const uint32_t *obs_val_dev;
    uint32_t *assign;
    double *value;
    uint32_t nvars, n_obs, n_rec, set_one;      // set_one: the plan has no result step, the value is the empty product
    uint32_t n_sum;                             // summed ids in rec (MAP plans)
    uint32_t obs_val[kDecodeInlineObs];
};

__global__ void mpe_decode(const __grid_constant__ MpeDecodeParams p)
{
    if (threadIdx.x || blockIdx.x) return;
    for (uint32_t v = 0; v < p.nvars; ++v) p.assign[v] = 0;
    const uint32_t *r = p.rec;
    const uint32_t *val = p.n_obs <= kDecodeInlineObs ? p.obs_val : p.obs_val_dev;
    for (uint32_t i = 0; i < p.n_obs; ++i) p.assign[r[i]] = val[i];
    r += p.n_obs;
    for (uint32_t i = 0; i < p.n_sum; ++i) p.assign[r[i]] = 0xffffffffu;
    r += p.n_sum;
    for (uint32_t s = 0; s < p.n_rec; ++s) {
        const uint64_t off = (uint64_t)r[1] | ((uint64_t)r[2] << 32);
        const uint32_t rank = r[3];
        uint64_t idx = 0;
        for (uint32_t j = 0; j < rank; ++j) idx += (uint64_t)p.assign[r[4 + 2 * j]] * r[5 + 2 * j];
        p.assign[r[0]] = p.arg[off + idx];
        r += 4 + 2 * rank;
    }
    if (p.set_one) *p.value = 1.0;
}

// Max-loc over the ranks of a sharded MPE / MAP run (bnpp_mpe_shard_select): record r = words [r * stride, + stride),
// its value (a double, words 0-1) and assignment (words 2..).  Candidates are ordered by: a number beats a NaN, a
// larger value beats a smaller one, then the lower rank -- a total order, so the strided scan and the tree give the
// winner of the sequential rule (start at rank 0, a later rank replaces it only if strictly greater) in any grouping,
// except that the sequential rule keeps rank 0 when its value is a NaN: that case is checked last.
constexpr int kSelectThreads = 256;

__device__ __forceinline__ double record_value(const uint32_t *rec)
{
    return __hiloint2double((int)rec[1], (int)rec[0]);
}

__device__ __forceinline__ bool select_beats(double v, uint32_t r, double bv, uint32_t br)
{
    if (r == UINT32_MAX) return false;
    if (br == UINT32_MAX) return true;
    const bool n = isnan(v), bn = isnan(bv);
    if (n != bn) return bn;
    if (!n && v != bv) return v > bv;
    return r < br;
}

__global__ void __launch_bounds__(kSelectThreads) mpe_shard_select(const uint32_t *rec, uint32_t nranks, uint32_t nvars,
                                                                   uint64_t stride, double *value, uint32_t *assign)
{
    __shared__ double s_v[kSelectThreads / 32];
    __shared__ uint32_t s_r[kSelectThreads / 32];
    double bv = 0.0;
    uint32_t br = UINT32_MAX;
    for (uint32_t r = threadIdx.x; r < nranks; r += blockDim.x) {
        const double v = record_value(rec + r * stride);
        if (select_beats(v, r, bv, br)) bv = v, br = r;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double v = __shfl_down_sync(0xffffffffu, bv, o);
        const uint32_t r = __shfl_down_sync(0xffffffffu, br, o);
        if (select_beats(v, r, bv, br)) bv = v, br = r;
    }
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) s_v[w] = bv, s_r[w] = br;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < (int)(blockDim.x >> 5); ++i)
            if (select_beats(s_v[i], s_r[i], bv, br)) bv = s_v[i], br = s_r[i];
        if (isnan(record_value(rec))) br = 0;
        s_r[0] = br;
    }
    __syncthreads();
    const uint32_t *win = rec + s_r[0] * stride;
    if (threadIdx.x == 0) *value = record_value(win);
    for (uint32_t v = threadIdx.x; v < nvars; v += blockDim.x) assign[v] = win[2 + v];
}

// MPE / MAP decode of a batch (bnpp_mpe_plan_run_batched): one thread per set of a slice walks the records of mpe_decode with
// the FIRST ARGMAX ROW of the step in words 1-2: the argmax of output entry o of a step for set t of the slice is
// arg[(row + o) * cur + t].  The records are the same for every set, so the threads of a warp always touch one
// variable's row of assign[v][nb] (coalesced); only the argmax byte a set's own assignment selects is scattered.
struct MpeBatchDecodeParams {
    const uint32_t *rec;
    const uint8_t *arg;             // [rows][cur]
    const uint8_t *ev;              // evidence value j of set t: ev[j * ev_col + t * ev_row] (already range-checked)
    uint64_t ev_col, ev_row;
    uint8_t *assign;                // [nvars][nb]: the column of the slice's first set
    uint32_t nb, cur, nvars, n_obs, n_rec, n_sum;
};

__global__ void mpe_decode_batched(const __grid_constant__ MpeBatchDecodeParams p)
{
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < p.cur; t += gridDim.x * blockDim.x) {
        uint8_t *a = p.assign + t;
        for (uint32_t v = 0; v < p.nvars; ++v) a[(uint64_t)v * p.nb] = 0;
        const uint32_t *r = p.rec;
        for (uint32_t i = 0; i < p.n_obs; ++i) a[(uint64_t)__ldg(r + i) * p.nb] = p.ev[i * p.ev_col + t * p.ev_row];
        r += p.n_obs;
        for (uint32_t i = 0; i < p.n_sum; ++i) a[(uint64_t)__ldg(r + i) * p.nb] = 0xff;
        r += p.n_sum;
        for (uint32_t s = 0; s < p.n_rec; ++s) {
            const uint64_t row = (uint64_t)__ldg(r + 1) | ((uint64_t)__ldg(r + 2) << 32);
            const uint32_t rank = __ldg(r + 3);
            uint64_t idx = 0;
            for (uint32_t j = 0; j < rank; ++j) idx += (uint64_t)a[(uint64_t)__ldg(r + 4 + 2 * j) * p.nb] * __ldg(r + 5 + 2 * j);
            a[(uint64_t)__ldg(r) * p.nb] = p.arg[(row + idx) * p.cur + t];
            r += 4 + 2 * rank;
        }
    }
}
}  // namespace bnpp

struct bnpp_ve_plan {
    bnpp_ctx *ctx = nullptr;
    int n_inputs = 0;
    int n_obs = 0;
    std::vector<uint32_t> obs_card;         // cardinality per observed variable (0 = no factor mentions it)
    uint32_t *obs_card_dev = nullptr;       // device copy, made by the first batched run
    uint8_t *ev_clean = nullptr;            // batched fused runs: the evidence matrix with out-of-range values zeroed
    uint64_t ev_clean_bytes = 0;
    bool normalize = true;                  // marginals plan: normalise the slices at the end of a run
    int fused_mode = 1;                     // 0: one launch per bucket always; 1: one launch per plan when every step is small
    bnpp::FusedProgram fused;
    // K10 -- TASKS (on unless BNPP_FUSED_SEGMENTS=0): a plan that is not one launch altogether is cut into tasks --
    // subtrees of the bucket tree whose steps are all small, run by ONE CTA with their intermediates in shared memory
    // (a "segment": a contiguous range of the re-ordered step list, with its own step program) -- and the tasks whose
    // inputs are ready form ONE ve_tasks launch (a "group" = the small tasks of one dependency level).  Wide steps
    // stay their own launches.  Hundreds of tiny launches become a few dozen.
    struct Segment { int a = 0, b = 0, G = 128; int level = 0; bnpp::FusedProgram prog; };
    struct Group {
        int a = 0, b = 0;                   // step range covered (all its steps are small and of one level)
        int first_seg = 0, n_segs = 0;
        uint32_t max_arena = 0;
        unsigned grid = 0, smem = 0;
        bnpp::TaskLaunch launch;            // parameters of the launch (evidence and result pointers patched per run)
        bool launch_valid = false;
    };
    int segments_mode = 1;
    uint32_t segments_max_steps = 0;        // > 0: at most this many steps per task (tests)
    bool segments_built = false, levels_built = false;
    std::vector<Segment> segs;
    std::vector<Group> groups;
    std::vector<int> group_at;              // per step: the group that STARTS here, or -1
    std::vector<int> step_level;            // per step (after build_levels): dependency level; steps of a level never read each other
    std::vector<int> step_task;             // per step: root step of its task (small steps), -1 for wide steps
    // all task programs of the plan in ONE device buffer each (one upload)
    std::vector<uint32_t> tasks_prog;
    size_t tasks_tab_words = 0;         // all offset tables of the tasks, each padded to 4 words (they stay in segs[i].prog.offtab)
    std::vector<bnpp::TaskRecord> tasks_rec;
    struct TaskSlot { uint32_t lo, hi; int kind, index; uint64_t addr; };
    std::vector<TaskSlot> tasks_slots;
    uint32_t *tasks_prog_dev = nullptr, *tasks_tab_dev = nullptr;
    bnpp::TaskRecord *tasks_rec_dev = nullptr;
    bool tasks_uploaded = false;
    std::vector<bnpp::PlanFactor> f;
    std::vector<bnpp::PlanStep> steps;
    std::vector<uint32_t> result_var, result_card;
    uint64_t result_size = 1;
    uint64_t union_entries = 0, bytes = 0, peak_bytes = 0, max_step_entries = 0;
    // replay state: one resolved launch per step and a fixed arena for the intermediates, so a
    // run is pointer patching + cudaLaunchKernel (the host must not be what small steps wait for)
    std::vector<std::unique_ptr<bnpp::LaunchDesc>> exec;     // resolved lazily: only the steps that run as their own launch
    std::vector<char> exec_planned;
    std::vector<uint64_t> arena_off;        // per PlanFactor, in doubles
    uint64_t arena_doubles = 0;
    double *arena = nullptr;
    bool exec_ok = false;
    // the whole schedule as one CUDA graph (a chain of kernel nodes): a replay is one
    // cudaGraphLaunch; only nodes whose pointers moved (other evidence values) are re-parameterised
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t graph_exec = nullptr;
    bool graph_groups = false;              // the graph was built with task groups as nodes
    std::vector<cudaGraphNode_t> nodes;
    // batched replay: per-step operand-offset tables (host copy + device copy, built on first use)
    std::vector<std::vector<uint32_t>> offtab_host;
    std::vector<uint32_t *> offtab_dev;
    // batched replay as a captured graph (allocations included), valid while the caller's buffers stay put
    cudaGraphExec_t batch_exec = nullptr;
    std::vector<const void *> batch_key;
    uint64_t batch_runs = 0;
    bool use_graph = true;
    uint64_t runs = 0;                      // the graph is built on the second run: a one-shot plan never pays for it
    // all-marginals plan (bucket-tree elimination): per variable the slice of the result buffer
    bool is_mar = false;
    std::vector<uint32_t> mar_off, mar_size;
    uint32_t *mar_off_dev = nullptr, *mar_size_dev = nullptr;
    // MPE plan (max-product): every eliminating step also writes its argmax table into a byte arena that is never
    // reused within a run (the decode reads all of them); single runs are launch-per-bucket (K10 only sums), batched
    // runs take K9 in max mode (ve_fused_max) or K8's max variants
    // MAP plan (marginal MAP): the same, with max steps only where the eliminated variable is a MAP variable -- the
    // other eliminating steps sum, the argmax arena / rows and decode records cover the max steps only
    bool is_mpe = false;                    // an MPE or MAP plan
    uint32_t mpe_nvars = 0;
    uint32_t n_max = 0, n_sum_steps = 0;    // max steps and summing eliminating steps
    uint32_t n_summed = 0;                  // summed variable ids in the decode records (MAP plans)
    std::vector<uint64_t> arg_off;          // per step: byte offset of its argmax table (eliminating steps only)
    uint64_t arg_bytes = 0;
    uint8_t *arg_arena = nullptr;
    std::vector<uint32_t> decode_rec;       // see MpeDecodeParams; uploaded once
    uint32_t *decode_rec_dev = nullptr, *obs_val_dev = nullptr;
    uint32_t n_decode_rec = 0;
    bnpp::MpeDecodeParams decode;           // parameters of the decode's node in the replay graph
    cudaGraphNode_t decode_node = nullptr;
    // batched MPE: eliminating step s (plan order) owns argmax rows [arg_row[s], arg_row[s] + its output entries) of a
    // byte scratch of arg_rows rows x slice sets, entry o of set b at (arg_row[s] + o) * slice + b
    std::vector<uint64_t> arg_row;
    uint64_t arg_rows = 0;
    std::vector<uint32_t> batch_rec;        // decode records of mpe_decode_batched (rows for byte offsets); uploaded once
    uint32_t *batch_rec_dev = nullptr;
    uint8_t *batch_arg = nullptr;
    uint64_t batch_arg_bytes = 0;
    bool profiling = false;
    std::vector<cudaEvent_t> ev;
    std::vector<float> step_ms;
    std::vector<std::string> step_kernel;
    // K11 -- WINDOWS (chain.hpp): runs of wide binary eliminations, each one contract_chain launch with its
    // intermediates in registers.  Steps [a, b) of the plan; the steps stay in the plan (the batched engines, the
    // emulator of the tests and bnpp_ve_plan_describe see them one by one), only the single-query run fuses them.
    struct Window {
        int a = 0, b = 0;
        int head = -1, out = -1;                        // PlanFactor ids
        int side[bnpp::kChainMaxLevels][bnpp::kChainMaxSides];
        int m = 0, add[bnpp::kChainMaxLevels] = {0, 0, 0, 0};
        const void *fn = nullptr;
        unsigned grid = 0;                              // resolved by the first run (occupancy)
        bnpp::ChainParams p;                            // pointers patched per run
        uint64_t bytes = 0, entries = 0;
        std::string name;
    };
    uint32_t chain_depth = 0;               // bnpp_tuning_set("chain_depth") at plan creation; <= 1: no windows
    std::vector<Window> windows;
    std::vector<int> window_at;             // per step: the window that STARTS here, or -1
    std::vector<int> launch_first;          // first step of every launch of a single run without task groups
};

using namespace bnpp;

namespace {

// device buffer of `count` elements of T, rounded up to whole doubles; *out is set only on success
template <class T>
int dev_alloc(bnpp_ctx *ctx, size_t count, T **out)
{
    double *store = nullptr;
    const int rc = bnpp_alloc(ctx, (count * sizeof(T) + sizeof(double) - 1) / sizeof(double), &store);
    if (rc == BNPP_OK) *out = static_cast<T *>(static_cast<void *>(store));
    return rc;
}

template <class T>
void dev_free(bnpp_ctx *ctx, T *&p)
{
    if (p) bnpp_free(ctx, static_cast<double *>(static_cast<void *>(p)));
    p = nullptr;
}

uint64_t table_size(const std::vector<uint32_t> &card)
{
    uint64_t n = 1;
    for (uint32_t c : card) n *= c;
    return n;
}

// one fused launch description: product of `ops`, optionally eliminating `elim`, output
// in canonical order (descending rank => the lowest-rank variable is the fastest axis)
int add_step(bnpp_ve_plan *pl, std::vector<int> ops, int64_t elim, const RankMap &rank, bool to_result,
             uint64_t roff = 0, bool want_z = true)
{
    std::vector<std::pair<uint64_t, std::pair<uint32_t, uint32_t>>> u;   // (rank, (var, card))
    for (int id : ops) {
        const PlanFactor &pf = pl->f[id];
        for (size_t i = 0; i < pf.var.size(); ++i) {
            bool seen = false;
            for (auto &e : u) seen |= (e.second.first == pf.var[i]);
            if (!seen) u.push_back({rank.at(pf.var[i]), {pf.var[i], pf.card[i]}});
        }
    }
    std::sort(u.begin(), u.end(), [](const auto &a, const auto &b) { return a.first > b.first; });
    PlanFactor out;
    uint64_t entries = 1;
    for (auto &e : u) {
        entries *= e.second.second;
        if (elim >= 0 && e.second.first == (uint64_t)elim) continue;
        out.var.push_back(e.second.first);
        out.card.push_back(e.second.second);
    }
    out.size = table_size(out.card);
    PlanStep st;
    st.operands = ops;
    st.elim = elim;
    st.union_entries = entries;
    st.bytes = 8 * out.size;
    for (int id : ops) st.bytes += 8 * pl->f[id].size;
    const int step_index = (int)pl->steps.size();
    for (int id : ops) pl->f[id].last_use = step_index;
    if (to_result) {
        st.out = -2;
        st.rvar = out.var;
        st.rcard = out.card;
        st.roff = roff;
        st.want_z = want_z;
        pl->result_var = out.var;
        pl->result_card = out.card;
        pl->result_size = out.size;
    } else {
        pl->f.push_back(std::move(out));
        st.out = (int)pl->f.size() - 1;
    }
    const int out_id = st.out;
    pl->steps.push_back(std::move(st));
    return out_id;
}

uint64_t union_size(const bnpp_ve_plan *pl, const std::vector<int> &ops)
{
    std::vector<uint32_t> seen;
    uint64_t n = 1;
    for (int id : ops)
        for (size_t i = 0; i < pl->f[id].var.size(); ++i) {
            const uint32_t v = pl->f[id].var[i];
            if (std::find(seen.begin(), seen.end(), v) != seen.end()) continue;
            seen.push_back(v);
            n *= pl->f[id].card[i];
        }
    return n;
}

// A bucket that streams a wide table usually also holds a handful of small CPTs.  Gathering
// from each of them costs instructions per entry of the WIDE table; multiplying them into
// one small (L2-resident) table first costs a negligible launch and leaves the streaming
// kernel with the wide operand(s) plus one small one (K <= 3: the `canon` variant).
constexpr uint64_t kWideEntries = 1ull << 20;
void fold_small(bnpp_ve_plan *pl, std::vector<int> &ops, const RankMap &rank)
{
    if (ops.empty()) return;
    const uint64_t whole = union_size(pl, ops);          // entries the bucket's launch iterates over
    if (whole < kWideEntries) return;
    const uint64_t cap = std::max<uint64_t>(1ull << 12, whole >> 5);
    auto merge = [&](std::vector<int> part) {
        const int t = add_step(pl, part, -1, rank, false);
        return t;
    };
    // repeatedly multiply together the two smallest operands while their joint table stays small
    for (;;) {
        std::stable_sort(ops.begin(), ops.end(), [pl](int a, int b) { return pl->f[a].size < pl->f[b].size; });
        if (ops.size() < 2) break;
        // the smallest operand and the partner giving the smallest joint table
        size_t best = 0;
        uint64_t best_size = UINT64_MAX;
        for (size_t j = 1; j < ops.size(); ++j) {
            const uint64_t u = union_size(pl, {ops[0], ops[j]});
            if (u < best_size) { best_size = u; best = j; }
        }
        if (best == 0 || best_size > cap || (ops.size() == 2 && pl->f[ops[1]].size > cap)) break;
        if (ops.size() == 2) {
            // two small tables left: one launch over `whole` entries either way, nothing to gain
            break;
        }
        const int a = ops[0], b = ops[best];
        ops.erase(ops.begin() + best);
        ops.erase(ops.begin());
        ops.push_back(merge({a, b}));
    }
    // a raw input view keeps its file-order layout, which forces scalar gathers in a wide launch:
    // copy it once into canonical axis order (K = 1 product)
    for (int &id : ops)
        if (pl->f[id].src >= 0 && pl->f[id].size <= cap) id = merge({id});
}

// the kernel takes at most BNPP_MAX_OPERANDS tables: fold the smallest ones first
void shrink(bnpp_ve_plan *pl, std::vector<int> &ops, const RankMap &rank)
{
    while ((int)ops.size() > kMaxK) {
        std::stable_sort(ops.begin(), ops.end(), [pl](int a, int b) { return pl->f[a].size < pl->f[b].size; });
        int m = (int)ops.size() - kMaxK + 1;
        if (m > kMaxK) m = kMaxK;
        std::vector<int> head(ops.begin(), ops.begin() + m);
        const int t = add_step(pl, head, -1, rank, false);
        ops.erase(ops.begin(), ops.begin() + m);
        ops.insert(ops.begin(), t);
    }
}

// the input tables as evidence-reduced views (code/domain.cpp:74-90: free axes keep their order)
int add_inputs(bnpp_ve_plan *pl, int nfac, const bnpp_scope *scopes, const std::map<uint32_t, int> &obs_index,
               RankMap &rank)
{
    for (int q = 0; q < nfac; ++q) {
        const bnpp_scope &s = scopes[q];
        if (s.rank < 0 || s.rank > BNPP_MAX_RANK) return BNPP_EINVAL;
        PlanFactor pf;
        pf.src = q;
        uint64_t dense = 1;
        std::vector<int64_t> st(s.rank);
        for (int i = s.rank - 1; i >= 0; --i) {
            st[i] = (int64_t)dense;
            dense *= s.card[i];
        }
        for (int i = 0; i < s.rank; ++i) {
            auto o = obs_index.find(s.var_id[i]);
            if (o != obs_index.end()) {
                pf.obs.push_back({st[i], o->second});
                if ((size_t)o->second < pl->obs_card.size()) pl->obs_card[o->second] = s.card[i];
                continue;
            }
            pf.var.push_back(s.var_id[i]);
            pf.card.push_back(s.card[i]);
            pf.stride.push_back(st[i]);
            if (!rank.count(s.var_id[i])) rank.set(s.var_id[i], (1ull << 40) + (0xffffffffull - s.var_id[i]));   // kept: ascending id, most significant first
        }
        pf.size = table_size(pf.card);
        pl->f.push_back(pf);
    }
    return BNPP_OK;
}

// product of `ops`, then every variable outside `keep` summed out one fused launch at a time
// (the first launch also does the product); -1 when there is nothing to multiply
int chain(bnpp_ve_plan *pl, std::vector<int> ops, const std::vector<uint32_t> &keep, const RankMap &rank,
          bool to_result, uint64_t roff)
{
    if (ops.empty()) return -1;
    std::vector<std::pair<uint64_t, uint32_t>> gone;   // (rank, var) of the variables to eliminate
    for (int id : ops)
        for (uint32_t v : pl->f[id].var) {
            bool kept = std::find(keep.begin(), keep.end(), v) != keep.end(), seen = false;
            for (auto &g : gone) seen |= (g.second == v);
            if (!kept && !seen) gone.push_back({rank.at(v), v});
        }
    std::sort(gone.begin(), gone.end());
    shrink(pl, ops, rank);
    if (gone.empty()) return add_step(pl, ops, -1, rank, to_result, roff, false);
    int t = -1;
    for (size_t i = 0; i < gone.size(); ++i) {
        const bool last = (i + 1 == gone.size());
        t = add_step(pl, i == 0 ? ops : std::vector<int>{t}, (int64_t)gone[i].second, rank, to_result && last, roff, false);
    }
    return t;
}

// Arena layout (first-fit over the step sequence, 256-byte granules) and one resolved launch per
// step.  Descriptors are planned against stand-in pointers that carry only the ALIGNMENT the
// real ones are guaranteed to have: intermediates sit on 256-byte boundaries of the arena;
// an input view is its table (required 32-byte aligned at run time, else the dynamic path
// is taken) plus a base offset that is a multiple of gcd(strides of its observed axes).
void build_exec(bnpp_ve_plan *pl)
{
    const uint64_t gran = 32;   // doubles
    pl->arena_off.assign(pl->f.size(), 0);
    std::vector<std::pair<uint64_t, uint64_t>> free_list;   // (offset, size)
    uint64_t top = 0;
    // first fit; `avoid`: regions the block must not overlap (the head and side tables a window's launch reads while
    // it writes its last level's output)
    std::vector<std::pair<uint64_t, uint64_t>> avoid;                 // (offset, end)
    auto clear_of = [&](uint64_t off, uint64_t n) {
        for (auto &a : avoid)
            if (off < a.second && a.first < off + n) return a.second;      // the first end to try next
        return uint64_t(0);
    };
    auto take = [&](uint64_t n) {
        n = (n + gran - 1) / gran * gran;
        for (size_t i = 0; i < free_list.size(); ++i) {
            const uint64_t lo = free_list[i].first, hi = lo + free_list[i].second;
            uint64_t off = lo;
            for (uint64_t e; off + n <= hi && (e = clear_of(off, n));) off = (e + gran - 1) / gran * gran;
            if (off + n > hi) continue;
            free_list.erase(free_list.begin() + i);
            if (off + n < hi) free_list.insert(free_list.begin() + i, {off + n, hi - off - n});
            if (lo < off) free_list.insert(free_list.begin() + i, {lo, off - lo});
            return off;
        }
        uint64_t off = top;
        for (uint64_t e; (e = clear_of(off, n));) off = (e + gran - 1) / gran * gran;
        if (top < off) {
            free_list.push_back({top, off - top});
            std::sort(free_list.begin(), free_list.end());
        }
        top = off + n;
        return off;
    };
    auto give = [&](uint64_t off, uint64_t n) {
        n = (n + gran - 1) / gran * gran;
        free_list.push_back({off, n});
        std::sort(free_list.begin(), free_list.end());
        for (size_t i = 0; i + 1 < free_list.size();)
            if (free_list[i].first + free_list[i].second == free_list[i + 1].first) {
                free_list[i].second += free_list[i + 1].second;
                free_list.erase(free_list.begin() + i + 1);
            } else ++i;
        if (!free_list.empty() && free_list.back().first + free_list.back().second == top) {
            top = free_list.back().first;
            free_list.pop_back();
        }
    };
    // steps of one dependency level may run concurrently (the tasks of a ve_tasks launch): what a level's steps read
    // is released only when the level ends
    std::vector<int> pending;
    const bool leveled = pl->step_level.size() == pl->steps.size();
    for (size_t s = 0; s < pl->steps.size(); ++s) {
        const PlanStep &st = pl->steps[s];
        avoid.clear();
        for (const auto &w : pl->windows)
            if ((int)s == w.b - 1) {
                auto add = [&](int id) {
                    if (pl->f[id].src < 0) avoid.push_back({pl->arena_off[id], pl->arena_off[id] + (pl->f[id].size + gran - 1) / gran * gran});
                };
                add(w.head);
                for (int j = 0; j < w.m; ++j)
                    for (int q = 0; q < w.p.lv[j].k; ++q) add(w.side[j][q]);
            }
        if (st.out >= 0) pl->arena_off[st.out] = take(pl->f[st.out].size);
        pl->arena_doubles = std::max(pl->arena_doubles, top);
        for (int id : st.operands)
            if (pl->f[id].src < 0 && pl->f[id].last_use == (int)s && std::find(pending.begin(), pending.end(), id) == pending.end())
                pending.push_back(id);
        const bool level_ends = !leveled || s + 1 == pl->steps.size() || pl->step_level[s + 1] != pl->step_level[s];
        if (level_ends) {
            for (int id : pending) give(pl->arena_off[id], pl->f[id].size);
            pending.clear();
        }
    }

    // launches are resolved lazily, step by step, during the first run (plan_step): the GPU already
    // executes the early buckets while the host is still resolving the later ones
    // (the descriptors themselves -- 4 KB each -- are allocated by the first launch-per-bucket run: a plan that
    // runs fused never needs them)
    pl->exec_ok = true;
}

// bytes of the live intermediates at their peak over the step order (an intermediate lives from its step to its last reader)
uint64_t live_peak(const bnpp_ve_plan *pl)
{
    uint64_t live = 0, peak = 0;
    for (size_t s = 0; s < pl->steps.size(); ++s) {
        const PlanStep &st = pl->steps[s];
        if (st.out >= 0) live += 8 * pl->f[st.out].size;
        peak = std::max(peak, live);
        for (int id : st.operands)
            if (pl->f[id].src < 0 && pl->f[id].last_use == (int)s) live -= 8 * pl->f[id].size;
    }
    return peak;
}

// resolve the launch of step s against stand-in pointers that carry only the guaranteed alignment
bool plan_step(bnpp_ve_plan *pl, size_t s)
{
    double *const arena_standin = reinterpret_cast<double *>(uintptr_t(1) << 32);
    double *const table_standin = reinterpret_cast<double *>(uintptr_t(2) << 32);
    double *const result_standin = reinterpret_cast<double *>((uintptr_t(3) << 32) + 8);   // only 8-byte alignment assumed
    const PlanStep &st = pl->steps[s];
    bnpp_operand ops[kMaxK];
    for (size_t q = 0; q < st.operands.size(); ++q) {
        const PlanFactor &pf = pl->f[st.operands[q]];
        if (pf.src < 0) {
            ops[q].data = arena_standin + pl->arena_off[st.operands[q]];
        } else {
            uint64_t g = 4;
            for (auto &o : pf.obs) g = std::__gcd<uint64_t>(g, (uint64_t)o.first);
            ops[q].data = table_standin + (g >= 4 ? 0 : g);
        }
        ops[q].scope.rank = (int32_t)pf.var.size();
        ops[q].scope.var_id = pf.var.data();
        ops[q].scope.card = pf.card.data();
        ops[q].stride = pf.stride.empty() ? nullptr : pf.stride.data();
    }
    bnpp_scope os;
    double *dst;
    if (st.out == -2) {
        os.rank = (int32_t)st.rvar.size();
        os.var_id = st.rvar.data();
        os.card = st.rcard.data();
        dst = result_standin;
    } else {
        const PlanFactor &of = pl->f[st.out];
        os.rank = (int32_t)of.var.size();
        os.var_id = of.var.data();
        os.card = of.card.data();
        dst = arena_standin + pl->arena_off[st.out];
    }
    pl->exec_planned[s] = 1;
    if (!pl->exec[s]) pl->exec[s].reset(new LaunchDesc());
    const bool max_mode = st.max;
    return contract_plan(pl->ctx, (int)st.operands.size(), ops, &os, st.elim, 0, dst, nullptr, pl->exec[s].get(), max_mode,
                         max_mode ? pl->arg_arena + pl->arg_off[s] : nullptr) == BNPP_OK;
}


// ---- K9: compile the plan into one fused launch (fused.hpp) -------------------------------------
constexpr uint64_t kFusedMaxUnion = 1ull << 14;      // widest step (union entries) a fused plan may contain
constexpr uint64_t kFusedMaxTabWords = 1ull << 21;   // operand-offset tables, all steps
constexpr uint64_t kFusedMaxLaneWork = 1ull << 13;   // union entries one lane may walk per evidence set (the steps of a set are serial)
constexpr size_t kFusedSmemLimit = 200u << 10;       // dynamic shared memory of one CTA

bool fused_default_on()
{
    static const int on = [] {
        const char *e = getenv("BNPP_FUSED");
        return (e && e[0] == '0') ? 0 : 1;
    }();
    return on != 0;
}

// Step order: the bucket tree is walked depth first, at every node the child whose subtree needs
// the most scratch beyond its own result first (Sethi-Ullman), so few intermediates are alive
// at any time -- the arena of one evidence set has to fit in shared memory many times over.
// Any topological order gives the same numbers: operand lists, hence the order of the
// multiplications inside a bucket, are untouched.
// Scratch of fused_encode, sized by the PLAN (steps, factors) and built once per thread: a plan of a thousand buckets is
// cut into a few hundred tasks, and a task must cost what ITS steps cost, not a pass over the plan.  Everything a call
// marks is put back before it returns.
struct EncodeScratch {
    std::vector<int> pos, last_use, producer, reads, side;
    std::vector<char> in_smem, read_inside, read_outside;
    std::vector<uint64_t> aoff, at;
    std::vector<int> cons_off, cons;        // consumers[f] = steps that read factor f (CSR)
    explicit EncodeScratch(const bnpp_ve_plan *pl);
};
void fused_encode(bnpp_ve_plan *pl, const std::vector<int> &order, bool segment, FusedProgram &fp, EncodeScratch *scratch = nullptr);

void fused_build(bnpp_ve_plan *pl)
{
    FusedProgram &fp = pl->fused;
    fp.built = true;
    fp.ok = false;
    const size_t ns = pl->steps.size();
    if (ns == 0 || ns >= (1u << 24)) return;
    if (!pl->is_mar && pl->steps.back().out != -2) return;      // the result is the scalar 1: nothing to fuse
    for (const PlanStep &st : pl->steps)
        if (st.union_entries > kFusedMaxUnion || st.operands.empty() || (int)st.operands.size() > kMaxK) return;

    std::vector<int> producer(pl->f.size(), -1);
    for (size_t s = 0; s < ns; ++s)
        if (pl->steps[s].out >= 0) producer[pl->steps[s].out] = (int)s;
    auto out_size = [&](size_t s) -> uint64_t {
        const PlanStep &st = pl->steps[s];
        return st.out >= 0 ? pl->f[st.out].size : table_size(st.rcard);
    };
    std::vector<char> consumed(ns, 0);
    std::vector<std::vector<int>> kids(ns);
    std::vector<uint64_t> need(ns, 0);
    for (size_t s = 0; s < ns; ++s) {
        for (int id : pl->steps[s].operands) {
            const int c = producer[id];
            if (c < 0) continue;
            if (c >= (int)s) return;                              // producers precede consumers in a plan
            consumed[c] = 1;
            if (std::find(kids[s].begin(), kids[s].end(), c) == kids[s].end()) kids[s].push_back(c);
        }
        std::stable_sort(kids[s].begin(), kids[s].end(), [&](int a, int b) {
            return (int64_t)(need[a] - out_size(a)) > (int64_t)(need[b] - out_size(b));
        });
        uint64_t held = 0, peak = 0;
        for (int c : kids[s]) {
            peak = std::max(peak, held + need[c]);
            held += out_size(c);
        }
        need[s] = std::max(peak, held + (pl->steps[s].out >= 0 ? out_size(s) : 0));
    }
    std::vector<int> order;
    std::vector<char> done(ns, 0);
    for (size_t root = 0; root < ns; ++root) {
        if (done[root] || (pl->steps[root].out != -2 && consumed[root])) continue;
        std::vector<std::pair<int, size_t>> stack{{(int)root, 0}};
        while (!stack.empty()) {
            const int s = stack.back().first;
            if (stack.back().second < kids[s].size()) {
                const int c = kids[s][stack.back().second++];
                if (!done[c]) {
                    done[c] = 1;
                    stack.push_back({c, 0});
                }
            } else {
                order.push_back(s);
                stack.pop_back();
            }
        }
        done[root] = 1;
    }
    if (order.size() != ns) return;
    fused_encode(pl, order, false, fp);
}

// The program of the steps `order` (plan step indices, a topological order).  segment = false: the whole plan.
// segment = true: a run of steps inside a launch-per-bucket plan -- intermediates made by earlier launches are read
// from the plan's global arena (operand kind 1 without observed axes), an output that a LATER launch reads is
// written there (kFusedToGlobal); only intermediates born and consumed inside the run live in shared memory.
// BNPP_FUSED_STACK=0: first-fit arenas only (tests run both layouts)
static bool fused_stack_arena()
{
    const char *e = getenv("BNPP_FUSED_STACK");
    return !(e && e[0] == '0');
}

EncodeScratch::EncodeScratch(const bnpp_ve_plan *pl)
    : pos(pl->steps.size(), -1), last_use(pl->f.size(), -1), producer(pl->f.size(), -1), reads(pl->f.size(), 0), side(pl->f.size(), 0),
      in_smem(pl->f.size(), 0), read_inside(pl->f.size(), 0), read_outside(pl->f.size(), 0), aoff(pl->f.size(), 0), at(pl->f.size(), 0),
      cons_off(pl->f.size() + 1, 0)
{
    const size_t all = pl->steps.size();
    for (size_t s = 0; s < all; ++s) {
        if (pl->steps[s].out >= 0) producer[pl->steps[s].out] = (int)s;
        for (int id : pl->steps[s].operands)
            if (pl->f[id].src < 0) ++cons_off[id + 1];
    }
    for (size_t i = 0; i < pl->f.size(); ++i) cons_off[i + 1] += cons_off[i];
    cons.resize(cons_off.back());
    std::vector<int> fill(cons_off.begin(), cons_off.end() - 1);
    for (size_t s = 0; s < all; ++s)
        for (int id : pl->steps[s].operands)
            if (pl->f[id].src < 0) cons[fill[id]++] = (int)s;
}

void fused_encode(bnpp_ve_plan *pl, const std::vector<int> &order, bool segment, FusedProgram &fp, EncodeScratch *scratch)
{
    fp.built = true;
    fp.ok = false;
    const size_t ns = order.size();
    if (ns == 0) return;
    std::unique_ptr<EncodeScratch> own;
    if (!scratch) {
        own.reset(new EncodeScratch(pl));
        scratch = own.get();
    }
    std::vector<int> &pos = scratch->pos, &last_use = scratch->last_use, &producer = scratch->producer;
    std::vector<char> &in_smem = scratch->in_smem, &read_inside = scratch->read_inside, &read_outside = scratch->read_outside;
    std::vector<uint64_t> &aoff = scratch->aoff;
    // whatever this call marks (its steps, the intermediates they make) goes back to the initial state on every way out
    struct Reset {
        EncodeScratch *sc;
        const bnpp_ve_plan *pl;
        const std::vector<int> &order;
        ~Reset()
        {
            for (int st : order) {
                sc->pos[st] = -1;
                const int id = pl->steps[st].out;
                if (id < 0) continue;
                sc->last_use[id] = -1;
                sc->reads[id] = sc->side[id] = 0;
                sc->in_smem[id] = sc->read_inside[id] = sc->read_outside[id] = 0;
                sc->aoff[id] = sc->at[id] = 0;
            }
        }
    } reset{scratch, pl, order};
    for (size_t i = 0; i < ns; ++i) pos[order[i]] = (int)i;
    // an intermediate lives in shared memory iff it is made here; then every reader must be here too
    for (size_t i = 0; i < ns; ++i) {
        const int id = pl->steps[order[i]].out;
        if (id < 0 || pl->f[id].src >= 0) continue;
        for (int c = scratch->cons_off[id]; c < scratch->cons_off[id + 1]; ++c) {
            const int s = scratch->cons[c];
            if (pos[s] >= 0) {
                read_inside[id] = 1;
                last_use[id] = std::max(last_use[id], pos[s]);
            } else {
                read_outside[id] = 1;
            }
        }
        if (!segment) in_smem[id] = 1;
        else if (read_inside[id] && read_outside[id]) return;       // two homes: not a run this builder takes
        else in_smem[id] = read_inside[id];
    }
    // arena of one evidence set: first fit over the order, in doubles
    std::vector<std::pair<uint64_t, uint64_t>> free_list;   // (offset, size)
    uint64_t top = 0, peak = 0;
    auto take = [&](uint64_t n) {
        n = (n + 1) & ~1ull;      // tables start on even offsets: the kernel moves pairs of doubles
        for (size_t i = 0; i < free_list.size(); ++i)
            if (free_list[i].second >= n) {
                const uint64_t off = free_list[i].first;
                free_list[i].first += n;
                free_list[i].second -= n;
                if (!free_list[i].second) free_list.erase(free_list.begin() + i);
                return off;
            }
        const uint64_t off = top;
        top += n;
        return off;
    };
    auto give = [&](uint64_t off, uint64_t n) {
        n = (n + 1) & ~1ull;
        free_list.push_back({off, n});
        std::sort(free_list.begin(), free_list.end());
        for (size_t i = 0; i + 1 < free_list.size();)
            if (free_list[i].first + free_list[i].second == free_list[i + 1].first) {
                free_list[i].second += free_list[i + 1].second;
                free_list.erase(free_list.begin() + i + 1);
            } else ++i;
        if (!free_list.empty() && free_list.back().first + free_list.back().second == top) {
            top = free_list.back().first;
            free_list.pop_back();
        }
    };
    for (size_t i = 0; i < ns; ++i) {
        const PlanStep &st = pl->steps[order[i]];
        if (st.out >= 0 && in_smem[st.out]) {
            aoff[st.out] = take(pl->f[st.out].size);
            peak = std::max(peak, top);
        }
        std::vector<int> seen;
        for (int id : st.operands) {
            if (pl->f[id].src >= 0 || !in_smem[id] || last_use[id] != (int)i || std::find(seen.begin(), seen.end(), id) != seen.end())
                continue;
            seen.push_back(id);
            give(aoff[id], pl->f[id].size);
        }
        if (st.out >= 0 && in_smem[st.out] && last_use[st.out] < 0) give(aoff[st.out], pl->f[st.out].size);   // never read
    }
    // When the steps form a forest (every shared-memory intermediate read by exactly one step) and `order` is a
    // post-order walk of it, a TWO-ENDED STACK lays the arena out without the holes of first fit: the result of a step
    // goes to the end opposite to its operands' (which are the top of their end: popped as soon as the step is done).
    // The peak is the live set of the walk itself (config 5: 192 doubles where first fit needs 240) -- the arena of a
    // set is what bounds the evidence sets resident on an SM.
    {
        std::vector<int> &reads = scratch->reads, &side = scratch->side;
        bool forest = true;
        for (size_t i = 0; i < ns && forest; ++i) {
            std::vector<int> seen;
            for (int id : pl->steps[order[i]].operands) {
                if (pl->f[id].src >= 0 || !in_smem[id] || std::find(seen.begin(), seen.end(), id) != seen.end()) continue;
                seen.push_back(id);
                if (++reads[id] > 1) forest = false;
            }
        }
        // sides top down: an output sits opposite to the outputs of the steps it feeds on
        for (size_t i = ns; i-- > 0 && forest;) {
            const PlanStep &st = pl->steps[order[i]];
            const int mine = (st.out >= 0 && in_smem[st.out]) ? side[st.out] : 0;
            for (int id : st.operands)
                if (pl->f[id].src < 0 && in_smem[id]) side[id] = 1 - mine;
        }
        std::vector<uint64_t> &at = scratch->at;        // distance of the table's START (side 0) / END (side 1) from its end of the arena
        uint64_t tops[2] = {0, 0}, best = 0;
        for (size_t i = 0; i < ns && forest; ++i) {
            const PlanStep &st = pl->steps[order[i]];
            if (st.out >= 0 && in_smem[st.out]) {
                const uint64_t n = (pl->f[st.out].size + 1) & ~1ull;
                const int sd = side[st.out];
                at[st.out] = sd == 0 ? tops[0] : tops[1] + n;
                tops[sd] += n;
                best = std::max(best, tops[0] + tops[1]);
            }
            std::vector<int> seen;
            for (int id : st.operands) {
                if (pl->f[id].src >= 0 || !in_smem[id] || std::find(seen.begin(), seen.end(), id) != seen.end()) continue;
                seen.push_back(id);
                tops[side[id]] -= (pl->f[id].size + 1) & ~1ull;
            }
            // popped tables must have been the top of their end: whatever is left starts below them
            for (int id : seen) {
                const uint64_t n = (pl->f[id].size + 1) & ~1ull;
                const uint64_t start = side[id] == 0 ? at[id] : at[id] - n;
                if (start < tops[side[id]]) forest = false;
            }
            if (st.out >= 0 && in_smem[st.out] && last_use[st.out] < 0) tops[side[st.out]] -= (pl->f[st.out].size + 1) & ~1ull;
        }
        if (forest && best > 0 && best < peak && fused_stack_arena()) {
            for (size_t i = 0; i < ns; ++i) {
                const int id = pl->steps[order[i]].out;
                if (id >= 0 && in_smem[id]) aoff[id] = side[id] == 0 ? at[id] : best - at[id];
            }
            peak = best;
        }
    }
    if (peak >= (1ull << 24)) return;

    // the program and the operand-offset tables
    fp.prog.clear();
    fp.offtab.clear();
    fp.ptr_slots.clear();
    fp.max_out = 0;
    for (size_t i = 0; i < ns; ++i) {
        const PlanStep &st = pl->steps[order[i]];
        const std::vector<uint32_t> &ovar = st.out == -2 ? st.rvar : pl->f[st.out].var;
        const std::vector<uint32_t> &ocard = st.out == -2 ? st.rcard : pl->f[st.out].card;
        const uint64_t n_out = table_size(ocard);
        const int k = (int)st.operands.size(), wr = (int)ovar.size();
        if (n_out > kFusedMaxUnion) return;
        if (fp.offtab.size() + (uint64_t)k * n_out > kFusedMaxTabWords) return;
        fp.max_out = std::max<uint32_t>(fp.max_out, (uint32_t)n_out);
        uint32_t cx = 1;
        std::vector<std::vector<uint64_t>> axs(k, std::vector<uint64_t>(wr, 0));
        std::vector<uint64_t> sx(k, 0);
        for (int q = 0; q < k; ++q) {
            const PlanFactor &pf = pl->f[st.operands[q]];
            uint64_t dense = 1;
            for (int a = (int)pf.var.size() - 1; a >= 0; --a) {
                const uint64_t stv = pf.stride.empty() ? dense : (uint64_t)pf.stride[a];
                dense *= pf.card[a];
                if (st.elim >= 0 && pf.var[a] == (uint64_t)st.elim) {
                    sx[q] = stv;
                    cx = pf.card[a];
                    continue;
                }
                int at = -1;
                for (int j = 0; j < wr; ++j)
                    if (ovar[j] == pf.var[a]) { at = j; break; }
                if (at < 0 || stv >= (1ull << 32)) return;
                axs[q][at] = stv;
            }
            if (sx[q] >= (1ull << 32) || pf.obs.size() > 255) return;
        }
        const uint32_t tab_off = (uint32_t)fp.offtab.size();
        fp.offtab.resize(fp.offtab.size() + (size_t)k * n_out, 0);
        {
            // odometer over the output axes, the operand offsets updated incrementally
            std::vector<uint32_t> digit(wr, 0);
            uint64_t cur[kMaxK] = {0};
            for (int q = 0; q < k; ++q) {
                uint64_t top = 0;
                for (int a = 0; a < wr; ++a) top += (uint64_t)(ocard[a] - 1) * axs[q][a];
                if (top >= (1ull << 32)) return;
            }
            for (uint64_t o = 0; o < n_out; ++o) {
                for (int q = 0; q < k; ++q) fp.offtab[tab_off + (size_t)q * n_out + o] = (uint32_t)cur[q];
                for (int a = wr - 1; a >= 0; --a) {
                    if (++digit[a] < ocard[a]) {
                        for (int q = 0; q < k; ++q) cur[q] += axs[q][a];
                        break;
                    }
                    digit[a] = 0;
                    for (int q = 0; q < k; ++q) cur[q] -= (uint64_t)(ocard[a] - 1) * axs[q][a];
                }
            }
        }
        // the pair form: binary eliminated variable at stride 1 in every arena operand, on even offsets
        bool pairs = cx == 2;
        for (int q = 0; q < k && pairs; ++q) {
            if (pl->f[st.operands[q]].src >= 0 || !in_smem[st.operands[q]]) continue;
            pairs = sx[q] == 1;
            for (uint64_t o = 0; o < n_out && pairs; ++o) pairs = (fp.offtab[tab_off + (size_t)q * n_out + o] & 1u) == 0;
        }
        uint32_t flags = pairs ? kFusedPairs : 0u, out_off;
        const bool argmax = st.max;
        if (argmax) {
            if (pl->arg_row[order[i]] >= (1ull << 32)) return;
            flags |= kFusedMax;
        }
        if (st.out == -2) {
            flags |= kFusedToResult | (st.want_z && !pl->is_mpe ? kFusedWantZ : 0u);
            if (st.roff >= (1ull << 32)) return;
            out_off = (uint32_t)st.roff;
        } else if (in_smem[st.out]) {
            out_off = (uint32_t)aoff[st.out];
        } else {
            flags |= kFusedToGlobal;      // a later launch reads it: absolute address in header words 5-6
            out_off = 0;
        }
        const uint32_t head[kFusedHeaderWords] = {(uint32_t)n_out, cx, (uint32_t)k | (flags << 8), out_off, tab_off, 0, 0,
                                                  argmax ? (uint32_t)pl->arg_row[order[i]] : 0u};
        if (flags & kFusedToGlobal) {
            const uint32_t at = (uint32_t)fp.prog.size();
            fp.ptr_slots.push_back({at + 5, at + 6, 1, st.out});
        }
        fp.prog.insert(fp.prog.end(), head, head + kFusedHeaderWords);
        for (int q = 0; q < k; ++q) {
            const PlanFactor &pf = pl->f[st.operands[q]];
            const uint32_t at = (uint32_t)fp.prog.size();
            if (pf.src < 0 && in_smem[st.operands[q]]) {
                const uint32_t rec[kFusedOperandWords] = {0u, (uint32_t)aoff[st.operands[q]], (uint32_t)sx[q], 0u};
                fp.prog.insert(fp.prog.end(), rec, rec + kFusedOperandWords);
                continue;
            }
            if (pf.src < 0) {
                // made by an earlier launch: a global table like a CPT, without observed axes
                if (producer[st.operands[q]] < 0 || pos[producer[st.operands[q]]] >= 0) return;
                const uint32_t rec[kFusedOperandWords] = {1u, 0u, (uint32_t)sx[q], 0u};
                fp.prog.insert(fp.prog.end(), rec, rec + kFusedOperandWords);
                fp.ptr_slots.push_back({at + 1, at + 3, 1, st.operands[q]});
                continue;
            }
            const uint32_t rec[kFusedOperandWords] = {1u | ((uint32_t)pf.obs.size() << 8), 0u, (uint32_t)sx[q], 0u};
            fp.prog.insert(fp.prog.end(), rec, rec + kFusedOperandWords);
            fp.ptr_slots.push_back({at + 1, at + 3, 0, pf.src});
            for (size_t j = 0; j < pf.obs.size(); j += 2) {
                uint32_t pair[4] = {(uint32_t)pf.obs[j].first, (uint32_t)pf.obs[j].second, 0u, 0u};
                if (pf.obs[j].first >= (1ll << 32)) return;
                if (j + 1 < pf.obs.size()) {
                    if (pf.obs[j + 1].first >= (1ll << 32)) return;
                    pair[2] = (uint32_t)pf.obs[j + 1].first;
                    pair[3] = (uint32_t)pf.obs[j + 1].second;
                }
                fp.prog.insert(fp.prog.end(), pair, pair + 4);
            }
        }
    }
    if (fp.prog.size() >= (1ull << 31)) return;
    fp.n_steps = (uint32_t)ns;
    fp.total_union = 0;
    for (int s : order) fp.total_union += pl->steps[s].union_entries;
    fp.arena = (uint32_t)std::max<uint64_t>((peak + 1) & ~1ull, 2);
    fp.slot_addr.assign(fp.ptr_slots.size(), 0);
    fp.ok = true;
}

// lanes per evidence set for a run over nb sets; 0 = this run is not fused
int fused_pick(bnpp_ve_plan *pl, uint32_t nb)
{
    if (!pl->fused_mode || pl->profiling) return 0;
    FusedProgram &fp = pl->fused;
    if (!fp.built) fused_build(pl);
    if (!fp.ok) return 0;
    int G = 0;
    if (nb == 1) {
        G = fp.max_out >= 128 ? 128 : 32;
        if (fused_smem_bytes(G, fp.arena) > kFusedSmemLimit) G = 128;
    } else {
        // at least ~16 warps per SM: the arena of one warp's sets within 13.75 KB
        for (int g : {8, 16, 32})
            if (!G && (uint64_t)(32 / g) * fp.arena * sizeof(double) <= 14080) G = g;
        if (!G) G = fused_smem_bytes(32, fp.arena) <= kFusedSmemLimit ? 32 : 128;
        if (const char *e = getenv("BNPP_FUSED_G")) {      // experiments: force the lanes per set of batched runs
            const int g = atoi(e);
            if (fused_valid_g(g)) G = g;
        }
    }
    // the steps of one set run one after the other on its G lanes: a set with much work needs a wider group,
    // and beyond a CTA per set the launch-per-bucket path (all SMs on every step) is the better one
    while (fp.total_union / G > kFusedMaxLaneWork && G < 128) G = G < 32 ? 2 * G : 128;
    if (fp.total_union / G > kFusedMaxLaneWork) return 0;
    if (fused_smem_bytes(G, fp.arena) > kFusedSmemLimit) return 0;
    // a batch wants many resident CTAs (the kernel hides latency with warps, measured: 4 -> 7 CTAs per SM = 5.6 -> 3.5 ms);
    // an arena that allows fewer than four per SM is better served by one launch per bucket
    if (nb > 1 && fused_smem_bytes(G, fp.arena) > (56u << 10)) return 0;
    return G;
}

// 0: off, 1: on, 2 (default): on for plans with at least kTasksMinSmall small steps -- cutting a plan into tasks is host
// work (the step programs of the tasks, ~0.3 ms) that a query with a few dozen buckets never earns back
int segments_default_mode()
{
    static const int mode = [] {
        const char *e = getenv("BNPP_FUSED_SEGMENTS");
        return !e ? 2 : (e[0] == '0' ? 0 : 1);
    }();
    return mode;
}
constexpr size_t kTasksMinSmall = 96;

constexpr uint64_t kTaskMaxWork = 1ull << 16;       // union entries one task (one CTA) may walk: a few microseconds, like a launch

bool step_is_small(const PlanStep &st)
{
    return st.union_entries <= kFusedMaxUnion && !st.operands.empty() && (int)st.operands.size() <= kMaxK;
}

void free_tasks(bnpp_ve_plan *pl)
{
    dev_free(pl->ctx, pl->tasks_prog_dev);
    dev_free(pl->ctx, pl->tasks_tab_dev);
    dev_free(pl->ctx, pl->tasks_rec_dev);
    pl->tasks_uploaded = false;
    pl->tasks_prog.clear();
    pl->tasks_tab_words = 0;
    pl->tasks_rec.clear();
    pl->tasks_slots.clear();
    pl->segs.clear();
    pl->groups.clear();
    pl->group_at.clear();
    pl->segments_built = false;
}

// Puts step order[j] at position j, with its level and task (a task root renumbered to its new position) when the plan
// is levelled.  Any topological order gives the same numbers: operand lists are untouched.  The arena is laid out
// again over the new order (around the plan's windows as they stand); the launches resolved for the old order and
// the K9 program are dropped.
void reorder_steps(bnpp_ve_plan *pl, const std::vector<int> &order)
{
    const size_t ns = pl->steps.size();
    const bool leveled = pl->step_level.size() == ns && pl->step_task.size() == ns;
    std::vector<int> pos(ns);
    for (size_t j = 0; j < ns; ++j) pos[order[j]] = (int)j;
    std::vector<PlanStep> steps;
    steps.reserve(ns);
    std::vector<int> level, task;
    for (size_t j = 0; j < ns; ++j) {
        steps.push_back(std::move(pl->steps[order[j]]));
        if (leveled) {
            level.push_back(pl->step_level[order[j]]);
            task.push_back(pl->step_task[order[j]] >= 0 ? pos[pl->step_task[order[j]]] : -1);
        }
    }
    pl->steps = std::move(steps);
    if (leveled) {
        pl->step_level = std::move(level);
        pl->step_task = std::move(task);
    }
    for (PlanFactor &pf : pl->f) pf.last_use = -1;
    for (size_t i = 0; i < ns; ++i)
        for (int id : pl->steps[i].operands) pl->f[id].last_use = (int)i;
    pl->arena_doubles = 0;
    build_exec(pl);
    // a levelled plan reports its arena (level-wide lifetimes), any other the live intermediates, as create_plan does
    pl->peak_bytes = leveled ? 8 * pl->arena_doubles : live_peak(pl);
    pl->exec.clear();
    pl->exec_planned.clear();
    dev_free(pl->ctx, pl->fused.prog_dev);
    dev_free(pl->ctx, pl->fused.offtab_dev);
    pl->fused = FusedProgram();
}

// Tasks and levels.  The steps of a plan form a DAG (a tree for PR plans).  A small step absorbs the tasks of its
// small producers while the task stays within kTaskMaxWork (and segments_max_steps) and the producer's output has no
// other reader -- such an intermediate then lives in the task's shared memory.  A task's level is one more than the
// highest level it reads from; wide steps are levelled the same way.  The step list is re-ordered by (level, task),
// which keeps it topological -- operand lists, hence the numbers, are untouched -- and the arena is laid out again
// with level-wide lifetimes.  Only before the first run of a plan.
void build_levels(bnpp_ve_plan *pl)
{
    if (pl->runs || pl->arena || pl->batch_runs || !pl->offtab_host.empty()) return;
    const size_t ns = pl->steps.size();
    if (pl->segments_mode == 2) {
        size_t n_small = 0;
        for (const PlanStep &st : pl->steps) n_small += step_is_small(st);
        if (n_small < kTasksMinSmall) {
            pl->segments_mode = 0;      // this plan: one launch per bucket, in elimination order
            return;
        }
        pl->segments_mode = 1;
    }
    free_tasks(pl);
    pl->levels_built = true;
    if (ns < 2) {
        pl->step_level.assign(ns, 0);
        pl->step_task.assign(ns, -1);
        return;
    }
    std::vector<int> producer(pl->f.size(), -1), readers(pl->f.size(), 0);
    for (size_t i = 0; i < ns; ++i) {
        if (pl->steps[i].out >= 0) producer[pl->steps[i].out] = (int)i;
        std::vector<int> seen;
        for (int id : pl->steps[i].operands)
            if (pl->f[id].src < 0 && std::find(seen.begin(), seen.end(), id) == seen.end()) {
                seen.push_back(id);
                readers[id]++;
            }
    }
    std::vector<int> parent(ns, -1), level(ns, 0), nst(ns, 1);
    std::vector<uint64_t> work(ns, 0);
    std::vector<char> small(ns, 0);
    for (size_t i = 0; i < ns; ++i) {
        const PlanStep &st = pl->steps[i];
        small[i] = step_is_small(st);
        work[i] = st.union_entries;
        std::vector<int> kids;
        for (int id : st.operands) {
            const int c = pl->f[id].src < 0 ? producer[id] : -1;
            if (c >= 0 && std::find(kids.begin(), kids.end(), c) == kids.end()) kids.push_back(c);
        }
        std::stable_sort(kids.begin(), kids.end(), [&](int x, int y) { return work[x] < work[y]; });
        for (int c : kids) {
            // within the work budget -- or a chain link (the only producer this step waits for): cutting a chain buys no
            // parallelism, only launches
            const bool absorb = small[i] && small[c] && parent[c] < 0 && readers[pl->steps[c].out] == 1 &&
                                (work[i] + work[c] <= kTaskMaxWork || (kids.size() == 1 && work[i] + work[c] <= 8 * kTaskMaxWork)) &&
                                (!pl->segments_max_steps || (uint32_t)(nst[i] + nst[c]) <= pl->segments_max_steps);
            if (absorb) {
                parent[c] = (int)i;
                work[i] += work[c];
                nst[i] += nst[c];
                level[i] = std::max(level[i], level[c]);
            } else {
                level[i] = std::max(level[i], level[c] + 1);
            }
        }
    }
    // root of every small step's task; a step absorbed into a task takes the task's level
    std::vector<int> root(ns, -1);
    for (size_t i = ns; i-- > 0;) {
        if (!small[i]) continue;
        root[i] = parent[i] >= 0 ? root[parent[i]] : (int)i;
        if (parent[i] >= 0) level[i] = level[root[i]];
    }
    std::vector<int> order(ns);
    for (size_t i = 0; i < ns; ++i) order[i] = (int)i;
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) {
        if (level[x] != level[y]) return level[x] < level[y];
        if (small[x] != small[y]) return small[x] > small[y];         // the level's tasks first, then its wide steps
        if (small[x] && root[x] != root[y]) return root[x] < root[y];
        return x < y;
    });
    pl->step_level = level;
    pl->step_task = root;       // -1 for wide steps
    reorder_steps(pl, order);
}

// the step program of every task, the groups (one ve_tasks launch each), and all programs in one buffer
void build_segments(bnpp_ve_plan *pl)
{
    free_tasks(pl);
    pl->segments_built = true;
    const size_t ns = pl->steps.size();
    pl->group_at.assign(ns, -1);
    if (!pl->levels_built || pl->step_task.size() != ns) return;
    // tasks = maximal runs of steps with the same task root; groups = maximal runs of tasks with the same level
    std::vector<bnpp_ve_plan::Segment> all;
    for (size_t t = 0; t < ns;) {
        if (pl->step_task[t] < 0) { ++t; continue; }
        size_t u = t;
        while (u < ns && pl->step_task[u] == pl->step_task[t]) ++u;
        bnpp_ve_plan::Segment seg;
        seg.a = (int)t;
        seg.b = (int)u;
        seg.level = pl->step_level[t];
        all.push_back(std::move(seg));
        t = u;
    }
    // the programs are independent of one another: encode them on a few host threads (the offset tables of a
    // 1000-bucket network are ~0.5 M words; a one-shot CLI query pays for them inside its timed region)
    auto encode = [&](size_t i, EncodeScratch *sc) {
        std::vector<int> order;
        for (int k = all[i].a; k < all[i].b; ++k) order.push_back(k);
        fused_encode(pl, order, true, all[i].prog, sc);
    };
    const auto tb0 = std::chrono::steady_clock::now();
    const unsigned hw = std::max(1u, std::min(8u, std::thread::hardware_concurrency()));
    if (all.size() >= 8 && hw > 1) {
        std::atomic<size_t> next(0);
        std::vector<std::thread> pool;
        for (unsigned w = 0; w < hw; ++w)
            pool.emplace_back([&] {
                EncodeScratch sc(pl);
                for (size_t i = next.fetch_add(1); i < all.size(); i = next.fetch_add(1)) encode(i, &sc);
            });
        for (auto &th : pool) th.join();
    } else if (!all.empty()) {
        EncodeScratch sc(pl);
        for (size_t i = 0; i < all.size(); ++i) encode(i, &sc);
    }
    const auto tb1 = std::chrono::steady_clock::now();
    if (getenv("BNPP_TIMING"))
        fprintf(stderr, "bnpp timing: %zu task programs encoded in %.3f ms on %u thread(s)\n", all.size(),
                std::chrono::duration<double, std::milli>(tb1 - tb0).count(), all.size() >= 8 ? hw : 1u);
    for (size_t i = 0; i < all.size();) {
        size_t j = i;
        while (j < all.size() && all[j].level == all[i].level && all[j].a == (j == i ? all[i].a : all[j - 1].b)) ++j;
        bnpp_ve_plan::Group g;
        g.a = all[i].a;
        g.b = all[j - 1].b;
        g.first_seg = (int)pl->segs.size();
        bool ok = true;
        for (size_t t = i; t < j && ok; ++t) ok = all[t].prog.ok && fused_smem_bytes(128, all[t].prog.arena) <= kFusedSmemLimit;
        if (ok) {
            for (size_t t = i; t < j; ++t) {
                g.max_arena = std::max(g.max_arena, all[t].prog.arena);
                pl->segs.push_back(std::move(all[t]));
            }
            g.n_segs = (int)(j - i);
            pl->group_at[g.a] = (int)pl->groups.size();
            pl->groups.push_back(g);
        }       // else: this level's small steps stay one launch each
        i = j;
    }
    const auto tb2 = std::chrono::steady_clock::now();
    // one buffer for all programs, one for all offset tables, one record per task
    size_t prog_words = 0;
    for (const auto &seg : pl->segs) prog_words += seg.prog.prog.size();
    pl->tasks_prog.reserve(prog_words);
    pl->tasks_rec.reserve(pl->segs.size());
    for (const auto &seg : pl->segs) {
        TaskRecord r;
        r.prog_off = (uint32_t)pl->tasks_prog.size();
        r.tab_base = (uint32_t)pl->tasks_tab_words;
        r.n_steps = seg.prog.n_steps;
        r.arena = seg.prog.arena;
        for (const auto &slot : seg.prog.ptr_slots)
            pl->tasks_slots.push_back({slot.lo + r.prog_off, slot.hi + r.prog_off, slot.kind, slot.index, 0});
        pl->tasks_prog.insert(pl->tasks_prog.end(), seg.prog.prog.begin(), seg.prog.prog.end());
        pl->tasks_tab_words += (seg.prog.offtab.size() + 3) / 4 * 4;
        pl->tasks_rec.push_back(r);
    }
    if (getenv("BNPP_TIMING"))
        fprintf(stderr, "bnpp timing: groups %.3f ms, one buffer %.3f ms\n", std::chrono::duration<double, std::milli>(tb2 - tb1).count(),
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tb2).count());
}

// ---- K11: windows (chain.hpp) ---------------------------------------------------------------------------------
// A LINK joins step s to step t when t is the only reader of s's output, neither is the result step nor wants Z, t
// eliminates the innermost axis of s's output, t's union has >= kChainMinUnion entries, every variable of both steps
// is binary and every other operand of t (a SIDE) has <= kChainMaxSide entries.  A window is a chain of links
// s0 -> t1 -> ... -> tm (2 <= m <= chain_depth) whose head -- s0's output -- holds the m eliminated variables as its
// m fastest axes; it is cut where a level's tile would exceed kChainTile doubles, where a variable a level adds would
// be eliminated inside the window, and where the shape has no contract_chain instantiation.  Plans with max steps
// (MPE / MAP) form none.
constexpr uint64_t kChainMinUnion = 1ull << 20;
constexpr uint64_t kChainMaxSide = 1ull << 16;

// stride of variable v in factor pf (0: absent); dense factors are row-major over (var, card)
int64_t factor_stride(const PlanFactor &pf, uint32_t v)
{
    int64_t dense = 1;
    for (size_t i = pf.var.size(); i-- > 0;) {
        const int64_t st = pf.stride.empty() ? dense : pf.stride[i];
        if (pf.var[i] == v) return st;
        dense *= pf.card[i];
    }
    return 0;
}

// rest index -> offset, as bit-fields: rest bit b is variable rest[b]
bool chain_fields(const PlanFactor &pf, const std::vector<uint32_t> &rest, Field *f, uint8_t &nf)
{
    nf = 0;
    for (size_t b = 0; b < rest.size();) {
        const int64_t st = factor_stride(pf, rest[b]);
        if (!st) { ++b; continue; }
        size_t len = 1;
        while (b + len < rest.size() && factor_stride(pf, rest[b + len]) == (st << len)) ++len;
        if (nf == kChainMaxFields || st > UINT32_MAX) return false;
        f[nf++] = Field{(uint32_t)((1ull << len) - 1), (uint32_t)st, (uint32_t)b};
        b += len;
    }
    return true;
}

// the window of head `head` over the levels `lv` (plan step indices) -> w, or false when it has no kernel
bool chain_shape(const bnpp_ve_plan *pl, int head, const std::vector<int> &lv, bnpp_ve_plan::Window &w)
{
    const int m = (int)lv.size();
    const PlanFactor &H = pl->f[head];
    const int nh = (int)H.var.size();
    if (m < 2 || m > kChainMaxLevels || nh < m || !H.stride.empty()) return false;
    std::vector<uint32_t> rest;                     // rest bit b -> variable (bit 0 = the fastest rest axis)
    for (int b = nh - m - 1; b >= 0; --b) rest.push_back(H.var[b]);
    const uint64_t n_items = H.size >> m;
    if (n_items % chain_chunk_items(m) || n_items > UINT32_MAX) return false;
    w = bnpp_ve_plan::Window();
    w.m = m;
    w.head = head;
    memset(&w.p, 0, sizeof w.p);
    w.p.n_items = (uint32_t)n_items;
    std::vector<uint32_t> added;                    // new variables, in order of addition
    std::vector<int> sides_seen;
    int in = head, nb = 0;
    w.bytes = 8 * H.size;
    for (int j = 0; j < m; ++j) {
        const PlanStep &st = pl->steps[lv[j]];
        if (st.elim != (int64_t)H.var[nh - 1 - j] || st.out < 0) return false;
        // union bits: the eliminated variable, the head's later tile variables, the added ones
        std::vector<uint32_t> ub;
        for (int i = j; i < m; ++i) ub.push_back(H.var[nh - 1 - i]);
        ub.insert(ub.end(), added.begin(), added.end());
        ChainLevel &L = w.p.lv[j];
        int hpos = -1, k = 0;
        for (size_t q = 0; q < st.operands.size(); ++q) {
            const int id = st.operands[q];
            if (id == in && hpos < 0) { hpos = (int)q; continue; }
            if (k == kChainMaxSides) return false;
            w.side[j][k++] = id;
        }
        if (hpos < 0) return false;
        // the kernel multiplies (s0 * s1) * h: a three-operand step lists its operands by size (fold_small), the head last
        if (k == 2 && hpos != 2) return false;
        L.k = (uint8_t)k;
        int add = 0;
        for (int q = 0; q < k; ++q)
            for (uint32_t v : pl->f[w.side[j][q]].var)
                if (std::find(ub.begin(), ub.end(), v) == ub.end() && std::find(rest.begin(), rest.end(), v) == rest.end()) {
                    ub.push_back(v);
                    added.push_back(v);
                    ++add;
                }
        if (add > kChainMaxAdd) return false;
        const int inb = m - j + nb, outb = inb - 1 + add;
        if (inb > 4 || outb > 4 || (int)ub.size() != inb + add) return false;
        w.add[j] = add;
        nb += add;
        for (int q = 0; q < k; ++q) {
            const PlanFactor &S = pl->f[w.side[j][q]];
            for (size_t b = 0; b < ub.size(); ++b) {
                const int64_t sv = factor_stride(S, ub[b]);
                if (sv > UINT32_MAX) return false;
                L.s[q].us[b] = (uint32_t)sv;
            }
            if (!chain_fields(S, rest, L.s[q].f, L.s[q].nf)) return false;
            if (std::find(sides_seen.begin(), sides_seen.end(), w.side[j][q]) == sides_seen.end()) {
                sides_seen.push_back(w.side[j][q]);
                w.bytes += 8 * S.size;
            }
        }
        // the step's output must be exactly (later tile variables, rest, added): what the next level reads
        const PlanFactor &O = pl->f[st.out];
        if (O.var.size() != ub.size() - 1 + rest.size()) return false;
        w.entries += st.union_entries;
        in = st.out;
    }
    const PlanFactor &O = pl->f[in];
    if (O.size > UINT32_MAX || !O.stride.empty()) return false;
    for (size_t i = 0; i < added.size(); ++i) w.p.os[i] = (uint32_t)factor_stride(O, added[i]);
    if (!chain_fields(O, rest, w.p.of, w.p.onf)) return false;
    w.out = in;
    w.bytes += 8 * O.size;
    w.fn = chain_kernel(m, w.add);
    if (!w.fn) return false;
    w.name = chain_name(m, w.add);
    return true;
}

void set_launches(bnpp_ve_plan *pl)
{
    const size_t ns = pl->steps.size();
    if (pl->window_at.size() != ns) pl->window_at.assign(ns, -1);
    pl->launch_first.clear();
    uint64_t bytes = 0;
    for (size_t s = 0; s < ns; ++s) {
        pl->launch_first.push_back((int)s);
        if (pl->window_at[s] >= 0) {
            const auto &w = pl->windows[pl->window_at[s]];
            bytes += w.bytes;
            s = (size_t)w.b - 1;
        } else {
            bytes += pl->steps[s].bytes;
        }
    }
    pl->bytes = bytes;
}

// Find the windows and move the steps that sit between a window's levels (the producers of its side tables among
// them) ahead of its first level, so every window is a contiguous run of the step list.  Any topological order gives
// the same numbers (operand lists are untouched), and no step between the levels reads a level's output (each has
// one reader, the next level), so the new order is topological.  The arena is laid out again over it.
void form_windows(bnpp_ve_plan *pl)
{
    if (pl->runs || pl->arena || pl->batch_runs || !pl->offtab_host.empty()) return;
    const size_t ns = pl->steps.size();
    pl->windows.clear();
    pl->window_at.assign(ns, -1);
    bool any_max = false;
    for (const PlanStep &st : pl->steps) any_max |= st.max;
    if (pl->is_mpe || pl->is_mar || any_max || pl->chain_depth < 2 || ns < 3) {
        set_launches(pl);
        return;
    }
    std::vector<int> producer(pl->f.size(), -1), nread(pl->f.size(), 0), reader(pl->f.size(), -1);
    for (size_t s = 0; s < ns; ++s) {
        const PlanStep &st = pl->steps[s];
        if (st.out >= 0) producer[st.out] = (int)s;
        std::vector<int> seen;
        for (int id : st.operands)
            if (std::find(seen.begin(), seen.end(), id) == seen.end()) {
                seen.push_back(id);
                nread[id]++;
                reader[id] = (int)s;
            }
    }
    auto binary = [&](const PlanStep &st) {
        for (int id : st.operands)
            for (uint32_t c : pl->f[id].card)
                if (c != 2) return false;
        return true;
    };
    auto link = [&](int s) {        // the step s links to, or -1
        const PlanStep &a = pl->steps[s];
        if (a.out < 0 || a.want_z || nread[a.out] != 1 || pl->f[a.out].var.empty()) return -1;
        const int t = reader[a.out];
        const PlanStep &b = pl->steps[t];
        if (b.out < 0 || b.want_z || b.elim < 0 || b.union_entries < kChainMinUnion) return -1;
        if (pl->f[a.out].var.back() != (uint32_t)b.elim || !binary(a) || !binary(b)) return -1;
        for (int id : b.operands)
            if (id != a.out && pl->f[id].size > kChainMaxSide) return -1;
        return t;
    };
    std::vector<int> order(ns), pos(ns);
    for (size_t i = 0; i < ns; ++i) order[i] = pos[i] = (int)i;
    std::vector<std::pair<int, bnpp_ve_plan::Window>> found;     // (first level, window) by plan step index
    for (size_t at = 0; at < ns; ++at) {
        const int t1 = order[at];
        int s0 = -1;
        for (int id : pl->steps[t1].operands)
            if (pl->f[id].src < 0 && producer[id] >= 0 && link(producer[id]) == t1) s0 = producer[id];
        if (s0 < 0) continue;
        std::vector<int> lv{t1};
        while ((uint32_t)lv.size() < std::min<uint32_t>(pl->chain_depth, kChainMaxLevels)) {
            const int t = link(lv.back());
            if (t < 0) break;
            lv.push_back(t);
        }
        bnpp_ve_plan::Window w;
        while (lv.size() >= 2 && !chain_shape(pl, pl->steps[s0].out, lv, w)) lv.pop_back();
        if (lv.size() < 2) continue;
        // [at, pos(tm)]: the steps between the levels first (in their order), then the levels
        std::vector<int> between, span(order.begin() + at, order.begin() + pos[lv.back()] + 1);
        for (int s : span)
            if (std::find(lv.begin(), lv.end(), s) == lv.end()) between.push_back(s);
        size_t q = at;
        for (int s : between) order[q++] = s;
        for (int s : lv) order[q++] = s;
        for (size_t i = at; i < q; ++i) pos[order[i]] = (int)i;
        found.push_back({t1, w});
        at = q - 1;
    }
    if (found.empty()) {
        set_launches(pl);
        return;
    }
    // the windows in the new step order first: the arena is laid out around them.  Every factor keeps its per-step
    // lifetime (the step-by-step engines and the emulator of the tests run them so); build_exec places a window's last
    // output clear of the head and side tables its launch reads meanwhile
    pl->window_at.assign(ns, -1);
    for (auto &fw : found) {
        bnpp_ve_plan::Window &w = fw.second;
        w.a = pos[fw.first];
        w.b = w.a + w.m;
        pl->window_at[w.a] = (int)pl->windows.size();
        pl->windows.push_back(w);
    }
    reorder_steps(pl, order);
    set_launches(pl);
}

// device copies of the task programs; addresses inside them (CPT tables, arena slots) patched when they moved
int upload_tasks(bnpp_ve_plan *pl, const double *const *tables_dev)
{
    bnpp_ctx *ctx = pl->ctx;
    if (pl->segs.empty()) return BNPP_OK;
    bool moved = !pl->tasks_uploaded;
    for (auto &slot : pl->tasks_slots) {
        const uint64_t a = slot.kind == 0 ? reinterpret_cast<uint64_t>(tables_dev[slot.index])
                                          : reinterpret_cast<uint64_t>(pl->arena + pl->arena_off[slot.index]);
        if (a != slot.addr) {
            slot.addr = a;
            pl->tasks_prog[slot.lo] = (uint32_t)a;
            pl->tasks_prog[slot.hi] = (uint32_t)(a >> 32);
            moved = true;
        }
    }
    if (!pl->tasks_prog_dev) {
        // the program last: it marks the three as allocated
        int rc = dev_alloc(ctx, pl->tasks_tab_words + 4, &pl->tasks_tab_dev);
        if (rc == BNPP_OK) rc = dev_alloc(ctx, pl->tasks_rec.size() + 1, &pl->tasks_rec_dev);
        if (rc == BNPP_OK) rc = dev_alloc(ctx, pl->tasks_prog.size() + 36, &pl->tasks_prog_dev);  // the kernel prefetches 32 words past a record
        if (rc != BNPP_OK) return rc;
        // the tables are gathered straight into the pinned ring (one copy to the device); too large for it: task by task
        if (uint32_t *stage = static_cast<uint32_t *>(stage_reserve(ctx, pl->tasks_tab_words * sizeof(uint32_t)))) {
            for (size_t i = 0; i < pl->segs.size(); ++i)
                if (!pl->segs[i].prog.offtab.empty())
                    memcpy(stage + pl->tasks_rec[i].tab_base, pl->segs[i].prog.offtab.data(), pl->segs[i].prog.offtab.size() * sizeof(uint32_t));
            BNPP_CUDA(ctx, cudaMemcpyAsync(pl->tasks_tab_dev, stage, pl->tasks_tab_words * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
        } else {
            for (size_t i = 0; i < pl->segs.size() && rc == BNPP_OK; ++i)
                rc = stage_upload(ctx, pl->tasks_tab_dev + pl->tasks_rec[i].tab_base, pl->segs[i].prog.offtab.data(),
                                  pl->segs[i].prog.offtab.size() * sizeof(uint32_t));
        }
        if (rc == BNPP_OK) rc = stage_upload(ctx, pl->tasks_rec_dev, pl->tasks_rec.data(), pl->tasks_rec.size() * sizeof(TaskRecord));
        if (rc != BNPP_OK) return rc;
    }
    if (moved) {    // stream-ordered after any launch still reading the previous contents
        const int rc = stage_upload(ctx, pl->tasks_prog_dev, pl->tasks_prog.data(), pl->tasks_prog.size() * sizeof(uint32_t));
        if (rc != BNPP_OK) return rc;
    }
    pl->tasks_uploaded = true;
    for (auto &g : pl->groups) {
        if (g.launch_valid) continue;
        const int rc = tasks_geometry(ctx, (uint32_t)g.n_segs, g.max_arena, &g.grid, &g.smem);
        if (rc != BNPP_OK) return rc;
        memset(&g.launch, 0, sizeof g.launch);
        g.launch.prog = pl->tasks_prog_dev;
        g.launch.offtab = pl->tasks_tab_dev;
        g.launch.tasks = pl->tasks_rec_dev + g.first_seg;
        g.launch.n_tasks = (uint32_t)g.n_segs;
        g.launch.n_obs = (uint32_t)pl->n_obs;
        g.launch_valid = true;
    }
    return BNPP_OK;
}

int run_fused(bnpp_ve_plan *pl, FusedProgram &fp, int G, const double *const *tables_dev, uint32_t nb, const uint8_t *ev_dev,
              const uint32_t *obs_val, double *result_dev, double *z_dev, uint8_t *arg_dev = nullptr);

// arg_dev != nullptr: an MPE / MAP program over a batch (ve_fused_max, or ve_fused_mixed when the plan also has summing
// eliminating steps), argmax rows [rows][nb] there
int run_fused(bnpp_ve_plan *pl, int G, const double *const *tables_dev, uint32_t nb, const uint8_t *ev_dev,
              const uint32_t *obs_val, double *result_dev, double *z_dev, uint8_t *arg_dev = nullptr)
{
    return run_fused(pl, pl->fused, G, tables_dev, nb, ev_dev, obs_val, result_dev, z_dev, arg_dev);
}

int run_fused(bnpp_ve_plan *pl, FusedProgram &fp, int G, const double *const *tables_dev, uint32_t nb, const uint8_t *ev_dev,
              const uint32_t *obs_val, double *result_dev, double *z_dev, uint8_t *arg_dev)
{
    bnpp_ctx *ctx = pl->ctx;
    auto address = [&](const FusedProgram::Slot &slot) {
        return slot.kind == 0 ? reinterpret_cast<uint64_t>(tables_dev[slot.index])
                              : reinterpret_cast<uint64_t>(pl->arena + pl->arena_off[slot.index]);
    };
    bool moved = fp.prog_dev == nullptr;
    for (size_t i = 0; i < fp.ptr_slots.size(); ++i) moved = moved || fp.slot_addr[i] != address(fp.ptr_slots[i]);
    if (moved) {
        for (size_t i = 0; i < fp.ptr_slots.size(); ++i) {
            const uint64_t a = address(fp.ptr_slots[i]);
            fp.prog[fp.ptr_slots[i].lo] = (uint32_t)a;
            fp.prog[fp.ptr_slots[i].hi] = (uint32_t)(a >> 32);
            fp.slot_addr[i] = a;
        }
        if (!fp.prog_dev) {
            const int rc = dev_alloc(ctx, fp.prog.size() + 36, &fp.prog_dev);      // the kernel prefetches 32 words past a record
            if (rc != BNPP_OK) return rc;
        }
        // stream-ordered after any launch still reading the previous contents; the pageable source is staged before the call returns
        BNPP_CUDA(ctx, cudaMemcpyAsync(fp.prog_dev, fp.prog.data(), fp.prog.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    }
    if (!fp.offtab_uploaded) {
        const int rc = dev_alloc(ctx, fp.offtab.size() + 4, &fp.offtab_dev);
        if (rc != BNPP_OK) return rc;
        if (!fp.offtab.empty())
            BNPP_CUDA(ctx, cudaMemcpyAsync(fp.offtab_dev, fp.offtab.data(), fp.offtab.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
        fp.offtab_uploaded = true;
    }
    FusedLaunch p;
    memset(&p, 0, sizeof p);
    p.prog = fp.prog_dev;
    p.offtab = fp.offtab_dev;
    p.ev = ev_dev;
    p.result = result_dev;
    p.z = nb == 1 ? z_dev : nullptr;
    p.nb = nb;
    p.n_obs = (uint32_t)pl->n_obs;
    p.n_steps = fp.n_steps;
    p.arena = fp.arena;
    if (!ev_dev && obs_val)
        for (int i = 0; i < pl->n_obs && i < kFusedInlineEv; ++i) p.ev_inline[i] = (uint8_t)obs_val[i];
    if (arg_dev && pl->n_max) {
        FusedMaxLaunch q;
        q.f = p;
        q.arg = arg_dev;
        // a MAP program with summing steps too: the interpreter that takes each step's mode from its kFusedMax flag
        return pl->n_sum_steps ? fused_mixed_launch(ctx, G, q) : fused_max_launch(ctx, G, q);
    }
    return fused_launch(ctx, G, p);
}

// the scopes of the CONDITIONED factors (code/model.cpp:283-287, 362): observed axes are gone
std::vector<std::vector<unsigned>> conditioned_scopes(const std::vector<char> &observed, int nvars, int nfac,
                                                     const bnpp_scope *scopes)
{
    std::vector<std::vector<unsigned>> sc(nfac);
    for (int f = 0; f < nfac; ++f)
        for (int i = 0; i < scopes[f].rank; ++i) {
            const uint32_t v = scopes[f].var_id[i];
            if (v >= (uint32_t)nvars || !observed[v]) sc[f].push_back(v);
        }
    return sc;
}

std::vector<char> observed_mask(int nvars, int n_obs, const uint32_t *obs_var)
{
    std::vector<char> observed(nvars > 0 ? nvars : 1, 0);
    for (int i = 0; i < n_obs; ++i)
        if (obs_var[i] < (uint32_t)nvars) observed[obs_var[i]] = 1;
    return observed;
}

std::vector<unsigned> unobserved(const std::vector<char> &observed, int nvars, int n, const uint32_t *vars)
{
    std::vector<unsigned> v;
    for (int i = 0; i < n; ++i)
        if (vars[i] >= (uint32_t)nvars || !observed[vars[i]]) v.push_back(vars[i]);
    return v;
}

}  // namespace

extern "C" {

static int mpe_finish(bnpp_ve_plan *pl, int nvars, int n_obs, const uint32_t *obs_var, const std::vector<char> *is_map);

// What every plan starts with: the plan, the elimination time of every ordered variable in `rank`, and the input tables
// as evidence-reduced views; no plan when the order or a scope is bad.
static int plan_prelude(bnpp_ctx *ctx, int nfac, const bnpp_scope *scopes, int n_obs, const uint32_t *obs_var, int n_order,
                        const uint32_t *order, bnpp_ve_plan *&plan, RankMap &rank)
{
    plan = nullptr;
    bnpp_ve_plan *pl = new bnpp_ve_plan();
    pl->ctx = ctx;
    pl->n_inputs = nfac;
    pl->n_obs = n_obs;
    pl->obs_card.assign(n_obs, 0);
    pl->fused_mode = fused_default_on() ? 1 : 0;
    pl->segments_mode = segments_default_mode();
    std::map<uint32_t, int> obs_index;
    for (int i = 0; i < n_obs; ++i) obs_index[obs_var[i]] = i;
    for (int i = 0; i < n_order; ++i) {
        if (rank.count(order[i]) || obs_index.count(order[i])) {
            delete pl;
            return fail(ctx, BNPP_EINVAL, "elimination order repeats a variable or names an observed one");
        }
        rank.set(order[i], (uint64_t)i);
    }
    if (int rc = add_inputs(pl, nfac, scopes, obs_index, rank)) {
        delete pl;
        return fail(ctx, rc, "bad factor scope");
    }
    plan = pl;
    return BNPP_OK;
}

// the bucket schedule of bnpp_ve_plan_create; mpe_card != NULL: an MPE plan over that many variables (bnpp_mpe_plan_create),
// or with is_map (per variable id, 1 = a MAP variable) a MAP plan (bnpp_map_plan_create)
static int create_plan(bnpp_ctx *ctx, int nfac, const bnpp_scope *scopes, int n_obs, const uint32_t *obs_var, int n_order,
                       const uint32_t *order, int mpe_nvars, const uint32_t *mpe_card, bnpp_ve_plan **out,
                       const std::vector<char> *is_map = nullptr)
{
    if (!out || nfac < 0 || n_obs < 0 || n_order < 0) return BNPP_EINVAL;   // ctx == NULL: a dry plan (inspect, never run)
    *out = nullptr;
    const auto tc0 = std::chrono::steady_clock::now();
    bnpp_ve_plan *pl;
    RankMap rank;           // elimination time; kept variables after all eliminated ones
    if (int rc = plan_prelude(ctx, nfac, scopes, n_obs, obs_var, n_order, order, pl, rank)) return rc;
    pl->chain_depth = mpe_card ? 0u : chain_depth_knob();
    if (mpe_card) {
        // MPE eliminates every unobserved variable; its argmax tables are uint8 (MAP: those of the MAP variables)
        for (const PlanFactor &pf : pl->f)
            for (size_t a = 0; a < pf.var.size(); ++a) {
                const char *why = nullptr;
                if (pf.var[a] >= (uint32_t)mpe_nvars) why = is_map ? "MAP plan: a scope names a variable id >= nvars"
                                                                   : "MPE plan: a scope names a variable id >= nvars";
                else if (rank.at(pf.var[a]) >= (uint64_t)n_order)
                    why = is_map ? "MAP plan: the order misses an unobserved variable" : "MPE plan: the order misses an unobserved variable";
                else if (pf.card[a] > 255 && !is_map) why = "MPE plan: a variable has more than 255 values (uint8 argmax tables)";
                if (why) {
                    delete pl;
                    return fail(ctx, BNPP_EINVAL, why);
                }
            }
    }

    // bucket = factors whose earliest-eliminated variable is order[i] (code/model.cpp:390-406)
    std::vector<std::vector<int>> bucket(n_order);
    std::vector<int> leftover;
    auto place = [&](int id) {
        uint64_t best = UINT64_MAX;
        for (uint32_t v : pl->f[id].var) best = std::min(best, rank.at(v));
        if (best < (uint64_t)n_order) bucket[best].push_back(id);
        else leftover.push_back(id);
    };
    for (int q = 0; q < nfac; ++q) place(q);

    const auto tc1 = std::chrono::steady_clock::now();
    // eliminate in order (code/model.cpp:409-439)
    for (int i = 0; i < n_order; ++i) {
        std::vector<int> ops = bucket[i];
        if (ops.empty()) continue;    // the reference makes a scalar 1 here; multiplying by it changes nothing
        fold_small(pl, ops, rank);
        shrink(pl, ops, rank);
        const int t = add_step(pl, ops, (int64_t)order[i], rank, false);
        pl->union_entries += pl->steps.back().union_entries;
        pl->max_step_entries = std::max(pl->max_step_entries, pl->steps.back().union_entries);
        place(t);
    }
    // result = product of everything that never entered (or left) a bucket (code/model.cpp:403-405, 436-438)
    if (leftover.empty()) {
        pl->result_size = 1;
    } else {
        shrink(pl, leftover, rank);
        add_step(pl, leftover, -1, rank, true);
    }

    // statistics: bytes, and the peak of live intermediates
    for (const PlanStep &st : pl->steps) pl->bytes += st.bytes;
    pl->peak_bytes = live_peak(pl);
    const auto tc2 = std::chrono::steady_clock::now();
    build_exec(pl);
    const auto tc3 = std::chrono::steady_clock::now();
    if (mpe_card) {
        if (int rc = mpe_finish(pl, mpe_nvars, n_obs, obs_var, is_map)) {
            delete pl;
            return fail(ctx, rc, is_map ? "MAP plan: bad observed variable" : "MPE plan: bad observed variable");
        }
    }
    if (pl->segments_mode) build_levels(pl);
    form_windows(pl);
    if (getenv("BNPP_TIMING")) {
        auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
            return std::chrono::duration<double, std::milli>(b - a).count();
        };
        fprintf(stderr, "bnpp timing: plan create: inputs %.3f ms, elimination steps %.3f ms, arena + exec %.3f ms, levels %.3f ms\n",
                ms(tc0, tc1), ms(tc1, tc2), ms(tc2, tc3), ms(tc3, std::chrono::steady_clock::now()));
    }
    *out = pl;
    return BNPP_OK;
}

int bnpp_ve_plan_create(bnpp_ctx *ctx, int nfac, const bnpp_scope *scopes, int n_obs, const uint32_t *obs_var,
                        int n_order, const uint32_t *order, bnpp_ve_plan **out)
{
    return create_plan(ctx, nfac, scopes, n_obs, obs_var, n_order, order, 0, nullptr, out);
}

int bnpp_mpe_plan_create(bnpp_ctx *ctx, int nvars, const uint32_t *card, int nfac, const bnpp_scope *scopes, int n_obs,
                         const uint32_t *obs_var, int n_order, const uint32_t *order, bnpp_ve_plan **out)
{
    if (!out || nvars < 0 || !card) return BNPP_EINVAL;
    for (int i = 0; i < n_order; ++i)
        if (order[i] >= (uint32_t)nvars) return fail(ctx, BNPP_EINVAL, "MPE plan: an order entry is >= nvars");
    return create_plan(ctx, nfac, scopes, n_obs, obs_var, n_order, order, nvars, card, out);
}

// Marginal MAP: the MPE plan machinery with max steps only where a MAP variable is eliminated; every other eliminating
// step sums.  Exact because the order must eliminate every summed variable before any MAP variable.
int bnpp_map_plan_create(bnpp_ctx *ctx, int nvars, const uint32_t *card, int nfac, const bnpp_scope *scopes, int n_obs,
                         const uint32_t *obs_var, int n_map, const uint32_t *map_var, int n_order, const uint32_t *order,
                         bnpp_ve_plan **out)
{
    if (!out || nvars < 0 || !card || n_map < 0 || n_obs < 0 || n_order < 0 || (n_map && !map_var)) return BNPP_EINVAL;
    std::vector<char> is_map(nvars > 0 ? nvars : 1, 0);
    const std::vector<char> observed = observed_mask(nvars, n_obs, obs_var);
    for (int i = 0; i < n_map; ++i) {
        const uint32_t v = map_var[i];
        const char *why = nullptr;
        if (v >= (uint32_t)nvars) why = "MAP plan: a MAP variable is >= nvars";
        else if (is_map[v]) why = "MAP plan: a MAP variable is repeated";
        else if (observed[v]) why = "MAP plan: a MAP variable is observed";
        else if (card[v] > 255) why = "MAP plan: a MAP variable has more than 255 values (uint8 argmax tables)";
        if (why) return fail(ctx, BNPP_EINVAL, why);
        is_map[v] = 1;
    }
    bool seen_map = false;
    for (int i = 0; i < n_order; ++i) {
        if (order[i] >= (uint32_t)nvars) return fail(ctx, BNPP_EINVAL, "MAP plan: an order entry is >= nvars");
        if (is_map[order[i]]) seen_map = true;
        else if (seen_map) return fail(ctx, BNPP_EINVAL, "MAP plan: the order eliminates a MAP variable before a summed one");
    }
    return create_plan(ctx, nfac, scopes, n_obs, obs_var, n_order, order, nvars, card, out, &is_map);
}

// Argmax arena, argmax rows of batched runs and decode records of an MPE / MAP plan (is_map: NULL = MPE, every
// eliminating step a max step); the K10 path off
static int mpe_finish(bnpp_ve_plan *pl, int nvars, int n_obs, const uint32_t *obs_var, const std::vector<char> *is_map)
{
    pl->is_mpe = true;
    pl->mpe_nvars = (uint32_t)nvars;
    pl->segments_mode = 0;
    pl->arg_off.assign(pl->steps.size(), 0);
    pl->arg_row.assign(pl->steps.size(), 0);
    for (PlanStep &st : pl->steps) {
        st.max = st.elim >= 0 && (!is_map || (*is_map)[st.elim]);
        if (st.max) pl->n_max++;
        else if (st.elim >= 0) pl->n_sum_steps++;
    }
    for (size_t s = 0; s < pl->steps.size(); ++s) {
        const PlanStep &st = pl->steps[s];
        if (!st.max) continue;
        pl->arg_off[s] = (pl->arg_bytes + 255) & ~(uint64_t)255;
        pl->arg_bytes = pl->arg_off[s] + pl->f[st.out].size;
        pl->arg_row[s] = pl->arg_rows;
        pl->arg_rows += pl->f[st.out].size;
    }
    pl->peak_bytes += pl->arg_bytes;
    std::vector<uint32_t> &r = pl->decode_rec;
    for (int i = 0; i < n_obs; ++i) {
        if (obs_var[i] >= (uint32_t)nvars) return BNPP_EINVAL;
        r.push_back(obs_var[i]);
    }
    if (is_map) {
        const std::vector<char> observed = observed_mask(nvars, n_obs, obs_var);
        for (int v = 0; v < nvars; ++v)
            if (!observed[v] && !(*is_map)[v]) {
                r.push_back((uint32_t)v);
                pl->n_summed++;
            }
    }
    for (size_t s = pl->steps.size(); s-- > 0;) {
        const PlanStep &st = pl->steps[s];
        if (!st.max) continue;
        const PlanFactor &of = pl->f[st.out];
        r.push_back((uint32_t)st.elim);
        r.push_back((uint32_t)pl->arg_off[s]);
        r.push_back((uint32_t)(pl->arg_off[s] >> 32));
        r.push_back((uint32_t)of.var.size());
        uint64_t stride = 1;
        std::vector<uint32_t> st_of(of.var.size());
        for (size_t a = of.var.size(); a-- > 0;) {
            st_of[a] = (uint32_t)stride;
            stride *= of.card[a];
        }
        for (size_t a = 0; a < of.var.size(); ++a) {
            r.push_back(of.var[a]);
            r.push_back(st_of[a]);
        }
        pl->n_decode_rec++;
    }
    // the same records with the step's first argmax row in place of its byte offset
    pl->batch_rec = r;
    uint32_t *w = pl->batch_rec.data() + n_obs + pl->n_summed;
    for (size_t s = pl->steps.size(); s-- > 0;) {
        if (!pl->steps[s].max) continue;
        w[1] = (uint32_t)pl->arg_row[s];
        w[2] = (uint32_t)(pl->arg_row[s] >> 32);
        w += 4 + 2 * w[3];
    }
    return BNPP_OK;
}

// All marginals in ONE plan: bucket-tree elimination (two passes over the bucket tree of the
// order) instead of the reference's N complete VE passes (code/model.cpp:326-334; SURVEY §8f
// row 2).  Upward pass = variable elimination, every bucket sends lambda to its parent
// bucket; downward pass, every bucket sends each child the product of everything else it
// holds, summed down to that child's separator.  The marginal of v is the product of all
// functions and messages in bucket v summed over the rest of its clique, normalised --
// mathematically the table the reference's pass for v produces (agreement ~1e-15).
// result layout: per variable id ascending, card(v) doubles, or ONE double (= 1) for an
// observed variable or one that no factor mentions (the reference's width-0 factor [1]).
int bnpp_mar_plan_create(bnpp_ctx *ctx, int nvars, const uint32_t *card, int nfac, const bnpp_scope *scopes, int n_obs,
                         const uint32_t *obs_var, int n_order, const uint32_t *order, bnpp_ve_plan **out)
{
    if (!out || nvars < 0 || nfac < 0 || n_obs < 0 || n_order < 0) return BNPP_EINVAL;   // ctx == NULL: a dry plan
    *out = nullptr;
    bnpp_ve_plan *pl;
    RankMap rank;
    if (int rc = plan_prelude(ctx, nfac, scopes, n_obs, obs_var, n_order, order, pl, rank)) return rc;
    pl->is_mar = true;
    for (const PlanFactor &pf : pl->f)
        for (uint32_t v : pf.var)
            if (rank.at(v) >= (uint64_t)n_order) {
                delete pl;
                return fail(ctx, BNPP_EINVAL, "marginals plan: the order must cover every unobserved variable of the factors");
            }

    // result slices
    std::vector<char> mentioned(nvars, 0);
    for (const PlanFactor &pf : pl->f)
        for (uint32_t v : pf.var)
            if (v < (uint32_t)nvars) mentioned[v] = 1;
    pl->mar_off.assign(nvars, 0);
    pl->mar_size.assign(nvars, 1);
    uint32_t total = 0;
    for (int v = 0; v < nvars; ++v) {
        pl->mar_off[v] = total;
        pl->mar_size[v] = mentioned[v] ? card[v] : 1;
        total += pl->mar_size[v];
    }
    pl->result_size = total;

    struct Bucket {
        std::vector<int> funcs;            // original views and lambdas of the children
        std::vector<int> child_of;         // for funcs[j]: the child bucket that sent it, or -1
        int mu = -1;                       // message from the parent bucket
    };
    std::vector<Bucket> B(n_order);
    auto place = [&](int id, int from) {
        uint64_t best = UINT64_MAX;
        for (uint32_t v : pl->f[id].var) best = std::min(best, rank.at(v));
        if (best < (uint64_t)n_order) {
            B[best].funcs.push_back(id);
            B[best].child_of.push_back(from);
        }
    };
    for (int q = 0; q < nfac; ++q) place(q, -1);
    // upward: lambda_i = sum over order[i] of everything in bucket i
    for (int i = 0; i < n_order; ++i) {
        if (B[i].funcs.empty()) continue;
        std::vector<int> ops = B[i].funcs;
        shrink(pl, ops, rank);
        const int lam = add_step(pl, ops, (int64_t)order[i], rank, false);
        pl->union_entries += pl->steps.back().union_entries;
        pl->max_step_entries = std::max(pl->max_step_entries, pl->steps.back().union_entries);
        place(lam, i);
    }
    // downward
    for (int i = n_order - 1; i >= 0; --i) {
        Bucket &b = B[i];
        if (b.funcs.empty()) continue;
        std::vector<int> G = b.funcs;
        if (b.mu >= 0) G.push_back(b.mu);
        const uint32_t v = order[i];
        if (v < (uint32_t)nvars) chain(pl, G, std::vector<uint32_t>{v}, rank, true, pl->mar_off[v]);
        for (size_t j = 0; j < b.funcs.size(); ++j) {
            const int c = b.child_of[j];
            if (c < 0) continue;
            std::vector<int> Gc;
            for (size_t t = 0; t < G.size(); ++t)
                if (t != j) Gc.push_back(G[t]);
            B[c].mu = chain(pl, Gc, pl->f[b.funcs[j]].var, rank, false, 0);
        }
    }
    pl->result_var.clear();
    pl->result_card.clear();
    pl->result_size = total;

    for (const PlanStep &st : pl->steps) pl->bytes += st.bytes;
    pl->peak_bytes = live_peak(pl);
    build_exec(pl);
    if (pl->segments_mode) build_levels(pl);
    if (!ctx) {
        *out = pl;
        return BNPP_OK;
    }
    if (int rc = dev_alloc(ctx, 2 * (size_t)nvars + 4, &pl->mar_off_dev)) {     // the offsets, then the sizes
        delete pl;
        return rc;
    }
    pl->mar_size_dev = pl->mar_off_dev + nvars;
    if (nvars) {
        cudaMemcpyAsync(pl->mar_off_dev, pl->mar_off.data(), sizeof(uint32_t) * nvars, cudaMemcpyHostToDevice, ctx->stream);
        cudaMemcpyAsync(pl->mar_size_dev, pl->mar_size.data(), sizeof(uint32_t) * nvars, cudaMemcpyHostToDevice, ctx->stream);
        cudaStreamSynchronize(ctx->stream);
    }
    *out = pl;
    return BNPP_OK;
}

// slices of the marginals result: offset and size (doubles) per variable id
int bnpp_mar_plan_layout(const bnpp_ve_plan *pl, int nvars, uint32_t *off, uint32_t *size, uint64_t *total)
{
    if (!pl || !pl->is_mar) return BNPP_EINVAL;
    for (int v = 0; v < nvars && v < (int)pl->mar_off.size(); ++v) {
        if (off) off[v] = pl->mar_off[v];
        if (size) size[v] = pl->mar_size[v];
    }
    if (total) *total = pl->result_size;
    return BNPP_OK;
}

int bnpp_ve_plan_destroy(bnpp_ve_plan *pl)
{
    if (!pl) return BNPP_OK;
    for (cudaEvent_t e : pl->ev) cudaEventDestroy(e);
    if (pl->batch_exec) {
        cudaGraphExecDestroy(pl->batch_exec);
        cudaDeviceGraphMemTrim(pl->ctx->device);   // hand the graph's allocations back
    }
    if (pl->graph_exec) cudaGraphExecDestroy(pl->graph_exec);
    if (pl->graph) cudaGraphDestroy(pl->graph);
    dev_free(pl->ctx, pl->arena);
    dev_free(pl->ctx, pl->arg_arena);
    dev_free(pl->ctx, pl->decode_rec_dev);
    dev_free(pl->ctx, pl->obs_val_dev);
    dev_free(pl->ctx, pl->batch_rec_dev);
    dev_free(pl->ctx, pl->batch_arg);
    for (auto &d : pl->exec)
        if (d) {
            contract_release(pl->ctx, *d);
            if (pl->ctx && pl->ctx->last_desc == d.get()) pl->ctx->last_desc = nullptr;      // bnpp_last_launch must not follow a pointer into a dead plan
        }
    free_tasks(pl);
    dev_free(pl->ctx, pl->fused.prog_dev);
    dev_free(pl->ctx, pl->fused.offtab_dev);
    dev_free(pl->ctx, pl->mar_off_dev);
    dev_free(pl->ctx, pl->obs_card_dev);
    dev_free(pl->ctx, pl->ev_clean);
    for (uint32_t *&t : pl->offtab_dev) dev_free(pl->ctx, t);
    delete pl;
    return BNPP_OK;
}

int bnpp_ve_plan_info(const bnpp_ve_plan *pl, int32_t *result_rank, uint32_t *result_var, uint32_t *result_card,
                      uint64_t *n_launches, uint64_t *union_entries, uint64_t *algorithmic_bytes,
                      uint64_t *peak_bytes, uint64_t *max_step_entries)
{
    if (!pl) return BNPP_EINVAL;
    if (result_rank) *result_rank = (int32_t)pl->result_var.size();
    for (size_t i = 0; i < pl->result_var.size(); ++i) {
        if (result_var) result_var[i] = pl->result_var[i];
        if (result_card) result_card[i] = pl->result_card[i];
    }
    if (n_launches) *n_launches = pl->windows.empty() ? pl->steps.size() : pl->launch_first.size();     // a window is one launch
    if (union_entries) *union_entries = pl->union_entries;
    if (algorithmic_bytes) *algorithmic_bytes = pl->bytes;
    if (peak_bytes) *peak_bytes = pl->peak_bytes;
    if (max_step_entries) *max_step_entries = pl->max_step_entries;
    return BNPP_OK;
}

int bnpp_ve_plan_result_size(const bnpp_ve_plan *pl, uint64_t *n)
{
    if (!pl || !n) return BNPP_EINVAL;
    *n = pl->result_size;
    return BNPP_OK;
}

int bnpp_ve_plan_set_normalize(bnpp_ve_plan *pl, int on)
{
    if (!pl) return BNPP_EINVAL;
    pl->normalize = on != 0;
    return BNPP_OK;
}

int bnpp_mar_plan_normalize(bnpp_ve_plan *pl, double *result_dev)
{
    if (!pl || !pl->ctx || !pl->is_mar || !result_dev) return BNPP_EINVAL;
    return normalize_segments(pl->ctx, result_dev, pl->mar_off_dev, pl->mar_size_dev, (int)pl->mar_off.size());
}

int bnpp_ve_plan_set_profiling(bnpp_ve_plan *pl, int on)
{
    if (!pl) return BNPP_EINVAL;
    pl->profiling = on != 0;
    if (pl->profiling && pl->ev.size() < pl->steps.size() + 1) {
        const size_t need = pl->steps.size() + 1;
        while (pl->ev.size() < need) {
            cudaEvent_t e;
            BNPP_CUDA(pl->ctx, cudaEventCreate(&e));
            pl->ev.push_back(e);
        }
    }
    return BNPP_OK;
}

int bnpp_ve_plan_set_fused(bnpp_ve_plan *pl, int on)
{
    if (!pl) return BNPP_EINVAL;
    pl->fused_mode = on != 0;
    return BNPP_OK;
}

int bnpp_ve_plan_fused_info(bnpp_ve_plan *pl, uint32_t nb, int32_t *lanes_per_set, uint32_t *arena_doubles, uint32_t *n_steps)
{
    if (!pl || nb == 0) return BNPP_EINVAL;
    const int G = fused_pick(pl, nb);
    if (lanes_per_set) *lanes_per_set = G;
    if (arena_doubles) *arena_doubles = G ? pl->fused.arena : 0;
    if (n_steps) *n_steps = G ? pl->fused.n_steps : 0;
    return BNPP_OK;
}

// The whole schedule as numbers, for inspection and for the CPU emulator of the tests (tests/plan_emulator.py): what
// every launch reads and writes and where the intermediates live in the plan's arena.  Stream of uint64 words:
//   n_factors, n_steps, arena_doubles, result_size,
//   per factor : src + 1 (0 = intermediate), size, arena_off, rank, rank x (var, card, stride), nobs, nobs x (stride, column)
//   per step   : elim + 1 (0 = none), out + 1 (0 = the result buffer), roff, want_z, k, k x operand factor,
//                rank of the output scope, rank x (var, card)
int bnpp_ve_plan_describe(const bnpp_ve_plan *pl, uint64_t *buf, uint64_t cap, uint64_t *words)
{
    if (!pl || !words) return BNPP_EINVAL;
    std::vector<uint64_t> w;
    w.push_back(pl->f.size());
    w.push_back(pl->steps.size());
    w.push_back(pl->arena_doubles);
    w.push_back(pl->result_size);
    for (size_t i = 0; i < pl->f.size(); ++i) {
        const PlanFactor &pf = pl->f[i];
        w.push_back((uint64_t)(pf.src + 1));
        w.push_back(pf.size);
        w.push_back(i < pl->arena_off.size() ? pl->arena_off[i] : 0);
        w.push_back(pf.var.size());
        uint64_t dense = 1;
        std::vector<uint64_t> st(pf.var.size());
        for (size_t a = pf.var.size(); a-- > 0;) {
            st[a] = pf.stride.empty() ? dense : (uint64_t)pf.stride[a];
            dense *= pf.card[a];
        }
        for (size_t a = 0; a < pf.var.size(); ++a) {
            w.push_back(pf.var[a]);
            w.push_back(pf.card[a]);
            w.push_back(st[a]);
        }
        w.push_back(pf.obs.size());
        for (auto &o : pf.obs) {
            w.push_back((uint64_t)o.first);
            w.push_back((uint64_t)o.second);
        }
    }
    for (const PlanStep &st : pl->steps) {
        w.push_back((uint64_t)(st.elim + 1));
        w.push_back(st.out == -2 ? 0 : (uint64_t)(st.out + 1));
        w.push_back(st.roff);
        w.push_back(st.want_z ? 1 : 0);
        w.push_back(st.operands.size());
        for (int id : st.operands) w.push_back((uint64_t)id);
        const std::vector<uint32_t> &ov = st.out == -2 ? st.rvar : pl->f[st.out].var;
        const std::vector<uint32_t> &oc = st.out == -2 ? st.rcard : pl->f[st.out].card;
        w.push_back(ov.size());
        for (size_t a = 0; a < ov.size(); ++a) {
            w.push_back(ov[a]);
            w.push_back(oc[a]);
        }
    }
    *words = w.size();
    if (buf) {
        if (cap < w.size()) return BNPP_EINVAL;
        std::copy(w.begin(), w.end(), buf);
    }
    return BNPP_OK;
}

int bnpp_ve_plan_set_segments(bnpp_ve_plan *pl, int on, uint32_t max_steps)
{
    if (!pl) return BNPP_EINVAL;
    if (pl->is_mpe && on) return fail(pl->ctx, BNPP_EINVAL, "MPE plans run one launch per bucket (ve_tasks only sums)");
    pl->segments_mode = on != 0 ? 1 : 0;
    if (pl->graph_exec && pl->graph_groups != (on != 0)) {      // the replay graph was built the other way
        cudaGraphExecDestroy(pl->graph_exec);
        cudaGraphDestroy(pl->graph);
        pl->graph_exec = nullptr;
        pl->graph = nullptr;
    }
    if (on && (!pl->levels_built || max_steps != pl->segments_max_steps)) {
        pl->segments_max_steps = max_steps;
        build_levels(pl);       // re-orders the steps; refused (the plan keeps its tasks) once the plan has run
        form_windows(pl);
    }
    return BNPP_OK;
}

static int dump_program(const FusedProgram &fp, uint32_t *prog, uint64_t prog_cap, uint64_t *prog_words, uint32_t *offtab,
                        uint64_t tab_cap, uint64_t *tab_words)
{
    if (prog_words) *prog_words = fp.prog.size();
    if (tab_words) *tab_words = fp.offtab.size();
    if (prog) {
        if (prog_cap < fp.prog.size()) return BNPP_EINVAL;
        std::copy(fp.prog.begin(), fp.prog.end(), prog);
        for (auto &slot : fp.ptr_slots) {
            prog[slot.lo] = (uint32_t)slot.index;
            prog[slot.hi] = slot.kind == 0 ? 0xffffffffu : 0xfffffffeu;      // input table | plan-arena intermediate
        }
    }
    if (offtab) {
        if (tab_cap < fp.offtab.size()) return BNPP_EINVAL;
        std::copy(fp.offtab.begin(), fp.offtab.end(), offtab);
    }
    return BNPP_OK;
}

// segments of a launch-per-bucket plan (experimental): [a, b) step ranges, lanes, arena, and each one's program
int bnpp_ve_plan_segments(bnpp_ve_plan *pl, uint32_t cap, uint32_t *n, uint32_t *first_step, uint32_t *end_step,
                          int32_t *lanes, uint32_t *arena_doubles)
{
    if (!pl || !n) return BNPP_EINVAL;
    if (!pl->segments_built) build_segments(pl);
    *n = (uint32_t)pl->segs.size();
    for (uint32_t i = 0; i < *n && i < cap; ++i) {
        if (first_step) first_step[i] = (uint32_t)pl->segs[i].a;
        if (end_step) end_step[i] = (uint32_t)pl->segs[i].b;
        if (lanes) lanes[i] = pl->segs[i].G;
        if (arena_doubles) arena_doubles[i] = pl->segs[i].prog.arena;
    }
    return BNPP_OK;
}

// kernel launches of one single-query run with tasks on: one per group (all small tasks of a dependency level) plus
// one per wide step; and the number of dependency levels
int bnpp_ve_plan_launches(bnpp_ve_plan *pl, uint64_t *launches, uint32_t *groups, uint32_t *levels)
{
    if (!pl) return BNPP_EINVAL;
    if (!pl->segments_built) build_segments(pl);
    uint64_t covered = 0;
    for (const auto &g : pl->groups) covered += (uint64_t)(g.b - g.a);
    for (const auto &w : pl->windows) covered += (uint64_t)(w.b - w.a - 1);
    if (launches) *launches = pl->steps.size() - covered + pl->groups.size();
    if (groups) *groups = (uint32_t)pl->groups.size();
    if (levels) *levels = pl->step_level.empty() ? 0u : (uint32_t)(*std::max_element(pl->step_level.begin(), pl->step_level.end()) + 1);
    return BNPP_OK;
}

int bnpp_ve_plan_windows(const bnpp_ve_plan *pl, uint32_t cap, uint32_t *n, uint32_t *first_step, uint32_t *n_steps)
{
    if (!pl || !n) return BNPP_EINVAL;
    *n = (uint32_t)pl->windows.size();
    for (uint32_t i = 0; i < *n && i < cap; ++i) {
        if (first_step) first_step[i] = (uint32_t)pl->windows[i].a;
        if (n_steps) n_steps[i] = (uint32_t)(pl->windows[i].b - pl->windows[i].a);
    }
    return BNPP_OK;
}

int bnpp_ve_plan_segment_program(bnpp_ve_plan *pl, uint32_t segment, uint32_t *prog, uint64_t prog_cap, uint64_t *prog_words,
                                 uint32_t *offtab, uint64_t tab_cap, uint64_t *tab_words)
{
    if (!pl) return BNPP_EINVAL;
    if (!pl->segments_built) build_segments(pl);
    if (segment >= pl->segs.size()) return BNPP_EINVAL;
    return dump_program(pl->segs[segment].prog, prog, prog_cap, prog_words, offtab, tab_cap, tab_words);
}

// The step program a fused run over nb sets would execute (fused.hpp), for inspection and for the
// CPU interpreter of the tests: CPT operand records carry the INDEX of their input table in word 1
// and 0xffffffff in word 3 instead of a device address.
int bnpp_ve_plan_fused_program(bnpp_ve_plan *pl, uint32_t nb, uint32_t *prog, uint64_t prog_cap, uint64_t *prog_words,
                               uint32_t *offtab, uint64_t tab_cap, uint64_t *tab_words)
{
    if (!pl || nb == 0) return BNPP_EINVAL;
    const bool was_profiling = pl->profiling;
    pl->profiling = false;
    const int G = fused_pick(pl, nb);
    pl->profiling = was_profiling;
    if (prog_words) *prog_words = G ? pl->fused.prog.size() : 0;
    if (tab_words) *tab_words = G ? pl->fused.offtab.size() : 0;
    if (!G) return BNPP_OK;
    return dump_program(pl->fused, prog, prog_cap, prog_words, offtab, tab_cap, tab_words);
}

int bnpp_ve_plan_step_stats(bnpp_ve_plan *pl, uint64_t n, float *ms, uint64_t *bytes, uint64_t *entries, int32_t *k)
{
    if (!pl) return BNPP_EINVAL;
    // one row per launch of a single run: a window is one row (its bytes: head + sides + output; its entries: the
    // union entries of its steps)
    const size_t ns = pl->steps.size();
    const bool win = !pl->windows.empty() && pl->window_at.size() == ns;
    auto launch_end = [&](size_t s) -> size_t { return win && pl->window_at[s] >= 0 ? (size_t)pl->windows[pl->window_at[s]].b : s + 1; };
    if (pl->profiling && !pl->ev.empty()) {
        BNPP_CUDA(pl->ctx, cudaEventSynchronize(pl->ev[ns]));
        pl->step_ms.clear();
        for (size_t s = 0; s < ns; s = launch_end(s)) {
            float t = 0.0f;
            BNPP_CUDA(pl->ctx, cudaEventElapsedTime(&t, pl->ev[s], pl->ev[launch_end(s)]));
            pl->step_ms.push_back(t);
        }
    }
    size_t row = 0;
    for (size_t s = 0; s < ns && row < n; s = launch_end(s), ++row) {
        const bool w = win && pl->window_at[s] >= 0;
        if (ms) ms[row] = row < pl->step_ms.size() ? pl->step_ms[row] : 0.0f;
        if (bytes) bytes[row] = w ? pl->windows[pl->window_at[s]].bytes : pl->steps[s].bytes;
        if (entries) entries[row] = w ? pl->windows[pl->window_at[s]].entries : pl->steps[s].union_entries;
        if (k) k[row] = (int32_t)pl->steps[s].operands.size();
    }
    return BNPP_OK;
}

int bnpp_ve_plan_step_kernel(const bnpp_ve_plan *pl, uint64_t step, char *name, size_t name_len)
{
    if (!pl || !name || !name_len) return BNPP_EINVAL;
    if (!pl->windows.empty()) step = step < pl->launch_first.size() ? (uint64_t)pl->launch_first[step] : UINT64_MAX;   // row = launch
    const std::string s = step < pl->step_kernel.size() ? pl->step_kernel[step] : std::string();
    strncpy(name, s.c_str(), name_len - 1);
    name[name_len - 1] = 0;
    return BNPP_OK;
}

// MPE / MAP plans: max steps are max-product steps writing their argmax tables into the plan's byte arena
static int run_dynamic(bnpp_ve_plan *pl, const std::vector<const double *> &ptr_in, double *result_dev, double *z_dev)
{
    bnpp_ctx *ctx = pl->ctx;
    std::vector<const double *> ptr = ptr_in;
    std::vector<double *> owned(pl->f.size(), nullptr);
    int rc = BNPP_OK;
    for (size_t s = 0; s < pl->steps.size() && rc == BNPP_OK; ++s) {
        const PlanStep &st = pl->steps[s];
        if (pl->profiling) cudaEventRecord(pl->ev[s], ctx->stream);
        bnpp_operand ops[kMaxK];
        for (size_t q = 0; q < st.operands.size(); ++q) {
            const PlanFactor &pf = pl->f[st.operands[q]];
            ops[q].data = ptr[st.operands[q]];
            ops[q].scope.rank = (int32_t)pf.var.size();
            ops[q].scope.var_id = pf.var.data();
            ops[q].scope.card = pf.card.data();
            ops[q].stride = pf.stride.empty() ? nullptr : pf.stride.data();
        }
        bnpp_scope os;
        double *dst;
        if (st.out == -2) {
            os.rank = (int32_t)st.rvar.size();
            os.var_id = st.rvar.data();
            os.card = st.rcard.data();
            dst = result_dev + st.roff;
        } else {
            const PlanFactor &of = pl->f[st.out];
            os.rank = (int32_t)of.var.size();
            os.var_id = of.var.data();
            os.card = of.card.data();
            rc = dev_alloc(ctx, of.size, &owned[st.out]);
            if (rc != BNPP_OK) break;
            dst = owned[st.out];
            ptr[st.out] = dst;
        }
        const bool max_mode = st.max;
        rc = contract(ctx, (int)st.operands.size(), ops, &os, st.elim, 0, dst, (st.out == -2 && st.want_z) ? z_dev : nullptr,
                      max_mode, max_mode ? pl->arg_arena + pl->arg_off[s] : nullptr);
        if (pl->profiling) {
            pl->step_kernel.resize(pl->steps.size());
            pl->step_kernel[s] = ctx->last_kernel;   // set by contract() below
        }
        for (int id : st.operands)
            if (pl->f[id].last_use == (int)s) dev_free(ctx, owned[id]);
    }
    for (double *&p : owned) dev_free(ctx, p);
    return rc;
}

// the parameters of an MPE run's decode (a launch, or the last node of the replay graph, set again on every replay:
// the evidence values travel in them); the decode records go to the device on the first run
static int mpe_decode_prepare(bnpp_ve_plan *pl, const uint32_t *obs_val, double *value_dev, uint32_t *assign_dev)
{
    bnpp_ctx *ctx = pl->ctx;
    if (!pl->decode_rec_dev && !pl->decode_rec.empty()) {
        const int rc = dev_alloc(ctx, pl->decode_rec.size(), &pl->decode_rec_dev);
        if (rc != BNPP_OK) return rc;
        BNPP_CUDA(ctx, cudaMemcpyAsync(pl->decode_rec_dev, pl->decode_rec.data(), 4 * pl->decode_rec.size(),
                                       cudaMemcpyHostToDevice, ctx->stream));
    }
    MpeDecodeParams &p = pl->decode;
    p.rec = pl->decode_rec_dev;
    p.arg = pl->arg_arena;
    p.assign = assign_dev;
    p.value = value_dev;
    p.nvars = pl->mpe_nvars;
    p.n_obs = (uint32_t)pl->n_obs;
    p.n_rec = pl->n_decode_rec;
    p.n_sum = pl->n_summed;
    p.set_one = (pl->steps.empty() || pl->steps.back().out != -2) ? 1u : 0u;
    if (p.n_obs <= kDecodeInlineObs) {
        for (uint32_t i = 0; i < p.n_obs; ++i) p.obs_val[i] = obs_val[i];
    } else {
        if (!pl->obs_val_dev) {
            const int rc = dev_alloc(ctx, p.n_obs, &pl->obs_val_dev);
            if (rc != BNPP_OK) return rc;
        }
        BNPP_CUDA(ctx, cudaMemcpyAsync(pl->obs_val_dev, obs_val, 4ull * p.n_obs, cudaMemcpyHostToDevice, ctx->stream));
        p.obs_val_dev = pl->obs_val_dev;
    }
    return BNPP_OK;
}

constexpr unsigned kDecodeThreads = 32;

// the decode as a launch of its own; bnpp_last_launch keeps reporting the plan's last step
static int decode_launch(bnpp_ve_plan *pl)
{
    bnpp_ctx *ctx = pl->ctx;
    mpe_decode<<<1, kDecodeThreads, 0, ctx->stream>>>(pl->decode);
    BNPP_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return BNPP_OK;
}

// one kernel run of the replay graph: a new node after `prev` while the graph is being built (it becomes `prev`), else
// the instantiated node's parameters set again
static cudaError_t graph_node(bnpp_ve_plan *pl, cudaGraphNode_t &node, cudaGraphNode_t &prev, const void *fn, unsigned grid,
                              unsigned block, unsigned smem, void *params)
{
    void *args[1] = {params};
    cudaKernelNodeParams kp;
    memset(&kp, 0, sizeof kp);
    kp.func = const_cast<void *>(fn);
    kp.gridDim = dim3(grid);
    kp.blockDim = dim3(block);
    kp.sharedMemBytes = smem;
    kp.kernelParams = args;
    if (pl->graph_exec) return cudaGraphExecKernelNodeSetParams(pl->graph_exec, node, &kp);
    const cudaError_t e = cudaGraphAddKernelNode(&node, pl->graph, prev ? &prev : nullptr, prev ? 1 : 0, &kp);
    prev = node;
    return e;
}

static int run_plan(bnpp_ve_plan *pl, const double *const *tables_dev, const uint32_t *obs_val, double *result_dev,
                    double *z_dev, uint32_t *assign_dev);

int bnpp_ve_plan_run(bnpp_ve_plan *pl, const double *const *tables_dev, const uint32_t *obs_val, double *result_dev,
                     double *z_dev)
{
    if (pl && pl->is_mpe) return fail(pl->ctx, BNPP_EINVAL, "MPE plan: run it with bnpp_mpe_plan_run");
    return run_plan(pl, tables_dev, obs_val, result_dev, z_dev, nullptr);
}

int bnpp_mpe_plan_run(bnpp_ve_plan *pl, const double *const *tables_dev, const uint32_t *obs_val, double *value_dev,
                      uint32_t *assignment_dev)
{
    if (!pl) return BNPP_EINVAL;
    if (!pl->is_mpe || !assignment_dev) return fail(pl->ctx, BNPP_EINVAL, "bnpp_mpe_plan_run: not an MPE plan, or no assignment buffer");
    return run_plan(pl, tables_dev, obs_val, value_dev, nullptr, assignment_dev);
}

int bnpp_mpe_plan_nvars(const bnpp_ve_plan *pl, uint32_t *nvars)
{
    if (!pl || !pl->is_mpe || !nvars) return BNPP_EINVAL;
    *nvars = pl->mpe_nvars;
    return BNPP_OK;
}

int bnpp_mpe_shard_select(bnpp_ctx *ctx, uint32_t nranks, uint32_t nvars, const uint32_t *records_dev, double *value_dev,
                          uint32_t *assignment_dev)
{
    if (!ctx) return BNPP_EINVAL;
    if (nranks == 0 || nvars == 0 || !records_dev || !value_dev || !assignment_dev)
        return fail(ctx, BNPP_EINVAL, "bnpp_mpe_shard_select: no ranks, no variables or a NULL buffer");
    const uint64_t stride = (2ull + nvars + 1) & ~1ull;
    mpe_shard_select<<<1, kSelectThreads, 0, ctx->stream>>>(records_dev, nranks, nvars, stride, value_dev, assignment_dev);
    BNPP_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    ctx->last_desc = nullptr;
    ctx->last_kernel = "mpe_shard_select";
    ctx->last_grid = 1;
    ctx->last_block = kSelectThreads;
    return BNPP_OK;
}

// assign_dev != NULL: an MPE run (result_dev is the value)
static int run_plan(bnpp_ve_plan *pl, const double *const *tables_dev, const uint32_t *obs_val, double *result_dev,
                    double *z_dev, uint32_t *assign_dev)
{
    if (!pl || !pl->ctx || !result_dev) return BNPP_EINVAL;
    bnpp_ctx *ctx = pl->ctx;
    const auto t_run0 = std::chrono::steady_clock::now();
    if (pl->n_obs && !obs_val) return fail(ctx, BNPP_EINVAL, "VE plan: evidence values missing");
    for (int i = 0; i < pl->n_obs; ++i)
        if (pl->obs_card[i] && obs_val[i] >= pl->obs_card[i])
            return fail(ctx, BNPP_EINVAL, "VE plan: evidence value out of range (Factor::operator[], code/factor.cpp:83-95)");
    std::vector<const double *> ptr(pl->f.size(), nullptr);
    bool aligned32 = true;
    for (size_t i = 0; i < pl->f.size(); ++i) {
        const PlanFactor &pf = pl->f[i];
        if (pf.src < 0) continue;
        uint64_t base = 0;
        for (auto &o : pf.obs) base += (uint64_t)o.first * obs_val[o.second];
        ptr[i] = tables_dev[pf.src] + base;
        aligned32 = aligned32 && (reinterpret_cast<uintptr_t>(tables_dev[pf.src]) % 32 == 0);
    }
    if (!pl->is_mar && !pl->is_mpe && (pl->steps.empty() || pl->steps.back().out != -2)) {
        int rc = fill(ctx, result_dev, 1, 1.0);   // no factor left: the scalar 1 (code/model.cpp:355)
        if (rc != BNPP_OK) return rc;
        if (z_dev) rc = fill(ctx, z_dev, 1, 1.0);
        if (rc != BNPP_OK) return rc;
    }
    int rc = BNPP_OK;
    int fused_g = 0;
    bool ev_inline = pl->n_obs <= kFusedInlineEv;      // the evidence values travel in the kernel parameters as bytes
    for (int i = 0; i < pl->n_obs && ev_inline; ++i) ev_inline = obs_val[i] <= 255;
    if (ev_inline && !pl->is_mpe) fused_g = fused_pick(pl, 1);
    if (pl->is_mpe) {
        if (!pl->arg_arena && pl->arg_bytes) {
            rc = dev_alloc(ctx, pl->arg_bytes, &pl->arg_arena);
            if (rc != BNPP_OK) return rc;
        }
        rc = mpe_decode_prepare(pl, obs_val, result_dev, assign_dev);
        if (rc != BNPP_OK) return rc;
    }
    if (getenv("BNPP_TIMING") && pl->runs == 0)
        fprintf(stderr, "bnpp timing: up to the choice of the path %.3f ms\n",
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_run0).count());
    if (fused_g) {
        // K9: every step is small -- the whole plan is one launch, intermediates in shared memory
        rc = run_fused(pl, fused_g, tables_dev, 1, nullptr, obs_val, result_dev, z_dev);
    } else if (!pl->exec_ok || !aligned32) {
        rc = run_dynamic(pl, ptr, result_dev, z_dev);
        if (rc == BNPP_OK && pl->is_mpe) rc = decode_launch(pl);
    } else {
        if (!pl->arena && pl->arena_doubles) {
            const auto t_a0 = std::chrono::steady_clock::now();
            rc = dev_alloc(ctx, pl->arena_doubles, &pl->arena);
            if (rc != BNPP_OK) return rc;
            if (getenv("BNPP_TIMING"))
                fprintf(stderr, "bnpp timing: arena of %.1f MB allocated in %.3f ms\n", pl->arena_doubles * 8e-6,
                        std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_a0).count());
        }
        if (pl->exec.size() != pl->steps.size()) {
            pl->exec.clear();
            pl->exec.resize(pl->steps.size());
            pl->exec_planned.assign(pl->steps.size(), 0);
        }
        for (size_t i = 0; i < pl->f.size(); ++i)
            if (pl->f[i].src < 0) ptr[i] = pl->arena + pl->arena_off[i];
        // K10: the small tasks of every dependency level as ONE ve_tasks launch (a node of the replay graph like any other)
        const bool seg_on = pl->segments_mode && pl->levels_built && ev_inline && !pl->profiling && !pl->is_mpe;
        static const bool timing = getenv("BNPP_TIMING") != nullptr;
        const auto t_0 = std::chrono::steady_clock::now();
        if (seg_on && !pl->segments_built) build_segments(pl);
        const auto t_1 = std::chrono::steady_clock::now();
        const bool use_groups = seg_on && !pl->groups.empty();
        if (use_groups) {
            rc = upload_tasks(pl, tables_dev);
            if (rc != BNPP_OK) return rc;
        }
        const auto t_2 = std::chrono::steady_clock::now();
        if (timing && pl->runs == 0)
            fprintf(stderr, "bnpp timing: build_segments %.3f ms, upload_tasks %.3f ms (%zu tasks, %zu groups, prog %zu words, tables %zu words)\n",
                    std::chrono::duration<double, std::milli>(t_1 - t_0).count(), std::chrono::duration<double, std::milli>(t_2 - t_1).count(),
                    pl->segs.size(), pl->groups.size(), pl->tasks_prog.size(), pl->tasks_tab_words);
        const bool graphed = pl->use_graph && !pl->profiling && pl->steps.size() > 1 && pl->runs >= 1 &&
                             (!pl->graph_exec || pl->graph_groups == use_groups);
        bool fresh = false;
        if (graphed && !pl->graph_exec) {
            if (cudaGraphCreate(&pl->graph, 0) != cudaSuccess) pl->use_graph = false;
            pl->nodes.assign(pl->steps.size(), nullptr);
            pl->graph_groups = use_groups;
            fresh = true;
        }
        cudaGraphNode_t prev = nullptr;
        uint64_t n_launched = 0;
        double t_plan_steps = 0.0;
        for (size_t s = 0; s < pl->steps.size() && rc == BNPP_OK; ++s) {
            if (use_groups && pl->group_at[s] >= 0) {
                bnpp_ve_plan::Group &g = pl->groups[pl->group_at[s]];
                TaskLaunch now = g.launch;
                now.result = result_dev;
                now.z = z_dev;
                memset(now.ev_inline, 0, sizeof now.ev_inline);
                for (int i = 0; i < pl->n_obs && i < kFusedInlineEv; ++i) now.ev_inline[i] = (uint8_t)obs_val[i];
                const bool changed = fresh || memcmp(&now, &g.launch, sizeof now) != 0;
                g.launch = now;
                ++n_launched;
                if (!(graphed && pl->use_graph)) {
                    rc = tasks_launch(ctx, g.launch, g.grid, g.smem);
                } else if (changed) {
                    const cudaError_t e = graph_node(pl, pl->nodes[s], prev, tasks_kernel(), g.grid, kFusedThreads, g.smem, &g.launch);
                    if (e != cudaSuccess) return cuda_fail(ctx, e, "CUDA graph node (tasks)");
                }
                s = (size_t)g.b - 1;
                continue;
            }
            if (!pl->windows.empty() && pl->window_at[s] >= 0) {
                // K11: a window of binary eliminations, one contract_chain launch
                bnpp_ve_plan::Window &w = pl->windows[pl->window_at[s]];
                if (pl->profiling) cudaEventRecord(pl->ev[s], ctx->stream);
                if (!w.grid) {
                    const int occ = chain_occupancy(w.fn);
                    if (occ <= 0) return fail(ctx, BNPP_ECUDA, "contract_chain: no occupancy");
                    const uint64_t chunks = w.p.n_items / (uint64_t)chain_chunk_items(w.m);
                    w.grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>(chunks, (uint64_t)occ * ctx->sm_count));
                }
                ChainParams now = w.p;
                now.head = ptr[w.head];
                now.out = pl->arena + pl->arena_off[w.out];
                for (int j = 0; j < w.m; ++j)
                    for (int q = 0; q < now.lv[j].k; ++q) now.lv[j].s[q].p = ptr[w.side[j][q]];
                bool moved = fresh || now.head != w.p.head || now.out != w.p.out;
                for (int j = 0; j < w.m; ++j)
                    for (int q = 0; q < now.lv[j].k; ++q) moved = moved || now.lv[j].s[q].p != w.p.lv[j].s[q].p;
                w.p = now;
                ++n_launched;
                if (!(graphed && pl->use_graph)) {
                    rc = chain_launch(ctx, w.fn, w.grid, w.p, w.name);
                } else if (moved) {
                    const cudaError_t e = graph_node(pl, pl->nodes[s], prev, w.fn, w.grid, kBlock, 0, &w.p);
                    if (e != cudaSuccess) return cuda_fail(ctx, e, "CUDA graph node (contract_chain)");
                }
                s = (size_t)w.b - 1;
                continue;
            }
            const PlanStep &st = pl->steps[s];
            if (pl->profiling) cudaEventRecord(pl->ev[s], ctx->stream);
            const double *in[kMaxK];
            for (size_t q = 0; q < st.operands.size(); ++q) in[q] = ptr[st.operands[q]];
            double *dst = st.out == -2 ? result_dev + st.roff : pl->arena + pl->arena_off[st.out];
            double *z = (st.out == -2 && st.want_z) ? z_dev : nullptr;
            if (!pl->exec_planned[s]) {
                const auto t_p0 = std::chrono::steady_clock::now();
                if (!plan_step(pl, s)) return fail(ctx, BNPP_EINVAL, "VE plan: a step could not be resolved");
                t_plan_steps += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_p0).count();
            }
            ++n_launched;
            if (!(graphed && pl->use_graph)) {
                rc = contract_launch(ctx, *pl->exec[s], in, dst, z);
                continue;
            }
            LaunchDesc &d = *pl->exec[s];
            ParamsHead &h = d.head();
            bool moved = fresh || h.out != dst || h.z != z;
            for (size_t q = 0; q < st.operands.size(); ++q) moved = moved || h.in[q] != in[q];
            if (!moved) continue;
            for (size_t q = 0; q < st.operands.size(); ++q) h.in[q] = in[q];
            h.out = dst;
            h.z = z;
            const cudaError_t e = graph_node(pl, pl->nodes[s], prev, d.fn, d.grid, kBlock, d.smem, d.params());
            if (e != cudaSuccess) return cuda_fail(ctx, e, "CUDA graph node");
        }
        if (pl->is_mpe && rc == BNPP_OK) {
            ++n_launched;
            if (!(graphed && pl->use_graph)) {
                rc = decode_launch(pl);
            } else {
                const cudaError_t e = graph_node(pl, pl->decode_node, prev, reinterpret_cast<const void *>(mpe_decode), 1,
                                                 kDecodeThreads, 0, &pl->decode);
                if (e != cudaSuccess) return cuda_fail(ctx, e, "CUDA graph node (MPE decode)");
            }
        }
        if (timing && pl->runs == 0)
            fprintf(stderr, "bnpp timing: resolving the wide steps' launches (contract_plan) %.3f ms, %llu launches, launch loop %.3f ms\n",
                    t_plan_steps, (unsigned long long)n_launched,
                    std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_2).count());
        if (graphed && pl->use_graph && rc == BNPP_OK) {
            if (fresh) BNPP_CUDA(ctx, cudaGraphInstantiate(&pl->graph_exec, pl->graph, 0));
            BNPP_CUDA(ctx, cudaGraphLaunch(pl->graph_exec, ctx->stream));
            ctx->launches += n_launched;
            ctx->last_desc = nullptr;
            ctx->last_kernel = "cudaGraphLaunch (VE plan replay)";
        }
        if (pl->profiling) {
            pl->step_kernel.resize(pl->steps.size());
            for (size_t s = 0; s < pl->steps.size(); ++s) pl->step_kernel[s] = pl->exec[s] ? pl->exec[s]->name() : std::string();
            for (const auto &w : pl->windows) pl->step_kernel[w.a] = w.name;
        }
    }
    if (rc == BNPP_OK && pl->is_mar && pl->normalize)
        rc = normalize_segments(ctx, result_dev, pl->mar_off_dev, pl->mar_size_dev, (int)pl->mar_off.size());
    if (pl->profiling) cudaEventRecord(pl->ev[pl->steps.size()], ctx->stream);
    if (getenv("BNPP_TIMING") && pl->runs == 0)
        fprintf(stderr, "bnpp timing: first run of the plan enqueued in %.3f ms (host)\n",
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_run0).count());
    pl->runs++;
    return rc;
}

// BN::partition for a whole batch of evidence sets over ONE plan (config 5): the observed
// ids are the plan's, ev_dev[b][j] is the value of obs_var[j] in set b.  result_dev receives
// [result_size][nb] (batch fastest).  Sets are processed in slices that keep the widest
// intermediate below ~1 GiB.
// assign_dev != nullptr: an MPE run (result_dev receives the values, assign_dev [nvars][nb] the assignments)
static int run_batched_once(bnpp_ve_plan *pl, const double *const *tables_dev, uint32_t nb, uint32_t n_obs,
                            const uint8_t *ev_dev, double *result_dev, uint8_t *assign_dev);
static int run_batched(bnpp_ve_plan *pl, const double *const *tables_dev, uint32_t nb, uint32_t n_obs, const uint8_t *ev_dev,
                       double *result_dev, uint8_t *assign_dev);

int bnpp_ve_plan_run_batched(bnpp_ve_plan *pl, const double *const *tables_dev, uint32_t nb, uint32_t n_obs,
                             const uint8_t *ev_dev, double *result_dev)
{
    if (!pl || !pl->ctx || !result_dev || nb == 0) return BNPP_EINVAL;
    if (pl->is_mpe) return fail(pl->ctx, BNPP_EINVAL, "MPE plan: run a batch with bnpp_mpe_plan_run_batched");
    return run_batched(pl, tables_dev, nb, n_obs, ev_dev, result_dev, nullptr);
}

int bnpp_mpe_plan_run_batched(bnpp_ve_plan *pl, const double *const *tables_dev, uint32_t nb, uint32_t n_obs,
                              const uint8_t *ev_dev, double *value_dev, uint8_t *assignment_dev)
{
    if (!pl || !pl->ctx || !value_dev || !assignment_dev || nb == 0) return BNPP_EINVAL;
    if (!pl->is_mpe) return fail(pl->ctx, BNPP_EINVAL, "bnpp_mpe_plan_run_batched: not an MPE plan");
    return run_batched(pl, tables_dev, nb, n_obs, ev_dev, value_dev, assignment_dev);
}

// Sets per slice of a batched run: K8 keeps its widest intermediate within ~1 GiB (k8 = true), and an MPE run its
// argmax rows (arg_rows bytes per set) within 1 GiB on either engine.
static uint32_t batch_slice(const bnpp_ve_plan *pl, uint32_t nb, bool k8)
{
    uint64_t slice = nb;
    if (k8) {
        uint64_t widest = 1;
        for (const PlanFactor &pf : pl->f)
            if (pf.src < 0) widest = std::max(widest, pf.size);
        widest = std::max(widest, pl->result_size);
        slice = std::min<uint64_t>(nb, std::max<uint64_t>(1, (1ull << 27) / widest));
        if (pl->result_size > 1) slice = nb;     // a multi-entry result is laid out [entries][nb]: no slicing
    }
    if (pl->is_mpe && pl->arg_rows) slice = std::min<uint64_t>(slice, std::max<uint64_t>(1, (1ull << 30) / pl->arg_rows));
    return (uint32_t)slice;
}

// the argmax rows of an MPE batch of `slice` sets, and the decode records on the device (before any capture)
static int mpe_batch_prepare(bnpp_ve_plan *pl, uint32_t slice)
{
    bnpp_ctx *ctx = pl->ctx;
    if (!pl->batch_rec_dev && !pl->batch_rec.empty()) {
        const int rc = dev_alloc(ctx, pl->batch_rec.size(), &pl->batch_rec_dev);
        if (rc != BNPP_OK) return rc;
        BNPP_CUDA(ctx, cudaMemcpyAsync(pl->batch_rec_dev, pl->batch_rec.data(), 4 * pl->batch_rec.size(), cudaMemcpyHostToDevice,
                                       ctx->stream));
    }
    const uint64_t need = pl->arg_rows * slice;
    if (need > pl->batch_arg_bytes) {
        dev_free(ctx, pl->batch_arg);
        pl->batch_arg_bytes = 0;
        const int rc = dev_alloc(ctx, need, &pl->batch_arg);
        if (rc != BNPP_OK) return rc;
        pl->batch_arg_bytes = need;
    }
    return BNPP_OK;
}

// the decode of the sets [b0, b0 + cur) of an MPE batch; ev: evidence value j of set b0 + t at ev[j * ev_col + t * ev_row]
static int mpe_decode_batch_launch(bnpp_ve_plan *pl, uint32_t nb, uint32_t b0, uint32_t cur, const uint8_t *ev, uint64_t ev_col,
                                   uint64_t ev_row, uint8_t *assign_dev)
{
    bnpp_ctx *ctx = pl->ctx;
    MpeBatchDecodeParams p;
    memset(&p, 0, sizeof p);
    p.rec = pl->batch_rec_dev;
    p.arg = pl->batch_arg;
    p.ev = ev;
    p.ev_col = ev_col;
    p.ev_row = ev_row;
    p.assign = assign_dev + b0;
    p.nb = nb;
    p.cur = cur;
    p.nvars = pl->mpe_nvars;
    p.n_obs = (uint32_t)pl->n_obs;
    p.n_rec = pl->n_decode_rec;
    p.n_sum = pl->n_summed;
    mpe_decode_batched<<<(cur + 127) / 128, 128, 0, ctx->stream>>>(p);
    BNPP_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return BNPP_OK;
}

// The launches of a batched run are tiny when the batch is sharded over many GPUs, so from the
// third run with the same buffers on, the whole run (stream-ordered allocations included) is
// replayed as one captured CUDA graph.
static int run_batched(bnpp_ve_plan *pl, const double *const *tables_dev, uint32_t nb, uint32_t n_obs, const uint8_t *ev_dev,
                       double *result_dev, uint8_t *assign_dev)
{
    bnpp_ctx *ctx = pl->ctx;
    if ((int)n_obs != pl->n_obs) return fail(ctx, BNPP_EINVAL, "batched VE: n_obs differs from the plan's");
    if (n_obs && !ev_dev) return fail(ctx, BNPP_EINVAL, "batched VE: evidence matrix missing");
    if (n_obs && !pl->obs_card_dev) {
        const int rc = dev_alloc(ctx, n_obs + 4, &pl->obs_card_dev);
        if (rc != BNPP_OK) return rc;
        std::vector<uint32_t> c(pl->obs_card);
        for (uint32_t &v : c)
            if (!v) v = 256;        // a variable no factor mentions: any byte is harmless
        BNPP_CUDA(ctx, cudaMemcpyAsync(pl->obs_card_dev, c.data(), sizeof(uint32_t) * n_obs, cudaMemcpyHostToDevice, ctx->stream));
        BNPP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));       // `c` dies here
    }
    if (nb > 1) {
        // K9: one launch for the whole batch, the intermediates of a set never leave shared memory
        const int G = fused_pick(pl, nb);
        if (G) {
            const uint8_t *ev = ev_dev;
            if (n_obs) {
                const uint64_t need = (uint64_t)nb * n_obs;
                if (pl->ev_clean_bytes < need) {
                    dev_free(ctx, pl->ev_clean);
                    const int rc = dev_alloc(ctx, need + 16, &pl->ev_clean);
                    if (rc != BNPP_OK) return rc;
                    pl->ev_clean_bytes = need;
                }
                const int rc = sanitize_evidence_launch(ctx, ev_dev, pl->ev_clean, nb, n_obs, pl->obs_card_dev, false);
                if (rc != BNPP_OK) return rc;
                ev = pl->ev_clean;
            }
            if (!assign_dev) {
                int rc = run_fused(pl, G, tables_dev, nb, ev, nullptr, result_dev, nullptr);
                if (rc == BNPP_OK && pl->is_mar && pl->normalize)
                    rc = normalize_segments_batched(ctx, result_dev, pl->mar_off_dev, pl->mar_size_dev, (int)pl->mar_off.size(), nb);
                return rc;
            }
            // MPE: slices whose argmax rows fit the scratch, each one ve_fused_max launch and its decode
            const uint32_t slice = batch_slice(pl, nb, false);
            int rc = mpe_batch_prepare(pl, slice);
            for (uint32_t b0 = 0; b0 < nb && rc == BNPP_OK; b0 += slice) {
                const uint32_t cur = std::min(slice, nb - b0);
                const uint8_t *ev_b = n_obs ? ev + (uint64_t)b0 * n_obs : ev;
                rc = run_fused(pl, G, tables_dev, cur, ev_b, nullptr, result_dev + b0, nullptr, pl->batch_arg);
                if (rc == BNPP_OK) rc = mpe_decode_batch_launch(pl, nb, b0, cur, ev_b, 1, n_obs, assign_dev);
            }
            return rc;
        }
    }
    if (assign_dev) {
        const int rc = mpe_batch_prepare(pl, batch_slice(pl, nb, true));
        if (rc != BNPP_OK) return rc;
    }
    std::vector<const void *> key;
    key.push_back(ev_dev);
    key.push_back(result_dev);
    key.push_back(reinterpret_cast<const void *>(static_cast<uintptr_t>(nb)));
    for (int q = 0; q < pl->n_inputs; ++q) key.push_back(tables_dev[q]);
    if (assign_dev) {
        key.push_back(assign_dev);
        key.push_back(pl->batch_arg);       // a captured run writes the argmax rows there
    }
    const bool mar_norm = pl->is_mar && pl->normalize;     // the captured run ends with the batched normaliser
    key.push_back(reinterpret_cast<const void *>(static_cast<uintptr_t>(mar_norm)));
    const uint64_t replay_launches = pl->steps.size() + 1 + (mar_norm ? 1 : 0);
    if (pl->batch_exec && key == pl->batch_key) {
        BNPP_CUDA(ctx, cudaGraphLaunch(pl->batch_exec, ctx->stream));
        ctx->launches += replay_launches;
        return BNPP_OK;
    }
    if (pl->batch_exec) {
        cudaGraphExecDestroy(pl->batch_exec);
        pl->batch_exec = nullptr;
        pl->batch_runs = 0;
    }
    // run 0 is plain (it uploads the offset tables from pageable memory, which a capture must not
    // contain); run 1 with the same buffers is captured and launched
    if (pl->use_graph && pl->batch_runs >= 1 && key == pl->batch_key) {
        cudaGraph_t g = nullptr;
        if (cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
            const uint64_t before = ctx->launches;
            const int rc = run_batched_once(pl, tables_dev, nb, n_obs, ev_dev, result_dev, assign_dev);
            const cudaError_t e = cudaStreamEndCapture(ctx->stream, &g);
            ctx->launches = before;
            if (rc == BNPP_OK && e == cudaSuccess && cudaGraphInstantiate(&pl->batch_exec, g, 0) == cudaSuccess) {
                cudaGraphDestroy(g);
                BNPP_CUDA(ctx, cudaGraphLaunch(pl->batch_exec, ctx->stream));
                ctx->launches += replay_launches;
                return BNPP_OK;
            }
            if (g) cudaGraphDestroy(g);
            cudaGetLastError();
            pl->batch_exec = nullptr;
            pl->use_graph = false;      // capture not possible here: stay on plain launches
        }
    }
    pl->batch_key = key;
    pl->batch_runs++;
    return run_batched_once(pl, tables_dev, nb, n_obs, ev_dev, result_dev, assign_dev);
}

static int run_batched_once(bnpp_ve_plan *pl, const double *const *tables_dev, uint32_t nb, uint32_t n_obs,
                            const uint8_t *ev_dev, double *result_dev, uint8_t *assign_dev)
{
    bnpp_ctx *ctx = pl->ctx;
    uint64_t widest = 1;
    for (const PlanFactor &pf : pl->f)
        if (pf.src < 0) widest = std::max(widest, pf.size);
    widest = std::max(widest, pl->result_size);
    const uint32_t slice = batch_slice(pl, nb, true);
    if ((uint64_t)widest * slice >= (1ull << 32)) return fail(ctx, BNPP_ETOOBIG, "batched VE: intermediate too large");
    static const std::vector<int64_t> dense;
    static const std::vector<std::pair<int64_t, int>> no_obs;
    int rc = BNPP_OK;
    // a CPT with more observed axes than a K8 operand holds is read through the base-256 digits of its evidence base,
    // extra evidence columns after the plan's own: (stride, column) per digit instead of its observed axes
    std::vector<std::vector<std::pair<int64_t, int>>> digit_obs(pl->f.size());
    uint32_t n_cols = n_obs;
    for (size_t i = 0; i < pl->f.size(); ++i) {
        const PlanFactor &pf = pl->f[i];
        if (pf.src < 0 || pf.obs.size() <= (size_t)kMaxObsPerOperand) continue;
        uint64_t max_base = 0;
        for (auto &o : pf.obs) max_base += (uint64_t)o.first * (pl->obs_card[o.second] - 1);
        if (max_base >> 32) return fail(ctx, BNPP_ETOOBIG, "batched VE: evidence base of a table beyond 32 bits");
        for (uint32_t d = 0; d == 0 || (d < 4 && (max_base >> (8 * d))); ++d) digit_obs[i].push_back({1ll << (8 * d), (int)n_cols++});
    }
    // evidence columns contiguous over the sets: every thread of a warp then reads neighbouring bytes
    uint8_t *evt = nullptr;
    rc = dev_alloc(ctx, (uint64_t)nb * (n_cols ? n_cols : 1) + 8, &evt);
    if (rc != BNPP_OK) return rc;
    if (pl->offtab_host.size() != pl->steps.size()) {
        pl->offtab_host.assign(pl->steps.size(), std::vector<uint32_t>());
        pl->offtab_dev.assign(pl->steps.size(), nullptr);
    }
    rc = sanitize_evidence_launch(ctx, ev_dev, evt, nb, n_obs, pl->obs_card_dev, true);
    for (size_t i = 0; i < pl->f.size() && rc == BNPP_OK; ++i)
        if (!digit_obs[i].empty())
            rc = evidence_digits_launch(ctx, pl->f[i].obs, evt, nb, (uint32_t)digit_obs[i][0].second, (uint32_t)digit_obs[i].size());
    for (uint32_t b0 = 0; b0 < nb && rc == BNPP_OK; b0 += slice) {
        const uint32_t cur = std::min(slice, nb - b0);
        std::vector<double *> owned(pl->f.size(), nullptr);
        for (size_t s = 0; s < pl->steps.size() && rc == BNPP_OK; ++s) {
            const PlanStep &st = pl->steps[s];
            BatchedOperandDesc ops[kMaxK];
            for (size_t q = 0; q < st.operands.size(); ++q) {
                const PlanFactor &pf = pl->f[st.operands[q]];
                ops[q].batched = pf.src < 0;
                ops[q].ptr = pf.src < 0 ? owned[st.operands[q]] : tables_dev[pf.src];
                ops[q].var = &pf.var;
                ops[q].card = &pf.card;
                ops[q].stride = pf.src < 0 ? &dense : &pf.stride;
                ops[q].obs = pf.src < 0 ? &no_obs : digit_obs[st.operands[q]].empty() ? &pf.obs : &digit_obs[st.operands[q]];
            }
            double *dst;
            const std::vector<uint32_t> *ov, *oc;
            if (st.out == -2) {
                ov = &st.rvar;
                oc = &st.rcard;
                // result entry i of set b at result_dev[i * nb + b]: a multi-entry result (a marginals plan) is never
                // sliced (batch_slice), so there b0 == 0 and cur == nb; a sliced plan's result is one entry, roff 0
                dst = result_dev + (uint64_t)st.roff * nb + b0;
            } else {
                const PlanFactor &of = pl->f[st.out];
                ov = &of.var;
                oc = &of.card;
                rc = dev_alloc(ctx, of.size * cur, &owned[st.out]);
                if (rc != BNPP_OK) break;
                dst = owned[st.out];
            }
            uint8_t *arg = assign_dev && st.max ? pl->batch_arg + pl->arg_row[s] * cur : nullptr;   // a max step: its rows
            rc = contract_batched_step(ctx, (int)st.operands.size(), ops, *ov, *oc, st.elim, cur, evt + b0, nb, n_cols, dst,
                                       &pl->offtab_host[s], &pl->offtab_dev[s], arg);
            for (int id : st.operands)
                if (pl->f[id].last_use == (int)s) dev_free(ctx, owned[id]);
        }
        for (double *&p : owned) dev_free(ctx, p);
        if (!pl->is_mar && (pl->steps.empty() || pl->steps.back().out != -2)) rc = fill(ctx, result_dev + b0, cur, 1.0);
        if (rc == BNPP_OK && assign_dev) rc = mpe_decode_batch_launch(pl, nb, b0, cur, evt + b0, nb, 1, assign_dev);
    }
    dev_free(ctx, evt);
    // inside the run, hence inside its captured graph: a replay normalises too
    if (rc == BNPP_OK && pl->is_mar && pl->normalize)
        rc = normalize_segments_batched(ctx, result_dev, pl->mar_off_dev, pl->mar_size_dev, (int)pl->mar_off.size(), nb);
    return rc;
}

// Graph::ordering on the host (code/graph.cpp:41-195), same tie-breaks as the reference.
// scopes: factor scopes AFTER conditioning; vars: the variables to order, in the caller's order.
int bnpp_elim_order(int nvars, const uint32_t *card, int nfac, const bnpp_scope *scopes, int n_obs,
                    const uint32_t *obs_var, int n_vars_to_order, const uint32_t *vars, int heuristic,
                    uint32_t *order_out, uint32_t *n_order_out, uint32_t *width_out)
{
    // heuristic | 0x100 runs the slow path on the reference's own containers (cross-check in tests)
    const bool reference_containers = (heuristic & 0x100) != 0;
    heuristic &= 0xff;
    if (nvars < 0 || nfac < 0 || n_obs < 0 || n_vars_to_order < 0 || heuristic < 0 || heuristic > 2) return BNPP_EINVAL;
    const std::vector<char> observed = observed_mask(nvars, n_obs, obs_var);
    const std::vector<std::vector<unsigned>> sc = conditioned_scopes(observed, nvars, nfac, scopes);
    std::vector<unsigned> c(card, card + nvars);
    const std::vector<unsigned> v = unobserved(observed, nvars, n_vars_to_order, vars);
    unsigned width = 0;
    std::vector<unsigned> order;
    if (reference_containers) order = InteractionGraph(sc, c).ordering(v, (Heuristic)heuristic, width);
    else order = FastOrderer(sc, c).ordering(v, (Heuristic)heuristic, width);
    for (size_t i = 0; i < order.size(); ++i) order_out[i] = order[i];
    if (n_order_out) *n_order_out = (uint32_t)order.size();
    if (width_out) *width_out = width;
    return BNPP_OK;
}

// Constrained order of marginal MAP: `first` (the summed variables) by the heuristic as bnpp_elim_order orders them,
// then `last` (the MAP variables) on the same graph, the fill edges of the first phase in place.  Width: both phases.
int bnpp_elim_order_constrained(int nvars, const uint32_t *card, int nfac, const bnpp_scope *scopes, int n_obs,
                                const uint32_t *obs_var, int n_first, const uint32_t *first, int n_last, const uint32_t *last,
                                int heuristic, uint32_t *order_out, uint32_t *n_order_out, uint32_t *width_out)
{
    const bool reference_containers = (heuristic & 0x100) != 0;
    heuristic &= 0xff;
    if (nvars < 0 || nfac < 0 || n_obs < 0 || n_first < 0 || n_last < 0 || heuristic < 0 || heuristic > 2) return BNPP_EINVAL;
    const std::vector<char> observed = observed_mask(nvars, n_obs, obs_var);
    const std::vector<std::vector<unsigned>> sc = conditioned_scopes(observed, nvars, nfac, scopes);
    std::vector<unsigned> c(card, card + nvars);
    const std::vector<unsigned> f = unobserved(observed, nvars, n_first, first), l = unobserved(observed, nvars, n_last, last);
    unsigned w1 = 0, w2 = 0;
    std::vector<unsigned> order, tail;
    if (reference_containers) {
        InteractionGraph g(sc, c);
        order = g.ordering_in_place(f, (Heuristic)heuristic, w1);
        tail = g.ordering_in_place(l, (Heuristic)heuristic, w2);
    } else {
        FastOrderer g(sc, c);
        order = g.ordering(f, (Heuristic)heuristic, w1);
        tail = g.ordering(l, (Heuristic)heuristic, w2);
    }
    order.insert(order.end(), tail.begin(), tail.end());
    for (size_t i = 0; i < order.size(); ++i) order_out[i] = order[i];
    if (n_order_out) *n_order_out = (uint32_t)order.size();
    if (width_out) *width_out = std::max(w1, w2);
    return BNPP_OK;
}

// The g variables of the widest elimination clique that `order` eliminates last (SURVEY §8e):
// with the canonical layout they are the leading axes of every wide table, so fixing them to
// a rank's values selects that rank's slab.  scopes: factor scopes (conditioned); host only.
int bnpp_pick_shard_vars(int nfac, const bnpp_scope *scopes, int n_order, const uint32_t *order, int g, uint32_t *out)
{
    if (nfac < 0 || n_order < 0 || g < 0 || (g > 0 && !out)) return BNPP_EINVAL;
    std::map<uint32_t, int> rank;
    for (int i = 0; i < n_order; ++i) rank[order[i]] = i;
    std::vector<std::vector<std::vector<uint32_t>>> bucket(n_order);
    auto place = [&](const std::vector<uint32_t> &sc) {
        int best = -1;
        for (uint32_t v : sc) {
            auto it = rank.find(v);
            if (it != rank.end() && (best < 0 || it->second < best)) best = it->second;
        }
        if (best >= 0) bucket[best].push_back(sc);
    };
    for (int f = 0; f < nfac; ++f) {
        std::vector<uint32_t> sc;
        for (int i = 0; i < scopes[f].rank; ++i)
            if (rank.count(scopes[f].var_id[i])) sc.push_back(scopes[f].var_id[i]);
        place(sc);
    }
    std::vector<uint32_t> widest;
    for (int i = 0; i < n_order; ++i) {
        if (bucket[i].empty()) continue;
        std::vector<uint32_t> u;
        for (auto &sc : bucket[i])
            for (uint32_t v : sc)
                if (std::find(u.begin(), u.end(), v) == u.end()) u.push_back(v);
        if (u.size() > widest.size()) widest = u;
        u.erase(std::remove(u.begin(), u.end(), order[i]), u.end());
        place(u);
    }
    std::sort(widest.begin(), widest.end(), [&](uint32_t a, uint32_t b) { return rank[a] < rank[b]; });
    const int n = (int)widest.size() < g ? (int)widest.size() : g;
    for (int i = 0; i < n; ++i) out[i] = widest[widest.size() - n + i];
    return n;
}

int bnpp_order_width(int nvars, const uint32_t *card, int nfac, const bnpp_scope *scopes, int n_order,
                     const uint32_t *order, uint32_t *width_out)
{
    if (nvars < 0 || nfac < 0 || n_order < 0 || !width_out) return BNPP_EINVAL;
    std::vector<std::vector<unsigned>> sc(nfac);
    for (int f = 0; f < nfac; ++f) sc[f].assign(scopes[f].var_id, scopes[f].var_id + scopes[f].rank);
    std::vector<unsigned> c(card, card + nvars);
    InteractionGraph g(sc, c);
    std::vector<unsigned> o(order, order + n_order);
    *width_out = g.order_width(o);
    return BNPP_OK;
}

}  // extern "C"
