// Multi-valued elimination: out[o] = sum_{x < cx} prod_k F_k[pi_k(o, x)] for cx > 2, any cardinalities.
//
// Replaces the same reference code as contract.cu -- `prod *= *pf` over a bucket, then `prod.sum_out(var)`
// (code/model.cpp:414-418; code/factor.cpp:117-147, 182-212) -- for the networks whose variables are not
// binary (Munin*, Link, Barley, Mildew, Water, Diabetes, Pigs ...).  With one output entry per thread a warp
// reads 32 runs of cx doubles that lie 8 * cx bytes apart: every load instruction touches 32 sectors for 256
// useful bytes.  Here the lanes walk the UNION table in the order that is contiguous in the large operands (the
// eliminated variable fastest when it is their stride-1 axis -- always so in the canonical layout of ve.cu --
// else the output index fastest), so a warp's load is one or a few 256-byte runs, and the sum over x happens in
// shared memory:
//
//   tile   = T consecutive output entries = [g digits of one "split" axis] x [all axes inside it], E = T * cx
//            union entries; T * cx <= 2048 so a thread owns up to 8 entries
//   phase 1: entry e -> operand offsets and stage slot come from a TABLE (the same for every tile: what depends
//            on the tile is one base offset per operand); all loads of a batch of entries are issued before the
//            first multiply; the product goes to stage[o * cxp + x], cxp odd => phase 2 is bank-conflict free
//   phase 2: thread j adds row j up in the reference's order (0 + p(x=0) + p(x=1) + ...) and stores out[j]
//            (consecutive threads, consecutive addresses)
// The table (<= 32 KB) is built by the plan, lives in device memory next to the launch descriptor and is brought
// into shared memory once per CTA by ONE bulk copy (cp.async.bulk -> mbarrier, the TMA engine; no thread moves
// it).  Tile bases are a mixed-radix decomposition of the tile index (multiply-high division, common.cuh) done by
// K+1 threads per tile one tile ahead.  Arithmetic: __dmul_rn / __dadd_rn in the reference's order => every
// entry bit-identical to code/factor.cpp.  HBM-bound: algorithmic bytes 8 * (sum #F_k + #out) (SURVEY 8d).
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <vector>

#include "common.cuh"
#include "contract.hpp"
#include "contract_mv.hpp"
#include "chain.hpp"

extern "C" int bnpp_alloc(bnpp_ctx *ctx, uint64_t n_doubles, double **dptr);
extern "C" int bnpp_free(bnpp_ctx *ctx, double *dptr);

namespace bnpp {

__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// base offset of operand `which` (< K), or (which == K) the tile's first output entry and its valid entries
template <int K>
__device__ __forceinline__ void mv_tile(const ParamsMV &p, uint32_t t, uint32_t which, uint32_t *dst)
{
    uint32_t outer = t, c = 0;
    if (p.n_split > 1) {
        outer = fastdiv(t, p.dsplit);
        c = t - outer * p.n_split;
    }
    if (which == (uint32_t)K) {
        dst[K] = outer * (p.ext_split * p.inner) + c * p.g * p.inner;
        return;
    }
    uint32_t b = c * p.g * p.s_split[which], rem = outer;
#pragma unroll 1
    for (int a = (int)p.R - 1; a > 0; --a) {
        const uint32_t q = fastdiv(rem, p.div[a]);
        b += (rem - q * p.div[a].d) * p.s[which][a];
        rem = q;
    }
    if (p.R > 0) b += rem * p.s[which][0];
    dst[which] = b;
}

template <int KP>
__device__ __forceinline__ void mv_entry(const uint32_t *tab, uint32_t e, uint32_t (&w)[KP])
{
    if (KP == 2) {
        const uint2 a = *reinterpret_cast<const uint2 *>(tab + 2 * e);
        w[0] = a.x; w[1] = a.y;
    } else {
#pragma unroll
        for (int i = 0; i < KP / 4; ++i) {
            const uint4 a = *reinterpret_cast<const uint4 *>(tab + KP * e + 4 * i);
            w[4 * i] = a.x; w[4 * i + 1] = a.y; w[4 * i + 2] = a.z; w[4 * i + 3] = a.w;
        }
    }
}

// the loads of one tile: every entry of the thread in flight at once.  The table holds UB * kBlock entries: those
// past the tile's E are padding that re-reads entry 0 and parks its product in a slot nobody sums, so there is no
// predicate anywhere (and no partial tile: the plan only cuts the split axis into equal chunks).
template <int K, int KP, int UB>
__device__ __forceinline__ void mv_load(const ParamsMV &p, const uint32_t *tab, const uint32_t *base, double (&v)[UB][K],
                                        uint32_t (&slot)[UB])
{
#pragma unroll
    for (int u = 0; u < UB; ++u) {
        uint32_t w[KP];
        mv_entry<KP>(tab, threadIdx.x + u * kBlock, w);
        slot[u] = w[KP - 1];
#pragma unroll
        for (int k = 0; k < K; ++k) v[u][k] = ld1(p.h.in[k] + (base[k] + w[k]));      // 32-bit index, one widening multiply-add
    }
}

// Software pipeline over a CTA's tiles: the loads of tile n+1 are issued (into registers) right after the barrier
// that publishes tile n's products, so they are in flight while tile n is summed up and stored -- a CTA has loads
// outstanding all the time except while it multiplies and stages.
template <int K, int KP, int UB>
__global__ void __launch_bounds__(kBlock) contract_mv(const __grid_constant__ ParamsMV p)
{
    extern __shared__ __align__(128) unsigned char mv_smem[];
    __shared__ uint32_t s_base[2][kMaxK + 2];
    __shared__ __align__(8) uint64_t s_bar;
    uint32_t *tab = reinterpret_cast<uint32_t *>(mv_smem);
    const uint32_t tab_bytes = UB * kBlock * KP * 4u;
    double *stage = reinterpret_cast<double *>(mv_smem + ((tab_bytes + 127u) & ~127u));
    const uint32_t tid = threadIdx.x;
    const uint32_t bar = smem_addr(&s_bar);

    // the entry table: one bulk copy global -> shared (TMA engine), completion counted in bytes on an mbarrier
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(tab_bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_addr(tab)), "l"(p.tab), "r"(tab_bytes), "r"(bar)
                     : "memory");
    }
    uint32_t t = blockIdx.x;
    if (tid <= (uint32_t)K && t < p.n_tiles) mv_tile<K>(p, t, tid, s_base[0]);
    asm volatile("{\n.reg .pred P1;\nMV_WAIT:\nmbarrier.try_wait.parity.shared::cta.b64 P1, [%0], 0;\n@P1 bra MV_DONE;\nbra MV_WAIT;\nMV_DONE:\n}"
                 ::"r"(bar)
                 : "memory");
    __syncthreads();

    const uint32_t cx = p.h.cx, cxp = p.cxp;
    double zacc = 0.0;
    double v[UB][K];
    uint32_t slot[UB];
    if (t < p.n_tiles) mv_load<K, KP, UB>(p, tab, s_base[0], v, slot);
    for (uint32_t buf = 0; t < p.n_tiles; buf ^= 1u) {
        const uint32_t tn = t + gridDim.x;
        // the bases of this CTA's next tile (read after the barrier below)
        if (tid <= (uint32_t)K && tn < p.n_tiles) mv_tile<K>(p, tn, tid, s_base[buf ^ 1u]);
        // products of this tile's union entries -> stage
#pragma unroll
        for (int u = 0; u < UB; ++u) {
            double a = v[u][0];
#pragma unroll
            for (int k = 1; k < K; ++k) a = __dmul_rn(a, v[u][k]);
            stage[slot[u]] = a;
        }
        __syncthreads();
        const uint32_t tv = p.T;
        double *dst = p.h.out + s_base[buf][K];
        if (tn < p.n_tiles) mv_load<K, KP, UB>(p, tab, s_base[buf ^ 1u], v, slot);
        // one thread per output entry adds its row up in the reference's order
        for (uint32_t j = tid; j < tv; j += kBlock) {
            const double *row = stage + j * cxp;
            double acc = 0.0;
#pragma unroll 4
            for (uint32_t x = 0; x < cx; ++x) acc = __dadd_rn(acc, row[x]);
            dst[j] = acc;
            zacc = __dadd_rn(zacc, acc);
        }
        __syncthreads();
        t = tn;
    }
    if (p.h.z) grid_sum_to(zacc, p.h.partials, p.h.ticket, p.h.z);
}

typedef void (*mv_fn)(const ParamsMV);

// UB = table entries per thread: 8 (tiles of up to 2048 union entries) or 4; K >= 4 keeps 4 (registers)
static mv_fn pick_mv(int k, int ub, int &KP)
{
    KP = k == 1 ? 2 : (k <= 3 ? 4 : 8);
    switch (k * 16 + ub) {
    case 1 * 16 + 8: return contract_mv<1, 2, 8>;
    case 1 * 16 + 4: return contract_mv<1, 2, 4>;
    case 2 * 16 + 8: return contract_mv<2, 4, 8>;
    case 2 * 16 + 4: return contract_mv<2, 4, 4>;
    case 3 * 16 + 8: return contract_mv<3, 4, 8>;
    case 3 * 16 + 4: return contract_mv<3, 4, 4>;
    case 4 * 16 + 4: return contract_mv<4, 8, 4>;
    case 5 * 16 + 4: return contract_mv<5, 8, 4>;
    case 6 * 16 + 4: return contract_mv<6, 8, 4>;
    default: return nullptr;
    }
}

// process-wide knobs (bnpp_tuning_set): seeded from the environment on first use
struct MvKnobs {
    uint64_t min_entries;
    uint32_t emax;
    uint32_t staged = 1;
    uint32_t staged_tma = 1;
    uint32_t staged_async = 1;
    uint32_t chain_depth = kChainDefaultDepth;      // levels of a ve.cu window (contract_chain); 0 or 1 = no windows
    MvKnobs()
    {
        const char *e = getenv("BNPP_MV_MIN_ENTRIES");
        min_entries = e ? (uint64_t)strtoull(e, nullptr, 10) : (uint64_t)(1u << 15);
        e = getenv("BNPP_MV_EMAX");
        emax = e ? (uint32_t)atoi(e) : 0u;
        e = getenv("BNPP_STAGED_TMA");
        if (e && e[0] == '0') staged_tma = 0;
        e = getenv("BNPP_STAGED_ASYNC");
        if (e && e[0] == '0') staged_async = 0;
        e = getenv("BNPP_CHAIN_DEPTH");
        if (e) chain_depth = (uint32_t)atoi(e);
    }
};
static MvKnobs &knobs()
{
    static MvKnobs k;
    return k;
}

uint64_t mv_min_entries() { return knobs().min_entries; }
bool mv_staged_enabled() { return knobs().staged != 0; }
bool staged_tma_enabled() { return knobs().staged_tma != 0; }
uint32_t chain_depth_knob() { return knobs().chain_depth; }
bool staged_async_enabled() { return knobs().staged_async != 0; }

static uint32_t mv_emax(int k)
{
    const uint32_t forced = knobs().emax;
    const uint32_t cap = k >= 4 ? 4u * kBlock : 8u * kBlock;      // entries per thread of a full tile (UB) x kBlock
    if (forced >= 64) return std::min(forced, cap);
    return cap;
}

// co-resident CTAs per SM of a variant at a given dynamic shared memory size; the opt-in above 48 KB is per
// device and function, so the cache is keyed by both
static int mv_resident(bnpp_ctx *ctx, mv_fn fn, unsigned smem)
{
    static std::mutex mu;
    static std::map<std::pair<int, const void *>, unsigned> granted;
    std::lock_guard<std::mutex> lock(mu);
    const auto key = std::make_pair(ctx->device, reinterpret_cast<const void *>(fn));
    smem = ((smem + 1023u) >> 10) << 10;        // opt-in and occupancy are asked per KB of shared memory (cached)
    auto it = granted.find(key);
    if (it == granted.end() || it->second < smem) {
        if (cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
            cudaGetLastError();
            return 0;
        }
        granted[key] = smem;
    }
    static std::map<std::pair<std::pair<int, const void *>, unsigned>, int> occupancy;       // (device, fn, KB of shared memory)
    const auto okey = std::make_pair(key, smem >> 10);
    auto oc = occupancy.find(okey);
    if (oc != occupancy.end()) return oc->second;
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kBlock, smem) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    occupancy[okey] = per_sm;
    return per_sm;
}

int plan_mv(bnpp_ctx *ctx, LaunchDesc *d, int k, uint32_t cx, const uint64_t *sx, const uint64_t *op_bytes,
            const std::vector<MVAxis> &axes, uint64_t n_out, const ParamsHead &h)
{
    if (k < 1 || k > kMaxK || cx < 2) return 1;
    const uint32_t emax = mv_emax(k);
    const uint32_t tmax = emax / cx;
    if (tmax < 1) return 1;
    const int n = (int)axes.size();

    // tile = [g digits of the split axis] x [every axis inside it]; g divides the extent, so all tiles are full
    uint64_t inner = 1;
    int split = n - 1;
    while (split >= 0 && inner * axes[split].ext <= tmax) inner *= axes[split--].ext;
    uint32_t g = 1, ext_split = 1;
    if (split >= 0) {
        ext_split = axes[split].ext;
        const uint32_t gmax = (uint32_t)std::min<uint64_t>(ext_split, tmax / inner);
        double best = -1.0;
        for (uint32_t c = 1; c <= gmax; ++c) {
            if (ext_split % c) continue;
            const uint64_t e = (uint64_t)c * inner * cx;
            const uint64_t slots = e <= 4u * kBlock ? 4u * kBlock : 8u * kBlock;
            const double lanes = (double)e / (double)slots;                    // table entries that are padding
            const double amort = (double)e / (double)(e + 192);              // barriers and bases per tile
            const double score = lanes * amort;
            if (score >= best) { best = score; g = c; }
        }
    }
    const uint32_t T = (uint32_t)(g * inner), E = T * cx, cxp = cx | 1u;
    if ((uint64_t)T * cxp + 1 >= (1u << 16)) return 1;
    const int UB = (E <= 4u * kBlock) ? 4 : 8;
    int KP = 0;
    mv_fn fn = pick_mv(k, UB, KP);
    if (!fn) return 1;

    // outer axes (outside the split axis), neighbours that are contiguous in every operand merged
    struct Outer { uint64_t ext; uint64_t s[kMaxK]; };
    std::vector<Outer> outer;
    for (int a = 0; a < split; ++a) {
        Outer o;
        o.ext = axes[a].ext;
        for (int q = 0; q < kMaxK; ++q) o.s[q] = q < k ? axes[a].s[q] : 0;
        if (!outer.empty()) {
            Outer &up = outer.back();
            bool ok = up.ext * o.ext < (1ull << 32);
            for (int q = 0; q < k && ok; ++q) ok = (up.s[q] == o.s[q] * o.ext);
            if (ok) {
                up.ext *= o.ext;
                for (int q = 0; q < k; ++q) up.s[q] = o.s[q];
                continue;
            }
        }
        outer.push_back(o);
    }
    if ((int)outer.size() > kMaxR) return 1;

    ParamsMV &p = d->mvp;
    memset(&p, 0, sizeof p);
    p.h = h;
    p.h.n_items = n_out;
    p.h.cx = cx;
    p.E = E;
    p.T = T;
    p.cxp = cxp;
    p.inner = (uint32_t)inner;
    p.g = g;
    p.ext_split = ext_split;
    p.n_split = ext_split / g;
    p.R = (uint32_t)outer.size();
    uint64_t n_outer = 1;
    for (size_t a = 0; a < outer.size(); ++a) {
        p.div[a] = make_fastdiv((uint32_t)outer[a].ext);
        n_outer *= outer[a].ext;
        for (int q = 0; q < k; ++q) {
            if (outer[a].s[q] >= (1ull << 32)) return 1;
            p.s[q][a] = (uint32_t)outer[a].s[q];
        }
    }
    if (n_outer * p.n_split >= (1ull << 32)) return 1;
    p.n_tiles = (uint32_t)(n_outer * p.n_split);
    if (p.n_split > 1) p.dsplit = make_fastdiv(p.n_split);
    for (int q = 0; q < k; ++q) {
        const uint64_t s = split >= 0 ? axes[split].s[q] : 0;
        if (s >= (1ull << 32) || sx[q] >= (1ull << 32)) return 1;
        p.s_split[q] = (uint32_t)s;
        p.h.sx[q] = (uint32_t)sx[q];
    }

    // enumeration order inside a tile: the eliminated variable fastest when it is the fastest axis of the
    // heaviest operand that has it (then a warp reads runs of cx doubles back to back), else the output index
    int heavy = -1;
    for (int q = 0; q < k; ++q)
        if (sx[q] && (heavy < 0 || op_bytes[q] > op_bytes[heavy])) heavy = q;
    bool x_fast = true;
    if (heavy >= 0)
        for (int a = std::max(split, 0); a < n; ++a)
            if (axes[a].s[heavy] && axes[a].s[heavy] < sx[heavy]) x_fast = false;

    // the eliminated variable is a slow axis of the heavy operand: one output entry per thread with a loop over its values
    // (contract_generic) already reads and writes whole rows of the fastest axes -- gathering through a table adds nothing
    if (!x_fast) return 1;
    // the entry table: E real entries, then padding up to UB * kBlock that re-reads entry 0 into a spare stage slot
    const size_t slots = (size_t)UB * kBlock;
    const size_t words = slots * KP;
    std::vector<uint32_t> tab(words, 0);
    {
        const int first = std::max(split, 0);
        std::vector<uint32_t> digit(n, 0);
        uint64_t loc[kMaxK] = {0};
        for (uint32_t o = 0; o < T; ++o) {
            for (uint32_t x = 0; x < cx; ++x) {
                const size_t e = x_fast ? (size_t)o * cx + x : (size_t)x * T + o;
                for (int q = 0; q < k; ++q) {
                    const uint64_t off = loc[q] + (uint64_t)x * sx[q];
                    if (off >= (1ull << 32)) return 1;
                    tab[e * KP + q] = (uint32_t)off;
                }
                tab[e * KP + KP - 1] = o * cxp + x;
            }
            // odometer over [split digit][inner axes], innermost fastest (the split digit never wraps inside a tile)
            for (int a = n - 1; a >= first; --a) {
                if (++digit[a] < axes[a].ext || a == first) {
                    for (int q = 0; q < k; ++q) loc[q] += axes[a].s[q];
                    break;
                }
                digit[a] = 0;
                for (int q = 0; q < k; ++q) loc[q] -= (uint64_t)(axes[a].ext - 1) * axes[a].s[q];
            }
        }
        for (size_t e = E; e < slots; ++e) {
            for (int q = 0; q < k; ++q) tab[e * KP + q] = tab[q];
            tab[e * KP + KP - 1] = T * cxp;                      // the spare slot after the last row
        }
    }

    const unsigned smem = (unsigned)(((words * 4 + 127) & ~(size_t)127) + ((size_t)T * cxp + 1) * sizeof(double));
    const int per_sm = mv_resident(ctx, fn, smem);
    if (per_sm < 1) return 1;
    double *store = nullptr;
    int rc = bnpp_alloc(ctx, words / 2 + 2, &store);
    if (rc != BNPP_OK) return rc;
    rc = stage_upload(ctx, store, tab.data(), words * 4);
    if (rc != BNPP_OK) {
        bnpp_free(ctx, store);
        return rc;
    }
    d->mv_tab = reinterpret_cast<uint32_t *>(store);
    p.tab = d->mv_tab;
    d->mv = true;
    d->p2 = false;
    d->staged = false;
    d->smem = smem;
    d->fn = reinterpret_cast<const void *>(fn);
    d->grid = (unsigned)std::min<uint64_t>(p.n_tiles, (uint64_t)ctx->sm_count * per_sm);
    d->k = k;
    d->variant = x_fast ? "mv/x" : "mv/o";
    d->C = (int)cx;
    d->V = 1;
    d->U = UB;
    d->div = false;
    d->generic = false;
    d->R = p.R;
    return BNPP_OK;
}

void contract_release(bnpp_ctx *ctx, LaunchDesc &d)
{
    if (d.mv_tab) {
        if (ctx) bnpp_free(ctx, reinterpret_cast<double *>(d.mv_tab));
        d.mv_tab = nullptr;
    }
}

}  // namespace bnpp

extern "C" int bnpp_tuning_set(const char *key, uint64_t value)
{
    if (!key) return BNPP_EINVAL;
    if (!strcmp(key, "mv_min_entries")) bnpp::knobs().min_entries = value;
    else if (!strcmp(key, "mv_emax")) bnpp::knobs().emax = (uint32_t)value;
    else if (!strcmp(key, "mv_staged")) bnpp::knobs().staged = (uint32_t)value;
    else if (!strcmp(key, "staged_tma")) bnpp::knobs().staged_tma = (uint32_t)value;
    else if (!strcmp(key, "staged_async")) bnpp::knobs().staged_async = (uint32_t)value;
    else if (!strcmp(key, "chain_depth")) bnpp::knobs().chain_depth = (uint32_t)value;
    else return BNPP_EINVAL;
    return BNPP_OK;
}

extern "C" int bnpp_tuning_get(const char *key, uint64_t *value)
{
    if (!key || !value) return BNPP_EINVAL;
    if (!strcmp(key, "mv_min_entries")) *value = bnpp::knobs().min_entries;
    else if (!strcmp(key, "mv_emax")) *value = bnpp::knobs().emax;
    else if (!strcmp(key, "mv_staged")) *value = bnpp::knobs().staged;
    else if (!strcmp(key, "staged_tma")) *value = bnpp::knobs().staged_tma;
    else if (!strcmp(key, "staged_async")) *value = bnpp::knobs().staged_async;
    else if (!strcmp(key, "chain_depth")) *value = bnpp::knobs().chain_depth;
    else return BNPP_EINVAL;
    return BNPP_OK;
}
