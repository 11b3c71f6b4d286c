// K9 -- variable elimination of a whole plan in one launch, intermediates in shared memory.
//
// Replaces, for plans whose steps are all small, the per-bucket launches of ve.cu / batched.cu
// (reference: the bucket loop of BN::variable_elimination, code/model.cpp:409-439, run once per
// evidence set by BN::partition, code/model.cpp:275-294).  A group of G lanes owns one evidence
// set and walks the step list of fused.hpp:
//   * the arena of a set (its live intermediates, first-fit over a depth-first step order that
//     keeps it small) sits in shared memory.  The sets of a warp are interleaved in PAIRS of
//     doubles -- element e of set s lives at  (e & ~1) * SPW + 2 s + (e & 1)  of the warp's slice
//     -- and lane l of set s is thread  l * SPW + s  of the warp: lanes reading consecutive
//     pairs of their sets then hit consecutive 16-byte slots (no bank conflicts), and the two
//     values of a binary eliminated variable (stride 1 in every intermediate, canonical layout
//     of ve.cu) arrive in ONE 128-bit shared load;
//   * a resident CPT is read in place through the base offset its observed axes select
//     (Factor::conditioning, code/factor.cpp:214-242, reduced to one multiply-add per axis);
//   * operand offsets per output entry come from the step's table (same numbers for every set);
//   * nothing but the result of the last step is written to HBM.
// Per entry the arithmetic is that of contract.cu / batched.cu -- operands multiplied in bucket
// order with __dmul_rn, values of the eliminated variable added in index order with __dadd_rn
// -- so a result is bit-identical to the launch-per-bucket paths.
// MAX (ve_fused_max, the batch engine of MPE plans): the same products, the maximum over the eliminated variable by the
// rule of contract.cu's max-product kernels (start at x = 0, a later x replaces it only if its product is strictly
// greater: ties keep the lowest x, a NaN never replaces a number), and the argmax byte of every output entry of a
// kFusedMax step in global memory -- ~14 KB of argmax per set of config 5 would not fit in shared memory.
// MIXED (ve_fused_mixed, the batch engine of MAP plans that also sum): a kFusedMax step takes the MAX path above, every
// other step the sum path of ve_fused (same products, same order of additions; no partition).
#include <cstdlib>
#include <map>
#include <mutex>

#include "common.cuh"
#include "fused.hpp"

namespace bnpp {

extern __shared__ __align__(16) double arena_smem[];

__device__ __forceinline__ uint4 ldg4(const uint32_t *p) { return __ldg(reinterpret_cast<const uint4 *>(p)); }

template <int G>
__device__ __forceinline__ void group_sync()
{
    if (G <= 32) __syncwarp();
    else __syncthreads();
}

// where this thread's evidence set keeps its arena, and where results go
template <int SPW>
struct SetView {
    uint32_t wbase;     // index (doubles) of element 0 of the set inside arena_smem; even
    __device__ __forceinline__ uint32_t at(uint32_t e) const { return wbase + (e & ~1u) * SPW + (e & 1u); }
    __device__ __forceinline__ uint32_t pair(uint32_t e) const { return wbase + e * SPW; }      // e even
};

struct Operands {
    uint32_t base[kMaxK];           // arena operand: element offset of the table inside the set's arena
    uint32_t sx[kMaxK];             // stride of the eliminated variable
    const double *cpt[kMaxK];       // CPT operand: the table, evidence offset applied
};

struct Dest {
    double *result;     // != nullptr: this step writes the result buffer, entry o at result[o * stride]
    uint64_t stride;
    uint32_t out_off;   // arena destination: element offset
    bool store;
    uint8_t *arg;       // MAX, != nullptr: the argmax of entry o goes to arg[o * arg_stride]
    uint32_t arg_stride;
};

template <int SPW, bool MAX = false>
__device__ __forceinline__ void put(const SetView<SPW> &v, const Dest &d, uint32_t o, double val, uint32_t best = 0)
{
    if (d.result) {
        if (d.store) d.result[(uint64_t)o * d.stride] = val;
    } else {
        arena_smem[v.at(d.out_off + o)] = val;
    }
    if (MAX && d.arg && d.store) d.arg[(uint64_t)o * d.arg_stride] = (uint8_t)best;
}

// Binary eliminated variable, every arena operand with the variable at stride 1 on an even
// offset (a 16-byte pair), AMASK = which operands are arena tables -- the shape of every bucket
// of an all-binary network.  Two output entries per trip, all loads of both before the math.
template <int K, unsigned AMASK, int G, int SPW, bool MAX>
__device__ __forceinline__ double entries_pairs(const SetView<SPW> &v, const Operands &op, const uint32_t *__restrict__ tab,
                                                uint32_t n_out, uint32_t lane, const Dest &d)
{
    double zacc = 0.0;
    for (uint32_t o0 = lane; o0 < n_out; o0 += 2 * G) {
        const bool two = o0 + G < n_out;
        const uint32_t o1 = two ? o0 + G : o0;
        uint32_t off0[K], off1[K];
#pragma unroll
        for (int q = 0; q < K; ++q) {
            off0[q] = __ldg(tab + (size_t)q * n_out + o0);
            off1[q] = __ldg(tab + (size_t)q * n_out + o1);
        }
        double a0[K], a1[K], b0[K], b1[K];
#pragma unroll
        for (int q = 0; q < K; ++q) {
            if ((AMASK >> q) & 1u) {
                const double2 pa = *reinterpret_cast<const double2 *>(&arena_smem[v.pair(op.base[q] + off0[q])]);
                const double2 pb = *reinterpret_cast<const double2 *>(&arena_smem[v.pair(op.base[q] + off1[q])]);
                a0[q] = pa.x; a1[q] = pa.y;
                b0[q] = pb.x; b1[q] = pb.y;
            } else {
                a0[q] = __ldg(op.cpt[q] + off0[q]);
                a1[q] = __ldg(op.cpt[q] + off0[q] + op.sx[q]);
                b0[q] = __ldg(op.cpt[q] + off1[q]);
                b1[q] = __ldg(op.cpt[q] + off1[q] + op.sx[q]);
            }
        }
        double x0 = a0[0], x1 = a1[0], y0 = b0[0], y1 = b1[0];
#pragma unroll
        for (int q = 1; q < K; ++q) {
            x0 = __dmul_rn(x0, a0[q]);
            x1 = __dmul_rn(x1, a1[q]);
            y0 = __dmul_rn(y0, b0[q]);
            y1 = __dmul_rn(y1, b1[q]);
        }
        if (MAX) {
            const bool ga = x1 > x0, gb = y1 > y0;
            put<SPW, true>(v, d, o0, ga ? x1 : x0, ga);
            if (two) put<SPW, true>(v, d, o1, gb ? y1 : y0, gb);
            continue;
        }
        const double ra = __dadd_rn(x0, x1), rb = __dadd_rn(y0, y1);
        put<SPW>(v, d, o0, ra);
        zacc = __dadd_rn(zacc, ra);
        if (two) {
            put<SPW>(v, d, o1, rb);
            zacc = __dadd_rn(zacc, rb);
        }
    }
    return zacc;
}

// any cardinality, any operand layout; amask: which operands are arena tables
template <int K, int G, int SPW, bool MAX>
__device__ __forceinline__ double entries_any(const SetView<SPW> &v, const Operands &op, uint32_t amask,
                                              const uint32_t *__restrict__ tab, uint32_t n_out, uint32_t cx, uint32_t lane,
                                              const Dest &d)
{
    double zacc = 0.0;
    for (uint32_t o = lane; o < n_out; o += G) {
        uint32_t off[K];
#pragma unroll
        for (int q = 0; q < K; ++q) off[q] = __ldg(tab + (size_t)q * n_out + o);
        double acc = 0.0;
        uint32_t best = 0;
        for (uint32_t x = 0; x < cx; ++x) {
            double val = 0.0;
#pragma unroll
            for (int q = 0; q < K; ++q) {
                const uint32_t e = off[q] + x * op.sx[q];
                const double t = ((amask >> q) & 1u) ? arena_smem[v.at(op.base[q] + e)] : __ldg(op.cpt[q] + e);
                val = (q == 0) ? t : __dmul_rn(val, t);
            }
            if (!MAX) {
                acc = (x == 0) ? val : __dadd_rn(acc, val);
            } else if (x == 0 || val > acc) {
                acc = val;
                best = x;
            }
        }
        if (MAX) {
            put<SPW, true>(v, d, o, acc, best);
            continue;
        }
        put<SPW>(v, d, o, acc);
        zacc = __dadd_rn(zacc, acc);
    }
    return zacc;
}

template <int K, int G, int SPW, bool MAX>
__device__ __forceinline__ double entries_dispatch(const SetView<SPW> &v, const Operands &op, uint32_t amask, bool pairs,
                                                   const uint32_t *tab, uint32_t n_out, uint32_t cx, uint32_t lane, const Dest &d)
{
    if (pairs && K <= 3) {
        // compile-time arena mask for the common operand counts
        switch (amask) {
        case 0: return entries_pairs<K, 0u, G, SPW, MAX>(v, op, tab, n_out, lane, d);
        case 1: return entries_pairs<K, 1u, G, SPW, MAX>(v, op, tab, n_out, lane, d);
        case 2: if (K >= 2) return entries_pairs<K, (K >= 2 ? 2u : 0u), G, SPW, MAX>(v, op, tab, n_out, lane, d); break;
        case 3: if (K >= 2) return entries_pairs<K, (K >= 2 ? 3u : 0u), G, SPW, MAX>(v, op, tab, n_out, lane, d); break;
        case 4: if (K >= 3) return entries_pairs<K, (K >= 3 ? 4u : 0u), G, SPW, MAX>(v, op, tab, n_out, lane, d); break;
        case 5: if (K >= 3) return entries_pairs<K, (K >= 3 ? 5u : 0u), G, SPW, MAX>(v, op, tab, n_out, lane, d); break;
        case 6: if (K >= 3) return entries_pairs<K, (K >= 3 ? 6u : 0u), G, SPW, MAX>(v, op, tab, n_out, lane, d); break;
        case 7: if (K >= 3) return entries_pairs<K, (K >= 3 ? 7u : 0u), G, SPW, MAX>(v, op, tab, n_out, lane, d); break;
        default: break;
        }
    }
    return entries_any<K, G, SPW, MAX>(v, op, amask, tab, n_out, cx, lane, d);
}

// the entries of one step, k operands
template <int G, int SPW, bool MAX>
__device__ __forceinline__ double step_entries(uint32_t k, const SetView<SPW> &v, const Operands &op, uint32_t amask, bool pairs,
                                               const uint32_t *tab, uint32_t n_out, uint32_t cx, uint32_t lane, const Dest &d)
{
    switch (k) {
    case 1: return entries_dispatch<1, G, SPW, MAX>(v, op, amask, pairs, tab, n_out, cx, lane, d);
    case 2: return entries_dispatch<2, G, SPW, MAX>(v, op, amask, pairs, tab, n_out, cx, lane, d);
    case 3: return entries_dispatch<3, G, SPW, MAX>(v, op, amask, pairs, tab, n_out, cx, lane, d);
    case 4: return entries_dispatch<4, G, SPW, MAX>(v, op, amask, pairs, tab, n_out, cx, lane, d);
    case 5: return entries_dispatch<5, G, SPW, MAX>(v, op, amask, pairs, tab, n_out, cx, lane, d);
    default: return entries_dispatch<6, G, SPW, MAX>(v, op, amask, pairs, tab, n_out, cx, lane, d);
    }
}

// the steps of one program for one evidence set (b), on the G lanes that own it.
// Decoding a step costs no memory round trip: the record of a step (header, operand records, observed axes -- the same
// words for every lane of the warp) is fetched with ONE coalesced load, lane i word i, while the PREVIOUS step runs, and
// read field by field with warp shuffles; the evidence values of the set sit in registers the same way (lane l of the
// set holds values 4l .. 4l+3).  Records longer than 32 words and plans with more than 32 observed variables read the
// rest from memory.  `prog` must be readable 32 words past the last record.  MAX: see ve_fused_max; MAX and MIXED: see
// ve_fused_mixed.
template <int G, int SPW, bool MAX = false, bool MIXED = false>
__device__ __forceinline__ void run_steps(const uint32_t *__restrict__ prog, const uint32_t *__restrict__ offtab, uint32_t n_steps,
                                          const uint8_t *ev, uint32_t n_obs, double *result, double *zout, uint32_t nb, uint32_t b,
                                          bool live, const SetView<SPW> &v, uint32_t lane, double *s_red, uint8_t *arg = nullptr)
{
    const uint32_t tw = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    constexpr uint32_t kEvLanes = G < 8 ? G : 8;                // lanes of a set inside one warp that hold evidence values
    const bool ev_regs = n_obs <= 4u * kEvLanes;
    const uint32_t l = (G < 32) ? lane : tw;                    // G = 128: every warp keeps its own copy
    uint32_t evw = 0;
    if (ev_regs && l < kEvLanes) {
#pragma unroll
        for (uint32_t j = 0; j < 4; ++j)
            if (4u * l + j < n_obs) evw |= (uint32_t)ev[4u * l + j] << (8u * j);
    }
    const uint32_t my_set = (G < 32) ? tw % SPW : 0u;
    auto evidence = [&](uint32_t i) -> uint32_t {
        if (ev_regs) return (__shfl_sync(0xffffffffu, evw, (i >> 2) * SPW + my_set) >> (8u * (i & 3u))) & 0xffu;
        return ev[i];
    };
    uint32_t rec0 = 0;                      // first word of the current step's record
    uint32_t w = __ldg(prog + tw);
    for (uint32_t s = 0; s < n_steps; ++s) {
        auto word = [&](uint32_t i) -> uint32_t { return i < 32u ? __shfl_sync(0xffffffffu, w, i) : __ldg(prog + rec0 + i); };
        const uint32_t n_out = word(0), cx = word(1), kf = word(2), k = kf & 0xffu, flags = kf >> 8, tab_off = word(4);
        Dest d;
        d.out_off = word(3);
        d.store = live;
        if (flags & kFusedToResult) {
            d.result = result + ((uint64_t)d.out_off * nb + b);
            d.stride = nb;
        } else if (flags & kFusedToGlobal) {      // single queries inside a launch-per-bucket plan: a later launch reads it
            d.result = reinterpret_cast<double *>(((uint64_t)word(6) << 32) | (uint64_t)word(5));
            d.stride = 1;
        } else {
            d.result = nullptr;
            d.stride = 0;
        }
        if (MAX) {
            d.arg = (flags & kFusedMax) ? arg + ((uint64_t)word(7) * nb + b) : nullptr;
            d.arg_stride = nb;
        }
        // operand records (the k of a step is uniform over its lanes)
        uint32_t at = kFusedHeaderWords;
        Operands op;
        uint32_t amask = 0;
#pragma unroll
        for (int q = 0; q < kMaxK; ++q) {
            if (q < (int)k) {
                const uint32_t r0 = word(at), r1 = word(at + 1), r2 = word(at + 2);
                op.sx[q] = r2;
                if ((r0 & 0xffu) == 0) {
                    at += kFusedOperandWords;
                    op.base[q] = r1;
                    op.cpt[q] = nullptr;
                    amask |= 1u << q;
                } else {
                    const uint32_t r3 = word(at + 3);
                    at += kFusedOperandWords;
                    const uint32_t nobs = r0 >> 8;
                    uint32_t e = 0;
                    for (uint32_t j = 0; j < nobs; j += 2) {
                        e += word(at) * evidence(word(at + 1));
                        if (j + 1 < nobs) e += word(at + 2) * evidence(word(at + 3));
                        at += 4;
                    }
                    op.base[q] = 0;
                    op.cpt[q] = reinterpret_cast<const double *>(((uint64_t)r3 << 32) | (uint64_t)r1) + e;
                }
            }
        }
        rec0 += at;
        const uint32_t w_next = __ldg(prog + rec0 + tw);       // the next step's record, on its way while this step runs
        const uint32_t *tab = offtab + tab_off;
        const bool pairs = (flags & kFusedPairs) != 0;
        double zacc;
        if (MIXED && !(flags & kFusedMax)) zacc = step_entries<G, SPW, false>(k, v, op, amask, pairs, tab, n_out, cx, lane, d);
        else zacc = step_entries<G, SPW, MAX>(k, v, op, amask, pairs, tab, n_out, cx, lane, d);
        if (!MAX && (flags & kFusedWantZ) && zout) {      // uniform over the lanes of the set; only single queries ask for it
            double z = zacc;
            if (G <= 32) {
                // the lanes of a set are the threads l * SPW + s of the warp
#pragma unroll
                for (int o = 16; o >= SPW; o >>= 1) z = __dadd_rn(z, __shfl_xor_sync(0xffffffffu, z, o));
            } else {
                z = warp_sum(z);
                if (tw == 0) s_red[warp] = z;
                __syncthreads();
                z = 0.0;
#pragma unroll
                for (int i = 0; i < kFusedThreads / 32; ++i) z = __dadd_rn(z, s_red[i]);
            }
            if (lane == 0 && live) zout[b] = z;
        }
        group_sync<G>();     // the step's output is complete, and its operands are dead, before the next step
        w = w_next;
    }
}

// the evidence sets of a launch, a group of G lanes each
template <int G, bool MAX, bool MIXED = false>
__device__ __forceinline__ void run_sets(const FusedLaunch &p, double *s_red, uint8_t *arg)
{
    constexpr int SPW = G >= 32 ? 1 : 32 / G;       // sets per warp, interleaved in the warp's slice of the arena
    constexpr int SPC = kFusedThreads / G;          // sets per CTA
    const uint32_t tw = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    uint32_t lane, set_in_cta;
    SetView<SPW> v;
    if (G < 32) {
        lane = tw / SPW;
        set_in_cta = warp * SPW + (tw % SPW);
        v.wbase = warp * SPW * p.arena + 2u * (tw % SPW);
    } else if (G == 32) {
        lane = tw;
        set_in_cta = warp;
        v.wbase = warp * p.arena;
    } else {
        lane = threadIdx.x;
        set_in_cta = 0;
        v.wbase = 0;
    }
    const uint32_t n_groups = (p.nb + SPC - 1) / SPC;
    for (uint32_t grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
        uint32_t b = grp * SPC + set_in_cta;
        const bool live = b < p.nb;      // lanes of a missing set repeat the last one (they take part in the syncs), stores off
        if (!live) b = p.nb - 1;
        const uint8_t *ev = p.ev ? p.ev + (uint64_t)b * p.n_obs : p.ev_inline;
        run_steps<G, SPW, MAX, MIXED>(p.prog, p.offtab, p.n_steps, ev, p.n_obs, p.result, p.z, p.nb, b, live, v, lane, s_red, arg);
    }
}

template <int G>
__global__ void __launch_bounds__(kFusedThreads) ve_fused(const __grid_constant__ FusedLaunch p)
{
    __shared__ double s_red[kFusedThreads / 32];
    run_sets<G, false>(p, s_red, nullptr);
}

// an MPE program over a batch: the value of every set to p.f.result, the argmax rows to p.arg (fused.hpp)
template <int G>
__global__ void __launch_bounds__(kFusedThreads) ve_fused_max(const __grid_constant__ FusedMaxLaunch p)
{
    run_sets<G, true>(p.f, nullptr, p.arg);
}

// a MAP program over a batch: kFusedMax steps take the maximum and write their argmax rows, the others sum (fused.hpp)
template <int G>
__global__ void __launch_bounds__(kFusedThreads) ve_fused_mixed(const __grid_constant__ FusedMaxLaunch p)
{
    run_sets<G, true, true>(p.f, nullptr, p.arg);
}

// K10 -- TASKS: one launch runs many independent programs of one query, a CTA each.  A mixed plan (hundreds of tiny
// buckets around a few wide ones: Munin*, Link, Pigs, andes ...) is cut into tasks -- subtrees of the bucket tree whose
// steps are all small -- and the tasks whose inputs are ready form one launch (ve.cu, build_levels); inside a task the
// intermediates live in shared memory, its root's output goes to the plan's global arena.
__global__ void __launch_bounds__(kFusedThreads) ve_tasks(const __grid_constant__ TaskLaunch p)
{
    __shared__ double s_red[kFusedThreads / 32];
    SetView<1> v;
    v.wbase = 0;
    for (uint32_t t = blockIdx.x; t < p.n_tasks; t += gridDim.x) {
        const uint4 task = ldg4(reinterpret_cast<const uint32_t *>(p.tasks + t));      // prog offset, offtab base, steps, arena
        run_steps<128, 1>(p.prog + task.x, p.offtab + task.y, task.z, p.ev_inline, p.n_obs, p.result, p.z, 1u, 0u, true, v, threadIdx.x, s_red);
        __syncthreads();
    }
}

bool fused_valid_g(int G) { return G == 2 || G == 4 || G == 8 || G == 16 || G == 32 || G == 128; }

size_t fused_smem_bytes(int G, uint32_t arena)
{
    const uint32_t even = (arena + 1u) & ~1u;      // pairs of doubles stay together
    return (size_t)(kFusedThreads / G) * (even ? even : 2) * sizeof(double);
}

typedef void (*fused_fn)(const FusedLaunch);
typedef void (*fused_max_fn)(const FusedMaxLaunch);

// fn: the kernel for G (nullptr: no such variant), args: its parameter block
static int launch_sets(bnpp_ctx *ctx, int G, const void *fn, void *args_block, const FusedLaunch &p, const char *const names[6]);

int fused_launch(bnpp_ctx *ctx, int G, const FusedLaunch &p)
{
    fused_fn fn = nullptr;
    switch (G) {
    case 2: fn = ve_fused<2>; break;
    case 4: fn = ve_fused<4>; break;
    case 8: fn = ve_fused<8>; break;
    case 16: fn = ve_fused<16>; break;
    case 32: fn = ve_fused<32>; break;
    case 128: fn = ve_fused<128>; break;
    default: break;
    }
    static const char *const names[6] = {"ve_fused<G=2>", "ve_fused<G=4>", "ve_fused<G=8>", "ve_fused<G=16>", "ve_fused<G=32>", "ve_fused<G=128>"};
    return launch_sets(ctx, G, reinterpret_cast<const void *>(fn), const_cast<FusedLaunch *>(&p), p, names);
}

int fused_max_launch(bnpp_ctx *ctx, int G, const FusedMaxLaunch &p)
{
    fused_max_fn fn = nullptr;
    switch (G) {
    case 2: fn = ve_fused_max<2>; break;
    case 4: fn = ve_fused_max<4>; break;
    case 8: fn = ve_fused_max<8>; break;
    case 16: fn = ve_fused_max<16>; break;
    case 32: fn = ve_fused_max<32>; break;
    case 128: fn = ve_fused_max<128>; break;
    default: break;
    }
    static const char *const names[6] = {"ve_fused_max<G=2>", "ve_fused_max<G=4>", "ve_fused_max<G=8>", "ve_fused_max<G=16>",
                                         "ve_fused_max<G=32>", "ve_fused_max<G=128>"};
    return launch_sets(ctx, G, reinterpret_cast<const void *>(fn), const_cast<FusedMaxLaunch *>(&p), p.f, names);
}

int fused_mixed_launch(bnpp_ctx *ctx, int G, const FusedMaxLaunch &p)
{
    fused_max_fn fn = nullptr;
    switch (G) {
    case 2: fn = ve_fused_mixed<2>; break;
    case 4: fn = ve_fused_mixed<4>; break;
    case 8: fn = ve_fused_mixed<8>; break;
    case 16: fn = ve_fused_mixed<16>; break;
    case 32: fn = ve_fused_mixed<32>; break;
    case 128: fn = ve_fused_mixed<128>; break;
    default: break;
    }
    static const char *const names[6] = {"ve_fused_mixed<G=2>", "ve_fused_mixed<G=4>", "ve_fused_mixed<G=8>", "ve_fused_mixed<G=16>",
                                         "ve_fused_mixed<G=32>", "ve_fused_mixed<G=128>"};
    return launch_sets(ctx, G, reinterpret_cast<const void *>(fn), const_cast<FusedMaxLaunch *>(&p), p.f, names);
}

static int launch_sets(bnpp_ctx *ctx, int G, const void *fn, void *args_block, const FusedLaunch &p, const char *const names[6])
{
    if (!fn) return fail(ctx, BNPP_EINVAL, "fused VE: lanes per set must be 8, 16, 32 or 128");
    if (p.arena & 1u) return fail(ctx, BNPP_EINVAL, "fused VE: the arena of a set must be an even number of doubles");
    const size_t smem = fused_smem_bytes(G, p.arena);
    {
        static std::map<std::pair<int, const void *>, size_t> granted;      // dynamic shared memory opted into, per device and variant
        static std::mutex mu;
        std::lock_guard<std::mutex> lock(mu);
        size_t &have = granted[{ctx->device, reinterpret_cast<const void *>(fn)}];
        if (smem > have) {
            BNPP_CUDA(ctx, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            have = smem;
        }
    }
    int per_sm = 0;
    BNPP_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kFusedThreads, smem));
    if (per_sm < 1) return fail(ctx, BNPP_ETOOBIG, "fused VE: the arena of one CTA does not fit in shared memory");
    if (const char *e = getenv("BNPP_FUSED_CTAS_PER_SM"))      // experiments: cap the resident CTAs per SM
        if (atoi(e) > 0 && atoi(e) < per_sm) per_sm = atoi(e);
    const uint32_t spc = kFusedThreads / G;
    uint64_t blocks = ((uint64_t)p.nb + spc - 1) / spc;
    const uint64_t resident = (uint64_t)ctx->sm_count * per_sm;
    if (blocks > resident) blocks = resident;
    if (blocks < 1) blocks = 1;
    void *args[1] = {args_block};
    BNPP_CUDA(ctx, cudaLaunchKernel(fn, dim3((unsigned)blocks), dim3(kFusedThreads), args, smem, ctx->stream));
    ctx->launches++;
    ctx->last_desc = nullptr;
    ctx->last_kernel = names[G == 2 ? 0 : G == 4 ? 1 : G == 8 ? 2 : G == 16 ? 3 : G == 32 ? 4 : 5];
    ctx->last_grid = (uint32_t)blocks;
    ctx->last_block = kFusedThreads;
    return BNPP_OK;
}

}  // namespace bnpp

namespace bnpp {

const void *tasks_kernel() { return reinterpret_cast<const void *>(ve_tasks); }

// grid and dynamic shared memory of a ve_tasks launch over n_tasks programs whose largest arena is `arena` doubles
int tasks_geometry(bnpp_ctx *ctx, uint32_t n_tasks, uint32_t arena, unsigned *grid, unsigned *smem)
{
    const size_t bytes = fused_smem_bytes(128, arena);
    {
        static std::map<std::pair<int, const void *>, size_t> granted;
        static std::mutex mu;
        std::lock_guard<std::mutex> lock(mu);
        size_t &have = granted[{ctx->device, tasks_kernel()}];
        if (bytes > have) {
            BNPP_CUDA(ctx, cudaFuncSetAttribute(ve_tasks, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
            have = bytes;
        }
    }
    int per_sm = 0;
    BNPP_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ve_tasks, kFusedThreads, bytes));
    if (per_sm < 1) return fail(ctx, BNPP_ETOOBIG, "task launch: the arena of one task does not fit in shared memory");
    uint64_t blocks = n_tasks;
    const uint64_t resident = (uint64_t)ctx->sm_count * per_sm;
    if (blocks > resident) blocks = resident;
    if (blocks < 1) blocks = 1;
    *grid = (unsigned)blocks;
    *smem = (unsigned)bytes;
    return BNPP_OK;
}

int tasks_launch(bnpp_ctx *ctx, const TaskLaunch &p, unsigned grid, unsigned smem)
{
    void *args[1] = {const_cast<TaskLaunch *>(&p)};
    BNPP_CUDA(ctx, cudaLaunchKernel(tasks_kernel(), dim3(grid), dim3(kFusedThreads), args, smem, ctx->stream));
    ctx->launches++;
    ctx->last_desc = nullptr;
    ctx->last_kernel = "ve_tasks";
    ctx->last_grid = grid;
    ctx->last_block = kFusedThreads;
    return BNPP_OK;
}

}  // namespace bnpp
