// K1/K2/K3/K4 -- the fused elimination-step kernel and its host-side plan.
//
//   out[o] = sum_{x < card(X)}  prod_k  F_k[ pi_k(o, x) ]        Z = sum_o out[o]
//
// replaces `prod *= *pf` over a bucket followed by `prod.sum_out(var)`
// (reference code/model.cpp:414-418, code/factor.cpp:117-147 and :182-212) without
// materialising the product table.  Factor::product / divide / sum_out / conditioning
// are the k=2 / k=1 special cases of the same kernel.
//
// Where the reference walks an odometer and does two hash lookups per scope variable
// per entry (code/domain.cpp:113-123,162-179), the plan below turns every operand
// into a stride vector over the OUTPUT's axes (stride 0 = axis absent = broadcast,
// SURVEY A.1) and the kernel recovers operand offsets from its linear item index:
//   * all extents powers of two (binary variables: every BASELINE config): offsets are
//     sums of bit-fields of the index, merged per operand;
//   * otherwise: mixed-radix digits by multiply-high division over merged axes.
// The ITERATION order is chosen by the plan, not dictated by the output layout: above a
// tile of the output's fastest axes, axes that a large operand lacks are iterated
// fastest, so that operand's tile is re-read from L2 instead of HBM.
// Each thread owns U items; an item is a [V x C] micro-tile: V (1 or 2) consecutive
// output entries times the C values of the eliminated variable, loaded with 128/256-bit
// accesses whenever the operand's layout makes them contiguous.  HBM-bound: algorithmic
// bytes per launch = 8 * (sum_k #F_k + #out)   (SURVEY §8d).
//
// Arithmetic is written with __dmul_rn/__dadd_rn (no FMA contraction) so every entry is
// bit-identical to the reference's `((1*f1)*f2)*...` then `0 + p(x=0) + p(x=1) + ...`.
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <tuple>
#include <vector>

#include "common.cuh"
#include "contract.hpp"
#include "contract_mv.hpp"

namespace bnpp {

// How the [V x C] micro-tile of one operand sits in memory.  A class fixes the LOADS
// (issued for all operands of all U items before anything consumes them) and the
// index map used later to pick micro-tile element (j, x) out of the loaded registers.
enum LoadClass : uint8_t {
    LC_BCAST = 0,   // one 8-byte load, same value for the whole micro-tile
    LC_VX,          // x contiguous (stride 1, C == 2): a 16-byte load per output entry      -> r[2j+x]
    LC_VX_B,        //   ... operand does not depend on the innermost output axis             -> r[x]
    LC_VL,          // innermost output axis contiguous (V == 2): a 16-byte load per x         -> r[2x+j]
    LC_VL_B,        //   ... operand does not depend on x                                     -> r[j]
    LC_V4,          // [j][x] contiguous: one 32-byte load                                    -> r[2j+x]
    LC_V4T,         // [x][j] contiguous: one 32-byte load                                    -> r[2x+j]
    LC_S_X,         // two 8-byte loads along x                                               -> r[x]
    LC_S_L,         // two 8-byte loads along the innermost output axis                       -> r[j]
    LC_S_JX,        // four 8-byte loads                                                      -> r[2j+x]
};

template <int K>
__device__ __forceinline__ void decompose(const ParamsMR &p, uint32_t item, uint32_t (&off)[K], uint32_t &ooff)
{
#pragma unroll
    for (int k = 0; k < K; ++k) off[k] = 0;
    ooff = 0;
    uint32_t rem = item;
    for (int a = (int)p.R - 1; a > 0; --a) {
        const uint32_t q = fastdiv(rem, p.div[a]);
        const uint32_t d = rem - q * p.div[a].d;
        rem = q;
#pragma unroll
        for (int k = 0; k < K; ++k) off[k] += d * p.s[k][a];
        ooff += d * p.so[a];
    }
    if (p.R > 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) off[k] += rem * p.s[k][0];
        ooff += rem * p.so[0];
    }
}

template <int K>
__device__ __forceinline__ void decompose(const ParamsP2 &p, uint32_t item, uint32_t (&off)[K], uint32_t &ooff)
{
#pragma unroll
    for (int k = 0; k < K; ++k) {
        uint32_t o = 0;
        for (int f = 0; f < (int)p.nf[k]; ++f) o += ((item >> p.f[k][f].sh) & p.f[k][f].mask) * p.f[k][f].mul;
        off[k] = o;
    }
    uint32_t o = 0;
    for (int f = 0; f < (int)p.nf[K]; ++f) o += ((item >> p.f[K][f].sh) & p.f[K][f].mask) * p.f[K][f].mul;
    ooff = o;
}

template <int C, int V>
__device__ __forceinline__ void issue_loads(const double *__restrict__ p, uint32_t sx, uint32_t sl, uint8_t cls,
                                            double (&r)[4])
{
    switch (cls) {
    case LC_BCAST:
        r[0] = ld1(p);
        break;
    case LC_VX_B:
    case LC_VL_B: {
        const double2 a = ld2(p);
        r[0] = a.x; r[1] = a.y;
        break;
    }
    case LC_VX: {
        const double2 a = ld2(p), b = ld2(p + sl);
        r[0] = a.x; r[1] = a.y; r[2] = b.x; r[3] = b.y;
        break;
    }
    case LC_VL: {
        const double2 a = ld2(p), b = ld2(p + sx);
        r[0] = a.x; r[1] = a.y; r[2] = b.x; r[3] = b.y;
        break;
    }
    case LC_V4:
    case LC_V4T: {
        const double4_t a = ld4(p);
        r[0] = a.x; r[1] = a.y; r[2] = a.z; r[3] = a.w;
        break;
    }
    case LC_S_X:
        r[0] = ld1(p); r[1] = ld1(p + sx);
        break;
    case LC_S_L:
        r[0] = ld1(p); r[1] = ld1(p + sl);
        break;
    default:
        r[0] = ld1(p); r[1] = ld1(p + sx); r[2] = ld1(p + sl); r[3] = ld1(p + sl + sx);
        break;
    }
}

// element (j, x) of the micro-tile; j and x are compile-time, cls is grid-uniform
__device__ __forceinline__ double pick(const double (&r)[4], uint8_t cls, int j, int x)
{
    switch (cls) {
    case LC_BCAST: return r[0];
    case LC_VX_B:
    case LC_S_X: return r[x];
    case LC_VL_B:
    case LC_S_L: return r[j];
    case LC_VL:
    case LC_V4T: return r[2 * x + j];
    default: return r[2 * j + x];
    }
}

// ---- per-operand dispatch hoisted over the thread's U items -----------------------------------
// One switch per operand and phase (not per element): phase 1 issues the loads of all U items of
// operand k inside the case of its class; phase 2 multiplies the accumulators IN PLACE inside
// the case, so no loaded value is ever copied or selected at run time.
template <int C, int V, int U>
__device__ __forceinline__ void issue_loads_all(const double *__restrict__ base, const uint32_t (&off)[U], uint32_t sx,
                                                uint32_t sl, uint8_t cls, double (&r)[U][4])
{
    switch (cls) {
    case LC_BCAST:
#pragma unroll
        for (int u = 0; u < U; ++u) r[u][0] = ld1(base + off[u]);
        break;
    case LC_VX_B:
    case LC_VL_B:
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const double2 a = ld2(base + off[u]);
            r[u][0] = a.x; r[u][1] = a.y;
        }
        break;
    case LC_VX:
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const double2 a = ld2(base + off[u]), b = ld2(base + off[u] + sl);
            r[u][0] = a.x; r[u][1] = a.y; r[u][2] = b.x; r[u][3] = b.y;
        }
        break;
    case LC_VL:
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const double2 a = ld2(base + off[u]), b = ld2(base + off[u] + sx);
            r[u][0] = a.x; r[u][1] = a.y; r[u][2] = b.x; r[u][3] = b.y;
        }
        break;
    case LC_V4:
    case LC_V4T:
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const double4_t a = ld4(base + off[u]);
            r[u][0] = a.x; r[u][1] = a.y; r[u][2] = a.z; r[u][3] = a.w;
        }
        break;
    case LC_S_X:
#pragma unroll
        for (int u = 0; u < U; ++u) { r[u][0] = ld1(base + off[u]); r[u][1] = ld1(base + off[u] + sx); }
        break;
    case LC_S_L:
#pragma unroll
        for (int u = 0; u < U; ++u) { r[u][0] = ld1(base + off[u]); r[u][1] = ld1(base + off[u] + sl); }
        break;
    default:
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const double *q = base + off[u];
            r[u][0] = ld1(q); r[u][1] = ld1(q + sx); r[u][2] = ld1(q + sl); r[u][3] = ld1(q + sl + sx);
        }
        break;
    }
}

// acc[u][j][x] (op)= element (j, x) of operand k's micro-tile;  IDX: 0 -> r[0], 1 -> r[x], 2 -> r[j], 3 -> r[2x+j], 4 -> r[2j+x]
template <int C, int V, int U, bool FIRST, bool DIV, int IDX>
__device__ __forceinline__ void apply_idx(const double (&r)[U][4], double (&acc)[U][V][C], bool &zero_div)
{
#pragma unroll
    for (int u = 0; u < U; ++u)
#pragma unroll
        for (int j = 0; j < V; ++j)
#pragma unroll
            for (int x = 0; x < C; ++x) {
                const int e = IDX == 0 ? 0 : (IDX == 1 ? x : (IDX == 2 ? j : (IDX == 3 ? 2 * x + j : 2 * j + x)));
                const double t = r[u][e];
                if (FIRST) acc[u][j][x] = t;
                else if (DIV) { zero_div |= (t == 0.0); acc[u][j][x] = __ddiv_rn(acc[u][j][x], t); }
                else acc[u][j][x] = __dmul_rn(acc[u][j][x], t);
            }
}

template <int C, int V, int U, bool FIRST, bool DIV>
__device__ __forceinline__ void apply_all(const double (&r)[U][4], uint8_t cls, double (&acc)[U][V][C], bool &zero_div)
{
    switch (cls) {
    case LC_BCAST: apply_idx<C, V, U, FIRST, DIV, 0>(r, acc, zero_div); break;
    case LC_VX_B:
    case LC_S_X: apply_idx<C, V, U, FIRST, DIV, 1>(r, acc, zero_div); break;
    case LC_VL_B:
    case LC_S_L: apply_idx<C, V, U, FIRST, DIV, 2>(r, acc, zero_div); break;
    case LC_VL:
    case LC_V4T: apply_idx<C, V, U, FIRST, DIV, 3>(r, acc, zero_div); break;
    default: apply_idx<C, V, U, FIRST, DIV, 4>(r, acc, zero_div); break;
    }
}

template <int K, int C, int V, int U, bool DIV, int k0 = 0>
struct ApplyOperands {
    static __device__ __forceinline__ void run(const double (&raw)[K][U][4], const uint8_t *cls, double (&acc)[U][V][C],
                                               bool &zero_div, int skip)
    {
        if (k0 != skip) apply_all<C, V, U, k0 == 0, DIV>(raw[k0], cls[k0], acc, zero_div);
        ApplyOperands<K, C, V, U, DIV, k0 + 1>::run(raw, cls, acc, zero_div, skip);
    }
};
template <int K, int C, int V, int U, bool DIV>
struct ApplyOperands<K, C, V, U, DIV, K> {
    static __device__ __forceinline__ void run(const double (&)[K][U][4], const uint8_t *, double (&)[U][V][C], bool &, int) {}
};

template <int K, int C, int V, int U, int k0 = 0>
struct ApplyOperandsStaged {
    static __device__ __forceinline__ void run(const double (&raw)[K][U][4], const uint8_t *cls, double (&acc)[U][V][C],
                                               bool &zero_div, int skip)
    {
        if (k0 != skip) apply_all<C, V, U, false, false>(raw[k0], cls[k0], acc, zero_div);
        ApplyOperandsStaged<K, C, V, U, k0 + 1>::run(raw, cls, acc, zero_div, skip);
    }
};
template <int K, int C, int V, int U>
struct ApplyOperandsStaged<K, C, V, U, K> {
    static __device__ __forceinline__ void run(const double (&)[K][U][4], const uint8_t *, double (&)[U][V][C], bool &, int) {}
};

// Fast path: eliminated variable binary (C = 2) or absent (C = 1).  Each CTA walks
// chunks of U * kBlock consecutive items.  Phase 1 issues the loads of all K operands of
// all U items of a thread back to back; nothing reads a loaded register until phase 2,
// so U * K requests per thread are in flight -- that, not occupancy, is what feeds HBM.
template <class P, int K, int C, int V, int U, bool DIV>
__global__ void __launch_bounds__(kBlock) contract_fast(const __grid_constant__ P p)
{
    const ParamsHead &h = p.h;
    const uint64_t chunk = (uint64_t)U * kBlock;
    const uint64_t step = (uint64_t)gridDim.x * chunk;
    const uint64_t last = h.n_items - 1;
    double zacc = 0.0;
    bool zero_div = false;
    for (uint64_t base = (uint64_t)blockIdx.x * chunk + threadIdx.x; base < h.n_items; base += step) {
        double raw[U][K][4];
        uint32_t ooff[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint64_t it = base + (uint64_t)u * kBlock;
            uint32_t off[K];
            decompose<K>(p, (uint32_t)(it < last ? it : last), off, ooff[u]);   // tail items clamp, their result is dropped
#pragma unroll
            for (int k = 0; k < K; ++k) {
#pragma unroll
                for (int e = 0; e < 4; ++e) raw[u][k][e] = 0.0;
                issue_loads<C, V>(h.in[k] + off[k], h.sx[k], h.sl[k], h.cls[k], raw[u][k]);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            double r[V];
#pragma unroll
            for (int j = 0; j < V; ++j) {
#pragma unroll
                for (int x = 0; x < C; ++x) {
                    double a = pick(raw[u][0], h.cls[0], j, x);
#pragma unroll
                    for (int k = 1; k < K; ++k) {
                        const double t = pick(raw[u][k], h.cls[k], j, x);
                        if (DIV) { zero_div |= (t == 0.0); a = __ddiv_rn(a, t); }
                        else a = __dmul_rn(a, t);
                    }
                    r[j] = (x == 0) ? a : __dadd_rn(r[j], a);
                }
            }
            if (base + (uint64_t)u * kBlock > last) continue;
            double *o = h.out + ooff[u];
            if (V == 2) {
                zacc = __dadd_rn(zacc, __dadd_rn(r[0], r[V - 1]));
                if (h.out_vec) *reinterpret_cast<double2 *>(o) = make_double2(r[0], r[V - 1]);
                else { o[0] = r[0]; o[h.sol] = r[V - 1]; }
            } else {
                zacc = __dadd_rn(zacc, r[0]);
                o[0] = r[0];
            }
        }
    }
    if (DIV && zero_div) atomicOr(h.status, BNPP_STATUS_ZERO_DIVISOR);
    if (h.z) grid_sum_to(zacc, h.partials, h.ticket, h.z);   // grid-uniform: intermediates of a VE plan need no partition
}

// Power-of-two iteration space, the hot variant.  A CTA owns chunks of CH = U * kBlock
// consecutive items (CH a power of two, dividing n_items).  Because offsets are sums of
// bit-fields of the item index and  item = chunk_base + (u * kBlock + tid)  has disjoint
// bits in its two terms,  off(item) = off(chunk_base) + off(u * kBlock + tid)  exactly:
// the second term is loop-invariant per thread, the first is computed once per chunk
// (uniform over the CTA) and shared by the U items -- U-fold less index arithmetic.
template <int K, int C, int V, int U, bool DIV>
__global__ void __launch_bounds__(kBlock) contract_fast_p2s(const __grid_constant__ ParamsP2 p)
{
    const ParamsHead &h = p.h;
    constexpr uint32_t CH = U * kBlock;
    uint32_t lo[U][K], olo[U];
#pragma unroll
    for (int u = 0; u < U; ++u) decompose<K>(p, threadIdx.x + u * kBlock, lo[u], olo[u]);
    const uint32_t n_chunks = (uint32_t)(h.n_items / CH);
    double zacc = 0.0;
    bool zero_div = false;
    for (uint32_t c = blockIdx.x; c < n_chunks; c += gridDim.x) {
        uint32_t hi[K], ohi;
        decompose<K>(p, c * CH, hi, ohi);
        double raw[K][U][4];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            uint32_t off[U];
#pragma unroll
            for (int u = 0; u < U; ++u) off[u] = hi[k] + lo[u][k];
            issue_loads_all<C, V, U>(h.in[k], off, h.sx[k], h.sl[k], h.cls[k], raw[k]);
        }
        double acc[U][V][C];
        ApplyOperands<K, C, V, U, DIV>::run(raw, h.cls, acc, zero_div, -1);
#pragma unroll
        for (int u = 0; u < U; ++u) {
            double r[V];
#pragma unroll
            for (int j = 0; j < V; ++j) {
                r[j] = acc[u][j][0];
#pragma unroll
                for (int x = 1; x < C; ++x) r[j] = __dadd_rn(r[j], acc[u][j][x]);
            }
            double *o = h.out + (ohi + olo[u]);
            if (V == 2) {
                zacc = __dadd_rn(zacc, __dadd_rn(r[0], r[V - 1]));
                if (h.out_vec) *reinterpret_cast<double2 *>(o) = make_double2(r[0], r[V - 1]);
                else { o[0] = r[0]; o[h.sol] = r[V - 1]; }
            } else {
                zacc = __dadd_rn(zacc, r[0]);
                o[0] = r[0];
            }
        }
    }
    if (DIV && zero_div) atomicOr(h.status, BNPP_STATUS_ZERO_DIVISOR);
    if (h.z) grid_sum_to(zacc, h.partials, h.ticket, h.z);   // grid-uniform: intermediates of a VE plan need no partition
}

// The variable-elimination hot variant.  With the canonical axis order of ve.cu every
// operand of a bucket has the eliminated (binary) variable as its fastest axis, so an
// operand's micro-tile is either 4 contiguous doubles (it also has the output's fastest
// axis: one 32-byte load) or 2 contiguous doubles shared by both output entries (one
// 16-byte load).  Which of the two is a compile-time bit of MASK: no class dispatch, no
// register shuffling -- per item K loads, 4(K-1) multiplies, 2+1 adds, one 16-byte store.
// INVK >= 0 names an operand that does not depend on the two axes the plan placed at the
// thread's unroll bits: its micro-tile is loaded once and reused for all U items.
// MAX: max-product instead -- r = the product at x = 0, replaced by x = 1's only if strictly
// greater (ties keep the lower x, a NaN never replaces a number); the two argmax bytes of an
// item go out as one 16-bit store at the (even) output index; no Z.
template <int K, unsigned MASK, int U, int INVK, bool MAX = false>
__global__ void __launch_bounds__(kBlock) contract_canon(const __grid_constant__ ParamsP2 p)
{
    const ParamsHead &h = p.h;
    constexpr uint32_t CH = U * kBlock;
    uint32_t lo[U][K], olo[U];
#pragma unroll
    for (int u = 0; u < U; ++u) decompose<K>(p, threadIdx.x + u * kBlock, lo[u], olo[u]);
    const uint32_t n_chunks = (uint32_t)(h.n_items / CH);
    double zacc = 0.0;
    for (uint32_t c = blockIdx.x; c < n_chunks; c += gridDim.x) {
        uint32_t hi[K], ohi;
        decompose<K>(p, c * CH, hi, ohi);
        double4_t t[U][K];
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int k = 0; k < K; ++k) {
                if (k == INVK && u > 0) continue;   // same element for all U items: loaded once, kept in registers
                const double *src = h.in[k] + (hi[k] + lo[u][k]);
                if ((MASK >> k) & 1u) {
                    t[u][k] = ld4(src);
                } else {
                    const double2 v = ld2(src);
                    t[u][k].x = v.x; t[u][k].y = v.y; t[u][k].z = v.x; t[u][k].w = v.y;
                }
            }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const double4_t &t0 = t[INVK == 0 ? 0 : u][0];
            double a = t0.x, b = t0.y, cc = t0.z, d = t0.w;
#pragma unroll
            for (int k = 1; k < K; ++k) {
                const double4_t &tk = t[INVK == k ? 0 : u][k];
                a = __dmul_rn(a, tk.x);
                b = __dmul_rn(b, tk.y);
                cc = __dmul_rn(cc, tk.z);
                d = __dmul_rn(d, tk.w);
            }
            if (MAX) {
                const bool x0 = b > a, x1 = d > cc;
                const uint32_t o = ohi + olo[u];
                *reinterpret_cast<double2 *>(h.out + o) = make_double2(x0 ? b : a, x1 ? d : cc);
                *reinterpret_cast<uint16_t *>(h.arg + o) = (uint16_t)((uint32_t)x0 | ((uint32_t)x1 << 8));
                continue;
            }
            const double r0 = __dadd_rn(a, b), r1 = __dadd_rn(cc, d);
            zacc = __dadd_rn(zacc, __dadd_rn(r0, r1));
            *reinterpret_cast<double2 *>(h.out + (ohi + olo[u])) = make_double2(r0, r1);
        }
    }
    if (!MAX && h.z) grid_sum_to(zacc, h.partials, h.ticket, h.z);   // grid-uniform: intermediates of a VE plan need no partition
}

// Transposing variant: operand `st.sk` comes through a shared-memory tile (see StageInfo).
// The plan puts the output's 6 fastest bits on the lanes (coalesced 512-byte rows for the
// output and the well laid-out operands) and the staged operand's fastest axes on the
// remaining chunk bits, so the tile is a few contiguous runs of that operand.  Slots are
// XOR-swizzled with the slot bits the lanes differ in, so a warp reads 32 distinct banks.
template <int K, int C>
__global__ void __launch_bounds__(kBlock, 2) contract_staged(const __grid_constant__ ParamsP2S ps)
{
    constexpr int U = 4, V = 2;
    constexpr uint32_t CH = U * kBlock;
    __shared__ double tile[4096];
    const ParamsP2 &p = ps.b;
    const ParamsHead &h = p.h;
    const StageInfo &st = ps.st;
    const int sk = st.sk;
    uint32_t lo[U][K], olo[U], slo[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const uint32_t local = threadIdx.x + u * kBlock;
        decompose<K>(p, local, lo[u], olo[u]);
        uint32_t sl = 0;
        for (int f = 0; f < (int)st.ncf; ++f) sl += ((local >> st.cf[f].sh) & st.cf[f].mask) * st.cf[f].mul;
        slo[u] = sl;
    }
    // Tile entry `slot = tid + 256 * i` lives at operand offset scatter(tid) + scatter(256 * i)
    // (disjoint bits): the first term is this thread's, the second is shared by the CTA.
    __shared__ uint32_t s_off[16], s_off2[8];
    uint32_t my_off = 0, my_off2 = 0;
    for (int f = 0; f < (int)st.nlf; ++f) {
        my_off += ((threadIdx.x >> st.lf[f].sh) & st.lf[f].mask) * st.lf[f].mul;
        my_off2 += (((2u * threadIdx.x) >> st.lf[f].sh) & st.lf[f].mask) * st.lf[f].mul;      // pair copies: slot 2 * tid
    }
    if (threadIdx.x < 16) {
        const uint32_t slot = threadIdx.x * kBlock;
        uint32_t o = 0, o2 = 0;
        for (int f = 0; f < (int)st.nlf; ++f) {
            o += ((slot >> st.lf[f].sh) & st.lf[f].mask) * st.lf[f].mul;
            o2 += (((2u * slot) >> st.lf[f].sh) & st.lf[f].mask) * st.lf[f].mul;                  // pair copies: block of 512 slots
        }
        s_off[threadIdx.x] = o;
        if (threadIdx.x < 8) s_off2[threadIdx.x] = o2;
    }
    __syncthreads();
    const uint32_t n_copy = (st.tile + kBlock - 1) / kBlock;
    const uint32_t tile_base = (uint32_t)__cvta_generic_to_shared(tile);
    const uint32_t n_chunks = (uint32_t)(h.n_items / CH);
    double zacc = 0.0;
    // the chunk's base offsets are the same for the whole CTA and, for a transposed operand, a sum over two dozen
    // one-bit fields: computed one chunk ahead, the CTA reads them after the barrier that ends the previous chunk
    __shared__ uint32_t s_hi[2][kMaxK + 1];
    // warp w <= K owns operand w (warp K the output), lane f its bit-field f: one warp-wide integer add per chunk
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    Field mine = Field{0u, 0u, 0u};
    if (warp <= (uint32_t)K && lane < p.nf[warp]) mine = p.f[warp][lane];
    auto chunk_base = [&](uint32_t c, uint32_t *dst) {
        if (warp <= (uint32_t)K) {
            const uint32_t o = __reduce_add_sync(0xffffffffu, (((c * CH) >> mine.sh) & mine.mask) * mine.mul);
            if (lane == 0) dst[warp] = o;
        }
    };
    if (blockIdx.x < n_chunks) chunk_base(blockIdx.x, s_hi[0]);
    __syncthreads();
    uint32_t buf = 0;
    for (uint32_t c = blockIdx.x; c < n_chunks; c += gridDim.x, buf ^= 1u) {
        if (c + gridDim.x < n_chunks) chunk_base(c + gridDim.x, s_hi[buf ^ 1u]);
        uint32_t hi[K], ohi;
#pragma unroll
        for (int k = 0; k < K; ++k) hi[k] = s_hi[buf][k];
        ohi = s_hi[buf][K];
        const double *src = h.in[0];
        uint32_t base = 0;
#pragma unroll
        for (int k = 0; k < K; ++k)
            if (k == sk) { src = h.in[k]; base = hi[k]; }
        const double *src2 = src + base + my_off2;
        src += base + my_off;
        // global -> shared without passing through registers (LDGSTS): 16 bytes per copy when slots 2m, 2m+1 are
        // neighbours in the operand (its stride-1 axis is slot bit 0; the swizzle leaves bit 0 alone), else 8
        if (st.pair) {
            for (uint32_t i = 0; i < n_copy; i += 2) {
                // thread t moves the pair of slots 2t, 2t+1 of every 512-slot block
                const uint32_t slot = 2u * threadIdx.x + i * kBlock;
                if (slot < st.tile) {
                    const uint32_t dst = tile_base + 8u * (slot ^ (((slot >> st.swz) & 15u) << 1));
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src2 + s_off2[i >> 1]) : "memory");
                }
            }
        } else {
            for (uint32_t i = 0; i < n_copy; ++i) {
                const uint32_t slot = threadIdx.x + i * kBlock;
                if (slot < st.tile) {
                    const uint32_t dst = tile_base + 8u * (slot ^ (((slot >> st.swz) & 15u) << 1));
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src + s_off[i]) : "memory");
                }
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        double raw[K][U][4];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            if (k == sk) continue;
            uint32_t off[U];
#pragma unroll
            for (int u = 0; u < U; ++u) off[u] = hi[k] + lo[u][k];
            issue_loads_all<C, V, U>(h.in[k], off, h.sx[k], h.sl[k], h.cls[k], raw[k]);
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        // the staged operand first (acc = its tile entries), then the others multiply in place
        double acc[U][V][C];
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int j = 0; j < V; ++j)
#pragma unroll
                for (int x = 0; x < C; ++x) {
                    const uint32_t slot = slo[u] + j * st.slot_j + x * st.slot_x;
                    acc[u][j][x] = tile[slot ^ (((slot >> st.swz) & 15u) << 1)];
                }
        bool zd = false;
        ApplyOperandsStaged<K, C, V, U>::run(raw, h.cls, acc, zd, sk);
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const double r0 = (C == 2) ? __dadd_rn(acc[u][0][0], acc[u][0][C - 1]) : acc[u][0][0];
            const double r1 = (C == 2) ? __dadd_rn(acc[u][1][0], acc[u][1][C - 1]) : acc[u][1][0];
            double *o = h.out + (ohi + olo[u]);
            zacc = __dadd_rn(zacc, __dadd_rn(r0, r1));
            if (h.out_vec) *reinterpret_cast<double2 *>(o) = make_double2(r0, r1);
            else { o[0] = r0; o[h.sol] = r1; }
        }
        __syncthreads();
    }
    if (h.z) grid_sum_to(zacc, h.partials, h.ticket, h.z);
}

// The tiles brought in by the TMA engine (see ParamsP2T): cp.async.bulk global -> shared of whole runs, one run per
// thread and operand, completion counted on the stage's mbarrier -- no per-element address arithmetic, no swizzle.  A
// ring of S stages: the copies of the next S-1 chunks are in flight while this one is consumed (without that the
// only bytes in flight are the current chunk's, and a step whose operands are all half the union table -- F-bcast --
// is latency-bound: a chunk is 48 KB, two CTAs per SM).  What a thread needs to find its entries of a tile (one
// index per item, the same for every chunk) lives in registers.  Products are taken in operand order.
template <int K, int C, int k0 = 0>
struct TmaApply {
    static constexpr int U = 4, V = 2;
    static __device__ __forceinline__ void run(const double *stage, const uint32_t (&idx)[U][K], const TmaOperand *t, uint32_t mask,
                                               const double (&raw)[K][U][4], const uint8_t *cls, double (&acc)[U][V][C], bool &zd)
    {
        if ((mask >> k0) & 1u) {
            const uint32_t dj = t[k0].dj, dx = t[k0].dx;
#pragma unroll
            for (int u = 0; u < U; ++u)
#pragma unroll
                for (int j = 0; j < V; ++j)
#pragma unroll
                    for (int x = 0; x < C; ++x) {
                        const double v = stage[idx[u][k0] + j * dj + x * dx];
                        acc[u][j][x] = (k0 == 0) ? v : __dmul_rn(acc[u][j][x], v);
                    }
        } else
            apply_all<C, V, U, k0 == 0, false>(raw[k0], cls[k0], acc, zd);
        TmaApply<K, C, k0 + 1>::run(stage, idx, t, mask, raw, cls, acc, zd);
    }
};
template <int K, int C>
struct TmaApply<K, C, K> {
    static __device__ __forceinline__ void run(const double *, const uint32_t (&)[4][K], const TmaOperand *, uint32_t,
                                               const double (&)[K][4][4], const uint8_t *, double (&)[4][2][C], bool &) {}
};

template <int K, int C>
__global__ void __launch_bounds__(kBlock, 2) contract_staged_tma(const __grid_constant__ ParamsP2T pt)
{
    constexpr int U = 4, V = 2;
    constexpr uint32_t CH = U * kBlock;
    extern __shared__ __align__(16) double stages[];        // [S][stage_doubles]
    __shared__ __align__(8) uint64_t s_full[kStagedMaxStages];
    __shared__ uint32_t s_hi[4][kMaxK + 1];                 // chunk bases, a ring over the chunks in flight
    const ParamsP2 &p = pt.b;
    const ParamsHead &h = p.h;
    const uint32_t mask = pt.mask;
    const uint32_t S = pt.stages, D = S - 1u;
    auto run_pos = [](const TmaOperand &t, uint32_t r) {
        uint32_t o = 0;
        for (int i = 0; i < (int)t.nrb; ++i) o |= ((r >> i) & 1u) << t.rpos[i];
        return o;
    };
    // idx[u][k]: shared-memory index of item u's entry (V bit and x at 0) for a staged operand, else its offset inside the chunk
    uint32_t idx[U][K], olo[U], run_off[K], run_dst[K];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const uint32_t local = threadIdx.x + u * kBlock;
        decompose<K>(p, local, idx[u], olo[u]);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            if (!((mask >> k) & 1u)) continue;
            const TmaOperand &t = pt.t[k];
            uint32_t sl = 0;
            for (int f = 0; f < (int)t.ncf; ++f) sl += ((local >> t.cf[f].sh) & t.cf[f].mask) * t.cf[f].mul;
            idx[u][k] = t.off + run_pos(t, sl >> t.rbits) * ((1u << t.rbits) + 2u) + (sl & ((1u << t.rbits) - 1u));
        }
    }
    // A bulk copy is a warp-uniform instruction: a warp issues the copies of its lanes one after the other (about ten
    // issue slots each), so runs are dealt round-robin over the WARPS -- this thread moves run `my_run` of every staged
    // operand's tile; run_off: where that run starts in the operand, relative to the chunk's base
    const uint32_t my_run = (threadIdx.x & 31u) * (kBlock / 32) + (threadIdx.x >> 5);
#pragma unroll
    for (int k = 0; k < K; ++k) {
        run_off[k] = run_dst[k] = 0;
        if (!((mask >> k) & 1u)) continue;
        const TmaOperand &t = pt.t[k];
        for (int f = 1; f < (int)t.nlf; ++f) run_off[k] += (((my_run << t.rbits) >> t.lf[f].sh) & t.lf[f].mask) * t.lf[f].mul;
        run_dst[k] = t.off + run_pos(t, my_run) * ((1u << t.rbits) + 2u);
    }
    const uint32_t bar0 = (uint32_t)__cvta_generic_to_shared(&s_full[0]);
    const uint32_t stage0 = (uint32_t)__cvta_generic_to_shared(stages);
    if (threadIdx.x == 0) {
        for (uint32_t s = 0; s < S; ++s) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0 + 8u * s) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    const uint32_t n_chunks = (uint32_t)(h.n_items / CH);
    // A chunk's base offsets are sums over up to two dozen bit-fields of the chunk index (a transposed operand has
    // one field per variable).  Warp w <= K owns operand w (warp K the output), lane f its field f: one shift-mask-
    // multiply per lane and a warp-wide integer add -- a serial loop here would keep the CTA waiting at the barrier.
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    Field mine = Field{0u, 0u, 0u};
    if (warp <= (uint32_t)K && lane < p.nf[warp]) mine = p.f[warp][lane];
    auto chunk_base = [&](uint32_t c, uint32_t *dst) {
        if (warp <= (uint32_t)K && c < n_chunks) {
            const uint32_t o = __reduce_add_sync(0xffffffffu, (((c * CH) >> mine.sh) & mine.mask) * mine.mul);
            if (lane == 0) dst[warp] = o;
        }
    };
    // the copies of chunk c into stage s: thread 0 announces the bytes, every thread moves its run of every staged operand
    auto fetch = [&](uint32_t c, const uint32_t *hi, uint32_t s) {
        if (c >= n_chunks) return;
        const uint32_t bar = bar0 + 8u * s;
        if (threadIdx.x == 0)
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(pt.stage_bytes) : "memory");
#pragma unroll
        for (int k = 0; k < K; ++k) {
            if (!((mask >> k) & 1u)) continue;
            const TmaOperand &t = pt.t[k];
            if (my_run < (t.tile >> t.rbits)) {
                const double *src = h.in[k] + (hi[k] + run_off[k]);
                const uint32_t dst = stage0 + 8u * (s * pt.stage_doubles + run_dst[k]);
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(dst), "l"(src), "r"(8u << t.rbits), "r"(bar)
                             : "memory");
            }
        }
    };
    for (uint32_t d = 0; d <= D; ++d) chunk_base(blockIdx.x + d * gridDim.x, s_hi[d]);
    __syncthreads();
    for (uint32_t d = 0; d < D; ++d) fetch(blockIdx.x + d * gridDim.x, s_hi[d], d);
    double zacc = 0.0;
    uint32_t stage = 0, parity = 0, it = 0;
    for (uint32_t c = blockIdx.x; c < n_chunks; c += gridDim.x, ++it) {
        // chunk it + D goes into the stage consumed in the previous iteration; its bases were computed one iteration ago
        fetch(c + D * gridDim.x, s_hi[(it + D) & 3u], stage == 0 ? D : stage - 1u);
        chunk_base(c + (D + 1u) * gridDim.x, s_hi[(it + D + 1u) & 3u]);
        uint32_t hi[K], ohi;
#pragma unroll
        for (int k = 0; k < K; ++k) hi[k] = s_hi[it & 3u][k];
        ohi = s_hi[it & 3u][K];
        double raw[K][U][4];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            if ((mask >> k) & 1u) continue;
            uint32_t off[U];
#pragma unroll
            for (int u = 0; u < U; ++u) off[u] = hi[k] + idx[u][k];
            issue_loads_all<C, V, U>(h.in[k], off, h.sx[k], h.sl[k], h.cls[k], raw[k]);
        }
        {
            const uint32_t bar = bar0 + 8u * stage;
            asm volatile("{\n.reg .pred P1;\nSTT_WAIT:\nmbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n@P1 bra STT_DONE;\nbra STT_WAIT;\nSTT_DONE:\n}"
                         ::"r"(bar), "r"(parity)
                         : "memory");
        }
        double acc[U][V][C];
        bool zd = false;
        TmaApply<K, C>::run(stages + stage * pt.stage_doubles, idx, pt.t, mask, raw, h.cls, acc, zd);
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const double r0 = (C == 2) ? __dadd_rn(acc[u][0][0], acc[u][0][C - 1]) : acc[u][0][0];
            const double r1 = (C == 2) ? __dadd_rn(acc[u][1][0], acc[u][1][C - 1]) : acc[u][1][0];
            double *o = h.out + (ohi + olo[u]);
            zacc = __dadd_rn(zacc, __dadd_rn(r0, r1));
            if (h.out_vec) *reinterpret_cast<double2 *>(o) = make_double2(r0, r1);
            else { o[0] = r0; o[h.sol] = r1; }
        }
        __syncthreads();        // the stage is consumed (the next iteration's copies land in it); s_hi is written
        if (++stage == S) { stage = 0; parity ^= 1u; }
    }
    if (h.z) grid_sum_to(zacc, h.partials, h.ticket, h.z);
}

// Generic path: any cardinality of the eliminated variable, one output entry per item.
// MAX: max-product (the rule of contract_canon<MAX>), arg[ooff] = the first maximising x; no Z.
template <class P, int K, bool DIV, bool MAX = false>
__global__ void __launch_bounds__(kBlock) contract_generic(const __grid_constant__ P p)
{
    const ParamsHead &h = p.h;
    const uint64_t step = (uint64_t)gridDim.x * kBlock;
    double zacc = 0.0;
    bool zero_div = false;
    for (uint64_t it = (uint64_t)blockIdx.x * kBlock + threadIdx.x; it < h.n_items; it += step) {
        uint32_t off[K], ooff;
        decompose<K>(p, (uint32_t)it, off, ooff);
        double acc = 0.0;
        uint32_t best = 0;
        for (uint32_t x = 0; x < h.cx; ++x) {
            double v = ld1(h.in[0] + off[0] + x * h.sx[0]);
#pragma unroll
            for (int k = 1; k < K; ++k) {
                const double t = ld1(h.in[k] + off[k] + x * h.sx[k]);
                if (DIV) { zero_div |= (t == 0.0); v = __ddiv_rn(v, t); }
                else v = __dmul_rn(v, t);
            }
            if (!MAX) acc = __dadd_rn(acc, v);
            else if (x == 0 || v > acc) { acc = v; best = x; }
        }
        h.out[ooff] = acc;
        if (MAX) h.arg[ooff] = (uint8_t)best;
        else zacc = __dadd_rn(zacc, acc);
    }
    if (DIV && zero_div) atomicOr(h.status, BNPP_STATUS_ZERO_DIVISOR);
    if (!MAX && h.z) grid_sum_to(zacc, h.partials, h.ticket, h.z);   // grid-uniform: intermediates of a VE plan need no partition
}

// ---------------------------------------------------------------------------
// kernel selection
// ---------------------------------------------------------------------------
template <class P>
struct Launch {
    typedef void (*fn_t)(const P);

    template <int K, int U>
    static fn_t fast(int C, int V)
    {
        if (C == 1) return V == 2 ? contract_fast<P, K, 1, 2, U, false> : contract_fast<P, K, 1, 1, U, false>;
        return V == 2 ? contract_fast<P, K, 2, 2, U, false> : contract_fast<P, K, 2, 1, U, false>;
    }

    // max-product: one output entry per item, any cardinality and layout
    static fn_t pick_max(int K)
    {
        switch (K) {
        case 1: return contract_generic<P, 1, false, true>;
        case 2: return contract_generic<P, 2, false, true>;
        case 3: return contract_generic<P, 3, false, true>;
        case 4: return contract_generic<P, 4, false, true>;
        case 5: return contract_generic<P, 5, false, true>;
        default: return contract_generic<P, 6, false, true>;
        }
    }

    static fn_t pick(int K, int C, int V, bool div, bool generic, int &U)
    {
        U = 1;
        if (generic) {
            if (div) return contract_generic<P, 2, true>;
            switch (K) {
            case 1: return contract_generic<P, 1, false>;
            case 2: return contract_generic<P, 2, false>;
            case 3: return contract_generic<P, 3, false>;
            case 4: return contract_generic<P, 4, false>;
            case 5: return contract_generic<P, 5, false>;
            default: return contract_generic<P, 6, false>;
            }
        }
        if (div) {
            U = 2;
            if (C == 1) return V == 2 ? contract_fast<P, 2, 1, 2, 2, true> : contract_fast<P, 2, 1, 1, 2, true>;
            return V == 2 ? contract_fast<P, 2, 2, 2, 2, true> : contract_fast<P, 2, 2, 1, 2, true>;
        }
        // U: items in flight per thread -- fewer operands => fewer bytes per item => more items
        switch (K) {
        case 1: U = 4; return fast<1, 4>(C, V);
        case 2: U = 2; return fast<2, 2>(C, V);
        case 3: U = 2; return fast<3, 2>(C, V);
        case 4: U = 1; return fast<4, 1>(C, V);
        case 5: U = 1; return fast<5, 1>(C, V);
        default: U = 1; return fast<6, 1>(C, V);
        }
    }
};

// ---------------------------------------------------------------------------
// host-side plan
// ---------------------------------------------------------------------------
struct Axis {
    uint32_t ext;
    uint64_t so;
    uint64_t s[kMaxK];
    uint64_t miss;   // bytes of large operands that do NOT depend on this axis
};

static bool aligned(const void *p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }
static bool is_pow2(uint32_t v) { return v && !(v & (v - 1)); }
static uint32_t ilog2(uint32_t v) { uint32_t l = 0; while ((1u << l) < v) ++l; return l; }

constexpr uint64_t kTileOutputs = 1u << 13;     // the output's fastest axes covering this many entries keep their order
constexpr uint64_t kReuseBytes = 32ull << 20;   // operands above this do not survive in L2 between passes

typedef void (*p2s_fn)(const ParamsP2);

constexpr int kCanonU = 4;

template <int K, unsigned MASK, bool MAX>
static p2s_fn canon_inv(int invk)
{
    switch (invk) {
    case 0: return contract_canon<K, MASK, kCanonU, 0, MAX>;
    case 1: return K > 1 ? contract_canon<K, MASK, kCanonU, (K > 1 ? 1 : -1), MAX> : nullptr;
    case 2: return K > 2 ? contract_canon<K, MASK, kCanonU, (K > 2 ? 2 : -1), MAX> : nullptr;
    default: return contract_canon<K, MASK, kCanonU, -1, MAX>;
    }
}

template <int K, unsigned MASK>
static p2s_fn canon_inv(int invk, bool max)
{
    return max ? canon_inv<K, MASK, true>(invk) : canon_inv<K, MASK, false>(invk);
}

static p2s_fn pick_canon(int K, unsigned mask, int invk, bool max)
{
    switch (K * 8 + (int)mask) {
    case 1 * 8 + 0: return canon_inv<1, 0>(-1, max);
    case 1 * 8 + 1: return canon_inv<1, 1>(-1, max);
    case 2 * 8 + 0: return canon_inv<2, 0>(invk, max);
    case 2 * 8 + 1: return canon_inv<2, 1>(invk, max);
    case 2 * 8 + 2: return canon_inv<2, 2>(invk, max);
    case 2 * 8 + 3: return canon_inv<2, 3>(invk, max);
    case 3 * 8 + 0: return canon_inv<3, 0>(invk, max);
    case 3 * 8 + 1: return canon_inv<3, 1>(invk, max);
    case 3 * 8 + 2: return canon_inv<3, 2>(invk, max);
    case 3 * 8 + 3: return canon_inv<3, 3>(invk, max);
    case 3 * 8 + 4: return canon_inv<3, 4>(invk, max);
    case 3 * 8 + 5: return canon_inv<3, 5>(invk, max);
    case 3 * 8 + 6: return canon_inv<3, 6>(invk, max);
    case 3 * 8 + 7: return canon_inv<3, 7>(invk, max);
    default: return nullptr;
    }
}

template <int K, int U>
static p2s_fn p2s_fast(int C, int V)
{
    if (C == 1) return V == 2 ? contract_fast_p2s<K, 1, 2, U, false> : contract_fast_p2s<K, 1, 1, U, false>;
    return V == 2 ? contract_fast_p2s<K, 2, 2, U, false> : contract_fast_p2s<K, 2, 1, U, false>;
}

static p2s_fn pick_p2s(int K, int C, int V, bool div, int &U)
{
    if (div) {
        U = 4;
        if (C == 1) return V == 2 ? contract_fast_p2s<2, 1, 2, 4, true> : contract_fast_p2s<2, 1, 1, 4, true>;
        return V == 2 ? contract_fast_p2s<2, 2, 2, 4, true> : contract_fast_p2s<2, 2, 1, 4, true>;
    }
    switch (K) {
    case 1: U = 4; return p2s_fast<1, 4>(C, V);
    case 2: U = 4; return p2s_fast<2, 4>(C, V);
    case 3: U = 2; return p2s_fast<3, 2>(C, V);
    case 4: U = 2; return p2s_fast<4, 2>(C, V);
    case 5: U = 2; return p2s_fast<5, 2>(C, V);
    default: U = 2; return p2s_fast<6, 2>(C, V);
    }
}

typedef void (*staged_fn)(const ParamsP2S);
static staged_fn pick_staged(int K, int C)
{
    switch (K * 2 + (C - 1)) {
    case 1 * 2 + 0: return contract_staged<1, 1>;
    case 1 * 2 + 1: return contract_staged<1, 2>;
    case 2 * 2 + 0: return contract_staged<2, 1>;
    case 2 * 2 + 1: return contract_staged<2, 2>;
    case 3 * 2 + 0: return contract_staged<3, 1>;
    case 3 * 2 + 1: return contract_staged<3, 2>;
    default: return nullptr;
    }
}

// persistent grid: as many CTAs as are co-resident (occupancy is register-bound and differs per variant)
typedef void (*tma_fn)(const ParamsP2T);
static tma_fn pick_staged_tma(int K, int C)
{
    switch (K * 2 + (C - 1)) {
    case 1 * 2 + 0: return contract_staged_tma<1, 1>;
    case 1 * 2 + 1: return contract_staged_tma<1, 2>;
    case 2 * 2 + 0: return contract_staged_tma<2, 1>;
    case 2 * 2 + 1: return contract_staged_tma<2, 2>;
    case 3 * 2 + 0: return contract_staged_tma<3, 1>;
    case 3 * 2 + 1: return contract_staged_tma<3, 2>;
    default: return nullptr;
    }
}

template <class F>
static uint64_t resident_ctas(bnpp_ctx *ctx, F fn)
{
    static std::map<std::pair<int, const void *>, int> cache;      // per device and variant
    static std::mutex mu;
    std::lock_guard<std::mutex> lock(mu);
    const auto key = std::make_pair(ctx->device, reinterpret_cast<const void *>(fn));
    auto it = cache.find(key);
    if (it == cache.end()) {
        int per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kBlock, 0) != cudaSuccess || per_sm < 1) per_sm = 2;
        it = cache.insert({key, per_sm}).first;
    }
    return (uint64_t)ctx->sm_count * it->second;
}

// the same for a kernel with dynamic shared memory (opt-in above 48 KB, granted once per device and variant); 0 on error
template <class F>
static uint64_t resident_ctas_dyn(bnpp_ctx *ctx, F fn, unsigned smem)
{
    static std::map<std::tuple<int, const void *, unsigned>, int> cache;       // per device, variant and KB of shared memory
    static std::map<std::pair<int, const void *>, bool> granted;
    static std::mutex mu;
    std::lock_guard<std::mutex> lock(mu);
    const void *f = reinterpret_cast<const void *>(fn);
    if (!granted[{ctx->device, f}]) {
        if (cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kStagedSmemBudget) != cudaSuccess) return 0;
        granted[{ctx->device, f}] = true;
    }
    const auto key = std::make_tuple(ctx->device, f, (smem + 1023u) / 1024u);
    auto it = cache.find(key);
    if (it == cache.end()) {
        int per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kBlock, smem) != cudaSuccess || per_sm < 1) return 0;
        it = cache.insert({key, per_sm}).first;
    }
    return (uint64_t)ctx->sm_count * it->second;
}

static void describe(LaunchDesc *d, const ParamsHead &h, const void *fn, uint64_t blocks, const char *variant, int k, int C,
                     int V, int U, bool div, bool generic, uint32_t R)
{
    d->fn = fn;
    d->grid = (unsigned)blocks;
    d->k = k;
    // the printable name is formatted only when somebody asks for it (LaunchDesc::name())
    d->variant = variant;
    d->C = C;
    d->V = V;
    d->U = U;
    d->div = div;
    d->generic = generic;
    d->max = false;
    d->R = R;
    (void)h;
}

std::string LaunchDesc::name()
{
    const ParamsHead &h = head();
    char nm[128];
    if (mvt) snprintf(nm, sizeof nm, "contract_mvt<%s,K=%d,stages=%d> cx=%u T=%u g=%u tiles=%u R=%u stage=%uB", variant, k, U, h.cx,
                      mvtp.T, mvtp.g, mvtp.n_tiles, R, mvtp.stage_doubles * 8u);
    else if (mv) snprintf(nm, sizeof nm, "contract_mv<%s,K=%d,U=%d> cx=%u T=%u E=%u g=%u tiles=%u R=%u", variant, k, U, h.cx, mvp.T, mvp.E,
                     mvp.g, mvp.n_tiles, R);
    else if (max && generic) snprintf(nm, sizeof nm, "contract_generic_max<%s,K=%d> cx=%u R=%u", variant, k, h.cx, R);
    else if (max) snprintf(nm, sizeof nm, "contract_canon_max<%s,K=%d,U=%d> R=%u cls=%d,%d,%d", variant, k, U, R, h.cls[0],
                           k > 1 ? h.cls[1] : -1, k > 2 ? h.cls[2] : -1);
    else if (generic) snprintf(nm, sizeof nm, "contract_generic<%s,K=%d,div=%d> cx=%u R=%u", variant, k, div, h.cx, R);
    else snprintf(nm, sizeof nm, "contract_fast<%s,K=%d,C=%d,V=%d,U=%d,div=%d> R=%u cls=%d,%d,%d", variant, k, C, V, U, div, R,
                  h.cls[0], k > 1 ? h.cls[1] : -1, k > 2 ? h.cls[2] : -1);
    return nm;
}

template <class P>
static int plan_launch(bnpp_ctx *ctx, LaunchDesc *d, const P &p, int k, int C, int V, bool div, bool generic, const char *mode,
                       uint32_t R, bool max = false)
{
    int U = 1;
    typename Launch<P>::fn_t fn = max ? Launch<P>::pick_max(k) : Launch<P>::pick(k, C, V, div, generic, U);
    uint64_t blocks = (p.h.n_items + (uint64_t)kBlock * U - 1) / ((uint64_t)kBlock * U);
    const uint64_t cap = resident_ctas(ctx, fn);
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    describe(d, p.h, reinterpret_cast<const void *>(fn), blocks, mode, k, C, V, U, div, generic, R);
    d->max = max;
    return BNPP_OK;
}

// max: only the canonical layout has a max-product variant here (false otherwise: contract_generic<MAX> takes the step)
static bool plan_launch_p2s(bnpp_ctx *ctx, LaunchDesc *d, const ParamsP2 &p, int k, int C, int V, bool div, uint32_t R,
                            bool max = false)
{
    int U = 1;
    p2s_fn fn = nullptr;
    const char *variant = "p2s";
    // canonical VE layout: every operand has the eliminated variable as its stride-1 axis
    if (!div && C == 2 && V == 2 && k <= 3 && p.h.out_vec) {
        unsigned mask = 0;
        bool canon = true;
        for (int q = 0; q < k; ++q) {
            if (p.h.cls[q] == LC_V4) mask |= 1u << q;
            else if (p.h.cls[q] != LC_VX_B) canon = false;
        }
        if (canon) {
            // an operand none of whose bit-fields touches item bits 8..9 (= u * kBlock) is the
            // same element for all U items of a thread; keep the heaviest such operand in registers
            int invk = -1;
            for (int q = 0; q < k; ++q) {
                bool touches = false;
                for (int f = 0; f < (int)p.nf[q]; ++f)
                    touches |= (((uint64_t)p.f[q][f].mask << p.f[q][f].sh) & (uint64_t)(kBlock * (kCanonU - 1))) != 0;
                if (!touches && (invk < 0 || (((mask >> q) & 1u) && !((mask >> invk) & 1u)))) invk = q;
            }
            fn = pick_canon(k, mask, invk, max);
            U = kCanonU;
            variant = invk < 0 ? "canon" : (invk == 0 ? "canon/inv0" : (invk == 1 ? "canon/inv1" : "canon/inv2"));
        }
    }
    if (max && (!fn || !aligned(p.h.arg, 2))) return false;
    if (!fn) fn = pick_p2s(k, C, V, div, U);
    const uint64_t ch = (uint64_t)kBlock * U;
    if (p.h.n_items < ch || p.h.n_items % ch) return false;   // tiny problem: per-item kernel
    uint64_t blocks = p.h.n_items / ch;
    const uint64_t cap = resident_ctas(ctx, fn);
    if (blocks > cap) blocks = cap;
    describe(d, p.h, reinterpret_cast<const void *>(fn), blocks, variant, k, C, V, U, div, false, R);
    d->max = max;
    return true;
}

int contract_launch(bnpp_ctx *ctx, LaunchDesc &d, const double *const *in, double *out, double *z)
{
    ParamsHead &h = d.head();
    for (int q = 0; q < d.k; ++q) h.in[q] = in[q];
    h.out = out;
    h.z = z;
    void *args[1];
    args[0] = d.params();
    BNPP_CUDA(ctx, cudaLaunchKernel(d.fn, dim3(d.grid), dim3(kBlock), args, d.smem, ctx->stream));
    ctx->launches++;
    ctx->last_desc = &d;
    ctx->last_kernel.clear();
    ctx->last_grid = d.grid;
    ctx->last_block = kBlock;
    return BNPP_OK;
}

int contract(bnpp_ctx *ctx, int k, const bnpp_operand *ops, const bnpp_scope *out_scope, int64_t elim_var, int divide,
             double *out_dev, double *z_dev, bool max_mode, uint8_t *arg_dev)
{
    LaunchDesc d;
    const int rc = contract_plan(ctx, k, ops, out_scope, elim_var, divide, out_dev, z_dev, &d, max_mode, arg_dev);
    if (rc != BNPP_OK) return rc;
    const double *in[kMaxK];
    for (int q = 0; q < k; ++q) in[q] = ops[q].data;
    const int rc2 = contract_launch(ctx, d, in, out_dev, z_dev);
    ctx->last_kernel = d.name();      // the descriptor dies here: keep the printable name, not the pointer
    ctx->last_desc = nullptr;
    contract_release(ctx, d);         // stream-ordered: after the launch that reads the table
    return rc2;
}

// max_mode: 0 = sum-product; 1 = max-product, canon<MAX> where the sum-mode plan takes canon; 2 = max-product, generic<MAX>
static int plan_impl(bnpp_ctx *ctx, int k, const bnpp_operand *ops, const bnpp_scope *out_scope, int64_t elim_var,
                     int divide, double *out_dev, double *z_dev, LaunchDesc *desc, int max_mode, uint8_t *arg_dev);

int contract_plan(bnpp_ctx *ctx, int k, const bnpp_operand *ops, const bnpp_scope *out_scope, int64_t elim_var,
                  int divide, double *out_dev, double *z_dev, LaunchDesc *desc, bool max_mode, uint8_t *arg_dev)
{
    if (!ctx || !desc) return BNPP_EINVAL;
    if (max_mode) {
        if (elim_var < 0) return fail(ctx, BNPP_EINVAL, "product_max_out: a max-product step eliminates a variable");
        if (divide) return fail(ctx, BNPP_EINVAL, "product_max_out: no divide");
        if (!arg_dev) return fail(ctx, BNPP_EINVAL, "product_max_out: argmax buffer missing");
    }
    return plan_impl(ctx, k, ops, out_scope, elim_var, divide, out_dev, z_dev, desc, max_mode ? 1 : 0, arg_dev);
}

static int plan_impl(bnpp_ctx *ctx, int k, const bnpp_operand *ops, const bnpp_scope *out_scope, int64_t elim_var,
                     int divide, double *out_dev, double *z_dev, LaunchDesc *desc, int max_mode, uint8_t *arg_dev)
{
    // the generic max-product kernel: one output entry per item (V = 1), planned again from scratch
    auto generic_max = [&]() { return plan_impl(ctx, k, ops, out_scope, elim_var, divide, out_dev, z_dev, desc, 2, arg_dev); };
    if (k < 1 || k > kMaxK) return fail(ctx, BNPP_ERANK, "product_sum_out: operand count must be 1..BNPP_MAX_OPERANDS");
    if (divide && k != 2) return fail(ctx, BNPP_EINVAL, "divide needs exactly two operands");
    if (!out_scope || out_scope->rank < 0 || out_scope->rank > BNPP_MAX_RANK)
        return fail(ctx, BNPP_EINVAL, "bad output scope");
    const int wr = out_scope->rank;

    // output axes, dense row-major, last fastest (code/domain.cpp:20-24)
    std::vector<Axis> axes(wr);
    uint64_t n_out = 1;
    for (int i = wr - 1; i >= 0; --i) {
        if (out_scope->card[i] == 0) return fail(ctx, BNPP_EINVAL, "zero cardinality");
        if (elim_var >= 0 && out_scope->var_id[i] == (uint64_t)elim_var)
            return fail(ctx, BNPP_EINVAL, "the eliminated variable is in the output scope");
        for (int j = i + 1; j < wr; ++j)
            if (out_scope->var_id[i] == out_scope->var_id[j]) return fail(ctx, BNPP_EINVAL, "duplicate variable in output scope");
        axes[i].ext = out_scope->card[i];
        axes[i].so = n_out;
        axes[i].miss = 0;
        for (int q = 0; q < kMaxK; ++q) axes[i].s[q] = 0;
        n_out *= out_scope->card[i];
        if (n_out >= (1ull << 32)) return fail(ctx, BNPP_ETOOBIG, "output table has >= 2^32 entries");
    }

    uint64_t sx[kMaxK] = {0};
    uint64_t op_bytes[kMaxK] = {0};
    uint32_t cx = 1;
    for (int q = 0; q < k; ++q) {
        const bnpp_operand &op = ops[q];
        if (op.scope.rank < 0 || op.scope.rank > BNPP_MAX_RANK) return fail(ctx, BNPP_EINVAL, "bad operand scope");
        uint64_t dense = 1, maxoff = 0;
        for (int i = op.scope.rank - 1; i >= 0; --i) {
            const uint32_t var = op.scope.var_id[i], card = op.scope.card[i];
            if (op.stride && op.stride[i] < 0) return fail(ctx, BNPP_EINVAL, "negative stride");
            const uint64_t st = op.stride ? (uint64_t)op.stride[i] : dense;
            dense *= card;
            maxoff += (uint64_t)(card - 1) * st;
            for (int j = i + 1; j < op.scope.rank; ++j)
                if (op.scope.var_id[j] == var) return fail(ctx, BNPP_EINVAL, "duplicate variable in operand scope");
            if (elim_var >= 0 && var == (uint64_t)elim_var) {
                sx[q] = st;
                if (cx != 1 && cx != card) return fail(ctx, BNPP_EINVAL, "inconsistent cardinality of the eliminated variable");
                cx = card;
                continue;
            }
            int pos = -1;
            for (int j = 0; j < wr; ++j)
                if (out_scope->var_id[j] == var) { pos = j; break; }
            if (pos < 0) return fail(ctx, BNPP_EINVAL, "operand variable is neither in the output scope nor eliminated");
            if (out_scope->card[pos] != card) return fail(ctx, BNPP_EINVAL, "cardinality mismatch between operand and output");
            axes[pos].s[q] = st;
        }
        if (maxoff >= (1ull << 32)) return fail(ctx, BNPP_ETOOBIG, "operand table has >= 2^32 entries");
        op_bytes[q] = 8 * dense;
    }
    if (max_mode && cx > 255)
        return fail(ctx, BNPP_EINVAL, "product_max_out: the eliminated variable has more than 255 values (uint8 argmax)");

    // ---- iteration order -------------------------------------------------------
    // keep the output's fastest axes (>= kTileOutputs entries) in place; above them iterate
    // fastest the axes that large operands lack, so their tiles are re-read from L2
    std::vector<Axis> it;
    for (int i = 0; i < wr; ++i)
        if (axes[i].ext > 1) it.push_back(axes[i]);
    {
        size_t first_tile = it.size();
        uint64_t cover = 1;
        while (first_tile > 0 && cover < kTileOutputs) cover *= it[--first_tile].ext;
        bool any = false;
        for (size_t a = 0; a < first_tile; ++a) {
            for (int q = 0; q < k; ++q)
                if (it[a].s[q] == 0 && op_bytes[q] > kReuseBytes) it[a].miss += op_bytes[q];
            any |= it[a].miss != 0;
        }
        if (any)
            std::stable_sort(it.begin(), it.begin() + first_tile, [](const Axis &x, const Axis &y) { return x.miss < y.miss; });
    }

    // The U items of a thread differ in item bits 8.. (u * kBlock).  Put there binary axes
    // that operands LACK: those operands then address the same element for several of the
    // thread's items, and the repeated loads merge in L1 instead of each crossing L2 (an
    // L2-resident broadcast operand costs L2 bandwidth like a streamed one).
    if (cx <= 2) {
        size_t split = it.size();
        uint64_t inner = 1;
        while (split > 0 && inner < 2u * kBlock) inner *= it[--split].ext;
        bool p2all = true;
        for (const Axis &a : it) p2all = p2all && is_pow2(a.ext);
        if (p2all && inner == 2u * kBlock && split > 0) {
            auto weight = [&](int q) { return (uint64_t)(sx[q] ? 2 : 1) * (it.back().s[q] ? 2 : 1); };
            auto score = [&](size_t a) {
                uint64_t sc = 0;
                for (int q = 0; q < k; ++q)
                    if (it[a].s[q] == 0) sc += weight(q);
                return sc;
            };
            // the heaviest operand that lacks at least two eligible axes gets both unroll bits
            int owner = -1;
            for (int q = 0; q < k; ++q) {
                int lacking = 0;
                for (size_t a = 0; a < split; ++a) lacking += (it[a].ext == 2 && it[a].s[q] == 0);
                if (lacking >= 2 && (owner < 0 || weight(q) > weight(owner))) owner = q;
            }
            for (int pick = 0; pick < 2; ++pick) {
                int best = -1;
                uint64_t best_score = 0;
                for (size_t a = 0; a + pick < split; ++a) {
                    if (it[a].ext != 2) continue;
                    if (owner >= 0 && it[a].s[owner] != 0) continue;
                    const uint64_t sc = score(a);
                    if (sc > best_score) { best_score = sc; best = (int)a; }
                }
                if (best < 0) break;
                const Axis ax = it[best];   // move it to just above the thread bits (and the axis placed before it)
                it.erase(it.begin() + best);
                it.insert(it.begin() + (split - 1 - pick), ax);
            }
        }
    }

    // ---- one transposed operand goes through shared memory -----------------------------------------
    // binary axes innermost first: b[0] is the V bit, b[1..10] the item bits of a 1024-item chunk
    int staged = -1;
    std::vector<Axis> bin;
    if (cx <= 2 && !divide && k <= 3 && n_out >= (1u << 11)) {
        bool p2all = true;
        for (const Axis &a : it) p2all = p2all && is_pow2(a.ext);
        if (p2all) {
            for (size_t i = it.size(); i-- > 0;)
                for (uint32_t t = 0, e = ilog2(it[i].ext); t < e; ++t) {
                    Axis a = it[i];
                    a.ext = 2;
                    a.so = it[i].so << t;
                    for (int q = 0; q < k; ++q) a.s[q] = it[i].s[q] << t;
                    bin.push_back(a);
                }
        }
        if (bin.size() >= 11) {
            uint64_t total = 8 * n_out;
            for (int q = 0; q < k; ++q) total += op_bytes[q];
            uint64_t best_bytes = 0;
            for (int q = 0; q < k; ++q) {
                int far = 0;   // lane-level axes (V bit + 5 lane bits) on which the operand jumps by >= 128 bytes
                for (int a = 0; a < 6; ++a) far += (bin[a].s[q] >= 16);
                if (far >= 4 && op_bytes[q] * 8 >= total && op_bytes[q] > best_bytes) { best_bytes = op_bytes[q]; staged = q; }
            }
        }
        if (staged >= 0) {
            // chunk bits 5..9 (b[6..10]) := the staged operand's fastest remaining axes, smallest stride first
            for (int slot = 6; slot <= 10; ++slot) {
                int best = -1;
                for (size_t a = slot; a < bin.size(); ++a)
                    if (bin[a].s[staged] != 0 && (best < 0 || bin[a].s[staged] < bin[best].s[staged])) best = (int)a;
                if (best < 0) break;
                const Axis ax = bin[best];
                bin.erase(bin.begin() + best);
                bin.insert(bin.begin() + slot, ax);
            }
            // The chunks in flight at one time (a few hundred CTAs, grid-stride) differ in the LOW chunk bits.  An axis
            // the staged operand lacks re-reads its tile: as a low chunk bit the second read comes right after the first
            // and hits L2; left among the slow axes it goes to DRAM again half a kernel later (F-bcast: +33% traffic).
            for (int moved = 0, slot = 11; moved < 4 && slot < (int)bin.size(); ++moved, ++slot) {
                int best = -1;
                for (size_t a = slot; a < bin.size() && best < 0; ++a)
                    if (bin[a].s[staged] == 0) best = (int)a;
                if (best < 0) break;
                const Axis ax = bin[best];
                bin.erase(bin.begin() + best);
                bin.insert(bin.begin() + slot, ax);
            }
            it.assign(bin.rbegin(), bin.rend());
        }
    }

    // merge neighbours that are contiguous in the output and in every operand
    std::vector<Axis> m;
    for (size_t i = 0; i < it.size(); ++i) {
        if (!m.empty()) {
            Axis &o = m.back();   // o is OUTER to it[i]
            bool ok = (o.so == it[i].so * it[i].ext);
            for (int q = 0; q < k && ok; ++q) ok = (o.s[q] == it[i].s[q] * it[i].ext);
            if (ok && (uint64_t)o.ext * it[i].ext < (1ull << 32)) {
                o.ext *= it[i].ext;
                o.so = it[i].so;
                for (int q = 0; q < k; ++q) o.s[q] = it[i].s[q];
                continue;
            }
        }
        m.push_back(it[i]);
    }

    const bool generic = (cx > 2) || max_mode == 2;
    // The tiled multi-valued kernels stream: they pay per union entry for bringing operand entries to the SM.  A step
    // whose operands are all much smaller than its union table (an outer product of small tables) re-reads them from
    // L1/L2 either way, and there the one-entry-per-thread kernel with its cached gathers is as fast or faster
    // (Munin1's widest step: 0.41 ms against 0.67 ms) -- so the tiled kernels take a step only when its heaviest
    // operand covers at least a sixteenth of the union table (Barley's widest step, 1/5: 0.023 ms -> 0.018 ms tiled).
    uint64_t heaviest = 0;
    for (int q = 0; q < k; ++q) heaviest = std::max(heaviest, op_bytes[q]);
    const bool streams = heaviest * 16 >= 8 * n_out * cx || mv_min_entries() == 0;
    if (generic && !divide && !max_mode && streams && n_out * cx >= mv_min_entries()) {
        // multi-valued elimination: the table-driven tile kernel (contract_mv.cu), in the output's own axis order
        std::vector<MVAxis> mva;
        for (int i = 0; i < wr; ++i) {
            if (axes[i].ext <= 1) continue;
            MVAxis a;
            a.ext = axes[i].ext;
            for (int q = 0; q < kMaxK; ++q) a.s[q] = axes[i].s[q];
            mva.push_back(a);
        }
        ParamsHead hm;
        memset(&hm, 0, sizeof hm);
        for (int q = 0; q < k; ++q) hm.in[q] = ops[q].data;
        hm.out = out_dev;
        hm.partials = ctx->partials;
        hm.ticket = ctx->ticket;
        hm.z = z_dev;
        hm.status = ctx->status;
        *desc = LaunchDesc();
        if (mv_staged_enabled()) {
            const int rct = plan_mvt(ctx, desc, k, cx, sx, op_bytes, mva, n_out, hm);
            if (rct <= 0) return rct;
            *desc = LaunchDesc();
        }
        const int rc = plan_mv(ctx, desc, k, cx, sx, op_bytes, mva, n_out, hm);
        if (rc <= 0) return rc;     // planned, or an error; 1 = not applicable: the one-entry-per-thread kernel below
    }
    desc->smem = 0;
    desc->mv = desc->mvt = desc->tma = false;
    const int C = generic ? 0 : (int)cx;
    int V = 1;
    if (!generic && !m.empty() && (m.back().ext % 2 == 0)) V = 2;

    ParamsHead h;
    memset(&h, 0, sizeof h);
    for (int q = 0; q < k; ++q) {
        h.in[q] = ops[q].data;
        h.sx[q] = (uint32_t)sx[q];
        h.sl[q] = m.empty() ? 0 : (uint32_t)m.back().s[q];
    }
    h.sol = m.empty() ? 0 : (uint32_t)m.back().so;
    if (V == 2) {
        Axis &l = m.back();
        l.ext /= 2;
        l.so *= 2;
        for (int q = 0; q < k; ++q) l.s[q] *= 2;
        if (l.ext == 1) m.pop_back();
    }
    const uint32_t R = (uint32_t)m.size();
    h.n_items = n_out / V;
    h.cx = cx;
    h.out = out_dev;
    h.arg = max_mode ? arg_dev : nullptr;
    h.out_vec = (V == 2 && h.sol == 1 && aligned(out_dev, 16)) ? 1 : 0;
    for (uint32_t a = 0; a < R && h.out_vec; ++a)
        if (m[a].so % 2) h.out_vec = 0;

    // load class per operand: how the [V x C] micro-tile sits in the operand's memory
    for (int q = 0; q < k && !generic; ++q) {
        const uint32_t x = h.sx[q], l = (V == 2) ? h.sl[q] : 0;
        bool mult2 = true, mult4 = true;
        for (uint32_t a = 0; a < R; ++a) {
            if (m[a].s[q] % 2) mult2 = false;
            if (m[a].s[q] % 4) mult4 = false;
        }
        const bool has_x = (C == 2 && x != 0), has_l = (V == 2 && l != 0);
        uint8_t c;
        if (!has_x && !has_l) c = LC_BCAST;
        else if (has_x && x == 1 && mult2 && aligned(h.in[q], 16) && (!has_l || l % 2 == 0)) {
            if (!has_l) c = LC_VX_B;
            else if (l == 2 && mult4 && aligned(h.in[q], 32)) c = LC_V4;
            else c = LC_VX;
        } else if (has_l && l == 1 && mult2 && aligned(h.in[q], 16) && (!has_x || x % 2 == 0)) {
            if (!has_x) c = LC_VL_B;
            else if (x == 2 && mult4 && aligned(h.in[q], 32)) c = LC_V4T;
            else c = LC_VL;
        } else if (has_x && has_l) c = LC_S_JX;
        else c = has_x ? LC_S_X : LC_S_L;
        h.cls[q] = c;
    }

    h.partials = ctx->partials;
    h.ticket = ctx->ticket;
    h.z = z_dev;
    h.status = ctx->status;

    // ---- power-of-two iteration space: per-operand bit-fields --------------------
    bool p2 = true;
    for (uint32_t a = 0; a < R; ++a) p2 = p2 && is_pow2(m[a].ext);
    if (p2) {
        ParamsP2 &p = desc->p2p.b;
        memset(&desc->p2p, 0, sizeof desc->p2p);
        p.h = h;
        bool fits = true;
        for (int q = 0; q <= k && fits; ++q) {
            int nf = 0;
            uint32_t sh = 0;
            // walk axes innermost first; a field grows while the next axis continues it in THIS operand
            uint32_t cur_sh = 0, cur_bits = 0;
            uint64_t cur_mul = 0;
            for (int a = (int)R - 1; a >= 0; --a) {
                const uint32_t bits = ilog2(m[a].ext);
                const uint64_t st = (q == k) ? m[a].so : m[a].s[q];
                if (cur_bits && st == (cur_mul << cur_bits) && st != 0) {
                    cur_bits += bits;
                } else {
                    if (cur_bits && cur_mul) {
                        if (nf == kMaxF) { fits = false; break; }
                        p.f[q][nf++] = Field{(cur_bits >= 32) ? 0xffffffffu : ((1u << cur_bits) - 1), (uint32_t)cur_mul, cur_sh};
                    }
                    cur_sh = sh;
                    cur_bits = bits;
                    cur_mul = st;
                }
                sh += bits;
            }
            if (fits && cur_bits && cur_mul) {
                if (nf == kMaxF) fits = false;
                else p.f[q][nf++] = Field{(cur_bits >= 32) ? 0xffffffffu : ((1u << cur_bits) - 1), (uint32_t)cur_mul, cur_sh};
            }
            p.nf[q] = (uint8_t)nf;
        }
        if (fits && staged >= 0 && V == 2 && h.n_items % (4 * kBlock) == 0 && h.n_items >= 4 * kBlock) {
            // slots of a tile: the chunk-local bits operand q depends on, ranked by ITS stride.  tma: its runs can be
            // bulk-copied (slot bit 0 is its stride-1 axis, every other bit and every chunk stride moves by an even number
            // of doubles, the table is 16-byte aligned); *low: the lowest slot bit a lane bit drives
            struct Loc { uint64_t stride; int item_bit; };   // item_bit: -2 = x, -1 = V bit, 0..9 = item bits
            int lane_rank[5];            // of the last build_stage call: slot bit each lane bit drives (-1: none)
            auto build_stage = [&](int q, StageInfo &st, bool &even, int &low) -> bool {
                std::vector<Loc> loc;
                if (C == 2 && sx[q]) loc.push_back({sx[q], -2});
                for (int a = 0; a <= 10; ++a)
                    if (bin[a].s[q]) loc.push_back({bin[a].s[q], a - 1});
                std::sort(loc.begin(), loc.end(), [](const Loc &x, const Loc &y) { return x.stride < y.stride; });
                memset(&st, 0, sizeof st);
                st.sk = q;
                st.tile = 1u << loc.size();
                bool ok = loc.size() <= 12;
                int rank_of_item[10];
                for (int i = 0; i < 10; ++i) rank_of_item[i] = -1;
                for (size_t r = 0; r < loc.size() && ok; ++r) {
                    if (loc[r].item_bit == -2) st.slot_x = 1u << r;
                    else if (loc[r].item_bit == -1) st.slot_j = 1u << r;
                    else rank_of_item[loc[r].item_bit] = (int)r;
                    // tile-load fields: runs of ranks whose strides keep doubling
                    if (st.nlf && loc[r].stride == ((uint64_t)st.lf[st.nlf - 1].mul << ilog2(st.lf[st.nlf - 1].mask + 1)))
                        st.lf[st.nlf - 1].mask = (st.lf[st.nlf - 1].mask << 1) | 1u;
                    else if (st.nlf < 12) st.lf[st.nlf++] = Field{1u, (uint32_t)loc[r].stride, (uint32_t)r};
                    else ok = false;
                }
                // consumption fields: runs of item bits whose ranks are consecutive
                for (int i = 0; i < 10 && ok; ++i) {
                    if (rank_of_item[i] < 0) continue;
                    if (st.ncf && i > 0 && rank_of_item[i - 1] >= 0 && rank_of_item[i] == rank_of_item[i - 1] + 1 &&
                        st.cf[st.ncf - 1].sh + ilog2(st.cf[st.ncf - 1].mask + 1) == (uint32_t)i)
                        st.cf[st.ncf - 1].mask = (st.cf[st.ncf - 1].mask << 1) | 1u;
                    else if (st.ncf < 12) st.cf[st.ncf++] = Field{1u, 1u << rank_of_item[i], (uint32_t)i};
                    else ok = false;
                }
                low = 32;
                for (int i = 0; i < 5; ++i) {
                    lane_rank[i] = rank_of_item[i];
                    if (rank_of_item[i] >= 0 && rank_of_item[i] < low) low = rank_of_item[i];
                }
                even = !loc.empty() && loc[0].stride == 1 && aligned(ops[q].data, 16);
                for (size_t r = 1; r < loc.size() && even; ++r)
                    if (loc[r].stride % 2) even = false;
                for (uint32_t a = 0; a < R && even; ++a)
                    if (m[a].s[q] % 2 && m[a].s[q] != 1) even = false;
                return ok;
            };
            // TMA: runs of at least 64 bytes, at most one run per thread
            auto tma_operand = [&](const StageInfo &st, bool even, TmaOperand &t) -> bool {
                if (!even || !st.nlf || st.lf[0].mul != 1 || st.lf[0].sh != 0) return false;
                const uint32_t rb = ilog2(st.lf[0].mask + 1);
                if (rb < 3 || (st.tile >> rb) > (uint32_t)kBlock) return false;
                memset(&t, 0, sizeof t);
                t.tile = st.tile;
                t.rbits = rb;
                // run positions: the run bits the lanes drive lowest, in lane order (measured: 70-76% of peak on the
                // reversed F-bcast shapes against 50-67% in stride order), then the others
                t.nrb = (uint8_t)(ilog2(st.tile) - rb);
                bool placed[12] = {false};
                int next = 0;
                for (int i = 0; i < 5; ++i)
                    if (lane_rank[i] >= (int)rb) { t.rpos[lane_rank[i] - rb] = (uint8_t)next++; placed[lane_rank[i] - rb] = true; }
                for (int i = 0; i < (int)t.nrb; ++i)
                    if (!placed[i]) t.rpos[i] = (uint8_t)next++;
                const uint32_t pitch = (1u << rb) + 2u;
                auto phys = [&](uint32_t slot) {
                    uint32_t r = 0;
                    for (int i = 0; i < (int)t.nrb; ++i) r |= (((slot >> rb) >> i) & 1u) << t.rpos[i];
                    return r * pitch + (slot & ((1u << rb) - 1u));
                };
                t.dj = phys(st.slot_j);
                t.dx = phys(st.slot_x);
                t.nlf = st.nlf;
                t.ncf = st.ncf;
                memcpy(t.lf, st.lf, sizeof t.lf);
                memcpy(t.cf, st.cf, sizeof t.cf);
                return true;
            };
            StageInfo &st = desc->p2p.st;
            bool even = false;
            int low = 32;
            const bool ok = build_stage(staged, st, even, low);
            uint64_t blocks = h.n_items / (4 * kBlock);
            ParamsP2T &pt = desc->p2t;
            if (ok && staged_tma_enabled() && k <= kTmaMaxK && tma_operand(st, even, pt.t[staged])) {
                pt.mask = 1u << staged;
                const uint32_t budget = kStagedSmemBudget;
                auto padded = [](const TmaOperand &t) { return t.tile + 2u * (t.tile >> t.rbits); };
                uint32_t doubles = padded(pt.t[staged]);
                // the other operands ride along while two stages of everything fit, smallest tile first
                if (staged_async_enabled()) {
                    std::vector<std::pair<uint32_t, int>> riders;
                    for (int q = 0; q < k; ++q) {
                        StageInfo sq;
                        bool eq = false;
                        int lq = 32;
                        if (q != staged && build_stage(q, sq, eq, lq) && tma_operand(sq, eq, pt.t[q])) riders.push_back({padded(pt.t[q]), q});
                    }
                    std::sort(riders.begin(), riders.end());
                    for (const auto &r : riders)
                        if (2u * (doubles + r.first) * 8u <= budget) {
                            doubles += r.first;
                            pt.mask |= 1u << r.second;
                        }
                }
                uint32_t off = 0;
                pt.stage_bytes = 0;
                for (int q = 0; q < k; ++q)
                    if ((pt.mask >> q) & 1u) {
                        pt.t[q].off = off;
                        off += padded(pt.t[q]);
                        pt.stage_bytes += pt.t[q].tile * 8u;
                    }
                pt.stage_doubles = off;
                pt.stages = (3u * off * 8u <= budget) ? 3u : 2u;
                // An operand that carries an eighth of the traffic and does NOT fit the ring would be loaded chunk by chunk
                // into registers: there the element-wise kernel below is the faster one (F-elem reversed: 89-92% of peak
                // against 82-83%), and this one wins when everything big is prefetched (F-bcast reversed: 70-80% against 61-66%)
                uint64_t total_bytes = 8 * n_out;
                for (int q = 0; q < k; ++q) total_bytes += op_bytes[q];
                bool all_big = true;
                for (int q = 0; q < k; ++q)
                    if (!((pt.mask >> q) & 1u) && op_bytes[q] * 8 >= total_bytes) all_big = false;
                tma_fn fn = pick_staged_tma(k, C);
                if (fn && all_big && 2u * off * 8u <= budget) {
                    if (max_mode) return generic_max();
                    pt.b = p;
                    desc->p2 = true;
                    desc->tma = true;
                    desc->smem = pt.stages * off * (unsigned)sizeof(double);
                    const uint64_t cap = resident_ctas_dyn(ctx, fn, desc->smem);
                    if (!cap) return fail(ctx, BNPP_ECUDA, "contract_staged_tma: shared memory not granted");
                    if (blocks > cap) blocks = cap;
                    static const char *const names[8] = {"tma", "tma/0", "tma/1", "tma/01", "tma/2", "tma/02", "tma/12", "tma/012"};
                    describe(desc, pt.b.h, reinterpret_cast<const void *>(fn), blocks, names[pt.mask & 7u], k, C, V, 4, false, false, R);
                    return BNPP_OK;
                }
            }
            // element-wise copies (LDGSTS).  Lanes are item bits 0..4: swizzle with the lowest slot bit any of them
            // drives (if it is high enough); 16-byte copies when slots 2m, 2m+1 are neighbours in the operand
            st.swz = (low >= 5 && low < 32) ? (uint32_t)low : 31u;
            st.pair = (even && st.tile >= 2 * kBlock) ? 1 : 0;
            staged_fn fn = ok ? pick_staged(k, C) : nullptr;
            if (fn) {
                if (max_mode) return generic_max();
                desc->p2 = true;
                desc->staged = true;
                const uint64_t cap = resident_ctas(ctx, fn);
                if (blocks > cap) blocks = cap;
                describe(desc, p.h, reinterpret_cast<const void *>(fn), blocks, staged == 0 ? "staged0" : (staged == 1 ? "staged1" : "staged2"),
                         k, C, V, 4, false, false, R);
                return BNPP_OK;
            }
        }
        if (fits) {
            desc->p2 = true;
            desc->staged = false;
            if (!generic && plan_launch_p2s(ctx, desc, p, k, C, V, divide != 0, R, max_mode != 0)) return BNPP_OK;
            if (max_mode && !generic) return generic_max();
            return plan_launch(ctx, desc, p, k, C, V, divide != 0, generic, "p2", R, max_mode != 0);
        }
    }

    if (max_mode && !generic) return generic_max();
    if ((int)R > kMaxR) return fail(ctx, BNPP_ERANK, "more than BNPP_MAX_AXES non-mergeable axes");
    ParamsMR &p = desc->mrp;
    memset(&p, 0, sizeof p);
    p.h = h;
    p.R = R;
    for (uint32_t a = 0; a < R; ++a) {
        p.div[a] = make_fastdiv(m[a].ext);
        p.so[a] = (uint32_t)m[a].so;
        for (int q = 0; q < k; ++q) p.s[q][a] = (uint32_t)m[a].s[q];
    }
    desc->p2 = false;
    return plan_launch(ctx, desc, p, k, C, V, divide != 0, generic, "mr", R, max_mode != 0);
}

}  // namespace bnpp
