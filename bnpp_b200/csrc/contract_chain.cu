// K11 -- contract_chain: a window of m binary eliminations of a VE plan in one launch (see chain.hpp).
//
// Per rest item r a thread loads the head's 2^m contiguous doubles (256-bit loads), runs level j = 0 .. m-1 on its
// register tile and stores the 2^n doubles of the last level.  Level j computes, for every output entry o,
//     p(u) = op0 * op1 * ...  (__dmul_rn, in the step's own operand order)   at u = 2o and u = 2o + 1,
//     out[o] = __dadd_rn(p(2o), p(2o + 1))
// -- what contract_canon / contract_fast_p2s compute for that step, so the results are the same bits.  Side operands
// (small tables, L1/L2-resident) are gathered at base(r) + sum over the union bits of bit * stride: the bits are
// compile-time constants of the unrolled tile loop, the strides are parameters.  Only the head is read from HBM and
// only the last level's output is written there.
#include <cstdio>
#include <string>
#include <utility>

#include "chain.hpp"
#include "common.cuh"

namespace bnpp {

__device__ __forceinline__ uint32_t chain_fields(const Field *f, uint32_t nf, uint32_t r)
{
    uint32_t o = 0;
    for (uint32_t i = 0; i < nf; ++i) o += ((r >> f[i].sh) & f[i].mask) * f[i].mul;
    return o;
}

// u is a constant of the unrolled tile loop: the sum is a handful of adds of parameters
__device__ __forceinline__ uint32_t ubit_off(const uint32_t (&us)[kChainMaxUBits], int nbits, int u)
{
    uint32_t o = 0;
#pragma unroll
    for (int b = 0; b < kChainMaxUBits; ++b)
        if (b < nbits && ((u >> b) & 1)) o += us[b];
    return o;
}

// level J of m = M levels, NB variables added before it, A added by it, KS side operands: in[0 .. IN) -> out[0 .. OUT).
// The side values of G output entries (2G union points) are loaded before any of them is used, so a thread has 2G (or
// 4G) L1 round trips in flight instead of one.
template <int M, int J, int NB, int A, int KS>
__device__ __forceinline__ void chain_level_k(const ChainLevel &L, const uint32_t (&base)[kChainMaxSides],
                                              const double (&in)[kChainTile], double (&out)[kChainTile])
{
    constexpr int INB = M - J + NB;             // input tile bits
    constexpr int UB = INB + A;                 // union bits
    constexpr int OUT = 1 << (UB - 1);
    constexpr int G = OUT < 4 ? OUT : (UB >= 5 ? 2 : 4);     // 2G union points per batch; 16 doubles of a 32-point tile
    static_assert(INB <= 4 && UB - 1 <= 4 && UB <= kChainMaxUBits, "chain tile too large");
    const double *s0 = L.s[0].p + base[0];
    const double *s1 = L.s[1].p + base[1];
#pragma unroll
    for (int g = 0; g < OUT; g += G) {
        double a[2 * G], b[2 * G];
#pragma unroll
        for (int i = 0; i < 2 * G; ++i) {
            if (KS >= 1) a[i] = __ldg(s0 + ubit_off(L.s[0].us, UB, 2 * g + i));
            if (KS >= 2) b[i] = __ldg(s1 + ubit_off(L.s[1].us, UB, 2 * g + i));
        }
#pragma unroll
        for (int o = 0; o < G; ++o) {
            double p[2];
#pragma unroll
            for (int x = 0; x < 2; ++x) {
                const int i = 2 * o + x;
                const double h = in[(2 * g + i) & ((1 << INB) - 1)];
                p[x] = KS == 0 ? h : (KS == 1 ? __dmul_rn(h, a[i]) : __dmul_rn(__dmul_rn(a[i], b[i]), h));
            }
            out[g + o] = __dadd_rn(p[0], p[1]);
        }
    }
}

// the step's own product order: h * s0 for two operands (in either order: a product of two is commutative), (s0 * s1) * h
// for three -- fold_small lists a wide bucket's operands by size, so the head comes last (the planner checks it)
template <int M, int J, int NB, int A>
__device__ __forceinline__ void chain_level(const ChainLevel &L, const uint32_t (&base)[kChainMaxSides],
                                            const double (&in)[kChainTile], double (&out)[kChainTile])
{
    if (L.k == 0) chain_level_k<M, J, NB, A, 0>(L, base, in, out);
    else if (L.k == 1) chain_level_k<M, J, NB, A, 1>(L, base, in, out);
    else chain_level_k<M, J, NB, A, 2>(L, base, in, out);
}

template <int M, int A0, int A1, int A2, int A3>
__global__ void __launch_bounds__(kBlock) contract_chain(const __grid_constant__ ChainParams p)
{
    constexpr uint32_t CH = chain_chunk_items(M);
    constexpr int U = CH / kBlock;              // rest items per thread
    constexpr int NT = A0 + (M > 1 ? A1 : 0) + (M > 2 ? A2 : 0) + (M > 3 ? A3 : 0);
    uint32_t slo[U][M][kChainMaxSides], olo[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const uint32_t r = threadIdx.x + u * kBlock;
        olo[u] = chain_fields(p.of, p.onf, r);
#pragma unroll
        for (int j = 0; j < M; ++j)
#pragma unroll
            for (int q = 0; q < kChainMaxSides; ++q)
                slo[u][j][q] = q < p.lv[j].k ? chain_fields(p.lv[j].s[q].f, p.lv[j].s[q].nf, r) : 0u;
    }
    const uint32_t n_chunks = p.n_items / CH;
    for (uint32_t c = blockIdx.x; c < n_chunks; c += gridDim.x) {
        const uint32_t rb = c * CH;
        uint32_t shi[M][kChainMaxSides];
#pragma unroll
        for (int j = 0; j < M; ++j)
#pragma unroll
            for (int q = 0; q < kChainMaxSides; ++q)
                shi[j][q] = q < p.lv[j].k ? chain_fields(p.lv[j].s[q].f, p.lv[j].s[q].nf, rb) : 0u;
        const uint32_t ohi = chain_fields(p.of, p.onf, rb);
        double a[U][kChainTile], b[U][kChainTile];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const double *src = p.head + ((uint64_t)(rb + threadIdx.x + u * kBlock) << M);
#pragma unroll
            for (int i = 0; i < (1 << M); i += 4) {
                const double4_t v = ld4(src + i);
                a[u][i] = v.x; a[u][i + 1] = v.y; a[u][i + 2] = v.z; a[u][i + 3] = v.w;
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            uint32_t base[kChainMaxLevels][kChainMaxSides];
#pragma unroll
            for (int j = 0; j < M; ++j)
#pragma unroll
                for (int q = 0; q < kChainMaxSides; ++q) base[j][q] = shi[j][q] + slo[u][j][q];
            chain_level<M, 0, 0, A0>(p.lv[0], base[0], a[u], b[u]);
            if constexpr (M > 1) chain_level<M, 1, A0, A1>(p.lv[1], base[1], b[u], a[u]);
            if constexpr (M > 2) chain_level<M, 2, A0 + A1, A2>(p.lv[2], base[2], a[u], b[u]);
            if constexpr (M > 3) chain_level<M, 3, A0 + A1 + A2, A3>(p.lv[3], base[3], b[u], a[u]);
            double *o = p.out + (ohi + olo[u]);
#pragma unroll
            for (int i = 0; i < (1 << NT); ++i) {
                uint32_t off = 0;
#pragma unroll
                for (int bit = 0; bit < NT; ++bit)
                    if ((i >> bit) & 1) off += p.os[bit];
                if constexpr (M & 1) o[off] = b[u][i];
                else o[off] = a[u][i];
            }
        }
    }
}

namespace {

// shapes: m levels (2 .. 4), level j adds add[j] (0 .. 2) variables; every level's input and output tile within
// kChainTile.  Code = (m - 2) * 81 + add[0] + 3 add[1] + 9 add[2] + 27 add[3] (add[j] = 0 for j >= m).
constexpr bool chain_shape_ok(int m, int a0, int a1, int a2, int a3)
{
    const int add[4] = {a0, a1, a2, a3};
    int nb = 0;
    for (int j = 0; j < 4; ++j) {
        if (j >= m) {
            if (add[j]) return false;
            continue;
        }
        const int inb = m - j + nb;
        const int outb = inb - 1 + add[j];
        if (inb > 4 || outb > 4) return false;
        nb += add[j];
    }
    return true;
}

constexpr int kChainCodes = 3 * 81;

template <int C>
constexpr const void *chain_entry()
{
    constexpr int m = C / 81 + 2, a0 = C % 3, a1 = C / 3 % 3, a2 = C / 9 % 3, a3 = C / 27 % 3;
    if constexpr (chain_shape_ok(m, a0, a1, a2, a3))
        return reinterpret_cast<const void *>(contract_chain<m, a0, a1, a2, a3>);
    else
        return nullptr;
}

template <int... C>
const void *chain_table(int code, std::integer_sequence<int, C...>)
{
    static const void *const table[] = {chain_entry<C>()...};
    return table[code];
}

}  // namespace

const void *chain_kernel(int m, const int *add)
{
    if (m < 2 || m > kChainMaxLevels) return nullptr;
    int code = (m - 2) * 81, w = 1;
    for (int j = 0; j < kChainMaxLevels; ++j, w *= 3) {
        const int a = j < m ? add[j] : 0;
        if (a < 0 || a > kChainMaxAdd) return nullptr;
        code += a * w;
    }
    return chain_table(code, std::make_integer_sequence<int, kChainCodes>());
}

int chain_launch(bnpp_ctx *ctx, const void *fn, unsigned grid, const ChainParams &p, const std::string &name)
{
    void *args[1] = {const_cast<ChainParams *>(&p)};
    BNPP_CUDA(ctx, cudaLaunchKernel(fn, dim3(grid), dim3(kBlock), args, 0, ctx->stream));
    ctx->launches++;
    ctx->last_desc = nullptr;
    ctx->last_kernel = name;
    ctx->last_grid = grid;
    ctx->last_block = kBlock;
    return BNPP_OK;
}

int chain_occupancy(const void *fn)
{
    int n = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, fn, kBlock, 0) != cudaSuccess) return 0;
    return n;
}

std::string chain_name(int m, const int *add)
{
    std::string s = "contract_chain<D=" + std::to_string(m) + ",add=";
    for (int j = 0; j < m; ++j) s += std::to_string(add[j]);
    return s + ">";
}

}  // namespace bnpp
