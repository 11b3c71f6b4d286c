// K8 -- batched-evidence variable elimination (BASELINE config 5: tens of thousands of
// evidence sets on one network, PR per set).
//
// Replaces running BN::partition (reference code/model.cpp:250-301) once per evidence
// set: with the observed variable IDS fixed, every set shares one elimination order and
// one plan (ve.cu); only the evidence VALUES differ.  Each intermediate gets the batch as
// its FASTEST axis, [entries][batch], so consecutive threads touch consecutive doubles;
// the resident CPTs are shared by all sets and read through a per-set base offset
//     base_k(b) = sum_j stride_kj * value[b][obs_kj]
// which is the whole of Factor::conditioning (code/factor.cpp:214-242) here.  One launch
// per bucket for the entire batch; nothing is materialised per evidence set.
#include <algorithm>
#include <cstring>
#include <vector>

#include "batched.hpp"
#include "common.cuh"

namespace bnpp {

struct BOperand {
    const double *ptr;
    uint32_t batched;                       // 1: intermediate [entries][batch]; 0: resident CPT view
    uint32_t sx;                            // stride of the eliminated variable
    uint32_t nobs;
    uint32_t ostride[kMaxObsPerOperand];    // stride of an observed axis ...
    uint32_t oidx[kMaxObsPerOperand];       // ... and its column in the evidence matrix
};

struct BParams {
    BOperand op[kMaxK];
    double *out;                            // [n_out][nb]
    const uint8_t *ev;                      // [n_obs][ev_stride] evidence values, set index fastest (column of this slice)
    uint32_t ev_stride;
    uint32_t n_obs, nb, n_out, cx;
    uint32_t oc, n_chunks;                  // a thread walks `oc` consecutive output entries for its evidence sets
    const uint32_t *offtab;                 // [K][n_out] operand offset of output entry o (built by the plan, L1-resident)
    FastDiv nbdiv;
};

// the max-product variant (MPE): out = the maximum over the eliminated variable (start at x = 0, a later x replaces it
// only if its product is strictly greater -- contract.cu's rule), arg = [n_out][nb] bytes, the first maximising x
struct BMaxParams {
    BParams p;
    uint8_t *arg;
};

// A thread owns VB evidence sets (2 when the slice is even: 16-byte accesses on the batched
// tables) and walks `oc` consecutive output entries for them.  What depends only on the sets
// -- the evidence base of every resident CPT -- is computed once per thread, what depends only
// on the output entry -- operand offsets -- comes from a small table that a warp reads as one
// broadcast (all lanes share the entry, the batch being the fastest axis).
template <int K, int VB, bool MAX>
__device__ __forceinline__ void batched_entries(const BParams &p, uint8_t *arg)
{
    const uint32_t nbv = p.nb / VB;
    const uint64_t total = (uint64_t)p.n_chunks * nbv;
    const uint64_t step = (uint64_t)gridDim.x * kBlock;
    for (uint64_t idx = (uint64_t)blockIdx.x * kBlock + threadIdx.x; idx < total; idx += step) {
        uint32_t chunk, bv;
        if (nbv == 1) { chunk = (uint32_t)idx; bv = 0; }
        else if (total < (1ull << 32)) { chunk = fastdiv((uint32_t)idx, p.nbdiv); bv = (uint32_t)idx - chunk * nbv; }
        else { chunk = (uint32_t)(idx / nbv); bv = (uint32_t)(idx - (uint64_t)chunk * nbv); }
        const uint32_t b = bv * VB;
        const double *base[K][VB];
        uint64_t xs[K], os[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const BOperand &op = p.op[k];
            if (op.batched) {
                base[k][0] = op.ptr + b;
                if (VB == 2) base[k][VB - 1] = base[k][0] + 1;
                xs[k] = (uint64_t)op.sx * p.nb;
                os[k] = p.nb;
            } else {
                uint32_t e[VB];
#pragma unroll
                for (int v = 0; v < VB; ++v) e[v] = 0;
                for (uint32_t j = 0; j < op.nobs; ++j) {
                    const uint8_t *col = p.ev + (uint64_t)op.oidx[j] * p.ev_stride + b;   // neighbouring threads, neighbouring bytes
#pragma unroll
                    for (int v = 0; v < VB; ++v) e[v] += op.ostride[j] * col[v];
                }
#pragma unroll
                for (int v = 0; v < VB; ++v) base[k][v] = op.ptr + e[v];
                xs[k] = op.sx;
                os[k] = 1;
            }
        }
        const uint32_t o_end = min(p.n_out, (chunk + 1) * p.oc);
        for (uint32_t o = chunk * p.oc; o < o_end; ++o) {
            const double *src[K][VB];
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const uint64_t off = (uint64_t)__ldg(p.offtab + (uint64_t)k * p.n_out + o) * os[k];
#pragma unroll
                for (int v = 0; v < VB; ++v) src[k][v] = base[k][v] + off;
            }
            double acc[VB];
            uint32_t best[VB];
#pragma unroll
            for (int w = 0; w < VB; ++w) best[w] = 0;
            for (uint32_t x = 0; x < p.cx; ++x) {
                double v[VB];
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    double t[VB];
                    if (VB == 2 && p.op[k].batched) {
                        const double2 d2 = ld2(src[k][0] + x * xs[k]);
                        t[0] = d2.x;
                        t[VB - 1] = d2.y;
                    } else {
#pragma unroll
                        for (int w = 0; w < VB; ++w) t[w] = ld1(src[k][w] + x * xs[k]);
                    }
#pragma unroll
                    for (int w = 0; w < VB; ++w) v[w] = (k == 0) ? t[w] : __dmul_rn(v[w], t[w]);
                }
#pragma unroll
                for (int w = 0; w < VB; ++w) {
                    if (!MAX) {
                        acc[w] = (x == 0) ? v[w] : __dadd_rn(acc[w], v[w]);
                    } else if (x == 0 || v[w] > acc[w]) {
                        acc[w] = v[w];
                        best[w] = x;
                    }
                }
            }
            double *dst = p.out + ((uint64_t)o * p.nb + b);
            if (VB == 2) *reinterpret_cast<double2 *>(dst) = make_double2(acc[0], acc[VB - 1]);
            else dst[0] = acc[0];
            if (MAX) {
#pragma unroll
                for (int w = 0; w < VB; ++w) arg[(uint64_t)o * p.nb + b + w] = (uint8_t)best[w];
            }
        }
    }
}

template <int K, int VB>
__global__ void __launch_bounds__(kBlock) contract_batched(const __grid_constant__ BParams p)
{
    batched_entries<K, VB, false>(p, nullptr);
}

template <int K, int VB>
__global__ void __launch_bounds__(kBlock) contract_batched_max(const __grid_constant__ BMaxParams q)
{
    batched_entries<K, VB, true>(q.p, q.arg);
}

// Binary eliminated variable (every BASELINE network): UO output entries of a thread are
// processed together -- all their loads are issued before the first multiply, so one wave of
// CTAs moves UO times the bytes per memory round trip (the launch is a handful of waves long,
// each paying a full DRAM latency).
template <int K, int VB, int UO, bool MAX>
__device__ __forceinline__ void batched_bin_entries(const BParams &p, uint8_t *arg)
{
    const uint32_t nbv = p.nb / VB;
    const uint64_t total = (uint64_t)p.n_chunks * nbv;
    const uint64_t step = (uint64_t)gridDim.x * kBlock;
    for (uint64_t idx = (uint64_t)blockIdx.x * kBlock + threadIdx.x; idx < total; idx += step) {
        uint32_t chunk, bv;
        if (nbv == 1) { chunk = (uint32_t)idx; bv = 0; }
        else if (total < (1ull << 32)) { chunk = fastdiv((uint32_t)idx, p.nbdiv); bv = (uint32_t)idx - chunk * nbv; }
        else { chunk = (uint32_t)(idx / nbv); bv = (uint32_t)(idx - (uint64_t)chunk * nbv); }
        const uint32_t b = bv * VB;
        const double *base[K][VB];
        uint64_t xs[K], os[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const BOperand &op = p.op[k];
            if (op.batched) {
                base[k][0] = op.ptr + b;
                if (VB == 2) base[k][VB - 1] = base[k][0] + 1;
                xs[k] = (uint64_t)op.sx * p.nb;
                os[k] = p.nb;
            } else {
                uint32_t e[VB];
#pragma unroll
                for (int v = 0; v < VB; ++v) e[v] = 0;
                for (uint32_t j = 0; j < op.nobs; ++j) {
                    const uint8_t *col = p.ev + (uint64_t)op.oidx[j] * p.ev_stride + b;
#pragma unroll
                    for (int v = 0; v < VB; ++v) e[v] += op.ostride[j] * col[v];
                }
#pragma unroll
                for (int v = 0; v < VB; ++v) base[k][v] = op.ptr + e[v];
                xs[k] = op.sx;
                os[k] = 1;
            }
        }
        const uint32_t o_end = min(p.n_out, (chunk + 1) * p.oc);
        for (uint32_t o0 = chunk * p.oc; o0 < o_end; o0 += UO) {
            double t[UO][K][2][VB];
#pragma unroll
            for (int i = 0; i < UO; ++i) {
                const uint32_t o = min(o0 + i, o_end - 1);      // tail entries repeat the last one, their result is dropped
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    const uint64_t off = (uint64_t)__ldg(p.offtab + (uint64_t)k * p.n_out + o) * os[k];
#pragma unroll
                    for (int x = 0; x < 2; ++x) {
                        if (VB == 2 && p.op[k].batched) {
                            const double2 d2 = ld2(base[k][0] + off + x * xs[k]);
                            t[i][k][x][0] = d2.x;
                            t[i][k][x][VB - 1] = d2.y;
                        } else {
#pragma unroll
                            for (int w = 0; w < VB; ++w) t[i][k][x][w] = ld1(base[k][w] + off + x * xs[k]);
                        }
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < UO; ++i) {
                if (o0 + i >= o_end) break;
                double acc[VB];
#pragma unroll
                for (int w = 0; w < VB; ++w) {
                    double v0 = t[i][0][0][w], v1 = t[i][0][1][w];
#pragma unroll
                    for (int k = 1; k < K; ++k) {
                        v0 = __dmul_rn(v0, t[i][k][0][w]);
                        v1 = __dmul_rn(v1, t[i][k][1][w]);
                    }
                    if (MAX) {
                        const bool gt = v1 > v0;
                        acc[w] = gt ? v1 : v0;
                        arg[(uint64_t)(o0 + i) * p.nb + b + w] = (uint8_t)gt;
                    } else {
                        acc[w] = __dadd_rn(v0, v1);
                    }
                }
                double *dst = p.out + ((uint64_t)(o0 + i) * p.nb + b);
                if (VB == 2) *reinterpret_cast<double2 *>(dst) = make_double2(acc[0], acc[VB - 1]);
                else dst[0] = acc[0];
            }
        }
    }
}

template <int K, int VB, int UO>
__global__ void __launch_bounds__(kBlock) contract_batched_bin(const __grid_constant__ BParams p)
{
    batched_bin_entries<K, VB, UO, false>(p, nullptr);
}

template <int K, int VB, int UO>
__global__ void __launch_bounds__(kBlock) contract_batched_bin_max(const __grid_constant__ BMaxParams q)
{
    batched_bin_entries<K, VB, UO, true>(q.p, q.arg);
}

// [nb][n_obs] (one row per evidence set, as the caller has it) -> [n_obs][nb] (transpose != 0) or a copy in place
// order.  A value outside its variable's cardinality would move a CPT view past its table: it is replaced by 0 and
// BNPP_STATUS_BAD_EVIDENCE is raised (the reference throws from Factor::operator[] there, code/factor.cpp:83-95).
__global__ void sanitize_evidence(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, uint32_t nb, uint32_t n_obs,
                                  const uint32_t *__restrict__ card, int transpose, unsigned int *status)
{
    const uint64_t n = (uint64_t)nb * n_obs;
    bool bad = false;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t j, b;
        if (transpose) {
            j = (uint32_t)(i / nb);
            b = (uint32_t)(i - (uint64_t)j * nb);
        } else {
            b = (uint32_t)(i / n_obs);
            j = (uint32_t)(i - (uint64_t)b * n_obs);
        }
        uint8_t v = in[(uint64_t)b * n_obs + j];
        if (v >= card[j]) {
            bad = true;
            v = 0;
        }
        out[i] = v;
    }
    if (bad) atomicOr(status, BNPP_STATUS_BAD_EVIDENCE);
}

int sanitize_evidence_launch(bnpp_ctx *ctx, const uint8_t *in, uint8_t *out, uint32_t nb, uint32_t n_obs, const uint32_t *card_dev,
                             bool transpose)
{
    if (!nb || !n_obs) return BNPP_OK;
    const uint64_t n = (uint64_t)nb * n_obs;
    uint64_t blocks = (n + 255) / 256;
    if (blocks > 4096) blocks = 4096;
    sanitize_evidence<<<(unsigned)blocks, 256, 0, ctx->stream>>>(in, out, nb, n_obs, card_dev, transpose ? 1 : 0, ctx->status);
    BNPP_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return BNPP_OK;
}

// The evidence base of a CPT with more observed axes than a K8 operand holds, sum_j stride_j * value[obs_j], for
// every set: up to kMaxObsPerOperand axes per launch, added to `acc`; the last launch (digits != 0) writes the sum as
// `digits` base-256 digits into the evidence columns digit_col, digit_col + 1, ... of the column-major matrix `ev`.
struct ObsAxes {
    uint32_t n;
    uint32_t stride[kMaxObsPerOperand];
    uint32_t col[kMaxObsPerOperand];
};

__global__ void evidence_digits(const __grid_constant__ ObsAxes a, uint8_t *ev, uint32_t nb, uint32_t *__restrict__ acc, int first,
                                uint32_t digit_col, uint32_t digits)
{
    for (uint32_t b = blockIdx.x * blockDim.x + threadIdx.x; b < nb; b += gridDim.x * blockDim.x) {
        uint32_t e = first ? 0 : acc[b];
        for (uint32_t j = 0; j < a.n; ++j) e += a.stride[j] * ev[(uint64_t)a.col[j] * nb + b];
        if (!digits) acc[b] = e;
        for (uint32_t d = 0; d < digits; ++d) ev[(uint64_t)(digit_col + d) * nb + b] = (uint8_t)(e >> (8 * d));
    }
}

int evidence_digits_launch(bnpp_ctx *ctx, const std::vector<std::pair<int64_t, int>> &obs, uint8_t *ev_dev, uint32_t nb,
                           uint32_t digit_col, uint32_t digits)
{
    if (!nb || obs.empty() || !digits) return BNPP_OK;
    double *acc = nullptr;
    if (obs.size() > (size_t)kMaxObsPerOperand) {
        const int rc = bnpp_alloc(ctx, nb / 2 + 1, &acc);
        if (rc != BNPP_OK) return rc;
    }
    const unsigned blocks = (unsigned)std::min<uint64_t>((nb + 255) / 256, 4096);
    for (size_t j0 = 0; j0 < obs.size(); j0 += kMaxObsPerOperand) {
        ObsAxes a;
        memset(&a, 0, sizeof a);
        a.n = (uint32_t)std::min<size_t>(kMaxObsPerOperand, obs.size() - j0);
        for (uint32_t j = 0; j < a.n; ++j) {
            a.stride[j] = (uint32_t)obs[j0 + j].first;
            a.col[j] = (uint32_t)obs[j0 + j].second;
        }
        const bool last = j0 + a.n == obs.size();
        evidence_digits<<<blocks, 256, 0, ctx->stream>>>(a, ev_dev, nb, reinterpret_cast<uint32_t *>(acc), j0 == 0, digit_col,
                                                         last ? digits : 0);
        BNPP_CUDA(ctx, cudaGetLastError());
        ctx->launches++;
    }
    return bnpp_free(ctx, acc);
}

typedef void (*batched_fn)(const BParams);
typedef void (*batched_max_fn)(const BMaxParams);

template <int VB>
static batched_fn pick_batched_bin(int K, int &uo)
{
    switch (K) {
    case 1: uo = 4; return contract_batched_bin<1, VB, 4>;
    case 2: uo = 4; return contract_batched_bin<2, VB, 4>;
    case 3: uo = 2; return contract_batched_bin<3, VB, 2>;
    case 4: uo = 2; return contract_batched_bin<4, VB, 2>;
    default: uo = 0; return nullptr;
    }
}

template <int VB>
static batched_fn pick_batched_v(int K)
{
    switch (K) {
    case 1: return contract_batched<1, VB>;
    case 2: return contract_batched<2, VB>;
    case 3: return contract_batched<3, VB>;
    case 4: return contract_batched<4, VB>;
    case 5: return contract_batched<5, VB>;
    default: return contract_batched<6, VB>;
    }
}

template <int VB>
static batched_max_fn pick_batched_bin_max(int K, int &uo)
{
    switch (K) {
    case 1: uo = 4; return contract_batched_bin_max<1, VB, 4>;
    case 2: uo = 4; return contract_batched_bin_max<2, VB, 4>;
    case 3: uo = 2; return contract_batched_bin_max<3, VB, 2>;
    case 4: uo = 2; return contract_batched_bin_max<4, VB, 2>;
    default: uo = 0; return nullptr;
    }
}

template <int VB>
static batched_max_fn pick_batched_v_max(int K)
{
    switch (K) {
    case 1: return contract_batched_max<1, VB>;
    case 2: return contract_batched_max<2, VB>;
    case 3: return contract_batched_max<3, VB>;
    case 4: return contract_batched_max<4, VB>;
    case 5: return contract_batched_max<5, VB>;
    default: return contract_batched_max<6, VB>;
    }
}

int contract_batched_step(bnpp_ctx *ctx, int k, const BatchedOperandDesc *ops, const std::vector<uint32_t> &out_var,
                          const std::vector<uint32_t> &out_card, int64_t elim, uint32_t nb, const uint8_t *ev_dev,
                          uint32_t ev_stride, uint32_t n_obs, double *out_dev, std::vector<uint32_t> *offtab_host,
                          uint32_t **offtab_dev, uint8_t *arg_dev)
{
    if (k < 1 || k > kMaxK) return fail(ctx, BNPP_ERANK, "batched step: operand count");
    BParams p;
    memset(&p, 0, sizeof p);
    const int wr = (int)out_var.size();
    struct Ax { uint32_t ext; uint64_t s[kMaxK]; };
    std::vector<Ax> axes(wr);
    uint64_t n_out = 1;
    for (int i = wr - 1; i >= 0; --i) {
        axes[i].ext = out_card[i];
        for (int q = 0; q < kMaxK; ++q) axes[i].s[q] = 0;
        n_out *= out_card[i];
    }
    if (n_out >= (1ull << 32)) return fail(ctx, BNPP_ETOOBIG, "batched step: output too large");
    uint32_t cx = 1;
    for (int q = 0; q < k; ++q) {
        const BatchedOperandDesc &op = ops[q];
        uint64_t dense = 1;
        for (int i = (int)op.var->size() - 1; i >= 0; --i) {
            const uint64_t st = op.stride->empty() ? dense : (uint64_t)(*op.stride)[i];
            dense *= (*op.card)[i];
            if (elim >= 0 && (*op.var)[i] == (uint64_t)elim) {
                p.op[q].sx = (uint32_t)st;
                cx = (*op.card)[i];
                continue;
            }
            int pos = -1;
            for (int j = 0; j < wr; ++j)
                if (out_var[j] == (*op.var)[i]) { pos = j; break; }
            if (pos < 0) return fail(ctx, BNPP_EINVAL, "batched step: operand variable not in the output");
            axes[pos].s[q] = st;
        }
        p.op[q].ptr = op.ptr;
        p.op[q].batched = op.batched ? 1 : 0;
        if (op.obs->size() > (size_t)kMaxObsPerOperand) return fail(ctx, BNPP_ERANK, "batched step: too many observed axes in one table");
        p.op[q].nobs = (uint32_t)op.obs->size();
        for (size_t j = 0; j < op.obs->size(); ++j) {
            p.op[q].ostride[j] = (uint32_t)(*op.obs)[j].first;
            p.op[q].oidx[j] = (uint32_t)(*op.obs)[j].second;
        }
    }
    // operand offset of every output entry (row-major odometer over the output axes)
    std::vector<uint32_t> &tab = *offtab_host;
    if (tab.empty()) {
        tab.assign((size_t)k * n_out, 0);
        std::vector<uint32_t> digit(wr, 0);
        for (uint64_t o = 0; o < n_out; ++o) {
            for (int q = 0; q < k; ++q) {
                uint64_t off = 0;
                for (int i = 0; i < wr; ++i) off += (uint64_t)digit[i] * axes[i].s[q];
                tab[(size_t)q * n_out + o] = (uint32_t)off;
            }
            for (int i = wr - 1; i >= 0; --i) {
                if (++digit[i] < axes[i].ext) break;
                digit[i] = 0;
            }
        }
    }
    if (!*offtab_dev) {
        double *store = nullptr;
        const int rc = bnpp_alloc(ctx, (tab.size() + 1) / 2 + 1, &store);
        if (rc != BNPP_OK) return rc;
        *offtab_dev = reinterpret_cast<uint32_t *>(store);
        BNPP_CUDA(ctx, cudaMemcpyAsync(*offtab_dev, tab.data(), tab.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    }
    p.offtab = *offtab_dev;
    p.out = out_dev;
    p.ev = ev_dev;
    p.ev_stride = ev_stride;
    p.n_obs = n_obs;
    p.nb = nb;
    p.n_out = (uint32_t)n_out;
    p.cx = cx;
    // two sets per thread when every batched table keeps 16-byte alignment: even slice, aligned bases
    int vb = (nb % 2 == 0 && reinterpret_cast<uintptr_t>(out_dev) % 16 == 0) ? 2 : 1;
    for (int q = 0; q < k && vb == 2; ++q)
        if (ops[q].batched && reinterpret_cast<uintptr_t>(ops[q].ptr) % 16 != 0) vb = 1;
    p.nbdiv = make_fastdiv(nb / vb > 1 ? nb / vb : 2);
    // binary eliminated variable with at most 4 operands: the unrolled variant
    int uo = 0;
    batched_fn fn = nullptr;
    batched_max_fn fn_max = nullptr;
    const bool max_mode = arg_dev && elim >= 0;
    if (max_mode) {
        if (cx == 2) fn_max = (vb == 2) ? pick_batched_bin_max<2>(k, uo) : pick_batched_bin_max<1>(k, uo);
        if (!fn_max) fn_max = (vb == 2) ? pick_batched_v_max<2>(k) : pick_batched_v_max<1>(k);
    } else {
        if (cx == 2) fn = (vb == 2) ? pick_batched_bin<2>(k, uo) : pick_batched_bin<1>(k, uo);
        if (!fn) fn = (vb == 2) ? pick_batched_v<2>(k) : pick_batched_v<1>(k);
    }
    // about one resident wave of threads, each walking `oc` consecutive output entries
    const uint64_t want_threads = (uint64_t)ctx->sm_count * (uo ? 768 : 2048);
    uint64_t oc = (n_out * (nb / vb) + want_threads - 1) / want_threads;
    if (oc < 1) oc = 1;
    if (uo && oc < (uint64_t)uo && n_out >= (uint64_t)uo) oc = uo;
    if (oc > 32) oc = 32;
    p.oc = (uint32_t)oc;
    p.n_chunks = (uint32_t)((n_out + oc - 1) / oc);
    const uint64_t total = (uint64_t)p.n_chunks * (nb / vb);
    uint64_t blocks = (total + kBlock - 1) / kBlock;
    const uint64_t cap = (uint64_t)ctx->sm_count * 8;
    if (blocks > cap) blocks = cap;
    if (max_mode) {
        BMaxParams q;
        q.p = p;
        q.arg = arg_dev;
        fn_max<<<(unsigned)blocks, kBlock, 0, ctx->stream>>>(q);
    } else {
        fn<<<(unsigned)blocks, kBlock, 0, ctx->stream>>>(p);
    }
    BNPP_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return BNPP_OK;
}

}  // namespace bnpp
