// K5 normalize, K6 reduce (sum / max / min), fill -- streaming, HBM-bound helpers.
#include "common.cuh"

namespace bnpp {

// Factor::normalize (reference code/factor.cpp:244-255): TRUE division by the cached
// partition, so Z = 0 gives NaN/inf exactly as the reference does.
__global__ void __launch_bounds__(kBlock) normalize_kernel(const double *__restrict__ in, double *__restrict__ out,
                                                           uint64_t n, const double *__restrict__ z_dev, double z_host,
                                                           int vec)
{
    const double z = z_dev ? *z_dev : z_host;
    const uint64_t step = (uint64_t)gridDim.x * kBlock;
    const uint64_t tid = (uint64_t)blockIdx.x * kBlock + threadIdx.x;
    if (vec) {
        const uint64_t n2 = n / 2;
        for (uint64_t i = tid; i < n2; i += step) {
            double2 v = ld2(in + 2 * i);
            v.x = v.x / z;
            v.y = v.y / z;
            *reinterpret_cast<double2 *>(out + 2 * i) = v;
        }
        if (tid == 0 && (n & 1)) out[n - 1] = in[n - 1] / z;
    } else {
        for (uint64_t i = tid; i < n; i += step) out[i] = in[i] / z;
    }
}

// op 0: sum; op 1: max starting from 0.0 (code/factor.cpp:97-105);
// op 2: min starting from `init` = the partition (code/factor.cpp:107-115).
// Comparisons are the reference's strict `>` / `<`, so NaN entries never win.
__global__ void __launch_bounds__(kBlock) reduce_kernel(const double *__restrict__ in, uint64_t n, int op, double init,
                                                        double *partials, unsigned int *ticket, double *result)
{
    const uint64_t step = (uint64_t)gridDim.x * kBlock;
    double acc = (op == 0) ? 0.0 : (op == 1 ? 0.0 : init);
    for (uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x; i < n; i += step) {
        const double v = ld1(in + i);
        if (op == 0) acc += v;
        else if (op == 1) { if (v > acc) acc = v; }
        else { if (v < acc) acc = v; }
    }
    if (op == 0) {
        grid_sum_to(acc, partials, ticket, result);
        return;
    }
    __shared__ double s_w[kBlock / 32];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    auto better = [op](double a, double b) { return op == 1 ? (b > a ? b : a) : (b < a ? b : a); };
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc = better(acc, __shfl_down_sync(0xffffffffu, acc, o));
    if (lane == 0) s_w[w] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double b = s_w[0];
        for (int i = 1; i < kBlock / 32; ++i) b = better(b, s_w[i]);
        partials[blockIdx.x] = b;
        __threadfence();
        s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        __threadfence();
        double b = __ldcg(partials);
        for (unsigned i = 1; i < gridDim.x; ++i) b = better(b, __ldcg(partials + i));
        *result = b;
        *ticket = 0;
    }
}

__global__ void __launch_bounds__(kBlock) fill_kernel(double *out, uint64_t n, double value)
{
    const uint64_t step = (uint64_t)gridDim.x * kBlock;
    for (uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x; i < n; i += step) out[i] = value;
}

// Factor::normalize for many small tables at once (the marginals of every variable, each a
// slice of one buffer): Z summed in index order like the reference's `partition +=`, then the
// same true division (code/factor.cpp:244-255).  A one-entry slice is the reference's width-0
// factor [1] of an observed variable (code/model.cpp:333 on a scalar VE result).
__global__ void normalize_segments_kernel(double *buf, const uint32_t *__restrict__ off, const uint32_t *__restrict__ size, int n)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    double *p = buf + off[s];
    const uint32_t m = size[s];
    if (m == 1) {
        p[0] = 1.0;
        return;
    }
    double z = 0.0;
    for (uint32_t i = 0; i < m; ++i) z = __dadd_rn(z, p[i]);
    for (uint32_t i = 0; i < m; ++i) p[i] = __ddiv_rn(p[i], z);
}

int normalize_segments(bnpp_ctx *ctx, double *buf, const uint32_t *off_dev, const uint32_t *size_dev, int n)
{
    if (n <= 0) return BNPP_OK;
    normalize_segments_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(buf, off_dev, size_dev, n);
    BNPP_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return BNPP_OK;
}

// normalize_segments_kernel for a batch laid out [entries][nb] (batch fastest): one thread per (slice, set), the same
// index-order sum and true division, so every set's column gets the bits of its own single run.  Neighbouring
// threads are neighbouring sets of one slice: every read and write of a warp is one contiguous run.
__global__ void normalize_segments_batched_kernel(double *buf, const uint32_t *__restrict__ off, const uint32_t *__restrict__ size,
                                                  uint64_t n_items, uint32_t nb)
{
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_items) return;
    const uint32_t s = (uint32_t)(t / nb);
    double *p = buf + (uint64_t)off[s] * nb + (t - (uint64_t)s * nb);
    const uint32_t m = size[s];
    if (m == 1) {
        p[0] = 1.0;
        return;
    }
    double z = 0.0;
    for (uint32_t i = 0; i < m; ++i) z = __dadd_rn(z, p[(uint64_t)i * nb]);
    for (uint32_t i = 0; i < m; ++i) p[(uint64_t)i * nb] = __ddiv_rn(p[(uint64_t)i * nb], z);
}

int normalize_segments_batched(bnpp_ctx *ctx, double *buf, const uint32_t *off_dev, const uint32_t *size_dev, int n, uint32_t nb)
{
    if (n <= 0 || nb == 0) return BNPP_OK;
    const uint64_t items = (uint64_t)n * nb;
    if ((items + 127) / 128 > 0x7fffffffull) return fail(ctx, BNPP_ETOOBIG, "batched marginals: too many slices x sets");
    normalize_segments_batched_kernel<<<(unsigned)((items + 127) / 128), 128, 0, ctx->stream>>>(buf, off_dev, size_dev, items, nb);
    BNPP_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return BNPP_OK;
}

static unsigned grid_for(bnpp_ctx *ctx, uint64_t n_items)
{
    uint64_t b = (n_items + kBlock - 1) / kBlock;
    const uint64_t cap = (uint64_t)ctx->sm_count * 8;
    if (b > cap) b = cap;
    return (unsigned)(b < 1 ? 1 : b);
}

int normalize(bnpp_ctx *ctx, uint64_t n, const double *in, const double *z_dev, double z_host, double *out)
{
    const int vec = ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) % 16 == 0) && n >= 2;
    normalize_kernel<<<grid_for(ctx, vec ? n / 2 : n), kBlock, 0, ctx->stream>>>(in, out, n, z_dev, z_host, vec);
    BNPP_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return BNPP_OK;
}

int reduce(bnpp_ctx *ctx, int op, uint64_t n, const double *in, double init, double *result)
{
    if (op < 0 || op > 2) return fail(ctx, BNPP_EINVAL, "reduce: op must be 0 (sum), 1 (max) or 2 (min)");
    reduce_kernel<<<grid_for(ctx, n), kBlock, 0, ctx->stream>>>(in, n, op, init, ctx->partials, ctx->ticket, result);
    BNPP_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return BNPP_OK;
}

int fill(bnpp_ctx *ctx, double *out, uint64_t n, double value)
{
    fill_kernel<<<grid_for(ctx, n), kBlock, 0, ctx->stream>>>(out, n, value);
    BNPP_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return BNPP_OK;
}

}  // namespace bnpp
