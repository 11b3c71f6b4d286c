// extern "C" entry points of include/bnpp_b200.h: context, memory and the
// reference-shaped single ops, all thin wrappers over the contraction engine.
#include <cstdio>
#include <cstring>
#include <vector>

#include "common.cuh"
#include "contract.hpp"

namespace bnpp {
int contract(bnpp_ctx *ctx, int k, const bnpp_operand *ops, const bnpp_scope *out_scope, int64_t elim_var, int divide,
             double *out_dev, double *z_dev, bool max_mode = false, uint8_t *arg_dev = nullptr);
int normalize(bnpp_ctx *ctx, uint64_t n, const double *in, const double *z_dev, double z_host, double *out);
int reduce(bnpp_ctx *ctx, int op, uint64_t n, const double *in, double init, double *result);
int fill(bnpp_ctx *ctx, double *out, uint64_t n, double value);

int fail(bnpp_ctx *ctx, int code, const std::string &msg)
{
    if (ctx) ctx->last_error = msg;
    return code;
}

int stage_upload(bnpp_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes)
{
    if (!bytes) return BNPP_OK;
    const size_t need = (bytes + 255) & ~(size_t)255;
    if (!ctx->stage || need > ctx->stage_bytes) {
        // no ring, or a table larger than the ring: the (synchronising) copy from pageable memory
        BNPP_CUDA(ctx, cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
        return BNPP_OK;
    }
    if (ctx->stage_off + need > ctx->stage_bytes) {
        BNPP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));      // every earlier copy out of the ring is done: wrap around
        ctx->stage_off = 0;
    }
    memcpy(ctx->stage + ctx->stage_off, src_host, bytes);
    BNPP_CUDA(ctx, cudaMemcpyAsync(dst_dev, ctx->stage + ctx->stage_off, bytes, cudaMemcpyHostToDevice, ctx->stream));
    ctx->stage_off += need;
    return BNPP_OK;
}

// A contiguous piece of the pinned ring to be filled IN PLACE (nullptr: no ring, or it does not fit) -- for data that
// is gathered from many small host buffers: gathering it into a fresh pageable vector first pays a page fault per 4 KB.
// The caller copies out of it with cudaMemcpyAsync on ctx->stream.
void *stage_reserve(bnpp_ctx *ctx, size_t bytes)
{
    const size_t need = (bytes + 255) & ~(size_t)255;
    if (!ctx->stage || !bytes || need > ctx->stage_bytes) return nullptr;
    if (ctx->stage_off + need > ctx->stage_bytes) {
        if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return nullptr;
        ctx->stage_off = 0;
    }
    void *p = ctx->stage + ctx->stage_off;
    ctx->stage_off += need;
    return p;
}

int cuda_fail(bnpp_ctx *ctx, cudaError_t e, const char *what)
{
    if (ctx) ctx->last_error = std::string(what) + ": " + cudaGetErrorString(e);
    return BNPP_ECUDA;
}
}  // namespace bnpp

using namespace bnpp;

static std::string g_create_error;

extern "C" {

int bnpp_version(void) { return 100; }

int bnpp_ctx_create(int device, void *stream, bnpp_ctx **out)
{
    if (!out) return BNPP_EINVAL;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0 || device < 0 || device >= count) {
        g_create_error = std::string("no usable CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "bad ordinal");
        fprintf(stderr, "bnpp_b200: %s (this library has no CPU fallback)\n", g_create_error.c_str());
        return BNPP_ECUDA;
    }
    bnpp_ctx *ctx = new bnpp_ctx();
    ctx->device = device;
    BNPP_CUDA(ctx, cudaSetDevice(device));
    if (stream) {
        ctx->stream = static_cast<cudaStream_t>(stream);
    } else {
        BNPP_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        ctx->own_stream = true;
    }
    cudaDeviceProp prop;
    BNPP_CUDA(ctx, cudaGetDeviceProperties(&prop, device));
    ctx->sm_count = prop.multiProcessorCount;
    BNPP_CUDA(ctx, cudaDeviceGetDefaultMemPool(&ctx->pool, device));
    uint64_t keep = UINT64_MAX;   // keep freed blocks cached: VE allocates and frees a table per step
    BNPP_CUDA(ctx, cudaMemPoolSetAttribute(ctx->pool, cudaMemPoolAttrReleaseThreshold, &keep));
    BNPP_CUDA(ctx, cudaMalloc(&ctx->partials, sizeof(double) * kMaxPartials));
    BNPP_CUDA(ctx, cudaMalloc(&ctx->ticket, 64));
    BNPP_CUDA(ctx, cudaMemset(ctx->ticket, 0, 64));
    ctx->status = ctx->ticket + 4;
    ctx->stage_bytes = 4u << 20;
    if (cudaHostAlloc(reinterpret_cast<void **>(&ctx->stage), ctx->stage_bytes, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        ctx->stage = nullptr;
        ctx->stage_bytes = 0;
    }
    *out = ctx;
    return BNPP_OK;
}

int bnpp_ctx_destroy(bnpp_ctx *ctx)
{
    if (!ctx) return BNPP_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaFree(ctx->partials);
    cudaFree(ctx->ticket);
    if (ctx->stage) cudaFreeHost(ctx->stage);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return BNPP_OK;
}

int bnpp_ctx_sync(bnpp_ctx *ctx)
{
    if (!ctx) return BNPP_EINVAL;
    BNPP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return BNPP_OK;
}

int bnpp_ctx_status(bnpp_ctx *ctx, uint32_t *status_bits, int clear)
{
    if (!ctx || !status_bits) return BNPP_EINVAL;
    BNPP_CUDA(ctx, cudaMemcpyAsync(status_bits, ctx->status, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (clear) BNPP_CUDA(ctx, cudaMemsetAsync(ctx->status, 0, sizeof(uint32_t), ctx->stream));
    BNPP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return BNPP_OK;
}

const char *bnpp_last_error(const bnpp_ctx *ctx) { return ctx ? ctx->last_error.c_str() : g_create_error.c_str(); }

uint64_t bnpp_launch_count(const bnpp_ctx *ctx) { return ctx ? ctx->launches : 0; }

int bnpp_last_launch(const bnpp_ctx *ctx, char *name, size_t name_len, uint32_t *grid, uint32_t *block)
{
    if (!ctx) return BNPP_EINVAL;
    if (name && name_len) {
        // valid right after the launch it describes (one-shot descriptors live on the caller's stack)
        const std::string nm = !ctx->last_kernel.empty() ? ctx->last_kernel
                               : (ctx->last_desc ? static_cast<bnpp::LaunchDesc *>(ctx->last_desc)->name() : std::string());
        strncpy(name, nm.c_str(), name_len - 1);
        name[name_len - 1] = 0;
    }
    if (grid) *grid = ctx->last_grid;
    if (block) *block = ctx->last_block;
    return BNPP_OK;
}

int bnpp_alloc(bnpp_ctx *ctx, uint64_t n_doubles, double **dptr)
{
    if (!ctx || !dptr) return BNPP_EINVAL;
    void *p = nullptr;
    cudaError_t e = cudaMallocAsync(&p, sizeof(double) * (n_doubles ? n_doubles : 1), ctx->stream);
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        return fail(ctx, BNPP_ENOMEM, "out of device memory");
    }
    BNPP_CUDA(ctx, e);
    *dptr = static_cast<double *>(p);
    return BNPP_OK;
}

int bnpp_free(bnpp_ctx *ctx, double *dptr)
{
    if (!ctx) return BNPP_EINVAL;
    if (dptr) BNPP_CUDA(ctx, cudaFreeAsync(dptr, ctx->stream));
    return BNPP_OK;
}

int bnpp_upload(bnpp_ctx *ctx, double *dst_dev, const double *src_host, uint64_t n)
{
    if (!ctx) return BNPP_EINVAL;
    BNPP_CUDA(ctx, cudaMemcpyAsync(dst_dev, src_host, sizeof(double) * n, cudaMemcpyHostToDevice, ctx->stream));
    return BNPP_OK;
}

int bnpp_download(bnpp_ctx *ctx, double *dst_host, const double *src_dev, uint64_t n)
{
    if (!ctx) return BNPP_EINVAL;
    BNPP_CUDA(ctx, cudaMemcpyAsync(dst_host, src_dev, sizeof(double) * n, cudaMemcpyDeviceToHost, ctx->stream));
    BNPP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return BNPP_OK;
}

int bnpp_fill(bnpp_ctx *ctx, double *dst_dev, uint64_t n, double value)
{
    if (!ctx) return BNPP_EINVAL;
    return fill(ctx, dst_dev, n, value);
}

int bnpp_union_scope(const bnpp_scope *a, const bnpp_scope *b, uint32_t *out_var_id, uint32_t *out_card)
{
    if (!a || !b || !out_var_id || !out_card) return BNPP_EINVAL;
    int w = 0;
    for (int i = 0; i < a->rank; ++i) {
        out_var_id[w] = a->var_id[i];
        out_card[w++] = a->card[i];
    }
    for (int i = 0; i < b->rank; ++i) {
        bool seen = false;
        for (int j = 0; j < a->rank && !seen; ++j) seen = (a->var_id[j] == b->var_id[i]);
        if (!seen) {
            out_var_id[w] = b->var_id[i];
            out_card[w++] = b->card[i];
        }
    }
    return w;
}

uint64_t bnpp_scope_size(const bnpp_scope *s)
{
    if (!s) return 0;
    unsigned __int128 n = 1;
    for (int i = 0; i < s->rank; ++i) {
        n *= s->card[i];
        if (n >> 64) return 0;
    }
    return (uint64_t)n;
}

int bnpp_product_sum_out(bnpp_ctx *ctx, int k, const bnpp_operand *operands, const bnpp_scope *out_scope,
                         int64_t elim_var, int divide, double *out_dev, double *z_dev)
{
    return contract(ctx, k, operands, out_scope, elim_var, divide, out_dev, z_dev);
}

int bnpp_product_max_out(bnpp_ctx *ctx, int k, const bnpp_operand *operands, const bnpp_scope *out_scope,
                         int64_t elim_var, double *out_dev, uint8_t *argmax_dev)
{
    return contract(ctx, k, operands, out_scope, elim_var, 0, out_dev, nullptr, true, argmax_dev);
}

int bnpp_product(bnpp_ctx *ctx, const bnpp_scope *sa, const double *a_dev, const bnpp_scope *sb, const double *b_dev,
                 int divide, double *out_dev, double *z_dev)
{
    if (!ctx || !sa || !sb) return BNPP_EINVAL;
    if (sa->rank < 0 || sb->rank < 0 || sa->rank > BNPP_MAX_RANK || sb->rank > BNPP_MAX_RANK)
        return fail(ctx, BNPP_EINVAL, "bad scope rank");
    uint32_t ids[2 * BNPP_MAX_RANK], cards[2 * BNPP_MAX_RANK];
    bnpp_scope u;
    u.rank = bnpp_union_scope(sa, sb, ids, cards);
    if (u.rank > BNPP_MAX_RANK) return fail(ctx, BNPP_EINVAL, "union scope wider than BNPP_MAX_RANK");
    u.var_id = ids;
    u.card = cards;
    bnpp_operand ops[2] = {{a_dev, *sa, nullptr}, {b_dev, *sb, nullptr}};
    return contract(ctx, 2, ops, &u, -1, divide, out_dev, z_dev);
}

int bnpp_sum_out(bnpp_ctx *ctx, const bnpp_scope *s, const double *in_dev, uint32_t var, double *out_dev, double *z_dev)
{
    if (!ctx || !s) return BNPP_EINVAL;
    if (s->rank < 0 || s->rank > BNPP_MAX_RANK) return fail(ctx, BNPP_EINVAL, "bad scope rank");
    uint32_t ids[BNPP_MAX_RANK], cards[BNPP_MAX_RANK];
    bnpp_scope o;
    o.rank = 0;
    for (int i = 0; i < s->rank; ++i) {
        if (s->var_id[i] == var) continue;
        ids[o.rank] = s->var_id[i];
        cards[o.rank++] = s->card[i];
    }
    o.var_id = ids;
    o.card = cards;
    bnpp_operand op = {in_dev, *s, nullptr};
    // var not in scope: o == s and the contraction degenerates to a copy (code/factor.cpp:185-188)
    return contract(ctx, 1, &op, &o, (int64_t)var, 0, out_dev, z_dev);
}

int bnpp_condition(bnpp_ctx *ctx, const bnpp_scope *s, const double *in_dev, int n_ev, const uint32_t *ev_var,
                   const uint32_t *ev_val, double *out_dev, double *z_dev)
{
    if (!ctx || !s || n_ev < 0) return BNPP_EINVAL;
    if (s->rank < 0 || s->rank > BNPP_MAX_RANK) return fail(ctx, BNPP_EINVAL, "bad scope rank");
    // evidence slice = strided view: observed axes vanish, their offset moves into the base pointer
    uint32_t ids[BNPP_MAX_RANK], cards[BNPP_MAX_RANK];
    int64_t strides[BNPP_MAX_RANK];
    bnpp_scope o;
    o.rank = 0;
    uint64_t base = 0, dense = 1;
    for (int i = s->rank - 1; i >= 0; --i) {
        int hit = -1;
        for (int e = 0; e < n_ev; ++e)
            if (ev_var[e] == s->var_id[i]) hit = e;   // last assignment wins, as in an unordered_map
        if (hit >= 0) {
            if (ev_val[hit] >= s->card[i]) return fail(ctx, BNPP_EINVAL, "evidence value out of range");
            base += dense * ev_val[hit];
        }
        dense *= s->card[i];
    }
    dense = 1;
    std::vector<int64_t> full(s->rank);
    for (int i = s->rank - 1; i >= 0; --i) {
        full[i] = (int64_t)dense;
        dense *= s->card[i];
    }
    for (int i = 0; i < s->rank; ++i) {
        bool obs = false;
        for (int e = 0; e < n_ev && !obs; ++e) obs = (ev_var[e] == s->var_id[i]);
        if (obs) continue;
        ids[o.rank] = s->var_id[i];
        cards[o.rank] = s->card[i];
        strides[o.rank++] = full[i];
    }
    o.var_id = ids;
    o.card = cards;
    bnpp_operand op = {in_dev + base, o, strides};
    return contract(ctx, 1, &op, &o, -1, 0, out_dev, z_dev);
}

int bnpp_normalize(bnpp_ctx *ctx, uint64_t n, const double *in_dev, const double *z_dev, double z_host, double *out_dev)
{
    if (!ctx) return BNPP_EINVAL;
    return normalize(ctx, n, in_dev, z_dev, z_host, out_dev);
}

int bnpp_reduce(bnpp_ctx *ctx, int op, uint64_t n, const double *in_dev, double init, double *result_dev)
{
    if (!ctx) return BNPP_EINVAL;
    return reduce(ctx, op, n, in_dev, init, result_dev);
}

}  // extern "C"
