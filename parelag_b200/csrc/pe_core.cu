// pe_core.cu -- context, vectors, matrix upload/download, halo exchange, CUDA graphs.
#include "pe_core.cuh"
#include "pe_stream.cuh"
#include <dlfcn.h>
#include <atomic>
#include <cstring>
#include <cstdio>

static thread_local std::string g_last_error;
void pe_set_error(const std::string &msg) { g_last_error = msg; }
extern "C" const char *pe_last_error(void) { return g_last_error.c_str(); }

// ---------------------------------------------------------------------------
// NCCL, resolved at run time so that a single-GPU process never needs it and a
// torch process reuses the libnccl.so.2 torch already mapped.
// ---------------------------------------------------------------------------
typedef struct { char internal[128]; } pe_ncclUniqueId;
typedef int (*fn_ncclGetUniqueId)(pe_ncclUniqueId *);
typedef int (*fn_ncclCommInitRank)(void **, int, pe_ncclUniqueId, int);
typedef int (*fn_ncclCommDestroy)(void *);
typedef int (*fn_ncclSend)(const void *, size_t, int, int, void *, cudaStream_t);
typedef int (*fn_ncclRecv)(void *, size_t, int, int, void *, cudaStream_t);
typedef int (*fn_ncclGroup)(void);
typedef int (*fn_ncclAllReduce)(const void *, void *, size_t, int, int, void *, cudaStream_t);
typedef const char *(*fn_ncclGetErrorString)(int);
static struct {
    void *h = nullptr;
    fn_ncclGetUniqueId GetUniqueId;
    fn_ncclCommInitRank CommInitRank;
    fn_ncclCommDestroy CommDestroy;
    fn_ncclSend Send;
    fn_ncclRecv Recv;
    fn_ncclGroup GroupStart, GroupEnd;
    fn_ncclAllReduce AllReduce;
    fn_ncclGetErrorString GetErrorString;
} g_nccl;
static const int PE_NCCL_FLOAT64 = 8; // ncclDouble
static const int PE_NCCL_SUM = 0;

static int nccl_load()
{
    if (g_nccl.h) return 0;
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char *n : names) {
        g_nccl.h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (g_nccl.h) break;
    }
    PE_CHECK(g_nccl.h, "cannot dlopen libnccl.so.2 (needed for nranks > 1)");
#define LD(sym) g_nccl.sym = (fn_nccl##sym)dlsym(g_nccl.h, "nccl" #sym); \
    PE_CHECK(g_nccl.sym, "missing NCCL symbol nccl" #sym)
    LD(GetUniqueId); LD(CommInitRank); LD(CommDestroy); LD(Send); LD(Recv);
    LD(AllReduce); LD(GetErrorString);
    g_nccl.GroupStart = (fn_ncclGroup)dlsym(g_nccl.h, "ncclGroupStart");
    g_nccl.GroupEnd = (fn_ncclGroup)dlsym(g_nccl.h, "ncclGroupEnd");
    PE_CHECK(g_nccl.GroupStart && g_nccl.GroupEnd, "missing ncclGroupStart/End");
#undef LD
    return 0;
}
#define PE_NCCL(call)                                                              \
    do {                                                                           \
        int r_ = (call);                                                           \
        if (r_ != 0) {                                                             \
            pe_set_error(std::string(#call) + " failed: " + g_nccl.GetErrorString(r_)); \
            return 3;                                                              \
        }                                                                          \
    } while (0)

extern "C" int pe_nccl_get_unique_id(void *id128)
{
    PE_TRY(nccl_load());
    pe_ncclUniqueId id;
    PE_NCCL(g_nccl.GetUniqueId(&id));
    memcpy(id128, &id, 128);
    return 0;
}

// ---------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------
extern "C" int pe_ctx_create(int rank, int nranks, int device, const void *nccl_unique_id,
                             pe_ctx **out)
{
    PE_CHECK(out, "null out pointer");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        pe_set_error(std::string("no CUDA device available (there is no CPU fallback): ")
                     + cudaGetErrorString(e));
        return 1;
    }
    PE_CHECK(device >= 0 && device < ndev, "device index out of range");
    PE_CUDA(cudaSetDevice(device));
    pe_ctx *c = new pe_ctx();
    c->rank = rank; c->nranks = nranks; c->device = device;
    PE_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    PE_CUDA(cudaStreamCreateWithFlags(&c->comm_stream, cudaStreamNonBlocking));
    PE_CUDA(cudaEventCreate(&c->ev_t0));
    PE_CUDA(cudaEventCreate(&c->ev_t1));
    PE_CUDA(cudaEventCreateWithFlags(&c->ev_pack, cudaEventDisableTiming));
    PE_CUDA(cudaEventCreateWithFlags(&c->ev_halo, cudaEventDisableTiming));
    PE_CUDA(cudaMalloc(&c->partials_d, sizeof(double) * PE_MAX_PARTIALS));
    PE_CUDA(cudaMalloc(&c->scalar_d, sizeof(double) * 8));
    PE_CUDA(cudaMallocHost(&c->scalar_h, sizeof(double) * 8));
    if (nranks > 1) {
        PE_CHECK(nccl_unique_id, "nranks > 1 needs an NCCL unique id");
        PE_TRY(nccl_load());
        pe_ncclUniqueId id;
        memcpy(&id, nccl_unique_id, 128);
        PE_NCCL(g_nccl.CommInitRank(&c->nccl, nranks, id, rank));
    }
    *out = c;
    return 0;
}

extern "C" int pe_ctx_destroy(pe_ctx *c)
{
    if (!c) return 0;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    cudaStreamSynchronize(c->comm_stream);
    pe_p2p_shutdown(c);
    if (c->nccl) g_nccl.CommDestroy(c->nccl);
    cudaFree(c->partials_d); cudaFree(c->scalar_d); cudaFreeHost(c->scalar_h);
    if (c->flush_d) cudaFree(c->flush_d);
    cudaEventDestroy(c->ev_t0); cudaEventDestroy(c->ev_t1);
    cudaEventDestroy(c->ev_pack); cudaEventDestroy(c->ev_halo);
    cudaStreamDestroy(c->stream); cudaStreamDestroy(c->comm_stream);
    delete c;
    return 0;
}

static int g_tuning[PE_TUNE_COUNT] = {200000, 0, 1, 0, 1, 0, 0, 0};
extern "C" int pe_set_tuning(int key, int value)
{
    PE_CHECK(key >= 0 && key < PE_TUNE_COUNT, "bad tuning key");
    g_tuning[key] = value;
    return 0;
}
extern "C" int pe_get_tuning(int key) { return key >= 0 && key < PE_TUNE_COUNT ? g_tuning[key] : 0; }

static std::atomic<int64_t> g_variant[PE_VARIANT_COUNT];
void pe_variant_add(int slot, int64_t count) { g_variant[slot].fetch_add(count, std::memory_order_relaxed); }
extern "C" int pe_variant_counts(int64_t *out, int n, int reset)
{
    PE_CHECK(n >= 0 && (out || n == 0), "pe_variant_counts: bad arguments");
    for (int k = 0; k < n; ++k) out[k] = k < PE_VARIANT_COUNT ? g_variant[k].load(std::memory_order_relaxed) : 0;
    if (reset)
        for (auto &c : g_variant) c.store(0, std::memory_order_relaxed);
    return 0;
}

extern "C" int pe_ctx_sync(pe_ctx *c)
{
    PE_CUDA(cudaStreamSynchronize(c->stream));
    PE_CUDA(cudaStreamSynchronize(c->comm_stream));
    return 0;
}
extern "C" int pe_ctx_rank(const pe_ctx *c) { return c->rank; }
extern "C" int pe_ctx_nranks(const pe_ctx *c) { return c->nranks; }
extern "C" int pe_ctx_p2p_enabled(const pe_ctx *c) { return c->p2p_base ? 1 : 0; }
extern "C" int64_t pe_ctx_launch_count(const pe_ctx *c) { return c->launches; }

extern "C" int pe_ctx_timer_start(pe_ctx *c)
{
    PE_CUDA(cudaEventRecord(c->ev_t0, c->stream));
    return 0;
}
extern "C" int pe_ctx_timer_stop(pe_ctx *c, float *ms)
{
    PE_CUDA(cudaEventRecord(c->ev_t1, c->stream));
    PE_CUDA(cudaEventSynchronize(c->ev_t1));
    PE_CUDA(cudaEventElapsedTime(ms, c->ev_t0, c->ev_t1));
    return 0;
}

__global__ void k_fill_u32(uint32_t *p, size_t n, uint32_t v)
{
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) p[i] = v;
}
extern "C" int pe_ctx_flush_l2(pe_ctx *c)
{
    if (!c->flush_d) {
        c->flush_bytes = (size_t)256 << 20;  // 256 MiB > 126 MB L2
        PE_CUDA(cudaMalloc(&c->flush_d, c->flush_bytes));
    }
    k_fill_u32<<<PE_SM_COUNT * 8, 256, 0, c->stream>>>((uint32_t *)c->flush_d,
                                                      c->flush_bytes / 4, 0u);
    PE_CUDA(cudaPeekAtLastError());
    return 0;
}

int pe_allreduce_sum(pe_ctx *c, double *d, int count)
{
    if (c->nranks == 1) return 0;
    PE_NCCL(g_nccl.AllReduce(d, d, (size_t)count, PE_NCCL_FLOAT64, PE_NCCL_SUM, c->nccl, c->stream));
    return 0;
}
// op: ncclRedOp_t (0 sum, 2 max)
int pe_allreduce(pe_ctx *c, double *d, int count, int op)
{
    if (c->nranks == 1) return 0;
    PE_NCCL(g_nccl.AllReduce(d, d, (size_t)count, PE_NCCL_FLOAT64, op, c->nccl, c->stream));
    return 0;
}

// ---------------------------------------------------------------------------
// per-kernel event profiling
// ---------------------------------------------------------------------------
static cudaEvent_t prof_event(pe_ctx *c)
{
    if (!c->prof_pool.empty()) { cudaEvent_t e = c->prof_pool.back(); c->prof_pool.pop_back(); return e; }
    cudaEvent_t e; cudaEventCreate(&e); return e;
}
int pe_prof_begin(pe_ctx *c, int id, double bytes)
{
    c->pending_bytes = bytes;
    if (!c->prof || c->capturing || c->rec) return 0;
    pe_ctx::ProfRec r{id, bytes, prof_event(c), prof_event(c)};
    PE_CUDA(cudaEventRecord(r.e0, c->stream));
    c->prof_recs.push_back(r);
    return 0;
}
int pe_prof_end(pe_ctx *c)
{
    if (!c->prof || c->capturing || c->rec) return 0;
    PE_CUDA(cudaEventRecord(c->prof_recs.back().e1, c->stream));
    return 0;
}
extern "C" int pe_ctx_profile(pe_ctx *c, int enable)
{
    PE_CUDA(cudaStreamSynchronize(c->stream));
    for (auto &r : c->prof_recs)
    {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.e0, r.e1) == cudaSuccess) { c->prof_ms[r.id] += ms; c->prof_bytes[r.id] += r.bytes; c->prof_count[r.id]++; }
        c->prof_pool.push_back(r.e0); c->prof_pool.push_back(r.e1);
    }
    c->prof_recs.clear();
    if (enable == 1 && !c->prof) for (int i = 0; i < 4; ++i) { c->prof_ms[i] = 0; c->prof_bytes[i] = 0; c->prof_count[i] = 0; }
    c->prof = enable != 0;
    return 0;
}
extern "C" int pe_ctx_profile_get(pe_ctx *c, int id, int64_t *count, double *total_ms, double *total_bytes)
{
    PE_CHECK(id >= 0 && id < 4, "bad kernel id");
    PE_TRY(pe_ctx_profile(c, c->prof ? 2 : 0));   // fold pending records, keep the state
    if (count) *count = c->prof_count[id];
    if (total_ms) *total_ms = c->prof_ms[id];
    if (total_bytes) *total_bytes = c->prof_bytes[id];
    return 0;
}

// ---------------------------------------------------------------------------
// CUDA graphs
// ---------------------------------------------------------------------------
struct pe_graph {
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    int64_t launches = 0;   // kernels recorded in the graph (counted at capture)
};
extern "C" int pe_graph_free(pe_graph *g);
extern "C" int pe_graph_begin(pe_ctx *c)
{
    PE_CHECK(!c->capturing, "graph capture already active");
    PE_CUDA(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
    c->capturing = true;
    c->scalar_h[7] = (double)c->launches;
    return 0;
}
extern "C" int pe_graph_end(pe_ctx *c, pe_graph **out)
{
    PE_CHECK(c->capturing, "no graph capture active");
    pe_graph *g = new pe_graph();
    c->capturing = false;
    g->launches = c->launches - (int64_t)c->scalar_h[7];
    c->launches = (int64_t)c->scalar_h[7];  // capture did not execute anything
    cudaError_t e = cudaStreamEndCapture(c->stream, &g->graph);
    if (e == cudaSuccess) e = cudaGraphInstantiate(&g->exec, g->graph, 0);
    if (e != cudaSuccess)
    {
        (void)cudaGetLastError();   // an invalidated capture leaves a sticky-looking error behind
        pe_set_error(std::string("CUDA graph capture failed: ") + cudaGetErrorString(e));
        pe_graph_free(g);
        return 1;
    }
    *out = g;
    return 0;
}
extern "C" int pe_graph_launch(pe_ctx *c, pe_graph *g)
{
    PE_CUDA(cudaGraphLaunch(g->exec, c->stream));
    c->launches += g->launches;
    return 0;
}
extern "C" int pe_graph_free(pe_graph *g)
{
    if (!g) return 0;
    if (g->exec) cudaGraphExecDestroy(g->exec);
    if (g->graph) cudaGraphDestroy(g->graph);
    delete g;
    return 0;
}

// ---------------------------------------------------------------------------
// vectors
// ---------------------------------------------------------------------------
extern "C" int pe_vec_create(pe_ctx *ctx, int64_t n, pe_vec **out)
{
    PE_CHECK(ctx && out && n >= 0, "bad arguments");
    pe_vec *v = new pe_vec{ctx, n, nullptr, false};
    PE_CUDA(cudaMalloc(&v->d, sizeof(double) * (size_t)(n > 0 ? n : 1)));
    PE_CUDA(cudaMemsetAsync(v->d, 0, sizeof(double) * (size_t)(n > 0 ? n : 1), ctx->stream));
    *out = v;
    return 0;
}
extern "C" int pe_vec_free(pe_vec *v)
{
    if (!v) return 0;
    if (!v->view)
    {
        cudaStreamSynchronize(v->ctx->stream);
        cudaFree(v->d);
    }
    delete v;
    return 0;
}
extern "C" int pe_vec_view(const pe_vec *base, int64_t offset, int64_t n, pe_vec **out)
{
    PE_CHECK(base && out && offset >= 0 && n >= 0 && offset + n <= base->n, "pe_vec_view: range outside the base vector");
    *out = new pe_vec{base->ctx, n, base->d + offset, true};
    return 0;
}
extern "C" int64_t pe_vec_size(const pe_vec *v) { return v->n; }
extern "C" void *pe_vec_device_ptr(pe_vec *v) { return v->d; }
extern "C" int pe_vec_upload(pe_vec *v, const double *host)
{
    PE_CUDA(cudaMemcpyAsync(v->d, host, sizeof(double) * (size_t)v->n, cudaMemcpyHostToDevice,
                            v->ctx->stream));
    PE_CUDA(cudaStreamSynchronize(v->ctx->stream));
    return 0;
}
extern "C" int pe_vec_download(const pe_vec *v, double *host)
{
    PE_CUDA(cudaMemcpyAsync(host, v->d, sizeof(double) * (size_t)v->n, cudaMemcpyDeviceToHost,
                            v->ctx->stream));
    PE_CUDA(cudaStreamSynchronize(v->ctx->stream));
    return 0;
}

// elementwise kernels: grid-stride, 2 doubles per thread per step via double2 when aligned
__global__ void k_fill(double *x, int64_t n, double v)
{
    pdl_trigger(); pdl_wait();   // operands come from the preceding kernel (see pe_launch_k)
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int64_t s = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += s) x[i] = v;
}
__global__ void k_axpby(int64_t n, double a, const double *x, double b,
                        double *y)
{
    pdl_trigger(); pdl_wait();   // operands come from the preceding kernel (see pe_launch_k)
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int64_t s = (int64_t)gridDim.x * blockDim.x;
    if (b == 0.0) { for (; i < n; i += s) y[i] = a * x[i]; }
    else { for (; i < n; i += s) y[i] = a * x[i] + b * y[i]; }
}
__global__ void k_add3(int64_t n, double a, const double *x, double b,
                       const double *y, double *z)
{
    pdl_trigger(); pdl_wait();   // operands come from the preceding kernel (see pe_launch_k)
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int64_t s = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += s) z[i] = a * x[i] + b * y[i];
}
__global__ void k_scale(int64_t n, double a, double *x)
{
    pdl_trigger(); pdl_wait();   // operands come from the preceding kernel (see pe_launch_k)
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int64_t s = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += s) x[i] *= a;
}
__global__ void k_mul(int64_t n, const double *d, double *x)
{
    pdl_trigger(); pdl_wait();   // operands come from the preceding kernel (see pe_launch_k)
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int64_t s = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += s) x[i] *= d[i];
}
static inline int ew_grid(int64_t n)
{
    int64_t g = (n + 255) / 256;
    int64_t cap = (int64_t)PE_SM_COUNT * 16;
    return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}
extern "C" int pe_vec_fill(pe_vec *v, double value)
{
    if (v->ctx->rec)
    {
        if (v->n == 0) return 0;
        PeOp o = pe_op(PE_OP_FILL); o.n = v->n; o.a = value; o.p[0] = v->d;
        pe_rec_push(v->ctx, o, 8.0 * v->n);
        return 0;
    }
    if (value == 0.0) {
        PE_CUDA(cudaMemsetAsync(v->d, 0, sizeof(double) * (size_t)v->n, v->ctx->stream));
        return 0;
    }
    PE_CUDA(pe_launch_k(v->ctx, k_fill, ew_grid(v->n), 256, v->d, v->n, value));
    PE_LAUNCHED(v->ctx);
    return 0;
}
extern "C" int pe_vec_copy(const pe_vec *src, pe_vec *dst)
{
    PE_CHECK(src->n == dst->n, "size mismatch");
    if (dst->ctx->rec)
    {
        if (src->n == 0) return 0;
        PeOp o = pe_op(PE_OP_COPY); o.n = src->n; o.p[0] = src->d; o.p[1] = dst->d;
        pe_rec_push(dst->ctx, o, 16.0 * src->n);
        return 0;
    }
    PE_CUDA(cudaMemcpyAsync(dst->d, src->d, sizeof(double) * (size_t)src->n,
                            cudaMemcpyDeviceToDevice, dst->ctx->stream));
    return 0;
}
extern "C" int pe_vec_axpby(double a, const pe_vec *x, double b, pe_vec *y)
{
    PE_CHECK(x->n == y->n, "size mismatch");
    if (y->ctx->rec)
    {
        if (x->n == 0) return 0;
        PeOp o = pe_op(PE_OP_AXPBY); o.n = x->n; o.a = a; o.b = b; o.p[0] = x->d; o.p[1] = y->d;
        pe_rec_push(y->ctx, o, (b == 0.0 ? 16.0 : 24.0) * x->n);
        return 0;
    }
    PE_CUDA(pe_launch_k(y->ctx, k_axpby, ew_grid(x->n), 256, x->n, a, x->d, b, y->d));
    PE_LAUNCHED(y->ctx);
    return 0;
}
extern "C" int pe_vec_add3(double a, const pe_vec *x, double b, const pe_vec *y, pe_vec *z)
{
    PE_CHECK(x->n == y->n && x->n == z->n, "size mismatch");
    if (z->ctx->rec)
    {
        if (x->n == 0) return 0;
        PeOp o = pe_op(PE_OP_ADD3); o.n = x->n; o.a = a; o.b = b; o.p[0] = x->d; o.p[1] = y->d; o.p[2] = z->d;
        pe_rec_push(z->ctx, o, 24.0 * x->n);
        return 0;
    }
    PE_CUDA(pe_launch_k(z->ctx, k_add3, ew_grid(x->n), 256, x->n, a, x->d, b, y->d, z->d));
    PE_LAUNCHED(z->ctx);
    return 0;
}
extern "C" int pe_vec_scale(pe_vec *x, double a)
{
    if (x->ctx->rec)
    {
        if (x->n == 0) return 0;
        PeOp o = pe_op(PE_OP_SCALE); o.n = x->n; o.a = a; o.p[0] = x->d;
        pe_rec_push(x->ctx, o, 16.0 * x->n);
        return 0;
    }
    PE_CUDA(pe_launch_k(x->ctx, k_scale, ew_grid(x->n), 256, x->n, a, x->d));
    PE_LAUNCHED(x->ctx);
    return 0;
}
extern "C" int pe_vec_mul(const pe_vec *d, pe_vec *x)
{
    PE_CHECK(d->n == x->n, "size mismatch");
    if (x->ctx->rec)
    {
        if (x->n == 0) return 0;
        PeOp o = pe_op(PE_OP_MUL); o.n = x->n; o.p[0] = d->d; o.p[1] = x->d;
        pe_rec_push(x->ctx, o, 24.0 * x->n);
        return 0;
    }
    PE_CUDA(pe_launch_k(x->ctx, k_mul, ew_grid(x->n), 256, x->n, d->d, x->d));
    PE_LAUNCHED(x->ctx);
    return 0;
}

// deterministic two-stage dot: fixed grid, fixed in-block tree, fixed final order
#define DOT_THREADS 256
__global__ void k_dot_stage1(int64_t n, const double *x, const double *y,
                             double *partials)
{
    pdl_trigger(); pdl_wait();   // operands come from the preceding kernel (see pe_launch_k)
    __shared__ double sh[DOT_THREADS];
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int64_t s = (int64_t)gridDim.x * blockDim.x;
    double acc = 0.0;
    for (; i < n; i += s) acc += x[i] * y[i];
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int w = DOT_THREADS / 2; w > 0; w >>= 1) {
        if (threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) partials[blockIdx.x] = sh[0];
}
__global__ void k_dot_stage2(int nparts, const double *partials, double *out)
{
    pdl_trigger(); pdl_wait();   // operands come from the preceding kernel (see pe_launch_k)
    __shared__ double sh[DOT_THREADS];
    double acc = 0.0;
    for (int i = threadIdx.x; i < nparts; i += DOT_THREADS) acc += partials[i];
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int w = DOT_THREADS / 2; w > 0; w >>= 1) {
        if (threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = sh[0];
}
extern "C" int pe_vec_dot(const pe_vec *x, const pe_vec *y, double *out)
{
    PE_CHECK(x->n == y->n, "size mismatch");
    pe_ctx *c = x->ctx;
    if (c->rec) pe_rec_fail(c, "pe_vec_dot (host-synchronising)", 0);
    int grid = ew_grid(x->n);
    if (grid > PE_MAX_PARTIALS) grid = PE_MAX_PARTIALS;
    PE_CUDA(pe_launch_k(c, k_dot_stage1, grid, DOT_THREADS, x->n, x->d, y->d, c->partials_d));
    PE_LAUNCHED(c);
    PE_CUDA(pe_launch_k(c, k_dot_stage2, 1, DOT_THREADS, grid, c->partials_d, c->scalar_d));
    PE_LAUNCHED(c);
    PE_TRY(pe_allreduce_sum(c, c->scalar_d, 1));
    PE_CUDA(cudaMemcpyAsync(c->scalar_h, c->scalar_d, sizeof(double), cudaMemcpyDeviceToHost,
                            c->stream));
    PE_CUDA(cudaStreamSynchronize(c->stream));
    *out = c->scalar_h[0];
    return 0;
}

// ---------------------------------------------------------------------------
// device-resident scalars (graph-capturable inner Krylov solves)
// ---------------------------------------------------------------------------
extern "C" int pe_ctx_is_capturing(const pe_ctx *c) { return c->capturing ? 1 : 0; }
extern "C" int pe_ctx_is_profiling(const pe_ctx *c) { return c->prof ? 1 : 0; }
extern "C" int pe_scalars_create(pe_ctx *ctx, int count, double **slots_d)
{
    PE_CHECK(ctx && slots_d && count > 0, "bad arguments");
    PE_CUDA(cudaMalloc(slots_d, sizeof(double) * (size_t)count));
    PE_CUDA(cudaMemsetAsync(*slots_d, 0, sizeof(double) * (size_t)count, ctx->stream));
    return 0;
}
extern "C" int pe_scalars_free(double *slots_d)
{
    if (slots_d) cudaFree(slots_d);
    return 0;
}
extern "C" int pe_scalars_download(pe_ctx *ctx, const double *slots_d, int count, double *host)
{
    PE_CUDA(cudaMemcpyAsync(host, slots_d, sizeof(double) * (size_t)count, cudaMemcpyDeviceToHost, ctx->stream));
    PE_CUDA(cudaStreamSynchronize(ctx->stream));
    return 0;
}
extern "C" int pe_vec_dot_dev(const pe_vec *x, const pe_vec *y, double *slots_d, int out_slot)
{
    PE_CHECK(x->n == y->n, "size mismatch");
    pe_ctx *c = x->ctx;
    if (c->rec)
    {
        PeOp o = pe_op(PE_OP_DOT); o.n = x->n; o.p[0] = x->d; o.p[1] = y->d; o.p[2] = c->partials_d;
        pe_rec_push(c, o, 16.0 * x->n);
        PeOp f = pe_op(PE_OP_DOT_FIN); f.p[0] = c->partials_d; f.p[1] = slots_d + out_slot;   // i0 = grid, set at program_end
        pe_rec_push(c, f, 0.0);
        return 0;
    }
    int grid = ew_grid(x->n);
    if (grid > PE_MAX_PARTIALS) grid = PE_MAX_PARTIALS;
    PE_CUDA(pe_launch_k(c, k_dot_stage1, grid, DOT_THREADS, x->n, x->d, y->d, c->partials_d));
    PE_LAUNCHED(c);
    PE_CUDA(pe_launch_k(c, k_dot_stage2, 1, DOT_THREADS, grid, c->partials_d, slots_d + out_slot));
    PE_LAUNCHED(c);
    return pe_allreduce_sum(c, slots_d + out_slot, 1);
}
__global__ void k_axpy_dev(int64_t n, const double *a, double sign, const double *x, double *y)
{
    pdl_trigger(); pdl_wait();   // operands come from the preceding kernel (see pe_launch_k)
    const double s = sign * a[0];
    if (s == 0.0) return;
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t st = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += st) y[i] += s * x[i];
}
__global__ void k_xpby_dev(int64_t n, const double *x, const double *b, double *y)
{
    pdl_trigger(); pdl_wait();   // operands come from the preceding kernel (see pe_launch_k)
    const double s = b[0];
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t st = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += st) y[i] = x[i] + s * y[i];
}
extern "C" int pe_vec_axpy_dev(const double *slots_d, int a_slot, double sign, const pe_vec *x, pe_vec *y)
{
    PE_CHECK(x->n == y->n, "size mismatch");
    if (y->ctx->rec)
    {
        if (x->n == 0) return 0;
        PeOp o = pe_op(PE_OP_AXPY_DEV); o.n = x->n; o.a = sign; o.p[0] = slots_d + a_slot; o.p[1] = x->d; o.p[2] = y->d;
        pe_rec_push(y->ctx, o, 24.0 * x->n);
        return 0;
    }
    PE_CUDA(pe_launch_k(y->ctx, k_axpy_dev, ew_grid(x->n), 256, x->n, slots_d + a_slot, sign, x->d, y->d));
    PE_LAUNCHED(y->ctx);
    return 0;
}
extern "C" int pe_vec_xpby_dev(const pe_vec *x, const double *slots_d, int b_slot, pe_vec *y)
{
    PE_CHECK(x->n == y->n, "size mismatch");
    if (y->ctx->rec)
    {
        if (x->n == 0) return 0;
        PeOp o = pe_op(PE_OP_XPBY_DEV); o.n = x->n; o.p[0] = x->d; o.p[1] = slots_d + b_slot; o.p[2] = y->d;
        pe_rec_push(y->ctx, o, 24.0 * x->n);
        return 0;
    }
    PE_CUDA(pe_launch_k(y->ctx, k_xpby_dev, ew_grid(x->n), 256, x->n, x->d, slots_d + b_slot, y->d));
    PE_LAUNCHED(y->ctx);
    return 0;
}
__global__ void k_pcg_scalar_step(double *s, int phase, int iter, int max_iter, double rel, double abs_tol)
{
    pdl_trigger(); pdl_wait();   // operands come from the preceding kernel (see pe_launch_k)
    pe_pcg_scalar_step_dev(s, phase, iter, max_iter, rel, abs_tol);
}
extern "C" int pe_pcg_scalar_step(pe_ctx *ctx, double *slots_d, int phase, int iter, int max_iter, double rel_tol, double abs_tol)
{
    PE_CHECK(phase >= 0 && phase <= 3, "bad phase");
    if (ctx->rec)
    {
        PeOp o = pe_op(PE_OP_PCG_STEP); o.i0 = phase; o.i1 = iter; o.i2 = max_iter; o.a = rel_tol; o.b = abs_tol; o.p[0] = slots_d;
        pe_rec_push(ctx, o, 0.0);
        return 0;
    }
    PE_CUDA(pe_launch_k(ctx, k_pcg_scalar_step, 1, 1, slots_d, phase, iter, max_iter, rel_tol, abs_tol));
    PE_LAUNCHED(ctx);
    return 0;
}

// ---------------------------------------------------------------------------
// matrices
// ---------------------------------------------------------------------------
int devcsr_alloc(DevCSR &m, int32_t nrows, int32_t ncols, int64_t nnz)
{
    m.nrows = nrows; m.ncols = ncols; m.nnz = nnz;
    PE_CUDA(cudaMalloc(&m.I, sizeof(int32_t) * (size_t)(nrows + 1)));
    PE_CUDA(cudaMalloc(&m.J, sizeof(int32_t) * (size_t)(nnz > 0 ? nnz : 1)));
    PE_CUDA(cudaMalloc(&m.A, sizeof(double) * (size_t)(nnz > 0 ? nnz : 1)));
    return 0;
}
void devcsr_free(DevCSR &m)
{
    if (m.rb) cudaFree(m.rb);
    if (m.sell) { pe_sell_free(*m.sell); delete m.sell; }
    if (m.I) cudaFree(m.I);
    if (m.J) cudaFree(m.J);
    if (m.A) cudaFree(m.A);
    m = DevCSR();
}

// Row blocks for the streaming kernels.  Host pass over the row pointer (once per matrix):
// greedy packing of consecutive rows up to PE_STREAM_NNZ non-zeros and 1024 rows; optional
// forced breaks (Gauss-Seidel set boundaries).
int pe_build_row_blocks(pe_ctx *ctx, DevCSR &m, const std::vector<int32_t> *forced_breaks)
{
    if (m.rb) { cudaFree(m.rb); m.rb = nullptr; }
    m.nrb = 0;
    const int n = m.nrows;
    if (n == 0) return 0;
    std::vector<int32_t> I(n + 1);
    PE_CUDA(cudaMemcpyAsync(I.data(), m.I, sizeof(int32_t) * (size_t)(n + 1), cudaMemcpyDeviceToHost, ctx->stream));
    PE_CUDA(cudaStreamSynchronize(ctx->stream));
    std::vector<int32_t> rb;
    rb.push_back(0);
    size_t fb = 0;
    while (forced_breaks && fb < forced_breaks->size() && (*forced_breaks)[fb] <= 0) ++fb;
    int start = 0;
    for (int r = 0; r < n; ++r)
    {
        const int len = I[r + 1] - I[r];
        if (len > PE_STREAM_MAXROW) { m.nrb = -1; return 0; }
        const bool forced = forced_breaks && fb < forced_breaks->size() && (*forced_breaks)[fb] == r;
        if (r > start && (forced || I[r + 1] - I[start] > PE_STREAM_NNZ || r - start >= 1024))
        {
            rb.push_back(r);
            start = r;
        }
        if (forced) ++fb;
    }
    rb.push_back(n);
    m.nrb = (int)rb.size() - 1;
    PE_CUDA(cudaMalloc(&m.rb, sizeof(int32_t) * rb.size()));
    PE_CUDA(cudaMemcpyAsync(m.rb, rb.data(), sizeof(int32_t) * rb.size(), cudaMemcpyHostToDevice, ctx->stream));
    PE_CUDA(cudaStreamSynchronize(ctx->stream));
    return 0;
}

void pe_mat_values_changed(pe_mat *A)
{
    if (A->T) { pe_mat_free(A->T); A->T = nullptr; }
    if (A->offdT_built) { devcsr_free(A->offdT); A->offdT_built = false; }
    for (DevCSR *m : {&A->diag, &A->offd})
    {
        if (m->sell) { pe_sell_free(*m->sell); delete m->sell; m->sell = nullptr; }
        m->sell_state = 0;
    }
}

int pe_choose_tpr(int64_t nnz, int32_t nrows)
{
    double avg = nrows > 0 ? (double)nnz / nrows : 0.0;
    int t = 1;
    while (t < 32 && t * 1.5 < avg) t <<= 1;   // avg 11 -> 8, 27..33 -> 32, 4 -> 4
    return t;
}

static int upload_block(pe_ctx *ctx, DevCSR &m, int32_t nrows, int32_t ncols, const int32_t *I,
                        const int32_t *J, const double *A)
{
    int64_t nnz = I ? I[nrows] : 0;
    PE_TRY(devcsr_alloc(m, nrows, ncols, nnz));
    if (I) PE_CUDA(cudaMemcpyAsync(m.I, I, sizeof(int32_t) * (size_t)(nrows + 1),
                                   cudaMemcpyHostToDevice, ctx->stream));
    else PE_CUDA(cudaMemsetAsync(m.I, 0, sizeof(int32_t) * (size_t)(nrows + 1), ctx->stream));
    if (nnz > 0) {
        PE_CUDA(cudaMemcpyAsync(m.J, J, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice,
                                ctx->stream));
        PE_CUDA(cudaMemcpyAsync(m.A, A, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice,
                                ctx->stream));
    }
    return 0;
}

// ghost / reverse-receive buffers live in the peer-visible halo arena when there is one (pe_p2p.cu)
static int halo_buffer_alloc(pe_ctx *ctx, size_t n, double **out)
{
    *out = static_cast<double *>(pe_p2p_alloc(ctx, sizeof(double) * (n > 0 ? n : 1)));
    if (!*out) PE_CUDA(cudaMalloc(out, sizeof(double) * (n > 0 ? n : 1)));
    return 0;
}

extern "C" int pe_mat_upload(pe_ctx *ctx, const pe_parcsr_host *H, pe_mat **out)
{
    PE_CHECK(ctx && H && out, "bad arguments");
    PE_CHECK(H->num_rows >= 0 && H->diag_i, "matrix needs diag_i");
    pe_mat *M = new pe_mat();
    M->ctx = ctx;
    M->global_num_rows = H->global_num_rows; M->global_num_cols = H->global_num_cols;
    M->first_row_index = H->first_row_index; M->first_col_diag = H->first_col_diag;
    PE_TRY(upload_block(ctx, M->diag, H->num_rows, H->num_cols_diag, H->diag_i, H->diag_j,
                        H->diag_data));
    PE_TRY(upload_block(ctx, M->offd, H->num_rows, H->num_cols_offd,
                        H->num_cols_offd > 0 ? H->offd_i : nullptr, H->offd_j, H->offd_data));
    if (H->num_cols_offd > 0) {
        PE_CHECK(H->col_map_offd, "offd block needs col_map_offd");
        M->col_map_offd.assign(H->col_map_offd, H->col_map_offd + H->num_cols_offd);
        PE_CHECK(ctx->nranks > 1, "ghost columns on a single-rank context");
        M->send_procs.assign(H->send_procs, H->send_procs + H->num_sends);
        M->send_map_starts.assign(H->send_map_starts, H->send_map_starts + H->num_sends + 1);
        int nsend = M->send_map_starts[H->num_sends];
        M->send_map_elmts.assign(H->send_map_elmts, H->send_map_elmts + nsend);
        M->recv_procs.assign(H->recv_procs, H->recv_procs + H->num_recvs);
        M->recv_vec_starts.assign(H->recv_vec_starts, H->recv_vec_starts + H->num_recvs + 1);
        PE_CUDA(cudaMalloc(&M->send_map_d, sizeof(int32_t) * (size_t)(nsend > 0 ? nsend : 1)));
        PE_CUDA(cudaMemcpyAsync(M->send_map_d, M->send_map_elmts.data(), sizeof(int32_t) * (size_t)nsend,
                                cudaMemcpyHostToDevice, ctx->stream));
        PE_TRY(halo_buffer_alloc(ctx, (size_t)(nsend > 0 ? nsend : 1), &M->send_buf_d));
        PE_TRY(halo_buffer_alloc(ctx, (size_t)H->num_cols_offd, &M->x_ext_d));
    } else if (H->num_sends > 0) {
        // a rank may own columns others need while having no ghosts itself
        M->send_procs.assign(H->send_procs, H->send_procs + H->num_sends);
        M->send_map_starts.assign(H->send_map_starts, H->send_map_starts + H->num_sends + 1);
        int nsend = M->send_map_starts[H->num_sends];
        M->send_map_elmts.assign(H->send_map_elmts, H->send_map_elmts + nsend);
        PE_CUDA(cudaMalloc(&M->send_map_d, sizeof(int32_t) * (size_t)(nsend > 0 ? nsend : 1)));
        PE_CUDA(cudaMemcpyAsync(M->send_map_d, M->send_map_elmts.data(), sizeof(int32_t) * (size_t)nsend,
                                cudaMemcpyHostToDevice, ctx->stream));
        PE_TRY(halo_buffer_alloc(ctx, (size_t)(nsend > 0 ? nsend : 1), &M->send_buf_d));
    }
    M->tpr = pe_choose_tpr(M->diag.nnz + M->offd.nnz, M->diag.nrows);
    M->distributed = ctx->nranks > 1 && (H->global_num_rows != H->num_rows || H->global_num_cols != H->num_cols_diag ||
                                         H->num_cols_offd > 0 || H->num_sends > 0);
    PE_CUDA(cudaStreamSynchronize(ctx->stream));
    *out = M;
    return 0;
}

int pe_mat_wrap_local(pe_ctx *ctx, DevCSR &diag, pe_mat **out)
{
    pe_mat *M = new pe_mat();
    M->ctx = ctx;
    M->diag = diag;
    diag = DevCSR();
    M->global_num_rows = M->diag.nrows; M->global_num_cols = M->diag.ncols;
    PE_TRY(devcsr_alloc(M->offd, M->diag.nrows, 0, 0));
    PE_CUDA(cudaMemsetAsync(M->offd.I, 0, sizeof(int32_t) * (size_t)(M->diag.nrows + 1), ctx->stream));
    M->tpr = pe_choose_tpr(M->diag.nnz, M->diag.nrows);
    *out = M;
    return 0;
}

extern "C" int pe_mat_info(const pe_mat *A, int32_t *num_rows, int32_t *num_cols_diag,
                           int32_t *num_cols_offd, int64_t *nnz_diag, int64_t *nnz_offd)
{
    if (num_rows) *num_rows = A->diag.nrows;
    if (num_cols_diag) *num_cols_diag = A->diag.ncols;
    if (num_cols_offd) *num_cols_offd = A->offd.ncols;
    if (nnz_diag) *nnz_diag = A->diag.nnz;
    if (nnz_offd) *nnz_offd = A->offd.nnz;
    return 0;
}

extern "C" int pe_mat_global_info(const pe_mat *A, int64_t *gr, int64_t *gc, int64_t *fr, int64_t *fc)
{
    if (gr) *gr = A->global_num_rows;
    if (gc) *gc = A->global_num_cols;
    if (fr) *fr = A->first_row_index;
    if (fc) *fc = A->first_col_diag;
    return 0;
}

extern "C" int pe_mat_download(const pe_mat *A, int32_t *diag_i, int32_t *diag_j, double *diag_data,
                               int32_t *offd_i, int32_t *offd_j, double *offd_data,
                               int64_t *col_map_offd)
{
    cudaStream_t s = A->ctx->stream;
    if (diag_i) PE_CUDA(cudaMemcpyAsync(diag_i, A->diag.I, sizeof(int32_t) * (size_t)(A->diag.nrows + 1), cudaMemcpyDeviceToHost, s));
    if (diag_j && A->diag.nnz) PE_CUDA(cudaMemcpyAsync(diag_j, A->diag.J, sizeof(int32_t) * (size_t)A->diag.nnz, cudaMemcpyDeviceToHost, s));
    if (diag_data && A->diag.nnz) PE_CUDA(cudaMemcpyAsync(diag_data, A->diag.A, sizeof(double) * (size_t)A->diag.nnz, cudaMemcpyDeviceToHost, s));
    if (offd_i) PE_CUDA(cudaMemcpyAsync(offd_i, A->offd.I, sizeof(int32_t) * (size_t)(A->offd.nrows + 1), cudaMemcpyDeviceToHost, s));
    if (offd_j && A->offd.nnz) PE_CUDA(cudaMemcpyAsync(offd_j, A->offd.J, sizeof(int32_t) * (size_t)A->offd.nnz, cudaMemcpyDeviceToHost, s));
    if (offd_data && A->offd.nnz) PE_CUDA(cudaMemcpyAsync(offd_data, A->offd.A, sizeof(double) * (size_t)A->offd.nnz, cudaMemcpyDeviceToHost, s));
    if (col_map_offd) memcpy(col_map_offd, A->col_map_offd.data(), sizeof(int64_t) * A->col_map_offd.size());
    PE_CUDA(cudaStreamSynchronize(s));
    return 0;
}

extern "C" int pe_mat_free(pe_mat *A)
{
    if (!A) return 0;
    cudaStreamSynchronize(A->ctx->stream);
    cudaStreamSynchronize(A->ctx->comm_stream);
    pe_p2p_unlink(A);
    devcsr_free(A->diag);
    devcsr_free(A->offd);
    if (A->send_map_d) cudaFree(A->send_map_d);
    if (A->send_buf_d && !pe_p2p_owns(A->ctx, A->send_buf_d)) cudaFree(A->send_buf_d);   // arena blocks are not returned
    if (A->x_ext_d && !pe_p2p_owns(A->ctx, A->x_ext_d)) cudaFree(A->x_ext_d);
    if (A->T) pe_mat_free(A->T);
    devcsr_free(A->offdT);
    if (A->unpack_rows_d) cudaFree(A->unpack_rows_d);
    if (A->unpack_I_d) cudaFree(A->unpack_I_d);
    if (A->unpack_pos_d) cudaFree(A->unpack_pos_d);
    delete A;
    return 0;
}

// ---------------------------------------------------------------------------
// halo exchange: pack x[send_map_elmts] -> grouped ncclSend/ncclRecv on the comm
// stream; the compute stream overlaps the diag pass and waits on ev_halo before the
// offd pass.  Same structure as hypre_ParCSRMatrixMatvecBoolInt.c:162-199.
// ---------------------------------------------------------------------------
__global__ void k_pack(int n, const int32_t *__restrict__ map, const double *__restrict__ x,
                       double *__restrict__ buf)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) buf[i] = x[map[i]];
}

// peer-memory path (pe_p2p.cu): linked at the first exchange of a matrix outside graph capture -- a collective
// step over ALL ranks (pe_p2p_link gathers the buffer offsets of every rank), so every rank of a distributed
// matrix enters it, also a rank that has no neighbour for this particular matrix (all ranks execute the same
// sequence of exchanges); matrices that are not distributed at all (no comm package on any rank: global == local
// size) never get here.
static int p2p_ready(pe_mat *A)
{
    pe_ctx *c = A->ctx;
    // rank-local matrix on a multi-rank context (global == local sizes: the MPI_COMM_SELF case): nothing to link
    if (A->global_num_rows == A->diag.nrows && A->global_num_cols == A->diag.ncols) return 0;
    if (A->p2p_state == 0 && c->p2p_base && !c->capturing) PE_TRY(pe_p2p_link(A));
    return 0;
}

int pe_halo_exchange(pe_mat *A, const double *x_d)
{
    pe_ctx *c = A->ctx;
    if (c->nranks == 1) return 0;
    int nsend = A->send_map_starts.empty() ? 0 : A->send_map_starts.back();
    int nrecv = A->recv_vec_starts.empty() ? 0 : A->recv_vec_starts.back();
    PE_TRY(p2p_ready(A));
    if (nsend == 0 && nrecv == 0) return 0;
    if (A->p2p_state == 1) return pe_p2p_push(A, 0, x_d);
    if (nsend > 0) {
        k_pack<<<pe_grid_for(nsend, 256), 256, 0, c->stream>>>(nsend, A->send_map_d, x_d, A->send_buf_d);
        PE_LAUNCHED(c);
    }
    PE_CUDA(cudaEventRecord(c->ev_pack, c->stream));
    PE_CUDA(cudaStreamWaitEvent(c->comm_stream, c->ev_pack, 0));
    PE_NCCL(g_nccl.GroupStart());
    for (size_t s = 0; s < A->send_procs.size(); ++s) {
        int lo = A->send_map_starts[s], hi = A->send_map_starts[s + 1];
        PE_NCCL(g_nccl.Send(A->send_buf_d + lo, (size_t)(hi - lo), PE_NCCL_FLOAT64, A->send_procs[s],
                            c->nccl, c->comm_stream));
    }
    for (size_t r = 0; r < A->recv_procs.size(); ++r) {
        int lo = A->recv_vec_starts[r], hi = A->recv_vec_starts[r + 1];
        PE_NCCL(g_nccl.Recv(A->x_ext_d + lo, (size_t)(hi - lo), PE_NCCL_FLOAT64, A->recv_procs[r],
                            c->nccl, c->comm_stream));
    }
    PE_NCCL(g_nccl.GroupEnd());
    PE_CUDA(cudaEventRecord(c->ev_halo, c->comm_stream));
    return 0;
}

int pe_halo_wait(pe_mat *A)
{
    pe_ctx *c = A->ctx;
    if (c->nranks == 1) return 0;
    if (A->p2p_state == 1)
    {
        const int nsend = A->send_map_starts.empty() ? 0 : A->send_map_starts.back();
        const int nrecv = A->recv_vec_starts.empty() ? 0 : A->recv_vec_starts.back();
        if (nsend == 0 && nrecv == 0) return 0;
        return pe_p2p_wait(A, 0);
    }
    PE_CUDA(cudaStreamWaitEvent(c->stream, c->ev_halo, 0));
    return 0;
}

// reverse exchange (MatvecT): the partial sums in x_ext_d travel to the owners of the ghost
// columns (recv_procs), land in send_buf_d (slots ordered like send_map_elmts) and are added to y.
int pe_reverse_halo_add(pe_mat *A, double alpha, double *y_d)
{
    pe_ctx *c = A->ctx;
    if (c->nranks == 1) return 0;
    int nsend = A->send_map_starts.empty() ? 0 : A->send_map_starts.back();
    int nrecv = A->recv_vec_starts.empty() ? 0 : A->recv_vec_starts.back();
    PE_TRY(p2p_ready(A));
    if (nsend == 0 && nrecv == 0) return 0;
    if (A->p2p_state == 1)
    {
        PE_TRY(pe_p2p_push(A, 1, A->x_ext_d));
        PE_TRY(pe_p2p_wait(A, 1));
        return pe_launch_unpack_add(c, A, alpha, y_d);
    }
    PE_CUDA(cudaEventRecord(c->ev_pack, c->stream));
    PE_CUDA(cudaStreamWaitEvent(c->comm_stream, c->ev_pack, 0));
    PE_NCCL(g_nccl.GroupStart());
    for (size_t r = 0; r < A->recv_procs.size(); ++r) {
        int lo = A->recv_vec_starts[r], hi = A->recv_vec_starts[r + 1];
        PE_NCCL(g_nccl.Send(A->x_ext_d + lo, (size_t)(hi - lo), PE_NCCL_FLOAT64, A->recv_procs[r], c->nccl, c->comm_stream));
    }
    for (size_t s = 0; s < A->send_procs.size(); ++s) {
        int lo = A->send_map_starts[s], hi = A->send_map_starts[s + 1];
        PE_NCCL(g_nccl.Recv(A->send_buf_d + lo, (size_t)(hi - lo), PE_NCCL_FLOAT64, A->send_procs[s], c->nccl, c->comm_stream));
    }
    PE_NCCL(g_nccl.GroupEnd());
    PE_CUDA(cudaEventRecord(c->ev_halo, c->comm_stream));
    PE_CUDA(cudaStreamWaitEvent(c->stream, c->ev_halo, 0));
    return pe_launch_unpack_add(c, A, alpha, y_d);
}
