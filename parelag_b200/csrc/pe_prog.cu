// pe_prog.cu -- the V-cycle as ONE persistent kernel.
//
// A multigrid V-cycle on the coarse levels is hundreds of tiny dependent steps (one colour of
// Gauss-Seidel on a few thousand rows, a restriction, a dot product ...).  As separate
// kernels -- even replayed from a CUDA graph -- every step pays a launch, a ramp-up and a
// drain (5-6 us measured on B200, see profiles/), which is ~30 % of the whole cycle.  Here the
// cycle is RECORDED once into a list of ops (the launchers in pe_sell.cu / pe_spmv.cu /
// pe_core.cu append a PeOp instead of launching while ctx->rec is set) and then executed by a
// single cooperative kernel with one 1024-thread CTA per SM: the whole grid walks the op list,
// every op is distributed over all warps of the grid, and ops are separated by a grid-wide
// barrier (one atomic arrive + acquire spin per CTA, ~1 us) instead of a kernel boundary.
//
// Memory model: vectors are written by one op and read by later ops on other SMs, so every
// vector access inside the program bypasses the (non-coherent) L1: loads are ld.global.cg,
// stores are write-through.  Matrix arrays are immutable during a program and keep the
// streaming, evict-first path.  The barrier is __syncthreads + __threadfence + atomic arrive,
// then ld.acquire spin: release/acquire at gpu scope, cumulative over the CTA via bar.sync.
#include "pe_core.cuh"
#include "pe_stream.cuh"
#include <cstring>

#define PROG_THREADS 1024
#define PROG_WARPS (PROG_THREADS / 32)

struct pe_program {
    pe_ctx *ctx = nullptr;
    PeOp *ops_d = nullptr;
    int nops = 0, grid = 0;
    unsigned long long *bar_d = nullptr;     // monotone arrival counter
    unsigned long long epoch = 0;            // arrivals consumed by earlier launches
    unsigned long long *ts_d = nullptr;      // nops+1 globaltimer stamps (profiling launches only)
    std::vector<int32_t> types;
    std::vector<double> bytes;
    double total_bytes = 0.0;
};

__device__ __forceinline__ unsigned long long ld_acquire_u64(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long globaltimer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// ---------------------------------------------------------------------------------------------
// ops.  gw: global warp index (consecutive indices sit on different SMs), W: warps in the grid
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double op_ld_value(const double *a, uint64_t pol) { return ld_stream_f64(a, pol); }
__device__ __forceinline__ double op_ld_value(const int8_t *a, uint64_t pol) { return ld_stream_s8(a, pol); }

// p: soff J A x yin yout S | i0 nslices i1 nrows | a alpha b beta      (S: sign codes in place of A, or null)
template <typename V>
__device__ __forceinline__ void sell_spmv_body(const PeOp &o, const V *A, int gw, int W, int lane)
{
    const int nslices = o.i0, nrows = o.i1;
    const int *soff = (const int *)o.p[0], *J = (const int *)o.p[1];
    const double *x = (const double *)o.p[3], *yin = (const double *)o.p[4];
    double *yout = (double *)o.p[5];
    const double alpha = o.a, beta = o.b;
    const uint64_t pol = l2_evict_first_policy();
    for (int s = gw; s < nslices; s += W)
    {
        const int o0 = __ldg(soff + s), w = __ldg(soff + s + 1) - o0;
        const int *j = J + (int64_t)o0 * 32 + lane;
        const V *a = A + (int64_t)o0 * 32 + lane;
        double acc = 0.0;
        int q = 0;
        for (; q + 4 <= w; q += 4)
        {
            const int c0 = ld_stream_s32(j + (q + 0) * 32, pol), c1 = ld_stream_s32(j + (q + 1) * 32, pol);
            const int c2 = ld_stream_s32(j + (q + 2) * 32, pol), c3 = ld_stream_s32(j + (q + 3) * 32, pol);
            const double a0 = op_ld_value(a + (q + 0) * 32, pol), a1 = op_ld_value(a + (q + 1) * 32, pol);
            const double a2 = op_ld_value(a + (q + 2) * 32, pol), a3 = op_ld_value(a + (q + 3) * 32, pol);
            const double x0 = __ldcg(x + c0), x1 = __ldcg(x + c1), x2 = __ldcg(x + c2), x3 = __ldcg(x + c3);
            acc += a0 * x0; acc += a1 * x1; acc += a2 * x2; acc += a3 * x3;
        }
        for (; q < w; ++q) acc += op_ld_value(a + q * 32, pol) * __ldcg(x + ld_stream_s32(j + q * 32, pol));
        const int row = s * 32 + lane;
        if (row < nrows)
        {
            double v = alpha * acc;
            if (beta != 0.0) v += beta * __ldcg(yin + row);
            yout[row] = v;
        }
    }
}
__device__ __noinline__ void op_sell_spmv(const PeOp &o, int gw, int W, int lane)
{
    if (o.p[6]) sell_spmv_body(o, (const int8_t *)o.p[6], gw, W, lane);
    else sell_spmv_body(o, (const double *)o.p[2], gw, W, lane);
}

// one colour of (l1-)Gauss-Seidel, slices [i0, i1) -- same arithmetic as k_sell_gs (pe_sell.cu)
// p: soff J A f u uext l1 | i2 ext_base
__device__ __noinline__ void op_sell_gs(const PeOp &o, int gw, int W, int lane)
{
    const int s0 = o.i0, s1 = o.i1, ext_base = o.i2;
    const int *soff = (const int *)o.p[0], *J = (const int *)o.p[1];
    const double *A = (const double *)o.p[2], *f = (const double *)o.p[3];
    double *u = (double *)o.p[4];
    const double *uext = (const double *)o.p[5], *l1 = (const double *)o.p[6];
    const uint64_t pol = l2_evict_first_policy();
#define PE_GATHER(c) ((uext && (c) >= ext_base) ? __ldcg(uext + ((c) - ext_base)) : __ldcg(u + (c)))
    for (int s = s0 + gw; s < s1; s += W)
    {
        const int o0 = __ldg(soff + s), w = __ldg(soff + s + 1) - o0;
        const int *j = J + (int64_t)o0 * 32 + lane;
        const double *a = A + (int64_t)o0 * 32 + lane;
        const int row = s * 32 + lane;
        const double d = __ldcg(l1 + row), fr = __ldcg(f + row);
        double acc = 0.0;
        int q = 0;
        int c0 = 0, c1 = 0, c2 = 0, c3 = 0;
        double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
        if (w >= 4)
        {
            c0 = ld_stream_s32(j, pol); c1 = ld_stream_s32(j + 32, pol); c2 = ld_stream_s32(j + 64, pol); c3 = ld_stream_s32(j + 96, pol);
            a0 = ld_stream_f64(a, pol); a1 = ld_stream_f64(a + 32, pol); a2 = ld_stream_f64(a + 64, pol); a3 = ld_stream_f64(a + 96, pol);
        }
        for (; q + 4 <= w; q += 4)
        {
            const double u0 = PE_GATHER(c0), u1 = PE_GATHER(c1), u2 = PE_GATHER(c2), u3 = PE_GATHER(c3);
            const double b0 = a0, b1 = a1, b2 = a2, b3 = a3;
            if (q + 8 <= w)
            {
                const int *jn = j + (q + 4) * 32; const double *an = a + (q + 4) * 32;
                c0 = ld_stream_s32(jn, pol); c1 = ld_stream_s32(jn + 32, pol); c2 = ld_stream_s32(jn + 64, pol); c3 = ld_stream_s32(jn + 96, pol);
                a0 = ld_stream_f64(an, pol); a1 = ld_stream_f64(an + 32, pol); a2 = ld_stream_f64(an + 64, pol); a3 = ld_stream_f64(an + 96, pol);
            }
            acc += b0 * u0; acc += b1 * u1; acc += b2 * u2; acc += b3 * u3;
        }
        for (; q < w; ++q) { const int c = ld_stream_s32(j + q * 32, pol); acc += ld_stream_f64(a + q * 32, pol) * PE_GATHER(c); }
        if (d != 0.0) u[row] = __ldcg(u + row) + (fr - acc) / d;
    }
#undef PE_GATHER
}

// CSR "vector" SpMV, TPR lanes per row (P, P^T and whatever has no SELL copy)
// p: I J A x yin yout | i0 nrows | a alpha b beta
template <int TPR>
__device__ __forceinline__ void csr_spmv_body(const PeOp &o, int gw, int W, int lane)
{
    const int n = o.i0;
    const int *I = (const int *)o.p[0], *J = (const int *)o.p[1];
    const double *A = (const double *)o.p[2], *x = (const double *)o.p[3], *yin = (const double *)o.p[4];
    double *yout = (double *)o.p[5];
    const double alpha = o.a, beta = o.b;
    const uint64_t pol = l2_evict_first_policy();
    constexpr int RPW = 32 / TPR;                    // rows per warp per step
    const int sub = lane / TPR, l = lane & (TPR - 1);
    for (int64_t base = (int64_t)gw * RPW; base < n; base += (int64_t)W * RPW)
    {
        const int64_t row = base + sub;
        double s = 0.0;
        if (row < n)
        {
            const int lo = __ldg(I + row), hi = __ldg(I + row + 1);
            for (int k = lo + l; k < hi; k += TPR) s += ld_stream_f64(A + k, pol) * __ldcg(x + ld_stream_s32(J + k, pol));
        }
#pragma unroll
        for (int w = TPR / 2; w > 0; w >>= 1) s += __shfl_down_sync(0xffffffffu, s, w, TPR);
        if (l == 0 && row < n)
        {
            double r = alpha * s;
            if (beta != 0.0) r += beta * __ldcg(yin + row);
            yout[row] = r;
        }
    }
}
__device__ __noinline__ void op_csr_spmv(const PeOp &o, int gw, int W, int lane)
{
    switch (o.i1)
    {
    case 1: csr_spmv_body<1>(o, gw, W, lane); break;
    case 2: csr_spmv_body<2>(o, gw, W, lane); break;
    case 4: csr_spmv_body<4>(o, gw, W, lane); break;
    case 8: csr_spmv_body<8>(o, gw, W, lane); break;
    case 16: csr_spmv_body<16>(o, gw, W, lane); break;
    default: csr_spmv_body<32>(o, gw, W, lane); break;
    }
}

// elementwise ops over n entries; gt: global thread index, T: threads in the grid
__device__ __noinline__ void op_elementwise(const PeOp &o, int64_t gt, int64_t T)
{
    const int64_t n = o.n;
    const double a = o.a, b = o.b;
    switch (o.type)
    {
    case PE_OP_PERM_IN:       // fp[pos[i]] = b[i]; up[pos[i]] = x ? x[i] : 0      p: pos b x fp up
    {
        const int *pos = (const int *)o.p[0];
        const double *bv = (const double *)o.p[1], *x = (const double *)o.p[2];
        double *fp = (double *)o.p[3], *up = (double *)o.p[4];
        for (int64_t i = gt; i < n; i += T) { const int p = __ldg(pos + i); fp[p] = __ldcg(bv + i); up[p] = x ? __ldcg(x + i) : 0.0; }
        break;
    }
    case PE_OP_PERM_IN_GS0:   // PERM_IN from a zero guess + the first colour, rows [r0, r1) (k_sell_perm_in_gs0)
    {                         //                                                    p: pos b l1 fp up | i0 r0 i1 r1
        const int *pos = (const int *)o.p[0];
        const double *bv = (const double *)o.p[1], *l1 = (const double *)o.p[2];
        double *fp = (double *)o.p[3], *up = (double *)o.p[4];
        for (int64_t i = gt; i < n; i += T)
        {
            const int p = __ldg(pos + i);
            const double d = (p >= o.i0 && p < o.i1) ? __ldcg(l1 + p) : 0.0;
            const double fr = __ldcg(bv + i), ur = 0.0, acc = 0.0;
            fp[p] = fr;
            up[p] = d != 0.0 ? ur + (fr - acc) / d : ur;
        }
        break;
    }
    case PE_OP_PERM_OUT:      // x[i] = up[pos[i]]                                  p: pos up x
    {
        const int *pos = (const int *)o.p[0];
        const double *up = (const double *)o.p[1];
        double *x = (double *)o.p[2];
        for (int64_t i = gt; i < n; i += T) x[i] = __ldcg(up + __ldg(pos + i));
        break;
    }
    case PE_OP_AXPBY:         // y = a x + b y                                      p: x y
    {
        const double *x = (const double *)o.p[0];
        double *y = (double *)o.p[1];
        if (b == 0.0) { for (int64_t i = gt; i < n; i += T) y[i] = a * __ldcg(x + i); }
        else { for (int64_t i = gt; i < n; i += T) y[i] = a * __ldcg(x + i) + b * __ldcg(y + i); }
        break;
    }
    case PE_OP_ADD3:          // z = a x + b y                                      p: x y z
    {
        const double *x = (const double *)o.p[0], *y = (const double *)o.p[1];
        double *z = (double *)o.p[2];
        for (int64_t i = gt; i < n; i += T) z[i] = a * __ldcg(x + i) + b * __ldcg(y + i);
        break;
    }
    case PE_OP_FILL:          // x = a                                               p: x
    {
        double *x = (double *)o.p[0];
        for (int64_t i = gt; i < n; i += T) x[i] = a;
        break;
    }
    case PE_OP_COPY:          // y = x                                               p: x y
    {
        const double *x = (const double *)o.p[0];
        double *y = (double *)o.p[1];
        for (int64_t i = gt; i < n; i += T) y[i] = __ldcg(x + i);
        break;
    }
    case PE_OP_SCALE:         // x *= a                                              p: x
    {
        double *x = (double *)o.p[0];
        for (int64_t i = gt; i < n; i += T) x[i] = a * __ldcg(x + i);
        break;
    }
    case PE_OP_MUL:           // x .*= d                                             p: d x
    {
        const double *d = (const double *)o.p[0];
        double *x = (double *)o.p[1];
        for (int64_t i = gt; i < n; i += T) x[i] = __ldcg(x + i) * __ldcg(d + i);
        break;
    }
    case PE_OP_AXPY_DEV:      // y += sign * slot * x (no-op when the scalar is 0)  p: slot x y | a sign
    {
        const double s = a * __ldcg((const double *)o.p[0]);
        if (s == 0.0) break;
        const double *x = (const double *)o.p[1];
        double *y = (double *)o.p[2];
        for (int64_t i = gt; i < n; i += T) y[i] = __ldcg(y + i) + s * __ldcg(x + i);
        break;
    }
    case PE_OP_XPBY_DEV:      // y = x + slot * y                                    p: x slot y
    {
        const double *x = (const double *)o.p[0];
        const double s = __ldcg((const double *)o.p[1]);
        double *y = (double *)o.p[2];
        for (int64_t i = gt; i < n; i += T) y[i] = __ldcg(x + i) + s * __ldcg(y + i);
        break;
    }
    default: break;
    }
}

// deterministic dot: fixed per-thread strides, fixed shuffle tree, fixed order over CTAs
// p: x y partials
__device__ __noinline__ void op_dot(const PeOp &o, int64_t gt, int64_t T, double *red)
{
    const double *x = (const double *)o.p[0], *y = (const double *)o.p[1];
    double *partials = (double *)o.p[2];
    double acc = 0.0;
    for (int64_t i = gt; i < o.n; i += T) acc += __ldcg(x + i) * __ldcg(y + i);
#pragma unroll
    for (int w = 16; w > 0; w >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, w);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) red[warp] = acc;
    __syncthreads();
    if (warp == 0)
    {
        double v = red[lane];
#pragma unroll
        for (int w = 16; w > 0; w >>= 1) v += __shfl_down_sync(0xffffffffu, v, w);
        if (lane == 0) partials[blockIdx.x] = v;
    }
}
// p: partials out | i0 nparts      (CTA 0 only)
__device__ __noinline__ void op_dot_fin(const PeOp &o, double *red)
{
    if (blockIdx.x != 0) return;
    const double *partials = (const double *)o.p[0];
    double *out = (double *)o.p[1];
    double acc = 0.0;
    for (int i = threadIdx.x; i < o.i0; i += PROG_THREADS) acc += __ldcg(partials + i);
#pragma unroll
    for (int w = 16; w > 0; w >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, w);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) red[warp] = acc;
    __syncthreads();
    if (warp == 0)
    {
        double v = red[lane];
#pragma unroll
        for (int w = 16; w > 0; w >>= 1) v += __shfl_down_sync(0xffffffffu, v, w);
        if (lane == 0) out[0] = v;
    }
}

__global__ void __launch_bounds__(PROG_THREADS, 1)
k_program(const PeOp *__restrict__ ops, int nops, unsigned long long *bar, unsigned long long epoch,
          unsigned long long *ts)
{
    __shared__ PeOp op;
    __shared__ double red[PROG_WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int W = gridDim.x * PROG_WARPS;
    const int gw = warp * gridDim.x + blockIdx.x;              // neighbouring work items -> different SMs
    const int64_t T = (int64_t)gridDim.x * PROG_THREADS;
    const int64_t gt = (int64_t)blockIdx.x * PROG_THREADS + threadIdx.x;
    unsigned long long target = epoch;
    if (ts && gt == 0) ts[0] = globaltimer_ns();
    for (int k = 0; k < nops; ++k)
    {
        if (threadIdx.x < 16) ((unsigned long long *)&op)[threadIdx.x] = __ldg((const unsigned long long *)(ops + k) + threadIdx.x);
        __syncthreads();
        switch (op.type)
        {
        case PE_OP_SELL_SPMV: op_sell_spmv(op, gw, W, lane); break;
        case PE_OP_SELL_GS: op_sell_gs(op, gw, W, lane); break;
        case PE_OP_CSR_SPMV: op_csr_spmv(op, gw, W, lane); break;
        case PE_OP_DOT: op_dot(op, gt, T, red); break;
        case PE_OP_DOT_FIN: op_dot_fin(op, red); break;
        case PE_OP_PCG_STEP:       // p: slots | i0 phase i1 iter i2 max_iter | a rel b abs
            if (gt == 0) pe_pcg_scalar_step_dev((double *)op.p[0], op.i0, op.i1, op.i2, op.a, op.b);
            break;
        default: op_elementwise(op, gt, T); break;
        }
        // grid-wide barrier
        target += gridDim.x;
        __syncthreads();
        if (threadIdx.x == 0)
        {
            __threadfence();
            atomicAdd(bar, 1ULL);
            while (ld_acquire_u64(bar) < target) { }
            if (ts && blockIdx.x == 0) ts[k + 1] = globaltimer_ns();
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
void pe_rec_fail(pe_ctx *ctx, const char *file, int line)
{
    if (!ctx->rec || ctx->rec->failed) return;
    ctx->rec->failed = true;
    ctx->rec->why = std::string("a kernel without a program op was launched at ") + file + ":" + std::to_string(line);
}

extern "C" int pe_program_begin(pe_ctx *ctx)
{
    PE_CHECK(ctx, "null context");
    PE_CHECK(!ctx->rec && !ctx->capturing, "a recording or graph capture is already active");
    PE_CHECK(ctx->nranks == 1, "programs are single-rank (halo exchanges are NCCL calls)");
    ctx->rec = new pe_recorder();
    return 0;
}

extern "C" int pe_program_free(pe_program *p)
{
    if (!p) return 0;
    cudaStreamSynchronize(p->ctx->stream);
    if (p->ops_d) cudaFree(p->ops_d);
    if (p->bar_d) cudaFree(p->bar_d);
    if (p->ts_d) cudaFree(p->ts_d);
    delete p;
    return 0;
}

extern "C" int pe_program_end(pe_ctx *ctx, pe_program **out)
{
    PE_CHECK(ctx && ctx->rec && out, "no recording active");
    pe_recorder *rec = ctx->rec;
    ctx->rec = nullptr;
    std::unique_ptr<pe_recorder> hold(rec);
    *out = nullptr;
    if (rec->failed) { pe_set_error("program recording failed: " + rec->why); return 4; }
    PE_CHECK(!rec->ops.empty(), "empty program");
    int coop = 0, nsm = 0, nb = 0;
    PE_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, ctx->device));
    PE_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, ctx->device));
    PE_CHECK(coop, "device does not support cooperative launches");
    PE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_program, PROG_THREADS, 0));
    PE_CHECK(nb >= 1, "k_program does not fit on an SM");
    pe_program *p = new pe_program();
    p->ctx = ctx;
    p->nops = (int)rec->ops.size();
    p->grid = nsm;                                  // one CTA per SM
    PE_CHECK(p->grid <= PE_MAX_PARTIALS && p->grid <= PROG_THREADS, "grid too large for the reduction scratch");
    for (size_t k = 0; k < rec->ops.size(); ++k)
    {
        PeOp &o = rec->ops[k];
        if (o.type == PE_OP_DOT_FIN) o.i0 = p->grid;
        p->types.push_back(o.type);
        p->total_bytes += rec->bytes[k];
    }
    p->bytes = rec->bytes;
    PE_CUDA(cudaMalloc(&p->ops_d, sizeof(PeOp) * rec->ops.size()));
    PE_CUDA(cudaMalloc(&p->bar_d, sizeof(unsigned long long)));
    PE_CUDA(cudaMemcpyAsync(p->ops_d, rec->ops.data(), sizeof(PeOp) * rec->ops.size(), cudaMemcpyHostToDevice, ctx->stream));
    PE_CUDA(cudaMemsetAsync(p->bar_d, 0, sizeof(unsigned long long), ctx->stream));
    PE_CUDA(cudaStreamSynchronize(ctx->stream));
    *out = p;
    return 0;
}

static int launch_program(pe_ctx *ctx, pe_program *p, unsigned long long *ts)
{
    const PeOp *ops = p->ops_d;
    int nops = p->nops;
    unsigned long long *bar = p->bar_d, epoch = p->epoch;
    void *args[] = {(void *)&ops, (void *)&nops, (void *)&bar, (void *)&epoch, (void *)&ts};
    PE_CUDA(cudaLaunchCooperativeKernel((const void *)k_program, dim3(p->grid), dim3(PROG_THREADS), args, 0, ctx->stream));
    p->epoch += (unsigned long long)p->nops * (unsigned long long)p->grid;
    ctx->launches++;
    return 0;
}

extern "C" int pe_program_launch(pe_ctx *ctx, pe_program *p)
{
    PE_CHECK(ctx && p && p->ctx == ctx, "bad arguments");
    PE_CHECK(!ctx->rec, "cannot launch a program while recording");
    return launch_program(ctx, p, nullptr);
}

extern "C" int pe_program_info(const pe_program *p, int32_t *nops, double *algorithmic_bytes)
{
    if (nops) *nops = p->nops;
    if (algorithmic_bytes) *algorithmic_bytes = p->total_bytes;
    return 0;
}

// one extra launch with per-op globaltimer stamps: duration (us), type and algorithmic bytes of
// every op, in program order (arrays of nops entries; NULL = skip)
extern "C" int pe_program_profile(pe_ctx *ctx, pe_program *p, int32_t *types, double *usec, double *bytes)
{
    PE_CHECK(ctx && p && p->ctx == ctx, "bad arguments");
    if (!p->ts_d) PE_CUDA(cudaMalloc(&p->ts_d, sizeof(unsigned long long) * (size_t)(p->nops + 1)));
    PE_TRY(launch_program(ctx, p, p->ts_d));
    std::vector<unsigned long long> ts((size_t)p->nops + 1);
    PE_CUDA(cudaMemcpyAsync(ts.data(), p->ts_d, sizeof(unsigned long long) * ts.size(), cudaMemcpyDeviceToHost, ctx->stream));
    PE_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < p->nops; ++k)
    {
        if (types) types[k] = p->types[k];
        if (usec) usec[k] = 1e-3 * (double)(ts[k + 1] - ts[k]);
        if (bytes) bytes[k] = p->bytes[k];
    }
    return 0;
}

extern "C" int pe_ctx_is_recording(const pe_ctx *ctx) { return ctx->rec ? 1 : 0; }
