// pe_sell.cu -- sliced-ELL (SELL-32) storage and the thread-per-row streaming kernels built
// on it: SpMV / residual / prolongation (K1/K2/K7) and one colour of multicolour
// (l1-)Gauss-Seidel (K4).
//
// Layout: rows are grouped in slices of 32 (one warp); slice s stores w_s = max row length
// of its rows, column-major: entry q of lane l sits at (soff[s] + q) * 32 + l.  A warp-wide
// load of J is one 128-byte line and of A two lines (always fully used), and because
// consecutive rows of a (locally) structured operator couple to consecutive columns, the
// x-gather of one q touches ~8-10 sectors instead of the ~25 of the CSR layout.  Short rows
// are padded with (col = last valid column of the row, val = 0).
//
// The SELL copy is what the kernels stream; the CSR block stays the interchange format of
// the C ABI (upload/download/SpGEMM).  Algorithmic bytes are counted on the CSR figures
// (12 B per true non-zero), see DESIGN.md.
#include "pe_core.cuh"
#include "pe_stream.cuh"
#include <cub/cub.cuh>
#include <algorithm>

// ---------------------------------------------------------------------------
// build
// ---------------------------------------------------------------------------
__device__ __forceinline__ int sell_src_row(const int *rowmap, int k, int nrows_src)
{
    if (rowmap) return rowmap[k];
    return k < nrows_src ? k : -1;
}

// one warp per slice: width = max over its rows of (diag + offd) row length
__global__ void k_sell_widths(int nslices, int nrows_src, const int *__restrict__ rowmap,
                              const int *__restrict__ dI, const int *__restrict__ oI, int *w)
{
    const int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (s >= nslices) return;
    const int r = sell_src_row(rowmap, s * 32 + lane, nrows_src);
    int len = 0;
    if (r >= 0) { len = dI[r + 1] - dI[r]; if (oI) len += oI[r + 1] - oI[r]; }
    len = __reduce_max_sync(0xffffffffu, len);
    if (lane == 0) { w[s + 1] = len; if (s == 0) w[0] = 0; }
}

__global__ void k_sell_fill(int nslices, int nrows_src, const int *__restrict__ rowmap,
                            const int *__restrict__ colpos, int ext_base,
                            const int *__restrict__ dI, const int *__restrict__ dJ, const double *__restrict__ dA,
                            const int *__restrict__ oI, const int *__restrict__ oJ, const double *__restrict__ oA,
                            const int *__restrict__ soff, int *J, double *A)
{
    const int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (s >= nslices) return;
    const int r = sell_src_row(rowmap, s * 32 + lane, nrows_src);
    const int o0 = soff[s], w = soff[s + 1] - o0;
    int64_t p = (int64_t)o0 * 32 + lane;
    int q = 0, last = 0;
    if (r >= 0)
    {
        for (int t = dI[r]; t < dI[r + 1]; ++t, ++q, p += 32)
        {
            last = colpos ? colpos[dJ[t]] : dJ[t];
            J[p] = last; A[p] = dA[t];
        }
        if (oI) for (int t = oI[r]; t < oI[r + 1]; ++t, ++q, p += 32)
        {
            last = ext_base + oJ[t];
            J[p] = last; A[p] = oA[t];
        }
    }
    for (; q < w; ++q, p += 32) { J[p] = last; A[p] = 0.0; }
}

void pe_sell_free(DevSELL &m)
{
    if (m.soff) cudaFree(m.soff);
    if (m.J) cudaFree(m.J);
    if (m.A) cudaFree(m.A);
    if (m.S) cudaFree(m.S);
    m = DevSELL();
}

// rowmap_d: nslices*32 source rows (-1 = padding row) or null for the identity over diag.nrows;
// colpos_d: new index of every diag column or null; ghost column j becomes ext_base + j.
int pe_sell_build(pe_ctx *ctx, const DevCSR &diag, const DevCSR *offd, const int32_t *rowmap_d, int32_t nslices,
                  const int32_t *colpos_d, int32_t ext_base, DevSELL &out, std::vector<int32_t> *soff_host)
{
    cudaStream_t st = ctx->stream;
    if (!rowmap_d) nslices = (diag.nrows + 31) / 32;
    out = DevSELL();
    out.nslices = nslices;
    out.nrows = diag.nrows;
    PE_CUDA(cudaMalloc(&out.soff, sizeof(int32_t) * (size_t)(nslices + 1)));
    if (nslices == 0) { PE_CUDA(cudaMemsetAsync(out.soff, 0, sizeof(int32_t), st)); return 0; }
    const int *oI = (offd && offd->nnz > 0) ? offd->I : nullptr;
    const int grid = pe_grid_for((int64_t)nslices * 32, 256);
    k_sell_widths<<<grid, 256, 0, st>>>(nslices, diag.nrows, rowmap_d, diag.I, oI, out.soff);
    PE_LAUNCHED(ctx);
    void *tmp = nullptr; size_t tb = 0;
    cub::DeviceScan::InclusiveSum(nullptr, tb, out.soff, out.soff, nslices + 1, st);
    PE_CUDA(cudaMalloc(&tmp, tb));
    PE_CUDA(cub::DeviceScan::InclusiveSum(tmp, tb, out.soff, out.soff, nslices + 1, st));
    ctx->launches++;
    std::vector<int32_t> soff_h((size_t)nslices + 1);
    PE_CUDA(cudaMemcpyAsync(soff_h.data(), out.soff, sizeof(int32_t) * (size_t)(nslices + 1), cudaMemcpyDeviceToHost, st));
    PE_CUDA(cudaStreamSynchronize(st));
    cudaFree(tmp);
    const int32_t total = soff_h[nslices];
    out.wmax = 0;
    for (int32_t k = 0; k < nslices; ++k) out.wmax = std::max(out.wmax, soff_h[k + 1] - soff_h[k]);
    if (soff_host) soff_host->swap(soff_h);
    out.nstored = (int64_t)total * 32;
    PE_CUDA(cudaMalloc(&out.J, sizeof(int32_t) * (size_t)(out.nstored > 0 ? out.nstored : 1)));
    PE_CUDA(cudaMalloc(&out.A, sizeof(double) * (size_t)(out.nstored > 0 ? out.nstored : 1)));
    if (out.nstored > 0)
    {
        k_sell_fill<<<grid, 256, 0, st>>>(nslices, diag.nrows, rowmap_d, colpos_d, ext_base, diag.I, diag.J, diag.A,
                                          oI, oI ? offd->J : nullptr, oI ? offd->A : nullptr, out.soff, out.J, out.A);
        PE_LAUNCHED(ctx);
    }
    return 0;
}

// sign codes of the stored values; *bad is set when a value is not -1, 0 or +1 (-0.0 counts as 0: the row sum starts
// at +0.0 and an fma only returns -0.0 from a -0.0 addend, so a +0 or -0 product leaves every sum bit-identical)
__global__ void k_sell_signs(int64_t n, const double *__restrict__ A, int8_t *S, int *bad)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double v = A[i];
    const int8_t c = v == 1.0 ? 1 : (v == -1.0 ? -1 : 0);
    if (c == 0 && v != 0.0) *bad = 1;
    S[i] = c;
}

// Replace the values of a SELL copy by sign codes when all of them are -1, 0 or +1 (the discrete derivatives of the
// fine de Rham sequence): 5 B per stored entry instead of 12, decoded to the same doubles.
static int sell_encode_signs(pe_ctx *ctx, DevSELL &s)
{
    if (s.nstored == 0) return 0;
    cudaStream_t st = ctx->stream;
    int *bad_d = nullptr, bad = 0;
    PE_CUDA(cudaMalloc(&s.S, (size_t)s.nstored));
    PE_CUDA(cudaMalloc(&bad_d, sizeof(int)));
    PE_CUDA(cudaMemsetAsync(bad_d, 0, sizeof(int), st));
    k_sell_signs<<<pe_grid_for(s.nstored, 256), 256, 0, st>>>(s.nstored, s.A, s.S, bad_d);
    PE_LAUNCHED(ctx);
    PE_CUDA(cudaMemcpyAsync(&bad, bad_d, sizeof(int), cudaMemcpyDeviceToHost, st));
    PE_CUDA(cudaStreamSynchronize(st));
    cudaFree(bad_d);
    if (bad) { cudaFree(s.S); s.S = nullptr; }
    else { cudaFree(s.A); s.A = nullptr; }
    return 0;
}

// Lazily attach a SELL copy to a CSR block used by SpMV.  Rejected (state -1) when padding
// would add more than 25 % to the stream.
int pe_sell_for_spmv(pe_ctx *ctx, DevCSR &m)
{
    if (m.sell_state != 0) return 0;
    m.sell_state = -1;
    if (m.nnz == 0 || m.nrows == 0) return 0;
    DevSELL *s = new DevSELL();
    int rc = pe_sell_build(ctx, m, nullptr, nullptr, 0, nullptr, 0, *s);
    if (rc) { delete s; return rc; }
    if ((double)s->nstored > 1.25 * (double)m.nnz) { pe_sell_free(*s); delete s; return 0; }
    rc = sell_encode_signs(ctx, *s);
    if (rc) { pe_sell_free(*s); delete s; return rc; }
    m.sell = s;
    m.sell_state = 1;
    return 0;
}

// ---------------------------------------------------------------------------
// Entry groups.  A thread walks its row in groups of G entries: the (col,val) loads of a whole
// group are issued back to back, then the G gathers, and the loads of group g+1 are in flight
// while the gathers of group g are outstanding.  The last group is predicated on the slice
// width (warp-uniform), so a row costs ceil(w/G)+2 dependent memory round trips instead of one
// per tail entry.  SINGLE: every slice of the launch has w <= G -- one group, no loop; this is
// what short rows (RT0: 11, D: 2, D^T: 4) need to keep enough bytes in flight.  The products are
// accumulated in entry order in every variant, so the result does not depend on G.
// ---------------------------------------------------------------------------
template <bool PRO>
__device__ __forceinline__ double sell_load_value(const double *a, uint64_t pol)
{ return PRO ? ld_stream_f64_pro(a, pol) : ld_stream_f64(a, pol); }
template <bool PRO>
__device__ __forceinline__ double sell_load_value(const int8_t *a, uint64_t pol)
{ return PRO ? ld_stream_s8_pro(a, pol) : ld_stream_s8(a, pol); }

template <int G, bool PRO = false, typename V>
__device__ __forceinline__ void sell_load_group(const int *j, const V *a, int q, int w, uint64_t pol,
                                                int (&c)[G], double (&v)[G])
{
#pragma unroll
    for (int k = 0; k < G; ++k)
        if (q + k < w)
        {
            c[k] = PRO ? ld_stream_s32_pro(j + (q + k) * 32, pol) : ld_stream_s32(j + (q + k) * 32, pol);
            v[k] = sell_load_value<PRO>(a + (q + k) * 32, pol);
        }
}

// pdl_wait() has acquire semantics only: ptxas is free to sink the (independent) prologue loads
// below it, which would serialise them behind the predecessor kernel.  Making a harmless
// instruction depend on every loaded word pins the loads ahead of the wait: the gathers need the
// column indices anyway, so nothing is lost when there is no predecessor to overlap with.
template <int G>
__device__ __forceinline__ void sell_pin_group_then_wait(const int (&c)[G], const double (&v)[G], int w)
{
    int t = 0;
#pragma unroll
    for (int k = 0; k < G; ++k) if (k < w) t ^= c[k] ^ __double2hiint(v[k]) ^ __double2loint(v[k]);
    if (t == 0x5bd1e995) pdl_trigger();      // a second trigger is a no-op
    pdl_wait();
}

// ---------------------------------------------------------------------------
// SpMV: yout = alpha * A x + beta * yin   (thread per row, warp per slice; V: double values or int8 sign codes)
// ---------------------------------------------------------------------------
template <int G, bool SINGLE, typename V>
__global__ void __launch_bounds__(256, ((SINGLE || G <= 4) ? 4 : 2))
k_sell_spmv(int nslices, int nrows, const int *__restrict__ soff, const int *__restrict__ J,
            const V *__restrict__ A, const double *x, double alpha, double beta,
            const double *yin, double *yout)
{
    // x, yin, f, u, uext are written by preceding kernels that may still be draining when this one
    // starts (PDL): they are plain pointers (no __restrict__/ld.global.nc) and only read after pdl_wait()
    pdl_trigger();
    const int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (s >= nslices) { pdl_wait(); return; }
    const int o0 = ld_nc_s32_pro(soff + s), w = ld_nc_s32_pro(soff + s + 1) - o0;
    const int *j = J + (int64_t)o0 * 32 + lane;
    const V *a = A + (int64_t)o0 * 32 + lane;
    const uint64_t pol = l2_evict_first_policy();
    double acc = 0.0;
    int c[G]; double v[G];
    sell_load_group<G, true>(j, a, 0, w, pol, c, v);
    sell_pin_group_then_wait<G>(c, v, w);    // x (and yin) come from the preceding kernel
    const int row = s * 32 + lane;
    const double yv = (beta != 0.0 && row < nrows) ? yin[row] : 0.0;   // issued with the first gathers, not after them
    for (int q = 0; q < w; q += G)
    {
        double xv[G], b[G];
#pragma unroll
        for (int k = 0; k < G; ++k) if (q + k < w) { xv[k] = x[c[k]]; b[k] = v[k]; }
        if (!SINGLE && q + G < w) sell_load_group<G>(j, a, q + G, w, pol, c, v);
#pragma unroll
        for (int k = 0; k < G; ++k) if (q + k < w) acc = __fma_rn(b[k], xv[k], acc);   // explicit: same rounding in every variant
        if (SINGLE) break;
    }
    if (row < nrows)
    {
        double r = alpha * acc;
        if (beta != 0.0) r += beta * yv;
        yout[row] = r;
    }
}

// ---------------------------------------------------------------------------
// L2 policy of the gathers (PE_TUNE_GATHER_KEEP_PCT)
// ---------------------------------------------------------------------------
__global__ void k_make_policy(int pct, uint64_t *out)
{
    uint64_t p;
    switch (pct)
    {
    case 25: asm("createpolicy.fractional.L2::evict_last.L2::evict_unchanged.b64 %0, 0.25;" : "=l"(p)); break;
    case 50: asm("createpolicy.fractional.L2::evict_last.L2::evict_unchanged.b64 %0, 0.5;" : "=l"(p)); break;
    case 60: asm("createpolicy.fractional.L2::evict_last.L2::evict_unchanged.b64 %0, 0.6;" : "=l"(p)); break;
    case 75: asm("createpolicy.fractional.L2::evict_last.L2::evict_unchanged.b64 %0, 0.75;" : "=l"(p)); break;
    case 90: asm("createpolicy.fractional.L2::evict_last.L2::evict_unchanged.b64 %0, 0.9;" : "=l"(p)); break;
    case 100: asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p)); break;
    default: asm("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p)); break;
    }
    *out = p;
}
int pe_make_gather_policy(pe_ctx *ctx, int keep_pct, uint64_t *pol)
{
    uint64_t *d = nullptr;
    PE_CUDA(cudaMalloc(&d, sizeof(uint64_t)));
    k_make_policy<<<1, 1, 0, ctx->stream>>>(keep_pct, d);
    PE_LAUNCHED(ctx);
    PE_CUDA(cudaMemcpyAsync(pol, d, sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    PE_CUDA(cudaStreamSynchronize(ctx->stream));
    cudaFree(d);
    return 0;
}
__device__ __forceinline__ double ld_hint_f64(const double *p, uint64_t pol)
{
    double v;
    asm volatile("ld.global.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol) : "memory");
    return v;
}

// group size for slices up to wmax entries wide (0 <= forced: PE_TUNE_SELL_GROUP)
static void sell_pick_group(int wmax, int &G, bool &single)
{
    const int forced = pe_get_tuning(PE_TUNE_SELL_GROUP);
    if (forced == 4 || forced == 8 || forced == 12) G = forced;
    else if (wmax <= 4) G = 4;
    else if (wmax <= 8) G = 8;
    else if (wmax <= 12) G = 12;
    else if (wmax <= 24) G = 8;
    else G = 4;
    single = wmax <= G;
}

// pe_variant_counts slot of a (G, single) choice: base = PE_VARIANT_SELL_GS_G4_SINGLE or PE_VARIANT_SELL_SPMV_G4_SINGLE
static int sell_group_slot(int base, int G, bool single)
{
    return base + 2 * (G / 4 - 1) + (single ? 0 : 1);
}

int pe_launch_sell_spmv(pe_ctx *ctx, const DevSELL &S, double alpha, const double *x, double beta,
                        const double *yin, double *yout)
{
    if (S.nslices == 0) return 0;
    if (ctx->rec)
    {
        PeOp o = pe_op(PE_OP_SELL_SPMV); o.i0 = S.nslices; o.i1 = S.nrows; o.a = alpha; o.b = beta;
        o.p[0] = S.soff; o.p[1] = S.J; o.p[2] = S.A; o.p[3] = x; o.p[4] = yin; o.p[5] = yout; o.p[6] = S.S;
        pe_rec_push(ctx, o, -1.0);
        return 0;
    }
    const int grid = pe_grid_for((int64_t)S.nslices * 32, 256);
    int G; bool single;
    sell_pick_group(S.wmax, G, single);
    pe_variant_add(sell_group_slot(PE_VARIANT_SELL_SPMV_G4_SINGLE, G, single), (int64_t)S.nslices * 32);
#define PE_SPMV_V(GG, SS, VV, AA) PE_CUDA(pe_launch_k(ctx, k_sell_spmv<GG, SS, VV>, grid, 256, S.nslices, S.nrows, S.soff, S.J, AA, x, alpha, beta, yin, yout))
#define PE_SPMV(GG, SS) do { if (S.S) PE_SPMV_V(GG, SS, int8_t, (const int8_t *)S.S); else PE_SPMV_V(GG, SS, double, (const double *)S.A); } while (0)
    if (G == 4) { if (single) PE_SPMV(4, true); else PE_SPMV(4, false); }
    else if (G == 8) { if (single) PE_SPMV(8, true); else PE_SPMV(8, false); }
    else { if (single) PE_SPMV(12, true); else PE_SPMV(12, false); }
#undef PE_SPMV
#undef PE_SPMV_V
    PE_LAUNCHED(ctx);
    return 0;
}

// ---------------------------------------------------------------------------
// One colour of (l1-)Gauss-Seidel on the colour-ordered SELL copy: slices [s0, s1), in-place
// update of u (colour-ordered numbering, padded rows have l1 = 0 and are skipped).  Columns
// >= ext_base address the halo.  Rows of one colour are mutually independent, so no thread
// reads a value another thread of this launch writes.
// ---------------------------------------------------------------------------
template <int G, bool SINGLE, bool OFFD>
__global__ void __launch_bounds__(256, ((SINGLE || G <= 4) ? 4 : 2))
k_sell_gs(int s0, int s1, const int *__restrict__ soff, const int *__restrict__ J, const double *__restrict__ A,
          int ext_base, const double *f, double *u, const double *uext,
          const double *__restrict__ l1, uint64_t pol_u)
{
    pdl_trigger();
    const int s = s0 + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (s >= s1) { pdl_wait(); return; }
    const int o0 = ld_nc_s32_pro(soff + s), w = ld_nc_s32_pro(soff + s + 1) - o0;
    const int *j = J + (int64_t)o0 * 32 + lane;
    const double *a = A + (int64_t)o0 * 32 + lane;
    const int row = s * 32 + lane;
    const uint64_t pol = l2_evict_first_policy();
    const double d = ld_stream_f64_pro(l1 + row, pol);       // l1, f: read once per sweep -> streaming, like the matrix
    double acc = 0.0;
#define PE_GATHER(cc) ((OFFD && (cc) >= ext_base) ? uext[(cc) - ext_base] : ld_hint_f64(u + (cc), pol_u))
    int c[G]; double v[G];
    sell_load_group<G, true>(j, a, 0, w, pol, c, v);
    sell_pin_group_then_wait<G>(c, v, w);    // u, f (and the halo) come from the preceding kernels
    const double fr = ld_hint_f64(f + row, pol), ur = u[row];   // issued with the first gathers: one round trip less at the end
    for (int q = 0; q < w; q += G)
    {
        double uv[G], b[G];
#pragma unroll
        for (int k = 0; k < G; ++k) if (q + k < w) { uv[k] = PE_GATHER(c[k]); b[k] = v[k]; }
        if (!SINGLE && q + G < w) sell_load_group<G>(j, a, q + G, w, pol, c, v);
#pragma unroll
        for (int k = 0; k < G; ++k) if (q + k < w) acc = __fma_rn(b[k], uv[k], acc);   // explicit: same rounding in every variant
        if (SINGLE) break;
    }
#undef PE_GATHER
    if (d != 0.0) u[row] = ur + (fr - acc) / d;
}

int pe_launch_sell_gs(pe_ctx *ctx, const DevSELL &S, int s0, int s1, int wmax, int ext_base, const double *f, double *u,
                      const double *uext, const double *l1, uint64_t pol_gather)
{
    if (s1 <= s0) return 0;
    if (ctx->rec)
    {
        PeOp o = pe_op(PE_OP_SELL_GS); o.i0 = s0; o.i1 = s1; o.i2 = ext_base;
        o.p[0] = S.soff; o.p[1] = S.J; o.p[2] = S.A; o.p[3] = f; o.p[4] = u; o.p[5] = uext; o.p[6] = l1;
        pe_rec_push(ctx, o, -1.0);
        return 0;
    }
    const int grid = pe_grid_for((int64_t)(s1 - s0) * 32, 256);
    int G; bool single;
    sell_pick_group(wmax > 0 ? wmax : S.wmax, G, single);
    pe_variant_add(sell_group_slot(PE_VARIANT_SELL_GS_G4_SINGLE, G, single), (int64_t)(s1 - s0) * 32);
#define PE_GS(GG, SS, OO) PE_CUDA(pe_launch_k(ctx, k_sell_gs<GG, SS, OO>, grid, 256, s0, s1, S.soff, S.J, S.A, ext_base, f, u, uext, l1, pol_gather))
#define PE_GS2(GG, SS) do { if (uext) PE_GS(GG, SS, true); else PE_GS(GG, SS, false); } while (0)
    if (G == 4) { if (single) PE_GS2(4, true); else PE_GS2(4, false); }
    else if (G == 8) { if (single) PE_GS2(8, true); else PE_GS2(8, false); }
    else { if (single) PE_GS2(12, true); else PE_GS2(12, false); }
#undef PE_GS2
#undef PE_GS
    PE_LAUNCHED(ctx);
    return 0;
}

// colour-ordered <-> caller numbering
__global__ void k_sell_perm_in(int n, const int *__restrict__ pos, const double *b,
                               const double *x, double *fp, double *up)
{
    pdl_trigger();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int p = i < n ? pos[i] : 0;
    pdl_wait();
    if (i >= n) return;
    fp[p] = b[i];
    up[p] = x ? x[i] : 0.0;
}
__global__ void k_sell_perm_out(int n, const int *__restrict__ pos, const double *up, double *x)
{
    pdl_trigger();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int p = i < n ? pos[i] : 0;
    pdl_wait();
    if (i < n) x[i] = up[p];
}
int pe_launch_perm_in(pe_ctx *ctx, int n, const int *pos, const double *b, const double *x, double *fp, double *up)
{
    if (n == 0) return 0;
    if (ctx->rec)
    {
        PeOp o = pe_op(PE_OP_PERM_IN); o.n = n; o.p[0] = pos; o.p[1] = b; o.p[2] = x; o.p[3] = fp; o.p[4] = up;
        pe_rec_push(ctx, o, 0.0);   // renumbering is our overhead, not algorithmic traffic
        return 0;
    }
    PE_CUDA(pe_launch_k(ctx, k_sell_perm_in, pe_grid_for(n, 256), 256, n, pos, b, x, fp, up));
    PE_LAUNCHED(ctx);
    return 0;
}

// Zero initial guess: perm_in of f, and the first colour of the sweep in the same pass.  u is +0 everywhere (ghosts
// too), so every gather of that colour returns +0 and its row sum is +0 (fma(a, +0, +0) = +0 for finite a): the rows
// [r0, r1) of that colour get k_sell_gs's update with acc = 0 -- the same expression, so the same bits, signed zeros
// included -- and every other row gets the 0 perm_in writes.
__global__ void k_sell_perm_in_gs0(int n, const int *__restrict__ pos, const double *b, int r0, int r1,
                                   const double *__restrict__ l1, double *fp, double *up)
{
    pdl_trigger();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int p = i < n ? pos[i] : 0;
    const double d = (i < n && p >= r0 && p < r1) ? l1[p] : 0.0;
    pdl_wait();
    if (i >= n) return;
    const double fr = b[i], ur = 0.0, acc = 0.0;
    fp[p] = fr;
    up[p] = d != 0.0 ? ur + (fr - acc) / d : ur;
}
int pe_launch_perm_in_gs0(pe_ctx *ctx, int n, const int *pos, const double *b, int r0, int r1, const double *l1,
                          double *fp, double *up)
{
    if (n == 0) return 0;
    if (ctx->rec)
    {
        PeOp o = pe_op(PE_OP_PERM_IN_GS0); o.n = n; o.i0 = r0; o.i1 = r1;
        o.p[0] = pos; o.p[1] = b; o.p[2] = l1; o.p[3] = fp; o.p[4] = up;
        pe_rec_push(ctx, o, 0.0);
        return 0;
    }
    PE_CUDA(pe_launch_k(ctx, k_sell_perm_in_gs0, pe_grid_for(n, 256), 256, n, pos, b, r0, r1, l1, fp, up));
    PE_LAUNCHED(ctx);
    return 0;
}
int pe_launch_perm_out(pe_ctx *ctx, int n, const int *pos, const double *up, double *x)
{
    if (n == 0) return 0;
    if (ctx->rec)
    {
        PeOp o = pe_op(PE_OP_PERM_OUT); o.n = n; o.p[0] = pos; o.p[1] = up; o.p[2] = x;
        pe_rec_push(ctx, o, 0.0);
        return 0;
    }
    PE_CUDA(pe_launch_k(ctx, k_sell_perm_out, pe_grid_for(n, 256), 256, n, pos, up, x));
    PE_LAUNCHED(ctx);
    return 0;
}
