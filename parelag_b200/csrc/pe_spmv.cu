// pe_spmv.cu -- K1/K2/K7: ParCSR SpMV (diag+offd), explicit-transpose SpMV^T, residual.
//
// Kernel: CSR "vector" SpMV with TPR (threads per row, power of two <= 32) lanes per
// row.  Consecutive lane groups own consecutive rows, so a warp streams one contiguous
// run of (col,val) pairs of 32/TPR rows: loads of J (int32) and A (fp64) are coalesced
// and read exactly once from HBM (ld.global.nc, no L1 allocation so L1 stays for the x
// gather).  Algorithmic bytes per launch: 12*nnz + 4*(n+1) + 8*n_cols + 8*n (+8*n when
// beta != 0), see DESIGN.md.
#include "pe_core.cuh"
#include <cub/cub.cuh>

__device__ __forceinline__ double ld_stream_f64(const double *p)
{
    double v;
    asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ int ld_stream_s32(const int *p)
{
    int v;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}

template <int TPR>
__global__ void __launch_bounds__(256)
k_spmv(int n, const int *__restrict__ dI, const int *__restrict__ dJ, const double *__restrict__ dA,
       const int *__restrict__ oI, const int *__restrict__ oJ, const double *__restrict__ oA,
       const double *x, const double *xext,
       double alpha, double beta, const double *yin, double *yout)
{
    // PDL (pe_launch_k): the first row extent is fetched before the wait; x, xext, yin after it
    pdl_trigger();
    const int lane = threadIdx.x & (TPR - 1);
    const int64_t gid = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / TPR;
    const int64_t ngroups = ((int64_t)gridDim.x * blockDim.x) / TPR;
    int lo = 0, hi = 0;
    if (gid < n) { lo = dI[gid]; hi = dI[gid + 1]; }
    if ((lo ^ hi) == 0x5bd1e995 && hi == -7) pdl_trigger();      // pins the two loads ahead of the wait
    pdl_wait();
    for (int64_t row = gid; row < n; row += ngroups) {
        if (row != gid) { lo = dI[row]; hi = dI[row + 1]; }
        double s = 0.0;
        for (int k = lo + lane; k < hi; k += TPR) s += ld_stream_f64(dA + k) * x[ld_stream_s32(dJ + k)];
        if (oI) {
            int olo = oI[row], ohi = oI[row + 1];
            for (int k = olo + lane; k < ohi; k += TPR) s += ld_stream_f64(oA + k) * xext[ld_stream_s32(oJ + k)];
        }
#pragma unroll
        for (int w = TPR / 2; w > 0; w >>= 1) s += __shfl_down_sync(0xffffffffu, s, w, TPR);
        if (lane == 0) {
            double r = alpha * s;
            if (beta != 0.0) r += beta * yin[row];
            yout[row] = r;
        }
    }
}

// Streaming SpMV: CTA b owns the consecutive rows [rb[b], rb[b+1]) (<= PE_STREAM_CAP non-zeros).
// Phase 1: the CTA streams its contiguous run of (col,val) pairs with fully coalesced,
// independent loads (8 in flight per thread), gathers x and parks the products in shared
// memory.  Phase 2: one thread per row sums its products and applies the alpha/beta epilogue.
#define SU 8
__global__ void __launch_bounds__(256)
k_spmv_stream(const int *__restrict__ rb, const int *__restrict__ I, const int *__restrict__ J,
              const double *__restrict__ A, const double *x, double alpha, double beta,
              const double *yin, double *yout)
{
    __shared__ double prod[PE_STREAM_CAP];
    pdl_trigger();
    const int tid = threadIdx.x;
    const int r0 = rb[blockIdx.x], r1 = rb[blockIdx.x + 1];
    const int k0 = I[r0], k1 = I[r1];
    if ((k0 ^ k1) == 0x5bd1e995 && k1 == -7) pdl_trigger();      // pins the row-block extent ahead of the wait
    pdl_wait();
    for (int base = k0; base < k1; base += 256 * SU)
    {
        int c[SU]; double a[SU];
#pragma unroll
        for (int u = 0; u < SU; ++u)
        {
            const int k = base + u * 256 + tid;
            c[u] = k < k1 ? ld_stream_s32(J + k) : -1;
            a[u] = k < k1 ? ld_stream_f64(A + k) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < SU; ++u) if (c[u] >= 0) a[u] *= x[c[u]];
#pragma unroll
        for (int u = 0; u < SU; ++u) { const int k = base + u * 256 + tid; if (k < k1) prod[k - k0] = a[u]; }
    }
    __syncthreads();
    for (int r = r0 + tid; r < r1; r += 256)
    {
        const int lo = I[r] - k0, hi = I[r + 1] - k0;
        double s = 0.0;
        for (int q = lo; q < hi; ++q) s += prod[q];
        double v = alpha * s;
        if (beta != 0.0) v += beta * yin[r];
        yout[r] = v;
    }
}

int pe_launch_spmv(pe_ctx *ctx, const DevCSR &diag, const DevCSR *offd, int tpr,
                   double alpha, const double *x, const double *xext,
                   double beta, const double *yin, double *yout)
{
    int n = diag.nrows;
    if (n == 0) return 0;
    const int *oI = nullptr, *oJ = nullptr;
    const double *oA = nullptr;
    if (offd && offd->nnz > 0) { oI = offd->I; oJ = offd->J; oA = offd->A; }
    if (!oI && diag.sell_state == 0) PE_TRY(pe_sell_for_spmv(ctx, const_cast<DevCSR &>(diag)));
    if (!oI && diag.sell)
    {
        pe_variant_add(PE_VARIANT_SPMV_SELL, n);
        if (diag.sell->S) pe_variant_add(PE_VARIANT_SPMV_SELL_SIGNS, n);
        const double per_nnz = diag.sell->S ? 5.0 : 12.0;     // sign-encoded values: 1 B instead of 8
        PE_TRY(pe_prof_begin(ctx, 0, per_nnz * (double)diag.nnz + 4.0 * (n + 1) + 8.0 * diag.ncols + 8.0 * n + (beta != 0.0 ? 8.0 * n : 0.0)));
        PE_TRY(pe_launch_sell_spmv(ctx, *diag.sell, alpha, x, beta, yin, yout));
        PE_TRY(pe_prof_end(ctx));
        return 0;
    }
    if (ctx->rec && !oI)
    {
        // persistent program: CSR-vector op (the CTA-tiled streaming kernel has no op equivalent)
        pe_variant_add(PE_VARIANT_SPMV_VECTOR, n);
        PeOp o = pe_op(PE_OP_CSR_SPMV); o.i0 = n; o.i1 = pe_choose_tpr(diag.nnz, n); o.a = alpha; o.b = beta;
        o.p[0] = diag.I; o.p[1] = diag.J; o.p[2] = diag.A; o.p[3] = x; o.p[4] = yin; o.p[5] = yout;
        pe_rec_push(ctx, o, 12.0 * (double)diag.nnz + 4.0 * (n + 1) + 8.0 * diag.ncols + 8.0 * n + (beta != 0.0 ? 8.0 * n : 0.0));
        return 0;
    }
    if (!oI && diag.nrb == 0 && diag.nnz > 0) PE_TRY(pe_build_row_blocks(ctx, const_cast<DevCSR &>(diag), nullptr));
    if (!oI && diag.nrb > 0)
    {
        pe_variant_add(PE_VARIANT_SPMV_STREAM, n);
        PE_TRY(pe_prof_begin(ctx, 0, 12.0 * (double)diag.nnz + 4.0 * (n + 1) + 8.0 * diag.ncols + 8.0 * n + (beta != 0.0 ? 8.0 * n : 0.0)));
        PE_CUDA(pe_launch_k(ctx, k_spmv_stream, diag.nrb, 256, diag.rb, diag.I, diag.J, diag.A, x, alpha, beta, yin, yout));
        PE_LAUNCHED(ctx);
        PE_TRY(pe_prof_end(ctx));
        return 0;
    }
    pe_variant_add(PE_VARIANT_SPMV_VECTOR, n);
    int64_t threads = (int64_t)n * tpr;
    int64_t cap = (int64_t)PE_SM_COUNT * 8 * 8;     // 8 CTAs of 256 threads per SM, x8 waves
    int grid = (int)std::min<int64_t>((threads + 255) / 256, cap);
    if (grid < 1) grid = 1;
#define LAUNCH(T) PE_CUDA(pe_launch_k(ctx, k_spmv<T>, grid, 256, n, diag.I, diag.J, diag.A, oI, oJ, oA, x, xext, alpha, beta, yin, yout))
    const double nnz_all = (double)diag.nnz + (oI ? (double)offd->nnz : 0.0);
    PE_TRY(pe_prof_begin(ctx, 0, 12.0 * nnz_all + 4.0 * (n + 1) + 8.0 * diag.ncols + 8.0 * n + (beta != 0.0 ? 8.0 * n : 0.0)));
    switch (tpr) {
    case 1: LAUNCH(1); break;
    case 2: LAUNCH(2); break;
    case 4: LAUNCH(4); break;
    case 8: LAUNCH(8); break;
    case 16: LAUNCH(16); break;
    default: LAUNCH(32); break;
    }
#undef LAUNCH
    PE_LAUNCHED(ctx);
    PE_TRY(pe_prof_end(ctx));
    return 0;
}

extern "C" int pe_spmv(pe_ctx *ctx, double alpha, pe_mat *A, const pe_vec *x, double beta, pe_vec *y)
{
    PE_CHECK(x->n == A->diag.ncols && y->n == A->diag.nrows, "pe_spmv: size mismatch");
    PE_CHECK(x->d != y->d, "pe_spmv: x and y must not alias");
    if (A->offd.nnz > 0) {
        // diag pass overlaps the exchange; offd pass accumulates (beta = 1) once the halo landed
        PE_TRY(pe_halo_exchange(A, x->d));
        PE_TRY(pe_launch_spmv(ctx, A->diag, nullptr, A->tpr, alpha, x->d, nullptr, beta, y->d, y->d));
        PE_TRY(pe_halo_wait(A));
        int otpr = pe_choose_tpr(A->offd.nnz, A->offd.nrows);
        PE_TRY(pe_launch_spmv(ctx, A->offd, nullptr, otpr, alpha, A->x_ext_d, nullptr, 1.0, y->d, y->d));
        return 0;
    }
    if (ctx->nranks > 1) { PE_TRY(pe_halo_exchange(A, x->d)); PE_TRY(pe_halo_wait(A)); }  // others may need our values
    return pe_launch_spmv(ctx, A->diag, nullptr, A->tpr, alpha, x->d, nullptr, beta, y->d, y->d);
}

extern "C" int pe_residual(pe_ctx *ctx, pe_mat *A, const pe_vec *x, const pe_vec *b, pe_vec *r)
{
    PE_CHECK(x->n == A->diag.ncols && b->n == A->diag.nrows && r->n == b->n, "pe_residual: size mismatch");
    if (A->offd.nnz > 0) {
        PE_TRY(pe_halo_exchange(A, x->d));
        PE_TRY(pe_launch_spmv(ctx, A->diag, nullptr, A->tpr, -1.0, x->d, nullptr, 1.0, b->d, r->d));
        PE_TRY(pe_halo_wait(A));
        int otpr = pe_choose_tpr(A->offd.nnz, A->offd.nrows);
        return pe_launch_spmv(ctx, A->offd, nullptr, otpr, -1.0, A->x_ext_d, nullptr, 1.0, r->d, r->d);
    }
    if (ctx->nranks > 1) { PE_TRY(pe_halo_exchange(A, x->d)); PE_TRY(pe_halo_wait(A)); }
    return pe_launch_spmv(ctx, A->diag, nullptr, A->tpr, -1.0, x->d, nullptr, 1.0, b->d, r->d);
}

// ---------------------------------------------------------------------------
// transpose: stable radix sort of (col -> entry index); rows of A^T come out with
// ascending column (= original row) order, identical to a counting-sort transpose.
// ---------------------------------------------------------------------------
__global__ void k_iota(int64_t n, int *p)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) p[i] = (int)i;
}
__global__ void k_expand_rows(int nrows, const int *__restrict__ I, int *__restrict__ rowof)
{
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < nrows) for (int k = I[r]; k < I[r + 1]; ++k) rowof[k] = r;
}
__global__ void k_count_cols(int64_t nnz, const int *__restrict__ J, int *cnt)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < nnz) atomicAdd(cnt + J[i] + 1, 1);
}
__global__ void k_gather_t(int64_t nnz, const int *__restrict__ perm, const int *__restrict__ rowof,
                           const double *__restrict__ A, int *TJ, double *TA)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < nnz) { int p = perm[i]; TJ[i] = rowof[p]; TA[i] = A[p]; }
}

int pe_devcsr_transpose(pe_ctx *ctx, const DevCSR &A, DevCSR &T)
{
    cudaStream_t s = ctx->stream;
    PE_TRY(devcsr_alloc(T, A.ncols, A.nrows, A.nnz));
    PE_CUDA(cudaMemsetAsync(T.I, 0, sizeof(int) * (size_t)(A.ncols + 1), s));
    if (A.nnz == 0) return 0;
    int64_t nnz = A.nnz;
    int *rowof, *idx, *keys_out, *idx_out;
    PE_CUDA(cudaMalloc(&rowof, sizeof(int) * nnz));
    PE_CUDA(cudaMalloc(&idx, sizeof(int) * nnz));
    PE_CUDA(cudaMalloc(&keys_out, sizeof(int) * nnz));
    PE_CUDA(cudaMalloc(&idx_out, sizeof(int) * nnz));
    k_expand_rows<<<pe_grid_for(A.nrows, 256), 256, 0, s>>>(A.nrows, A.I, rowof); PE_LAUNCHED(ctx);
    k_iota<<<pe_grid_for(nnz, 256), 256, 0, s>>>(nnz, idx); PE_LAUNCHED(ctx);
    k_count_cols<<<pe_grid_for(nnz, 256), 256, 0, s>>>(nnz, A.J, T.I); PE_LAUNCHED(ctx);
    void *tmp = nullptr; size_t tmp_bytes = 0, b2 = 0;
    int end_bit = 1; while ((1ll << end_bit) < A.ncols && end_bit < 31) ++end_bit;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, A.J, keys_out, idx, idx_out, (int)nnz, 0, end_bit, s);
    cub::DeviceScan::InclusiveSum(nullptr, b2, T.I, T.I, A.ncols + 1, s);
    if (b2 > tmp_bytes) tmp_bytes = b2;
    PE_CUDA(cudaMalloc(&tmp, tmp_bytes));
    PE_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, A.J, keys_out, idx, idx_out, (int)nnz, 0, end_bit, s));
    PE_CUDA(cub::DeviceScan::InclusiveSum(tmp, tmp_bytes, T.I, T.I, A.ncols + 1, s));
    ctx->launches += 2;
    k_gather_t<<<pe_grid_for(nnz, 256), 256, 0, s>>>(nnz, idx_out, rowof, A.A, T.J, T.A); PE_LAUNCHED(ctx);
    PE_CUDA(cudaStreamSynchronize(s));
    cudaFree(tmp); cudaFree(rowof); cudaFree(idx); cudaFree(keys_out); cudaFree(idx_out);
    return 0;
}

extern "C" int pe_mat_transpose(pe_ctx *ctx, const pe_mat *A, pe_mat **out)
{
    if (A->distributed) return pe_transpose_distributed(ctx, A, out);
    DevCSR T;
    PE_TRY(pe_devcsr_transpose(ctx, A->diag, T));
    PE_TRY(pe_mat_wrap_local(ctx, T, out));
    (*out)->global_num_rows = A->global_num_cols;
    (*out)->global_num_cols = A->global_num_rows;
    return 0;
}

extern "C" int pe_spmv_t(pe_ctx *ctx, double alpha, pe_mat *A, const pe_vec *x, double beta, pe_vec *y)
{
    PE_CHECK(x->n == A->diag.nrows && y->n == A->diag.ncols, "pe_spmv_t: size mismatch");
    if (A->distributed) return pe_spmv_t_distributed(ctx, alpha, A, x, beta, y);
    if (!A->T) PE_TRY(pe_mat_transpose(ctx, A, &A->T));
    return pe_spmv(ctx, alpha, A->T, x, beta, y);
}

// ---------------------------------------------------------------------------
__global__ void k_get_diag(int n, const int *__restrict__ I, const int *__restrict__ J,
                           const double *__restrict__ A, double *d)
{
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    double v = 0.0;
    for (int k = I[r]; k < I[r + 1]; ++k) if (J[k] == r) { v = A[k]; break; }
    d[r] = v;
}
extern "C" int pe_mat_get_diag(const pe_mat *A, pe_vec *d)
{
    PE_CHECK(d->n == A->diag.nrows, "size mismatch");
    k_get_diag<<<pe_grid_for(A->diag.nrows, 256), 256, 0, A->ctx->stream>>>(A->diag.nrows, A->diag.I, A->diag.J, A->diag.A, d->d);
    PE_LAUNCHED(A->ctx);
    return 0;
}
__global__ void k_scale_rows(int n, const int *__restrict__ I, double *A, const double *__restrict__ d, int invert)
{
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    double s = invert ? 1.0 / d[r] : d[r];
    for (int k = I[r]; k < I[r + 1]; ++k) A[k] *= s;
}
extern "C" int pe_mat_scale_rows(pe_mat *A, const pe_vec *d, int invert)
{
    PE_CHECK(d->n == A->diag.nrows, "size mismatch");
    int n = A->diag.nrows;
    k_scale_rows<<<pe_grid_for(n, 256), 256, 0, A->ctx->stream>>>(n, A->diag.I, A->diag.A, d->d, invert);
    PE_LAUNCHED(A->ctx);
    if (A->offd.nnz > 0) {
        k_scale_rows<<<pe_grid_for(n, 256), 256, 0, A->ctx->stream>>>(n, A->offd.I, A->offd.A, d->d, invert);
        PE_LAUNCHED(A->ctx);
    }
    pe_mat_values_changed(A);
    return 0;
}

__global__ void k_scale_all(int64_t nnz, double *A, double a)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < nnz) A[i] *= a;
}
extern "C" int pe_mat_scale(pe_mat *A, double a)
{
    for (DevCSR *m : {&A->diag, &A->offd})
        if (m->nnz > 0)
        {
            k_scale_all<<<pe_grid_for(m->nnz, 256), 256, 0, A->ctx->stream>>>(m->nnz, m->A, a);
            PE_LAUNCHED(A->ctx);
        }
    pe_mat_values_changed(A);
    return 0;
}
__global__ void k_abs_row_sums(int n, const int *__restrict__ dI, const double *__restrict__ dA, const int *__restrict__ oI,
                               const double *__restrict__ oA, double *d)
{
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    double s = 0.0;
    for (int k = dI[r]; k < dI[r + 1]; ++k) s += fabs(dA[k]);
    if (oI) for (int k = oI[r]; k < oI[r + 1]; ++k) s += fabs(oA[k]);
    d[r] = s;
}
extern "C" int pe_mat_abs_row_sums(const pe_mat *A, pe_vec *d)
{
    PE_CHECK(d->n == A->diag.nrows, "size mismatch");
    const int n = A->diag.nrows;
    if (n == 0) return 0;
    k_abs_row_sums<<<pe_grid_for(n, 256), 256, 0, A->ctx->stream>>>(n, A->diag.I, A->diag.A, A->offd.nnz > 0 ? A->offd.I : nullptr, A->offd.A, d->d);
    PE_LAUNCHED(A->ctx);
    return 0;
}
