// pe_util.cu -- the ParCSR utilities of src/hypreExtension (SURVEY 2.2) on device matrices:
// delete-zeros, sign transformation, identity / diagonal factories, matrix norms, compare, R^T diag(d) P.
#include "pe_core.cuh"
#include <cub/cub.cuh>
#include <algorithm>
#include <cmath>

// ---- hypre_CSRMatrixDeleteZeros (hypre, called by hypre_ParCSRMatrixDeleteZeros, deleteZeros.c:16-47): entries with
// |a| <= tol are deleted, i.e. |a| > tol is kept (tol = 0 removes the stored zeros) ---------------------------------
__global__ void k_count_keep(int n, const int *__restrict__ I, const double *__restrict__ A, double tol, int *len)
{
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    int c = 0;
    for (int k = I[r]; k < I[r + 1]; ++k) c += fabs(A[k]) > tol;
    len[r] = c;
}
__global__ void k_fill_keep(int n, const int *__restrict__ I, const int *__restrict__ J, const double *__restrict__ A, double tol,
                            const int *__restrict__ OI, int *OJ, double *OA)
{
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    int p = OI[r];
    for (int k = I[r]; k < I[r + 1]; ++k) if (fabs(A[k]) > tol) { OJ[p] = J[k]; OA[p] = A[k]; ++p; }
}
static int compress_block(pe_ctx *ctx, DevCSR &m, double tol)
{
    cudaStream_t st = ctx->stream;
    const int n = m.nrows;
    if (m.nnz == 0) return 0;
    int *len, *OI;
    PE_CUDA(cudaMalloc(&len, sizeof(int) * (size_t)(n + 1)));
    PE_CUDA(cudaMalloc(&OI, sizeof(int) * (size_t)(n + 1)));
    PE_CUDA(cudaMemsetAsync(len, 0, sizeof(int) * (size_t)(n + 1), st));
    k_count_keep<<<pe_grid_for(n, 256), 256, 0, st>>>(n, m.I, m.A, tol, len); PE_LAUNCHED(ctx);
    void *tmp = nullptr; size_t tb = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tb, len, OI, n + 1, st);
    PE_CUDA(cudaMalloc(&tmp, tb));
    PE_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tb, len, OI, n + 1, st));
    ctx->launches++;
    int nnz = 0;
    PE_CUDA(cudaMemcpyAsync(&nnz, OI + n, sizeof(int), cudaMemcpyDeviceToHost, st));
    PE_CUDA(cudaStreamSynchronize(st));
    cudaFree(tmp); cudaFree(len);
    int *OJ; double *OA;
    PE_CUDA(cudaMalloc(&OJ, sizeof(int) * (size_t)(nnz > 0 ? nnz : 1)));
    PE_CUDA(cudaMalloc(&OA, sizeof(double) * (size_t)(nnz > 0 ? nnz : 1)));
    k_fill_keep<<<pe_grid_for(n, 256), 256, 0, st>>>(n, m.I, m.J, m.A, tol, OI, OJ, OA); PE_LAUNCHED(ctx);
    PE_CUDA(cudaStreamSynchronize(st));
    cudaFree(m.I); cudaFree(m.J); cudaFree(m.A);
    if (m.rb) { cudaFree(m.rb); m.rb = nullptr; m.nrb = 0; }
    m.I = OI; m.J = OJ; m.A = OA; m.nnz = nnz;
    return 0;
}
/* hypre_ParCSRMatrixDeleteZeros (deleteZeros.c:16-47), in place.  The ghost-column map and comm package
 * are kept (columns that lost all entries stay as unused ghosts); hypre rebuilds them. */
extern "C" int pe_mat_delete_zeros(pe_ctx *ctx, pe_mat *A, double tol)
{
    PE_CHECK(ctx && A, "bad arguments");
    PE_TRY(compress_block(ctx, A->diag, tol));
    PE_TRY(compress_block(ctx, A->offd, tol));
    pe_mat_values_changed(A);
    A->tpr = pe_choose_tpr(A->diag.nnz + A->offd.nnz, A->diag.nrows);
    return 0;
}

// ---- hypre_ParCSRDataTransformationSign (hypre_ParCSRDataTransformationSign.c:16-33) -----------------
__global__ void k_sign(int64_t nnz, double *A, double tol)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < nnz) { const double a = A[i]; A[i] = a > tol ? 1.0 : (a < -tol ? -1.0 : 0.0); }
}
extern "C" int pe_mat_sign(pe_ctx *ctx, pe_mat *A, double tol)
{
    for (DevCSR *m : {&A->diag, &A->offd})
        if (m->nnz > 0) { k_sign<<<pe_grid_for(m->nnz, 256), 256, 0, ctx->stream>>>(m->nnz, m->A, tol); PE_LAUNCHED(ctx); }
    pe_mat_values_changed(A);
    return 0;
}

// ---- hypre_IdentityCSRMatrix / hypre_DiagonalCSRMatrix (hypre_CSRFactory.c:16-250), rank-local ------
__global__ void k_diag_fill(int n, const double *__restrict__ d, int *I, int *J, double *A)
{
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r > n) return;
    I[r] = r;
    if (r < n) { J[r] = r; A[r] = d ? d[r] : 1.0; }
}
extern "C" int pe_mat_diagonal(pe_ctx *ctx, int32_t n, const pe_vec *d_or_null, pe_mat **out)
{
    PE_CHECK(ctx && out && n >= 0 && (!d_or_null || d_or_null->n == n), "bad arguments");
    DevCSR m;
    PE_TRY(devcsr_alloc(m, n, n, n));
    k_diag_fill<<<pe_grid_for(n + 1, 256), 256, 0, ctx->stream>>>(n, d_or_null ? d_or_null->d : nullptr, m.I, m.J, m.A);
    PE_LAUNCHED(ctx);
    return pe_mat_wrap_local(ctx, m, out);
}

// ---- norms (hypre_ParCSRMatrixNorms.c:18-195): out = {l1, linf, max, frobenius} ---------------------
__global__ void k_row_stats(int n, const int *__restrict__ dI, const double *__restrict__ dA, const int *__restrict__ oI,
                            const double *__restrict__ oA, double *rowsum, double *rowmax, double *rowsq)
{
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    double s = 0, m = 0, q = 0;
    for (int k = dI[r]; k < dI[r + 1]; ++k) { const double a = fabs(dA[k]); s += a; m = fmax(m, a); q += a * a; }
    if (oI) for (int k = oI[r]; k < oI[r + 1]; ++k) { const double a = fabs(oA[k]); s += a; m = fmax(m, a); q += a * a; }
    rowsum[r] = s; rowmax[r] = m; rowsq[r] = q;
}
__global__ void k_abs_vals(int64_t nnz, const double *__restrict__ in, double *out)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < nnz) out[i] = fabs(in[i]);
}
int pe_allreduce(pe_ctx *c, double *d, int count, int op);   // pe_core.cu: op 0 sum, 2 max
static int reduce_dev(pe_ctx *ctx, const double *v, int n, bool do_max, double *out_h)
{
    double *out_d = ctx->scalar_d + 5;
    void *tmp = nullptr; size_t tb = 0;
    if (n == 0) { *out_h = 0.0; }
    else
    {
        if (do_max) cub::DeviceReduce::Max(nullptr, tb, v, out_d, n, ctx->stream); else cub::DeviceReduce::Sum(nullptr, tb, v, out_d, n, ctx->stream);
        PE_CUDA(cudaMalloc(&tmp, tb));
        if (do_max) PE_CUDA(cub::DeviceReduce::Max(tmp, tb, v, out_d, n, ctx->stream)); else PE_CUDA(cub::DeviceReduce::Sum(tmp, tb, v, out_d, n, ctx->stream));
        ctx->launches++;
    }
    if (n == 0) PE_CUDA(cudaMemsetAsync(out_d, 0, sizeof(double), ctx->stream));
    PE_TRY(pe_allreduce(ctx, out_d, 1, do_max ? 2 : 0));
    PE_CUDA(cudaMemcpyAsync(out_h, out_d, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    PE_CUDA(cudaStreamSynchronize(ctx->stream));
    if (tmp) cudaFree(tmp);
    return 0;
}
extern "C" int pe_mat_norms(pe_ctx *ctx, pe_mat *A, double *out4)
{
    PE_CHECK(ctx && A && out4, "bad arguments");
    const int n = A->diag.nrows, nc = A->diag.ncols;
    double *buf;
    PE_CUDA(cudaMalloc(&buf, sizeof(double) * (size_t)(3 * (n > 0 ? n : 1))));
    if (n > 0)
    {
        k_row_stats<<<pe_grid_for(n, 256), 256, 0, ctx->stream>>>(n, A->diag.I, A->diag.A, A->offd.nnz > 0 ? A->offd.I : nullptr, A->offd.A,
                                                                 buf, buf + n, buf + 2 * n);
        PE_LAUNCHED(ctx);
    }
    PE_TRY(reduce_dev(ctx, buf, n, true, out4 + 1));            // linf: max abs row sum
    PE_TRY(reduce_dev(ctx, buf + n, n, true, out4 + 2));        // max norm
    double fro2 = 0.0;
    PE_TRY(reduce_dev(ctx, buf + 2 * n, n, false, &fro2));
    out4[3] = std::sqrt(fro2);
    cudaFree(buf);
    // l1: max abs column sum = max(|A|^T 1) through the (distributed) transpose product; the values are
    // replaced by their moduli for the duration of the product and restored afterwards
    double *save_d = nullptr, *save_o = nullptr;
    for (int blk = 0; blk < 2; ++blk)
    {
        DevCSR &m = blk == 0 ? A->diag : A->offd;
        double *&sv = blk == 0 ? save_d : save_o;
        if (m.nnz == 0) continue;
        PE_CUDA(cudaMalloc(&sv, sizeof(double) * (size_t)m.nnz));
        PE_CUDA(cudaMemcpyAsync(sv, m.A, sizeof(double) * (size_t)m.nnz, cudaMemcpyDeviceToDevice, ctx->stream));
        k_abs_vals<<<pe_grid_for(m.nnz, 256), 256, 0, ctx->stream>>>(m.nnz, sv, m.A); PE_LAUNCHED(ctx);
    }
    pe_mat_values_changed(A);
    pe_vec *ones = nullptr, *cs = nullptr;
    PE_TRY(pe_vec_create(ctx, n, &ones)); PE_TRY(pe_vec_create(ctx, nc, &cs));
    PE_TRY(pe_vec_fill(ones, 1.0));
    int rc = pe_spmv_t(ctx, 1.0, A, ones, 0.0, cs);
    if (!rc) rc = reduce_dev(ctx, cs->d, nc, true, out4 + 0);
    for (int blk = 0; blk < 2; ++blk)
    {
        DevCSR &m = blk == 0 ? A->diag : A->offd;
        double *sv = blk == 0 ? save_d : save_o;
        if (!sv) continue;
        cudaMemcpyAsync(m.A, sv, sizeof(double) * (size_t)m.nnz, cudaMemcpyDeviceToDevice, ctx->stream);
        cudaStreamSynchronize(ctx->stream);
        cudaFree(sv);
    }
    pe_mat_values_changed(A);
    pe_vec_free(ones); pe_vec_free(cs);
    return rc;
}

// ---- hypre_ParCSRMatrixCompare (hypre_ParCSRMatrixCompare.c:125-195): bit flags
//  1 global rows, 2 global cols, 4 first row, 8 last row, 16 first col, 32 last col, 64 ||A - B||_max > tol
__global__ void k_maxdiff_rows(int n, const int *__restrict__ AI, const int *__restrict__ AJ, const double *__restrict__ AA,
                               const int *__restrict__ BI, const int *__restrict__ BJ, const double *__restrict__ BA, double *rowmax)
{
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    double m = 0.0;
    // entries of A minus the matching entry of B, then the entries of B that A lacks
    for (int ka = AI[r]; ka < AI[r + 1]; ++ka)
    {
        double b = 0.0;
        for (int kb = BI[r]; kb < BI[r + 1]; ++kb) if (BJ[kb] == AJ[ka]) b += BA[kb];
        m = fmax(m, fabs(AA[ka] - b));
    }
    for (int kb = BI[r]; kb < BI[r + 1]; ++kb)
    {
        bool found = false;
        for (int ka = AI[r]; ka < AI[r + 1]; ++ka) if (AJ[ka] == BJ[kb]) { found = true; break; }
        if (!found) m = fmax(m, fabs(BA[kb]));
    }
    rowmax[r] = m;
}
extern "C" int pe_mat_compare(pe_ctx *ctx, const pe_mat *A, const pe_mat *B, double tol, int32_t *flags)
{
    PE_CHECK(ctx && A && B && flags, "bad arguments");
    int cmp = 0;
    if (A->global_num_rows != B->global_num_rows) cmp |= 1;
    if (A->global_num_cols != B->global_num_cols) cmp |= 2;
    if (A->first_row_index != B->first_row_index) cmp |= 4;
    if (A->first_row_index + A->diag.nrows != B->first_row_index + B->diag.nrows) cmp |= 8;
    if (A->first_col_diag != B->first_col_diag) cmp |= 16;
    if (A->first_col_diag + A->diag.ncols != B->first_col_diag + B->diag.ncols) cmp |= 32;
    double diff = 0.0;
    if (A->diag.nrows == B->diag.nrows)
    {
        const int n = A->diag.nrows;
        double *rm;
        PE_CUDA(cudaMalloc(&rm, sizeof(double) * (size_t)(n > 0 ? n : 1)));
        double d1 = 0.0, d2 = 0.0;
        if (n > 0) { k_maxdiff_rows<<<pe_grid_for(n, 256), 256, 0, ctx->stream>>>(n, A->diag.I, A->diag.J, A->diag.A, B->diag.I, B->diag.J, B->diag.A, rm); PE_LAUNCHED(ctx); }
        PE_TRY(reduce_dev(ctx, rm, n, true, &d1));
        if (A->col_map_offd == B->col_map_offd)
        {
            if (n > 0 && (A->offd.nnz > 0 || B->offd.nnz > 0))
            { k_maxdiff_rows<<<pe_grid_for(n, 256), 256, 0, ctx->stream>>>(n, A->offd.I, A->offd.J, A->offd.A, B->offd.I, B->offd.J, B->offd.A, rm); PE_LAUNCHED(ctx); }
            else if (n > 0) PE_CUDA(cudaMemsetAsync(rm, 0, sizeof(double) * (size_t)n, ctx->stream));
            PE_TRY(reduce_dev(ctx, rm, n, true, &d2));
        }
        else d2 = INFINITY;    // different ghost numbering: not comparable block-wise
        cudaFree(rm);
        diff = std::fmax(d1, d2);
    }
    else diff = INFINITY;
    if (diff > tol) cmp |= 64;
    *flags = cmp;
    return 0;
}

// ---- hypre_RDP (par_Tmatmul.c:17-39): R^T diag(d) P, rank-local -------------------------------------
extern "C" int pe_rdp(pe_ctx *ctx, const pe_mat *R, const pe_vec *d, const pe_mat *P, pe_mat **out)
{
    PE_CHECK(ctx && R && d && P && out, "bad arguments");
    PE_CHECK(!R->distributed && !P->distributed, "pe_rdp: rank-local matrices only");
    PE_CHECK(R->diag.nrows == P->diag.nrows && d->n == P->diag.nrows, "pe_rdp: size mismatch");
    pe_mat *DP = nullptr;
    PE_TRY(pe_spadd(ctx, 1.0, P, 0.0, P, &DP));          // copy of P
    int rc = pe_mat_scale_rows(DP, d, 0);
    DevCSR Rt, C;
    if (!rc) rc = pe_devcsr_transpose(ctx, R->diag, Rt);
    if (!rc) rc = pe_devcsr_spgemm(ctx, Rt, DP->diag, C);
    devcsr_free(Rt);
    pe_mat_free(DP);
    if (rc) return rc;
    return pe_mat_wrap_local(ctx, C, out);
}

// ---- same sparsity pattern: sizes on the host, then row pointers and column indices in one pass whose threads raise
// a shared flag (every writer stores 1, so the stores need no ordering); one int is downloaded
__global__ void k_pattern_differs(int64_t n, int nrows, int64_t nnz, const int *__restrict__ AI, const int *__restrict__ AJ,
                                  const int *__restrict__ BI, const int *__restrict__ BJ, int *flag)
{
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    if ((k < nnz && AJ[k] != BJ[k]) || (k <= nrows && AI[k] != BI[k])) *flag = 1;
}
extern "C" int pe_mat_same_pattern(pe_ctx *ctx, const pe_mat *A, const pe_mat *B, int32_t *same)
{
    PE_CHECK(ctx && A && B && same, "bad arguments");
    *same = 0;
    if (A == B) { *same = 1; return 0; }
    PE_CHECK(!A->distributed && !B->distributed && A->offd.nnz == 0 && B->offd.nnz == 0,
             "pe_mat_same_pattern: single-rank matrices only");
    if (A->diag.nrows != B->diag.nrows || A->diag.ncols != B->diag.ncols || A->diag.nnz != B->diag.nnz) return 0;
    int *flag = reinterpret_cast<int *>(ctx->scalar_d + 4);
    PE_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), ctx->stream));
    const int64_t n = std::max<int64_t>(A->diag.nnz, (int64_t)A->diag.nrows + 1);
    k_pattern_differs<<<pe_grid_for(n, 256), 256, 0, ctx->stream>>>(n, A->diag.nrows, A->diag.nnz, A->diag.I, A->diag.J,
                                                                     B->diag.I, B->diag.J, flag);
    PE_LAUNCHED(ctx);
    int h = 0;
    PE_CUDA(cudaMemcpyAsync(&h, flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    PE_CUDA(cudaStreamSynchronize(ctx->stream));
    *same = h == 0;
    return 0;
}
