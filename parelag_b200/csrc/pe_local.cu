// pe_local.cu -- K11/K12/K13: the per-agglomerate dense work of DeRhamSequence::Coarsen
// as batched one-agglomerate-per-CTA kernels; every local matrix lives in shared memory.
//
//   pe_batched_traces      ComputeCoarseTracesWithTargets hot loop
//                          (src/amge/DeRhamSequence.cpp:1818-1926): Deflate, weighted SVD,
//                          rank truncation, p_loc = [pv | sqrt(pv.M.pv) U], coarse trace mass,
//                          dof functional.
//   pe_batched_extension   hFacetExtension hot loop (:2364-2556) with FacetSaddlePoint
//                          [M B^T 0; B 0 T^T; 0 T 0]  (ParELAG_SaddlePointSolver.cpp:70-130) and
//                          hRidgePeakExtension hot loop (:2779-3027) with RidgePeakSaddlePoint
//                          [M B^T; B -C] (:150-189): local assembly of M, W, D blocks from the
//                          entity matrices, all right-hand sides at once, pivoted LU, target
//                          residual SVD, CochainProjector::CreateDofFunctional
//                          (src/amge/CochainProjector.cpp:53-137) and CoarsenMassMatrixPart.
//
// The reference factors with dsytrf (Bunch-Kaufman) and uses dgesvd; here the small
// systems (order 7..60) are solved by Gaussian elimination with partial pivoting and the
// thin SVDs (<= 8 columns) by one-sided Jacobi, both in FP64 FMA -- far below DMMA tile
// sizes, so no tensor cores (SURVEY K11/K12).  SVD sign convention: largest-magnitude
// entry of every retained singular vector is positive; near-ties (relative 1e-6) go to the
// smallest index (warp_sign_pivot).
#include "pe_core.cuh"
#include <chrono>
#include <map>
#include "../../include/parelag_b200_local.h"
#include <algorithm>
#include <cmath>
#include <cstring>

#define LT 128   // threads per CTA in the extension kernel

// ---------------------------------------------------------------------------
// CTA-cooperative dense helpers (row-major, data in shared memory)
// ---------------------------------------------------------------------------
// Solve A X = R in place (A n x n, lda; R n x nrhs, ldr) by Gaussian elimination with
// partial pivoting (ties -> smallest row index).  Returns 0, or k+1 if pivot k is zero.
__device__ int cta_lu_solve(double *A, int n, int lda, double *R, int nrhs, int ldr, int *s_piv, int tid, int nt)
{
    __shared__ int s_info;
    if (tid == 0) s_info = 0;
    __syncthreads();
    for (int k = 0; k < n; ++k)
    {
        if (tid < 32)
        {
            double best = -1.0; int bi = k;
            for (int i = k + tid; i < n; i += 32) { double v = fabs(A[i * lda + k]); if (v > best) { best = v; bi = i; } }
            for (int o = 16; o > 0; o >>= 1)
            {
                double ob = __shfl_down_sync(0xffffffffu, best, o);
                int oi = __shfl_down_sync(0xffffffffu, bi, o);
                if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
            }
            if (tid == 0) { *s_piv = bi; if (!(best > 0.0) && s_info == 0) s_info = k + 1; }
        }
        __syncthreads();
        const int p = *s_piv;
        if (s_info) return s_info;
        if (p != k)
        {
            for (int j = tid; j < n; j += nt) { double t = A[k * lda + j]; A[k * lda + j] = A[p * lda + j]; A[p * lda + j] = t; }
            for (int j = tid; j < nrhs; j += nt) { double t = R[k * ldr + j]; R[k * ldr + j] = R[p * ldr + j]; R[p * ldr + j] = t; }
            __syncthreads();
        }
        const double inv = 1.0 / A[k * lda + k];
        for (int i = k + 1 + tid; i < n; i += nt) A[i * lda + k] *= inv;     // multipliers
        __syncthreads();
        const int rem = n - k - 1, wtot = rem + nrhs;
        for (int idx = tid; idx < rem * wtot; idx += nt)
        {
            const int i = k + 1 + idx / wtot, c = idx % wtot;
            const double l = A[i * lda + k];
            if (c < rem) A[i * lda + k + 1 + c] -= l * A[k * lda + k + 1 + c];
            else R[i * ldr + (c - rem)] -= l * R[k * ldr + (c - rem)];
        }
        __syncthreads();
    }
    for (int k = n - 1; k >= 0; --k)
    {
        const double inv = 1.0 / A[k * lda + k];
        for (int j = tid; j < nrhs; j += nt) R[k * ldr + j] *= inv;
        __syncthreads();
        for (int idx = tid; idx < k * nrhs; idx += nt)
        {
            const int i = idx / nrhs, j = idx % nrhs;
            R[i * ldr + j] -= A[i * lda + k] * R[k * ldr + j];
        }
        __syncthreads();
    }
    return 0;
}

// Index of the entry that fixes the sign of a singular vector: the FIRST entry (in index order)
// whose magnitude is within a relative 1e-6 of the largest one.  Identical to "largest-magnitude
// entry" whenever that entry is unique; on (near-)ties -- congruent fine entities inside an
// agglomerate give entries of equal magnitude up to rounding -- the choice no longer depends on the
// last bits, which LAPACK (oracle/amge.py:fix_sign follows the same rule) and the Jacobi SVD need not share.
#define PE_SIGN_TIE_REL 1e-6
__device__ __forceinline__ int warp_sign_pivot(const double *col, int m, int lane)
{
    const unsigned FULL = 0xffffffffu;
    double best = 0.0;
    for (int i = lane; i < m; i += 32) best = fmax(best, fabs(col[i]));
    for (int o = 16; o > 0; o >>= 1) best = fmax(best, __shfl_xor_sync(FULL, best, o));
    const double thr = best * (1.0 - PE_SIGN_TIE_REL);
    int bi = m;
    for (int i = lane; i < m; i += 32) if (fabs(col[i]) >= thr) { bi = i; break; }
    for (int o = 16; o > 0; o >>= 1) bi = min(bi, __shfl_xor_sync(FULL, bi, o));
    return bi < m ? bi : 0;
}

// One-sided (Hestenes) Jacobi SVD of X (m x k, COLUMN-major, ldx >= m) by warp 0.
// On exit: columns of X are the left singular vectors (sign-fixed) scaled to unit norm
// where sigma > 0, ordered by descending sigma; sv[0..min(m,k)) the singular values.
__device__ void warp_jacobi_svd(double *X, int m, int k, int ldx, double *sv, int lane)
{
    const unsigned FULL = 0xffffffffu;
    for (int sweep = 0; sweep < 40; ++sweep)
    {
        double off = 0.0;
        for (int p = 0; p < k - 1; ++p)
            for (int q = p + 1; q < k; ++q)
            {
                double a = 0, b = 0, g = 0;
                for (int i = lane; i < m; i += 32) { double xp = X[p * ldx + i], xq = X[q * ldx + i]; a += xp * xp; b += xq * xq; g += xp * xq; }
                for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(FULL, a, o); b += __shfl_xor_sync(FULL, b, o); g += __shfl_xor_sync(FULL, g, o); }
                if (a == 0.0 || b == 0.0) continue;
                const double r = fabs(g) / sqrt(a * b);
                if (r > off) off = r;
                if (r < 1e-16) continue;
                const double zeta = (b - a) / (2.0 * g);
                const double t = (zeta >= 0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
                const double c = 1.0 / sqrt(1.0 + t * t), s = c * t;
                for (int i = lane; i < m; i += 32)
                {
                    double xp = X[p * ldx + i], xq = X[q * ldx + i];
                    X[p * ldx + i] = c * xp - s * xq;
                    X[q * ldx + i] = s * xp + c * xq;
                }
                __syncwarp();
            }
        if (off < 1e-15) break;
    }
    // norms
    for (int p = 0; p < k; ++p)
    {
        double a = 0;
        for (int i = lane; i < m; i += 32) a += X[p * ldx + i] * X[p * ldx + i];
        for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(FULL, a, o);
        if (lane == 0) sv[p] = sqrt(a);
    }
    __syncwarp();
    // selection sort by descending sigma (k is tiny); stable for ties
    for (int p = 0; p < k - 1; ++p)
    {
        int best = p;
        for (int q = p + 1; q < k; ++q) if (sv[q] > sv[best]) best = q;
        if (best != p)
        {
            for (int i = lane; i < m; i += 32) { double t = X[p * ldx + i]; X[p * ldx + i] = X[best * ldx + i]; X[best * ldx + i] = t; }
            __syncwarp();
            if (lane == 0) { double t = sv[p]; sv[p] = sv[best]; sv[best] = t; }
            __syncwarp();
        }
    }
    // normalise + canonical sign
    for (int p = 0; p < k; ++p)
    {
        const double s = sv[p];
        const int bi = warp_sign_pivot(X + p * ldx, m, lane);
        const double sgn = (m > 0 && X[p * ldx + bi] < 0.0) ? -1.0 : 1.0;
        const double sc = s > 0.0 ? sgn / s : 0.0;
        __syncwarp();
        for (int i = lane; i < m; i += 32) X[p * ldx + i] *= sc;
    }
    __syncwarp();
    // LAPACK returns min(m,k) singular values: the remaining ones are exactly zero
    if (lane == 0) for (int p = (m < k ? m : k); p < k; ++p) sv[p] = 0.0;
    __syncwarp();
}

// functional F = (P^T M P)^{-1} (M P)^T : P nu x nc column-major (ldp), M nu x nu row-major (ldm)
// work: MP (nu*nc, column-major) + cM (nc*nc) ; F out row-major nc x nu (ldf = nu)
__device__ int cta_dof_functional(const double *P, int nu, int nc, int ldp, const double *M, int ldm,
                                  double *MP, double *cM, double *F, int *s_piv, int tid, int nt)
{
    if (nc == 0) return 0;
    for (int idx = tid; idx < nu * nc; idx += nt)
    {
        const int i = idx % nu, c = idx / nu;
        double s = 0.0;
        for (int t = 0; t < nu; ++t) s += M[i * ldm + t] * P[c * ldp + t];
        MP[c * nu + i] = s;
    }
    __syncthreads();
    for (int idx = tid; idx < nc * nc; idx += nt)
    {
        const int a = idx / nc, b = idx % nc;
        double s = 0.0;
        for (int t = 0; t < nu; ++t) s += P[a * ldp + t] * MP[b * nu + t];
        cM[a * nc + b] = s;
    }
    for (int idx = tid; idx < nc * nu; idx += nt) F[idx] = MP[idx];   // (M P)^T row-major nc x nu == MP column-major
    __syncthreads();
    return cta_lu_solve(cM, nc, nc, F, nu, nu, s_piv, tid, nt);
}

// Symmetric eigendecomposition W = V diag(lambda) V^T by cyclic Jacobi rotations, one warp
// (SymEigensolver::ComputeAll -- dsyevx in the reference, ParELAG_Eigensolver.cpp:57-135; every use on this path goes
// through W^{1/2} and W^{-1/2}, which do not depend on the choice of eigenvectors inside a cluster).
// W: m x m row-major, overwritten (diagonal = eigenvalues on exit); V: m x m row-major, columns = eigenvectors.
__device__ void warp_jacobi_eig(double *W, double *V, int m, int lane)
{
    for (int i = lane; i < m * m; i += 32) V[i] = (i / m == i % m) ? 1.0 : 0.0;
    __syncwarp();
    for (int sweep = 0; sweep < 60; ++sweep)
    {
        double off = 0.0;
        for (int p = 0; p < m - 1; ++p)
            for (int q = p + 1; q < m; ++q)
            {
                const double apq = W[p * m + q], app = W[p * m + p], aqq = W[q * m + q];
                if (apq == 0.0) continue;
                const double r = fabs(apq) / sqrt(fabs(app * aqq));
                if (r > off) off = r;
                if (r < 1e-17) { __syncwarp(); if (lane == 0) { W[p * m + q] = 0.0; W[q * m + p] = 0.0; } __syncwarp(); continue; }
                const double theta = (aqq - app) / (2.0 * apq);
                const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(1.0 + theta * theta));
                const double c = 1.0 / sqrt(1.0 + t * t), sn = c * t;
                __syncwarp();                                   // everybody has read app, aqq, apq
                for (int k = lane; k < m; k += 32)              // columns p, q  (W <- W J)
                {
                    const double wkp = W[k * m + p], wkq = W[k * m + q];
                    W[k * m + p] = c * wkp - sn * wkq; W[k * m + q] = sn * wkp + c * wkq;
                    const double vkp = V[k * m + p], vkq = V[k * m + q];
                    V[k * m + p] = c * vkp - sn * vkq; V[k * m + q] = sn * vkp + c * vkq;
                }
                __syncwarp();
                for (int k = lane; k < m; k += 32)              // rows p, q  (W <- J^T W)
                {
                    const double wpk = W[p * m + k], wqk = W[q * m + k];
                    W[p * m + k] = c * wpk - sn * wqk; W[q * m + k] = sn * wpk + c * wqk;
                }
                __syncwarp();
            }
        if (off < 1e-15) break;
    }
}
// x <- V diag(f(lambda)) V^T x for the columns of X (m x k column-major, ldx); f = sqrt (inv = false) or 1/sqrt;
// y: scratch of m doubles; lambda = diagonal of Wd
__device__ void warp_apply_sqrt(const double *V, const double *Wd, int m, double *X, int k, int ldx, double *y, bool inv, int lane)
{
    for (int t = 0; t < k; ++t)
    {
        for (int c = lane; c < m; c += 32)
        {
            double s = 0.0;
            for (int i = 0; i < m; ++i) s += V[i * m + c] * X[t * ldx + i];
            const double l = sqrt(Wd[c * m + c]);
            y[c] = inv ? s / l : s * l;
        }
        __syncwarp();
        for (int i = lane; i < m; i += 32)
        {
            double s = 0.0;
            for (int c = 0; c < m; ++c) s += V[i * m + c] * y[c];
            X[t * ldx + i] = s;
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------
// traces
// ---------------------------------------------------------------------------
struct TraceArgs
{
    int nAE;
    const int *I, *J;
    const double *pv, *diagM;     // pv per fine dof; diagM per ADof
    const double *denseM;         // dense mass blocks of the entities that have one (dense_off[ae] >= 0)
    const long long *dense_off;
    int max_md;                   // largest such block
    int nT, ldT;
    const double *T;
    double svd_tol;
    const long long *out_off;
    double *out;                  // per AE: p (m x (nT+1)) | mass ((nT+1)^2) | func ((nT+1) x m) | sv (nT)
    int *ndofs_out, *info_out;
    int max_m;
};

// sm: the CTA's workspace -- dynamic shared memory (k_traces) or, for agglomerated entities too large for it, a
// slab of global memory (k_traces_gmem; __syncwarp/__syncthreads order global accesses inside the CTA as well)
__device__ __forceinline__ void traces_one(const TraceArgs &a, int ae, double *sm)
{
    const int lane = threadIdx.x;
    const int s = a.I[ae], m = a.I[ae + 1] - s, nT = a.nT, nc_max = nT + 1;
    double *X = sm;                       // m x nT column-major (ld = max_m)
    double *pvl = X + a.max_m * (nT > 0 ? nT : 1);
    double *dg = pvl + a.max_m;
    double *sv = dg + a.max_m;            // nT
    double *Pl = sv + (nT > 0 ? nT : 1);  // m x nc_max column-major (ld = max_m)
    double *MP = Pl + a.max_m * nc_max;
    double *cM = MP + a.max_m * nc_max;
    double *Mm = cM + nc_max * nc_max;        // dense entities only: mass block, working copy, eigenvectors, scratch
    double *Me = Mm + a.max_md * a.max_md;
    double *V = Me + a.max_md * a.max_md;
    double *ys = V + a.max_md * a.max_md;
    __shared__ int s_piv;
    const int ld = a.max_m;
    const bool dense = a.dense_off && a.dense_off[ae] >= 0;
    double pvMpv = 0.0;
    if (dense)
    {
        const double *Mg = a.denseM + a.dense_off[ae];
        for (int i = lane; i < m * m; i += 32) { const double v = Mg[i]; Mm[i] = v; Me[i] = v; }
        for (int i = lane; i < m; i += 32)
        {
            const int d = a.J[s + i];
            pvl[i] = a.pv[d];
            for (int t = 0; t < nT; ++t) X[t * ld + i] = a.T[(size_t)t * a.ldT + d];
        }
        __syncwarp();
        for (int i = lane; i < m; i += 32)            // dg <- M pv (scratch)
        {
            double sacc = 0.0;
            for (int c = 0; c < m; ++c) sacc += Mm[i * m + c] * pvl[c];
            dg[i] = sacc;
            pvMpv += pvl[i] * sacc;
        }
    }
    else
        for (int i = lane; i < m; i += 32)
        {
            const int d = a.J[s + i];
            pvl[i] = a.pv[d]; dg[i] = a.diagM[s + i];
            pvMpv += pvl[i] * dg[i] * pvl[i];
            for (int t = 0; t < nT; ++t) X[t * ld + i] = a.T[(size_t)t * a.ldT + d];
        }
    for (int o = 16; o > 0; o >>= 1) pvMpv += __shfl_xor_sync(0xffffffffu, pvMpv, o);
    __syncwarp();
    // Deflate: t += (-(pv.M.t)/(pv.M.pv)) pv ; then the weighted SVD: rows scaled by sqrt(diag M), or X = M^{1/2}
    const double sc = -1.0 / pvMpv;
    for (int t = 0; t < nT; ++t)
    {
        double dot = 0.0;
        if (dense) for (int i = lane; i < m; i += 32) dot += dg[i] * X[t * ld + i];
        else for (int i = lane; i < m; i += 32) dot += pvl[i] * dg[i] * X[t * ld + i];
        for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
        if (dense) for (int i = lane; i < m; i += 32) X[t * ld + i] = X[t * ld + i] + (dot * sc) * pvl[i];
        else for (int i = lane; i < m; i += 32) X[t * ld + i] = (X[t * ld + i] + (dot * sc) * pvl[i]) * sqrt(dg[i]);
    }
    __syncwarp();
    if (dense && nT > 0)
    {
        warp_jacobi_eig(Me, V, m, lane);
        warp_apply_sqrt(V, Me, m, X, nT, ld, ys, false, lane);
    }
    if (nT > 0) warp_jacobi_svd(X, m, nT, ld, sv, lane);
    const double s_max_tol = pvMpv * a.svd_tol;
    int k = 0;
    const int nsv = m < nT ? m : nT;
    while (k < nsv && !(sv[k] < s_max_tol)) ++k;
    const int nc = k + 1;
    const double sq = sqrt(pvMpv);
    if (dense && k > 0) warp_apply_sqrt(V, Me, m, X, k, ld, ys, true, lane);
    for (int i = lane; i < m; i += 32)
    {
        Pl[i] = pvl[i];
        if (dense) for (int c = 0; c < k; ++c) Pl[(c + 1) * ld + i] = X[c * ld + i];
        else for (int c = 0; c < k; ++c) Pl[(c + 1) * ld + i] = X[c * ld + i] / sqrt(dg[i]);
    }
    __syncwarp();
    // canonical sign again after the inverse scaling (largest |entry| may have moved), then the scaling by sqrt(pv.M.pv)
    for (int c = 1; c < nc; ++c)
    {
        const int bi = warp_sign_pivot(Pl + c * ld, m, lane);
        const double sg = Pl[c * ld + bi] < 0.0 ? -sq : sq;
        __syncwarp();
        for (int i = lane; i < m; i += 32) Pl[c * ld + i] *= sg;
        __syncwarp();
    }
    double *out = a.out + a.out_off[ae];
    double *p_out = out, *mass_out = out + (size_t)m * nc_max, *func_out = mass_out + nc_max * nc_max, *sv_out = func_out + (size_t)nc_max * m;
    for (int idx = lane; idx < m * nc; idx += 32) { int i = idx % m, c = idx / m; p_out[c * m + i] = Pl[c * ld + i]; }
    // mass = P^T M P (symmetrised), functional = (P^T M P)^{-1} P^T M
    if (dense)
        for (int idx = lane; idx < m * nc; idx += 32)
        {
            int i = idx % m, c = idx / m;
            double sacc = 0.0;
            for (int q = 0; q < m; ++q) sacc += Mm[i * m + q] * Pl[c * ld + q];
            MP[c * m + i] = sacc;
        }
    else
        for (int idx = lane; idx < m * nc; idx += 32) { int i = idx % m, c = idx / m; MP[c * m + i] = dg[i] * Pl[c * ld + i]; }
    __syncwarp();
    for (int idx = lane; idx < nc * nc; idx += 32)
    {
        int x = idx / nc, y = idx % nc;
        double v = 0.0, w = 0.0;
        for (int i = 0; i < m; ++i) { v += Pl[x * ld + i] * MP[y * m + i]; w += Pl[y * ld + i] * MP[x * m + i]; }
        cM[idx] = v;
        mass_out[x * nc + y] = 0.5 * (v + w);
    }
    double *F = func_out;
    for (int idx = lane; idx < nc * m; idx += 32) F[idx] = MP[idx];
    __syncwarp();
    // tiny LU by the warp (same routine, nt = 32)
    int info = 0;
    {
        // cta_lu_solve uses __syncthreads: the CTA is exactly one warp here
        info = cta_lu_solve(cM, nc, nc, F, m, m, &s_piv, lane, 32);
    }
    for (int t = lane; t < nT; t += 32) sv_out[t] = t < nsv ? sv[t] : 0.0;
    if (lane == 0) { a.ndofs_out[ae] = nc; a.info_out[ae] = info; }
}
__global__ void __launch_bounds__(32) k_traces(TraceArgs a)
{
    extern __shared__ double sm[];
    if (blockIdx.x < a.nAE) traces_one(a, blockIdx.x, sm);
}
__global__ void __launch_bounds__(32) k_traces_gmem(TraceArgs a, double *work, size_t stride)
{
    double *sm = work + (size_t)blockIdx.x * stride;
    for (int ae = blockIdx.x; ae < a.nAE; ae += gridDim.x) { traces_one(a, ae, sm); __syncthreads(); }
}

// ---------------------------------------------------------------------------
// extension (facet / ridge / peak)
// ---------------------------------------------------------------------------
struct PoolV { const long long *off; const int *size, *rdoff; const double *vals; };
struct CsrV { const int *I, *J; const double *A; };
struct RowPoolV { const long long *start; const int *len, *J; const double *A; };

struct ExtArgs
{
    int nAE, facet, compute_null;
    const int *uI, *uJ, *uN, *pI, *pJ, *pN, *qI, *qJ;
    const int *aeI, *aeJ;
    PoolV Mu, Mp, Mq;
    const int *slot_u, *slot_p, *slot_q;
    CsrV Dj, Dj1;
    const int *cbI, *cbJ;
    RowPoolV Pj, Dc;
    CsrV Pj1;
    const int *pvc, *pnI, *pnJ;
    int nT, ldT;
    const double *T;
    double svd_tol, smallest_entry;
    const long long *out_off;
    double *out;
    int *k_out, *info_out;
    int mxu, mxp, mxq, mxui, mxpi, mxcb, mxrt;   // max sizes (for the shared-memory carve-up)
};

__device__ __forceinline__ int find_lin(const int *list, int n, int key)
{
    for (int i = 0; i < n; ++i) if (list[i] == key) return i;
    return -1;
}
__device__ __forceinline__ int find_bin(const int *list, int n, int key)
{
    int lo = 0, hi = n - 1;
    while (lo <= hi) { int mid = (lo + hi) >> 1; int v = list[mid]; if (v == key) return mid; if (v < key) lo = mid + 1; else hi = mid - 1; }
    return -1;
}
// assemble the agglomerate matrix from the entity blocks (AssembleAgglomerateMatrix)
__device__ void cta_assemble(double *Mall, int n, const PoolV &P, const int *slot, const int *ents, int nents, int tid)
{
    for (int i = tid; i < n * n; i += LT) Mall[i] = 0.0;
    __syncthreads();
    for (int q = 0; q < nents; ++q)
    {
        const int e = ents[q], m = P.size[e], rd0 = P.rdoff[e];
        const double *blk = P.vals + P.off[e];
        for (int idx = tid; idx < m * m; idx += LT)
        {
            const int la = slot[rd0 + idx / m], lb = slot[rd0 + idx % m];
            Mall[la * n + lb] += blk[idx];
        }
        __syncthreads();
    }
}

// sm: the CTA's workspace -- dynamic shared memory (k_extension) or a slab of global memory (k_extension_gmem) for
// agglomerates whose local matrices do not fit (coarse levels carrying many dofs per entity)
__device__ __forceinline__ void extension_one(const ExtArgs &a, int ae, double *sm)
{
    const int tid = threadIdx.x;
    const int us = a.uI[ae], nua = a.uI[ae + 1] - us, nui = a.uN[ae], nub = nua - nui;
    const int ps = a.pI[ae], npa = a.pI[ae + 1] - ps, npi = a.pN[ae];
    const int qs = a.facet ? 0 : a.qI[ae], nqa = a.facet ? 0 : a.qI[ae + 1] - qs;
    const int cbs = a.cbI[ae], ncb = a.cbI[ae + 1] - cbs;
    const int nrt = a.pnI[ae + 1] - a.pnI[ae];
    const int nT = (a.compute_null && nui > nrt) ? a.nT : 0;
    const int n = a.facet ? nui + npi + 1 : nui + npi;
    const int nrhs = ncb + nrt + nT;
    const int nents = a.aeI[ae + 1] - a.aeI[ae];
    const int *ents = a.aeJ + a.aeI[ae];
    // ---- shared memory carve-up (upper bounds from the host)
    const int nmax = a.mxui + a.mxpi + 1, rmax = a.mxcb + a.mxrt + a.nT, cmax = a.mxrt + a.nT, lbmax = a.mxcb + cmax;
    double *Mall = sm;                                  // nua x nua
    double *Wall = Mall + a.mxu * a.mxu;                // npa x npa
    double *Dall = Wall + a.mxp * a.mxp;                // npa x nua
    double *Brow = Dall + a.mxp * a.mxu;                // npi x nua
    double *A = Brow + a.mxpi * a.mxu;                  // n x n
    double *R = A + nmax * nmax;                        // n x nrhs
    double *Rb = R + nmax * rmax;                       // nub x ncb
    double *G = Rb + a.mxu * a.mxcb;                    // npa x ncb (ridge) / scratch
    double *X = G + a.mxp * a.mxcb;                     // nui x nT column-major (target residual)
    double *PL = X + a.mxui * (a.nT > 0 ? a.nT : 1);    // nui x (nrt+nT) column-major: [bub | nul]
    double *MP = PL + a.mxui * (cmax > 0 ? cmax : 1);   // scratch nui x cmax
    double *cM = MP + (a.mxu > a.mxp ? a.mxu : a.mxp) * (lbmax > 0 ? lbmax : 1);  // (MP is reused as MB: nua x lbmax)
    double *W2 = cM + lbmax * lbmax;                    // nqa x nqa (ridge)
    double *D2 = W2 + a.mxq * a.mxq;                    // nqa x npi
    double *TMP = D2 + a.mxq * a.mxpi;                  // nqa x npi
    double *sv = TMP + a.mxq * a.mxpi;                  // nT
    int *su = reinterpret_cast<int *>(sv + (a.nT > 0 ? a.nT : 1));
    int *sp = su + a.mxu;
    int *sq = sp + a.mxp;
    int *scb = sq + a.mxq;
    __shared__ int s_piv, s_k;
    for (int i = tid; i < nua; i += LT) su[i] = a.uJ[us + i];
    for (int i = tid; i < npa; i += LT) sp[i] = a.pJ[ps + i];
    for (int i = tid; i < nqa; i += LT) sq[i] = a.qJ[qs + i];
    for (int i = tid; i < ncb; i += LT) scb[i] = a.cbJ[cbs + i];
    __syncthreads();
    // ---- local matrices
    cta_assemble(Mall, nua, a.Mu, a.slot_u, ents, nents, tid);
    cta_assemble(Wall, npa, a.Mp, a.slot_p, ents, nents, tid);
    for (int i = tid; i < npa * nua; i += LT) Dall[i] = 0.0;
    __syncthreads();
    for (int r = tid; r < npa; r += LT)
    {
        const int row = sp[r];
        for (int k = a.Dj.I[row]; k < a.Dj.I[row + 1]; ++k)
        {
            const int lu = find_lin(su, nua, a.Dj.J[k]);
            if (lu >= 0) Dall[r * nua + lu] = a.Dj.A[k];
        }
    }
    __syncthreads();
    for (int idx = tid; idx < npi * nua; idx += LT)      // B = (W D) rows of interior p dofs
    {
        const int i = idx / nua, c = idx % nua;
        double s = 0.0;
        for (int t = 0; t < npa; ++t) s += Wall[i * npa + t] * Dall[t * nua + c];
        Brow[idx] = s;
    }
    for (int i = tid; i < n * n; i += LT) A[i] = 0.0;
    __syncthreads();
    for (int idx = tid; idx < nui * nui; idx += LT) A[(idx / nui) * n + idx % nui] = Mall[(idx / nui) * nua + idx % nui];
    for (int idx = tid; idx < npi * nui; idx += LT)
    {
        const int i = idx / nui, c = idx % nui;
        const double v = Brow[i * nua + c];
        A[(nui + i) * n + c] = v; A[c * n + nui + i] = v;
    }
    if (a.facet)
    {
        // T block: tloc = Wloc * pvloc, pvloc = column pv of P_{j+1} on the interior p dofs
        const int pvc = a.pvc[ae];
        for (int i = tid; i < npi; i += LT)
        {
            const int row = sp[i];
            double v = 0.0;
            for (int k = a.Pj1.I[row]; k < a.Pj1.I[row + 1]; ++k) if (a.Pj1.J[k] == pvc) { v = a.Pj1.A[k]; break; }
            G[i] = v;
        }
        __syncthreads();
        for (int i = tid; i < npi; i += LT)
        {
            double s = 0.0;
            for (int t = 0; t < npi; ++t) s += Wall[i * npa + t] * G[t];
            A[(n - 1) * n + nui + i] = s; A[(nui + i) * n + n - 1] = s;
        }
        __syncthreads();
    }
    else
    {
        // -C = -(D2^T W2 D2) on the interior p dofs (GetMinusC)
        cta_assemble(W2, nqa, a.Mq, a.slot_q, ents, nents, tid);
        for (int i = tid; i < nqa * npi; i += LT) D2[i] = 0.0;
        __syncthreads();
        for (int r = tid; r < nqa; r += LT)
        {
            const int row = sq[r];
            for (int k = a.Dj1.I[row]; k < a.Dj1.I[row + 1]; ++k)
            {
                const int lp = find_lin(sp, npi, a.Dj1.J[k]);
                if (lp >= 0) D2[r * npi + lp] = a.Dj1.A[k];
            }
        }
        __syncthreads();
        for (int idx = tid; idx < nqa * npi; idx += LT)
        {
            const int r = idx / npi, c = idx % npi;
            double s = 0.0;
            for (int t = 0; t < nqa; ++t) s += W2[r * nqa + t] * D2[t * npi + c];
            TMP[idx] = s;
        }
        __syncthreads();
        for (int idx = tid; idx < npi * npi; idx += LT)
        {
            const int i = idx / npi, j = idx % npi;
            double s = 0.0;
            for (int t = 0; t < nqa; ++t) s += D2[t * npi + i] * TMP[t * npi + j];
            A[(nui + i) * n + nui + j] = -s;
        }
        __syncthreads();
    }
    // ---- boundary traces R_b (nub x ncb) from the rows of P_j written by earlier stages
    for (int i = tid; i < nub * ncb; i += LT) Rb[i] = 0.0;
    __syncthreads();
    for (int r = tid; r < nub; r += LT)
    {
        const int d = su[nui + r];
        const long long st = a.Pj.start[d];
        for (int k = 0; k < a.Pj.len[d]; ++k)
        {
            const int c = find_bin(scb, ncb, a.Pj.J[st + k]);
            if (c >= 0) Rb[r * ncb + c] = a.Pj.A[st + k];
        }
    }
    for (int i = tid; i < n * nrhs; i += LT) R[i] = 0.0;
    __syncthreads();
    // ---- right-hand sides: [extension of the boundary traces | bubbles | targets]
    for (int idx = tid; idx < nui * ncb; idx += LT)
    {
        const int i = idx / ncb, c = idx % ncb;
        double s = 0.0;
        for (int t = 0; t < nub; ++t) s += Mall[i * nua + nui + t] * Rb[t * ncb + c];
        R[i * nrhs + c] = -s;
    }
    if (a.facet)
    {
        for (int idx = tid; idx < npi * ncb; idx += LT)
        {
            const int i = idx / ncb, c = idx % ncb;
            double s = 0.0;
            for (int t = 0; t < nub; ++t) s += Brow[i * nua + nui + t] * Rb[t * ncb + c];
            R[(nui + i) * nrhs + c] = -s;
        }
    }
    else
    {
        // G = (P_{j+1} D_c)_loc - D_loc[:, bdr] R_b  on ALL p dofs of the agglomerate
        for (int r = tid; r < npa; r += LT)
        {
            for (int c = 0; c < ncb; ++c) G[r * ncb + c] = 0.0;
            const int row = sp[r];
            for (int k = a.Pj1.I[row]; k < a.Pj1.I[row + 1]; ++k)
            {
                const int kc = a.Pj1.J[k];
                const double v = a.Pj1.A[k];
                const long long st = a.Dc.start[kc];
                for (int t = 0; t < a.Dc.len[kc]; ++t)
                {
                    const int c = find_bin(scb, ncb, a.Dc.J[st + t]);
                    if (c >= 0) G[r * ncb + c] += v * a.Dc.A[st + t];
                }
            }
            for (int c = 0; c < ncb; ++c)
            {
                double s = 0.0;
                for (int t = 0; t < nub; ++t) s += Dall[r * nua + nui + t] * Rb[t * ncb + c];
                G[r * ncb + c] -= s;
            }
        }
        __syncthreads();
        for (int idx = tid; idx < npi * ncb; idx += LT)
        {
            const int i = idx / ncb, c = idx % ncb;
            double s = 0.0;
            for (int t = 0; t < npa; ++t) s += Wall[i * npa + t] * G[t * ncb + c];
            R[(nui + i) * nrhs + c] = s;
        }
    }
    // bubbles: rhs_p = Wloc * P_{j+1}[p_int, null coarse dofs]
    if (nrt > 0)
    {
        __syncthreads();
        const int *pn = a.pnJ + a.pnI[ae];
        for (int idx = tid; idx < npi * nrt; idx += LT)     // sub -> MP scratch (npi x nrt row-major)
        {
            const int i = idx / nrt, q = idx % nrt, row = sp[i];
            double v = 0.0;
            for (int k = a.Pj1.I[row]; k < a.Pj1.I[row + 1]; ++k) if (a.Pj1.J[k] == pn[q]) { v = a.Pj1.A[k]; break; }
            MP[idx] = v;
        }
        __syncthreads();
        for (int idx = tid; idx < npi * nrt; idx += LT)
        {
            const int i = idx / nrt, q = idx % nrt;
            double s = 0.0;
            for (int t = 0; t < npi; ++t) s += Wall[i * npa + t] * MP[t * nrt + q];
            R[(nui + i) * nrhs + ncb + q] = s;
        }
    }
    // targets: rhs_u = -M_ib T_bdr ; rhs_p = B_ii T_int
    for (int idx = tid; idx < nui * nT; idx += LT)
    {
        const int i = idx / nT, t = idx % nT;
        double s = 0.0;
        for (int b = 0; b < nub; ++b) s += Mall[i * nua + nui + b] * a.T[(size_t)t * a.ldT + su[nui + b]];
        R[i * nrhs + ncb + nrt + t] = -s;
    }
    for (int idx = tid; idx < npi * nT; idx += LT)
    {
        const int i = idx / nT, t = idx % nT;
        double s = 0.0;
        for (int c = 0; c < nui; ++c) s += Brow[i * nua + c] * a.T[(size_t)t * a.ldT + su[c]];
        R[(nui + i) * nrhs + ncb + nrt + t] = s;
    }
    __syncthreads();
    // ---- solve all right-hand sides at once
    int info = 0;
    // without interior u dofs only the facet stage still needs the solve: its last unknown is the multiplier that becomes
    // the coarse derivative row of the PV dof (an agglomerated entity with a single member: [0 t; t 0] [p; lambda])
    if (nui > 0 || a.facet) info = cta_lu_solve(A, n, n, R, nrhs, nrhs, &s_piv, tid, LT);
    __syncthreads();
    // ---- outputs
    double *out = a.out + a.out_off[ae];
    double *ext_o = out;                                   // nui x ncb   (row-major)
    double *bub_o = ext_o + (size_t)nui * ncb;             // nui x nrt
    double *nul_o = bub_o + (size_t)nui * nrt;             // nui x a.nT  (first k columns valid)
    double *lam_o = nul_o + (size_t)nui * a.nT;            // ncb
    double *func_o = lam_o + ncb;                          // (nrt + a.nT) x nui
    double *mass_o = func_o + (size_t)(nrt + a.nT) * nui;  // (ncb + nrt + a.nT)^2, leading (ncb+nrt+k)^2 valid
    double *sv_o = mass_o + (size_t)(ncb + nrt + a.nT) * (ncb + nrt + a.nT);
    for (int idx = tid; idx < nui * ncb; idx += LT) ext_o[idx] = R[(idx / ncb) * nrhs + idx % ncb];
    for (int idx = tid; idx < nui * nrt; idx += LT) { const int i = idx / nrt, q = idx % nrt; const double v = R[i * nrhs + ncb + q]; bub_o[idx] = v; PL[q * nui + i] = v; }
    if (a.facet)
        for (int c = tid; c < ncb; c += LT) { const double l = R[(n - 1) * nrhs + c]; lam_o[c] = fabs(l) > a.smallest_entry ? -l : 0.0; }
    // target residual -> SVD -> NullSpace dofs
    for (int idx = tid; idx < nui * nT; idx += LT)
    {
        const int i = idx / nT, t = idx % nT;
        X[t * nui + i] = a.T[(size_t)t * a.ldT + su[i]] - R[i * nrhs + ncb + nrt + t];
    }
    if (tid == 0) s_k = 0;
    __syncthreads();
    if (nT > 0 && tid < 32)
    {
        warp_jacobi_svd(X, nui, nT, nui, sv, tid);
        if (tid == 0)
        {
            int k = 0;
            const int nsv = nui < nT ? nui : nT;
            while (k < nsv && !(sv[k] < a.svd_tol)) ++k;
            s_k = k;
        }
    }
    __syncthreads();
    const int k = s_k, nc = nrt + k, nlb = ncb + nc;
    for (int idx = tid; idx < nui * k; idx += LT) { const int i = idx % nui, c = idx / nui; const double v = X[c * nui + i]; PL[(nrt + c) * nui + i] = v; nul_o[i * a.nT + c] = v; }
    for (int t = tid; t < a.nT; t += LT) sv_o[t] = (t < nT && t < (nui < nT ? nui : nT)) ? sv[t] : 0.0;
    __syncthreads();
    // dof functional of the interior coarse dofs [RangeT | Null] w.r.t. M_ii
    int info2 = 0;
    if (nc > 0)
    {
        // M_ii as a compact nui x nui matrix in A (the factorisation is no longer needed)
        for (int idx = tid; idx < nui * nui; idx += LT) A[idx] = Mall[(idx / nui) * nua + idx % nui];
        __syncthreads();
        info2 = cta_dof_functional(PL, nui, nc, nui, A, nui, MP, cM, R, &s_piv, tid, LT);
        __syncthreads();
        for (int idx = tid; idx < nc * nui; idx += LT) func_o[idx] = R[idx];
    }
    __syncthreads();
    // coarse mass: basis^T M_aa basis, basis = [[ext bub nul]; [Rb 0 0]]  (order [bdr | RangeT | Null])
    double *MB = MP;     // nua x nlb row-major
    for (int idx = tid; idx < nua * nlb; idx += LT)
    {
        const int i = idx / nlb, c = idx % nlb;
        double s = 0.0;
        for (int t = 0; t < nua; ++t)
        {
            double b;
            if (t < nui) b = c < ncb ? ext_o[t * ncb + c] : PL[(c - ncb) * nui + t];
            else b = c < ncb ? Rb[(t - nui) * ncb + c] : 0.0;
            s += Mall[i * nua + t] * b;
        }
        MB[idx] = s;
    }
    __syncthreads();
    const int ldm = ncb + nrt + a.nT;
    for (int idx = tid; idx < nlb * nlb; idx += LT)
    {
        const int x = idx / nlb, y = idx % nlb;
        double v = 0.0, w = 0.0;
        for (int t = 0; t < nua; ++t)
        {
            double bx, by;
            if (t < nui) { bx = x < ncb ? ext_o[t * ncb + x] : PL[(x - ncb) * nui + t]; by = y < ncb ? ext_o[t * ncb + y] : PL[(y - ncb) * nui + t]; }
            else { bx = x < ncb ? Rb[(t - nui) * ncb + x] : 0.0; by = y < ncb ? Rb[(t - nui) * ncb + y] : 0.0; }
            v += bx * MB[t * nlb + y];
            w += by * MB[t * nlb + x];
        }
        mass_o[x * ldm + y] = 0.5 * (v + w);
    }
    if (tid == 0) { a.k_out[ae] = k; a.info_out[ae] = info ? info : (info2 ? 1000 + info2 : 0); }
}
// list: the agglomerates of this launch (null: all of them)
__global__ void __launch_bounds__(LT) k_extension(ExtArgs a, const int *__restrict__ list, int nlist)
{
    extern __shared__ double sm[];
    if ((int)blockIdx.x < nlist) extension_one(a, list ? list[blockIdx.x] : (int)blockIdx.x, sm);
}
__global__ void __launch_bounds__(LT) k_extension_gmem(ExtArgs a, const int *__restrict__ list, int nlist, double *work, size_t stride)
{
    double *sm = work + (size_t)blockIdx.x * stride;
    for (int i = blockIdx.x; i < nlist; i += gridDim.x) { extension_one(a, list[i], sm); __syncthreads(); }
}

// ---------------------------------------------------------------------------
// host wrappers: upload the batch description, run, download the results
// ---------------------------------------------------------------------------
namespace
{
// wall-clock split of the batched calls (pe_local_stage_seconds): [0] H2D staging incl. cudaMalloc,
// [1] kernel, [2] D2H of the results, [3] bytes uploaded, [4] bytes downloaded, [5] calls
static double g_stage[6] = {0, 0, 0, 0, 0, 0};
static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
// workspace bytes above which an agglomerate goes to the global-memory kernel: the built-in limit, or PE_TUNE_LOCAL_SMEM_BYTES
// when that is set (clamped to the built-in limit)
static size_t local_smem_limit(size_t builtin)
{
    const int v = pe_get_tuning(PE_TUNE_LOCAL_SMEM_BYTES);
    return v > 0 ? std::min(builtin, (size_t)v) : builtin;
}
// Device copies of inputs that stay constant over one Coarsen() (entity mass pools, agglomerate tables, the
// fine D_j): uploaded once per pe_local_cache(1) ... pe_local_cache(0) scope and shared by the per-form,
// per-codimension batched calls, keyed by host address and size.  At 144^3 hexahedra the 24 extension
// calls of the first level re-sent 31 GB without it.
static bool g_cache_on = false;
static std::map<std::pair<const void *, size_t>, void *> g_cache;
// Large host -> device copies of the setup go through two pinned staging buffers: host threads copy the next chunk
// into pinned memory while the previous chunk travels (pageable cudaMemcpy ran at ~5 GB/s on the B200 host: 17 GB of
// constant inputs per Coarsen() of the 144^3 level cost 3.5 s).
static int staged_h2d(void *dst, const void *src, size_t bytes, cudaStream_t st)
{
    const size_t CH = (size_t)32 << 20;
    if (bytes < 2 * CH) { PE_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st)); return 0; }
    static char *pin[2] = {nullptr, nullptr};
    static cudaEvent_t done[2];
    if (!pin[0])
    {
        if (cudaMallocHost(&pin[0], CH) != cudaSuccess || cudaMallocHost(&pin[1], CH) != cudaSuccess)
        {
            (void)cudaGetLastError();
            pin[0] = nullptr;
            PE_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
            return 0;
        }
        PE_CUDA(cudaEventCreateWithFlags(&done[0], cudaEventDisableTiming));
        PE_CUDA(cudaEventCreateWithFlags(&done[1], cudaEventDisableTiming));
    }
    int k = 0;
    bool used[2] = {false, false};
    for (size_t off = 0; off < bytes; off += CH, k ^= 1)
    {
        const size_t len = std::min(CH, bytes - off);
        if (used[k]) PE_CUDA(cudaEventSynchronize(done[k]));
        const char *s0 = static_cast<const char *>(src) + off;
        const size_t piece = (size_t)4 << 20;
        const int np = (int)((len + piece - 1) / piece);
#pragma omp parallel for schedule(static)
        for (int q = 0; q < np; ++q)
        {
            const size_t o = (size_t)q * piece;
            memcpy(pin[k] + o, s0 + o, std::min(piece, len - o));
        }
        PE_CUDA(cudaMemcpyAsync(static_cast<char *>(dst) + off, pin[k], len, cudaMemcpyHostToDevice, st));
        PE_CUDA(cudaEventRecord(done[k], st));
        used[k] = true;
    }
    for (int q = 0; q < 2; ++q) if (used[q]) PE_CUDA(cudaEventSynchronize(done[q]));
    return 0;
}
struct DevBuf
{
    std::vector<void *> ptrs;
    cudaStream_t st;
    explicit DevBuf(cudaStream_t s) : st(s) {}
    ~DevBuf() { for (void *p : ptrs) cudaFree(p); }
    // constant input: served from the cache when a scope is open
    template <class T> int upc(const T *h, size_t n, const T **out)
    {
        const size_t bytes = sizeof(T) * n;
        if (!g_cache_on || !h || bytes < ((size_t)1 << 16)) return up(h, n, out);
        auto key = std::make_pair((const void *)h, bytes);
        auto it = g_cache.find(key);
        if (it == g_cache.end())
        {
            T *d = nullptr;
            PE_CUDA(cudaMalloc(&d, bytes));
            PE_TRY(staged_h2d(d, h, bytes, st));
            g_stage[3] += (double)bytes;
            it = g_cache.emplace(key, (void *)d).first;
        }
        *out = static_cast<const T *>(it->second);
        return 0;
    }
    template <class T> int up(const T *h, size_t n, const T **out)
    {
        T *d = nullptr;
        PE_CUDA(cudaMalloc(&d, sizeof(T) * (n > 0 ? n : 1)));
        ptrs.push_back(d);
        if (n > 0 && h) { PE_TRY(staged_h2d(d, h, sizeof(T) * n, st)); g_stage[3] += (double)(sizeof(T) * n); }
        *out = d;
        return 0;
    }
    template <class T> int alloc(size_t n, T **out)
    {
        PE_CUDA(cudaMalloc(out, sizeof(T) * (n > 0 ? n : 1)));
        ptrs.push_back(*out);
        return 0;
    }
};
}

extern "C" int pe_local_cache(pe_ctx *ctx, int enable)
{
    PE_CHECK(ctx, "bad arguments");
    if (!enable)
    {
        PE_CUDA(cudaStreamSynchronize(ctx->stream));
        for (auto &kv : g_cache) cudaFree(kv.second);
        g_cache.clear();
    }
    g_cache_on = enable != 0;
    return 0;
}

extern "C" int pe_local_stage_seconds(double *out6, int reset)
{
    if (out6) for (int i = 0; i < 6; ++i) out6[i] = g_stage[i];
    if (reset) for (int i = 0; i < 6; ++i) g_stage[i] = 0.0;
    return 0;
}

extern "C" int pe_batched_traces(pe_ctx *ctx, const pe_trace_batch *b)
{
    PE_CHECK(ctx && b, "bad arguments");
    if (b->nAE == 0) return 0;
    cudaStream_t st = ctx->stream;
    DevBuf D(st);
    TraceArgs a{};
    a.nAE = b->nAE; a.nT = b->nT; a.ldT = b->ldT; a.svd_tol = b->svd_tol;
    const int nadof = b->I[b->nAE];
    int max_m = 0;
    for (int e = 0; e < b->nAE; ++e) max_m = std::max(max_m, b->I[e + 1] - b->I[e]);
    a.max_m = max_m;
    PE_TRY(D.up(b->I, (size_t)b->nAE + 1, &a.I));
    PE_TRY(D.up(b->J, (size_t)nadof, &a.J));
    PE_TRY(D.up(b->pv, (size_t)b->ndofs, &a.pv));
    PE_TRY(D.up(b->diagM, (size_t)nadof, &a.diagM));
    a.max_md = 0;
    if (b->denseM && b->dense_off)
    {
        size_t total = 0;
        for (int e = 0; e < b->nAE; ++e)
            if (b->dense_off[e] >= 0)
            {
                const int m = b->I[e + 1] - b->I[e];
                a.max_md = std::max(a.max_md, m);
                total = std::max(total, (size_t)b->dense_off[e] + (size_t)m * m);
            }
        if (a.max_md > 0)
        {
            PE_TRY(D.up(b->denseM, total, &a.denseM));
            PE_TRY(D.up(b->dense_off, (size_t)b->nAE, (const long long **)&a.dense_off));
        }
    }
    PE_TRY(D.upc(b->T, (size_t)b->ldT * b->nT, &a.T));
    PE_TRY(D.up(b->out_off, (size_t)b->nAE + 1, (const long long **)&a.out_off));
    const size_t out_n = (size_t)b->out_off[b->nAE];
    PE_TRY(D.alloc(out_n, &a.out));
    PE_CUDA(cudaMemsetAsync(a.out, 0, sizeof(double) * out_n, st));
    PE_TRY(D.alloc((size_t)b->nAE, &a.ndofs_out));
    PE_TRY(D.alloc((size_t)b->nAE, &a.info_out));
    const int nT1 = b->nT > 0 ? b->nT : 1, ncm = b->nT + 1;
    size_t smem = sizeof(double) * ((size_t)max_m * nT1 + 2 * (size_t)max_m + nT1 + 2 * (size_t)max_m * ncm + (size_t)ncm * ncm + (size_t)max_m * ncm
                                    + 3 * (size_t)a.max_md * a.max_md + (size_t)a.max_md);
    if (smem <= local_smem_limit(200 * 1024))
    {
        pe_variant_add(PE_VARIANT_TRACES_SMEM, b->nAE);
        PE_CUDA(cudaFuncSetAttribute(k_traces, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_traces<<<b->nAE, 32, smem, st>>>(a);
    }
    else
    {
        pe_variant_add(PE_VARIANT_TRACES_GMEM, b->nAE);
        // agglomerated entity too large for shared memory (coarse levels with many dofs per entity): global workspace
        const int grid = std::min(b->nAE, 148 * 16);
        pe_variant_add(PE_VARIANT_TRACES_GMEM_REUSE, b->nAE - grid);
        const size_t stride = (smem / sizeof(double) + 31) & ~(size_t)31;
        double *work = nullptr;
        PE_TRY(D.alloc(stride * (size_t)grid, &work));
        k_traces_gmem<<<grid, 32, 0, st>>>(a, work, stride);
    }
    PE_LAUNCHED(ctx);
    PE_CUDA(cudaMemcpyAsync(b->out, a.out, sizeof(double) * out_n, cudaMemcpyDeviceToHost, st));
    PE_CUDA(cudaMemcpyAsync(b->ndofs_out, a.ndofs_out, sizeof(int) * (size_t)b->nAE, cudaMemcpyDeviceToHost, st));
    std::vector<int> info(b->nAE);
    PE_CUDA(cudaMemcpyAsync(info.data(), a.info_out, sizeof(int) * (size_t)b->nAE, cudaMemcpyDeviceToHost, st));
    PE_CUDA(cudaStreamSynchronize(st));
    for (int e = 0; e < b->nAE; ++e)
        PE_CHECK(info[e] == 0, "pe_batched_traces: singular local coarse mass matrix (agglomerate " + std::to_string(e) + ")");
    return 0;
}

static int up_pool(DevBuf &D, const pe_blockpool_view &h, PoolV &d)
{
    PE_TRY(D.upc(h.off, (size_t)h.n + 1, (const long long **)&d.off));
    PE_TRY(D.upc(h.size, (size_t)h.n, &d.size));
    PE_TRY(D.up(h.rdoff, (size_t)h.n + 1, &d.rdoff));       // a temporary of the caller
    PE_TRY(D.upc(h.vals, (size_t)(h.n > 0 ? h.off[h.n] : 0), &d.vals));
    return 0;
}
static int up_csr(DevBuf &D, const pe_csr_view &h, CsrV &d, bool constant = false)
{
    const size_t nnz = h.nrows > 0 && h.I ? (size_t)h.I[h.nrows] : 0;
    if (constant)
    {
        PE_TRY(D.upc(h.I, (size_t)h.nrows + 1, &d.I));
        PE_TRY(D.upc(h.J, nnz, &d.J));
        PE_TRY(D.upc(h.A, nnz, &d.A));
        return 0;
    }
    PE_TRY(D.up(h.I, (size_t)h.nrows + 1, &d.I));
    PE_TRY(D.up(h.J, nnz, &d.J));
    PE_TRY(D.up(h.A, nnz, &d.A));
    return 0;
}
// Row pools (P_j, coarse D_j under construction) change between calls and are sent every time.  (An incremental
// device mirror that uploaded only the appended entries was measured and removed: when the extension of form j runs,
// P_j holds only the trace rows, so the pools are a small part of the 17 GB the level uploads.)
static int up_rowpool(DevBuf &D, const pe_rowpool_view &h, RowPoolV &d)
{
    PE_TRY(D.up(h.start, (size_t)h.nrows, (const long long **)&d.start));
    PE_TRY(D.up(h.len, (size_t)h.nrows, &d.len));
    PE_TRY(D.up(h.J, (size_t)h.pool_size, &d.J));
    PE_TRY(D.up(h.A, (size_t)h.pool_size, &d.A));
    return 0;
}

extern "C" int pe_batched_extension(pe_ctx *ctx, const pe_extension_batch *b)
{
    PE_CHECK(ctx && b, "bad arguments");
    if (b->nAE == 0) return 0;
    cudaStream_t st = ctx->stream;
    const double t_begin = now_s();
    DevBuf D(st);
    ExtArgs a{};
    const int nAE = b->nAE;
    a.nAE = nAE; a.facet = b->facet; a.compute_null = b->compute_null;
    a.nT = b->nT; a.ldT = b->ldT; a.svd_tol = b->svd_tol; a.smallest_entry = b->smallest_entry;
    // constant over the Coarsen() scope: DofAgglomeration tables, AE -> entity table, mass pools, slots, fine D_j
    PE_TRY(D.upc(b->uI, (size_t)nAE + 1, &a.uI)); PE_TRY(D.upc(b->uJ, (size_t)b->uI[nAE], &a.uJ)); PE_TRY(D.upc(b->uNint, (size_t)nAE, &a.uN));
    PE_TRY(D.upc(b->pI, (size_t)nAE + 1, &a.pI)); PE_TRY(D.upc(b->pJ, (size_t)b->pI[nAE], &a.pJ)); PE_TRY(D.upc(b->pNint, (size_t)nAE, &a.pN));
    PE_TRY(D.upc(b->aeI, (size_t)nAE + 1, &a.aeI)); PE_TRY(D.upc(b->aeJ, (size_t)b->aeI[nAE], &a.aeJ));
    PE_TRY(up_pool(D, b->Mu, a.Mu)); PE_TRY(up_pool(D, b->Mp, a.Mp));
    PE_TRY(D.upc(b->slot_u, (size_t)b->Mu.rdoff[b->Mu.n], &a.slot_u));
    PE_TRY(D.upc(b->slot_p, (size_t)b->Mp.rdoff[b->Mp.n], &a.slot_p));
    PE_TRY(up_csr(D, b->Dj, a.Dj, true));
    PE_TRY(D.up(b->cbI, (size_t)nAE + 1, &a.cbI)); PE_TRY(D.up(b->cbJ, (size_t)b->cbI[nAE], &a.cbJ));
    PE_TRY(up_rowpool(D, b->Pj, a.Pj));
    PE_TRY(up_csr(D, b->Pj1, a.Pj1, true));                 // the finished P of form j+1
    PE_TRY(D.up(b->pnI, (size_t)nAE + 1, &a.pnI)); PE_TRY(D.up(b->pnJ, (size_t)b->pnI[nAE], &a.pnJ));
    if (b->facet) PE_TRY(D.up(b->pvc, (size_t)nAE, &a.pvc));
    else
    {
        PE_TRY(D.upc(b->qI, (size_t)nAE + 1, &a.qI)); PE_TRY(D.upc(b->qJ, (size_t)b->qI[nAE], &a.qJ));
        PE_TRY(up_pool(D, b->Mq, a.Mq));
        PE_TRY(D.upc(b->slot_q, (size_t)b->Mq.rdoff[b->Mq.n], &a.slot_q));
        PE_TRY(up_csr(D, b->Dj1, a.Dj1, true));
        PE_TRY(up_rowpool(D, b->Dc, a.Dc));
    }
    PE_TRY(D.upc(b->T, (size_t)b->ldT * b->nT, &a.T));
    PE_TRY(D.up(b->out_off, (size_t)nAE + 1, (const long long **)&a.out_off));
    const size_t out_n = (size_t)b->out_off[nAE];
    PE_TRY(D.alloc(out_n, &a.out));
    PE_CUDA(cudaMemsetAsync(a.out, 0, sizeof(double) * out_n, st));
    PE_TRY(D.alloc((size_t)nAE, &a.k_out));
    PE_TRY(D.alloc((size_t)nAE, &a.info_out));
    // Workspace of one agglomerate as a function of the size bounds of its launch.  Agglomerates that fit into shared
    // memory go to k_extension (carve-up from the maxima over THAT set); the others -- coarse levels carrying many dofs
    // per entity, e.g. the NullSpace dofs of a deformed mesh -- to k_extension_gmem with a workspace slab in HBM.
    struct Bounds { int mxu = 0, mxp = 0, mxq = 0, mxui = 0, mxpi = 0, mxcb = 0, mxrt = 0; };
    auto grow = [&](Bounds &B, int e) {
        B.mxu = std::max(B.mxu, b->uI[e + 1] - b->uI[e]); B.mxui = std::max(B.mxui, b->uNint[e]);
        B.mxp = std::max(B.mxp, b->pI[e + 1] - b->pI[e]); B.mxpi = std::max(B.mxpi, b->pNint[e]);
        if (!b->facet) B.mxq = std::max(B.mxq, b->qI[e + 1] - b->qI[e]);
        B.mxcb = std::max(B.mxcb, b->cbI[e + 1] - b->cbI[e]); B.mxrt = std::max(B.mxrt, b->pnI[e + 1] - b->pnI[e]);
    };
    const int nTa = a.nT;
    auto bytes_of = [nTa](const Bounds &B) -> size_t {
        const size_t nmax = (size_t)B.mxui + B.mxpi + 1, rmax = (size_t)B.mxcb + B.mxrt + nTa, cmax = (size_t)B.mxrt + nTa, lbmax = B.mxcb + cmax;
        const size_t nT1 = nTa > 0 ? nTa : 1;
        // the functional / solve scratch reuses R (n x nrhs) for an nc x nui matrix and MP for nua x nlb: covered by
        // nmax*rmax >= cmax*mxui only if rmax >= cmax (true) and nmax >= mxui (true)
        const size_t nd = (size_t)B.mxu * B.mxu + (size_t)B.mxp * B.mxp + (size_t)B.mxp * B.mxu + (size_t)B.mxpi * B.mxu + nmax * nmax + nmax * rmax
                          + (size_t)B.mxu * B.mxcb + (size_t)B.mxp * B.mxcb + (size_t)B.mxui * nT1 + (size_t)B.mxui * (cmax > 0 ? cmax : 1)
                          + (size_t)std::max(B.mxu, B.mxp) * (lbmax > 0 ? lbmax : 1) + lbmax * lbmax + (size_t)B.mxq * B.mxq + 2 * (size_t)B.mxq * B.mxpi + nT1;
        return sizeof(double) * nd + sizeof(int) * ((size_t)B.mxu + B.mxp + B.mxq + B.mxcb) + 16;
    };
    const size_t SMEM_LIMIT = local_smem_limit(220 * 1024);
    Bounds all, fit, big;
    std::vector<int> fit_list, big_list;
    for (int e = 0; e < nAE; ++e) grow(all, e);
    if (bytes_of(all) > SMEM_LIMIT)
    {
        for (int e = 0; e < nAE; ++e)
        {
            Bounds one; grow(one, e);
            if (bytes_of(one) <= SMEM_LIMIT) { fit_list.push_back(e); grow(fit, e); } else { big_list.push_back(e); grow(big, e); }
        }
        if (bytes_of(fit) > SMEM_LIMIT)      // maxima attained by different agglomerates: keep it simple
        {
            big_list.resize(nAE); for (int e = 0; e < nAE; ++e) big_list[e] = e;
            fit_list.clear(); big = all;
        }
    }
    auto set_bounds = [&](const Bounds &B) { a.mxu = B.mxu; a.mxp = B.mxp; a.mxq = B.mxq; a.mxui = B.mxui; a.mxpi = B.mxpi; a.mxcb = B.mxcb; a.mxrt = B.mxrt; };
    PE_CUDA(cudaStreamSynchronize(st));
    const double t_up = now_s();
    pe_variant_add(PE_VARIANT_EXT_SMEM, big_list.empty() ? nAE : (int64_t)fit_list.size());
    pe_variant_add(PE_VARIANT_EXT_GMEM, (int64_t)big_list.size());
    if (big_list.empty())
    {
        set_bounds(all);
        const size_t smem = bytes_of(all);
        PE_CUDA(cudaFuncSetAttribute(k_extension, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_extension<<<nAE, LT, smem, st>>>(a, nullptr, nAE);
    }
    else
    {
        const int *list_d = nullptr;
        if (!fit_list.empty())
        {
            set_bounds(fit);
            const size_t smem = bytes_of(fit);
            PE_TRY(D.up(fit_list.data(), fit_list.size(), &list_d));
            pe_variant_add(PE_VARIANT_EXT_SPLIT_SMEM, (int64_t)fit_list.size());
            PE_CUDA(cudaFuncSetAttribute(k_extension, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            k_extension<<<(int)fit_list.size(), LT, smem, st>>>(a, list_d, (int)fit_list.size());
            PE_LAUNCHED(ctx);
        }
        set_bounds(big);
        const size_t stride = (bytes_of(big) / sizeof(double) + 31) & ~(size_t)31;
        const int grid = std::min((int)big_list.size(), 148 * 4);
        pe_variant_add(PE_VARIANT_EXT_GMEM_REUSE, (int64_t)big_list.size() - grid);
        double *work = nullptr;
        PE_TRY(D.alloc(stride * (size_t)grid, &work));
        PE_TRY(D.up(big_list.data(), big_list.size(), &list_d));
        k_extension_gmem<<<grid, LT, 0, st>>>(a, list_d, (int)big_list.size(), work, stride);
    }
    PE_LAUNCHED(ctx);
    PE_CUDA(cudaStreamSynchronize(st));
    const double t_kern = now_s();
    PE_CUDA(cudaMemcpyAsync(b->out, a.out, sizeof(double) * out_n, cudaMemcpyDeviceToHost, st));
    PE_CUDA(cudaMemcpyAsync(b->k_out, a.k_out, sizeof(int) * (size_t)nAE, cudaMemcpyDeviceToHost, st));
    std::vector<int> info(nAE);
    PE_CUDA(cudaMemcpyAsync(info.data(), a.info_out, sizeof(int) * (size_t)nAE, cudaMemcpyDeviceToHost, st));
    PE_CUDA(cudaStreamSynchronize(st));
    g_stage[0] += t_up - t_begin; g_stage[1] += t_kern - t_up; g_stage[2] += now_s() - t_kern;
    g_stage[4] += (double)(sizeof(double) * out_n); g_stage[5] += 1.0;
    for (int e = 0; e < nAE; ++e)
        PE_CHECK(info[e] == 0, "pe_batched_extension: singular local system on agglomerate " + std::to_string(e)
                                   + " (code " + std::to_string(info[e]) + "); a bad topology (e.g. a torus-shaped agglomerate) can cause this");
    return 0;
}
