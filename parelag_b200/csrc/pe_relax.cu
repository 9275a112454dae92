// pe_relax.cu -- K3/K4/K5: hypre-type relaxation as fused residual-update kernels.
//
//  * l1-Jacobi / Jacobi:  one pass over A computes v = w*(f - A u)/l1, a second
//    vector pass adds it (hypre_ParCSRRelax option 1).
//  * symmetric (l1-)Gauss-Seidel: hypre sweeps rows sequentially in natural order.
//    On the GPU the rows are split into SETS of mutually independent rows that are
//    processed set by set (forward), then in reverse (backward):
//      - PE_GS_ORDER_NATURAL: sets = levels of the dependency DAG of the natural
//        order, which reproduces hypre's result exactly (same operand values per row);
//      - PE_GS_ORDER_MULTICOLOR: sets = colours of a greedy first-fit colouring
//        (rows visited in natural order, smallest colour not used by a neighbour).
//    A set-ordered copy of the matrix (diag and offd merged per row) is kept in HBM so
//    every set streams a contiguous CSR range; x stays in the caller's numbering.
//  * Chebyshev: hypre_ParCSRRelax_Cheby with D^{-1/2} scaling, eigenvalue bounds from
//    10 CG steps (hypre_ParCSRMaxEigEstimateCG) started from hypre's LCG random vector.
#include "pe_core.cuh"
#include "pe_stream.cuh"
#include <algorithm>
#include <cmath>
#include <cstring>

struct pe_smoother {
    pe_ctx *ctx = nullptr;
    pe_mat *A = nullptr;      // borrowed
    int type = 2, sweeps = 1, cheby_order = 2, ordering = 0;
    double weight = 1.0, omega = 1.0, cheby_fraction = 0.3;
    double *l1_d = nullptr;
    double *v_d = nullptr, *w_d = nullptr, *z_d = nullptr, *r_d = nullptr; // scratch (n)
    // GS schedule
    int32_t nsets = 0;
    std::vector<int32_t> set_starts;   // nsets+1 (positions in permuted row order)
    std::vector<int32_t> order;        // permuted position -> row
    int32_t *perm_d = nullptr;         // same on device
    DevCSR P;                          // set-ordered merged copy; col >= ncols_diag => ghost
    uint8_t *before_d = nullptr;       // per entry: column visited earlier in forward pass
    int tpr = 8;
    std::vector<int> set_pI;           // P.I at the set boundaries (host copy, for profiling)
    std::vector<int> set_rb;           // first row block of each set (streaming kernel)
    int pI_at(int k) const { for (size_t c = 0; c < set_starts.size(); ++c) if (set_starts[c] == k) return set_pI[c]; return 0; }
    // colour-ordered SELL path (multicolour ordering with weight = omega = 1): rows AND columns
    // renumbered colour by colour, every colour padded to whole slices of 32 rows
    bool use_sell = false;
    DevSELL S;
    int32_t npad = 0;                   // padded length of the colour-ordered vectors
    std::vector<int32_t> slice_starts;  // nsets+1: first slice of every colour
    std::vector<int32_t> set_wmax;      // widest slice of every colour (selects the kernel's entry-group size)
    std::vector<double> set_bytes;      // algorithmic bytes of one colour launch
    uint64_t pol_gather = 0;            // L2 policy word of the u-gathers (PE_TUNE_GATHER_KEEP_PCT at creation)
    bool skip_turn = false;             // the backward pass may start at the second-to-last colour (see build_gs_schedule)
    int32_t *pos_d = nullptr;           // row -> colour-ordered position
    double *l1p_d = nullptr, *fp_d = nullptr, *up_d = nullptr;
    // fused sweep (PE_TUNE_FUSED_GS_MAX_MB): all colours of a symmetric sweep in one cooperative kernel
    bool fused = false;
    int fused_grid = 0, fused_nsteps = 0;
    int2 *fused_steps_d = nullptr;      // per step: row range of the set-ordered copy / slice range of the SELL copy
    unsigned *fused_bar_d = nullptr;    // {arrivals, generation}
    double fused_bytes = 0.0;           // algorithmic bytes of one fused sweep
    // Chebyshev
    double max_eig = 0, min_eig = 0;
    double coefs[5] = {0, 0, 0, 0, 0};
    double *ds_d = nullptr;
};

// ---------------------------------------------------------------------------
__global__ void k_l1_norms(int n, const int *__restrict__ dI, const int *__restrict__ dJ,
                           const double *__restrict__ dA, const int *__restrict__ oI,
                           const double *__restrict__ oA, int option, double *l1)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double diag = 0, off = 0, full = 0, lump = 0;
    for (int k = dI[i]; k < dI[i + 1]; ++k) {
        double a = dA[k];
        full += fabs(a); lump += a;
        if (dJ[k] == i) diag = a;
    }
    if (oI) for (int k = oI[i]; k < oI[i + 1]; ++k) { off += fabs(oA[k]); lump += oA[k]; }
    double d;
    if (option == 1) d = full + off;
    else if (option == 2) d = fabs(diag) + off;
    else if (option == 4) { d = fabs(diag) + off; if (d <= 4.0 / 3.0 * fabs(diag)) d = fabs(diag); }
    else if (option == 5) d = lump;
    else d = diag;
    if (option >= 1 && option <= 4 && diag < 0.0) d = -d;
    l1[i] = d;
}

// v = w * (f - A u) / l1   (TPR lanes per row; same streaming pattern as k_spmv)
template <int TPR>
__global__ void __launch_bounds__(256)
k_jacobi_update(int n, const int *__restrict__ dI, const int *__restrict__ dJ, const double *__restrict__ dA,
                const int *__restrict__ oI, const int *__restrict__ oJ, const double *__restrict__ oA,
                const double *__restrict__ u, const double *__restrict__ uext,
                const double *__restrict__ f, const double *__restrict__ l1, double w, double *v)
{
    const int lane = threadIdx.x & (TPR - 1);
    const int64_t gid = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / TPR;
    const int64_t ngroups = ((int64_t)gridDim.x * blockDim.x) / TPR;
    for (int64_t row = gid; row < n; row += ngroups) {
        double s = 0.0;
        for (int k = dI[row] + lane; k < dI[row + 1]; k += TPR) s += dA[k] * __ldg(u + dJ[k]);
        if (oI) for (int k = oI[row] + lane; k < oI[row + 1]; k += TPR) s += oA[k] * __ldg(uext + oJ[k]);
#pragma unroll
        for (int o = TPR / 2; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o, TPR);
        if (lane == 0) v[row] = w * (f[row] - s) / l1[row];
    }
}

// one GS set: rows [k0,k1) of the set-ordered matrix; in-place update of u.
template <int TPR, bool GENERAL>
__global__ void __launch_bounds__(256)
k_gs_set(int k0, int k1, const int *__restrict__ pI, const int *__restrict__ pJ,
         const double *__restrict__ pA, const int *__restrict__ perm, int ncd,
         const double *f, double *u, const double *uext,
         const double *__restrict__ l1, const uint8_t *__restrict__ before, int forward,
         const double *uold, double c1, double c2)
{
    // PDL: the row extent, the first (col,val) of every lane, the row's position and its l1 norm are
    // matrix data -- fetched while the preceding colour is still draining; f, u, uext, uold after the wait
    pdl_trigger();
    const int lane = threadIdx.x & (TPR - 1);
    const int gid = (blockIdx.x * blockDim.x + threadIdx.x) / TPR;
    const int k = k0 + gid;
    if (k >= k1) { pdl_wait(); return; }
    const int lo = ld_nc_s32_pro(pI + k), hi = ld_nc_s32_pro(pI + k + 1);
    const int i = ld_nc_s32_pro(perm + k);
    const double d = ld_nc_f64_pro(l1 + i);
    int q = lo + lane;
    int cn = 0; double an = 0.0;
    if (q < hi) { cn = ld_nc_s32_pro(pJ + q); an = ld_nc_f64_pro(pA + q); }
    if ((cn ^ __double2hiint(an) ^ __double2loint(an) ^ __double2hiint(d)) == 0x5bd1e995) pdl_trigger();   // pins the loads ahead of the wait
    pdl_wait();
    double fi = 0.0, ui = 0.0;
    if (lane == 0) { fi = f[i]; ui = u[i]; }     // issued with the gathers, not after the reduction
    double s = 0.0, s2 = 0.0;
    while (q < hi) {
        const int c = cn;
        const double a = an;
        const int qn = q + TPR;
        if (qn < hi) { cn = pJ[qn]; an = pA[qn]; }
        if (c < ncd) {
            double uc = u[c];
            s += a * uc;
            if (GENERAL) {
                bool vis = forward ? (before[q] != 0) : (before[q] == 0 && c != i);
                if (vis) s2 += a * (uold[c] - uc);
            }
        } else {
            s += a * uext[c - ncd];
        }
        q = qn;
    }
#pragma unroll
    for (int o = TPR / 2; o > 0; o >>= 1) {
        s += __shfl_down_sync(0xffffffffu, s, o, TPR);
        if (GENERAL) s2 += __shfl_down_sync(0xffffffffu, s2, o, TPR);
    }
    if (lane == 0) {
        if (d != 0.0) {
            if (GENERAL) u[i] = ui + (c1 * (fi - s) + c2 * s2) / d;
            else u[i] = ui + (fi - s) / d;
        }
    }
}

// ---------------------------------------------------------------------------
// Fused symmetric sweep: every colour of the forward and of the backward pass in ONE persistent kernel with a grid-wide
// barrier between colours.  On the coarse levels a colour is a few hundred to a few thousand rows: a launch per colour
// costs 3-10x the colour's work.  The rows a step touches, their lanes and the summation order are those of the
// per-colour kernels (k_gs_set<TPR, false>, k_sell_gs), so the result is bit-identical.  u is read and written past the
// (non-coherent) L1 (ld/st.global.cg); a colour's updates are published by __threadfence + the barrier's release.
// Launched cooperatively (all CTAs resident); grid <= SMs x occupancy.
// ---------------------------------------------------------------------------
__device__ __forceinline__ unsigned ld_acquire_gpu_u32(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu_u32(unsigned *p, unsigned v)
{
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// bar[0] = arrivals of the current barrier, bar[1] = generation; reusable across launches (graph replays)
__device__ __forceinline__ void grid_barrier(unsigned *bar)
{
    __syncthreads();
    if (threadIdx.x == 0)
    {
        __threadfence();
        const unsigned gen = ld_acquire_gpu_u32(bar + 1);
        if (atomicAdd(bar, 1u) == gridDim.x - 1) { atomicExch(bar, 0u); __threadfence(); st_release_gpu_u32(bar + 1, gen + 1); }
        else while (ld_acquire_gpu_u32(bar + 1) == gen) { }
    }
    __syncthreads();
}

template <int TPR>
__global__ void __launch_bounds__(256)
k_gs_sweep(int nsteps, const int2 *__restrict__ steps, const int *__restrict__ pI, const int *__restrict__ pJ,
           const double *__restrict__ pA, const int *__restrict__ perm, int ncd,
           const double *f, double *u, const double *uext, const double *__restrict__ l1, unsigned *bar)
{
    pdl_wait();
    const int lane = threadIdx.x & (TPR - 1);
    const int g0 = (blockIdx.x * blockDim.x + threadIdx.x) / TPR, gstride = (gridDim.x * blockDim.x) / TPR;
    for (int t = 0; t < nsteps; ++t)
    {
        const int2 st = steps[t];
        // the trip count is uniform over the CTA (kb does not depend on the thread): the full-mask shuffles below are
        // executed by every lane, rows past the end of the colour are predicated off
        for (int kb = st.x; kb < st.y; kb += gstride)
        {
            const int k = kb + g0;
            const bool on = k < st.y;
            int lo = 0, hi = 0, i = 0;
            double d = 0.0, fi = 0.0, ui = 0.0;
            if (on) { lo = pI[k]; hi = pI[k + 1]; i = perm[k]; d = l1[i]; if (lane == 0) { fi = f[i]; ui = __ldcg(u + i); } }
            double s = 0.0;
            for (int q = lo + lane; q < hi; q += TPR)
            {
                const int c = pJ[q];
                const double a = pA[q];
                s += a * (c < ncd ? __ldcg(u + c) : uext[c - ncd]);
            }
#pragma unroll
            for (int o = TPR / 2; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o, TPR);
            if (on && lane == 0 && d != 0.0) __stcg(u + i, ui + (fi - s) / d);
        }
        if (t + 1 < nsteps) grid_barrier(bar);
    }
}

// SELL variant: vectors in colour order; steps[0] and the last step are the renumbering passes
// (x.y < 0: renumber in, x.y == -2: renumber out), the others slice ranges [x, y) of one colour
__global__ void __launch_bounds__(256)
k_sell_gs_sweep(int nsteps, const int2 *__restrict__ steps, const int *__restrict__ soff, const int *__restrict__ J,
                const double *__restrict__ A, int ext_base, int n, const int *__restrict__ pos, const double *b,
                double *x, int zero_guess, double *f, double *u, const double *uext, const double *__restrict__ l1, unsigned *bar)
{
    pdl_wait();
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nthr = gridDim.x * blockDim.x;
    const int lane = threadIdx.x & 31, w0 = tid >> 5, nw = nthr >> 5;
    for (int t = 0; t < nsteps; ++t)
    {
        const int2 st = steps[t];
        if (st.y == -1)
            for (int i = tid; i < n; i += nthr) { const int p = pos[i]; __stcg(f + p, b[i]); __stcg(u + p, zero_guess ? 0.0 : x[i]); }
        else if (st.y == -2)
            for (int i = tid; i < n; i += nthr) x[i] = __ldcg(u + pos[i]);
        else
            for (int sl = st.x + w0; sl < st.y; sl += nw)
            {
                const int o0 = soff[sl], w = soff[sl + 1] - o0;
                const int *j = J + (int64_t)o0 * 32 + lane;
                const double *a = A + (int64_t)o0 * 32 + lane;
                const int row = sl * 32 + lane;
                const double d = l1[row], fr = __ldcg(f + row), ur = __ldcg(u + row);
                double acc = 0.0;
                for (int q = 0; q < w; q += 4)
                {
                    int c[4]; double v[4], uv[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) if (q + k < w) { c[k] = j[(q + k) * 32]; v[k] = a[(q + k) * 32]; }
#pragma unroll
                    for (int k = 0; k < 4; ++k) if (q + k < w) uv[k] = (uext && c[k] >= ext_base) ? uext[c[k] - ext_base] : __ldcg(u + c[k]);
#pragma unroll
                    for (int k = 0; k < 4; ++k) if (q + k < w) acc = __fma_rn(v[k], uv[k], acc);
                }
                if (d != 0.0) __stcg(u + row, ur + (fr - acc) / d);
            }
        if (t + 1 < nsteps) grid_barrier(bar);
    }
}

// Streaming variant of one GS set (same structure as k_spmv_stream): CTA b owns rows
// [rb[b], rb[b+1]) of the set-ordered matrix; row blocks never straddle a set boundary.
__global__ void __launch_bounds__(256)
k_gs_set_stream(int b0, const int *__restrict__ rb, const int *__restrict__ pI, const int *__restrict__ pJ,
                const double *__restrict__ pA, const int *__restrict__ perm, int ncd,
                const double *__restrict__ f, double *u, const double *__restrict__ uext,
                const double *__restrict__ l1)
{
    __shared__ double prod[PE_STREAM_CAP];
    const int tid = threadIdx.x;
    const int r0 = rb[b0 + blockIdx.x], r1 = rb[b0 + blockIdx.x + 1];
    const int k0 = pI[r0], k1 = pI[r1];
    for (int base = k0; base < k1; base += 256 * 8)
    {
        int c[8]; double a[8];
#pragma unroll
        for (int q = 0; q < 8; ++q)
        {
            const int k = base + q * 256 + tid;
            c[q] = k < k1 ? pJ[k] : -1;
            a[q] = k < k1 ? pA[k] : 0.0;
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) if (c[q] >= 0) a[q] *= (c[q] < ncd ? u[c[q]] : uext[c[q] - ncd]);
#pragma unroll
        for (int q = 0; q < 8; ++q) { const int k = base + q * 256 + tid; if (k < k1) prod[k - k0] = a[q]; }
    }
    __syncthreads();
    for (int r = r0 + tid; r < r1; r += 256)
    {
        const int lo = pI[r] - k0, hi = pI[r + 1] - k0;
        double s = 0.0;
        for (int q = lo; q < hi; ++q) s += prod[q];
        const int i = perm[r];
        const double d = l1[i];
        if (d != 0.0) u[i] += (f[i] - s) / d;
    }
}

// build the set-ordered merged matrix
__global__ void k_perm_rowlen(int n, const int *__restrict__ perm, const int *__restrict__ dI,
                              const int *__restrict__ oI, int *len)
{
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    int i = perm[k];
    int l = dI[i + 1] - dI[i];
    if (oI) l += oI[i + 1] - oI[i];
    len[k + 1] = l;
    if (k == 0) len[0] = 0;
}
__global__ void k_perm_fill(int n, const int *__restrict__ perm, const int *__restrict__ pos,
                            const int *__restrict__ dI, const int *__restrict__ dJ, const double *__restrict__ dA,
                            const int *__restrict__ oI, const int *__restrict__ oJ, const double *__restrict__ oA,
                            int ncd, const int *__restrict__ pI, int *pJ, double *pA, uint8_t *before)
{
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    int i = perm[k];
    int q = pI[k];
    for (int t = dI[i]; t < dI[i + 1]; ++t, ++q) {
        pJ[q] = dJ[t]; pA[q] = dA[t];
        if (before) before[q] = pos[dJ[t]] < k ? 1 : 0;
    }
    if (oI) for (int t = oI[i]; t < oI[i + 1]; ++t, ++q) {
        pJ[q] = ncd + oJ[t]; pA[q] = oA[t];
        if (before) before[q] = 0;
    }
}

// host: schedule construction -------------------------------------------------
static void build_levels(int n, const int *I, const int *J, std::vector<int> &level, int &nlev)
{
    // level(i) = 1 + max level(j), j < i coupled to i  (forward natural-order DAG)
    level.assign(n, 0);
    nlev = 0;
    for (int i = 0; i < n; ++i) {
        int l = 0;
        for (int k = I[i]; k < I[i + 1]; ++k) { int j = J[k]; if (j < i && level[j] + 1 > l) l = level[j] + 1; }
        level[i] = l;
        if (l + 1 > nlev) nlev = l + 1;
    }
}
static void build_colors(int n, const int *I, const int *J, std::vector<int> &color, int &ncol)
{
    // greedy first fit in natural order over the (structurally symmetrised by
    // assumption) diag pattern
    color.assign(n, -1);
    ncol = 0;
    std::vector<int> mark;
    for (int i = 0; i < n; ++i) {
        if ((int)mark.size() < ncol + 1) mark.resize(ncol + 1, -1);
        for (int k = I[i]; k < I[i + 1]; ++k) { int j = J[k]; if (j != i && color[j] >= 0) mark[color[j]] = i; }
        int c = 0;
        while (c < ncol && mark[c] == i) ++c;
        color[i] = c;
        if (c == ncol) { ++ncol; }
    }
}

// PE_TUNE_GS_SLABS: slab index of every row = quantile of its breadth-first level in the matrix graph (start: row 0;
// rows the search does not reach -- eliminated boundary rows are isolated -- continue the level count)
static void build_slabs(int n, const int *I, const int *J, int nslabs, std::vector<int> &slab)
{
    std::vector<int> level(n, -1), frontier, next;
    std::vector<int64_t> count;
    int lev = 0, seed = 0;
    int64_t visited = 0;
    while (visited < n)
    {
        while (seed < n && level[seed] >= 0) ++seed;
        frontier.assign(1, seed);
        level[seed] = lev;
        while (!frontier.empty())
        {
            count.push_back((int64_t)frontier.size());
            visited += (int64_t)frontier.size();
            next.clear();
            for (int i : frontier)
                for (int k = I[i]; k < I[i + 1]; ++k)
                {
                    const int j = J[k];
                    if (j < n && level[j] < 0) { level[j] = lev + 1; next.push_back(j); }
                }
            frontier.swap(next);
            ++lev;
        }
    }
    std::vector<int> slab_of_level(count.size());
    int64_t before = 0;
    for (size_t l = 0; l < count.size(); ++l)
    {
        slab_of_level[l] = (int)std::min<int64_t>(nslabs - 1, before * nslabs / std::max(n, 1));
        before += count[l];
    }
    slab.resize(n);
    for (int i = 0; i < n; ++i) slab[i] = slab_of_level[level[i]];
}

#include <cub/cub.cuh>

static int fused_setup(pe_smoother *s);
static int build_gs_schedule(pe_smoother *s)
{
    pe_ctx *ctx = s->ctx;
    pe_mat *A = s->A;
    int n = A->diag.nrows;
    std::vector<int> I(n + 1), J((size_t)A->diag.nnz);
    PE_CUDA(cudaMemcpyAsync(I.data(), A->diag.I, sizeof(int) * (size_t)(n + 1), cudaMemcpyDeviceToHost, ctx->stream));
    if (A->diag.nnz) PE_CUDA(cudaMemcpyAsync(J.data(), A->diag.J, sizeof(int) * (size_t)A->diag.nnz, cudaMemcpyDeviceToHost, ctx->stream));
    PE_CUDA(cudaStreamSynchronize(ctx->stream));
    std::vector<int> key;
    int nsets = 0;
    if (s->ordering == PE_GS_ORDER_NATURAL) {
        build_levels(n, I.data(), J.data(), key, nsets);
        // the backward pass replays the sets in reverse; that is a valid schedule of the
        // reverse sweep iff the pattern is structurally symmetric.  Verify.
        std::vector<int> pos_in_row;
        for (int i = 0; i < n; ++i)
            for (int k = I[i]; k < I[i + 1]; ++k) {
                int j = J[k];
                if (j > i && key[j] <= key[i]) {
                    // dependency j>i (backward) not ordered by levels: need symmetric pattern
                    bool found = false;
                    for (int t = I[j]; t < I[j + 1]; ++t) if (J[t] == i) { found = true; break; }
                    PE_CHECK(found, "natural-order GS needs a structurally symmetric matrix");
                }
            }
    } else {
        build_colors(n, I.data(), J.data(), key, nsets);
        const int nslabs = pe_get_tuning(PE_TUNE_GS_SLABS);
        if (nslabs > 1 && n >= 4000000 && nsets >= 2)
        {
            // slab-major order: set = slab * colours + colour (rows of one set are still mutually independent)
            std::vector<int> slab;
            build_slabs(n, I.data(), J.data(), nslabs, slab);
            for (int i = 0; i < n; ++i) key[i] += slab[i] * nsets;
            nsets *= nslabs;
        }
    }
    // stable counting sort of rows by set id
    s->nsets = nsets;
    s->set_starts.assign(nsets + 1, 0);
    for (int i = 0; i < n; ++i) s->set_starts[key[i] + 1]++;
    for (int c = 0; c < nsets; ++c) s->set_starts[c + 1] += s->set_starts[c];
    s->order.resize(n);
    std::vector<int> next(s->set_starts.begin(), s->set_starts.end() - 1), pos(n);
    for (int i = 0; i < n; ++i) { int p = next[key[i]]++; s->order[p] = i; pos[i] = p; }

    // The forward pass ends and the backward pass starts with the LAST set.  Its rows are mutually
    // independent, so right after the forward update row i has residual f_i - sum_j a_ij u_j =
    // (1 - a_ii / d_i) r_i, which is exactly 0 when d_i == a_ii: the repeated update adds only the
    // rounding error of that zero.  When every row of the last set has d_i == a_ii (no ghost entries,
    // l1 == diagonal) the second visit is skipped -- 1/nsets of the matrix traffic of a sweep.
    if (nsets >= 2 && s->type == 2 && s->ordering == PE_GS_ORDER_MULTICOLOR && s->weight == 1.0 && s->omega == 1.0)
    {
        std::vector<double> l1h(n), Ah((size_t)A->diag.nnz);
        std::vector<int> oIt;
        PE_CUDA(cudaMemcpy(l1h.data(), s->l1_d, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost));
        if (A->diag.nnz) PE_CUDA(cudaMemcpy(Ah.data(), A->diag.A, sizeof(double) * (size_t)A->diag.nnz, cudaMemcpyDeviceToHost));
        if (A->offd.nnz > 0) { oIt.resize(n + 1); PE_CUDA(cudaMemcpy(oIt.data(), A->offd.I, sizeof(int) * (size_t)(n + 1), cudaMemcpyDeviceToHost)); }
        bool ok = true;
        for (int k = s->set_starts[nsets - 1]; k < s->set_starts[nsets] && ok; ++k)
        {
            const int i = s->order[k];
            double aii = 0.0;
            for (int q = I[i]; q < I[i + 1]; ++q) if (J[q] == i) aii = Ah[q];
            ok = aii > 0.0 && l1h[i] == aii && (oIt.empty() || oIt[i + 1] == oIt[i]);
        }
        s->skip_turn = ok;
    }

    bool general = !(s->weight == 1.0 && s->omega == 1.0);
    // Colour-ordered SELL streaming (thread per row) for bandwidth-bound levels; below
    // PE_TUNE_SELL_MIN_ROWS rows a colour is a few thousand rows and latency-bound, where the
    // lanes-per-row CSR kernel (k_gs_set<TPR>: one coalesced load of the row, shuffle reduction, no
    // renumbering passes) has the shorter dependent chain.
    // A second condition on the rows PER COLOUR: irregular coarse operators (the NullSpace dofs of the deformed configs[4]
    // mesh: 25-50 entries per row) need 40-50 colours, so a 430 k-row level has < 10 k rows per colour -- one thread per
    // row leaves the GPU empty there, while the lanes-per-row kernel has 32 lanes per row in flight.  Measured on one
    // box of configs[4] (144^3, profiles/README.md round 2): V-cycle 17.3 ms with the row rule alone, 15.1 ms when the
    // 430 k-row level (9.5 k rows per colour) takes the CSR kernel, 17.0 ms when the 2.6 M-row level (65 k rows per
    // colour) takes it as well.  The row threshold 0 (tests) forces the SELL path.
    const int sell_min = pe_get_tuning(PE_TUNE_SELL_MIN_ROWS);
    const bool enough_per_colour = sell_min <= 0 || (int64_t)n >= (int64_t)nsets * 32768;
    if (s->ordering == PE_GS_ORDER_MULTICOLOR && !general && n >= sell_min && enough_per_colour)
    {
        // colour-ordered, slice-padded numbering
        s->slice_starts.assign(nsets + 1, 0);
        for (int c = 0; c < nsets; ++c)
            s->slice_starts[c + 1] = s->slice_starts[c] + (s->set_starts[c + 1] - s->set_starts[c] + 31) / 32;
        const int nslices = s->slice_starts[nsets];
        s->npad = nslices * 32;
        std::vector<int32_t> rowmap((size_t)s->npad, -1), ppos(n);
        std::vector<int> oIh;
        if (A->offd.nnz > 0)
        {
            oIh.resize(n + 1);
            PE_CUDA(cudaMemcpy(oIh.data(), A->offd.I, sizeof(int) * (size_t)(n + 1), cudaMemcpyDeviceToHost));
        }
        s->set_bytes.assign(nsets, 0.0);
        for (int c = 0; c < nsets; ++c)
        {
            double nnz_c = 0;
            for (int k = s->set_starts[c]; k < s->set_starts[c + 1]; ++k)
            {
                const int i = s->order[k], p = s->slice_starts[c] * 32 + (k - s->set_starts[c]);
                rowmap[p] = i; ppos[i] = p;
                nnz_c += I[i + 1] - I[i];
                if (!oIh.empty()) nnz_c += oIh[i + 1] - oIh[i];
            }
            const double rows = s->set_starts[c + 1] - s->set_starts[c];
            s->set_bytes[c] = 12.0 * nnz_c + 4.0 * rows + 32.0 * rows;
        }
        int32_t *rowmap_d = nullptr;
        const size_t np = (size_t)(s->npad > 0 ? s->npad : 1);
        PE_CUDA(cudaMalloc(&rowmap_d, sizeof(int32_t) * np));
        PE_CUDA(cudaMalloc(&s->pos_d, sizeof(int32_t) * (size_t)(n > 0 ? n : 1)));
        PE_CUDA(cudaMalloc(&s->l1p_d, sizeof(double) * np));
        PE_CUDA(cudaMalloc(&s->fp_d, sizeof(double) * np));
        PE_CUDA(cudaMalloc(&s->up_d, sizeof(double) * np));
        PE_CUDA(cudaMemcpyAsync(rowmap_d, rowmap.data(), sizeof(int32_t) * (size_t)s->npad, cudaMemcpyHostToDevice, ctx->stream));
        PE_CUDA(cudaMemcpyAsync(s->pos_d, ppos.data(), sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
        PE_CUDA(cudaMemsetAsync(s->l1p_d, 0, sizeof(double) * np, ctx->stream));
        PE_CUDA(cudaMemsetAsync(s->fp_d, 0, sizeof(double) * np, ctx->stream));
        PE_CUDA(cudaMemsetAsync(s->up_d, 0, sizeof(double) * np, ctx->stream));
        std::vector<int32_t> soff_h;
        PE_TRY(pe_sell_build(ctx, A->diag, &A->offd, rowmap_d, nslices, s->pos_d, s->npad, s->S, &soff_h));
        s->set_wmax.assign(nsets, 0);
        for (int c = 0; c < nsets; ++c)
            for (int k = s->slice_starts[c]; k < s->slice_starts[c + 1]; ++k)
                s->set_wmax[c] = std::max(s->set_wmax[c], soff_h[k + 1] - soff_h[k]);

        // l1 in colour order (padded rows keep 0 => never updated)
        PE_TRY(pe_launch_perm_in(ctx, n, s->pos_d, s->l1_d, nullptr, s->l1p_d, s->up_d));
        PE_CUDA(cudaStreamSynchronize(ctx->stream));
        cudaFree(rowmap_d);
        PE_TRY(pe_make_gather_policy(ctx, pe_get_tuning(PE_TUNE_GATHER_KEEP_PCT), &s->pol_gather));
        s->use_sell = true;
        return 0;
    }
    int *pos_d = nullptr, *len_d = nullptr;
    PE_CUDA(cudaMalloc(&s->perm_d, sizeof(int) * (size_t)(n > 0 ? n : 1)));
    PE_CUDA(cudaMalloc(&pos_d, sizeof(int) * (size_t)(n > 0 ? n : 1)));
    PE_CUDA(cudaMemcpyAsync(s->perm_d, s->order.data(), sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    PE_CUDA(cudaMemcpyAsync(pos_d, pos.data(), sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    int64_t nnz = A->diag.nnz + A->offd.nnz;
    PE_TRY(devcsr_alloc(s->P, n, A->diag.ncols + A->offd.ncols, nnz));
    if (general) PE_CUDA(cudaMalloc(&s->before_d, (size_t)(nnz > 0 ? nnz : 1)));
    const int *oI = A->offd.nnz > 0 ? A->offd.I : nullptr;
    len_d = s->P.I;
    if (n > 0) {
        k_perm_rowlen<<<pe_grid_for(n, 256), 256, 0, ctx->stream>>>(n, s->perm_d, A->diag.I, oI, len_d);
        PE_LAUNCHED(ctx);
        void *tmp = nullptr; size_t tb = 0;
        cub::DeviceScan::InclusiveSum(nullptr, tb, len_d, len_d, n + 1, ctx->stream);
        PE_CUDA(cudaMalloc(&tmp, tb));
        PE_CUDA(cub::DeviceScan::InclusiveSum(tmp, tb, len_d, len_d, n + 1, ctx->stream));
        ctx->launches++;
        k_perm_fill<<<pe_grid_for(n, 256), 256, 0, ctx->stream>>>(n, s->perm_d, pos_d, A->diag.I, A->diag.J, A->diag.A,
                                                                 oI, A->offd.J, A->offd.A, A->diag.ncols,
                                                                 s->P.I, s->P.J, s->P.A, s->before_d);
        PE_LAUNCHED(ctx);
        PE_CUDA(cudaStreamSynchronize(ctx->stream));
        cudaFree(tmp);
    } else {
        PE_CUDA(cudaMemsetAsync(s->P.I, 0, sizeof(int), ctx->stream));
    }
    cudaFree(pos_d);
    s->tpr = pe_choose_tpr(nnz, n);
    {
        std::vector<int32_t> breaks(s->set_starts.begin(), s->set_starts.end());
        PE_TRY(pe_build_row_blocks(ctx, s->P, &breaks));
        // first row block of every set
        s->set_rb.assign(s->set_starts.size(), 0);
        if (s->P.nrb > 0)
        {
            std::vector<int32_t> rb(s->P.nrb + 1);
            PE_CUDA(cudaMemcpy(rb.data(), s->P.rb, sizeof(int32_t) * rb.size(), cudaMemcpyDeviceToHost));
            size_t c = 0;
            for (int b = 0; b <= s->P.nrb; ++b)
                while (c < s->set_starts.size() && s->set_starts[c] == rb[b]) s->set_rb[c++] = b;
            for (; c < s->set_starts.size(); ++c) s->set_rb[c] = s->P.nrb;
        }
    }
    s->set_pI.resize(s->set_starts.size());
    for (size_t c = 0; c < s->set_starts.size(); ++c)
        PE_CUDA(cudaMemcpy(&s->set_pI[c], s->P.I + s->set_starts[c], sizeof(int), cudaMemcpyDeviceToHost));
    return 0;
}

// hypre's Park-Miller LCG (utilities/random.c), as in hypre_SeqVectorSetRandomValues
static void hypre_rand_vector(int n, int seed, std::vector<double> &v)
{
    const int a = 16807, m = 2147483647, q = 127773, r = 2836;
    int s = seed;
    v.resize(n);
    for (int i = 0; i < n; ++i) {
        int low = s % q, high = s / q;
        int test = a * low - r * high;
        s = test > 0 ? test : test + m;
        v[i] = 2.0 * ((double)s / m) - 1.0;
    }
}

// eigenvalues of a symmetric tridiagonal matrix (implicit QL, as EISPACK tql1)
static void tridiag_eigs(int n, std::vector<double> d, std::vector<double> e, double &lmin, double &lmax)
{
    // e[1..n-1] subdiagonal; shift to e[0..n-2]
    for (int i = 1; i < n; ++i) e[i - 1] = e[i];
    e[n - 1] = 0.0;
    for (int l = 0; l < n; ++l) {
        int iter = 0, m;
        do {
            for (m = l; m < n - 1; ++m) {
                double dd = fabs(d[m]) + fabs(d[m + 1]);
                if (fabs(e[m]) <= 2.220446049250313e-16 * dd) break;
            }
            if (m != l) {
                if (iter++ == 60) break;
                double g = (d[l + 1] - d[l]) / (2.0 * e[l]);
                double r = hypot(g, 1.0);
                g = d[m] - d[l] + e[l] / (g + (g >= 0 ? fabs(r) : -fabs(r)));
                double s = 1.0, c = 1.0, p = 0.0;
                int i;
                for (i = m - 1; i >= l; --i) {
                    double f = s * e[i], b = c * e[i];
                    e[i + 1] = (r = hypot(f, g));
                    if (r == 0.0) { d[i + 1] -= p; e[m] = 0.0; break; }
                    s = f / r; c = g / r;
                    g = d[i + 1] - p;
                    r = (d[i] - g) * s + 2.0 * c * b;
                    d[i + 1] = g + (p = s * r);
                    g = c * r - b;
                }
                if (r == 0.0 && i >= l) continue;
                d[l] -= p; e[l] = g; e[m] = 0.0;
            }
        } while (m != l);
    }
    lmin = *std::min_element(d.begin(), d.begin() + n);
    lmax = *std::max_element(d.begin(), d.begin() + n);
}

__global__ void k_inv_sqrt_diag(int n, const int *__restrict__ I, const int *__restrict__ J,
                                const double *__restrict__ A, double *ds)
{
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    double v = 0.0;
    for (int k = I[r]; k < I[r + 1]; ++k) if (J[k] == r) { v = A[k]; break; }
    ds[r] = 1.0 / sqrt(v);
}
__global__ void k_vmul3(int64_t n, const double *__restrict__ a, const double *__restrict__ b, double *c)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) c[i] = a[i] * b[i];
}
// u = coef * r + ds .* v
__global__ void k_cheb_step(int64_t n, double coef, const double *__restrict__ r, const double *__restrict__ ds,
                            const double *__restrict__ v, double *u)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) u[i] = coef * r[i] + ds[i] * v[i];
}
// r = ds .* r ; uo = u ; u = r * coef
__global__ void k_cheb_begin(int64_t n, double coef, const double *__restrict__ ds, double *r, double *uo, double *u)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) { double t = r[i] * ds[i]; r[i] = t; uo[i] = u[i]; u[i] = t * coef; }
}
// u = uo + ds .* u
__global__ void k_cheb_end(int64_t n, const double *__restrict__ ds, const double *__restrict__ uo, double *u)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) u[i] = uo[i] + ds[i] * u[i];
}

static int spmv_full(pe_ctx *ctx, pe_mat *A, double alpha, const double *x, double beta, const double *yin, double *yout)
{
    if (A->offd.nnz > 0) {
        PE_TRY(pe_halo_exchange(A, x));
        PE_TRY(pe_launch_spmv(ctx, A->diag, nullptr, A->tpr, alpha, x, nullptr, beta, yin, yout));
        PE_TRY(pe_halo_wait(A));
        return pe_launch_spmv(ctx, A->offd, nullptr, pe_choose_tpr(A->offd.nnz, A->offd.nrows), alpha, A->x_ext_d, nullptr, 1.0, yout, yout);
    }
    if (ctx->nranks > 1) { PE_TRY(pe_halo_exchange(A, x)); PE_TRY(pe_halo_wait(A)); }
    return pe_launch_spmv(ctx, A->diag, nullptr, A->tpr, alpha, x, nullptr, beta, yin, yout);
}

static int dot_dev(pe_ctx *ctx, int64_t n, const double *x, const double *y, double *out)
{
    pe_vec vx{ctx, n, const_cast<double *>(x)}, vy{ctx, n, const_cast<double *>(y)};
    return pe_vec_dot(&vx, &vy, out);
}

static int cheby_setup(pe_smoother *s)
{
    pe_ctx *ctx = s->ctx;
    pe_mat *A = s->A;
    int n = A->diag.nrows;
    cudaStream_t st = ctx->stream;
    PE_CUDA(cudaMalloc(&s->ds_d, sizeof(double) * (size_t)(n > 0 ? n : 1)));
    k_inv_sqrt_diag<<<pe_grid_for(n, 256), 256, 0, st>>>(n, A->diag.I, A->diag.J, A->diag.A, s->ds_d);
    PE_LAUNCHED(ctx);
    // hypre_ParCSRMaxEigEstimateCG(A, scale=1, max_iter=10)
    int max_iter = 10;
    if (A->global_num_rows < max_iter) max_iter = (int)A->global_num_rows;
    std::vector<double> rnd;
    hypre_rand_vector(n, 1 * (ctx->rank + 1), rnd);
    double *r = s->r_d, *p = s->v_d, *sv = s->w_d, *u = s->z_d;
    PE_CUDA(cudaMemcpyAsync(r, rnd.data(), sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st));
    std::vector<double> tridiag(max_iter + 1, 0.0), trioffd(max_iter + 1, 0.0);
    double gamma = 0, gamma_old, beta, sdotp, alpha;
    PE_TRY(dot_dev(ctx, n, r, r, &gamma));
    for (int i = 0; i < max_iter; ++i) {
        gamma_old = gamma;
        PE_TRY(dot_dev(ctx, n, r, r, &gamma));
        // stop once the residual vanishes (the start vector spans fewer than max_iter eigenvectors, as on
        // a small coarse level); the Lanczos matrix of the steps taken holds the estimate.  Going on divides 0 by 0.
        if (i > 0 && gamma < 2.220446049250313e-16) { max_iter = i; break; }
        pe_vec vr{ctx, n, r}, vp{ctx, n, p}, vs{ctx, n, sv};
        if (i == 0) { beta = 1.0; PE_TRY(pe_vec_copy(&vr, &vp)); }
        else { beta = gamma / gamma_old; PE_TRY(pe_vec_axpby(1.0, &vr, beta, &vp)); }
        k_vmul3<<<pe_grid_for(n, 256), 256, 0, st>>>(n, s->ds_d, p, u); PE_LAUNCHED(ctx);
        PE_TRY(spmv_full(ctx, A, 1.0, u, 0.0, sv, sv));
        pe_vec vds{ctx, n, s->ds_d};
        PE_TRY(pe_vec_mul(&vds, &vs));
        PE_TRY(dot_dev(ctx, n, sv, p, &sdotp));
        alpha = gamma / sdotp;
        double alphainv = 1.0 / alpha;
        tridiag[i + 1] = alphainv;
        tridiag[i] *= beta;
        tridiag[i] += alphainv;
        trioffd[i + 1] = alphainv;
        trioffd[i] *= sqrt(beta);
        PE_TRY(pe_vec_axpby(-alpha, &vs, 1.0, &vr));
    }
    tridiag_eigs(max_iter, tridiag, trioffd, s->min_eig, s->max_eig);
    // coefficients (hypre par_cheby.c)
    int order = s->cheby_order;
    if (order > 4) order = 4;
    if (order < 1) order = 1;
    s->cheby_order = order;
    int co = order - 1;
    double upper = s->max_eig * 1.1;
    double lower = (upper - s->min_eig) * s->cheby_fraction + s->min_eig;
    double theta = (upper + lower) / 2, delta = (upper - lower) / 2, den;
    double *c = s->coefs;
    switch (co) {
    case 0: c[0] = 1.0 / theta; break;
    case 1: den = theta * theta + delta * theta; c[0] = (delta + 2 * theta) / den; c[1] = -1.0 / den; break;
    case 2:
        den = 2 * delta * theta * theta - delta * delta * theta - pow(delta, 3) + 2 * pow(theta, 3);
        c[0] = (4 * delta * theta - pow(delta, 2) + 6 * pow(theta, 2)) / den;
        c[1] = -(2 * delta + 6 * theta) / den; c[2] = 2 / den; break;
    case 3:
        den = -(4 * delta * pow(theta, 3) - 3 * pow(delta, 2) * pow(theta, 2) - 3 * pow(delta, 3) * theta + 4 * pow(theta, 4));
        c[0] = (6 * pow(delta, 2) * theta - 12 * delta * pow(theta, 2) + 3 * pow(delta, 3) - 16 * pow(theta, 3)) / den;
        c[1] = (12 * delta * theta - 3 * pow(delta, 2) + 24 * pow(theta, 2)) / den;
        c[2] = -(4 * delta + 16 * theta) / den; c[3] = 4 / den; break;
    }
    return 0;
}

// ---------------------------------------------------------------------------
extern "C" int pe_smoother_create(pe_ctx *ctx, pe_mat *A, int type, int sweeps, double damping,
                                  double omega, int cheby_order, double cheby_fraction,
                                  int gs_ordering, pe_smoother **out)
{
    PE_CHECK(ctx && A && out, "bad arguments");
    PE_CHECK(A->diag.nrows == A->diag.ncols, "smoother needs a square matrix");
    PE_CHECK(type == 0 || type == 1 || type == 2 || type == 4 || type == 5 || type == 6 || type == 16,
             "unsupported hypre relaxation type (supported: 0,1,2,4,5,6,16)");
    pe_smoother *s = new pe_smoother();
    s->ctx = ctx; s->A = A; s->type = type; s->sweeps = sweeps; s->weight = damping; s->omega = omega;
    s->cheby_order = cheby_order; s->cheby_fraction = cheby_fraction; s->ordering = gs_ordering;
    int n = A->diag.nrows;
    size_t nb = sizeof(double) * (size_t)(n > 0 ? n : 1);
    PE_CUDA(cudaMalloc(&s->l1_d, nb));
    PE_CUDA(cudaMalloc(&s->v_d, nb));
    // type 6 (hybrid symmetric Gauss-Seidel, hypre_BoomerAMGRelax): the update of types 2/4 with the diagonal entry in
    // the place of the l1 norm, relaxation weight and omega included (c1 = omega w, c2 = omega (1 - w) on a saved copy)
    int l1opt = (type == 0 || type == 6 || type == 16) ? 0 : type;
    const int *oI = A->offd.nnz > 0 ? A->offd.I : nullptr;
    k_l1_norms<<<pe_grid_for(n, 256), 256, 0, ctx->stream>>>(n, A->diag.I, A->diag.J, A->diag.A, oI, A->offd.A, l1opt, s->l1_d);
    PE_LAUNCHED(ctx);
    if (type == 2 || type == 4 || type == 6) {
        if (!(damping == 1.0 && omega == 1.0)) PE_CUDA(cudaMalloc(&s->w_d, nb));
        PE_TRY(build_gs_schedule(s));
        PE_TRY(fused_setup(s));
    } else if (type == 16) {
        PE_CUDA(cudaMalloc(&s->w_d, nb));
        PE_CUDA(cudaMalloc(&s->z_d, nb));
        PE_CUDA(cudaMalloc(&s->r_d, nb));
        PE_TRY(cheby_setup(s));
    }
    PE_CUDA(cudaStreamSynchronize(ctx->stream));
    *out = s;
    return 0;
}

extern "C" int pe_smoother_free(pe_smoother *s)
{
    if (!s) return 0;
    cudaStreamSynchronize(s->ctx->stream);
    cudaFree(s->l1_d); cudaFree(s->v_d);
    if (s->w_d) cudaFree(s->w_d);
    if (s->z_d) cudaFree(s->z_d);
    if (s->r_d) cudaFree(s->r_d);
    if (s->ds_d) cudaFree(s->ds_d);
    if (s->perm_d) cudaFree(s->perm_d);
    if (s->before_d) cudaFree(s->before_d);
    if (s->pos_d) cudaFree(s->pos_d);
    if (s->l1p_d) cudaFree(s->l1p_d);
    if (s->fp_d) cudaFree(s->fp_d);
    if (s->up_d) cudaFree(s->up_d);
    if (s->fused_steps_d) cudaFree(s->fused_steps_d);
    if (s->fused_bar_d) cudaFree(s->fused_bar_d);
    pe_sell_free(s->S);
    devcsr_free(s->P);
    delete s;
    return 0;
}

// ---- fused sweep: schedule and launch
static int fused_setup(pe_smoother *s)
{
    pe_ctx *ctx = s->ctx;
    const int limit_mb = pe_get_tuning(PE_TUNE_FUSED_GS_MAX_MB);
    const bool general = !(s->weight == 1.0 && s->omega == 1.0);
    if (limit_mb <= 0 || general || s->nsets < 2 || !(s->type == 2 || s->type == 4 || s->type == 6)) return 0;
    const int nsets = s->nsets;
    std::vector<double> bytes(nsets, 0.0);
    std::vector<int2> steps;
    int max_units = 1;                       // rows (CSR) or slices (SELL) of the largest step
    for (int c = 0; c < nsets; ++c)
    {
        const double rows = s->set_starts[c + 1] - s->set_starts[c];
        bytes[c] = s->use_sell ? s->set_bytes[c] : 12.0 * (double)(s->set_pI[c + 1] - s->set_pI[c]) + 36.0 * rows;
        if (bytes[c] >= 1e6 * limit_mb) return 0;                 // a bandwidth-bound colour: keep one launch per colour
    }
    if (s->use_sell) steps.push_back(make_int2(-1, -1));
    s->fused_bytes = 0.0;
    for (int pass = 0; pass < 2; ++pass)
        for (int cc = (pass == 1 && s->skip_turn) ? 1 : 0; cc < nsets; ++cc)
        {
            const int c = pass == 0 ? cc : nsets - 1 - cc;
            const int a = s->use_sell ? s->slice_starts[c] : s->set_starts[c], b = s->use_sell ? s->slice_starts[c + 1] : s->set_starts[c + 1];
            if (b <= a) continue;
            steps.push_back(make_int2(a, b));
            max_units = std::max(max_units, b - a);
            s->fused_bytes += bytes[c];
        }
    if (s->use_sell) steps.push_back(make_int2(-2, -2));
    int nsm = 0, occ = 0, coop = 0;
    PE_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, ctx->device));
    PE_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, ctx->device));
    if (!coop) return 0;
    const void *kern = nullptr;
    if (s->use_sell) kern = (const void *)k_sell_gs_sweep;
    else switch (s->tpr) {
        case 1: kern = (const void *)k_gs_sweep<1>; break;
        case 2: kern = (const void *)k_gs_sweep<2>; break;
        case 4: kern = (const void *)k_gs_sweep<4>; break;
        case 8: kern = (const void *)k_gs_sweep<8>; break;
        case 16: kern = (const void *)k_gs_sweep<16>; break;
        default: kern = (const void *)k_gs_sweep<32>; break;
    }
    PE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 256, 0));
    if (occ < 1) return 0;
    const int64_t threads = s->use_sell ? (int64_t)max_units * 32 : (int64_t)max_units * s->tpr;
    int64_t want = (threads + 255) / 256;
    if (s->use_sell) want = std::max<int64_t>(want, ((int64_t)s->A->diag.nrows + 255) / 256 / 4);   // the renumbering passes
    s->fused_grid = (int)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)nsm * std::min(occ, 4)));
    s->fused_nsteps = (int)steps.size();
    PE_CUDA(cudaMalloc(&s->fused_steps_d, sizeof(int2) * steps.size()));
    PE_CUDA(cudaMemcpy(s->fused_steps_d, steps.data(), sizeof(int2) * steps.size(), cudaMemcpyHostToDevice));
    PE_CUDA(cudaMalloc(&s->fused_bar_d, 2 * sizeof(unsigned)));
    PE_CUDA(cudaMemset(s->fused_bar_d, 0, 2 * sizeof(unsigned)));
    s->fused = true;
    return 0;
}

// The grid never exceeds what is resident at once (fused_setup), nothing else runs on the device while the kernel does
// (the stream is serial; the kernel never triggers its dependents early, and its PDL predecessor completes on its own),
// so an ordinary launch through pe_launch_k -- programmatic dependent launch included -- is enough for the grid barrier.
// Inside a CUDA graph the cooperative attribute proved expensive (measured: 16 fused launches per V-cycle cost +1.4 ms
// as cooperative nodes); PE_FUSED_COOP=1 forces it for debugging.
template <typename... KArgs, typename... Args>
static cudaError_t launch_cooperative(pe_ctx *ctx, void (*kern)(KArgs...), int grid, Args... args)
{
    static const bool coop = getenv("PE_FUSED_COOP") && atoi(getenv("PE_FUSED_COOP")) != 0;
    if (!coop) return pe_launch_k(ctx, kern, grid, 256, args...);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid, 1, 1);
    cfg.blockDim = dim3(256, 1, 1);
    cfg.stream = ctx->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative;
    at[0].val.cooperative = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

static int launch_fused_sweep(pe_smoother *s, const double *b, double *x, bool zero_guess)
{
    pe_ctx *ctx = s->ctx;
    pe_mat *A = s->A;
    if (ctx->prof) PE_TRY(pe_prof_begin(ctx, 3, s->fused_bytes));
    if (s->use_sell)
        PE_CUDA(launch_cooperative(ctx, k_sell_gs_sweep, s->fused_grid, s->fused_nsteps, s->fused_steps_d, s->S.soff, s->S.J, s->S.A, s->npad,
                                   A->diag.nrows, s->pos_d, b, x, zero_guess ? 1 : 0, s->fp_d, s->up_d, A->offd.nnz > 0 ? A->x_ext_d : nullptr,
                                   s->l1p_d, s->fused_bar_d));
    else
    {
#define LAUNCH(T) PE_CUDA(launch_cooperative(ctx, k_gs_sweep<T>, s->fused_grid, s->fused_nsteps, s->fused_steps_d, s->P.I, s->P.J, s->P.A, s->perm_d, \
                                             A->diag.ncols, b, x, A->x_ext_d, s->l1_d, s->fused_bar_d))
        switch (s->tpr) {
        case 1: LAUNCH(1); break;
        case 2: LAUNCH(2); break;
        case 4: LAUNCH(4); break;
        case 8: LAUNCH(8); break;
        case 16: LAUNCH(16); break;
        default: LAUNCH(32); break;
        }
#undef LAUNCH
    }
    PE_LAUNCHED(ctx);
    PE_TRY(pe_prof_end(ctx));
    return 0;
}

template <bool GENERAL>
static int launch_gs_set(pe_smoother *s, int k0, int k1, const double *f, double *u, int forward, double c1, double c2)
{
    pe_ctx *ctx = s->ctx;
    int rows = k1 - k0;
    if (rows <= 0) return 0;
    if (!GENERAL && s->P.nrb > 0 && s->A->diag.nrows >= pe_get_tuning(PE_TUNE_SELL_MIN_ROWS))
    {
        int c = 0;
        while (s->set_starts[c] != k0) ++c;
        const int b0 = s->set_rb[c], b1 = s->set_rb[c + 1];
        if (ctx->prof) PE_TRY(pe_prof_begin(ctx, 3, 12.0 * (double)(s->set_pI[c + 1] - s->set_pI[c]) + 4.0 * rows + 32.0 * rows));
        k_gs_set_stream<<<b1 - b0, 256, 0, ctx->stream>>>(b0, s->P.rb, s->P.I, s->P.J, s->P.A, s->perm_d, s->A->diag.ncols,
                                                         f, u, s->A->x_ext_d, s->l1_d);
        PE_LAUNCHED(ctx);
        PE_TRY(pe_prof_end(ctx));
        return 0;
    }
    int tpr = s->tpr;
    pe_variant_add(PE_VARIANT_RELAX_TPR_1 + __builtin_ctz(tpr), rows);
    int grid = pe_grid_for((int64_t)rows * tpr, 256);
    int ncd = s->A->diag.ncols;
#define LAUNCH(T) PE_CUDA(pe_launch_k(ctx, k_gs_set<T, GENERAL>, grid, 256, k0, k1, s->P.I, s->P.J, s->P.A, s->perm_d, ncd, f, u, s->A->x_ext_d, s->l1_d, s->before_d, forward, s->w_d, c1, c2))
    if (ctx->prof)
    {
        const double nnz_set = (double)(s->pI_at(k1) - s->pI_at(k0));
        PE_TRY(pe_prof_begin(ctx, 3, 12.0 * nnz_set + 4.0 * rows + 32.0 * rows));
    }
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

// ghost values for one sweep: a zero initial guess is zero on every rank, so the exchange is replaced
// by clearing the ghost buffer (all ranks take the same branch: iterative_mode is a collective argument)
static int sweep_halo(pe_mat *A, const double *x_d, bool all_zero)
{
    pe_ctx *ctx = A->ctx;
    if (ctx->nranks == 1) return 0;
    if (all_zero)
    {
        if (A->offd.ncols > 0) PE_CUDA(cudaMemsetAsync(A->x_ext_d, 0, sizeof(double) * (size_t)A->offd.ncols, ctx->stream));
        return 0;
    }
    PE_TRY(pe_halo_exchange(A, x_d));
    return pe_halo_wait(A);
}

extern "C" int pe_smoother_apply(pe_smoother *s, const pe_vec *b, pe_vec *x, int iterative_mode)
{
    pe_ctx *ctx = s->ctx;
    pe_mat *A = s->A;
    int n = A->diag.nrows;
    PE_CHECK(b->n == n && x->n == n, "pe_smoother_apply: size mismatch");
    cudaStream_t st = ctx->stream;
    if (s->use_sell)
    {
        // colour-ordered SELL path: f and u are carried in colour order across the whole sweep
        const bool ghosts = A->offd.nnz > 0;
        for (int sweep = 0; sweep < s->sweeps; ++sweep)
        {
            const bool zero_guess = !iterative_mode && sweep == 0;
            PE_TRY(sweep_halo(A, x->d, zero_guess));
            if (s->fused && !ctx->rec) { PE_TRY(launch_fused_sweep(s, b->d, x->d, zero_guess)); continue; }
            // from a zero guess the first colour only sees zeros: it is done by the renumbering pass
            int first = -1;
            if (zero_guess && s->nsets > 0)
            {
                first = 0;
                while (first < s->nsets - 1 && s->slice_starts[first + 1] == s->slice_starts[first]) ++first;
                PE_TRY(pe_launch_perm_in_gs0(ctx, n, s->pos_d, b->d, 32 * s->slice_starts[first], 32 * s->slice_starts[first + 1],
                                             s->l1p_d, s->fp_d, s->up_d));
            }
            else PE_TRY(pe_launch_perm_in(ctx, n, s->pos_d, b->d, zero_guess ? nullptr : x->d, s->fp_d, s->up_d));
            for (int pass = 0; pass < 2; ++pass)
                for (int cc = (pass == 1 && s->skip_turn) ? 1 : 0; cc < s->nsets; ++cc)
                {
                    const int c = pass == 0 ? cc : s->nsets - 1 - cc;
                    if (s->slice_starts[c + 1] == s->slice_starts[c] || (pass == 0 && c == first)) continue;
                    PE_TRY(pe_prof_begin(ctx, s->set_bytes[c] >= 64e6 ? 1 : 3, s->set_bytes[c]));
                    PE_TRY(pe_launch_sell_gs(ctx, s->S, s->slice_starts[c], s->slice_starts[c + 1], s->set_wmax[c], s->npad, s->fp_d, s->up_d,
                                             ghosts ? A->x_ext_d : nullptr, s->l1p_d, s->pol_gather));
                    PE_TRY(pe_prof_end(ctx));
                }
            PE_TRY(pe_launch_perm_out(ctx, n, s->pos_d, s->up_d, x->d));
        }
        return 0;
    }
    if (!iterative_mode) PE_CUDA(cudaMemsetAsync(x->d, 0, sizeof(double) * (size_t)n, st));
    const int *oI = A->offd.nnz > 0 ? A->offd.I : nullptr;
    for (int sweep = 0; sweep < s->sweeps; ++sweep) {
        if (s->type == 0 || s->type == 1 || s->type == 5) {
            PE_TRY(sweep_halo(A, x->d, !iterative_mode && sweep == 0));
            int tpr = A->tpr;
            pe_variant_add(PE_VARIANT_RELAX_TPR_1 + __builtin_ctz(tpr), n);
            int64_t threads = (int64_t)n * tpr;
            int grid = (int)std::min<int64_t>((threads + 255) / 256, (int64_t)PE_SM_COUNT * 64);
            if (grid < 1) grid = 1;
            PE_TRY(pe_prof_begin(ctx, 2, 12.0 * (double)(A->diag.nnz + A->offd.nnz) + 4.0 * (n + 1) + 8.0 * n * 4));
#define LAUNCH(T) k_jacobi_update<T><<<grid, 256, 0, st>>>(n, A->diag.I, A->diag.J, A->diag.A, oI, A->offd.J, A->offd.A, x->d, A->x_ext_d, b->d, s->l1_d, s->weight, s->v_d)
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
            pe_vec vv{ctx, n, s->v_d};
            PE_TRY(pe_vec_axpby(1.0, &vv, 1.0, x));
        } else if (s->type == 2 || s->type == 4 || s->type == 6) {
            PE_TRY(sweep_halo(A, x->d, !iterative_mode && sweep == 0));
            bool general = !(s->weight == 1.0 && s->omega == 1.0);
            double c1 = s->omega * s->weight, c2 = s->omega * (1.0 - s->weight);
            if (s->fused && !ctx->rec) { PE_TRY(launch_fused_sweep(s, b->d, x->d, false)); continue; }
            for (int pass = 0; pass < 2; ++pass) {
                if (general) PE_CUDA(cudaMemcpyAsync(s->w_d, x->d, sizeof(double) * (size_t)n, cudaMemcpyDeviceToDevice, st));
                for (int cc = (pass == 1 && s->skip_turn) ? 1 : 0; cc < s->nsets; ++cc) {
                    int c = pass == 0 ? cc : s->nsets - 1 - cc;
                    if (general) PE_TRY(launch_gs_set<true>(s, s->set_starts[c], s->set_starts[c + 1], b->d, x->d, pass == 0, c1, c2));
                    else PE_TRY(launch_gs_set<false>(s, s->set_starts[c], s->set_starts[c + 1], b->d, x->d, pass == 0, c1, c2));
                }
            }
        } else if (s->type == 16) {
            int co = s->cheby_order - 1;
            double *r = s->r_d, *uo = s->w_d, *v = s->v_d, *t = s->z_d;
            PE_TRY(spmv_full(ctx, A, -1.0, x->d, 1.0, b->d, r));
            k_cheb_begin<<<pe_grid_for(n, 256), 256, 0, st>>>(n, s->coefs[co], s->ds_d, r, uo, x->d); PE_LAUNCHED(ctx);
            for (int c = co - 1; c >= 0; --c) {
                k_vmul3<<<pe_grid_for(n, 256), 256, 0, st>>>(n, s->ds_d, x->d, v); PE_LAUNCHED(ctx);
                PE_TRY(spmv_full(ctx, A, 1.0, v, 0.0, t, t));
                k_cheb_step<<<pe_grid_for(n, 256), 256, 0, st>>>(n, s->coefs[c], r, s->ds_d, t, x->d); PE_LAUNCHED(ctx);
            }
            k_cheb_end<<<pe_grid_for(n, 256), 256, 0, st>>>(n, s->ds_d, uo, x->d); PE_LAUNCHED(ctx);
        }
    }
    return 0;
}

extern "C" int pe_smoother_get_l1(const pe_smoother *s, double *l1_host)
{
    PE_CUDA(cudaMemcpyAsync(l1_host, s->l1_d, sizeof(double) * (size_t)s->A->diag.nrows, cudaMemcpyDeviceToHost, s->ctx->stream));
    PE_CUDA(cudaStreamSynchronize(s->ctx->stream));
    return 0;
}
extern "C" int pe_smoother_get_order(const pe_smoother *s, int32_t *order_host, int32_t *num_sets, int32_t *set_starts_host)
{
    if (num_sets) *num_sets = s->nsets;
    if (order_host && !s->order.empty()) memcpy(order_host, s->order.data(), sizeof(int32_t) * s->order.size());
    if (set_starts_host && !s->set_starts.empty()) memcpy(set_starts_host, s->set_starts.data(), sizeof(int32_t) * s->set_starts.size());
    return 0;
}
extern "C" int pe_smoother_get_eig(const pe_smoother *s, double *max_eig, double *min_eig)
{
    if (max_eig) *max_eig = s->max_eig;
    if (min_eig) *min_eig = s->min_eig;
    return 0;
}
