// pe_spgemm.cu -- K8/K9: two-pass (symbolic / numeric) hash SpGEMM, Galerkin RAP,
// FixZeroRows and sparse add.
//
// C = A*B row by row (Gustavson).  Each row of C is owned by one GROUP of threads
// (a warp, or a whole CTA for long rows) that accumulates the row in a hash table in
// shared memory (open addressing, linear probing; keys int32 column, values FP64):
//   pass 0  upper bound  ub[i] = sum_{k in A(i,:)} nnz(B(k,:))        -> bins
//   pass 1  symbolic     insert keys only, count distinct               -> C.I (scan)
//   pass 2  numeric      insert keys + atomicAdd values in shared memory, compact,
//                        bitonic-sort by column, write C.J / C.A
// Rows whose table would not fit in shared memory use a table in global memory.
// Rows of C have ascending columns; explicit zeros are kept (they are part of the
// pattern the reference produces, hypre_BoomerAMGBuildCoarseOperator).
#include "pe_core.cuh"
#include <cub/cub.cuh>
#include <algorithm>
#include <climits>

#define HASH_EMPTY (-1)
__device__ __forceinline__ unsigned hash_slot(int key, unsigned mask) { return ((unsigned)key * 2654435761u) & mask; }

// insert key; returns slot index.  `added` set when the key is new.
__device__ __forceinline__ int table_insert(int *keys, unsigned mask, int key, bool &added)
{
    unsigned s = hash_slot(key, mask);
    added = false;
    while (true) {
        int cur = keys[s];
        if (cur == key) return (int)s;
        if (cur == HASH_EMPTY) {
            int old = atomicCAS(keys + s, HASH_EMPTY, key);
            if (old == HASH_EMPTY) { added = true; return (int)s; }
            if (old == key) return (int)s;
        }
        s = (s + 1) & mask;
    }
}

__global__ void k_row_ub(int n, const int *__restrict__ AI, const int *__restrict__ AJ,
                         const int *__restrict__ BI, int *ub)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    long long s = 0;
    for (int k = AI[i]; k < AI[i + 1]; ++k) { int c = AJ[k]; s += BI[c + 1] - BI[c]; }
    ub[i] = s > INT_MAX ? INT_MAX : (int)s;
}

// bin rows by a size measure: bin b holds rows with limits[b-1] < size <= limits[b]
__global__ void k_bin_rows(int n, const int *__restrict__ size, int l0, int l1, int l2,
                           int *counts, int *lists /* 4 lists of capacity n */)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int s = size[i];
    int b = s <= l0 ? 0 : (s <= l1 ? 1 : (s <= l2 ? 2 : 3));
    int p = atomicAdd(counts + b, 1);
    lists[(size_t)b * n + p] = i;
}

// group-level bitonic sort of (keys, vals) in shared/global memory, m padded to pow2
template <int GT>
__device__ void group_sort(int *keys, double *vals, int m2, int tid)
{
    for (int k = 2; k <= m2; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = tid; t < m2; t += GT) {
                int ixj = t ^ j;
                if (ixj > t) {
                    bool up = ((t & k) == 0);
                    int a = keys[t], b = keys[ixj];
                    if ((a > b) == up) {
                        keys[t] = b; keys[ixj] = a;
                        double va = vals[t]; vals[t] = vals[ixj]; vals[ixj] = va;
                    }
                }
            }
            if (GT == 32) __syncwarp(); else __syncthreads();
        }
    }
}

// One group (GT threads: 32 = warp, else whole CTA) per row; TABLE slots per group.
// NUMERIC=false: count distinct columns -> rownnz.  NUMERIC=true: fill CJ/CA sorted.
template <int GT, int TABLE, bool NUMERIC>
__global__ void __launch_bounds__(256)
k_spgemm_smem(int nlist, const int *__restrict__ list,
              const int *__restrict__ AI, const int *__restrict__ AJ, const double *__restrict__ AA,
              const int *__restrict__ BI, const int *__restrict__ BJ, const double *__restrict__ BA,
              int *rownnz, const int *__restrict__ CI, int *CJ, double *CA)
{
    extern __shared__ unsigned char smem_raw[];
    constexpr int GROUPS = 256 / GT;
    const int g = threadIdx.x / GT, tid = threadIdx.x % GT;
    // layout: vals (double) first for alignment, then keys
    double *vals_all = reinterpret_cast<double *>(smem_raw);
    int *keys_all = reinterpret_cast<int *>(smem_raw + (NUMERIC ? sizeof(double) * TABLE * GROUPS : 0));
    int *keys = keys_all + g * TABLE;
    double *vals = NUMERIC ? vals_all + g * TABLE : nullptr;
    __shared__ int cnt[GROUPS];
    const int li = blockIdx.x * GROUPS + g;
    const bool active = li < nlist;   // whole group is uniform
    for (int t = tid; t < TABLE; t += GT) { keys[t] = HASH_EMPTY; if (NUMERIC) vals[t] = 0.0; }
    if (tid == 0) cnt[g] = 0;
    if (GT == 32) __syncwarp(); else __syncthreads();
    int row = active ? list[li] : 0;
    if (active) {
        const int alo = AI[row], ahi = AI[row + 1];
        // lanes stride over the entries of B rows; A entries are walked sequentially
        for (int ka = alo; ka < ahi; ++ka) {
            const int k = AJ[ka];
            const double a = NUMERIC ? AA[ka] : 0.0;
            const int blo = BI[k], bhi = BI[k + 1];
            for (int kb = blo + tid; kb < bhi; kb += GT) {
                bool added;
                int s = table_insert(keys, TABLE - 1, BJ[kb], added);
                if (NUMERIC) atomicAdd(vals + s, a * BA[kb]);   // columns of one B row are distinct: one add per slot and ka
                else if (added) atomicAdd(&cnt[g], 1);
            }
            // products are accumulated in the order of A's row entries (like the serial hypre RAP): the
            // group finishes entry ka before anyone starts ka+1, so every C entry has ONE summation order
            if (NUMERIC) { if (GT == 32) __syncwarp(); else __syncthreads(); }
        }
    }
    if (GT == 32) __syncwarp(); else __syncthreads();
    if (!NUMERIC) {
        if (active && tid == 0) rownnz[row] = cnt[g];
        return;
    }
    // compact occupied slots to the front (order irrelevant, sorted next)
    if (active) {
        const int m = CI[row + 1] - CI[row];
        // serial-free compaction: each occupied slot grabs a position
        // (reuse cnt as cursor); then move in two steps through registers
        // step 1: read own candidates
        int m2 = 1; while (m2 < m) m2 <<= 1;
        // gather into registers chunk by chunk to avoid overwriting unread slots:
        // we compact into the output arrays directly (global), then sort there if small
        int *outJ = CJ + CI[row];
        double *outA = CA + CI[row];
        for (int t = tid; t < TABLE; t += GT) {
            int key = keys[t];
            if (key != HASH_EMPTY) {
                int p = atomicAdd(&cnt[g], 1);
                outJ[p] = key; outA[p] = vals[t];
            }
        }
        if (GT == 32) __syncwarp(); else __syncthreads();
        // bring back to shared memory (dense, padded) and sort
        for (int t = tid; t < m2; t += GT) {
            if (t < m) { keys[t] = outJ[t]; vals[t] = outA[t]; }
            else { keys[t] = INT_MAX; vals[t] = 0.0; }
        }
        if (GT == 32) __syncwarp(); else __syncthreads();
        group_sort<GT>(keys, vals, m2, tid);
        for (int t = tid; t < m; t += GT) { outJ[t] = keys[t]; outA[t] = vals[t]; }
    } else if (GT != 32) {
        // keep CTA-wide barriers matched (only reachable when the whole CTA is inactive)
    }
}

// global-memory table variant for very long rows: one CTA per row
template <bool NUMERIC>
__global__ void __launch_bounds__(256)
k_spgemm_gmem(int nlist, const int *__restrict__ list, const long long *__restrict__ tab_off,
              const int *__restrict__ tab_size, int *gkeys, double *gvals,
              const int *__restrict__ AI, const int *__restrict__ AJ, const double *__restrict__ AA,
              const int *__restrict__ BI, const int *__restrict__ BJ, const double *__restrict__ BA,
              int *rownnz, const int *__restrict__ CI, int *CJ, double *CA)
{
    const int li = blockIdx.x;
    if (li >= nlist) return;
    const int row = list[li], tid = threadIdx.x;
    int *keys = gkeys + tab_off[li];
    double *vals = NUMERIC ? gvals + tab_off[li] : nullptr;
    const int T = tab_size[li];
    __shared__ int cnt;
    for (int t = tid; t < T; t += 256) { keys[t] = HASH_EMPTY; if (NUMERIC) vals[t] = 0.0; }
    if (tid == 0) cnt = 0;
    __syncthreads();
    for (int ka = AI[row]; ka < AI[row + 1]; ++ka) {
        const int k = AJ[ka];
        const double a = NUMERIC ? AA[ka] : 0.0;
        for (int kb = BI[k] + tid; kb < BI[k + 1]; kb += 256) {
            bool added;
            int s = table_insert(keys, (unsigned)T - 1, BJ[kb], added);
            if (NUMERIC) atomicAdd(vals + s, a * BA[kb]);
            else if (added) atomicAdd(&cnt, 1);
        }
        if (NUMERIC) __syncthreads();                // fixed summation order, see k_spgemm_smem
    }
    __syncthreads();
    if (!NUMERIC) { if (tid == 0) rownnz[row] = cnt; return; }
    const int m = CI[row + 1] - CI[row];
    int m2 = 1; while (m2 < m) m2 <<= 1;
    __shared__ int cursor;
    if (tid == 0) cursor = 0;
    __syncthreads();
    int *outJ = CJ + CI[row];
    double *outA = CA + CI[row];
    for (int t = tid; t < T; t += 256) {
        int key = keys[t];
        if (key != HASH_EMPTY) { int p = atomicAdd(&cursor, 1); outJ[p] = key; outA[p] = vals[t]; }
    }
    __syncthreads();
    // sort in the (now free) global table, padded
    for (int t = tid; t < m2; t += 256) {
        if (t < m) { keys[t] = outJ[t]; vals[t] = outA[t]; } else { keys[t] = INT_MAX; vals[t] = 0.0; }
    }
    __syncthreads();
    group_sort<256>(keys, vals, m2, tid);
    for (int t = tid; t < m; t += 256) { outJ[t] = keys[t]; outA[t] = vals[t]; }
}

template <bool NUMERIC>
static int run_bins(pe_ctx *ctx, int n, const int *size_d, const DevCSR &A, const DevCSR &B,
                    int *rownnz_d, const DevCSR *C)
{
    cudaStream_t st = ctx->stream;
    // table sizes: W128 holds <=64, W1024 holds <=512, B8192 holds <=4096 entries
    const int L0 = 64, L1 = 512, L2 = 4096;
    int *counts_d, *lists_d;
    PE_CUDA(cudaMalloc(&counts_d, sizeof(int) * 4));
    PE_CUDA(cudaMalloc(&lists_d, sizeof(int) * 4 * (size_t)n));
    PE_CUDA(cudaMemsetAsync(counts_d, 0, sizeof(int) * 4, st));
    k_bin_rows<<<pe_grid_for(n, 256), 256, 0, st>>>(n, size_d, L0, L1, L2, counts_d, lists_d);
    PE_LAUNCHED(ctx);
    int counts[4];
    PE_CUDA(cudaMemcpyAsync(counts, counts_d, sizeof(int) * 4, cudaMemcpyDeviceToHost, st));
    PE_CUDA(cudaStreamSynchronize(st));
    for (int b = 0; b < 4; ++b) pe_variant_add((NUMERIC ? PE_VARIANT_SPGEMM_NUM_T128 : PE_VARIANT_SPGEMM_SYM_T128) + b, counts[b]);
    const int *CI = C ? C->I : nullptr;
    int *CJ = C ? C->J : nullptr;
    double *CA = C ? C->A : nullptr;
    const size_t per_slot = NUMERIC ? 12 : 4;
    if (counts[0] > 0) {
        size_t sm = per_slot * 128 * 8;
        k_spgemm_smem<32, 128, NUMERIC><<<pe_grid_for(counts[0], 8), 256, sm, st>>>(counts[0], lists_d, A.I, A.J, A.A, B.I, B.J, B.A, rownnz_d, CI, CJ, CA);
        PE_LAUNCHED(ctx);
    }
    if (counts[1] > 0) {
        size_t sm = per_slot * 1024 * 8;
        PE_CUDA(cudaFuncSetAttribute(k_spgemm_smem<32, 1024, NUMERIC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        k_spgemm_smem<32, 1024, NUMERIC><<<pe_grid_for(counts[1], 8), 256, sm, st>>>(counts[1], lists_d + (size_t)n, A.I, A.J, A.A, B.I, B.J, B.A, rownnz_d, CI, CJ, CA);
        PE_LAUNCHED(ctx);
    }
    if (counts[2] > 0) {
        size_t sm = per_slot * 8192;
        PE_CUDA(cudaFuncSetAttribute(k_spgemm_smem<256, 8192, NUMERIC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        k_spgemm_smem<256, 8192, NUMERIC><<<counts[2], 256, sm, st>>>(counts[2], lists_d + 2 * (size_t)n, A.I, A.J, A.A, B.I, B.J, B.A, rownnz_d, CI, CJ, CA);
        PE_LAUNCHED(ctx);
    }
    if (counts[3] > 0) {
        // global tables, processed in chunks bounded by ~1 GiB of table memory
        std::vector<int> rows(counts[3]), sizes(n);
        PE_CUDA(cudaMemcpy(rows.data(), lists_d + 3 * (size_t)n, sizeof(int) * counts[3], cudaMemcpyDeviceToHost));
        PE_CUDA(cudaMemcpy(sizes.data(), size_d, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost));
        std::sort(rows.begin(), rows.end());
        size_t pos = 0;
        const long long cap = (1ll << 30) / 12;
        while (pos < rows.size()) {
            std::vector<long long> off; std::vector<int> tsz, chunk;
            long long tot = 0;
            while (pos < rows.size()) {
                long long need = 2ll * sizes[rows[pos]];
                long long t = 1; while (t < need) t <<= 1;
                if (t > (1ll << 30)) t = 1ll << 30;
                if (!chunk.empty() && tot + t > cap) break;
                off.push_back(tot); tsz.push_back((int)t); chunk.push_back(rows[pos]); tot += t; ++pos;
            }
            int *gk, *chunk_d, *tsz_d; double *gv = nullptr; long long *off_d;
            PE_CUDA(cudaMalloc(&gk, sizeof(int) * (size_t)tot));
            if (NUMERIC) PE_CUDA(cudaMalloc(&gv, sizeof(double) * (size_t)tot));
            PE_CUDA(cudaMalloc(&chunk_d, sizeof(int) * chunk.size()));
            PE_CUDA(cudaMalloc(&tsz_d, sizeof(int) * chunk.size()));
            PE_CUDA(cudaMalloc(&off_d, sizeof(long long) * chunk.size()));
            PE_CUDA(cudaMemcpy(chunk_d, chunk.data(), sizeof(int) * chunk.size(), cudaMemcpyHostToDevice));
            PE_CUDA(cudaMemcpy(tsz_d, tsz.data(), sizeof(int) * chunk.size(), cudaMemcpyHostToDevice));
            PE_CUDA(cudaMemcpy(off_d, off.data(), sizeof(long long) * chunk.size(), cudaMemcpyHostToDevice));
            k_spgemm_gmem<NUMERIC><<<(int)chunk.size(), 256, 0, st>>>((int)chunk.size(), chunk_d, off_d, tsz_d, gk, gv, A.I, A.J, A.A, B.I, B.J, B.A, rownnz_d, CI, CJ, CA);
            PE_LAUNCHED(ctx);
            PE_CUDA(cudaStreamSynchronize(st));
            cudaFree(gk); if (gv) cudaFree(gv); cudaFree(chunk_d); cudaFree(tsz_d); cudaFree(off_d);
        }
    }
    PE_CUDA(cudaStreamSynchronize(st));
    cudaFree(counts_d); cudaFree(lists_d);
    return 0;
}

int pe_devcsr_spgemm(pe_ctx *ctx, const DevCSR &A, const DevCSR &B, DevCSR &C)
{
    PE_CHECK(A.ncols == B.nrows, "spgemm: inner dimensions differ");
    cudaStream_t st = ctx->stream;
    int n = A.nrows;
    int *ub_d, *rownnz_d;
    PE_CUDA(cudaMalloc(&ub_d, sizeof(int) * (size_t)(n + 1)));
    PE_CUDA(cudaMalloc(&rownnz_d, sizeof(int) * (size_t)(n + 2)));
    PE_CUDA(cudaMemsetAsync(rownnz_d, 0, sizeof(int) * (size_t)(n + 2), st));
    if (n > 0) {
        k_row_ub<<<pe_grid_for(n, 256), 256, 0, st>>>(n, A.I, A.J, B.I, ub_d); PE_LAUNCHED(ctx);
        PE_TRY((run_bins<false>(ctx, n, ub_d, A, B, rownnz_d, nullptr)));
    }
    // C.I = exclusive scan of rownnz
    int *CI;
    PE_CUDA(cudaMalloc(&CI, sizeof(int) * (size_t)(n + 1)));
    void *tmp = nullptr; size_t tb = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tb, rownnz_d, CI, n + 1, st);
    PE_CUDA(cudaMalloc(&tmp, tb));
    PE_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tb, rownnz_d, CI, n + 1, st));
    ctx->launches++;
    int nnz = 0;
    PE_CUDA(cudaMemcpyAsync(&nnz, CI + n, sizeof(int), cudaMemcpyDeviceToHost, st));
    PE_CUDA(cudaStreamSynchronize(st));
    cudaFree(tmp);
    C.nrows = n; C.ncols = B.ncols; C.nnz = nnz; C.I = CI;
    PE_CUDA(cudaMalloc(&C.J, sizeof(int) * (size_t)(nnz > 0 ? nnz : 1)));
    PE_CUDA(cudaMalloc(&C.A, sizeof(double) * (size_t)(nnz > 0 ? nnz : 1)));
    if (n > 0 && nnz > 0) {
        // numeric tables are sized from the exact row counts: the bin limits are half the
        // table capacities, so the row counts themselves select the bin
        PE_TRY((run_bins<true>(ctx, n, rownnz_d, A, B, rownnz_d, &C)));
    }
    cudaFree(ub_d); cudaFree(rownnz_d);
    return 0;
}

extern "C" int pe_spgemm(pe_ctx *ctx, const pe_mat *A, const pe_mat *B, pe_mat **C)
{
    if (A->distributed || B->distributed)
    {
        PE_CHECK(A->distributed && B->distributed, "pe_spgemm: A and B must both be distributed matrices");
        return pe_spgemm_distributed(ctx, A, B, C);
    }
    DevCSR c;
    PE_TRY(pe_devcsr_spgemm(ctx, A->diag, B->diag, c));
    PE_TRY(pe_mat_wrap_local(ctx, c, C));
    (*C)->global_num_rows = A->global_num_rows;
    (*C)->global_num_cols = B->global_num_cols;
    return 0;
}

extern "C" int pe_rap(pe_ctx *ctx, const pe_mat *R, const pe_mat *A, const pe_mat *P, pe_mat **Ac)
{
    if (A->distributed || P->distributed)
    {
        PE_CHECK(A->distributed && P->distributed, "pe_rap: A and P must both be distributed matrices");
        PE_CHECK(!R || R->distributed, "pe_rap: R must be a distributed matrix as well");
        return pe_rap_distributed(ctx, R, A, P, Ac);
    }
    const pe_mat *Rm = R ? R : P;
    PE_CHECK(Rm->diag.nrows == A->diag.nrows && A->diag.ncols == P->diag.nrows, "pe_rap: size mismatch");
    DevCSR AP, Rt, C;
    PE_TRY(pe_devcsr_spgemm(ctx, A->diag, P->diag, AP));
    bool own_rt = true;
    if (Rm->T) { Rt = Rm->T->diag; own_rt = false; }
    else PE_TRY(pe_devcsr_transpose(ctx, Rm->diag, Rt));
    PE_TRY(pe_devcsr_spgemm(ctx, Rt, AP, C));
    devcsr_free(AP);
    if (own_rt) devcsr_free(Rt);
    PE_TRY(pe_mat_wrap_local(ctx, C, Ac));
    return 0;
}

// ---------------------------------------------------------------------------
// Numeric pass into a known pattern (pe_spgemm_numeric / pe_rap_numeric): the sorted columns of a row of C are its slot
// table, and a product a_ik * b_kj lands on the slot of column j found by binary search.  The group finishes entry ka of
// A's row before any thread starts ka+1, and every slot gets at most one add per ka (the columns of a B row are
// distinct), so every entry of C is summed in the order of k_spgemm_smem / k_spgemm_gmem, starting from 0.0, and the
// values are theirs bit for bit.  The product and the add are rounded separately, as the atomicAdd of those kernels.
// CAP > 0: the row is staged in shared memory (CAP slots per group); CAP == 0: one CTA per row, in place in C.
// SCALE: B's row k is read multiplied by s_k = 1.0 / d[k] (C = A diag(d)^-1 B), each b_kj * s_k rounded once, as
// k_scale_rows rounds it on a scaled copy of B before the two-pass product.
__global__ void k_row_len(int n, const int *__restrict__ I, int *len)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) len[i] = I[i + 1] - I[i];
}

template <int GT, int CAP, bool SCALE>
__global__ void __launch_bounds__(256)
k_spgemm_refill(int nlist, const int *__restrict__ list,
                const int *__restrict__ AI, const int *__restrict__ AJ, const double *__restrict__ AA,
                const int *__restrict__ BI, const int *__restrict__ BJ, const double *__restrict__ BA,
                const double *__restrict__ d, const int *__restrict__ CI, const int *__restrict__ CJ, double *CA)
{
    extern __shared__ unsigned char smem_raw[];
    constexpr int GROUPS = 256 / GT;
    const int g = threadIdx.x / GT, tid = threadIdx.x % GT;
    const int li = blockIdx.x * GROUPS + g;
    const bool active = li < nlist;   // whole group is uniform
    const int row = active ? list[li] : 0;
    const int c0 = active ? CI[row] : 0, m = active ? CI[row + 1] - c0 : 0;
    const int *keys;
    double *vals;
    if (CAP > 0)
    {
        vals = reinterpret_cast<double *>(smem_raw) + g * CAP;
        int *k = reinterpret_cast<int *>(smem_raw + sizeof(double) * CAP * GROUPS) + g * CAP;
        for (int t = tid; t < m; t += GT) { k[t] = CJ[c0 + t]; vals[t] = 0.0; }
        keys = k;
    }
    else
    {
        keys = CJ + c0;
        vals = CA + c0;
        for (int t = tid; t < m; t += GT) vals[t] = 0.0;
    }
    if (GT == 32) __syncwarp(); else __syncthreads();
    if (active)
    {
        for (int ka = AI[row]; ka < AI[row + 1]; ++ka)
        {
            const int k = AJ[ka];
            const double a = AA[ka];
            const double sk = SCALE ? __ddiv_rn(1.0, d[k]) : 1.0;
            for (int kb = BI[k] + tid; kb < BI[k + 1]; kb += GT)
            {
                const int col = BJ[kb];
                int lo = 0, hi = m;
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (keys[mid] < col) lo = mid + 1; else hi = mid; }
                const double b = SCALE ? __dmul_rn(BA[kb], sk) : BA[kb];
                if (lo < m && keys[lo] == col) vals[lo] = __dadd_rn(vals[lo], __dmul_rn(a, b));
            }
            if (GT == 32) __syncwarp(); else __syncthreads();
        }
    }
    if (CAP > 0) for (int t = tid; t < m; t += GT) CA[c0 + t] = vals[t];
}

template <bool SCALE>
static int refill_bins(pe_ctx *ctx, const int *counts, const int *lists_d, int n, const DevCSR &A, const DevCSR &B,
                       const double *d, DevCSR &C)
{
    cudaStream_t st = ctx->stream;
    if (counts[0] > 0)
    {
        k_spgemm_refill<32, 64, SCALE><<<pe_grid_for(counts[0], 8), 256, 12 * 64 * 8, st>>>(
            counts[0], lists_d, A.I, A.J, A.A, B.I, B.J, B.A, d, C.I, C.J, C.A);
        PE_LAUNCHED(ctx);
    }
    if (counts[1] > 0)
    {
        const int sm = 12 * 512 * 8;
        PE_CUDA(cudaFuncSetAttribute(k_spgemm_refill<32, 512, SCALE>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm));
        k_spgemm_refill<32, 512, SCALE><<<pe_grid_for(counts[1], 8), 256, sm, st>>>(
            counts[1], lists_d + (size_t)n, A.I, A.J, A.A, B.I, B.J, B.A, d, C.I, C.J, C.A);
        PE_LAUNCHED(ctx);
    }
    if (counts[2] > 0)
    {
        const int sm = 12 * 4096;
        PE_CUDA(cudaFuncSetAttribute(k_spgemm_refill<256, 4096, SCALE>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm));
        k_spgemm_refill<256, 4096, SCALE><<<counts[2], 256, sm, st>>>(
            counts[2], lists_d + 2 * (size_t)n, A.I, A.J, A.A, B.I, B.J, B.A, d, C.I, C.J, C.A);
        PE_LAUNCHED(ctx);
    }
    if (counts[3] > 0)
    {
        k_spgemm_refill<256, 0, SCALE><<<counts[3], 256, 0, st>>>(
            counts[3], lists_d + 3 * (size_t)n, A.I, A.J, A.A, B.I, B.J, B.A, d, C.I, C.J, C.A);
        PE_LAUNCHED(ctx);
    }
    return 0;
}

/// C (held pattern) = A B, or A diag(d)^-1 B when d is given (d: device array of B's row count)
int pe_devcsr_spgemm_numeric(pe_ctx *ctx, const DevCSR &A, const DevCSR &B, DevCSR &C, const double *d = nullptr)
{
    PE_CHECK(A.ncols == B.nrows && C.nrows == A.nrows && C.ncols == B.ncols, "spgemm_numeric: size mismatch");
    const int n = A.nrows;
    if (n == 0 || C.nnz == 0) return 0;
    cudaStream_t st = ctx->stream;
    // bins by the row length of C: <= 64 and <= 512 entries (a warp per row), <= 4096 (a CTA per row, shared memory),
    // longer rows in place in global memory
    const int L0 = 64, L1 = 512, L2 = 4096;
    int *len_d, *counts_d, *lists_d;
    PE_CUDA(cudaMalloc(&len_d, sizeof(int) * (size_t)n));
    PE_CUDA(cudaMalloc(&counts_d, sizeof(int) * 4));
    PE_CUDA(cudaMalloc(&lists_d, sizeof(int) * 4 * (size_t)n));
    PE_CUDA(cudaMemsetAsync(counts_d, 0, sizeof(int) * 4, st));
    k_row_len<<<pe_grid_for(n, 256), 256, 0, st>>>(n, C.I, len_d);
    PE_LAUNCHED(ctx);
    k_bin_rows<<<pe_grid_for(n, 256), 256, 0, st>>>(n, len_d, L0, L1, L2, counts_d, lists_d);
    PE_LAUNCHED(ctx);
    int counts[4];
    PE_CUDA(cudaMemcpyAsync(counts, counts_d, sizeof(int) * 4, cudaMemcpyDeviceToHost, st));
    PE_CUDA(cudaStreamSynchronize(st));
    const int rc = d ? refill_bins<true>(ctx, counts, lists_d, n, A, B, d, C) : refill_bins<false>(ctx, counts, lists_d, n, A, B, d, C);
    PE_CUDA(cudaStreamSynchronize(st));
    cudaFree(len_d); cudaFree(counts_d); cudaFree(lists_d);
    return rc;
}

extern "C" int pe_spgemm_numeric(pe_ctx *ctx, const pe_mat *A, const pe_mat *B, pe_mat *C)
{
    PE_CHECK(ctx && A && B && C, "bad arguments");
    PE_CHECK(!A->distributed && !B->distributed && !C->distributed && C->offd.nnz == 0,
             "pe_spgemm_numeric: single-rank matrices only");
    PE_TRY(pe_devcsr_spgemm_numeric(ctx, A->diag, B->diag, C->diag));
    pe_mat_values_changed(C);
    return 0;
}

// C = A diag(d)^-1 B into C's pattern: the Schur complement's A10 D^-1 A01 without the build's scaled copy of A01.
// That copy (pe_spadd(1, A01, 0, A01), then k_scale_rows) holds 1*b + 0*b = b for every finite entry b, -0.0
// included (-0.0 + -0.0 = -0.0); and a signed zero product cannot change a sum that starts from +0.0.  The scale
// 1.0 / d[k] and the products are rounded as k_scale_rows and the two-pass product round them, so the values are the
// build's bit for bit.
extern "C" int pe_spgemm_numeric_scaled(pe_ctx *ctx, const pe_mat *A, const pe_vec *d, const pe_mat *B, pe_mat *C)
{
    PE_CHECK(ctx && A && d && B && C, "bad arguments");
    PE_CHECK(!A->distributed && !B->distributed && !C->distributed && C->offd.nnz == 0,
             "pe_spgemm_numeric_scaled: single-rank matrices only");
    PE_CHECK(d->n == B->diag.nrows, "pe_spgemm_numeric_scaled: d must have one entry per row of B");
    PE_TRY(pe_devcsr_spgemm_numeric(ctx, A->diag, B->diag, C->diag, d->d));
    pe_mat_values_changed(C);
    return 0;
}

// A*P is recomputed with the two-pass product (its pattern is not kept from the build: no extra memory between
// updates); the outer product R^T (A P) is the numeric pass into Ac's pattern, with R's cached transpose when it has
// one (R = P when R is null), as pe_rap.
extern "C" int pe_rap_numeric(pe_ctx *ctx, const pe_mat *R, const pe_mat *A, const pe_mat *P, pe_mat *Ac)
{
    PE_CHECK(ctx && A && P && Ac, "bad arguments");
    const pe_mat *Rm = R ? R : P;
    PE_CHECK(!A->distributed && !P->distributed && !Rm->distributed && !Ac->distributed && Ac->offd.nnz == 0,
             "pe_rap_numeric: single-rank matrices only");
    PE_CHECK(Rm->diag.nrows == A->diag.nrows && A->diag.ncols == P->diag.nrows && Ac->diag.nrows == Rm->diag.ncols &&
             Ac->diag.ncols == P->diag.ncols, "pe_rap_numeric: size mismatch");
    DevCSR AP, Rt;
    PE_TRY(pe_devcsr_spgemm(ctx, A->diag, P->diag, AP));
    const bool own_rt = !Rm->T;
    if (Rm->T) Rt = Rm->T->diag;
    else PE_TRY(pe_devcsr_transpose(ctx, Rm->diag, Rt));
    const int rc = pe_devcsr_spgemm_numeric(ctx, Rt, AP, Ac->diag);
    devcsr_free(AP);
    if (own_rt) devcsr_free(Rt);
    PE_TRY(rc);
    pe_mat_values_changed(Ac);
    return 0;
}

// ---------------------------------------------------------------------------
// mask_i = 1 where hypre_ParCSRMatrixFixZeroRows rewrites row i (l1 norm below DBL_EPSILON, as k_fix_zero_rows);
// with `changed` set, *changed = 1 where that differs from the mask instead (the mask is only read)
__global__ void k_zero_rows(int n, const int *__restrict__ dI, const double *__restrict__ dA,
                            const int *__restrict__ oI, const double *__restrict__ oA, double *mask, int *changed)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double l1 = 0.0;
    for (int k = dI[i]; k < dI[i + 1]; ++k) l1 += fabs(dA[k]);
    if (oI) for (int k = oI[i]; k < oI[i + 1]; ++k) l1 += fabs(oA[k]);
    const double z = l1 < 2.2204460492503131e-16 ? 1.0 : 0.0;
    if (!changed) mask[i] = z;
    else if (mask[i] != z) *changed = 1;
}
extern "C" int pe_mat_zero_rows(pe_ctx *ctx, const pe_mat *A, pe_vec *mask, int32_t *changed)
{
    PE_CHECK(ctx && A && mask && mask->n == A->diag.nrows, "pe_mat_zero_rows: mask length differs from the rows of A");
    const int n = A->diag.nrows;
    int *flag = reinterpret_cast<int *>(ctx->scalar_d + 4);
    if (changed) PE_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), ctx->stream));
    if (n > 0)
    {
        k_zero_rows<<<pe_grid_for(n, 256), 256, 0, ctx->stream>>>(n, A->diag.I, A->diag.A, A->offd.nnz > 0 ? A->offd.I : nullptr,
                                                                  A->offd.A, mask->d, changed ? flag : nullptr);
        PE_LAUNCHED(ctx);
    }
    if (changed)
    {
        int h = 0;
        PE_CUDA(cudaMemcpyAsync(&h, flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        PE_CUDA(cudaStreamSynchronize(ctx->stream));
        *changed = h;
    }
    return 0;
}

// ---------------------------------------------------------------------------
__global__ void k_fix_zero_rows(int n, const int *__restrict__ dI, const int *__restrict__ dJ, double *dA,
                                const int *__restrict__ oI, double *oA, int *nfixed)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double l1 = 0.0;
    for (int k = dI[i]; k < dI[i + 1]; ++k) l1 += fabs(dA[k]);
    if (oI) for (int k = oI[i]; k < oI[i + 1]; ++k) l1 += fabs(oA[k]);
    if (l1 < 2.2204460492503131e-16) {
        for (int k = dI[i]; k < dI[i + 1]; ++k) dA[k] = (dJ[k] == i) ? 1.0 : 0.0;
        if (oI) for (int k = oI[i]; k < oI[i + 1]; ++k) oA[k] = 0.0;
        atomicAdd(nfixed, 1);
    }
}
extern "C" int pe_fix_zero_rows(pe_ctx *ctx, pe_mat *A, int32_t *num_fixed)
{
    int n = A->diag.nrows;
    int *cnt = reinterpret_cast<int *>(ctx->scalar_d + 4);
    PE_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int), ctx->stream));
    if (n > 0) {
        k_fix_zero_rows<<<pe_grid_for(n, 256), 256, 0, ctx->stream>>>(n, A->diag.I, A->diag.J, A->diag.A,
                                                                     A->offd.nnz > 0 ? A->offd.I : nullptr, A->offd.A, cnt);
        PE_LAUNCHED(ctx);
    }
    int h = 0;
    PE_CUDA(cudaMemcpyAsync(&h, cnt, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    PE_CUDA(cudaStreamSynchronize(ctx->stream));
    if (num_fixed) *num_fixed = h;
    if (h > 0) pe_mat_values_changed(A);
    return 0;
}

// C = a*A + b*B: entries of A in their order, then the entries of B not in A
// (hypre_CSRMatrixAdd2 two-pass count/fill with a marker; here a row-local search).
__global__ void k_spadd_count(int n, const int *__restrict__ AI, const int *__restrict__ AJ,
                              const int *__restrict__ BI, const int *__restrict__ BJ, int *len)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int c = AI[i + 1] - AI[i];
    for (int kb = BI[i]; kb < BI[i + 1]; ++kb) {
        bool found = false;
        for (int ka = AI[i]; ka < AI[i + 1]; ++ka) if (AJ[ka] == BJ[kb]) { found = true; break; }
        if (!found) ++c;
    }
    len[i] = c;
}
// PATTERN = false (pe_spadd_numeric): C already holds this pattern; only its values are written, with the same
// arithmetic, so they are pe_spadd's bit for bit.
template <bool PATTERN>
__global__ void k_spadd_fill(int n, double a, const int *__restrict__ AI, const int *__restrict__ AJ, const double *__restrict__ AA,
                             double b, const int *__restrict__ BI, const int *__restrict__ BJ, const double *__restrict__ BA,
                             const int *__restrict__ CI, int *CJ, double *CA)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int p = CI[i];
    const int p0 = p;
    for (int ka = AI[i]; ka < AI[i + 1]; ++ka, ++p) { if (PATTERN) CJ[p] = AJ[ka]; CA[p] = a * AA[ka]; }
    const int na = p - p0;
    for (int kb = BI[i]; kb < BI[i + 1]; ++kb) {
        int hit = -1;
        for (int q = 0; q < na; ++q) if (CJ[p0 + q] == BJ[kb]) { hit = p0 + q; break; }
        if (hit >= 0) CA[hit] += b * BA[kb];
        else { if (PATTERN) CJ[p] = BJ[kb]; CA[p] = b * BA[kb]; ++p; }
    }
}
int pe_devcsr_spadd(pe_ctx *ctx, double a, const DevCSR &A, double b, const DevCSR &B, DevCSR &C)
{
    PE_CHECK(A.nrows == B.nrows && A.ncols == B.ncols, "pe_spadd: size mismatch");
    cudaStream_t st = ctx->stream;
    int n = A.nrows;
    int *len;
    PE_CUDA(cudaMalloc(&len, sizeof(int) * (size_t)(n + 1)));
    PE_CUDA(cudaMemsetAsync(len, 0, sizeof(int) * (size_t)(n + 1), st));
    if (n > 0) { k_spadd_count<<<pe_grid_for(n, 256), 256, 0, st>>>(n, A.I, A.J, B.I, B.J, len); PE_LAUNCHED(ctx); }
    C = DevCSR();
    PE_CUDA(cudaMalloc(&C.I, sizeof(int) * (size_t)(n + 1)));
    void *tmp = nullptr; size_t tb = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tb, len, C.I, n + 1, st);
    PE_CUDA(cudaMalloc(&tmp, tb));
    PE_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tb, len, C.I, n + 1, st));
    ctx->launches++;
    int nnz = 0;
    PE_CUDA(cudaMemcpyAsync(&nnz, C.I + n, sizeof(int), cudaMemcpyDeviceToHost, st));
    PE_CUDA(cudaStreamSynchronize(st));
    cudaFree(tmp); cudaFree(len);
    C.nrows = n; C.ncols = A.ncols; C.nnz = nnz;
    PE_CUDA(cudaMalloc(&C.J, sizeof(int) * (size_t)(nnz > 0 ? nnz : 1)));
    PE_CUDA(cudaMalloc(&C.A, sizeof(double) * (size_t)(nnz > 0 ? nnz : 1)));
    if (n > 0) { k_spadd_fill<true><<<pe_grid_for(n, 256), 256, 0, st>>>(n, a, A.I, A.J, A.A, b, B.I, B.J, B.A, C.I, C.J, C.A); PE_LAUNCHED(ctx); }
    return 0;
}
extern "C" int pe_spadd(pe_ctx *ctx, double a, const pe_mat *A, double b, const pe_mat *B, pe_mat **Cout)
{
    if (A->distributed || B->distributed)
    {
        PE_CHECK(A->distributed && B->distributed, "pe_spadd: A and B must both be distributed matrices");
        return pe_spadd_distributed(ctx, a, A, b, B, Cout);
    }
    PE_CHECK(A->offd.nnz == 0 && B->offd.nnz == 0, "pe_spadd: local blocks only");
    DevCSR C;
    PE_TRY(pe_devcsr_spadd(ctx, a, A->diag, b, B->diag, C));
    PE_TRY(pe_mat_wrap_local(ctx, C, Cout));
    return 0;
}

extern "C" int pe_spadd_numeric(pe_ctx *ctx, double a, const pe_mat *A, double b, const pe_mat *B, pe_mat *C)
{
    PE_CHECK(ctx && A && B && C, "bad arguments");
    PE_CHECK(!A->distributed && !B->distributed && !C->distributed && A->offd.nnz == 0 && B->offd.nnz == 0 && C->offd.nnz == 0,
             "pe_spadd_numeric: single-rank matrices only");
    PE_CHECK(A->diag.nrows == B->diag.nrows && A->diag.ncols == B->diag.ncols && C->diag.nrows == A->diag.nrows &&
             C->diag.ncols == A->diag.ncols, "pe_spadd_numeric: size mismatch");
    PE_CHECK(C->diag.nnz >= A->diag.nnz && C->diag.nnz <= A->diag.nnz + B->diag.nnz,
             "pe_spadd_numeric: C does not hold the pattern of a A + b B");
    const int n = A->diag.nrows;
    if (n > 0)
    {
        k_spadd_fill<false><<<pe_grid_for(n, 256), 256, 0, ctx->stream>>>(n, a, A->diag.I, A->diag.J, A->diag.A, b, B->diag.I,
                                                                           B->diag.J, B->diag.A, C->diag.I, C->diag.J, C->diag.A);
        PE_LAUNCHED(ctx);
    }
    pe_mat_values_changed(C);
    return 0;
}

// ---------------------------------------------------------------------------
__global__ void k_eliminate_rowcol(int n, const int *__restrict__ I, const int *__restrict__ J, double *A,
                                   const int *__restrict__ marker)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const bool mi = marker[i] != 0;
    for (int k = I[i]; k < I[i + 1]; ++k)
    {
        const int j = J[k];
        if (mi) A[k] = (j == i) ? 1.0 : 0.0;
        else if (marker[j]) A[k] = 0.0;
    }
}
extern "C" int pe_mat_eliminate_rowcol(pe_ctx *ctx, pe_mat *A, const int32_t *marker_host)
{
    PE_CHECK(A->offd.nnz == 0 && A->diag.nrows == A->diag.ncols, "pe_mat_eliminate_rowcol: square local matrices only");
    int n = A->diag.nrows;
    int *m_d;
    PE_CUDA(cudaMalloc(&m_d, sizeof(int) * (size_t)(n > 0 ? n : 1)));
    PE_CUDA(cudaMemcpyAsync(m_d, marker_host, sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    if (n > 0) { k_eliminate_rowcol<<<pe_grid_for(n, 256), 256, 0, ctx->stream>>>(n, A->diag.I, A->diag.J, A->diag.A, m_d); PE_LAUNCHED(ctx); }
    PE_CUDA(cudaStreamSynchronize(ctx->stream));
    cudaFree(m_d);
    pe_mat_values_changed(A);
    return 0;
}
