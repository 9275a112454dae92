// pe_core.cuh -- internal structures shared by the CUDA translation units.
// Data layout in HBM (see DESIGN.md): every ParCSR matrix is two CSR blocks
// (diag: owned columns, offd: compressed ghost columns) with int32 indices and FP64
// values, plus device-resident halo index lists.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <memory>
#include <string>
#include <vector>
#include "../../include/parelag_b200.h"

#define PE_SM_COUNT 148

void pe_set_error(const std::string &msg);

#define PE_CUDA(call)                                                              \
    do {                                                                           \
        cudaError_t e_ = (call);                                                   \
        if (e_ != cudaSuccess) {                                                   \
            pe_set_error(std::string(#call) + " failed: " + cudaGetErrorString(e_) \
                         + " at " + __FILE__ + ":" + std::to_string(__LINE__));    \
            return 1;                                                              \
        }                                                                          \
    } while (0)

#define PE_CHECK(cond, msg)                                     \
    do {                                                        \
        if (!(cond)) {                                          \
            pe_set_error(std::string(msg) + " (" #cond ")");    \
            return 2;                                           \
        }                                                       \
    } while (0)

#define PE_TRY(expr)              \
    do {                          \
        int rc_ = (expr);         \
        if (rc_) return rc_;      \
    } while (0)

// count one kernel launch on ctx and check the launch status.  A launch that reaches this
// macro while a program is being recorded (pe_prog.cu) has no op equivalent: the recording is
// marked failed and the caller falls back to direct launches / a CUDA graph.
#define PE_LAUNCHED(ctx)                                     \
    do {                                                     \
        (ctx)->launches++;                                   \
        if ((ctx)->rec) pe_rec_fail((ctx), __FILE__, __LINE__); \
        PE_CUDA(cudaPeekAtLastError());                      \
    } while (0)

// ---- persistent "program" kernel (pe_prog.cu): the ops a recorded V-cycle is made of
enum PeOpType : int32_t {
    PE_OP_SELL_SPMV = 1, PE_OP_SELL_GS, PE_OP_CSR_SPMV, PE_OP_PERM_IN, PE_OP_PERM_OUT, PE_OP_AXPBY, PE_OP_ADD3,
    PE_OP_FILL, PE_OP_COPY, PE_OP_SCALE, PE_OP_MUL, PE_OP_DOT, PE_OP_DOT_FIN, PE_OP_AXPY_DEV, PE_OP_XPBY_DEV,
    PE_OP_PCG_STEP, PE_OP_PERM_IN_GS0
};
struct PeOp {               // 128 bytes, copied to shared memory by the interpreter
    int32_t type, i0, i1, i2, i3, i4, i5, flags;
    int64_t n;
    double a, b;
    const void *p[9];
};
struct pe_recorder {
    std::vector<PeOp> ops;
    std::vector<double> bytes;     // algorithmic bytes per op (DESIGN.md)
    bool failed = false;
    std::string why;
};
struct pe_ctx;
void pe_rec_fail(pe_ctx *ctx, const char *file, int line);

struct pe_ctx {
    int rank = 0, nranks = 1, device = 0;
    cudaStream_t stream = nullptr;       // compute stream
    cudaStream_t comm_stream = nullptr;  // halo exchange stream
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;
    cudaEvent_t ev_pack = nullptr, ev_halo = nullptr;
    void *nccl = nullptr;                // ncclComm_t (opaque; resolved by dlopen)
    int64_t launches = 0;
    double *partials_d = nullptr;        // reduction scratch (PE_MAX_PARTIALS doubles)
    double *scalar_d = nullptr;          // 8 device scalars
    double *scalar_h = nullptr;          // pinned host mirror
    void *flush_d = nullptr;
    size_t flush_bytes = 0;
    bool capturing = false;
    pe_recorder *rec = nullptr;          // non-null while a program is being recorded
    double pending_bytes = 0.0;          // algorithmic bytes announced by the last pe_prof_begin
    const struct pe_host_comm *hcomm = nullptr;   // setup-time host communicator (borrowed)
    // peer-visible halo arena (pe_p2p.cu): my block and every rank's block mapped through CUDA IPC
    char *p2p_base = nullptr;
    size_t p2p_size = 0, p2p_used = 0;
    std::vector<char *> p2p_peer;
    // optional per-kernel CUDA-event profiling (bench.py roofline): id 0 SpMV, 1 GS set, 2 Jacobi
    bool prof = false;
    struct ProfRec { int id; double bytes; cudaEvent_t e0, e1; };
    std::vector<ProfRec> prof_recs;
    std::vector<cudaEvent_t> prof_pool;
    double prof_ms[4] = {0, 0, 0, 0}, prof_bytes[4] = {0, 0, 0, 0};
    long long prof_count[4] = {0, 0, 0, 0};
};
// record an op instead of launching (returns true when ctx is recording)
// bytes < 0: use the figure announced by the enclosing pe_prof_begin
static inline bool pe_rec_push(pe_ctx *ctx, const PeOp &op, double bytes)
{
    if (!ctx->rec) return false;
    ctx->rec->ops.push_back(op);
    ctx->rec->bytes.push_back(bytes < 0.0 ? ctx->pending_bytes : bytes);
    ctx->pending_bytes = 0.0;
    return true;
}
static inline PeOp pe_op(int32_t type)
{
    PeOp o{};
    o.type = type;
    return o;
}
// ---- programmatic dependent launch (PDL).  A kernel launched through pe_launch_k may start while
// its predecessor on the stream is still draining: everything it does before pdl_wait() must touch
// only data no kernel of the sequence writes (matrix arrays, index lists, l1 norms); pdl_wait()
// returns once the predecessor has completed and its writes are visible.  Every kernel launched
// this way executes pdl_wait() in at least one thread, so completion stays transitive along the
// stream.  Without the launch attribute both instructions are no-ops.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
template <typename... KArgs, typename... Args>
static inline cudaError_t pe_launch_k(pe_ctx *ctx, void (*kern)(KArgs...), int grid, int block, Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid, 1, 1);
    cfg.blockDim = dim3((unsigned)block, 1, 1);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute at[1];
    // multi-rank: only when the halo exchange is made of ordinary kernels (peer-memory path); the NCCL path forks to
    // a communication stream with events around its launches
    if ((ctx->nranks == 1 || ctx->p2p_base) && pe_get_tuning(PE_TUNE_PDL) != 0)
    {
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
    }
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}
#endif
int pe_prof_begin(pe_ctx *ctx, int id, double bytes);
int pe_prof_end(pe_ctx *ctx);
#define PE_MAX_PARTIALS 4096

// sliced-ELL copy of a CSR block (pe_sell.cu): slices of 32 rows, column-major inside a slice
struct DevSELL {
    int32_t nslices = 0, nrows = 0;   // nrows: rows that receive output (<= nslices*32)
    int32_t wmax = 0;                 // widest slice (selects the entry-group size of the kernels)
    int64_t nstored = 0;              // stored entries incl. padding
    int32_t *soff = nullptr;          // nslices+1 slice offsets, in units of 32 entries
    int32_t *J = nullptr;
    double *A = nullptr;              // null when the values are sign-encoded
    int8_t *S = nullptr;              // SpMV copies whose values are all -1, 0 or +1 (discrete derivatives): 1 B per entry
};

struct DevCSR {
    int32_t nrows = 0, ncols = 0;
    int64_t nnz = 0;
    int32_t *I = nullptr, *J = nullptr;
    double *A = nullptr;
    // row blocks of the streaming kernels: block b owns rows [rb[b], rb[b+1]) holding <= PE_STREAM_CAP
    // non-zeros (built lazily; nrb == -1: matrix has rows too long for the streaming kernel)
    int32_t *rb = nullptr;
    int32_t nrb = 0;
    // SELL-32 copy streamed by SpMV (built lazily; state 0 untested, 1 built, -1 rejected: too much padding)
    DevSELL *sell = nullptr;
    int sell_state = 0;
};
void pe_sell_free(DevSELL &m);
int pe_sell_build(pe_ctx *ctx, const DevCSR &diag, const DevCSR *offd, const int32_t *rowmap_d, int32_t nslices,
                  const int32_t *colpos_d, int32_t ext_base, DevSELL &out,
                  std::vector<int32_t> *soff_host = nullptr);
int pe_sell_for_spmv(pe_ctx *ctx, DevCSR &m, bool force = false);
void pe_mat_values_changed(struct pe_mat *A);   // drop cached transposes / SELL copies after an in-place edit
int pe_launch_sell_spmv(pe_ctx *ctx, const DevSELL &S, double alpha, const double *x, double beta,
                        const double *yin, double *yout);
int pe_launch_sell_gs(pe_ctx *ctx, const DevSELL &S, int s0, int s1, int wmax, int ext_base, const double *f, double *u,
                      const double *uext, const double *l1, uint64_t pol_gather);
// L2 cache policy word for the u-gathers: keep_pct % of the lines evict_last, the rest unchanged (0: evict_normal)
int pe_make_gather_policy(pe_ctx *ctx, int keep_pct, uint64_t *pol);
int pe_launch_perm_in(pe_ctx *ctx, int n, const int *pos, const double *b, const double *x, double *fp, double *up);
int pe_launch_perm_out(pe_ctx *ctx, int n, const int *pos, const double *up, double *x);
int pe_launch_perm_in_gs0(pe_ctx *ctx, int n, const int *pos, const double *b, int r0, int r1, const double *l1,
                          double *fp, double *up);
#define PE_STREAM_NNZ 2048      // target non-zeros per CTA
#define PE_STREAM_CAP 2560      // shared-memory capacity (target + longest admissible row)
#define PE_STREAM_MAXROW 512
int pe_build_row_blocks(pe_ctx *ctx, DevCSR &m, const std::vector<int32_t> *forced_breaks);
int devcsr_alloc(DevCSR &m, int32_t nrows, int32_t ncols, int64_t nnz);
void devcsr_free(DevCSR &m);

struct pe_vec {
    pe_ctx *ctx;
    int64_t n;
    double *d;
    bool view = false;      // aliases another vector's buffer (pe_vec_view)
};

struct pe_mat {
    pe_ctx *ctx = nullptr;
    int64_t global_num_rows = 0, global_num_cols = 0, first_row_index = 0, first_col_diag = 0;
    DevCSR diag, offd;
    std::vector<int64_t> col_map_offd;
    // comm package (host copies + device send map)
    std::vector<int32_t> send_procs, send_map_starts, send_map_elmts, recv_procs, recv_vec_starts;
    int32_t *send_map_d = nullptr;
    double *send_buf_d = nullptr;
    double *x_ext_d = nullptr;
    pe_mat *T = nullptr;     // cached explicit transpose (owned); distributed: transpose of the diag block
    int tpr = 0;             // threads per row chosen for SpMV (power of two <= 32)
    // multi-rank: rows/columns are a slice of a global matrix (set at upload)
    bool distributed = false;
    DevCSR offdT;            // transpose of the offd block (ghost col x local row), built on first MatvecT
    bool offdT_built = false, unpack_built = false;
    int n_unpack = 0;        // reverse exchange: distinct target rows, CSR of receive-buffer slots per row
    int *unpack_rows_d = nullptr, *unpack_I_d = nullptr, *unpack_pos_d = nullptr;
    // peer-memory halo exchange (pe_p2p.cu): 0 = not linked yet, 1 = linked, -1 = NCCL path
    int p2p_state = 0;
    struct PeP2PDir *p2p[2] = {nullptr, nullptr};   // forward (ghost fill), reverse (MatvecT partial sums)
};
int pe_p2p_init(pe_ctx *ctx);
void pe_p2p_shutdown(pe_ctx *ctx);
void *pe_p2p_alloc(pe_ctx *ctx, size_t bytes);
bool pe_p2p_owns(const pe_ctx *ctx, const void *p);
int pe_p2p_link(pe_mat *A);
void pe_p2p_unlink(pe_mat *A);
int pe_p2p_push(pe_mat *A, int dir, const double *src);
int pe_p2p_wait(pe_mat *A, int dir);
int pe_rap_distributed(pe_ctx *ctx, const pe_mat *R, const pe_mat *A, const pe_mat *P, pe_mat **Ac);
int pe_spgemm_distributed(pe_ctx *ctx, const pe_mat *A, const pe_mat *B, pe_mat **C);
int pe_transpose_distributed(pe_ctx *ctx, const pe_mat *A, pe_mat **out);
int pe_spadd_distributed(pe_ctx *ctx, double a, const pe_mat *A, double b, const pe_mat *B, pe_mat **out);
int pe_spmv_t_distributed(pe_ctx *ctx, double alpha, pe_mat *A, const pe_vec *x, double beta, pe_vec *y);
int pe_launch_unpack_add(pe_ctx *ctx, pe_mat *A, double alpha, double *y_d);
int pe_reverse_halo_add(pe_mat *A, double alpha, double *y_d);

// ---- internal helpers used across translation units
int pe_halo_exchange(pe_mat *A, const double *x_d);   // fills A->x_ext_d (no-op single rank)
int pe_halo_wait(pe_mat *A);                           // compute stream waits for halo
int pe_devcsr_transpose(pe_ctx *ctx, const DevCSR &A, DevCSR &T);
int pe_devcsr_spgemm(pe_ctx *ctx, const DevCSR &A, const DevCSR &B, DevCSR &C);
int pe_choose_tpr(int64_t nnz, int32_t nrows);
void pe_variant_add(int slot, int64_t count);   // pe_variant_counts: rows / agglomerates handed to one kernel variant
int pe_mat_wrap_local(pe_ctx *ctx, DevCSR &diag, pe_mat **out);  // takes ownership of diag
int pe_allreduce_sum(pe_ctx *ctx, double *d, int count);

// spmv launcher on raw pointers: yout = alpha*(diag*x + offd*xext) + beta*yin
int pe_launch_spmv(pe_ctx *ctx, const DevCSR &diag, const DevCSR *offd, int tpr,
                   double alpha, const double *x, const double *xext,
                   double beta, const double *yin, double *yout);

static inline int pe_grid_for(int64_t work_items, int per_block)
{
    int64_t g = (work_items + per_block - 1) / per_block;
    if (g < 1) g = 1;
    return (int)g;
}
