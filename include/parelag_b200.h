/*
 * parelag_b200.h -- C ABI of the B200-native AMGe solve-and-coarsen path.
 *
 * This is the drop-in boundary (SURVEY.md 8b): plain pointers and sizes, no C++ or
 * torch types.  ParElag's C++ classes (re-created under parelag_b200/src with the
 * reference's names and signatures) call these functions from Mult()/BuildSolver();
 * a maintainer of the reference would call them from the same places -- see
 * INTEGRATION.md.  Every entry point names the reference interface it replaces
 * (paths relative to the reference tree).
 *
 * Conventions
 *   - all functions return 0 on success, non-zero on error; pe_last_error() returns
 *     the message of the last failing call on this thread.  No exception crosses
 *     the ABI.
 *   - pointers are HOST pointers unless the parameter is an opaque handle;
 *     handles own device memory (HBM) and are freed by the matching *_free.
 *   - HYPRE_Int is 32-bit in all reference usage (src/hypreExtension/parcsr-add.c:32-41):
 *     indices are int32, values are FP64, global ids are int64.
 *   - work is enqueued on the context's stream; calls that return host scalars or
 *     copy to host synchronise that stream.
 *   - there is NO CPU fallback: if no CUDA device is usable pe_ctx_create fails.
 */
#ifndef PARELAG_B200_H
#define PARELAG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pe_ctx pe_ctx;             /* device, streams, NCCL communicator    */
typedef struct pe_mat pe_mat;             /* device ParCSR matrix (diag+offd+halo) */
typedef struct pe_vec pe_vec;             /* device FP64 vector                    */
typedef struct pe_smoother pe_smoother;   /* hypre-type relaxation on one matrix   */
typedef struct pe_graph pe_graph;         /* captured CUDA graph                   */

/* Host-side description of a ParCSR matrix: the fields of hypre_ParCSRMatrix the
 * path reads (hypre_ParCSRMatrixMatvecBoolInt.c:148-196, parcsr-add.c:31-41,
 * hypre_CSRFactory.c:186-247).  All arrays are borrowed for the duration of the
 * call only.  A single-rank matrix has num_cols_offd = 0 and no comm package. */
typedef struct pe_parcsr_host {
    int64_t global_num_rows, global_num_cols;
    int64_t first_row_index, first_col_diag;
    int32_t num_rows;         /* local rows                                   */
    int32_t num_cols_diag;    /* local (owned) columns                        */
    int32_t num_cols_offd;    /* ghost columns                                */
    const int32_t *diag_i, *diag_j;
    const double *diag_data;
    const int32_t *offd_i, *offd_j;      /* may be NULL when num_cols_offd==0 */
    const double *offd_data;
    const int64_t *col_map_offd;         /* global ids, ascending             */
    /* hypre_ParCSRCommPkg */
    int32_t num_sends;
    const int32_t *send_procs, *send_map_starts, *send_map_elmts;
    int32_t num_recvs;
    const int32_t *recv_procs, *recv_vec_starts;
} pe_parcsr_host;

/* ---- context (replaces parelag::mpi_session, src/utilities/mpiUtils.cpp:23-31) */
/* nccl_unique_id: 128 bytes from pe_nccl_get_unique_id on rank 0 (broadcast by the
 * launcher), or NULL when nranks == 1. */
int pe_ctx_create(int rank, int nranks, int device, const void *nccl_unique_id, pe_ctx **out);
int pe_ctx_destroy(pe_ctx *ctx);
int pe_ctx_sync(pe_ctx *ctx);
int pe_nccl_get_unique_id(void *id128);
const char *pe_last_error(void);
int pe_ctx_rank(const pe_ctx *ctx);
int pe_ctx_nranks(const pe_ctx *ctx);
/* 1 when the halo exchange of this context goes through NVLink peer memory (PE_TUNE_P2P_HALO), 0 = NCCL send/recv */
int pe_ctx_p2p_enabled(const pe_ctx *ctx);
/* number of kernels this library has launched on ctx since creation */
int64_t pe_ctx_launch_count(const pe_ctx *ctx);
/* stream-ordered CUDA-event timer on the context's stream (milliseconds) */
int pe_ctx_timer_start(pe_ctx *ctx);
int pe_ctx_timer_stop(pe_ctx *ctx, float *ms);
/* per-kernel CUDA-event profiling on the context's stream (roofline in bench.py): enable=1
 * resets and starts, 0 stops.  kernel ids: 0 = SpMV (all variants), 1 = k_sell_gs colour launches of the
 * bandwidth-bound class (>= 64 MB algorithmic bytes: the fine level), 2 = Jacobi update, 3 = the other
 * Gauss-Seidel launches (coarse levels: k_gs_set<TPR>, small k_sell_gs).  total_bytes = algorithmic bytes
 * of the launches (DESIGN.md). */
int pe_ctx_profile(pe_ctx *ctx, int enable);
int pe_ctx_profile_get(pe_ctx *ctx, int kernel_id, int64_t *count, double *total_ms, double *total_bytes);
/* process-wide tuning knobs (tests force either kernel family; defaults in brackets):
 * PE_TUNE_SELL_MIN_ROWS [200000]: multicolour Gauss-Seidel uses the colour-ordered SELL-32 streaming
 * kernel for matrices with at least this many rows and the lanes-per-row CSR kernel below it.
 * PE_TUNE_SELL_GROUP [0]: entries per load group of the SELL kernels (0 = chosen from the slice widths;
 * 4, 8 or 12 forces one).  Results do not depend on it (the summation order of a row is fixed).
 * PE_TUNE_PDL [1]: launch the solve-path kernels with programmatic stream serialization (single rank, and
 * multi-rank when the halo exchange runs over peer memory):
 * the matrix prologue of a kernel overlaps the tail of its predecessor.
 * PE_TUNE_GATHER_KEEP_PCT [0]: percentage (0, 25, 50, 60, 75, 90, 100) of the u-gather lines of the SELL
 * Gauss-Seidel kernel that get L2 priority evict_last (the rest evict_unchanged); 0 = normal priority.
 * The colour-ordered iterate is re-read by every colour launch while 30-50x its size streams through
 * L2; keeping a fixed fraction resident turns an all-miss cyclic pattern into that fraction of hits.
 * Read when a smoother is created.
 * PE_TUNE_P2P_HALO [1]: multi-rank, one node: ParCSR halo exchange by direct stores into the neighbours' ghost
 * buffers over NVLink peer memory (CUDA IPC) with device-side arrival flags instead of ncclSend/ncclRecv.
 * Read at pe_ctx_set_host_comm; falls back to NCCL when a rank cannot map a peer.
 * PE_TUNE_FUSED_GS_MAX_MB [0 = off]: a multicolour Gauss-Seidel sweep whose LARGEST colour moves fewer algorithmic megabytes
 * than this runs as ONE persistent kernel (all colours of the forward and backward pass, grid barriers in between, the
 * colour-order renumbering of the SELL path included) instead of one launch per colour.  Results are bit-identical (same
 * rows, same summation order).  Measured on B200 (profiles/README.md, round 2): inside the CUDA graph with programmatic
 * dependent launch a colour launch costs ~2.5 us, a grid-barrier step ~4.2 us -- the V-cycle got slower (7.46 -> 8.29 ms
 * at 24 MB), so the default is off; the kernels stay for devices / drivers where launches are dearer.
 * Read when a smoother is created.
 * PE_TUNE_GS_SLABS [0 = off]: multicolour Gauss-Seidel on matrices with at least 4 million rows: the rows are cut into this
 * many contiguous pieces of the matrix graph (breadth-first levels from row 0, equal row counts) and the sweep visits
 * (slab 0: colours 0..C-1), (slab 1: colours 0..C-1), ... -- still Gauss-Seidel in an order made of independent sets.
 * The idea: the iterate of one slab stays in L2 across its C colour launches instead of being re-read from HBM by
 * every colour (each colour gathers (C-1)/C of the vector: the 1.2x DRAM traffic over the algorithmic bytes).  Measured
 * (round 2): 4 slabs 9.38 ms, 8 slabs 9.76 ms against 7.46 ms -- the smaller launches cost more than the gathers save
 * and the L2 hit rate of the gathers did not rise; default off.  Read when a smoother is created.
 * PE_TUNE_LOCAL_SMEM_BYTES [0 = built-in limits]: workspace bytes above which an agglomerate of the batched local solves
 * of Coarsen() leaves shared memory for a global-memory slab (k_traces_gmem, k_extension_gmem).  The built-in limits are
 * 200 KB (traces) and 220 KB (extension); a value > 0 replaces both and is clamped to them, so 1 sends every
 * agglomerate to the global-memory kernels.  Results do not depend on it (same arithmetic, same order). */
enum { PE_TUNE_SELL_MIN_ROWS = 0, PE_TUNE_SELL_GROUP = 1, PE_TUNE_PDL = 2, PE_TUNE_GATHER_KEEP_PCT = 3, PE_TUNE_P2P_HALO = 4,
       PE_TUNE_FUSED_GS_MAX_MB = 5, PE_TUNE_GS_SLABS = 6, PE_TUNE_LOCAL_SMEM_BYTES = 7, PE_TUNE_COUNT = 8 };
int pe_set_tuning(int key, int value);
int pe_get_tuning(int key);
/* process-wide counts of the work each size-dispatched kernel variant was given, kept on the host at the place that
 * chooses the variant (no device work, no synchronisation).  Units: rows for SpMV (per call), SpGEMM (per bin of the
 * symbolic / numeric pass) and relaxation (per launch of k_jacobi_update<TPR> / k_gs_set<TPR>), agglomerates for the
 * batched local solves.  An operation recorded into a persistent program or captured into a CUDA graph counts once,
 * when it is recorded.  Three slots refine the local solves: EXT_SPLIT_SMEM counts the agglomerates of the listed
 * shared-memory extension launch of a batch split between both kernels (also counted in EXT_SMEM); TRACES_GMEM_REUSE and
 * EXT_GMEM_REUSE count the agglomerates a global-workspace CTA takes after its first one (a launch with more agglomerates
 * than CTAs reuses each workspace slab).  SPMV_SELL_SIGNS counts the rows of SELL SpMVs whose values are stored as int8
 * sign codes (every value -1, 0 or +1; also counted in SPMV_SELL).  SELL_GS_* and SELL_SPMV_* count the entry-group variant
 * of each k_sell_gs (one colour of a multicolour sweep) and k_sell_spmv launch: G = 4, 8 or 12 entries per group, SINGLE
 * when every slice of the launch fits one group, PIPE otherwise; the unit is padded slice rows (32 per slice of the
 * launch, padding rows of a partly filled slice included).  Recording a persistent program pushes an op and picks no
 * variant, so it counts nothing; capturing a CUDA graph counts once, at capture, and a replay counts nothing.
 * out: n slots (slots past PE_VARIANT_COUNT are set to 0; NULL with n = 0 copies nothing);
 * reset != 0 zeroes every counter after the copy. */
enum { PE_VARIANT_SPMV_SELL = 0, PE_VARIANT_SPMV_STREAM = 1, PE_VARIANT_SPMV_VECTOR = 2,
       PE_VARIANT_SPGEMM_SYM_T128 = 3, PE_VARIANT_SPGEMM_SYM_T1024 = 4, PE_VARIANT_SPGEMM_SYM_T8192 = 5, PE_VARIANT_SPGEMM_SYM_GMEM = 6,
       PE_VARIANT_SPGEMM_NUM_T128 = 7, PE_VARIANT_SPGEMM_NUM_T1024 = 8, PE_VARIANT_SPGEMM_NUM_T8192 = 9, PE_VARIANT_SPGEMM_NUM_GMEM = 10,
       PE_VARIANT_RELAX_TPR_1 = 11, PE_VARIANT_RELAX_TPR_2 = 12, PE_VARIANT_RELAX_TPR_4 = 13, PE_VARIANT_RELAX_TPR_8 = 14,
       PE_VARIANT_RELAX_TPR_16 = 15, PE_VARIANT_RELAX_TPR_32 = 16,
       PE_VARIANT_TRACES_SMEM = 17, PE_VARIANT_TRACES_GMEM = 18, PE_VARIANT_EXT_SMEM = 19, PE_VARIANT_EXT_GMEM = 20,
       PE_VARIANT_EXT_SPLIT_SMEM = 21, PE_VARIANT_TRACES_GMEM_REUSE = 22, PE_VARIANT_EXT_GMEM_REUSE = 23,
       PE_VARIANT_SPMV_SELL_SIGNS = 24,
       PE_VARIANT_SELL_GS_G4_SINGLE = 25, PE_VARIANT_SELL_GS_G4_PIPE = 26, PE_VARIANT_SELL_GS_G8_SINGLE = 27,
       PE_VARIANT_SELL_GS_G8_PIPE = 28, PE_VARIANT_SELL_GS_G12_SINGLE = 29, PE_VARIANT_SELL_GS_G12_PIPE = 30,
       PE_VARIANT_SELL_SPMV_G4_SINGLE = 31, PE_VARIANT_SELL_SPMV_G4_PIPE = 32, PE_VARIANT_SELL_SPMV_G8_SINGLE = 33,
       PE_VARIANT_SELL_SPMV_G8_PIPE = 34, PE_VARIANT_SELL_SPMV_G12_SINGLE = 35, PE_VARIANT_SELL_SPMV_G12_PIPE = 36,
       PE_VARIANT_COUNT = 37 };
int pe_variant_counts(int64_t *out, int n, int reset);
/* write a scratch buffer larger than L2 (bench hygiene) */
int pe_ctx_flush_l2(pe_ctx *ctx);

/* ---- CUDA graphs (Hierarchy::Mult replays a captured V-cycle) */
int pe_graph_begin(pe_ctx *ctx);
int pe_graph_end(pe_ctx *ctx, pe_graph **out);
int pe_graph_launch(pe_ctx *ctx, pe_graph *g);
int pe_graph_free(pe_graph *g);

/* ---- persistent programs: a recorded sequence of solve-path operations (a whole
 * Hierarchy::Mult V-cycle) executed by ONE cooperative kernel, one CTA per SM, with
 * grid-wide barriers between the operations instead of kernel boundaries.
 * Between pe_program_begin and pe_program_end the solve-path entry points (pe_spmv,
 * pe_residual, pe_smoother_apply, pe_vec_*, pe_pcg_scalar_step ...) record instead of
 * executing; pe_program_end fails (non-zero) when an operation without a program
 * equivalent was requested -- the caller then falls back to a CUDA graph.
 * pe_program_profile runs the program once with a device timestamp after every barrier. */
typedef struct pe_program pe_program;
int pe_program_begin(pe_ctx *ctx);
int pe_program_end(pe_ctx *ctx, pe_program **out);
int pe_program_launch(pe_ctx *ctx, pe_program *p);
int pe_program_free(pe_program *p);
int pe_program_info(const pe_program *p, int32_t *nops, double *algorithmic_bytes);
int pe_program_profile(pe_ctx *ctx, pe_program *p, int32_t *op_types, double *op_usec, double *op_bytes);
int pe_ctx_is_recording(const pe_ctx *ctx);

/* ---- vectors (replace mfem::Vector on the path) */
int pe_vec_create(pe_ctx *ctx, int64_t n, pe_vec **out);
int pe_vec_free(pe_vec *v);
/* non-owning view of n entries of base starting at offset (block vectors, mfem::BlockVector::GetBlock);
 * free it with pe_vec_free before the base */
int pe_vec_view(const pe_vec *base, int64_t offset, int64_t n, pe_vec **out);
int64_t pe_vec_size(const pe_vec *v);
int pe_vec_upload(pe_vec *v, const double *host);       /* n doubles, H2D   */
int pe_vec_download(const pe_vec *v, double *host);     /* n doubles, D2H   */
int pe_vec_fill(pe_vec *v, double value);
int pe_vec_copy(const pe_vec *src, pe_vec *dst);
int pe_vec_axpby(double a, const pe_vec *x, double b, pe_vec *y);          /* y=a x+b y */
int pe_vec_add3(double a, const pe_vec *x, double b, const pe_vec *y, pe_vec *z); /* z=a x+b y */
int pe_vec_scale(pe_vec *x, double a);
int pe_vec_mul(const pe_vec *d, pe_vec *x);                                 /* x .*= d */
/* global dot (sum over ranks via ncclAllReduce); deterministic two-stage reduce.
 * Replaces mfem::CGSolver::Dot / MPI_Allreduce (ParELAG_StationarySolver.cpp:64). */
int pe_vec_dot(const pe_vec *x, const pe_vec *y, double *out);
/* Device-resident scalars: short inner Krylov solves (the AMGe coarse solver) keep every
 * scalar of the recurrence in HBM so that no host synchronisation interrupts the V-cycle and
 * the whole cycle can be replayed as one CUDA graph.  pe_scalars_* manage a block of doubles;
 * the *_dev variants read/write one of its slots.
 *   pe_vec_dot_dev : slots[out_slot] = <x,y> (all ranks)
 *   pe_vec_axpy_dev: y += sign * slots[a_slot] * x      (no-op when the scalar is 0)
 *   pe_vec_xpby_dev: y  = x + slots[b_slot] * y
 *   pe_pcg_scalar_step: the scalar part of one phase of mfem::CGSolver::Mult (same tests and
 *     formulas as the host loop in parelag_solvers.hpp); after convergence or breakdown the step
 *     lengths become 0, so the remaining fixed-trip iterations leave x unchanged.
 *     slot layout: PE_PCG_* below; history of (B r, r) starts at PE_PCG_HIST. */
enum { PE_PCG_DOT = 0, PE_PCG_NOM = 1, PE_PCG_DEN = 2, PE_PCG_BETANOM = 3, PE_PCG_ALPHA = 4, PE_PCG_BETA = 5,
       PE_PCG_R0 = 6, PE_PCG_DONE = 7, PE_PCG_CONVERGED = 8, PE_PCG_FINAL_ITER = 9, PE_PCG_NOM0 = 10,
       PE_PCG_NHIST = 11, PE_PCG_HIST = 16 };
int pe_scalars_create(pe_ctx *ctx, int count, double **slots_d);
int pe_scalars_free(double *slots_d);
int pe_scalars_download(pe_ctx *ctx, const double *slots_d, int count, double *host);
int pe_vec_dot_dev(const pe_vec *x, const pe_vec *y, double *slots_d, int out_slot);
int pe_vec_axpy_dev(const double *slots_d, int a_slot, double sign, const pe_vec *x, pe_vec *y);
int pe_vec_xpby_dev(const pe_vec *x, const double *slots_d, int b_slot, pe_vec *y);
int pe_pcg_scalar_step(pe_ctx *ctx, double *slots_d, int phase, int iter, int max_iter, double rel_tol, double abs_tol);
/* non-zero while a CUDA graph is being captured / while per-kernel profiling is on */
int pe_ctx_is_capturing(const pe_ctx *ctx);
int pe_ctx_is_profiling(const pe_ctx *ctx);
/* raw device pointer, for callers that own a CUDA stream themselves */
void *pe_vec_device_ptr(pe_vec *v);

/* ---- matrices (ParCSR in/out; replaces mfem::HypreParMatrix on the path) */
int pe_mat_upload(pe_ctx *ctx, const pe_parcsr_host *A, pe_mat **out);
/* query sizes, then download into caller-allocated arrays (NULL = skip) */
int pe_mat_info(const pe_mat *A, int32_t *num_rows, int32_t *num_cols_diag,
                int32_t *num_cols_offd, int64_t *nnz_diag, int64_t *nnz_offd);
int pe_mat_global_info(const pe_mat *A, int64_t *global_num_rows, int64_t *global_num_cols,
                       int64_t *first_row_index, int64_t *first_col_diag);
int pe_mat_download(const pe_mat *A, int32_t *diag_i, int32_t *diag_j, double *diag_data,
                    int32_t *offd_i, int32_t *offd_j, double *offd_data,
                    int64_t *col_map_offd);
int pe_mat_free(pe_mat *A);
/* copy of a single-rank matrix: its row pointers, columns and values (no cached transpose or SELL copy) */
int pe_mat_clone(pe_ctx *ctx, const pe_mat *A, pe_mat **out);
/* explicit local transpose (counting-sort order: ascending columns per row).
 * mfem::Transpose / hypre_ParCSRMatrixTranspose2 (src/hypreExtension/par_Tmatmul.c:41-79) */
int pe_mat_transpose(pe_ctx *ctx, const pe_mat *A, pe_mat **out);
/* diag(A) and inverse-scaled rows (SchurComplementFactory.cpp:51-166 InvScaleRows) */
int pe_mat_get_diag(const pe_mat *A, pe_vec *d);
int pe_mat_scale_rows(pe_mat *A, const pe_vec *d, int invert);
/* A *= a (HypreParMatrix::operator*=, Block2x2JacobiSolverFactory.cpp:86-91); d_i = sum_j |a_ij| over
 * diag and offd ("ABSROWSUM", SchurComplementFactory.cpp:70-96) */
int pe_mat_scale(pe_mat *A, double a);
int pe_mat_abs_row_sums(const pe_mat *A, pe_vec *d);

/* ---- K1/K2/K7: SpMV, SpMV^T, residual
 * y = alpha*A*x + beta*y : hypre_ParCSRMatrixMatvec via mfem::HypreParMatrix::Mult,
 *   src/linalg/solver_ops/ParELAG_Hierarchy.cpp:193,234.
 * y = alpha*A^T*x + beta*y : hypre_ParCSRMatrixMatvecT via P->MultTranspose,
 *   Hierarchy.cpp:202, HiptmairSmoother.cpp:63.  The explicit transpose is built
 *   on first use and cached on A (no atomics on the solve path).
 * r = b - A*x : mg_utils::ComputeResidual, src/linalg/utilities/ParELAG_MG_Utils.hpp:405-467. */
int pe_spmv(pe_ctx *ctx, double alpha, pe_mat *A, const pe_vec *x, double beta, pe_vec *y);
int pe_spmv_t(pe_ctx *ctx, double alpha, pe_mat *A, const pe_vec *x, double beta, pe_vec *y);
int pe_residual(pe_ctx *ctx, pe_mat *A, const pe_vec *x, const pe_vec *b, pe_vec *r);
/* Renumbered copy of A (transpose != 0: of A^T) for products on vectors in other numberings, single rank: row i of A
 * becomes row rpos[i] of a matrix of nrows_out rows, column j becomes column cpos[j] of ncols_out; NULL keeps the
 * natural numbering of that side.  rpos / cpos are device arrays, e.g. the colour numbering of
 * pe_smoother_colour_numbering.  Each row keeps its entries, their order, and A's SpMV format, so every mapped entry
 * of a product equals the natural product's bit for bit; rows no row of A maps to are empty (their result is
 * beta * y).  Free with pe_mat_free. */
int pe_mat_renumbered(pe_ctx *ctx, pe_mat *A, int transpose, const int32_t *rpos, int32_t nrows_out,
                      const int32_t *cpos, int32_t ncols_out, pe_mat **out);
/* Values only: R, made by pe_mat_renumbered(ctx, B, 0, rpos, ...) from a matrix B with A's pattern, takes A's values
 * (the same row map rpos); its pattern is kept and its products equal those of pe_mat_renumbered(A) bit for bit. */
int pe_mat_renumbered_values(pe_ctx *ctx, pe_mat *A, const int32_t *rpos, pe_mat *R);
/* *same = 1 when A and B (single rank) have the same sizes, row pointers and column indices: one device pass, one
 * flag downloaded */
int pe_mat_same_pattern(pe_ctx *ctx, const pe_mat *A, const pe_mat *B, int32_t *same);

/* ---- K3/K4/K5: hypre relaxation (mfem::HypreSmoother behind
 * parelag::HypreSmootherWrapper, src/linalg/solver_ops/ParELAG_HypreSmootherWrapper.cpp:20-35;
 * type ids as in src/linalg/factories/ParELAG_HypreSmootherFactory.cpp:92-109:
 * 0 Jacobi, 1 l1-Jacobi, 2 l1-GS, 4 truncated l1-GS, 5 lumped Jacobi, 6 GS, 16 Chebyshev).
 * ordering: how the sequential Gauss-Seidel order of hypre is realised on the GPU */
enum { PE_GS_ORDER_NATURAL = 0,     /* exact natural row order via level scheduling */
       PE_GS_ORDER_MULTICOLOR = 1   /* greedy first-fit colouring, colour by colour  */ };
int pe_smoother_create(pe_ctx *ctx, pe_mat *A, int type, int sweeps, double damping,
                       double omega, int cheby_order, double cheby_fraction,
                       int gs_ordering, pe_smoother **out);
/* x <- smoothed x (iterative_mode != 0) or smoother applied to zero initial guess */
int pe_smoother_apply(pe_smoother *s, const pe_vec *b, pe_vec *x, int iterative_mode);
int pe_smoother_free(pe_smoother *s);
/* introspection for parity tests: l1 norms, GS row order (sets concatenated),
 * number of sets, Chebyshev eigenvalue estimates */
int pe_smoother_get_l1(const pe_smoother *s, double *l1_host);
int pe_smoother_get_order(const pe_smoother *s, int32_t *order_host, int32_t *num_sets,
                          int32_t *set_starts_host /* num_sets+1, may be NULL */);
int pe_smoother_get_eig(const pe_smoother *s, double *max_eig, double *min_eig);
/* Colour numbering of a multicolour SELL Gauss-Seidel smoother (one rank): *npad = padded length of the colour-ordered
 * vectors, *pos_d = device array row -> position (owned by the smoother).  *npad = 0 and *pos_d = NULL when the
 * smoother has no such numbering (other types, CSR path, fused sweeps). */
int pe_smoother_colour_numbering(const pe_smoother *s, int32_t *npad, const int32_t **pos_d);
/* The smoother on colour-numbered vectors f, u of npad entries, no renumbering passes.  Padding entries of f must be 0;
 * those of u stay 0.  mode 0: u holds the initial guess; 1: zero initial guess (u's content is ignored); 2: u is what
 * pe_smoother_colour_in left (the first colour of a sweep from a zero guess is done). */
int pe_smoother_apply_colour(pe_smoother *s, const pe_vec *f, pe_vec *u, int mode);
/* b (natural) -> f (colour order) and u = the first colour of a sweep from a zero guess, in one pass; then
 * pe_smoother_apply_colour(mode 2).  pe_smoother_colour_out: x (natural) = u (colour order). */
int pe_smoother_colour_in(pe_smoother *s, const pe_vec *b, pe_vec *f, pe_vec *u);
int pe_smoother_colour_out(pe_smoother *s, const pe_vec *u, pe_vec *x);
/* New values for a smoother (mfem::Solver::SetOperator on a built HypreSmootherWrapper): A (borrowed) must have the
 * size and sparsity pattern of the smoother's matrix, else the call fails and changes nothing.  The smoother then
 * works on A, with everything recomputed that a pe_smoother_create on A would compute from the values (l1 norms,
 * diagonal, the values of its set-ordered CSR / colour-ordered SELL copy, Chebyshev bounds and coefficients), and
 * with its colouring, level sets, copy layouts and colour numbering (pos_d) kept. */
int pe_smoother_update(pe_smoother *s, pe_mat *A);

/* ---- K8/K9: sparse products
 * C = A*B (mfem::ParMult / hypre_ParMatmul; SchurComplementFactory.cpp:51-166)
 * Ac = P^T*A*P  (R == NULL)  or  R^T*A*P : mfem::RAP -> hypre_BoomerAMGBuildCoarseOperator,
 *   Hierarchy.cpp:365,511-513; HiptmairSmootherFactory.cpp:160-161.
 * Two-pass symbolic/numeric hash SpGEMM; rows of the result have ascending columns,
 * explicit zeros are kept.
 * pe_fix_zero_rows: hypre_ParCSRMatrixFixZeroRows (Hierarchy.cpp:366-371).
 * pe_spadd: C = a*A + b*B, hypre_ParCSRMatrixAdd2 (src/hypreExtension/parcsr-add.c:199-245). */
int pe_spgemm(pe_ctx *ctx, const pe_mat *A, const pe_mat *B, pe_mat **C);
int pe_rap(pe_ctx *ctx, const pe_mat *R_or_null, const pe_mat *A, const pe_mat *P, pe_mat **Ac);
int pe_fix_zero_rows(pe_ctx *ctx, pe_mat *A, int32_t *num_fixed);
/* Numeric pass only (single rank): C / Ac already hold the pattern of the product (row pointers, ascending columns),
 * e.g. from an earlier pe_spgemm / pe_rap with operands of the same patterns; only their values are overwritten, with
 * the summation order of the two-pass product, so the values are those pe_spgemm / pe_rap compute, bit for bit.
 * pe_rap_numeric recomputes the intermediate A*P with the two-pass product and, as pe_rap, uses the cached transpose
 * of R (of P when R_or_null is NULL).  pe_spgemm_numeric_scaled: C = A diag(d)^-1 B with the values pe_spgemm of A and
 * a copy of B whose rows were scaled by pe_mat_scale_rows(copy, d, 1) computes (the Schur complement's A10 D^-1 A01). */
int pe_spgemm_numeric(pe_ctx *ctx, const pe_mat *A, const pe_mat *B, pe_mat *C);
int pe_spgemm_numeric_scaled(pe_ctx *ctx, const pe_mat *A, const pe_vec *d, const pe_mat *B, pe_mat *C);
int pe_rap_numeric(pe_ctx *ctx, const pe_mat *R_or_null, const pe_mat *A, const pe_mat *P, pe_mat *Ac);
/* The rows pe_fix_zero_rows rewrites (l1 norm below DBL_EPSILON).  changed == NULL: mask (length = rows of A) becomes
 * 1.0 on those rows and 0.0 elsewhere.  Otherwise mask is only read and *changed = 1 when that set differs from it. */
int pe_mat_zero_rows(pe_ctx *ctx, const pe_mat *A, pe_vec *mask, int32_t *changed);
int pe_spadd(pe_ctx *ctx, double a, const pe_mat *A, double b, const pe_mat *B, pe_mat **C);
/* Values only (single rank): C holds the pattern pe_spadd(a, A, b, B) produced for operands of A's and B's patterns
 * (A's entries in their order, then B's entries not in A); its values become those of pe_spadd, bit for bit. */
int pe_spadd_numeric(pe_ctx *ctx, double a, const pe_mat *A, double b, const pe_mat *B, pe_mat *C);
/* mfem::SparseMatrix::EliminateRowCol(rc, DIAG_ONE) for every marked dof (marker_host[n],
 * non-zero = essential): marked rows become unit rows, marked columns are zeroed; entries
 * stay in the pattern (examples/MultigridTest2Form.cpp:457-464). */
int pe_mat_eliminate_rowcol(pe_ctx *ctx, pe_mat *A, const int32_t *marker_host);

/* ---- src/hypreExtension utilities on device matrices (SURVEY 2.2)
 * pe_mat_delete_zeros : hypre_ParCSRMatrixDeleteZeros (deleteZeros.c:16-47), in place; entries with |a| <= tol are
 *                       dropped as in hypre_CSRMatrixDeleteZeros (tol = 0: stored zeros only)
 * pe_mat_sign         : hypre_ParCSRDataTransformationSign (entries -> -1 / 0 / +1 with threshold tol)
 * pe_mat_diagonal     : hypre_IdentityCSRMatrix (d == NULL) / hypre_DiagonalCSRMatrix (hypre_CSRFactory.c:16-250)
 * pe_mat_norms        : {l1, linf, max, Frobenius} (hypre_ParCSRMatrixNorms.c:18-195), all-reduced over ranks
 * pe_mat_compare      : hypre_ParCSRMatrixCompare bit flags (1 rows, 2 cols, 4/8 first/last row, 16/32 first/last
 *                       diag column, 64 ||A - B||_max > tol) -- the parity comparator
 * pe_rdp              : hypre_RDP, R^T diag(d) P (par_Tmatmul.c:17-39), rank-local */
int pe_mat_delete_zeros(pe_ctx *ctx, pe_mat *A, double tol);
int pe_mat_sign(pe_ctx *ctx, pe_mat *A, double tol);
int pe_mat_diagonal(pe_ctx *ctx, int32_t n, const pe_vec *d_or_null, pe_mat **out);
int pe_mat_norms(pe_ctx *ctx, pe_mat *A, double *out4);
int pe_mat_compare(pe_ctx *ctx, const pe_mat *A, const pe_mat *B, double tol, int32_t *flags);
int pe_rdp(pe_ctx *ctx, const pe_mat *R, const pe_vec *d, const pe_mat *P, pe_mat **out);

#ifdef __cplusplus
}
#endif
#endif /* PARELAG_B200_H */
