/* bp4.h -- C ABI of the B200-native CEED BP4 hot path (drop-in boundary).
 *
 * This is the only interface between the host side (the C++ mirror of the reference's
 * operator/solver surface in mf_data_locality_b200/host/, or a deal.II application
 * through the stubs shown in INTEGRATION.md) and the CUDA (sm_100a, FP64) kernels.
 * Plain pointers and sizes only; no C++/torch/deal.II types.
 *
 * Each entry point cites the reference interface it replaces; paths are relative to
 * peterrum/mf_data_locality/common_code/.
 *
 * Conventions
 *   - every function returns 0 on success, a negative bp4_status otherwise;
 *     bp4_last_error() returns a thread-local message for the last failure.
 *   - a context is bound to one CUDA device and one stream and must be driven by one
 *     host thread (the reference runs one thread per MPI rank, benchmark.h:278).  The stream
 *     is the context's own, or the caller's after bp4_ctx_set_stream.
 *   - calls are asynchronous on that stream except those that return host scalars (bp4_dot,
 *     bp4_l2_norm, bp4_add_and_dot, bp4_all_zero, bp4_vmult_merged, bp4_vec_download,
 *     bp4_solve_cg, bp4_solve_cg_merged), which synchronise it.
 *   - vectors hold n_owned + n_ghost doubles: owned DoFs first (renumbered, three
 *     components interleaved per node), then ghost DoFs sorted by global index --
 *     the layout of LinearAlgebra::distributed::Vector<double>.
 *   - there is NO CPU fallback: without a CUDA device every call fails with
 *     BP4_ERR_CUDA.
 */
#ifndef BP4_H
#define BP4_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BP4_INVALID_INDEX 0xFFFFFFFFu /* numbers::invalid_unsigned_int, poisson_operator.h:114 */

typedef enum bp4_status
{
  BP4_OK           = 0,
  BP4_ERR_ARG      = -1, /* bad argument / unsupported degree */
  BP4_ERR_CUDA     = -2, /* CUDA runtime error (message in bp4_last_error) */
  BP4_ERR_NCCL     = -3, /* NCCL error */
  BP4_ERR_STATE    = -4  /* call sequence error (e.g. exchange without bp4_comm_init) */
} bp4_status;

typedef struct bp4_ctx bp4_ctx; /* operator + device mesh data  (Poisson::LaplaceOperator)   */
typedef struct bp4_vec bp4_vec; /* device vector                (LA::distributed::Vector)    */

/* Problem description = the arrays LaplaceOperator::initialize() builds
 * (poisson_operator.h:101-293) plus the partitioner's ghost-exchange plan. */
typedef struct bp4_desc
{
  int      degree;   /* fe_degree p, 2..8;  n_q_points_1d = p + 2 (benchmark.h:290-311)      */
  int      device;   /* CUDA device ordinal                                                   */
  uint64_t n_cells;  /* locally owned cells, in matrix-free loop order                        */
  uint64_t n_owned;  /* owned DoFs (multiple of 3)                                            */
  uint64_t n_ghost;  /* ghost DoFs (multiple of 3)                                            */
  /* [n_cells][27] first local DoF of each of the 27 cell entities, lexicographic entity
   * order a = ex + 3 ey + 9 ez, BP4_INVALID_INDEX for Dirichlet entities
   * = compressed_dof_indices (poisson_operator.h:183-261), one lane per cell.            */
  const uint32_t *entity_index;
  /* [n_cells][8][3] vertex coordinates, deal.II vertex order x + 2y + 4z
   * (poisson_operator.h:153-160); the tri-linear coefficients (:161-178) are derived.    */
  const double *vertices;
  uint64_t        n_constrained; /* MatrixFree::get_constrained_dofs(), poisson_operator.h:311 */
  const uint32_t *constrained;   /* local indices of owned Dirichlet DoFs                      */
  /* ghost exchange plan (Utilities::MPI::Partitioner); n_peers = 0 on a single rank.
   * Ghost DoFs owned by peer k occupy [n_owned+import_offset[k], n_owned+import_offset[k+1]);
   * export_index[export_offset[k] .. export_offset[k+1]) are the owned local DoFs peer k
   * ghosts, in the order of that peer's ghost range.                                         */
  int             n_peers;
  const int      *peer_rank;      /* [n_peers]     */
  const uint64_t *import_offset;  /* [n_peers + 1] */
  const uint64_t *export_offset;  /* [n_peers + 1] */
  const uint32_t *export_index;   /* [export_offset[n_peers]] */
  /* cell partitions of MatrixFree::cell_loop (SURVEY App. B1): cells [0, n_cells_before_comm)
   * and [n_cells_before_comm + n_cells_comm, n_cells) touch no ghost DoF; the exchange of
   * ghost values / ghost contributions is overlapped with them.  0/0 = no overlap.           */
  uint64_t n_cells_before_comm;
  uint64_t n_cells_comm;
  /* cell-batch ranges of the loop (MatrixFree task_info.cell_partition_data, as walked by
   * renumber_dofs_for_mf.h:622-671) and the owned DoFs PRIVATE to each of them: touched by the
   * cells of exactly one range, unconstrained, not shared with another rank.  These are the
   * DoF ranges on which MatrixFree::cell_loop runs the pre/post hooks of
   * vmult_with_merged_sums right around the range's own cells (poisson_operator.h:339-364).
   * Renumber(0,1,2) numbers them first and range by range (renumber_dofs_for_mf.h:556-590), so
   * range r owns the contiguous run [range_private_offset[r], range_private_offset[r+1]).
   * range_cell_offset[r] = first cell of range r, [0] = 0, [n_ranges] = n_cells; ranges do not
   * straddle the cell partitions above.  n_ranges = 0 (or an all-zero private table): the
   * vector updates are streamed over the whole vector before/after the cell loop instead.    */
  uint64_t        n_ranges;
  const uint64_t *range_cell_offset;    /* [n_ranges + 1] */
  const uint64_t *range_private_offset; /* [n_ranges + 1] local DoF indices, multiples of 3 */
  /* optional: [n_cells][27][3] ALL coefficient vectors of the cell geometry
   * X(xi) = sum_m v_m xi^a eta^b zeta^c, m = a + 3b + 9c, a,b,c in {0,1,2} -- the array
   * cell_quadratic_coefficients that local_apply evaluates (poisson_operator.h:577-602, :690).
   * The reference itself only fills the 8 tri-linear ones from the vertices (:161-178, "for now
   * use only constant and linear term"); with this field a caller can hand genuinely quadratic
   * cells (the MappingQCache(2) TODO of benchmark.h:75-77).  When given, `vertices` is ignored.  */
  const double *coefficients;
  /* 1: deterministic mode (see bp4_deterministic_info), 0: default.  The environment variable
   * BP4_DETERMINISTIC=1 turns it on for every context.  One rank only: with n_peers > 0 it is
   * BP4_ERR_ARG.                                                                               */
  int deterministic;
} bp4_desc;

const char *bp4_last_error(void);
int         bp4_device_count(int *count);

/* ---- context: LaplaceOperator::initialize (poisson_operator.h:101-293) ------------------ */
int bp4_ctx_create(const bp4_desc *desc, bp4_ctx **ctx);
int bp4_ctx_destroy(bp4_ctx *ctx);
int bp4_ctx_synchronize(bp4_ctx *ctx);
/* cudaStream_t the context currently queues its work on, as an opaque pointer: its own stream,
 * or the one bp4_ctx_set_stream bound */
int bp4_ctx_stream(bp4_ctx *ctx, void **stream);
/* From now on every piece of work of the context goes on `stream` (a cudaStream_t), as with the
 * stream argument of cuBLAS or NCCL: kernels, copies, memsets, solve-graph launches, NCCL calls
 * and the timing events of bp4_profile_*.  The ghost exchange still forks onto a second stream of
 * the context and joins back.  stream = NULL returns the context to its own stream; the legacy
 * default stream is accepted as cudaStreamLegacy (and cudaStreamPerThread as itself), since NULL
 * means "the context's own".
 *   - switching is safe: the new stream waits, through an event, for everything the context
 *     queued on the old one (pooled vectors, solve temporaries and the reduction scratch may still
 *     be in use there); the host does not wait.
 *   - a stream of another device, or not a stream, is BP4_ERR_ARG; switching while the old or
 *     the new stream is being captured into a graph is BP4_ERR_STATE.  Nothing is queued then.
 *   - the stream must stay valid while it is bound: until the next bp4_ctx_set_stream or
 *     bp4_ctx_destroy.  bp4_ctx_destroy never destroys or drains it; it waits for an event
 *     recorded there after the context's last call.
 *   - while the bound stream is being captured into a caller's graph, asynchronous calls
 *     (bp4_vmult, the BLAS-1 updates, ...) are captured with it; calls that synchronise, allocate
 *     or launch a solve graph (the host-scalar calls above, bp4_vec_alloc*, bp4_vec_upload,
 *     bp4_inverse_diagonal, the solves, bp4_ctx_synchronize, bp4_profile_*, bp4_comm_init) are
 *     BP4_ERR_STATE before anything is queued.
 *   - multi-rank: nothing here is rank-specific (the exchange and the all-reduce run on the bound
 *     stream), but only one rank is tested.                                                      */
int bp4_ctx_set_stream(bp4_ctx *ctx, void *stream);

/* ---- vectors: initialize_dof_vector (poisson_operator.h:298-302), reinit/operator= ------- */
int bp4_vec_alloc(bp4_ctx *ctx, uint64_t n, bp4_vec **v); /* zero-initialised, n doubles */
/* reinit(v, omit_zeroing_entries = true), solver_cg_optimized.h:215-217: contents undefined */
int bp4_vec_alloc_uninitialized(bp4_ctx *ctx, uint64_t n, bp4_vec **v);
int bp4_vec_free(bp4_ctx *ctx, bp4_vec *v);
int bp4_vec_size(const bp4_vec *v, uint64_t *n);
int bp4_vec_set_zero(bp4_ctx *ctx, bp4_vec *v);                            /* v = 0 */
int bp4_vec_upload(bp4_ctx *ctx, bp4_vec *v, const double *host, uint64_t n);
int bp4_vec_download(bp4_ctx *ctx, const bp4_vec *v, double *host, uint64_t n);
int bp4_vec_device_ptr(bp4_ctx *ctx, bp4_vec *v, double **dev);            /* current buffer */
/* v views n doubles of caller-owned device memory at dev: no copy, no allocation.  Every entry
 * point that takes a bp4_vec accepts it, with the usual length checks (n_owned + n_ghost for
 * operator operands, n_owned/3 for prec).
 *   - dev must be device memory (cudaMalloc, a caching allocator's block) of the context's device,
 *     16-byte aligned; n > 0.  A host pointer, managed memory, another GPU's memory, a null or
 *     misaligned pointer is BP4_ERR_ARG and nothing is launched.
 *   - lifetime: the memory must stay valid until bp4_vec_free and until the context's queued work
 *     on it has run.  bp4_vec_free releases the handle only; the memory stays the caller's and
 *     never enters the context's buffer pool.
 *   - stream order is the caller's: the context reads and writes the memory on its stream
 *     (bp4_ctx_stream).  Bind the stream that produces and consumes the data (bp4_ctx_set_stream),
 *     or make the context's stream wait for the producer and the consumer wait for the context's
 *     stream, e.g. with cudaEventRecord + cudaStreamWaitEvent.
 *   - device-resident solves cache their graph and three temporaries per (x, b, prec) address;
 *     bp4_vec_free of a wrapped vector drops the entries that name its memory, so wrapping a
 *     fresh x for every solve keeps one entry.                                                   */
int bp4_vec_wrap(bp4_ctx *ctx, double *dev, uint64_t n, bp4_vec **v);

/* ---- operator ------------------------------------------------------------------------- */
/* dst = A src, identity on constrained rows: LaplaceOperator::vmult, poisson_operator.h:307 */
int bp4_vmult(bp4_ctx *ctx, bp4_vec *dst, const bp4_vec *src);
/* LaplaceOperator::vmult_with_merged_sums (poisson_operator.h:327-377): pre-update of
 * x,g,d (do_cg_update4b, solver_cg_optimized.h:65), h = A d, the seven sums
 * (do_cg_update3b, :12), reduced over all ranks into out[7].  prec holds n_owned/3 entries.
 * With range tables in the descriptor the two vector kernels run INSIDE the cell loop on the
 * DoFs private to each cell-batch range (every vector is streamed once there) and as two
 * streaming kernels on the remaining DoFs (shared between ranges or ranks, Dirichlet).       */
int bp4_vmult_merged(bp4_ctx *ctx, bp4_vec *x, bp4_vec *g, bp4_vec *d, bp4_vec *h,
                     const bp4_vec *prec, double alpha, double beta, double alpha_old,
                     double beta_old, double out[7]);
/* 1/diag of the scalar GLL(p+1) Laplacian per node, 1 where 0:
 * LaplaceOperator::compute_inverse_diagonal + extraction (poisson_operator.h:392-426,
 * benchmark.h:141-147).  out holds n_owned/3 entries.                                       */
int bp4_inverse_diagonal(bp4_ctx *ctx, bp4_vec *out);
/* the same in the reference's own result layout (poisson_operator.h:392-426): a DoF vector
 * (n_owned + n_ghost entries) with 1/diag on component 0 of every node and 1 elsewhere ...     */
int bp4_inverse_diagonal_vector(bp4_ctx *ctx, bp4_vec *out);
/* ... and the extraction loop of benchmark.h:141-147: dst[i] = src[n_components * i + component] */
int bp4_extract_component(bp4_ctx *ctx, bp4_vec *dst, const bp4_vec *src, int n_components,
                          int component);
/* dst[3i+c] = diag[i] * src[3i+c]: DiagonalMatrixBlocked::vmult, diagonal_matrix_blocked.h:13 */
int bp4_jacobi_vmult(bp4_ctx *ctx, bp4_vec *dst, const bp4_vec *src, const bp4_vec *diag);
/* x += c1 * d + c2 * P g: final x update on even iterations, solver_cg_optimized.h:260-288  */
int bp4_x_finalize_even(bp4_ctx *ctx, bp4_vec *x, const bp4_vec *d, const bp4_vec *g,
                        const bp4_vec *prec, double c1, double c2);

/* ---- BLAS-1 on owned entries (LA::distributed::Vector members used by SolverCG and
 *      SolverCGFullMerge, solver_cg_optimized.h:215-228, :257) ---------------------------- */
int bp4_equ(bp4_ctx *ctx, bp4_vec *dst, double a, const bp4_vec *src);           /* dst = a src        */
int bp4_add(bp4_ctx *ctx, bp4_vec *dst, double a, const bp4_vec *src);           /* dst += a src       */
int bp4_sadd(bp4_ctx *ctx, bp4_vec *dst, double s, double a, const bp4_vec *src);/* dst = s dst + a src*/
int bp4_dot(bp4_ctx *ctx, const bp4_vec *a, const bp4_vec *b, double *result);   /* all ranks          */
int bp4_add_and_dot(bp4_ctx *ctx, bp4_vec *g, double a, const bp4_vec *h, const bp4_vec *w,
                    double *result);                                /* g += a h; return g.w */
int bp4_l2_norm(bp4_ctx *ctx, const bp4_vec *v, double *result);
int bp4_all_zero(bp4_ctx *ctx, const bp4_vec *v, int *result);

/* ---- whole solves on the device ---------------------------------------------------------
 * The two CG solvers of the benchmark with the host out of the iteration loop: every scalar
 * (alpha, beta, the residual, the stopping test) is computed on the device, in the host solver's
 * arithmetic, and the whole solve runs as one CUDA graph: step 0 (start residual g = A x - b, or
 * -b for a zero x, chosen on the device by an IF node, its norm and the first check) with the
 * kernels of the entry points above, then a conditional WHILE node runs the iterations until the
 * stopping test ends them.  A solve that ends at step 0 runs no iteration and leaves x untouched.
 *   - stopping test: ReductionControl::check (solver_control.h): step 0 sets
 *     reduced_tol = |g_0| * reduce; success if value < reduced_tol or value <= tol; failure if
 *     step >= max_steps or the value is NaN.  reduce = 0 is a plain SolverControl(max_steps, tol).
 *   - hitting max_steps is not an error: the call returns 0 with state = 2 and x holds the last
 *     iterate, as the host-driven solvers leave it.
 *   - one rank only: a context with a ghost-exchange plan (n_peers > 0) or a communicator over
 *     several ranks gives BP4_ERR_STATE.
 *   - the merged solve uses the context's in-loop / streamed form (bp4_debug_set_fused), i.e.
 *     the vector kernels of bp4_vmult_merged.
 *   - bp4_solve_cg / bp4_solve_cg_merged block: they are the _async call, a synchronisation of
 *     the stream and a copy of the result into *out.  The instantiated graph is cached in the
 *     context per (solver, x, b, prec, in-loop form) together with its temporaries g, d, h; a
 *     repeated solve re-uses it, whatever its max_steps, tolerances, result and history: those are
 *     kernel parameters of the graph's first node, replaced per launch without a new graph.
 *     bp4_vec_free of a wrapped x, b or prec drops the entries that name it and returns their
 *     temporaries to the context's pool.
 *   - measurement: bp4_launch_count adds one per graph launch; the kernels of the graph, step 0
 *     included, are counted once, when it is built.  bp4_profile_* time no kernel inside the
 *     graph.                                                                                  */
typedef struct bp4_solve_result
{
  int      state;         /* 1 = success, 2 = failure (SolverControl::State)   */
  unsigned last_step;     /* SolverControl::last_step()                        */
  double   last_value;    /* residual norm checked at last_step                */
  double   initial_value; /* residual norm at step 0                           */
} bp4_solve_result;
/* deal.II SolverCG with DiagonalMatrixBlocked (benchmark_precond/bench.cc:11-16, SURVEY App. B3);
 * prec holds n_owned/3 inverse-diagonal entries                                               */
int bp4_solve_cg(bp4_ctx *ctx, bp4_vec *x, const bp4_vec *b, const bp4_vec *prec, unsigned max_steps,
                 double tol, double reduce, bp4_solve_result *out);
/* SolverCGFullMerge (solver_cg_optimized.h:192-302): x every second iteration, odd/even fix-up */
int bp4_solve_cg_merged(bp4_ctx *ctx, bp4_vec *x, const bp4_vec *b, const bp4_vec *prec,
                        unsigned max_steps, double tol, double reduce, bp4_solve_result *out);
/* The same solves, queued on the context's stream without any host synchronisation: the call
 * returns once the graph launch is queued, and the stream writes *result when the solve ends, so
 * that a caller can queue solve k + 1, or the work that reads x, behind solve k.
 *   - result: device memory of the context's device or mapped pinned host memory
 *     (cudaHostAlloc / cudaMallocHost, cudaHostRegister with cudaHostRegisterMapped), 8-byte
 *     aligned; anything else is BP4_ERR_ARG and nothing is queued.  Read it after the stream
 *     (or an event recorded behind the call) has completed.
 *   - history (optional, NULL for none): the same kinds of memory, room for max_steps + 1
 *     doubles (the ABI cannot check the size: a plain pointer carries none).  It receives the
 *     residual norm checked at steps 0 .. last_step, the values deal.II's SolverControl records
 *     with enable_history_data(); the entries after last_step are left untouched.
 *   - x, b, prec and the memory behind result and history must stay valid until the solve has
 *     run.  Several solves may be queued back to back; each keeps its own arguments.        */
int bp4_solve_cg_async(bp4_ctx *ctx, bp4_vec *x, const bp4_vec *b, const bp4_vec *prec, unsigned max_steps,
                       double tol, double reduce, bp4_solve_result *result, double *history);
int bp4_solve_cg_merged_async(bp4_ctx *ctx, bp4_vec *x, const bp4_vec *b, const bp4_vec *prec,
                              unsigned max_steps, double tol, double reduce, bp4_solve_result *result,
                              double *history);

/* ---- mixed-precision solve --------------------------------------------------------------
 * CG to an FP64-accurate answer with most of the operator work in FP32 (DESIGN.md 4.7): iterative
 * refinement whose outer loop computes the true residual b - A x with the FP64 operator and tests
 * it, and whose inner loop solves for the correction with merged CG (SolverCGFullMerge's
 * recurrences, streamed form) on an FP32 cell kernel and FP32 vectors.  One CUDA graph, one rank.
 *   - stopping test: tol, reduce and the NaN rule are ReductionControl::check on the FP64 true
 *     residual |b - A x|; initial_value is that residual at the given x (step 0), last_value the
 *     one at the last refinement step.
 *   - max_steps caps the total number of inner FP32 iterations over all refinement steps.
 *   - every refinement step starts the inner solve from zero on the residual scaled to norm 1 and
 *     stops it at a fixed relative reduction (1e-3, chosen by measurement: DESIGN.md 4.7) or when the
 *     remaining step budget runs out; x += the correction scaled back.
 *   - history (optional): room for max_steps + 1 doubles; it receives the FP64 true residual of
 *     every refinement step 0 .. refinements.
 *   - state 1: success.  state 2 when the step budget is used up, when a refinement step does not
 *     reduce the true residual (stagnation: FP32 cannot resolve a smaller correction) or when the
 *     residual is NaN; x then holds the last iterate.  A solve that ends at step 0 (a zero right-
 *     hand side, an x that already passes, max_steps = 0) leaves x untouched.
 *   - refused like the solves above: BP4_ERR_STATE on a context with a ghost-exchange plan or a
 *     communicator over several ranks, BP4_ERR_ARG for result / history memory the device cannot
 *     use; also BP4_ERR_STATE in the deterministic mode (FP32 ordered reductions are not built).
 *   - the graph is cached per (x, b, prec) with its temporaries: an FP64 A x and the FP32 residual,
 *     direction, product, correction and preconditioner (4.33 floats per DoF); bp4_vec_free of a
 *     wrapped x, b or prec drops it.  The _async form queues the solve like bp4_solve_cg_async;
 *     bp4_solve_cg_mixed is the async call, a synchronisation and a copy into *out.            */
typedef struct bp4_mixed_result
{
  int      state;         /* 1 = success, 2 = failure                                  */
  unsigned refinements;   /* last refinement step checked                              */
  unsigned inner_steps;   /* FP32 iterations over all refinement steps                 */
  double   last_value;    /* FP64 true residual at the last refinement step            */
  double   initial_value; /* FP64 true residual at step 0                              */
} bp4_mixed_result;
int bp4_solve_cg_mixed_async(bp4_ctx *ctx, bp4_vec *x, const bp4_vec *b, const bp4_vec *prec, unsigned max_steps,
                             double tol, double reduce, bp4_mixed_result *result, double *history);
int bp4_solve_cg_mixed(bp4_ctx *ctx, bp4_vec *x, const bp4_vec *b, const bp4_vec *prec, unsigned max_steps,
                       double tol, double reduce, bp4_mixed_result *out);

/* ---- deterministic mode -----------------------------------------------------------------
 * With bp4_desc::deterministic (or BP4_DETERMINISTIC=1) every result of bp4_vmult,
 * bp4_vmult_merged (vector and sums), bp4_inverse_diagonal / _vector, bp4_dot, bp4_add_and_dot,
 * bp4_l2_norm, bp4_solve_cg and bp4_solve_cg_merged is a function of the inputs alone: repeated
 * calls and repeated runs give the same bits, given the same build, the same device model and the
 * same SM count, on one rank (no ghost-exchange plan; bp4_comm_init over several ranks is
 * BP4_ERR_STATE).  How:
 *   - the cells are coloured greedily in the given order (a cell takes the lowest colour that no
 *     earlier cell sharing one of its valid entities has; at most 64 colours, else BP4_ERR_ARG)
 *     and the cell loop and the diagonal assembly run one launch per colour: within a colour no
 *     two cells touch the same DoF, so the additions into every entry happen in colour order;
 *   - every reduction sums its per-block partials in a fixed order instead of with atomics, and
 *     the host-driven and device-resident solves use the same reductions, so they give the same
 *     sums and the same iterates, bit for bit;
 *   - vmult_with_merged_sums always runs in the streamed form (bp4_debug_set_fused(ctx, 1) is
 *     BP4_ERR_STATE).
 * bp4_deterministic_info: *on = 1 in this mode; *n_colors = number of colours (0 when off);
 * cell_color (optional, [n_cells], the caller's cell order) receives each cell's colour when on. */
int bp4_deterministic_info(bp4_ctx *ctx, int *on, uint32_t *n_colors, uint32_t *cell_color);

/* ---- multi-GPU (Utilities::MPI::Partitioner / MPI_Allreduce call sites, SURVEY 2a) ------- */
#define BP4_NCCL_ID_BYTES 128
int bp4_comm_unique_id(unsigned char id[BP4_NCCL_ID_BYTES]);                 /* rank 0 */
/* once per context: a second call is BP4_ERR_STATE and leaves the first communicator in place  */
int bp4_comm_init(bp4_ctx *ctx, int rank, int n_ranks, const unsigned char id[BP4_NCCL_ID_BYTES]);
/* n_ranks of the communicator; peer_copies = 1 when the ghost exchange runs as copy-engine peer
 * copies into IPC-shared buffers with stream-memory-operation flags (no SM involved; the analogue
 * of the reference's USE_SHMEM path, benchmark.h:35, :105-108), 0 when it runs as NCCL send/recv
 * (BP4_P2P=0, more than 16 ranks, or IPC / stream memory operations unavailable)             */
int bp4_comm_info(bp4_ctx *ctx, int *n_ranks, int *peer_copies);
int bp4_update_ghost_values(bp4_ctx *ctx, bp4_vec *v);   /* owners -> ghost copies            */
int bp4_compress_add(bp4_ctx *ctx, bp4_vec *v);          /* ghost contributions -> owners, +=  */

/* ---- measurement / developer hooks (not part of the drop-in surface) ------------------- */
/* fused = 1: do_cg_update4b/3b inside the cell kernel on the private DoFs of the ranges
 * (degrees 2..4, tri-linear geometry, descriptor with range tables; anything else is a state
 * error), 0: streamed over the whole vector by pre_kernel / post_kernel.  Default: the form
 * measured faster - fused at degree 4 on a single rank, streamed otherwise; the environment
 * variable BP4_FUSED=0/1 or this call pin it.  Same sums up to summation order.             */
int bp4_debug_set_fused(bp4_ctx *ctx, int on);
int bp4_fused_info(bp4_ctx *ctx, int *fused, uint64_t *n_private, uint64_t *n_units);
/* dst = A src with the FP32 cell kernel of the mixed solve: src rounded to float, the result
 * widened to double; constrained rows are the identity as in bp4_vmult.  One rank, not in the
 * deterministic mode (BP4_ERR_STATE).                                                        */
int bp4_debug_vmult_f32(bp4_ctx *ctx, bp4_vec *dst, const bp4_vec *src);
typedef enum bp4_kernel_id
{
  BP4_K_VMULT  = 0, /* cell kernel, plain                                   */
  BP4_K_MERGED = 1, /* cell kernel with the in-loop vector updates (fused) */
  BP4_K_PRE    = 2,
  BP4_K_POST   = 3,
  BP4_K_BLAS1  = 4,
  BP4_K_COUNT  = 5
} bp4_kernel_id;
int bp4_profile_enable(bp4_ctx *ctx, int on); /* CUDA-event timing of every launch, per id */
int bp4_profile_reset(bp4_ctx *ctx);
int bp4_profile_get(bp4_ctx *ctx, int kernel_id, double *total_ms, uint64_t *launches);
int bp4_launch_count(bp4_ctx *ctx, uint64_t *launches); /* all kernel launches since create/reset */

#ifdef __cplusplus
}
#endif
#endif /* BP4_H */
