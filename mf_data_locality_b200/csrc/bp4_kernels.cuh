// bp4_kernels.cuh -- sm_100a kernels of the BP4 hot path (FP64).
//   cell kernel, plain : dst += A src                              (a1/a3/a6/a7 of SURVEY 8a)
//   cell kernel, fused : the same loop with do_cg_update4b run on a cell-batch range's private
//                        DoFs before its first cell and do_cg_update3b after its last cell
//                        (poisson_operator.h:339-364)                          (a2/a8/a9)
//   streaming kernels for the DoFs shared between ranges, the plain-CG BLAS-1 and the Jacobi apply.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "bp4_cell.cuh"

namespace bp4
{
  // 128 threads (one warp per SM sub-partition) and two resident blocks per SM: the block
  // may use up to 255 registers per thread (phase 2 keeps 9*Q doubles live), and while one
  // block waits on its gather or a barrier the other keeps the FP64 pipe busy.
  constexpr int kThreads     = 128;
  constexpr int kBlocksPerSM = 2;

  // Every per-degree choice of the cell kernel, each one measured on B200 (DESIGN.md 4.1-4.2, 6).
  // QUAD: all 27 geometry coefficients per cell (81 doubles) instead of the 8 tri-linear ones (24)
  template <int P, bool QUAD = false>
  struct Cfg
  {
    using G = Geom<P>;
    static constexpr int NCOEF = QUAD ? 81 : 24;
    // resident blocks per SM of the cell kernel: three (<= 168 registers, smaller batches)
    // measured faster at Q2 (+12 %) and Q6 (+13 %), slower or equal elsewhere
    static constexpr int BLOCKS   = (P == 2 || P == 6) ? 3 : kBlocksPerSM;
    static constexpr int budget   = (227 * 1024) / BLOCKS - 512;
    static constexpr int per_cell = (G::WORK + 2 * NCOEF) * 8 + 2 * 28 * 4;
    static constexpr int fit      = (budget - 4 * G::DOF - 16 * G::Q - 256) / per_cell;
    // phase 2 carries ~2/3 of the FP64 work: prefer Q^2*CPB close to two rounds of the block
    static constexpr int want = (2 * kThreads) / (G::Q * G::Q) > 0 ? (2 * kThreads) / (G::Q * G::Q) : 1;
    static constexpr int CPB  = fit < 1 ? 1 : (fit < want ? fit : want);
    // phases 1 and 3 as one sweep per 1-D contraction (phase1a..c, phase3a..c): with 3N rows per
    // cell the high degrees have too few items for 128 threads (29-52 % barrier wait at Q6-Q8)
    static constexpr bool FINE = P >= 6;
    // phase 2 called out of line (phase2_call)
    static constexpr bool P2_CALL = P >= 6;
    // the gather of batch i+1 is in flight during the scatter of batch i
    static constexpr bool PIPE_GATHER = P <= 4;
    // batches / units are claimed from an atomic counter instead of strided.  Measured on B200
    // (operator apply at ~50-100 M DoFs): Q2 +13 %, Q3 +5 %, Q4 +8 %, Q5 +11 %; Q6 -6 %, Q7 -11 %,
    // Q8 -10 % (the claim bookkeeping makes the register-starved high-degree kernels spill)
    static constexpr bool DYNAMIC = P <= 5;
    // a fused cell kernel (in-loop vector updates staged through shared memory) is built; see Stage
    static constexpr bool STAGED = P <= 4;
    // the form of vmult_with_merged_sums a context starts with when it has private DoF runs:
    // in-loop updates (true) or streamed before/after the cell loop.  The in-loop form wins at Q4
    // on one rank (2.12 vs 2.14 ms per iteration) and loses at Q2/Q3; on several ranks the loop is
    // three launches with a unit-granular tail each, which has not been measured to pay, so
    // bp4_comm_init goes back to the streamed form.  bp4_debug_set_fused / BP4_FUSED override both.
    static constexpr bool FUSED_DEFAULT = P == 4;
  };

  template <int P, int CPB, int NCOEF = 24>
  struct alignas(16) CellSmem
  {
    using G = Geom<P>;
    // the gathered DoFs, the three phases and the result all live in the work rows: gather
    // fills the first N*N slots of each row, phases 1 and 3 run in place
    double   work[CPB * G::WORK];
    double   coef[2][CPB][NCOEF]; // double-buffered: the next batch's metadata is prefetched
    double   xq[G::Q];
    double   wq[G::Q];
    double   red[8];           // (spare)
    uint32_t units[8];         // ring of the units this block has claimed
    uint32_t n_claimed;
    uint32_t eidx[2][CPB][28];
    uint32_t dtab[G::DOF];
  };

  // One batch of the fused cell loop: CPB consecutive cells of one unit (= a group of whole
  // cell-batch ranges owned by one thread block) and the two DoF intervals the vector updates
  // are hooked to (MatrixFree::cell_loop's pre/post contract, SURVEY App. B1):
  //   [pre_begin, pre_end)   private DoFs of the ranges whose FIRST cell lies in this batch:
  //                          do_cg_update4b must run on them before the batch is gathered
  //   [post_begin, post_end) private DoFs of the ranges whose LAST cell lies in this batch:
  //                          do_cg_update3b runs on them once the batch has been scattered
  // "private" = touched by the cells of exactly one range: the first group of Renumber's
  // cellbatch_range grouping (renumber_dofs_for_mf.h:556-590, :622-671), contiguous per range.
  struct alignas(16) BatchDesc
  {
    uint32_t cell0, n_cells;
    uint32_t pre_begin, pre_end;
    uint32_t post_begin, post_end;
    uint32_t pad[2];
  };

  // Staging rows of the fused cell loop (appended to CellSmem in dynamic shared memory).  The
  // in-loop do_cg_update4b / do_cg_update3b are cut into "jobs" of at most JOB DoFs; asynchronous
  // copies (cp.async + mbarrier) bring a job's r, p, h and diagonal entries into these rows while
  // the block runs a compute phase, the threads consume them from shared memory at the end of
  // that phase: no thread waits for a DRAM round trip or holds loaded values in registers
  // (the register-staged variant made the memory window 3x longer, DESIGN.md 4.2).
  // A job [b, e) may start at an odd index: the copy is widened to 16-byte boundaries, element i
  // sits at row[..][i - (b & ~1)], diagonal entry i/3 at prec[i/3 - ((b/3) & ~1)].
  template <int JOB>
  struct alignas(16) JobSmem
  {
    static constexpr int ROW  = JOB + 2;
    static constexpr int PREC = ((JOB / 3 + 4) + 1) & ~1;
    double             row[3][ROW]; // r, p (= d), h
    double             prec[PREC];
    double             redw[8][8]; // the seven merged sums, one row per warp
    BatchDesc          ring[8];    // descriptors of the batches i-2 .. i+4 of this block
    unsigned long long mbar;
    unsigned long long pad;
  };
  // JOB = DoFs per job that fit next to the cell kernel's own shared memory; a batch's pre / post
  // run is handled by two jobs -> LIMIT.  OK: the degree has a fused kernel at all (the runs of
  // the high degrees are far longer than what is left of the shared memory: Q5 2187 DoFs per range
  // vs 146 per job)
  template <int P>
  struct Stage
  {
    static constexpr long avail = (long)Cfg<P>::budget - (long)sizeof(CellSmem<P, Cfg<P>::CPB, 24>) - 16 - 512 - 256;
    // 3 rows of (JOB + 2) + JOB / 3 + 5 doubles
    static constexpr long cap   = ((avail / 8 - 11) * 3) / 10;
    static constexpr int  JOB   = cap < 64 ? 0 : (int)(cap & ~1L);
    static constexpr int  LIMIT = 2 * JOB;
    static constexpr bool OK    = Cfg<P>::STAGED && JOB >= 64;
  };

  // Scratch of the ordered reductions of the deterministic mode (DESIGN.md 4.6): every block of a
  // reduction writes its K partial sums to slot[k * gridDim.x + blockIdx.x]; the last block to
  // take a ticket sums them in a fixed order.  slot = nullptr: the reductions end with one
  // atomicAdd per block instead (default).
  struct DetSlots
  {
    double   *slot   = nullptr; // [K][grid], grid <= 8 * SMs
    uint32_t *ticket = nullptr; // zero between launches: the last block re-arms it
  };

  struct SolveState;
  struct CellArgs
  {
    const uint32_t *entity_index; // [n_cells][27]
    const double   *coef;         // [n_cells][24] tri-linear or [n_cells][81] quadratic coefficients
    const uint32_t *dtab;         // [3 N^3] gather/scatter table (build_dof_table)
    uint64_t        n_cells;      // plain: cells of this launch, batches are cut on the fly
    const double   *src;          // plain: input vector; fused: the search direction d (= p)
    double         *dst;          // plain: output vector; fused: h
    uint32_t       *sched;        // unit counter of this launch (zero at launch), null: strided
    // ---- fused (vmult_with_merged_sums) only ----
    const BatchDesc *batch;       // batches of all units
    const uint32_t  *unit_batch;  // [n_units + 1] first batch of every unit of this launch
    uint32_t         n_units;
    double          *r, *p, *x;   // g, d, x of SolverCGFullMerge; p == src
    const double    *prec;        // [n_owned / 3]
    double           alpha, beta, c1, c2; // c1 = alpha + alpha_old/beta_old, c2 = alpha_old/beta_old
    int              first;       // alpha == 0: p = -P r, h = 0 only
    int              update_x;    // alpha_old != 0
    double          *acc;         // [7]
    // device-resident solve (cell_kernel<..., DEV = true>): alpha, beta, first, update_x, c1, c2
    // are derived in-kernel from state->alpha .. beta_old instead of the fields above
    const SolveState *state;
  };

  // Solver state of a device-resident CG solve (bp4_solve_cg / bp4_solve_cg_merged), one block
  // per context.  The scalar kernels write it, the vector kernels of the next sweep read it.
  struct SolveState
  {
    // arguments of the next vmult_with_merged_sums exactly as SolverCGFullMerge passes them
    // (alpha_old = 0 on even iterations); after the stopping check: alpha, and the true
    // alpha_old / beta_old of the final x update.  The plain solve keeps alpha and beta here.
    double   alpha, beta, alpha_old, beta_old;
    double   gh;                     // plain: g.h of the current iteration
    double   tol, reduced_tol;       // ReductionControl: absolute and reduced tolerance
    double   last_value, initial_value;
    uint32_t max_steps, step;        // step = last checked step
    int32_t  state, pad;             // SolverControl::State: 0 iterate, 1 success, 2 failure
  };
} // namespace bp4
