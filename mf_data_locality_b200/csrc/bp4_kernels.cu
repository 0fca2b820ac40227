// bp4_kernels.cu -- kernel definitions and launchers (sm_100a, FP64).  See bp4_kernels.cuh.
#include <algorithm>
#include <cstdio>
#include <cstdlib>

#include "bp4_kernels.cuh"
#include "bp4_launch.h"
#include "bp4_tables.h"

namespace bp4
{
  // one table per degree in the constant bank: with fully unrolled contractions every
  // matrix entry becomes a c[bank][offset] operand of a DFMA, no load instruction
  template <int P>
  __constant__ Tab<P> c_tab;

  template <int P, int CPB, int NC>
  __device__ __forceinline__ void load_tables(CellSmem<P, CPB, NC> &sm, const uint32_t *dtab)
  {
    for (int i = threadIdx.x; i < Geom<P>::DOF; i += blockDim.x)
      sm.dtab[i] = dtab[i];
    if (threadIdx.x < Geom<P>::Q)
      {
        sm.xq[threadIdx.x] = c_tab<P>.xq[threadIdx.x];
        sm.wq[threadIdx.x] = c_tab<P>.wq[threadIdx.x];
      }
    if (threadIdx.x < 8)
      sm.red[threadIdx.x] = 0.;
  }

  // optional per-phase clock accounting (compile with -DBP4_PHASE_TIMING, run with
  // BP4_PHASE_TIMING=1): how a warp's time splits over metadata / gather / phases / scatter
#ifdef BP4_PHASE_TIMING
  __device__ unsigned long long g_phase_clk[8];
#  define BP4_TICK_INIT unsigned long long tc[8] = {0, 0, 0, 0, 0, 0, 0, 0}; long long t0 = clock64();
#  define BP4_TICK(k) { const long long t1 = clock64(); tc[k] += t1 - t0; t0 = t1; }
#  define BP4_TICK_FLUSH if ((threadIdx.x & 31) == 0) for (int k = 0; k < 8; ++k) atomicAdd(&g_phase_clk[k], tc[k]);
  // per-block timeline of the first kTraceBatches batches (BP4_TRACE=<file>): globaltimer at the
  // top of the batch, after phase 3, after the scatter, at the end of the memory window; + SM id
  constexpr int kTraceBatches = 48;
#  ifndef BP4_TRACE_TID
#    define BP4_TRACE_TID 0
#  endif
  __device__ unsigned long long *g_trace;
  __device__ __forceinline__ unsigned long long gtime()
  {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
  }
  __device__ __forceinline__ unsigned smid()
  {
    unsigned r;
    asm volatile("mov.u32 %0, %smid;" : "=r"(r));
    return r;
  }
#  define BP4_TRACE(i, k)                                                                     \
    if (g_trace && threadIdx.x == BP4_TRACE_TID && (i) < kTraceBatches)                                   \
      g_trace[((size_t)blockIdx.x * kTraceBatches + (i)) * 20 + (k)] = (k) == 4 ? smid() : gtime();
#else
#  define BP4_TICK_INIT
#  define BP4_TICK(k)
#  define BP4_TICK_FLUSH
#  define BP4_TRACE(i, k)
#endif

  // Phase 2 as a real call for the high degrees: its ~100 live doubles get a register allocation
  // of their own instead of competing with whatever the gather/scatter code around it keeps
  // alive (the inlined form spilled 2.6x more after an unrelated change to the gather).
  template <int P, bool QUAD>
  __device__ __noinline__ void phase2_call(const uint32_t cf_off, const uint32_t work_off, const int qx,
                                           const int qz, const double x, const double z, const double wxz)
  {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    phase2<P, QUAD>(c_tab<P>, reinterpret_cast<const double *>(smem_raw + cf_off),
              reinterpret_cast<double *>(smem_raw + work_off), qx, qz, x, z, wxz);
  }

  __device__ __forceinline__ double warp_sum(double v)
  {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
      v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
  }

  // the seven merged sums of do_cg_update3b (solver_cg_optimized.h:37-44) for one entry
  __device__ __forceinline__ void post_terms(double (&s)[7], const double ri, const double di,
                                             const double hi, const double pr)
  {
    const double zi = pr * hi;
    s[0] += di * hi;
    s[1] += hi * hi;
    s[2] += ri * hi;
    s[3] += ri * ri;
    s[4] += ri * zi;
    s[5] += hi * zi;
    s[6] += ri * pr * ri;
  }

  // i / 3 for 32-bit i without an integer division
  __device__ __forceinline__ uint32_t div3(const uint32_t i) { return __umulhi(i, 0xAAAAAAABu) >> 1; }

  // ---- mbarrier / asynchronous-copy wrappers (PTX ISA: mbarrier, cp.async) ----
  __device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
  __device__ __forceinline__ void mbar_init(const uint32_t bar, const uint32_t count)
  {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __device__ __forceinline__ void mbar_wait(const uint32_t bar, const uint32_t parity)
  {
    asm volatile("{\n\t.reg .pred p;\n"
                 "WAIT_%=:\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
                 "@p bra DONE_%=;\n\t"
                 "bra WAIT_%=;\n"
                 "DONE_%=:\n\t}" ::"r"(bar),
                 "r"(parity)
                 : "memory");
  }
  __device__ __forceinline__ void cp_async16(const uint32_t smem_dst, const void *gmem_src)
  {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gmem_src) : "memory");
  }
  __device__ __forceinline__ void cp_async8(const uint32_t smem_dst, const void *gmem_src)
  {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_dst), "l"(gmem_src) : "memory");
  }
  __device__ __forceinline__ void cp_async4(const uint32_t smem_dst, const void *gmem_src)
  {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_dst), "l"(gmem_src) : "memory");
  }

  // ---------------------------------------------------------------------------------------
  // The cell kernel.  Every warp does every phase; two (or three) blocks per SM overlap one
  // block's memory phases with the other's FP64 phases.  The memory phases are kept short:
  //  * the next batch's metadata (27 indices + 24 coefficients per cell) is loaded into
  //    registers before phase 1 and parked in the other half of a double buffer after phase 3;
  //  * the gather issues all loads of the batch before the first use (one latency, not many);
  //  * the scatter reads its table/index/value operands for several DoFs before the REDs go out.
  //
  // FUSED = LaplaceOperator::vmult_with_merged_sums (poisson_operator.h:327-377) in the cell
  // loop.  The reference hooks do_cg_update4b "before the first touch" and do_cg_update3b "after
  // the last touch" of a DoF range into MatrixFree::cell_loop; Renumber(0,1,2) has made the DoFs
  // touched by exactly one cell-batch range a contiguous run per range
  // (renumber_dofs_for_mf.h:556-590).  Here a thread block owns whole ranges (a "unit" = a few
  // consecutive ranges, cut into batches of CPB cells), so those runs are private to the block:
  //   before the batch that holds a range's first cell is gathered -> do_cg_update4b on the run
  //   (streamed, coalesced; r, p, x updated in place, h zeroed), one batch ahead of its use;
  //   after the batch that holds its last cell has been scattered -> __threadfence, barrier,
  //   do_cg_update3b on the run while h, r, p are still in L2; 7 sums -> warp -> block -> acc.
  // No counters, no ping-pong buffers, no inter-block ordering.  The DoFs shared between ranges
  // (and between ranks, and the Dirichlet ones) are the tail [n_private, n_owned) of the vector:
  // pre_kernel / post_kernel stream them before / after this kernel.
  // ---------------------------------------------------------------------------------------
  // DEV (fused only): the scalars of do_cg_update4b come from the solver state of a device-resident
  // solve (a.state) instead of the launch arguments
  template <int P, int CPB, bool FUSED, bool QUAD, bool DEV = false>
  __global__ void __launch_bounds__(kThreads, Cfg<P>::BLOCKS) cell_kernel(const CellArgs a)
  {
    constexpr int NC = Cfg<P, QUAD>::NCOEF;
    using G         = Geom<P>;
    constexpr int Q = G::Q;
    constexpr bool kFine = Cfg<P>::FINE;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CellSmem<P, CPB, NC> &sm  = *reinterpret_cast<CellSmem<P, CPB, NC> *>(smem_raw);
    const int             tid = threadIdx.x;
    const Tab<P>         &tb  = c_tab<P>;
    load_tables<P, CPB, NC>(sm, a.dtab);
    BP4_TICK_INIT
    // ---- work list of this block: a unit is one batch (plain) or the batches
    // [unit_batch[u], unit_batch[u+1]) of whole ranges (fused).  Units are claimed dynamically
    // (Cfg<P>::DYNAMIC): the first one is blockIdx.x, the following ones come from an atomic counter,
    // a few units ahead of their use so that the claim's latency never shows.  The two blocks of
    // an SM run at different speeds (the warp scheduler favours one of them: measured 10.2 vs
    // 14.1 us per batch at Q4), a static split would leave the slower one with a long tail.
    struct It
    {
      uint32_t j, u, b, b_end; // j = position in this block's unit sequence
      bool     valid;
    };
    const uint32_t n_units = FUSED ? a.n_units : (uint32_t)((a.n_cells + CPB - 1) / CPB);
    const bool     dynamic = Cfg<P>::DYNAMIC && a.sched != nullptr;
    auto           unit_at = [&](const uint32_t j) {
      return dynamic ? sm.units[j & 7u] : blockIdx.x + j * gridDim.x;
    };
    // units a block holds claimed (the current one included) in the plain and in the fused loop
    constexpr uint32_t kClaimDepth = 5, kClaimDepthFused = 2;
    // thread 0 only; visible after the next barrier
    auto claim_ahead = [&](const uint32_t j_from, const uint32_t depth) {
      if (dynamic)
        while (sm.n_claimed < j_from + depth)
          {
            sm.units[sm.n_claimed & 7u] = gridDim.x + atomicAdd(a.sched, 1u);
            ++sm.n_claimed;
          }
    };
    auto enter = [&](It &it) {
      it.u     = unit_at(it.j);
      it.valid = it.u < n_units;
      if (FUSED && it.valid)
        {
          it.b     = __ldg(a.unit_batch + it.u);
          it.b_end = __ldg(a.unit_batch + it.u + 1);
        }
    };
    auto advance = [&](It it) {
      if (FUSED && it.valid && it.b + 1 < it.b_end)
        {
          ++it.b;
          return it;
        }
      if (it.valid)
        {
          ++it.j;
          enter(it);
        }
      return it;
    };
    struct Batch // plain kernel: cut on the fly
    {
      uint32_t cell0;
      int      nc;
    };
    auto describe = [&](const It &it) {
      Batch d;
      d.cell0 = it.u * CPB;
      d.nc    = (int)min((uint64_t)CPB, a.n_cells - (uint64_t)d.cell0);
      return d;
    };

    // metadata items of a batch handled by this thread: at most ME indices and MC coefficients
    constexpr int ME = (CPB * 27 + kThreads - 1) / kThreads, MC = (CPB * NC + kThreads - 1) / kThreads;
    uint32_t      me[ME];
    double        mc[MC];
    auto          fetch_meta = [&](const uint32_t cell0, const int nc) {
#pragma unroll
      for (int u = 0; u < ME; ++u)
        {
          const int k = tid + u * kThreads;
          me[u]       = k < nc * 27 ? __ldg(a.entity_index + (uint64_t)cell0 * 27 + k) : 0xFFFFFFFFu;
        }
#pragma unroll
      for (int u = 0; u < MC; ++u)
        {
          const int k = tid + u * kThreads;
          mc[u]       = k < nc * NC ? __ldg(a.coef + (uint64_t)cell0 * NC + k) : 0.;
        }
    };
    auto park_meta = [&](const int bf) {
#pragma unroll
      for (int u = 0; u < ME; ++u)
        {
          const int k = tid + u * kThreads;
          if (k < CPB * 27)
            sm.eidx[bf][k / 27][k % 27] = me[u];
        }
#pragma unroll
      for (int u = 0; u < MC; ++u)
        {
          const int k = tid + u * kThreads;
          if (k < CPB * NC)
            sm.coef[bf][k / NC][k % NC] = mc[u];
        }
    };
    // fused: the same items go from global to shared memory asynchronously (no registers held
    // over the phases); they count towards the next mbarrier arrival of this thread
    auto meta_async = [&](const int bf, const uint32_t cell0, const int nc) {
#pragma unroll
      for (int u = 0; u < ME; ++u)
        {
          const int k = tid + u * kThreads;
          if (k < nc * 27)
            cp_async4(smem_u32(&sm.eidx[bf][k / 27][k % 27]), a.entity_index + (uint64_t)cell0 * 27 + k);
          else if (k < CPB * 27)
            sm.eidx[bf][k / 27][k % 27] = 0xFFFFFFFFu;
        }
#pragma unroll
      for (int u = 0; u < MC; ++u)
        {
          const int k = tid + u * kThreads;
          if (k < nc * NC)
            cp_async8(smem_u32(&sm.coef[bf][k / NC][k % NC]), a.coef + (uint64_t)cell0 * NC + k);
        }
    };

    // gather (vector_access_reduced.h:175-258): consecutive threads walk an entity's contiguous
    // DoF segment.  Thread tid owns elements tid + r * kThreads of EVERY cell of the batch, so the
    // table entry is decoded once per r and the (cell, r) slots unroll with compile-time cell
    // offsets: ~7 instructions per element, all loads of the batch in flight together.  Cells
    // missing from a ragged last batch carry invalid entity indices (fetch_meta) and gather zeros.
    // With kPipe the gather is software-pipelined: the loads of batch i+1 are issued
    // (gather_issue) right after the scatter of batch i and land in registers while the block
    // does other memory work; they are stored to the work rows (gather_store) afterwards.
    // The fused kernel reads the direction with plain loads, not ld.global.nc: it was written by
    // this block's own do_cg_update4b moments ago (the L1 sees the stores of its own SM, every
    // other DoF the block reads is constant during the kernel).
    constexpr bool kPipe = Cfg<P>::PIPE_GATHER;
    constexpr int R = (G::DOF + kThreads - 1) / kThreads, S = CPB * R;
    // only the last r can run past the end of the cell
    const bool last_on = tid < G::DOF - (R - 1) * kThreads;
    auto       on      = [&](const int r) { return r < R - 1 || last_on; };
    double     gv[S];
    auto       gather_issue = [&](const int bf) {
      uint32_t tt[R], idx[S];
#pragma unroll
      for (int r = 0; r < R; ++r)
        tt[r] = sm.dtab[on(r) ? tid + r * kThreads : 0];
#pragma unroll
      for (int s1 = 0; s1 < S; ++s1)
        {
          const int      cell = s1 / R, r = s1 % R;
          const uint32_t base = sm.eidx[bf][cell][dtab_ent(tt[r])];
          idx[s1] = on(r) && base != 0xFFFFFFFFu ? base + dtab_rel(tt[r]) : 0xFFFFFFFFu;
        }
#pragma unroll
      for (int s1 = 0; s1 < S; ++s1)
        gv[s1] = idx[s1] != 0xFFFFFFFFu ? (FUSED ? a.src[idx[s1]] : __ldg(a.src + idx[s1])) : 0.;
    };
    auto gather_store = [&]() {
      uint32_t tt[R];
#pragma unroll
      for (int r = 0; r < R; ++r)
        tt[r] = sm.dtab[on(r) ? tid + r * kThreads : 0];
#pragma unroll
      for (int s1 = 0; s1 < S; ++s1)
        {
          const int cell = s1 / R, r = s1 % R;
          if (on(r))
            sm.work[cell * G::WORK + dtab_off_work<P>(tt[r])] = gv[s1];
        }
    };
    // scatter-add (vector_access_reduced.h:437-521); the cell-interior entity (13) is touched by
    // this cell only -> plain store
    auto scatter = [&](const int bf) {
      constexpr int SU = 6; // DoFs whose operands are read before their REDs go out
      uint32_t      tt[R];
#pragma unroll
      for (int r = 0; r < R; ++r)
        tt[r] = sm.dtab[on(r) ? tid + r * kThreads : 0];
#pragma unroll
      for (int s0 = 0; s0 < S; s0 += SU)
        {
          double   v[SU];
          uint32_t adr[SU];
#pragma unroll
          for (int u = 0; u < SU; ++u)
            if (s0 + u < S)
              {
                const int      cell = (s0 + u) / R, r = (s0 + u) % R;
                const uint32_t base = sm.eidx[bf][cell][dtab_ent(tt[r])];
                adr[u] = on(r) && base != 0xFFFFFFFFu ? base + dtab_rel(tt[r]) : 0xFFFFFFFFu;
                v[u]   = sm.work[cell * G::WORK + dtab_off_work<P>(tt[r])];
              }
#pragma unroll
          for (int u = 0; u < SU; ++u)
            if (s0 + u < S && adr[u] != 0xFFFFFFFFu)
              {
                if (dtab_ent(tt[(s0 + u) % R]) == 13u)
                  a.dst[adr[u]] = v[u];
                else
                  atomicAdd(a.dst + adr[u], v[u]);
              }
        }
    };
    // the three compute phases on the nc cells in the work rows; `between` runs at the end of
    // phase 1 and of phase 2 (before the barrier that closes them) and right after those barriers
    auto phase_1 = [&](const int nc) {
      // phase 1/3 items are handed out from the LAST thread downwards: the ragged final round
      // of phase 2 lands on the first warps, so the two kinds of partial rounds end up on
      // different warps (= different SM sub-partitions) instead of piling up on warp 0
      if (!kFine)
        {
          for (int it = kThreads - 1 - tid; it < nc * G::ITEMS13; it += kThreads)
            phase1<P>(tb, sm.work + it * G::RW, sm.work + it * G::RW);
        }
      else
        {
          // one 1-D line per item, consecutive lanes on consecutive rows (odd row stride:
          // no bank conflicts); see phase1a
          const int n_rows = nc * G::ITEMS13;
          for (int it = tid; it < n_rows * G::N; it += kThreads)
            phase1a<P>(tb, sm.work + (it % n_rows) * G::RW, it / n_rows);
          __syncthreads();
          for (int it = tid; it < n_rows * Q; it += kThreads)
            phase1b<P>(tb, sm.work + (it % n_rows) * G::RW, it / n_rows);
          __syncthreads();
          for (int it = tid; it < n_rows * Q; it += kThreads)
            phase1c<P>(tb, sm.work + (it % n_rows) * G::RW, it / n_rows);
        }
    };
    auto phase_2 = [&](const int nc, const int bf) {
      for (int it = tid; it < nc * G::ITEMS2; it += kThreads)
        {
          const int cell = it / G::ITEMS2, r = it % G::ITEMS2;
          const int qz = r / Q, qx = r % Q;
          if constexpr (Cfg<P>::P2_CALL)
            phase2_call<P, QUAD>((uint32_t)((const unsigned char *)sm.coef[bf][cell] - smem_raw),
                                 (uint32_t)((const unsigned char *)(sm.work + cell * G::WORK) - smem_raw), qx, qz,
                                 sm.xq[qx], sm.xq[qz], sm.wq[qx] * sm.wq[qz]);
          else
            phase2<P, QUAD>(tb, sm.coef[bf][cell], sm.work + cell * G::WORK, qx, qz, sm.xq[qx], sm.xq[qz],
                            sm.wq[qx] * sm.wq[qz]);
        }
    };
    auto phase_3 = [&](const int nc) {
      if (!kFine)
        {
          for (int it = kThreads - 1 - tid; it < nc * G::ITEMS13; it += kThreads)
            phase3<P>(tb, sm.work + it * G::RW, sm.work + it * G::RW);
        }
      else
        {
          const int n_rows = nc * G::ITEMS13;
          for (int it = tid; it < n_rows * Q; it += kThreads)
            phase3a<P>(tb, sm.work + (it % n_rows) * G::RW, it / n_rows);
          __syncthreads();
          for (int it = tid; it < n_rows * Q; it += kThreads)
            phase3b<P>(tb, sm.work + (it % n_rows) * G::RW, it / n_rows);
          __syncthreads();
          for (int it = tid; it < n_rows * G::N; it += kThreads)
            phase3c<P>(tb, sm.work + (it % n_rows) * G::RW, it / n_rows);
        }
    };

    if (tid == 0)
      {
        sm.units[0]  = blockIdx.x;
        sm.n_claimed = 1;
        claim_ahead(0, kClaimDepth);
      }
    __syncthreads();

    if constexpr (!FUSED)
      {
        // cur = the batch in the work rows, nxt = the one being gathered; the iterators run
        // three batches ahead so that a claimed unit is known long before it is needed
        It cur_it;
        cur_it.j = 0, cur_it.b = cur_it.b_end = 0;
        enter(cur_it);
        Batch cur{}, nxt{}, nn{};
        It    nxt_it = cur_it, nn_it = cur_it;
        if (cur_it.valid)
          {
            cur = describe(cur_it);
            fetch_meta(cur.cell0, cur.nc);
            park_meta(0);
            nxt_it = advance(cur_it);
            nn_it  = nxt_it;
            if (nxt_it.valid)
              {
                nxt   = describe(nxt_it);
                nn_it = advance(nxt_it);
                if (nn_it.valid)
                  nn = describe(nn_it);
              }
          }
        __syncthreads();
        if (kPipe && cur_it.valid)
          {
            gather_issue(0);
            gather_store();
          }
        for (int i = 0; cur_it.valid; ++i)
          {
            const int nc = cur.nc, bf = i & 1;
            BP4_TICK(0)
            if (!kPipe)
              {
                gather_issue(bf);
                gather_store();
              }
            BP4_TICK(1)
            __syncthreads();
            BP4_TICK(2)
            BP4_TRACE(i, 0)
            BP4_TRACE(i, 4)
            if (tid == 0)
              claim_ahead(cur_it.j, kClaimDepth);
            if (nxt_it.valid)
              fetch_meta(nxt.cell0, nxt.nc); // lands during the phases
            phase_1(nc);
            BP4_TRACE(i, 5)
            BP4_TICK(3)
            __syncthreads();
            BP4_TICK(2)
            phase_2(nc, bf);
            BP4_TRACE(i, 7)
            BP4_TICK(4)
            __syncthreads();
            BP4_TICK(2)
            phase_3(nc);
            if (nxt_it.valid)
              park_meta(bf ^ 1);
            BP4_TRACE(i, 9)
            BP4_TICK(5)
            __syncthreads();
            BP4_TICK(2)
            BP4_TRACE(i, 1)
            // ---- memory window: the next batch's gather loads are issued, then the scatter goes
            // out while they travel
            if (kPipe && nxt_it.valid)
              gather_issue(bf ^ 1);
            BP4_TRACE(i, 12)
            scatter(bf);
            BP4_TICK(6)
            BP4_TRACE(i, 2)
            const It n3_it = nn_it.valid ? advance(nn_it) : nn_it;
            Batch    n3{};
            if (n3_it.valid)
              n3 = describe(n3_it);
            BP4_TICK(7)
            __syncthreads();
            BP4_TICK(2)
            BP4_TRACE(i, 3)
            if (kPipe && nxt_it.valid)
              gather_store(); // the barrier after it is the one at the top of the next iteration
            BP4_TRACE(i, 18)
            cur_it = nxt_it, cur = nxt;
            nxt_it = nn_it, nxt = nn;
            nn_it = n3_it, nn = n3;
          }
      }
    else
      {
        // ---- fused: do_cg_update4b / do_cg_update3b on the private runs ride along as "jobs".
        // job_issue (right after a barrier: every thread is done with the rows) copies [b, e) of
        // r, p, h and the diagonal into the staging rows asynchronously: every thread copies its
        // share in 16-byte pieces (LDGSTS) and lets the mbarrier count it once those have landed.
        // pre_job / post_job (one compute phase later) wait for the bytes and do the update from
        // shared memory.  A run is cut into a first job of at most JOB DoFs and a second one.
        // (cp.async.bulk was measured first: the request blocks the issuing warp for ~0.25 us
        // per 5 KB row and the rows queue up behind each other - whoever asked last kept the
        // whole block waiting at the next barrier for ~1 us per job.)
        constexpr int  JOB        = Stage<P>::JOB;
        JobSmem<JOB>  &js         = *reinterpret_cast<JobSmem<JOB> *>(smem_raw + sizeof(CellSmem<P, CPB, NC>));
        const uint32_t job_bar    = smem_u32(&js.mbar);
        uint32_t       job_parity = 0;
        int            trace_i    = 0;
        if (tid == 0)
          mbar_init(job_bar, kThreads);
        if (tid < 8 * (kThreads / 32))
          js.redw[tid >> 3][tid & 7] = 0.;
        auto job_split = [&](const uint32_t b, const uint32_t e) { return min(b + (uint32_t)JOB, e); };
        // A job [b, e) is handled in 16-byte pieces ("pairs" of DoFs, the first one at the even
        // index lo = b & ~1): thread tid owns the pairs tid + k * kThreads, for the copy and for
        // the update, so every shared-memory and global access of a job is a 128-bit one.
        constexpr int      KC   = ((JOB + 2) / 2 + kThreads - 1) / kThreads; // pairs per thread
        constexpr uint32_t ROWB = JobSmem<JOB>::ROW * 8u;                    // bytes per staging row
        constexpr int      KQ   = (JobSmem<JOB>::PREC / 2 + kThreads - 1) / kThreads;
        // `always`: the arrival (and the matching wait) happens for an empty range too - the job
        // then only carries the other asynchronous copies of its threads (metadata, descriptors)
        auto job_issue = [&](const uint32_t b, const uint32_t e, const bool always) {
          if (e > b)
            {
              const uint32_t lo = b & ~1u, n2 = (((e + 1u) & ~1u) - lo) >> 1;
              const uint32_t q0 = div3(b) & ~1u, nq2 = (((div3(e - 1u) + 2u) & ~1u) - q0) >> 1;
              const uint32_t s0 = smem_u32(&js.row[0][0]);
              const double  *gr = a.r + lo, *gp = a.p + lo, *gh = a.dst + lo;
#pragma unroll
              for (int k = 0; k < KC; ++k)
                {
                  const uint32_t c = tid + k * kThreads;
                  if (c < n2)
                    {
                      cp_async16(s0 + 16u * c, gr + 2 * c);
                      cp_async16(s0 + ROWB + 16u * c, gp + 2 * c);
                      cp_async16(s0 + 2u * ROWB + 16u * c, gh + 2 * c);
                    }
                }
#pragma unroll
              for (int k = 0; k < KQ; ++k)
                {
                  const uint32_t c = tid + k * kThreads;
                  if (c < nq2)
                    cp_async16(smem_u32(&js.prec[2 * c]), a.prec + q0 + 2 * c);
                }
            }
          if (e > b || always)
            asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(job_bar) : "memory");
        };
        auto job_wait = [&](const int ts) {
          mbar_wait(job_bar, job_parity);
          job_parity ^= 1u;
          BP4_TRACE(trace_i, ts)
        };
        // the full pairs of a job [b, e) start at the first even index >= b and end at the last
        // even index <= e; an odd first / last element is left to one thread each (job_edges)
        struct Pairs
        {
          double2 r[KC], p[KC], h[KC], d[KC];
          bool    ok[KC];
        };
        auto job_load = [&](Pairs &w, const uint32_t b, const uint32_t e) {
          const uint32_t lo = b & ~1u, c0 = b & 1u, q0 = div3(b) & ~1u;
          const uint32_t nf = (e & ~1u) > lo + 2u * c0 ? (((e & ~1u) - lo) >> 1) - c0 : 0u; // full pairs
#pragma unroll
          for (int k = 0; k < KC; ++k)
            {
              const uint32_t t = tid + k * kThreads;
              w.ok[k]          = t < nf;
              const uint32_t cc = c0 + (w.ok[k] ? t : 0u), i0 = lo + 2u * cc;
              w.r[k]   = *reinterpret_cast<const double2 *>(&js.row[0][2 * cc]);
              w.p[k]   = *reinterpret_cast<const double2 *>(&js.row[1][2 * cc]);
              w.h[k]   = *reinterpret_cast<const double2 *>(&js.row[2][2 * cc]);
              w.d[k].x = js.prec[div3(min(i0, e - 1u)) - q0];
              w.d[k].y = js.prec[div3(min(i0 + 1u, e - 1u)) - q0];
            }
        };
        // f(i) for the odd element at either end of [b, e), on the last two threads of the block
        auto job_edges = [&](const uint32_t b, const uint32_t e, auto &&f) {
          if (tid == kThreads - 1 && (b & 1u))
            f(b);
          if (tid == kThreads - 2 && (e & 1u)) // e - 1 is even: never the odd first element
            f(e - 1u);
        };
        // the scalars of do_cg_update4b (sc.alpha, beta, first, update_x, c1, c2): the launch
        // arguments, or (DEV) derived from the solver state exactly as cell_range (bp4_capi.cu)
        // derives them on the host
        CellArgs dev_args;
        if constexpr (DEV)
          {
            dev_args        = a;
            const double al = a.state->alpha, ao = a.state->alpha_old, bo = a.state->beta_old;
            dev_args.alpha    = al;
            dev_args.beta     = a.state->beta;
            dev_args.first    = al == 0. ? 1 : 0;
            dev_args.update_x = (al != 0. && ao != 0.) ? 1 : 0;
            dev_args.c1       = dev_args.update_x ? __dadd_rn(al, __ddiv_rn(ao, bo)) : 0.;
            dev_args.c2       = dev_args.update_x ? __ddiv_rn(ao, bo) : 0.;
          }
        const CellArgs &sc = DEV ? dev_args : a;
        auto pre_one = [&](const uint32_t i, const double rr, const double pp, const double hh, const double pr) {
          if (sc.first)
            a.p[i] = -pr * rr;
          else
            {
              if (sc.update_x)
                atomicAdd(a.x + i, sc.c1 * pp + sc.c2 * pr * rr);
              const double rn = rr + sc.alpha * hh;
              a.r[i]          = rn;
              a.p[i]          = sc.beta * pp - pr * rn;
            }
          a.dst[i] = 0.;
        };
        // do_cg_update4b<3,double,true> (solver_cg_optimized.h:65-161) on [b, e)
        auto pre_job = [&](const uint32_t b, const uint32_t e, const bool always, const int ts) {
          if (e > b || always)
            job_wait(ts);
          if (e <= b)
            return;
          Pairs w;
          job_load(w, b, e);
          const uint32_t lo = b & ~1u, c0 = b & 1u, q0 = div3(b) & ~1u;
#pragma unroll
          for (int k = 0; k < KC; ++k)
            if (w.ok[k])
              {
                const uint32_t i0 = lo + 2u * (c0 + tid + k * kThreads);
                if (sc.first)
                  *reinterpret_cast<double2 *>(a.p + i0) = make_double2(-w.d[k].x * w.r[k].x, -w.d[k].y * w.r[k].y);
                else
                  {
                    if (sc.update_x) // x += ..., fire and forget: x is not read in this kernel
                      {
                        atomicAdd(a.x + i0, sc.c1 * w.p[k].x + sc.c2 * w.d[k].x * w.r[k].x);
                        atomicAdd(a.x + i0 + 1, sc.c1 * w.p[k].y + sc.c2 * w.d[k].y * w.r[k].y);
                      }
                    const double r0 = w.r[k].x + sc.alpha * w.h[k].x, r1 = w.r[k].y + sc.alpha * w.h[k].y;
                    *reinterpret_cast<double2 *>(a.r + i0) = make_double2(r0, r1);
                    *reinterpret_cast<double2 *>(a.p + i0) =
                      make_double2(sc.beta * w.p[k].x - w.d[k].x * r0, sc.beta * w.p[k].y - w.d[k].y * r1);
                  }
                *reinterpret_cast<double2 *>(a.dst + i0) = make_double2(0., 0.);
              }
          job_edges(b, e, [&](const uint32_t i) {
            pre_one(i, js.row[0][i - lo], js.row[1][i - lo], js.row[2][i - lo], js.prec[div3(i) - q0]);
          });
        };
        // do_cg_update3b<3,double> (solver_cg_optimized.h:12-61) on [b, e): the seven sums of a
        // thread stay in registers from the first to the second post job of an iteration, then
        // one warp reduction and a plain add into the warp's own slots (post_sums)
        auto post_job = [&](double (&sj)[7], const uint32_t b, const uint32_t e, const bool always, const int ts) {
          if (e > b || always)
            job_wait(ts);
          if (e <= b)
            return;
          Pairs w;
          job_load(w, b, e);
          const uint32_t lo = b & ~1u, q0 = div3(b) & ~1u;
#pragma unroll
          for (int k = 0; k < KC; ++k)
            {
              // (a thread without a pair reads whatever sits at the first pair's slot: mask all of it)
              if (w.ok[k])
                {
                  post_terms(sj, w.r[k].x, w.p[k].x, w.h[k].x, w.d[k].x);
                  post_terms(sj, w.r[k].y, w.p[k].y, w.h[k].y, w.d[k].y);
                }
            }
          job_edges(b, e, [&](const uint32_t i) {
            post_terms(sj, js.row[0][i - lo], js.row[1][i - lo], js.row[2][i - lo], js.prec[div3(i) - q0]);
          });
        };
        // Transposed butterfly: at every step a lane keeps half of its values and hands the
        // other half to its partner, so 7 sums over 32 lanes take 9 shuffles instead of 35;
        // lane 4 m ends up with the warp's total of sum m.
        auto post_sums = [&](double (&sj)[7]) {
          const int  lane = tid & 31;
          const bool h16 = lane & 16, h8 = lane & 8, h4 = lane & 4;
          double     w[4], u[2], t;
#pragma unroll
          for (int k = 0; k < 4; ++k)
            {
              const double hi = k + 4 < 7 ? sj[k + 4] : 0.;
              w[k] = (h16 ? hi : sj[k]) + __shfl_xor_sync(0xffffffffu, h16 ? sj[k] : hi, 16);
            }
#pragma unroll
          for (int k = 0; k < 2; ++k)
            u[k] = (h8 ? w[k + 2] : w[k]) + __shfl_xor_sync(0xffffffffu, h8 ? w[k] : w[k + 2], 8);
          t = (h4 ? u[1] : u[0]) + __shfl_xor_sync(0xffffffffu, h4 ? u[0] : u[1], 4);
          t += __shfl_xor_sync(0xffffffffu, t, 2);
          t += __shfl_xor_sync(0xffffffffu, t, 1);
          if ((lane & 3) == 0 && lane < 28)
            js.redw[tid >> 5][lane >> 2] += t;
        };

        // The descriptors of the batches i-2 .. i+4 live in a ring in shared memory and are read
        // where they are needed; the only iterator kept in registers is the head (batch i+3).
        // vm: bit k-1 set <=> batch i+k exists (k = 1..3).  All of this is uniform over the block.
        auto ring_put = [&](const uint32_t k, const It &it) { // synchronous (prologue)
          const uint4 w0 = __ldg(reinterpret_cast<const uint4 *>(a.batch + it.b));
          const uint4 w1 = __ldg(reinterpret_cast<const uint4 *>(a.batch + it.b) + 1);
          if (tid == 0)
            {
              uint4 *dst = reinterpret_cast<uint4 *>(&js.ring[k & 7u]);
              dst[0] = w0, dst[1] = w1;
            }
        };
        auto ring_fetch = [&](const uint32_t k, const It &it) { // asynchronous, see job_issue(always)
          if (tid < 2)
            cp_async16(smem_u32(&js.ring[k & 7u]) + 16u * tid,
                       reinterpret_cast<const unsigned char *>(a.batch + it.b) + 16u * tid);
        };
        It hd;
        hd.j = 0, hd.b = hd.b_end = 0;
        enter(hd);
        const bool any = hd.valid;
        uint32_t   vm  = 0;
        if (any)
          {
            ring_put(0, hd);
            for (uint32_t k = 1; k <= 3; ++k)
              if (hd.valid)
                {
                  hd = advance(hd);
                  if (hd.valid)
                    {
                      ring_put(k, hd);
                      vm |= 1u << (k - 1);
                    }
                }
          }
        __syncthreads();
        if (any)
          {
            // batch 0: metadata and the pre-update of its runs, synchronously
            const BatchDesc &d0 = js.ring[0];
            fetch_meta(d0.cell0, (int)d0.n_cells);
            park_meta(0);
            const uint32_t pb = d0.pre_begin, pe = d0.pre_end, pm = job_split(pb, pe);
            job_issue(pb, pm, false);
            pre_job(pb, pm, false, 16);
            __syncthreads();
            job_issue(pm, pe, false);
            pre_job(pm, pe, false, 17);
            __syncthreads();
            if (kPipe)
              {
                gather_issue(0);
                gather_store();
              }
          }
        // Schedule of one iteration - each job is requested right after a barrier and consumed
        // before the next one, one compute phase later:
        //   phase 1: first part of the next batch's pre-update      phase 2: its second part
        //   phase 3: first part of the post-update of the runs finished two batches ago (their
        //            REDs went out a whole batch earlier)
        //   window : its second part; it is consumed last, after the gathered values have been
        //            parked - the copies that travel while the scatter's REDs go out are slow
        int    i = 0;
        double sj[7]; // lives from the end of phase 3 to the end of the iteration only
        for (bool cur_ok = any; cur_ok; ++i)
          {
            const int bf = i & 1;
            trace_i      = i;
            if (!kPipe)
              {
                gather_issue(bf);
                gather_store();
              }
            __syncthreads();
            BP4_TRACE(i, 0)
            BP4_TRACE(i, 4)
            const int        nc = (int)js.ring[i & 7].n_cells;
            const BatchDesc &dn = js.ring[(i + 1) & 7];
            {
              // the arrival also covers the descriptor requested in the previous window
              const uint32_t pb = (vm & 1u) ? dn.pre_begin : 0u, pe = (vm & 1u) ? dn.pre_end : 0u;
              job_issue(pb, job_split(pb, pe), true);
            }
            if (tid == 0)
              claim_ahead(hd.j, kClaimDepthFused);
            if (vm & 1u)
              meta_async(bf ^ 1, dn.cell0, (int)dn.n_cells);
            phase_1(nc);
            BP4_TRACE(i, 5)
            {
              const uint32_t pb = (vm & 1u) ? dn.pre_begin : 0u, pe = (vm & 1u) ? dn.pre_end : 0u;
              const uint32_t pm = job_split(pb, pe);
              pre_job(pb, pm, true, 16);
              BP4_TRACE(i, 6)
              __syncthreads();
              job_issue(pm, pe, false);
              phase_2(nc, bf);
              BP4_TRACE(i, 7)
              pre_job(pm, pe, false, 17);
              BP4_TRACE(i, 8)
            }
            __syncthreads();
            const BatchDesc &dold = js.ring[(i + 6) & 7]; // batch i - 2
            const uint32_t   ob = i >= 2 ? dold.post_begin : 0u, oe = i >= 2 ? dold.post_end : 0u;
            const uint32_t   om = job_split(ob, oe);
            job_issue(ob, om, true); // carries the next batch's metadata too
            phase_3(nc);
            BP4_TRACE(i, 9)
#pragma unroll
            for (int k = 0; k < 7; ++k)
              sj[k] = 0.;
            post_job(sj, ob, om, true, 14);
            BP4_TRACE(i, 10)
            // every consumer of this block's stores and REDs is a thread of this block (its loads
            // and asynchronous copies): the barriers order them.  No GPU-scope fence here:
            // __threadfence is MEMBAR.SC.GPU + CCTL.IVALL, measured 0.7 us per batch and the
            // whole L1 gone each time.
            __syncthreads();
            BP4_TRACE(i, 1)
            job_issue(om, oe, false);
            // ---- memory window
            if (kPipe && (vm & 1u))
              gather_issue(bf ^ 1); // the next batch's DoFs (pre-updated during this batch)
            BP4_TRACE(i, 12)
            scatter(bf);
            BP4_TRACE(i, 2)
            // the head moves on to batch i + 4
            bool hv = false;
            if (vm & 4u)
              {
                hd = advance(hd);
                hv = hd.valid;
                if (hv)
                  ring_fetch(i + 4, hd);
              }
            __syncthreads();
            BP4_TRACE(i, 3)
            if (kPipe && (vm & 1u))
              gather_store(); // the barrier after it is the one at the top of the next iteration
            BP4_TRACE(i, 18)
            if (oe > ob)
              {
                post_job(sj, om, oe, false, 15);
                post_sums(sj);
              }
            BP4_TRACE(i, 13)
            cur_ok = (vm & 1u) != 0;
            vm     = (vm >> 1) | (hv ? 4u : 0u);
          }
        if (any)
          {
            // the post-updates of the last two batches, synchronously
            __syncthreads();
#pragma unroll
            for (int k = 0; k < 7; ++k)
              sj[k] = 0.;
            for (int k = max(i - 2, 0); k < i; ++k)
              {
                const BatchDesc &dk = js.ring[k & 7];
                const uint32_t   ob = dk.post_begin, oe = dk.post_end, om = job_split(ob, oe);
                job_issue(ob, om, false);
                post_job(sj, ob, om, false, 14);
                __syncthreads();
                job_issue(om, oe, false);
                post_job(sj, om, oe, false, 15);
                __syncthreads();
              }
            post_sums(sj);
          }
        __syncthreads();
        if (tid < 7)
          {
            double v = 0.;
#pragma unroll
            for (int wp = 0; wp < kThreads / 32; ++wp)
              v += js.redw[wp][tid];
            atomicAdd(a.acc + tid, v);
          }
      }
    BP4_TICK_FLUSH
  }

  // block-reduce K partial sums and atomically add them to acc[0..K)
  template <int K>
  __device__ __forceinline__ void block_accumulate(double (&s)[K], double *acc)
  {
    __shared__ double red[K][32];
    const int         lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int         nw = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int k = 0; k < K; ++k)
      {
        s[k] = warp_sum(s[k]);
        if (lane == 0)
          red[k][warp] = s[k];
      }
    __syncthreads();
    if (warp == 0)
      {
#pragma unroll
        for (int k = 0; k < K; ++k)
          {
            double v = lane < nw ? red[k][lane] : 0.;
            v        = warp_sum(v);
            if (lane == 0)
              atomicAdd(acc + k, v);
          }
      }
  }

  // the ordered form of block_accumulate (deterministic mode): the same warp / block tree, then the
  // block's K partials go to ds.slot[k][blockIdx.x]; the last block to take a ticket sums the
  // slots in a fixed order (thread t: blocks t, t + blockDim.x, ...; then the tree) and adds the
  // totals to acc[0..K).  The result depends on the data and gridDim.x only.  The last block
  // re-arms the ticket, so a replayed graph finds it at zero.
  template <int K>
  __device__ __forceinline__ void block_accumulate_ordered(double (&s)[K], double *acc, const DetSlots ds)
  {
    __shared__ double red[K][32];
    __shared__ int    is_last;
    const int         lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int         nw = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int k = 0; k < K; ++k)
      {
        s[k] = warp_sum(s[k]);
        if (lane == 0)
          red[k][warp] = s[k];
      }
    __syncthreads();
    if (warp == 0)
      {
        double v[K];
#pragma unroll
        for (int k = 0; k < K; ++k)
          v[k] = warp_sum(lane < nw ? red[k][lane] : 0.);
        if (lane == 0)
          {
#pragma unroll
            for (int k = 0; k < K; ++k)
              ds.slot[(size_t)k * gridDim.x + blockIdx.x] = v[k];
            __threadfence();
            is_last = atomicAdd(ds.ticket, 1u) == gridDim.x - 1;
          }
      }
    __syncthreads();
    if (!is_last)
      return;
    __threadfence();
#pragma unroll
    for (int k = 0; k < K; ++k)
      {
        double t = 0.;
        for (unsigned b = threadIdx.x; b < gridDim.x; b += blockDim.x)
          t += __ldcg(ds.slot + (size_t)k * gridDim.x + b);
        t = warp_sum(t);
        if (lane == 0)
          red[k][warp] = t;
      }
    __syncthreads();
    if (warp == 0)
      {
#pragma unroll
        for (int k = 0; k < K; ++k)
          {
            const double v = warp_sum(lane < nw ? red[k][lane] : 0.);
            if (lane == 0)
              acc[k] += v;
          }
        if (lane == 0)
          *ds.ticket = 0u;
      }
  }

  template <bool DET, int K>
  __device__ __forceinline__ void accumulate(double (&s)[K], double *acc, const DetSlots ds)
  {
    if constexpr (DET)
      block_accumulate_ordered<K>(s, acc, ds);
    else
      block_accumulate<K>(s, acc);
  }

  // ---------------------------------------------------------------------------------------
  // streaming kernels
  // ---------------------------------------------------------------------------------------
  // do_cg_update4b<3,double,true>, solver_cg_optimized.h:65-161, over [begin, end): the DoFs that
  // are not private to one cell-batch range (all of them when the numbering has no such group).
  // Also clears the reduction scratch of this iteration (stream order: before any post).
  // DEV: the four scalars come from the solver state of a device-resident solve (st).
  template <bool DEV>
  __global__ void __launch_bounds__(256) pre_kernel(const uint64_t begin, const uint64_t end,
                                                    double *__restrict__ h, double *__restrict__ x,
                                                    double *__restrict__ r, double *__restrict__ p,
                                                    const double *__restrict__ prec,
                                                    double alpha, double beta,
                                                    double alpha_old, double beta_old,
                                                    double *acc_to_zero, const SolveState *st)
  {
    if constexpr (DEV)
      {
        alpha     = st->alpha;
        beta      = st->beta;
        alpha_old = st->alpha_old;
        beta_old  = st->beta_old;
      }
    if (acc_to_zero && blockIdx.x == 0 && threadIdx.x < 8)
      acc_to_zero[threadIdx.x] = 0.;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const double   c1 = alpha_old != 0. ? alpha + alpha_old / beta_old : 0.;
    const double   c2 = alpha_old != 0. ? alpha_old / beta_old : 0.;
    // U independent elements per trip: all their loads are in flight together.  Measured at Q4
    // s=18: U = 1 -> 0.496 ms, 2 -> 0.484, 4 -> 0.474 (6.3 TB/s), 6/8 -> 0.48
    constexpr int U = 4;
    for (uint64_t i0 = begin + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < end; i0 += U * stride)
      {
        double pr[U], ri[U], pi[U], hi[U], xi[U];
#pragma unroll
        for (int u = 0; u < U; ++u)
          {
            const uint64_t i  = i0 + u * stride;
            const bool     ok = i < end;
            pr[u] = ok ? prec[i / 3] : 0.;
            ri[u] = ok ? r[i] : 0.;
            pi[u] = ok && alpha != 0. ? p[i] : 0.;
            hi[u] = ok && alpha != 0. ? h[i] : 0.;
            xi[u] = ok && alpha_old != 0. ? x[i] : 0.;
          }
#pragma unroll
        for (int u = 0; u < U; ++u)
          {
            const uint64_t i = i0 + u * stride;
            if (i < end)
              {
                if (alpha == 0.)
                  p[i] = -pr[u] * ri[u];
                else
                  {
                    if (alpha_old != 0.)
                      x[i] = xi[u] + (c1 * pi[u] + c2 * pr[u] * ri[u]);
                    const double rn = ri[u] + alpha * hi[u];
                    r[i] = rn;
                    p[i] = beta * pi[u] - pr[u] * rn;
                  }
                h[i] = 0.;
              }
          }
      }
  }

  // do_cg_update3b<3,double>, solver_cg_optimized.h:12-61, over [begin, end) -> acc[7]
  // DET: ordered cross-block sum (block_accumulate_ordered) instead of atomics
  template <bool DET>
  __global__ void __launch_bounds__(256) post_kernel(const uint64_t begin, const uint64_t end,
                                                     const double *__restrict__ r,
                                                     const double *__restrict__ d,
                                                     const double *__restrict__ h,
                                                     const double *__restrict__ prec, double *acc,
                                                     const DetSlots ds)
  {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    double         s[7]   = {0., 0., 0., 0., 0., 0., 0.};
    // U independent element groups per trip: all their loads are in flight together.  Measured at
    // Q4 s=18: U = 1 -> 0.233 ms, 4 -> 0.211 ms (6.45 TB/s), 2 and 8 slower
    constexpr int U = 4;
    for (uint64_t i0 = begin + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < end; i0 += U * stride)
      {
        double rr[U], dd[U], hh[U], pp[U];
#pragma unroll
        for (int u = 0; u < U; ++u)
          {
            const uint64_t i  = i0 + u * stride;
            const bool     ok = i < end;
            rr[u] = ok ? r[i] : 0.;
            dd[u] = ok ? d[i] : 0.;
            hh[u] = ok ? h[i] : 0.;
            pp[u] = ok ? prec[i / 3] : 0.;
          }
#pragma unroll
        for (int u = 0; u < U; ++u)
          post_terms(s, rr[u], dd[u], hh[u], pp[u]);
      }
    accumulate<DET>(s, acc, ds);
  }

  __global__ void __launch_bounds__(256) fixup_kernel(const uint64_t n, const uint32_t *__restrict__ con,
                                                      double *__restrict__ dst,
                                                      const double *__restrict__ src)
  {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n)
      dst[con[i]] = src[con[i]];
  }

  // dst = s*dst + a*src   (s == 0: dst = a*src without reading dst); DEV: s = *s_dev
  template <bool DEV>
  __global__ void __launch_bounds__(256) sadd_kernel(const uint64_t n, double *__restrict__ dst,
                                                     double s, const double a,
                                                     const double *__restrict__ src, const double *s_dev)
  {
    if constexpr (DEV)
      s = *s_dev;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
      dst[i] = (s == 0. ? 0. : s * dst[i]) + a * src[i];
  }

  template <bool DET>
  __global__ void __launch_bounds__(256) dot_kernel(const uint64_t n, const double *__restrict__ a,
                                                    const double *__restrict__ b, double *acc, const DetSlots ds)
  {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    double         s[1]   = {0.};
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
      s[0] += a[i] * b[i];
    accumulate<DET>(s, acc, ds);
  }

  // g += a*h ; acc += g.w   (w may alias g)
  template <bool DET>
  __global__ void __launch_bounds__(256) add_and_dot_kernel(const uint64_t n, double *g, const double a,
                                                            const double *__restrict__ h,
                                                            const double *w, double *acc, const DetSlots ds)
  {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    double         s[1]   = {0.};
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
      {
        const double gi = g[i] + a * h[i];
        const double wi = (w == g) ? gi : w[i];
        g[i]            = gi;
        s[0] += gi * wi;
      }
    accumulate<DET>(s, acc, ds);
  }

  __global__ void __launch_bounds__(256) nonzero_kernel(const uint64_t n, const double *__restrict__ v,
                                                        int *flag)
  {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    int            nz     = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
      nz |= (v[i] != 0.);
    if (__any_sync(0xffffffffu, nz) && (threadIdx.x & 31) == 0)
      atomicOr(flag, 1);
  }

  // hand k reduced values to the host through mapped pinned memory: values first, then a system
  // fence, then the sequence number the host is spinning on (a few microseconds less per host
  // round trip than a device-to-host copy plus stream synchronisation)
  // The accumulators are cleared on the way out: the next reduction needs no memset.
  __global__ void publish_kernel(double *acc, const int k, volatile double *host_vals,
                                 volatile unsigned long long *host_seq, const unsigned long long seq)
  {
    if (threadIdx.x == 0 && blockIdx.x == 0)
      {
        for (int i = 0; i < k; ++i)
          {
            host_vals[i] = acc[i];
            acc[i]       = 0.;
          }
        __threadfence_system();
        *host_seq = seq;
      }
  }

  // ghost exchange helpers: buf[k] = v[idx[k]] and v[idx[k]] += buf[k]
  __global__ void __launch_bounds__(256) pack_kernel(const uint64_t n, const uint32_t *__restrict__ idx,
                                                     const double *__restrict__ v, double *__restrict__ buf)
  {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n)
      buf[i] = v[idx[i]];
  }
  __global__ void __launch_bounds__(256) unpack_add_kernel(const uint64_t n, const uint32_t *__restrict__ idx,
                                                           const double *__restrict__ buf, double *v)
  {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n)
      atomicAdd(v + idx[i], buf[i]); // export lists of different peers may repeat an index
  }
  // out[i] = in[3 i]
  __global__ void __launch_bounds__(256) stride3_kernel(const uint64_t n, const double *__restrict__ in,
                                                        double *__restrict__ out)
  {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n)
      out[i] = in[3 * i];
  }

  // dst[3i+c] = diag[i]*src[3i+c]   (diagonal_matrix_blocked.h:21-26)
  __global__ void __launch_bounds__(256) jacobi_kernel(const uint64_t n, double *__restrict__ dst,
                                                       const double *__restrict__ src,
                                                       const double *__restrict__ diag)
  {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
      dst[i] = diag[i / 3] * src[i];
  }

  // x += c1*d + c2*prec*g   (solver_cg_optimized.h:260-288)
  __global__ void __launch_bounds__(256) xfinal_kernel(const uint64_t n, double *__restrict__ x,
                                                       const double *__restrict__ d,
                                                       const double *__restrict__ g,
                                                       const double *__restrict__ prec, const double c1,
                                                       const double c2)
  {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
      x[i] += c1 * d[i] + c2 * prec[i / 3] * g[i];
  }

  // ---------------------------------------------------------------------------------------
  // device-resident CG solves (bp4_solve_cg, bp4_solve_cg_merged): the vector sweeps the plain
  // solve needs beyond the operator, the scalar recurrences of both solvers and the final x update
  // ---------------------------------------------------------------------------------------
  // h = P g (diagonal_matrix_blocked.h:21-26) and acc += g.h in one sweep
  template <bool DET>
  __global__ void __launch_bounds__(256) jacobi_dot_kernel(const uint64_t n, double *__restrict__ h,
                                                           const double *__restrict__ g,
                                                           const double *__restrict__ diag, double *acc,
                                                           const DetSlots ds)
  {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    double         s[1]   = {0.};
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
      {
        const double gi = g[i], hi = diag[i / 3] * gi;
        h[i]            = hi;
        s[0] += gi * hi;
      }
    accumulate<DET>(s, acc, ds);
  }

  // x += alpha d; g += alpha h; acc += g.g   (SolverCG: x.add, g.add_and_dot), alpha from the state.
  // DET: x + alpha d rounded as bp4_add rounds it (product, then sum), so that the iterates equal the
  // host-driven solver's bit for bit; the default form contracts it into one FMA
  template <bool DET>
  __global__ void __launch_bounds__(256) cg_xg_kernel(const uint64_t n, double *__restrict__ x,
                                                      double *__restrict__ g, const double *__restrict__ d,
                                                      const double *__restrict__ h, const SolveState *st,
                                                      double *acc, const DetSlots ds)
  {
    const double   alpha  = st->alpha;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    double         s[1]   = {0.};
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
      {
        if constexpr (DET)
          x[i] = __dadd_rn(x[i], __dmul_rn(alpha, d[i]));
        else
          x[i] += alpha * d[i];
        const double gi = g[i] + alpha * h[i];
        g[i]            = gi;
        s[0] += gi * gi;
      }
    accumulate<DET>(s, acc, ds);
  }

  // ReductionControl::check (host/solver_control.h) for a step > 0
  __device__ int control_check(SolveState &st, const uint32_t step, const double value)
  {
    st.step       = step;
    st.last_value = value;
    if (value < st.reduced_tol || value <= st.tol)
      return 1;
    if (step >= st.max_steps || isnan(value))
      return 2;
    return 0;
  }

  // The scalar work of one iteration on one thread, in the host's association order with
  // explicitly rounded operations (the host build emits no FMA): for equal sums the scalars are
  // bit-identical to those of the host-driven solvers.  acc is left zero for the next reduction.
  //   kMergedStep: SolverCGFullMerge::solve (host/solver_cg_optimized.h) from the seven sums
  //   kPlainInit : gh = g.h before the first iteration (acc[2])
  //   kPlainAlpha: alpha = gh / d.h (acc[0])
  //   kPlainCheck: residual from g.g (acc[1]), the check, beta from the new g.h (acc[2])
  // kMergedStep and kPlainCheck end the iteration: they set the loop condition.
  __global__ void solve_scalar_kernel(const int kind, SolveState *stp, double *acc,
                                      const cudaGraphConditionalHandle loop)
  {
    if (threadIdx.x != 0)
      return;
    SolveState &st = *stp;
    if (kind == kSolveMergedStep)
      {
        double s[7];
        for (int k = 0; k < 7; ++k)
          s[k] = acc[k], acc[k] = 0.;
        const uint32_t it         = st.step + 1;
        const double   prev_alpha = st.alpha, prev_beta = st.beta;
        const double   alpha      = __ddiv_rn(s[6], s[0]);
        const double   res        = __dsqrt_rn(__dadd_rn(__dadd_rn(s[3], __dmul_rn(__dmul_rn(2., alpha), s[2])),
                                                         __dmul_rn(__dmul_rn(alpha, alpha), s[1])));
        const int      state      = control_check(st, it, res);
        st.alpha    = alpha;
        st.beta_old = prev_beta;
        if (state == 0) // the arguments of iteration it + 1: alpha_old only on odd iterations
          {
            st.beta      = __ddiv_rn(__dmul_rn(alpha, __dadd_rn(s[4], __dmul_rn(alpha, s[5]))), s[6]);
            st.alpha_old = ((it + 1) & 1u) ? prev_alpha : 0.;
          }
        else // kept for the final x update
          st.alpha_old = prev_alpha;
        st.state = state;
        cudaGraphSetConditional(loop, state == 0 ? 1u : 0u);
      }
    else if (kind == kSolvePlainInit)
      {
        st.gh  = acc[2];
        acc[2] = 0.;
      }
    else if (kind == kSolvePlainAlpha)
      {
        st.alpha = __ddiv_rn(st.gh, acc[0]);
        acc[0]   = 0.;
      }
    else // kSolvePlainCheck
      {
        const int state = control_check(st, st.step + 1, __dsqrt_rn(fabs(acc[1])));
        st.state        = state;
        // after the stopping check only the temporaries h, d and gh / beta change (the loop
        // body runs to its end)
        const double beta_den = st.gh;
        st.gh                 = acc[2];
        st.beta               = __ddiv_rn(st.gh, beta_den);
        acc[1] = acc[2] = 0.;
        cudaGraphSetConditional(loop, state == 0 ? 1u : 0u);
      }
  }

  // the pending x update of SolverCGFullMerge after its last iteration
  // (solver_cg_optimized.h:256-288): odd step x += alpha d, even step bp4_x_finalize_even's formula.
  // DET: the odd step rounded as bp4_add rounds it (see cg_xg_kernel)
  template <bool DET>
  __global__ void __launch_bounds__(256) solve_final_kernel(const uint64_t n, double *__restrict__ x,
                                                            const double *__restrict__ d,
                                                            const double *__restrict__ g,
                                                            const double *__restrict__ prec,
                                                            const SolveState *st)
  {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const double   alpha  = st->alpha;
    if (st->step & 1u)
      {
        for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
          if constexpr (DET)
            x[i] = __dadd_rn(x[i], __dmul_rn(alpha, d[i]));
          else
            x[i] += alpha * d[i];
        return;
      }
    const double c2 = __ddiv_rn(st->alpha_old, st->beta_old), c1 = __dadd_rn(alpha, c2);
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
      x[i] += c1 * d[i] + c2 * prec[i / 3] * g[i];
  }

  // inverse diagonal of the scalar GLL(p+1) Laplacian (poisson_operator.h:392-426): one
  // thread per (cell, node); collocation makes the unit-vector gradient non-zero only on
  // the three grid lines through the node.  gll holds x[N], w[N], Dg[N][N] (Dg[i][q]=l_i'(x_q)).
  __device__ __forceinline__ void metric_at(const double *cf, const int n_coef, double x, double y, double z,
                                            double w, double &g00, double &g01, double &g02, double &g11,
                                            double &g12, double &g22)
  {
    double r0[3], r1[3], r2[3];
    if (n_coef == 24)
      {
#pragma unroll
        for (int d = 0; d < 3; ++d)
          {
            const double v1 = cf[3 + d], v3 = cf[6 + d], v4 = cf[9 + d], v9 = cf[12 + d],
                         v10 = cf[15 + d], v12 = cf[18 + d], v13 = cf[21 + d];
            r0[d] = (v1 + z * v10) + y * (v4 + z * v13);
            r1[d] = (v3 + z * v12) + x * (v4 + z * v13);
            r2[d] = (v9 + y * v12) + x * (v10 + y * v13);
          }
      }
    else // all 27 coefficients of X = sum v_{a+3b+9c} x^a y^b z^c (poisson_operator.h:577-602)
      {
        const double px[3] = {1., x, x * x}, py[3] = {1., y, y * y}, pz[3] = {1., z, z * z};
        const double dx[3] = {0., 1., x + x}, dy[3] = {0., 1., y + y}, dz[3] = {0., 1., z + z};
        for (int d = 0; d < 3; ++d)
          {
            double s0 = 0., s1 = 0., s2 = 0.;
            for (int c = 0; c < 3; ++c)
              for (int b = 0; b < 3; ++b)
                for (int a = 0; a < 3; ++a)
                  {
                    const double v = cf[3 * (a + 3 * b + 9 * c) + d];
                    s0 += v * dx[a] * py[b] * pz[c];
                    s1 += v * px[a] * dy[b] * pz[c];
                    s2 += v * px[a] * py[b] * dz[c];
                  }
            r0[d] = s0, r1[d] = s1, r2[d] = s2;
          }
      }
    double k0[3], k1[3], k2[3];
    k0[0] = r1[1] * r2[2] - r1[2] * r2[1];
    k0[1] = r1[2] * r2[0] - r1[0] * r2[2];
    k0[2] = r1[0] * r2[1] - r1[1] * r2[0];
    k1[0] = r2[1] * r0[2] - r2[2] * r0[1];
    k1[1] = r2[2] * r0[0] - r2[0] * r0[2];
    k1[2] = r2[0] * r0[1] - r2[1] * r0[0];
    k2[0] = r0[1] * r1[2] - r0[2] * r1[1];
    k2[1] = r0[2] * r1[0] - r0[0] * r1[2];
    k2[2] = r0[0] * r1[1] - r0[1] * r1[0];
    const double det = r0[0] * k0[0] + r0[1] * k0[1] + r0[2] * k0[2];
    const double sc  = w / det;
    g00 = sc * (k0[0] * k0[0] + k0[1] * k0[1] + k0[2] * k0[2]);
    g01 = sc * (k0[0] * k1[0] + k0[1] * k1[1] + k0[2] * k1[2]);
    g02 = sc * (k0[0] * k2[0] + k0[1] * k2[1] + k0[2] * k2[2]);
    g11 = sc * (k1[0] * k1[0] + k1[1] * k1[1] + k1[2] * k1[2]);
    g12 = sc * (k1[0] * k2[0] + k1[1] * k2[1] + k1[2] * k2[2]);
    g22 = sc * (k2[0] * k2[0] + k2[1] * k2[1] + k2[2] * k2[2]);
  }

  __global__ void __launch_bounds__(128) diag_kernel(const int p, const uint64_t n_cells,
                                                     const uint32_t *__restrict__ entity_index,
                                                     const double *__restrict__ coef, const int n_coef,
                                                     const double *__restrict__ gll, double *diag,
                                                     const int stride)
  {
    const int      N  = p + 1, N3 = N * N * N;
    const uint64_t id = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= n_cells * N3)
      return;
    const uint64_t cell = id / N3;
    const int      l = (int)(id % N3), i = l % N, j = (l / N) % N, k = l / (N * N);
    const int      ex = i == 0 ? 0 : (i == p ? 2 : 1), ey = j == 0 ? 0 : (j == p ? 2 : 1),
              ez = k == 0 ? 0 : (k == p ? 2 : 1);
    const uint32_t base = entity_index[cell * 27 + ex + 3 * ey + 9 * ez];
    if (base == 0xFFFFFFFFu)
      return;
    const int oi = ex == 1 ? i - 1 : 0, oj = ey == 1 ? j - 1 : 0, ok = ez == 1 ? k - 1 : 0;
    const int sx = ex == 1 ? p - 1 : 1, sy = ey == 1 ? p - 1 : 1;
    const int pos = oi + sx * (oj + sy * ok);
    const double *x = gll, *w = gll + N, *Dg = gll + 2 * N;
    const double *cf = coef + cell * n_coef;
    double        s = 0., g00, g01, g02, g11, g12, g22;
    for (int q = 0; q < N; ++q)
      {
        const double dx = Dg[i * N + q], dy = Dg[j * N + q], dz = Dg[k * N + q];
        metric_at(cf, n_coef, x[q], x[j], x[k], w[q] * w[j] * w[k], g00, g01, g02, g11, g12, g22);
        s += dx * dx * g00;
        metric_at(cf, n_coef, x[i], x[q], x[k], w[i] * w[q] * w[k], g00, g01, g02, g11, g12, g22);
        s += dy * dy * g11;
        metric_at(cf, n_coef, x[i], x[j], x[q], w[i] * w[j] * w[q], g00, g01, g02, g11, g12, g22);
        s += dz * dz * g22;
      }
    metric_at(cf, n_coef, x[i], x[j], x[k], w[i] * w[j] * w[k], g00, g01, g02, g11, g12, g22);
    const double di = Dg[i * N + i], dj = Dg[j * N + j], dk = Dg[k * N + k];
    s += 2. * (di * dj * g01 + di * dk * g02 + dj * dk * g12);
    atomicAdd(diag + ((size_t)base / 3 + pos) * stride, s);
  }

  __global__ void __launch_bounds__(256) invert_diag_kernel(const uint64_t n, double *d)
  {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n)
      d[i] = d[i] == 0. ? 1. : 1. / d[i];
  }

  // ---------------------------------------------------------------------------------------

  // ---------------------------------------------------------------------------------------
  // launchers
  // ---------------------------------------------------------------------------------------
  static inline int stream_grid(uint64_t n, int sms)
  {
    const uint64_t blocks = (n + 255) / 256;
    return (int)std::min<uint64_t>(std::max<uint64_t>(blocks, 1), (uint64_t)sms * 8);
  }

  // dynamic shared memory of the fused instantiation: the staging rows follow the cell rows
  template <int P>
  constexpr size_t fused_smem()
  {
    return sizeof(CellSmem<P, Cfg<P>::CPB, 24>) + sizeof(JobSmem<(Stage<P>::OK ? Stage<P>::JOB : 2)>);
  }

  template <int P>
  static cudaError_t init_degree(std::vector<uint32_t> &walk)
  {
    Tab<P> tb;
    fill_tab<P>(tb);
    walk.resize(Geom<P>::DOF);
    build_dof_table<P>(walk.data());
    cudaError_t e = cudaMemcpyToSymbol(c_tab<P>, &tb, sizeof(tb));
    if (e != cudaSuccess)
      return e;
    constexpr int CPB = Cfg<P>::CPB, CPBQ = Cfg<P, true>::CPB;
    e = cudaFuncSetAttribute(cell_kernel<P, CPB, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)sizeof(CellSmem<P, CPB, 24>));
    if (e != cudaSuccess)
      return e;
    e = cudaFuncSetAttribute(cell_kernel<P, CPBQ, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)sizeof(CellSmem<P, CPBQ, 81>));
    if (e != cudaSuccess)
      return e;
    if constexpr (Stage<P>::OK)
      {
        e = cudaFuncSetAttribute(cell_kernel<P, CPB, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)fused_smem<P>());
        if (e != cudaSuccess)
          return e;
        e = cudaFuncSetAttribute(cell_kernel<P, CPB, true, false, true>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fused_smem<P>());
      }
    return e;
  }

  template <int P>
  static cudaError_t run_cell(const bool fused, const bool quad, const CellArgs &a, int sms, cudaStream_t st)
  {
    constexpr int  CPB = Cfg<P>::CPB, CPBQ = Cfg<P, true>::CPB;
    if (fused && (quad || !Stage<P>::OK))
      return cudaErrorInvalidValue;
    const uint64_t units = fused ? a.n_units : (a.n_cells + (quad ? CPBQ : CPB) - 1) / (quad ? CPBQ : CPB);
    const int      grid  = (int)std::min<uint64_t>(units, (uint64_t)sms * Cfg<P>::BLOCKS);
    if (grid == 0)
      return cudaSuccess;
#ifdef BP4_PHASE_TIMING
    unsigned long long *d_trace = nullptr;
    const size_t        n_trace = (size_t)grid * kTraceBatches * 20;
    if (getenv("BP4_TRACE"))
      {
        cudaMalloc(&d_trace, n_trace * 8);
        cudaMemsetAsync(d_trace, 0, n_trace * 8, st);
      }
    cudaMemcpyToSymbolAsync(g_trace, &d_trace, sizeof(d_trace), 0, cudaMemcpyHostToDevice, st);
#endif
    if (fused)
      {
        if constexpr (Stage<P>::OK)
          {
            if (a.state)
              cell_kernel<P, CPB, true, false, true><<<grid, kThreads, fused_smem<P>(), st>>>(a);
            else
              cell_kernel<P, CPB, true, false><<<grid, kThreads, fused_smem<P>(), st>>>(a);
          }
      }
    else if (quad)
      cell_kernel<P, CPBQ, false, true><<<grid, kThreads, sizeof(CellSmem<P, CPBQ, 81>), st>>>(a);
    else
      cell_kernel<P, CPB, false, false><<<grid, kThreads, sizeof(CellSmem<P, CPB, 24>), st>>>(a);
#ifdef BP4_PHASE_TIMING
    if (d_trace)
      {
        cudaStreamSynchronize(st);
        std::vector<unsigned long long> h(n_trace);
        cudaMemcpy(h.data(), d_trace, n_trace * 8, cudaMemcpyDeviceToHost);
        cudaFree(d_trace);
        if (FILE *f = fopen(getenv("BP4_TRACE"), "ab"))
          {
            const unsigned long long hdr[4] = {0xB4B4B4B4ull, (unsigned long long)grid, kTraceBatches, fused ? 1ull : 0ull};
            fwrite(hdr, 8, 4, f);
            fwrite(h.data(), 8, n_trace, f);
            fclose(f);
          }
      }
    if (getenv("BP4_PHASE_TIMING"))
      {
        cudaStreamSynchronize(st);
        unsigned long long h[8], z[8] = {0};
        cudaMemcpyFromSymbol(h, g_phase_clk, sizeof(h));
        cudaMemcpyToSymbol(g_phase_clk, z, sizeof(z));
        double tot = 0;
        for (int k = 0; k < 8; ++k)
          tot += double(h[k]);
        fprintf(stderr, "phase clk share: meta %.1f%% gather %.1f%% barrier %.1f%% P1 %.1f%% P2 %.1f%% P3 %.1f%% scatter %.1f%% post %.1f%% | per-warp total %.0f clk\n",
                100 * h[0] / tot, 100 * h[1] / tot, 100 * h[2] / tot, 100 * h[3] / tot, 100 * h[4] / tot,
                100 * h[5] / tot, 100 * h[6] / tot, 100 * h[7] / tot, tot / (grid * (kThreads / 32)));
      }
#endif
    return cudaGetLastError();
  }

#define BP4_DISPATCH(degree, CALL)         \
  switch (degree)                          \
    {                                      \
      case 2: return CALL(2);              \
      case 3: return CALL(3);              \
      case 4: return CALL(4);              \
      case 5: return CALL(5);              \
      case 6: return CALL(6);              \
      case 7: return CALL(7);              \
      case 8: return CALL(8);              \
      default: return cudaErrorInvalidValue; \
    }

  cudaError_t launch_init_degree(int degree, std::vector<uint32_t> &walk)
  {
#define CALL(P) init_degree<P>(walk)
    BP4_DISPATCH(degree, CALL)
#undef CALL
  }

  cudaError_t launch_cell(int degree, bool fused, bool quad, const CellArgs &a, int sms, cudaStream_t st)
  {
#define CALL(P) run_cell<P>(fused, quad, a, sms, st)
    BP4_DISPATCH(degree, CALL)
#undef CALL
  }

  template <int P>
  static cudaError_t fused_loop_cfg(FusedLoopCfg &out)
  {
    out = {(uint32_t)Cfg<P>::CPB, Stage<P>::OK ? (uint32_t)Stage<P>::LIMIT : 0u, Cfg<P>::FUSED_DEFAULT};
    return cudaSuccess;
  }

  cudaError_t fused_loop_config(int degree, FusedLoopCfg &out)
  {
#define CALL(P) fused_loop_cfg<P>(out)
    BP4_DISPATCH(degree, CALL)
#undef CALL
  }

  cudaError_t launch_pre(uint64_t begin, uint64_t end, double *h, double *x, double *r, double *p,
                         const double *prec, double alpha, double beta, double alpha_old,
                         double beta_old, double *acc_to_zero, int sms, cudaStream_t st)
  {
    pre_kernel<false><<<stream_grid(end > begin ? end - begin : 0, sms), 256, 0, st>>>(
      begin, end, h, x, r, p, prec, alpha, beta, alpha_old, beta_old, acc_to_zero, nullptr);
    return cudaGetLastError();
  }

  cudaError_t launch_pre_dev(uint64_t begin, uint64_t end, double *h, double *x, double *r, double *p,
                             const double *prec, const SolveState *state, double *acc_to_zero, int sms,
                             cudaStream_t st)
  {
    pre_kernel<true><<<stream_grid(end > begin ? end - begin : 0, sms), 256, 0, st>>>(
      begin, end, h, x, r, p, prec, 0., 0., 0., 0., acc_to_zero, state);
    return cudaGetLastError();
  }

  cudaError_t launch_post(uint64_t begin, uint64_t end, const double *r, const double *d,
                          const double *h, const double *prec, double *acc, const DetSlots &det, int sms,
                          cudaStream_t st)
  {
    if (end <= begin)
      return cudaSuccess;
    if (det.slot)
      post_kernel<true><<<stream_grid(end - begin, sms), 256, 0, st>>>(begin, end, r, d, h, prec, acc, det);
    else
      post_kernel<false><<<stream_grid(end - begin, sms), 256, 0, st>>>(begin, end, r, d, h, prec, acc, det);
    return cudaGetLastError();
  }

  cudaError_t launch_fixup(uint64_t n, const uint32_t *con, double *dst, const double *src,
                           cudaStream_t st)
  {
    if (n == 0)
      return cudaSuccess;
    fixup_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, con, dst, src);
    return cudaGetLastError();
  }

  cudaError_t launch_sadd(uint64_t n, double *dst, double s, double a, const double *src, int sms,
                          cudaStream_t st)
  {
    if (n == 0)
      return cudaSuccess;
    sadd_kernel<false><<<stream_grid(n, sms), 256, 0, st>>>(n, dst, s, a, src, nullptr);
    return cudaGetLastError();
  }

  cudaError_t launch_sadd_dev(uint64_t n, double *dst, const double *s, double a, const double *src, int sms,
                              cudaStream_t st)
  {
    if (n == 0)
      return cudaSuccess;
    sadd_kernel<true><<<stream_grid(n, sms), 256, 0, st>>>(n, dst, 0., a, src, s);
    return cudaGetLastError();
  }

  cudaError_t launch_jacobi_dot(uint64_t n, double *h, const double *g, const double *diag, double *acc,
                                const DetSlots &det, int sms, cudaStream_t st)
  {
    if (n == 0)
      return cudaSuccess;
    if (det.slot)
      jacobi_dot_kernel<true><<<stream_grid(n, sms), 256, 0, st>>>(n, h, g, diag, acc, det);
    else
      jacobi_dot_kernel<false><<<stream_grid(n, sms), 256, 0, st>>>(n, h, g, diag, acc, det);
    return cudaGetLastError();
  }

  cudaError_t launch_cg_xg(uint64_t n, double *x, double *g, const double *d, const double *h,
                           const SolveState *state, double *acc, const DetSlots &det, int sms, cudaStream_t st)
  {
    if (n == 0)
      return cudaSuccess;
    if (det.slot)
      cg_xg_kernel<true><<<stream_grid(n, sms), 256, 0, st>>>(n, x, g, d, h, state, acc, det);
    else
      cg_xg_kernel<false><<<stream_grid(n, sms), 256, 0, st>>>(n, x, g, d, h, state, acc, det);
    return cudaGetLastError();
  }

  cudaError_t launch_solve_scalar(int kind, SolveState *state, double *acc, cudaGraphConditionalHandle loop,
                                  cudaStream_t st)
  {
    solve_scalar_kernel<<<1, 32, 0, st>>>(kind, state, acc, loop);
    return cudaGetLastError();
  }

  cudaError_t launch_solve_final(uint64_t n, double *x, const double *d, const double *g, const double *prec,
                                 const SolveState *state, bool det, int sms, cudaStream_t st)
  {
    if (n == 0)
      return cudaSuccess;
    if (det)
      solve_final_kernel<true><<<stream_grid(n, sms), 256, 0, st>>>(n, x, d, g, prec, state);
    else
      solve_final_kernel<false><<<stream_grid(n, sms), 256, 0, st>>>(n, x, d, g, prec, state);
    return cudaGetLastError();
  }

  cudaError_t launch_dot(uint64_t n, const double *a, const double *b, double *acc, const DetSlots &det,
                         int sms, cudaStream_t st)
  {
    if (n == 0)
      return cudaSuccess;
    if (det.slot)
      dot_kernel<true><<<stream_grid(n, sms), 256, 0, st>>>(n, a, b, acc, det);
    else
      dot_kernel<false><<<stream_grid(n, sms), 256, 0, st>>>(n, a, b, acc, det);
    return cudaGetLastError();
  }

  cudaError_t launch_add_and_dot(uint64_t n, double *g, double a, const double *h, const double *w,
                                 double *acc, const DetSlots &det, int sms, cudaStream_t st)
  {
    if (n == 0)
      return cudaSuccess;
    if (det.slot)
      add_and_dot_kernel<true><<<stream_grid(n, sms), 256, 0, st>>>(n, g, a, h, w, acc, det);
    else
      add_and_dot_kernel<false><<<stream_grid(n, sms), 256, 0, st>>>(n, g, a, h, w, acc, det);
    return cudaGetLastError();
  }

  cudaError_t launch_nonzero(uint64_t n, const double *v, int *flag, int sms, cudaStream_t st)
  {
    if (n == 0)
      return cudaSuccess;
    nonzero_kernel<<<stream_grid(n, sms), 256, 0, st>>>(n, v, flag);
    return cudaGetLastError();
  }

  cudaError_t launch_jacobi(uint64_t n, double *dst, const double *src, const double *diag, int sms,
                            cudaStream_t st)
  {
    if (n == 0)
      return cudaSuccess;
    jacobi_kernel<<<stream_grid(n, sms), 256, 0, st>>>(n, dst, src, diag);
    return cudaGetLastError();
  }

  cudaError_t launch_xfinal(uint64_t n, double *x, const double *d, const double *g, const double *prec,
                            double c1, double c2, int sms, cudaStream_t st)
  {
    if (n == 0)
      return cudaSuccess;
    xfinal_kernel<<<stream_grid(n, sms), 256, 0, st>>>(n, x, d, g, prec, c1, c2);
    return cudaGetLastError();
  }

  // assemble the scalar GLL diagonal: entry of node i goes to diag[i * stride]
  cudaError_t launch_diag_assemble(int degree, uint64_t n_cells, const uint32_t *entity_index,
                                   const double *coef, int n_coef, const double *gll, double *diag,
                                   int stride, cudaStream_t st)
  {
    const int      N3 = (degree + 1) * (degree + 1) * (degree + 1);
    const uint64_t n  = n_cells * N3;
    if (n > 0)
      diag_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(degree, n_cells, entity_index, coef, n_coef,
                                                                gll, diag, stride);
    return cudaGetLastError();
  }

  cudaError_t launch_diag_invert(uint64_t n_nodes, double *diag, cudaStream_t st)
  {
    if (n_nodes > 0)
      invert_diag_kernel<<<(unsigned)((n_nodes + 255) / 256), 256, 0, st>>>(n_nodes, diag);
    return cudaGetLastError();
  }

  cudaError_t launch_publish(double *acc, int k, double *host_vals, unsigned long long *host_seq,
                             unsigned long long seq, cudaStream_t st)
  {
    publish_kernel<<<1, 32, 0, st>>>(acc, k, host_vals, host_seq, seq);
    return cudaGetLastError();
  }

  cudaError_t launch_pack(uint64_t n, const uint32_t *idx, const double *v, double *buf, cudaStream_t st)
  {
    if (n > 0)
      pack_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, idx, v, buf);
    return cudaGetLastError();
  }

  cudaError_t launch_unpack_add(uint64_t n, const uint32_t *idx, const double *buf, double *v, cudaStream_t st)
  {
    if (n > 0)
      unpack_add_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, idx, buf, v);
    return cudaGetLastError();
  }

  cudaError_t launch_stride3(uint64_t n, const double *in, double *out, cudaStream_t st)
  {
    if (n > 0)
      stride3_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, in, out);
    return cudaGetLastError();
  }

  // host table for the diagonal kernel: x[N], w[N], Dg[N][N]
  void gll_table(int degree, std::vector<double> &out)
  {
    const int           N = degree + 1;
    std::vector<double> x, w;
    gauss_lobatto_01(N, x, w);
    out.assign(2 * N + N * N, 0.);
    for (int i = 0; i < N; ++i)
      {
        out[i]     = x[i];
        out[N + i] = w[i];
        for (int q = 0; q < N; ++q)
          out[2 * N + i * N + q] = lagrange_deriv(x, i, x[q]);
      }
  }
} // namespace bp4
