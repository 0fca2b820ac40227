// bp4_kernels.cu -- the cell kernel and its launchers (sm_100a, FP64).  See bp4_kernels.cuh; the
// vector kernels are in bp4_vector_kernels.cuh.
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
  // instantiated here, ahead of the float tables, so that the FP64 tables keep their constant-bank
  // offsets (and the FP64 kernels their code) whatever the FP32 kernel adds
  template __constant__ Tab<2> c_tab<2>;
  template __constant__ Tab<3> c_tab<3>;
  template __constant__ Tab<4> c_tab<4>;
  template __constant__ Tab<5> c_tab<5>;
  template __constant__ Tab<6> c_tab<6>;
  template __constant__ Tab<7> c_tab<7>;
  template __constant__ Tab<8> c_tab<8>;
  // the same tables rounded to float, for the FP32 kernel (a second constant bank)
  template <int P>
  __constant__ Tab<P, float> c_tab32;

  template <int P, typename T>
  __device__ __forceinline__ const Tab<P, T> &ctab()
  {
    if constexpr (sizeof(T) == 4)
      return c_tab32<P>;
    else
      return c_tab<P>;
  }

  template <int P, int CPB, int NC, typename T>
  __device__ __forceinline__ void load_tables(CellSmem<P, CPB, NC, T> &sm, const uint32_t *dtab)
  {
    for (int i = threadIdx.x; i < Geom<P>::DOF; i += blockDim.x)
      sm.dtab[i] = dtab[i];
    if (threadIdx.x < Geom<P>::Q)
      {
        sm.xq[threadIdx.x] = ctab<P, T>().xq[threadIdx.x];
        sm.wq[threadIdx.x] = ctab<P, T>().wq[threadIdx.x];
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
  template <int P, bool QUAD, typename T>
  __device__ __noinline__ void phase2_call(const uint32_t cf_off, const uint32_t work_off, const int qx,
                                           const int qz, const T x, const T z, const T wxz)
  {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    phase2<P, QUAD>(ctab<P, T>(), reinterpret_cast<const T *>(smem_raw + cf_off),
              reinterpret_cast<T *>(smem_raw + work_off), qx, qz, x, z, wxz);
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
  // pre_kernel / post_kernel stream them before / after this kernel.  The scalars of
  // do_cg_update4b are the ones pre_kernel derived and left in *a.scalars, from the caller's
  // arguments or from the solver state of a device-resident solve.
  //
  // T = float: the FP32 plain kernel of the mixed-precision solve -- the same code with float work
  // rows, coefficients, tables and phase-2 arithmetic, and float REDs in the scatter.
  // ---------------------------------------------------------------------------------------
  template <int P, int CPB, bool FUSED, bool QUAD, typename T = double>
  __global__ void __launch_bounds__(kThreads, Cfg<P, QUAD, T>::BLOCKS) cell_kernel(const CellArgsT<T> a)
  {
    constexpr int NC = Cfg<P, QUAD>::NCOEF;
    using G         = Geom<P>;
    constexpr int Q = G::Q;
    constexpr bool kFine = Cfg<P>::FINE;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CellSmem<P, CPB, NC, T> &sm  = *reinterpret_cast<CellSmem<P, CPB, NC, T> *>(smem_raw);
    const int                tid = threadIdx.x;
    const Tab<P, T>         &tb  = ctab<P, T>();
    load_tables<P, CPB, NC, T>(sm, a.dtab);
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
    const bool     dynamic = Cfg<P, QUAD, T>::DYNAMIC && a.sched != nullptr;
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
    T             mc[MC];
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
          mc[u]       = k < nc * NC ? __ldg(a.coef + (uint64_t)cell0 * NC + k) : T(0);
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
    constexpr bool kPipe = Cfg<P, QUAD, T>::PIPE_GATHER;
    constexpr int R = (G::DOF + kThreads - 1) / kThreads, S = CPB * R;
    // only the last r can run past the end of the cell
    const bool last_on = tid < G::DOF - (R - 1) * kThreads;
    auto       on      = [&](const int r) { return r < R - 1 || last_on; };
    T          gv[S];
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
        gv[s1] = idx[s1] != 0xFFFFFFFFu ? (FUSED ? a.src[idx[s1]] : __ldg(a.src + idx[s1])) : T(0);
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
          T        v[SU];
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
            phase2_call<P, QUAD, T>((uint32_t)((const unsigned char *)sm.coef[bf][cell] - smem_raw),
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
        auto pre_one = [&](const Update4b &sc, const uint32_t i, const double rr, const double pp, const double hh,
                           const double pr) {
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
          // the scalars as pre_kernel derived them, read per job: held over the compute phases they
          // would take registers that phase 2 needs (Q4 spilled 80/40 instead of 52/32 bytes)
          const Update4b sc = *a.scalars;
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
            pre_one(sc, i, js.row[0][i - lo], js.row[1][i - lo], js.row[2][i - lo], js.prec[div3(i) - q0]);
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

  // ---------------------------------------------------------------------------------------
  // launchers
  // ---------------------------------------------------------------------------------------
  // One instance of the cell kernel and its dynamic shared memory.  A degree has five: plain
  // tri-linear, plain quadratic, fused tri-linear if Stage<P>::OK (its staging rows follow the
  // cell rows), and the FP32 plain tri-linear and quadratic ones.
  template <int P, bool FUSED, bool QUAD, typename T = double>
  struct CellInstance
  {
    static constexpr int CPB  = Cfg<P, QUAD, T>::CPB;
    static constexpr int SMEM = (int)(sizeof(CellSmem<P, CPB, Cfg<P, QUAD>::NCOEF, T>) +
                                      (FUSED ? sizeof(JobSmem<Stage<P>::JOB>) : 0));
    static cudaError_t init()
    {
      return cudaFuncSetAttribute(cell_kernel<P, CPB, FUSED, QUAD, T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  SMEM);
    }
    static void launch(const int grid, const CellArgsT<T> &a, cudaStream_t st)
    {
      cell_kernel<P, CPB, FUSED, QUAD, T><<<grid, kThreads, SMEM, st>>>(a);
    }
  };

  template <int P>
  static cudaError_t init_degree(std::vector<uint32_t> &walk)
  {
    Tab<P> tb;
    fill_tab<P>(tb);
    walk.resize(Geom<P>::DOF);
    build_dof_table<P>(walk.data());
    // the FP32 tables: every entry of the FP64 ones rounded to float
    Tab<P, float> tb32;
    const double *from = &tb.S[0][0];
    float        *to   = &tb32.S[0][0];
    static_assert(sizeof(tb) == 2 * sizeof(tb32), "Tab<P> is an array of doubles");
    for (size_t i = 0; i < sizeof(tb32) / sizeof(float); ++i)
      to[i] = (float)from[i];
    cudaError_t e = cudaMemcpyToSymbol(c_tab<P>, &tb, sizeof(tb));
    if (e == cudaSuccess)
      e = cudaMemcpyToSymbol(c_tab32<P>, &tb32, sizeof(tb32));
    if (e == cudaSuccess)
      e = CellInstance<P, false, false>::init();
    if (e == cudaSuccess)
      e = CellInstance<P, false, true>::init();
    if (e == cudaSuccess)
      e = CellInstance<P, false, false, float>::init();
    if (e == cudaSuccess)
      e = CellInstance<P, false, true, float>::init();
    if constexpr (Stage<P>::OK)
      if (e == cudaSuccess)
        e = CellInstance<P, true, false>::init();
    return e;
  }

  template <int P, typename T>
  static cudaError_t run_cell(const bool fused, const bool quad, const CellArgsT<T> &a, int sms, cudaStream_t st)
  {
    constexpr bool F64 = sizeof(T) == 8;
    constexpr int  CPB = Cfg<P, false, T>::CPB, CPBQ = Cfg<P, true, T>::CPB;
    if (fused && (quad || !Stage<P>::OK || !F64))
      return cudaErrorInvalidValue;
    const uint64_t units = fused ? a.n_units : (a.n_cells + (quad ? CPBQ : CPB) - 1) / (quad ? CPBQ : CPB);
    const int      grid  = (int)std::min<uint64_t>(units, (uint64_t)sms * Cfg<P, false, T>::BLOCKS);
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
        if constexpr (Stage<P>::OK && F64)
          CellInstance<P, true, false>::launch(grid, a, st);
      }
    else if (quad)
      CellInstance<P, false, true, T>::launch(grid, a, st);
    else
      CellInstance<P, false, false, T>::launch(grid, a, st);
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

  cudaError_t launch_cell_f32(int degree, bool quad, const CellArgsT<float> &a, int sms, cudaStream_t st)
  {
#define CALL(P) run_cell<P>(false, quad, a, sms, st)
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
