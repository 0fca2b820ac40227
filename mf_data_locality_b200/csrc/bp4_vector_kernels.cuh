// bp4_vector_kernels.cuh -- the vector kernels of the C ABI (sm_100a, FP64): the CG sweeps, the
// device-resident solves, the ghost exchange, the diagonal and the reductions they share.
// Included by bp4_capi.cu only, which launches them: a __global__ function defined in a header
// that two translation units include would be defined twice at link time.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/bp4.h"
#include "bp4_kernels.cuh"

namespace bp4
{
  __device__ __forceinline__ double warp_sum(double v)
  {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
      v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
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
  // Also clears the reduction scratch of this iteration (stream order: before any post) and leaves
  // its scalars in *scalars for the fused cell kernel that follows.
  // DEV: the four scalars come from the solver state of a device-resident solve (st).
  // T = float: the vectors of the inner FP32 solve of bp4_solve_cg_mixed (the scalars stay double)
  template <bool DEV, typename T = double>
  __global__ void __launch_bounds__(256) pre_kernel(const uint64_t begin, const uint64_t end,
                                                    T *__restrict__ h, T *__restrict__ x,
                                                    T *__restrict__ r, T *__restrict__ p,
                                                    const T *__restrict__ prec,
                                                    const double alpha, const double beta,
                                                    const double alpha_old, const double beta_old,
                                                    double *acc_to_zero, Update4b *scalars,
                                                    const SolveState *st)
  {
    const Update4b sc = DEV ? update4b(st->alpha, st->beta, st->alpha_old, st->beta_old)
                            : update4b(alpha, beta, alpha_old, beta_old);
    if (acc_to_zero && blockIdx.x == 0 && threadIdx.x < 8)
      acc_to_zero[threadIdx.x] = 0.;
    if (blockIdx.x == 0 && threadIdx.x == 0)
      *scalars = sc;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    // U independent elements per trip: all their loads are in flight together.  Measured at Q4
    // s=18: U = 1 -> 0.496 ms, 2 -> 0.484, 4 -> 0.474 (6.3 TB/s), 6/8 -> 0.48
    constexpr int U = 4;
    for (uint64_t i0 = begin + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < end; i0 += U * stride)
      {
        T pr[U], ri[U], pi[U], hi[U], xi[U];
#pragma unroll
        for (int u = 0; u < U; ++u)
          {
            const uint64_t i  = i0 + u * stride;
            const bool     ok = i < end;
            pr[u] = ok ? prec[i / 3] : T(0);
            ri[u] = ok ? r[i] : T(0);
            pi[u] = ok && !sc.first ? p[i] : T(0);
            hi[u] = ok && !sc.first ? h[i] : T(0);
            xi[u] = ok && sc.update_x ? x[i] : T(0);
          }
#pragma unroll
        for (int u = 0; u < U; ++u)
          {
            const uint64_t i = i0 + u * stride;
            if (i < end)
              {
                if (sc.first)
                  p[i] = -pr[u] * ri[u];
                else
                  {
                    if (sc.update_x)
                      x[i] = xi[u] + (sc.c1 * pi[u] + sc.c2 * pr[u] * ri[u]);
                    const double rn = ri[u] + sc.alpha * hi[u];
                    r[i] = rn;
                    p[i] = sc.beta * pi[u] - pr[u] * rn;
                  }
                h[i] = T(0);
              }
          }
      }
  }

  // do_cg_update3b<3,double>, solver_cg_optimized.h:12-61, over [begin, end) -> acc[7]
  // DET: ordered cross-block sum (block_accumulate_ordered) instead of atomics.  T = float: FP32
  // vectors, the sums still accumulated in double
  template <bool DET, typename T = double>
  __global__ void __launch_bounds__(256) post_kernel(const uint64_t begin, const uint64_t end,
                                                     const T *__restrict__ r,
                                                     const T *__restrict__ d,
                                                     const T *__restrict__ h,
                                                     const T *__restrict__ prec, double *acc,
                                                     const DetSlots ds)
  {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    double         s[7]   = {0., 0., 0., 0., 0., 0., 0.};
    // U independent element groups per trip: all their loads are in flight together.  Measured at
    // Q4 s=18: U = 1 -> 0.233 ms, 4 -> 0.211 ms (6.45 TB/s), 2 and 8 slower
    constexpr int U = 4;
    for (uint64_t i0 = begin + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < end; i0 += U * stride)
      {
        T rr[U], dd[U], hh[U], pp[U];
#pragma unroll
        for (int u = 0; u < U; ++u)
          {
            const uint64_t i  = i0 + u * stride;
            const bool     ok = i < end;
            rr[u] = ok ? r[i] : T(0);
            dd[u] = ok ? d[i] : T(0);
            hh[u] = ok ? h[i] : T(0);
            pp[u] = ok ? prec[i / 3] : T(0);
          }
#pragma unroll
        for (int u = 0; u < U; ++u)
          post_terms(s, rr[u], dd[u], hh[u], pp[u]);
      }
    accumulate<DET>(s, acc, ds);
  }

  template <typename T>
  __global__ void __launch_bounds__(256) fixup_kernel(const uint64_t n, const uint32_t *__restrict__ con,
                                                      T *__restrict__ dst, const T *__restrict__ src)
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

  // Step 0 of a device-resident solve, first node of its graph.  The per-call arguments are this
  // kernel's parameters, replaced per launch in the instantiated graph (cudaGraphExecKernelNodeSetParams),
  // so that solves queued back to back share no host buffer.  Starts a fresh solver state and
  // reads the flag nonzero_kernel left: x != 0 runs the IF node `apply` (g = A x) and makes the
  // sadd_kernel<true> that follows g = 1 g - b, x == 0 skips it and makes that sadd g = -b
  // (bp4_add / bp4_equ of the host-driven solvers).
  __global__ void solve_begin_kernel(SolveState *stp, const int *nonzero, const uint32_t max_steps, const double tol,
                                     const double reduce, double *history, void *result,
                                     const cudaGraphConditionalHandle apply)
  {
    if (threadIdx.x != 0)
      return;
    SolveState st{};
    st.max_steps = max_steps;
    st.tol       = tol;
    st.reduce    = reduce;
    st.history   = history;
    st.result    = result;
    st.g_scale   = *nonzero ? 1. : 0.;
    *stp         = st;
    cudaGraphSetConditional(apply, *nonzero ? 1u : 0u);
  }

  // ReductionControl::check(0, |g|) from g.g in acc[0] (sqrt rounded as std::sqrt rounds it):
  // reduced_tol = |g| reduce; success below either tolerance, failure for max_steps = 0 or NaN.
  // `loop` (the WHILE node) and `iterated` (the IF node of the final x update) stay 0 when the
  // solve ends here, so that x is not touched.
  __global__ void solve_step0_kernel(SolveState *stp, double *acc, const cudaGraphConditionalHandle loop,
                                     const cudaGraphConditionalHandle iterated)
  {
    if (threadIdx.x != 0)
      return;
    SolveState  &st  = *stp;
    const double res = __dsqrt_rn(acc[0]);
    acc[0]           = 0.;
    st.reduced_tol   = __dmul_rn(res, st.reduce);
    st.initial_value = st.last_value = res;
    st.step                          = 0;
    if (st.history)
      st.history[0] = res;
    st.state = (res < st.reduced_tol || res <= st.tol) ? 1 : ((st.max_steps == 0 || isnan(res)) ? 2 : 0);
    cudaGraphSetConditional(loop, st.state == 0 ? 1u : 0u);
    cudaGraphSetConditional(iterated, st.state == 0 ? 1u : 0u);
  }

  // last node of a device-resident solve: the outcome to the caller's bp4_solve_result
  __global__ void solve_result_kernel(const SolveState *st)
  {
    if (threadIdx.x == 0)
      *static_cast<bp4_solve_result *>(st->result) =
        bp4_solve_result{st->state, st->step, st->last_value, st->initial_value};
  }

  // ReductionControl::check (host/solver_control.h) for a step > 0; the value also goes to the
  // caller's history
  __device__ int control_check(SolveState &st, const uint32_t step, const double value)
  {
    st.step       = step;
    st.last_value = value;
    if (st.history)
      st.history[step] = value;
    if (value < st.reduced_tol || value <= st.tol)
      return 1;
    if (step >= st.max_steps || isnan(value))
      return 2;
    return 0;
  }

  // the `kind` of solve_scalar_kernel
  constexpr int kSolveMergedStep = 0, kSolvePlainInit = 1, kSolvePlainAlpha = 2, kSolvePlainCheck = 3;

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
  // DET: the odd step rounded as bp4_add rounds it (see cg_xg_kernel).  T = float: the inner FP32
  // solve of bp4_solve_cg_mixed
  template <bool DET, typename T = double>
  __global__ void __launch_bounds__(256) solve_final_kernel(const uint64_t n, T *__restrict__ x,
                                                            const T *__restrict__ d,
                                                            const T *__restrict__ g,
                                                            const T *__restrict__ prec,
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

  // ---------------------------------------------------------------------------------------
  // mixed-precision solve (bp4_solve_cg_mixed): FP64 refinement around an inner FP32 merged CG
  // ---------------------------------------------------------------------------------------
  // The inner FP32 solve stops at this relative reduction of its residual (DESIGN.md 4.7)
  constexpr double kMixedInnerReduce = 1e-3;

  // Solver state of a mixed solve, one block per context.  `outer` is the FP64 ReductionControl on
  // the true residual |b - A x| (step = refinement step); `inner` the state of the FP32 merged CG,
  // which the scalar kernels of the device-resident merged solve drive unchanged.
  struct MixedState
  {
    SolveState outer, inner;
    double     scale;       // 1 / |b - A x| of the current refinement step
    uint32_t   inner_steps; // inner iterations of the finished refinement steps
    int32_t    checked;     // step 0 has been checked
  };

  // first node of a mixed solve: the per-call arguments (replaced per launch, as solve_begin_kernel's)
  __global__ void mixed_begin_kernel(MixedState *msp, const int *nonzero, const uint32_t max_steps, const double tol,
                                     const double reduce, double *history, void *result,
                                     const cudaGraphConditionalHandle apply)
  {
    if (threadIdx.x != 0)
      return;
    MixedState ms{};
    ms.outer.max_steps = max_steps;
    ms.outer.tol       = tol;
    ms.outer.reduce    = reduce;
    ms.outer.history   = history;
    ms.outer.result    = result;
    ms.outer.g_scale   = *nonzero ? 1. : 0.;
    *msp               = ms;
    cudaGraphSetConditional(apply, *nonzero ? 1u : 0u);
  }

  // ReductionControl::check on the FP64 true residual (|g|^2 in acc[0], g = A x - b), once per
  // refinement step, plus the two rules of the refinement: a step that does not reduce the residual
  // (stagnation) and a used-up inner step budget end the solve with state 2.  Continuing: the inner
  // solve gets a fresh state (zero start, the remaining budget, the fixed relative reduction of a
  // right-hand side of norm 1) and `go` runs the refinement body; `loop` is the outer WHILE.
  __global__ void mixed_check_kernel(MixedState *msp, double *acc, const cudaGraphConditionalHandle loop,
                                     const cudaGraphConditionalHandle go)
  {
    if (threadIdx.x != 0)
      return;
    MixedState  &ms  = *msp;
    SolveState  &st  = ms.outer;
    const double res = __dsqrt_rn(acc[0]);
    acc[0]           = 0.;
    uint32_t step    = 0;
    int      state;
    if (!ms.checked)
      {
        ms.checked       = 1;
        st.reduced_tol   = __dmul_rn(res, st.reduce);
        st.initial_value = res;
      }
    else
      {
        step = st.step + 1;
        ms.inner_steps += ms.inner.step;
      }
    const double prev = st.last_value;
    st.step           = step;
    st.last_value     = res;
    if (st.history)
      st.history[step] = res;
    if (res < st.reduced_tol || res <= st.tol)
      state = 1;
    else if (isnan(res) || ms.inner_steps >= st.max_steps || (step > 0 && !(res < prev)))
      state = 2;
    else
      state = 0;
    st.state = state;
    if (state == 0)
      {
        ms.scale   = __drcp_rn(res);
        st.g_scale = 1.; // the refinement body leaves A x in g
        SolveState in{};
        in.max_steps   = st.max_steps - ms.inner_steps;
        in.reduced_tol = kMixedInnerReduce;
        ms.inner       = in;
      }
    cudaGraphSetConditional(loop, state == 0 ? 1u : 0u);
    cudaGraphSetConditional(go, state == 0 ? 1u : 0u);
  }

  // r32 = (float)(s (A x - b)) = the inner solve's starting residual (the merged CG's g = A e - rhs at
  // e = 0 for rhs = s (b - A x)), s = 1 / |b - A x|: O(1) at every refinement step.  Sets `inner`
  // (the WHILE node that follows it in the same body) to run.
  __global__ void __launch_bounds__(256) mixed_residual_kernel(const uint64_t n, float *__restrict__ r32,
                                                               const double *__restrict__ g, const MixedState *ms,
                                                               const cudaGraphConditionalHandle inner)
  {
    const double   s      = ms->scale;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
      r32[i] = (float)(s * g[i]);
    if (blockIdx.x == 0 && threadIdx.x == 0)
      cudaGraphSetConditional(inner, 1u);
  }

  // x += (double) e32 / s: the inner correction scaled back (1 / s = the residual it was made for)
  __global__ void __launch_bounds__(256) mixed_update_kernel(const uint64_t n, double *__restrict__ x,
                                                             const float *__restrict__ e32, const MixedState *ms)
  {
    const double   res    = ms->outer.last_value;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
      x[i] += (double)e32[i] * res;
  }

  // last node of a mixed solve: the outcome to the caller's bp4_mixed_result
  __global__ void mixed_result_kernel(const MixedState *ms)
  {
    if (threadIdx.x == 0)
      *static_cast<bp4_mixed_result *>(ms->outer.result) = bp4_mixed_result{
        ms->outer.state, ms->outer.step, ms->inner_steps, ms->outer.last_value, ms->outer.initial_value};
  }

  // out = (float) in: the preconditioner of the inner solve, and the FP32 operator's input (debug hook)
  __global__ void __launch_bounds__(256) narrow_kernel(const uint64_t n, const double *__restrict__ in,
                                                       float *__restrict__ out)
  {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
      out[i] = (float)in[i];
  }

  // out = (double) in: the FP32 operator's output (debug hook)
  __global__ void __launch_bounds__(256) widen_kernel(const uint64_t n, const float *__restrict__ in,
                                                      double *__restrict__ out)
  {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
      out[i] = (double)in[i];
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
} // namespace bp4
