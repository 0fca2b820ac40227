// bp4_launch.h -- launcher prototypes shared by bp4_kernels.cu and bp4_capi.cu
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

#include "bp4_kernels.cuh"

namespace bp4
{
  cudaError_t launch_init_degree(int degree, std::vector<uint32_t> &walk);
  // what the host needs to plan the fused cell loop of a degree (from Cfg<P> and Stage<P>)
  struct FusedLoopCfg
  {
    uint32_t cpb;        // cells per batch of the tri-linear kernel
    uint32_t run_limit;  // longest private run (DoFs) one batch may carry; 0 = no fused kernel
    bool     is_default; // Cfg<P>::FUSED_DEFAULT
  };
  cudaError_t fused_loop_config(int degree, FusedLoopCfg &out);
  // plain: a.n_cells cells from a.entity_index on; fused: a.n_units units of a.unit_batch;
  // quad: a.coef holds all 27 coefficients per cell (plain kernel only)
  cudaError_t launch_cell(int degree, bool fused, bool quad, const CellArgs &a, int sms, cudaStream_t st);
  // do_cg_update4b / do_cg_update3b on the DoF interval [begin, end) (the DoFs no range owns)
  cudaError_t launch_pre(uint64_t begin, uint64_t end, double *h, double *x, double *r, double *p,
                         const double *prec, double alpha, double beta, double alpha_old,
                         double beta_old, double *acc_to_zero, int sms, cudaStream_t st);
  // the same with alpha, beta, alpha_old, beta_old read from a device-resident solve's state
  cudaError_t launch_pre_dev(uint64_t begin, uint64_t end, double *h, double *x, double *r, double *p,
                             const double *prec, const SolveState *state, double *acc_to_zero, int sms,
                             cudaStream_t st);
  // the reductions below: det.slot set = ordered cross-block sums (deterministic mode), else atomics
  cudaError_t launch_post(uint64_t begin, uint64_t end, const double *r, const double *d,
                          const double *h, const double *prec, double *acc, const DetSlots &det, int sms,
                          cudaStream_t st);
  cudaError_t launch_fixup(uint64_t n, const uint32_t *con, double *dst, const double *src,
                           cudaStream_t st);
  cudaError_t launch_sadd(uint64_t n, double *dst, double s, double a, const double *src, int sms,
                          cudaStream_t st);
  cudaError_t launch_sadd_dev(uint64_t n, double *dst, const double *s, double a, const double *src, int sms,
                              cudaStream_t st); // s read on the device
  cudaError_t launch_dot(uint64_t n, const double *a, const double *b, double *acc, const DetSlots &det,
                         int sms, cudaStream_t st);
  cudaError_t launch_add_and_dot(uint64_t n, double *g, double a, const double *h, const double *w,
                                 double *acc, const DetSlots &det, int sms, cudaStream_t st);
  cudaError_t launch_nonzero(uint64_t n, const double *v, int *flag, int sms, cudaStream_t st);
  cudaError_t launch_jacobi(uint64_t n, double *dst, const double *src, const double *diag, int sms,
                            cudaStream_t st);
  cudaError_t launch_xfinal(uint64_t n, double *x, const double *d, const double *g, const double *prec,
                            double c1, double c2, int sms, cudaStream_t st);
  // device-resident solves (bp4_solve_cg / bp4_solve_cg_merged)
  enum SolveScalarKind
  {
    kSolveMergedStep = 0,
    kSolvePlainInit  = 1,
    kSolvePlainAlpha = 2,
    kSolvePlainCheck = 3
  };
  cudaError_t launch_jacobi_dot(uint64_t n, double *h, const double *g, const double *diag, double *acc,
                                const DetSlots &det, int sms, cudaStream_t st);
  cudaError_t launch_cg_xg(uint64_t n, double *x, double *g, const double *d, const double *h,
                           const SolveState *state, double *acc, const DetSlots &det, int sms, cudaStream_t st);
  cudaError_t launch_solve_scalar(int kind, SolveState *state, double *acc, cudaGraphConditionalHandle loop,
                                  cudaStream_t st);
  // det: the odd-step update rounded as bp4_add rounds it (deterministic mode)
  cudaError_t launch_solve_final(uint64_t n, double *x, const double *d, const double *g, const double *prec,
                                 const SolveState *state, bool det, int sms, cudaStream_t st);
  cudaError_t launch_diag_assemble(int degree, uint64_t n_cells, const uint32_t *entity_index,
                                   const double *coef, int n_coef, const double *gll, double *diag,
                                   int stride, cudaStream_t st);
  cudaError_t launch_diag_invert(uint64_t n_nodes, double *diag, cudaStream_t st);
  cudaError_t launch_publish(double *acc, int k, double *host_vals, unsigned long long *host_seq,
                             unsigned long long seq, cudaStream_t st);
  cudaError_t launch_pack(uint64_t n, const uint32_t *idx, const double *v, double *buf, cudaStream_t st);
  cudaError_t launch_unpack_add(uint64_t n, const uint32_t *idx, const double *buf, double *v, cudaStream_t st);
  cudaError_t launch_stride3(uint64_t n, const double *in, double *out, cudaStream_t st);
  void        gll_table(int degree, std::vector<double> &out);
} // namespace bp4
