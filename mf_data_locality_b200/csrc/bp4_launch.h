// bp4_launch.h -- what the cell-kernel unit (bp4_kernels.cu) exports to bp4_capi.cu
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
  // the FP32 plain kernel: a.src, a.dst and a.coef in float (the float copy of the coefficients)
  cudaError_t launch_cell_f32(int degree, bool quad, const CellArgsT<float> &a, int sms, cudaStream_t st);
  void        gll_table(int degree, std::vector<double> &out);
} // namespace bp4
