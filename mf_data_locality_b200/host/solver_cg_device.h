// solver_cg_device.h -- SolverCG and SolverCGFullMerge with the whole iteration loop on the
// device (bp4_solve_cg_async / bp4_solve_cg_merged_async): same constructor and solve() as the host-driven
// classes, same algorithm and stopping test, but no host round trip per iteration.  One rank only.
#pragma once
#include <cstring>
#include <vector>

#include "device_vector.h"
#include "solver_control.h"

namespace dealii
{
  template <typename VectorType, bool merged>
  class SolverCGOnDevice : public SolverBase<VectorType>
  {
  public:
    explicit SolverCGOnDevice(SolverControl &cn) : SolverBase<VectorType>(cn) {}

    template <typename MatrixType, typename PreconditionerType>
    void solve(const MatrixType &, VectorType &x, const VectorType &b, const PreconditionerType &preconditioner)
    {
      SolverControl &control = this->control;
      // a plain SolverControl is a ReductionControl that never reduces
      const auto      *rc     = dynamic_cast<const ReductionControl *>(&control);
      const double     reduce = rc ? rc->reduction() : 0.;
      // queued on the context's stream with the residual of every checked step; the result and
      // the history share one vector [bp4_solve_result (3 doubles) | history (max_steps + 1)],
      // read back with one download
      static_assert(sizeof(bp4_solve_result) == 3 * sizeof(double), "result = three doubles");
      bp4_ctx       *ctx = x.context();
      const unsigned max_steps = control.max_steps();
      std::vector<double> out(3 + max_steps + 1);
      bp4_vec       *buf = nullptr;
      double        *dev = nullptr;
      bp4_check(bp4_vec_alloc_uninitialized(ctx, out.size(), &buf));
      int err = bp4_vec_device_ptr(ctx, buf, &dev);
      if (!err)
        err = (merged ? bp4_solve_cg_merged_async : bp4_solve_cg_async)(
          ctx, x.handle(), b.handle(), preconditioner.get_vector().handle(), max_steps, control.tolerance(), reduce,
          reinterpret_cast<bp4_solve_result *>(dev), dev + 3);
      if (!err)
        err = bp4_vec_download(ctx, buf, out.data(), out.size());
      bp4_vec_free(ctx, buf);
      bp4_check(err);
      bp4_solve_result r;
      std::memcpy(&r, out.data(), sizeof(r));
      // replay every check, so that last_step(), last_value(), last_check() and the history data
      // read as the host-driven solver leaves them
      SolverControl::State conv = SolverControl::iterate;
      for (unsigned int k = 0; k <= r.last_step; ++k)
        conv = control.check(k, out[3 + k]);
      if (conv != SolverControl::success)
        throw SolverControl::NoConvergence(r.last_step, r.last_value);
    }
  };

  // Mixed-precision CG on the device (bp4_solve_cg_mixed_async): FP64 refinement steps around an
  // inner FP32 merged CG.  The control's tolerance, reduction and max_steps mean what
  // bp4_solve_cg_mixed makes of them: the FP64 true residual is checked once per refinement step,
  // and max_steps caps the inner FP32 iterations.  The replayed checks are those of the refinement
  // steps, so last_step() is the last refinement step.  One rank only.
  template <typename VectorType>
  class SolverCGMixedDevice : public SolverBase<VectorType>
  {
  public:
    explicit SolverCGMixedDevice(SolverControl &cn) : SolverBase<VectorType>(cn) {}

    template <typename MatrixType, typename PreconditionerType>
    void solve(const MatrixType &, VectorType &x, const VectorType &b, const PreconditionerType &preconditioner)
    {
      SolverControl &control = this->control;
      const auto    *rc      = dynamic_cast<const ReductionControl *>(&control);
      const double   reduce  = rc ? rc->reduction() : 0.;
      // [bp4_mixed_result (4 doubles) | history (max_steps + 1)], read back with one download
      static_assert(sizeof(bp4_mixed_result) == 4 * sizeof(double), "result = four doubles");
      bp4_ctx       *ctx       = x.context();
      const unsigned max_steps = control.max_steps();
      std::vector<double> out(4 + max_steps + 1);
      bp4_vec       *buf = nullptr;
      double        *dev = nullptr;
      bp4_check(bp4_vec_alloc_uninitialized(ctx, out.size(), &buf));
      int err = bp4_vec_device_ptr(ctx, buf, &dev);
      if (!err)
        err = bp4_solve_cg_mixed_async(ctx, x.handle(), b.handle(), preconditioner.get_vector().handle(), max_steps,
                                       control.tolerance(), reduce, reinterpret_cast<bp4_mixed_result *>(dev), dev + 4);
      if (!err)
        err = bp4_vec_download(ctx, buf, out.data(), out.size());
      bp4_vec_free(ctx, buf);
      bp4_check(err);
      bp4_mixed_result r;
      std::memcpy(&r, out.data(), sizeof(r));
      SolverControl::State conv = SolverControl::iterate;
      for (unsigned int k = 0; k <= r.refinements; ++k)
        conv = control.check(k, out[4 + k]);
      if (conv != SolverControl::success)
        throw SolverControl::NoConvergence(r.refinements, r.last_value);
    }
  };
} // namespace dealii

template <typename VectorType>
using SolverCGDevice = dealii::SolverCGOnDevice<VectorType, false>;
template <typename VectorType>
using SolverCGFullMergeDevice = dealii::SolverCGOnDevice<VectorType, true>;
