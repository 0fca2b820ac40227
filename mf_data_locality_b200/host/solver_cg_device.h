// solver_cg_device.h -- SolverCG and SolverCGFullMerge with the whole iteration loop on the
// device (bp4_solve_cg / bp4_solve_cg_merged): same constructor and solve() as the host-driven
// classes, same algorithm and stopping test, but no host round trip per iteration.  One rank only.
#pragma once
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
      bp4_solve_result r{};
      bp4_check((merged ? bp4_solve_cg_merged : bp4_solve_cg)(x.context(), x.handle(), b.handle(),
                                                               preconditioner.get_vector().handle(),
                                                               control.max_steps(), control.tolerance(),
                                                               reduce, &r));
      // replay the checks so that last_step(), last_value() and last_check() read as the
      // host-driven solver leaves them
      SolverControl::State conv = control.check(0, r.initial_value);
      if (r.last_step > 0)
        conv = control.check(r.last_step, r.last_value);
      if (conv != SolverControl::success)
        throw SolverControl::NoConvergence(r.last_step, r.last_value);
    }
  };
} // namespace dealii

template <typename VectorType>
using SolverCGDevice = dealii::SolverCGOnDevice<VectorType, false>;
template <typename VectorType>
using SolverCGFullMergeDevice = dealii::SolverCGOnDevice<VectorType, true>;
