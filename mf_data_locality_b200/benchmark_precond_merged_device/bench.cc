// benchmark_precond_merged_device: BP4 with the fully merged CG (SolverCGFullMerge), the whole
// iteration loop on the device (SolverCGFullMergeDevice, one rank).  The `run_cg_solver` plugin of
// host/benchmark.h; CLI and table row as benchmark_precond_merged.
#include "../host/benchmark.h"
#include "../host/solver_cg_device.h"

using DeviceVector = LinearAlgebra::distributed::Vector<double>;

template <typename Operator, typename Preconditioner>
unsigned int run_cg_solver(const Operator &A, DeviceVector &x, const DeviceVector &b, const Preconditioner &P)
{
  return solve_and_count<SolverCGFullMergeDevice<DeviceVector>>(A, x, b, P); // ReductionControl(100, 1e-15, 1e-8)
}

#ifndef BP4_NO_MAIN
int main(int argc, char **argv)
{
  run(argc, argv); // bench <degree> [s] [compact_output]
}
#endif
