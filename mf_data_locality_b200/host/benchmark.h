// benchmark.h -- host-side mirror of the reference driver (benchmark.h:38-318): the BP4
// problem definition (mesh, Q_p^3 DoFs, Dirichlet set, Renumber(0,1,2), Jacobi diagonal,
// right-hand side), the `run_cg_solver` plugin seam, the timing protocol and the one-line
// table row.  deal.II objects are replaced by the stand-ins in this directory; the solver
// and operator arithmetic runs on the B200 through include/bp4.h.
//
// Differences that are deliberate:
//   * no MPI: one process per GPU; `n_ranks`/`rank` describe the partition this process
//     holds (see INTEGRATION.md for the multi-GPU launch);
//   * warmup_code() (CPU spin-up, curved_manifold.h:90-106) has no GPU counterpart;
//   * the set-up half of run_templated() is factored into BenchmarkProblem so that the
//     C entry points used by tests/bench (host_capi.cc) share it with the CLI.
#pragma once
#include <chrono>
#include <cstdlib>
#include <iomanip>
#include <iostream>
#include <memory>

#include "curved_manifold.h"
#include "device_vector.h"
#include "diagonal_matrix_blocked.h"
#include "matrix_free_standin.h"
#include "poisson_operator.h"
#include "renumber_dofs_for_mf.h"
#include "solver_cg_optimized.h"
#include "solver_control.h"

using namespace dealii;

// the benchmark is the vector-valued Laplacian in 3-D (benchmark.h:38-39)
constexpr unsigned int dimension    = 3;
constexpr unsigned int n_components = dimension;

// plugin seam: declared here, defined once per benchmark directory
// (benchmark_precond/bench.cc, benchmark_precond_merged/bench.cc), called at benchmark.h:193
template <typename Operator, typename Preconditioner>
unsigned int run_cg_solver(const Operator &laplace_operator, LinearAlgebra::distributed::Vector<double> &x,
                           const LinearAlgebra::distributed::Vector<double> &b,
                           const Preconditioner                             &preconditioner);

// stopping rule used by both plugins; the defaults are the reference's
// ReductionControl(100, 1e-15, 1e-8) (bench.cc:11); north_star also asks for 1e-10 runs
struct SolverSettings
{
  unsigned int max_steps = 100;
  double       abs_tol = 1e-15, rel_tol = 1e-8;
};
inline SolverSettings &solver_settings()
{
  static SolverSettings s;
  return s;
}

// shared body of the two plugins: build the solver on the benchmark's stopping rule, solve, and
// report the iteration count -- hitting the iteration cap is a normal outcome here, not an error
// (the reference swallows NoConvergence the same way, bench.cc:19-24)
template <typename SolverType, typename Operator, typename VectorType, typename Preconditioner>
unsigned int solve_and_count(const Operator &A, VectorType &x, const VectorType &b, const Preconditioner &P)
{
  const SolverSettings &st = solver_settings();
  ReductionControl      control(st.max_steps, st.abs_tol, st.rel_tol);
  SolverType            solver(control);
  try
    {
      solver.solve(A, x, b, P);
    }
  catch (const SolverControl::NoConvergence &)
    {}
  return control.last_step();
}

struct BenchmarkOptions
{
  unsigned int n_ranks = 1, rank = 0; // partition held by this process
  int          device  = 0;
  unsigned int n_lanes = 8, batches_per_range = 1; // deal.II batch/range model (SURVEY B1)
  unsigned int renumber_a = 0, renumber_r = 1, renumber_g = 2;
  // multi-GPU: the 128-byte ncclUniqueId all ranks share (created by rank 0 with
  // bp4_comm_unique_id and distributed by the launcher); plays the role of MPI_COMM_WORLD
  const unsigned char *nccl_id = nullptr;
  unsigned int mapping_degree = 1; // 2: genuinely quadratic cells (the TODO of benchmark.h:75-77)
  bool numbering_only = false; // stop after Renumber + MatrixFree::reinit (inspection of numberings)
  bool deterministic  = false; // bit-reproducible results on one rank (bp4_desc::deterministic)
};

class Timer
{
public:
  Timer() { restart(); }
  void   restart() { t0 = std::chrono::steady_clock::now(); }
  double wall_time() const
  {
    return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  }

private:
  std::chrono::steady_clock::time_point t0;
};

// everything run_templated() sets up before its timing loops (benchmark.h:66-176)
template <int dim, int fe_degree, int n_q_points>
struct BenchmarkProblem
{
  using VectorType = LinearAlgebra::distributed::Vector<double>;
  using OperatorType = Poisson::LaplaceOperator<dim, fe_degree, n_q_points, n_components, double, VectorType>;

  BenchmarkProblem(const unsigned int s, const BenchmarkOptions &opt)
    : tria(opt.n_ranks, opt.rank), dof_handler(tria)
  {
    Timer      lap;
    const bool show = std::getenv("BP4_SETUP_TIMING") != nullptr;
    auto       tick = [&](const char *what) {
      if (show)
        std::cerr << "  setup[" << opt.rank << "] " << what << ": " << lap.wall_time() << " s" << std::endl;
      lap.restart();
    };
    // box [0,2]^r x [0,1]^(3-r), r = s % 3, refined s / 3 times, vertices moved by the chart
    const unsigned int          n_refine = s / 3, remainder = s % 3;
    std::array<unsigned int, 3> subdivisions{{1, 1, 1}};
    for (unsigned int d = 0; d < remainder; ++d)
      subdivisions[d] = 2;
    MyManifold<dim> manifold;
    tria.build(subdivisions, n_refine, [manifold](const Point3 &p) { return manifold.push_forward(p); });

    tick("triangulation");
    dof_handler.distribute_dofs(FESystem{fe_degree, n_components});
    VectorTools::interpolate_boundary_values(dof_handler, constraints);
    constraints.close();
    tick("distribute_dofs");

    mf_data.n_lanes           = opt.n_lanes;
    mf_data.batches_per_range = opt.batches_per_range;
    mf_data.mapping_degree    = opt.mapping_degree;

    Renumber<dim, double> renum(opt.renumber_a, opt.renumber_r, opt.renumber_g);
    renum.renumber(dof_handler, constraints, mf_data);
    tick("renumber");

    // Dirichlet constraints are geometric here, so they need no rebuild after renumbering
    // (the reference re-creates them at benchmark.h:115-120)
    matrix_free = std::make_shared<MatrixFree>();

    // Jacobi preconditioner from the diagonal under GLL(p+1) quadrature (benchmark.h:124-148);
    // the device routine evaluates exactly that quadrature
    matrix_free->reinit(dof_handler, constraints, n_q_points, mf_data);
    tick("matrix_free.reinit");
    if (opt.numbering_only)
      return;
    laplace_operator.initialize(matrix_free, constraints, opt.device, opt.deterministic);
    tick("operator.initialize");
    if (opt.device < 0)
      return; // tables only
    if (opt.n_ranks > 1)
      {
        AssertThrow(opt.nccl_id != nullptr, "n_ranks > 1 needs BenchmarkOptions::nccl_id");
        bp4_check(bp4_comm_init(laplace_operator.context(), (int)opt.rank, (int)opt.n_ranks, opt.nccl_id));
      }
    {
      // benchmark.h:139-147: keep the first component's entry of every node
      const auto                         vector = laplace_operator.compute_inverse_diagonal();
      const Utilities::MPI::Partitioner &part   = *matrix_free->get_dof_info().vector_partitioner;
      diag_mat.diagonal.reinit(laplace_operator.context(), part.locally_owned_size() / n_components, 0,
                               dof_handler.n_dofs() / n_components);
      diag_mat.diagonal.extract_component(vector, n_components, 0);
    }

    // right-hand side i % 8 on unconstrained local entries, start vector 0 (benchmark.h:170-176)
    laplace_operator.initialize_dof_vector(input);
    laplace_operator.initialize_dof_vector(output);
    std::vector<double> rhs(input.local_size());
    for (std::size_t i = 0; i < rhs.size(); ++i)
      rhs[i] = double(i % 8);
    for (const unsigned int i : matrix_free->get_constrained_dofs())
      rhs[i] = 0.;
    input.upload(rhs.data(), rhs.size());
    bp4_check(bp4_ctx_synchronize(laplace_operator.context()));
  }

  unsigned int solve()
  {
    output = 0;
    return run_cg_solver(laplace_operator, output, input, diag_mat);
  }

  Triangulation                               tria;
  DoFHandler                                  dof_handler;
  AffineConstraints                           constraints;
  MatrixFree::AdditionalData                  mf_data;
  std::shared_ptr<MatrixFree>                 matrix_free;
  OperatorType                                laplace_operator;
  DiagonalMatrixBlocked<n_components, double> diag_mat;
  VectorType                                  input, output;
};

struct BenchmarkResult
{
  unsigned int  fe_degree = 0, n_q_points = 0, n_iterations = 0;
  std::uint64_t n_cells = 0, n_dofs = 0;
  double        solver_time = 0, matvec_time = 0, setup_time = 0;
};

// timing protocol of run_templated (benchmark.h:184-225): best of 4 solves, best of 2 x 50 vmults
template <int dim, int fe_degree, int n_q_points>
BenchmarkResult run_templated(const unsigned int s, const bool short_output, const BenchmarkOptions &opt = BenchmarkOptions())
{
  Timer                                        time;
  BenchmarkProblem<dim, fe_degree, n_q_points> problem(s, opt);
  BenchmarkResult                              res;
  res.fe_degree  = fe_degree;
  res.n_q_points = n_q_points;
  res.n_cells    = problem.tria.n_global_active_cells();
  res.n_dofs     = problem.dof_handler.n_dofs();
  if (!short_output)
    {
      const double diag_norm = problem.diag_mat.diagonal.l2_norm(); // benchmark.h:149-154
      if (opt.rank == 0)
        std::cout << "Norm of diagonal for preconditioner: " << diag_norm << std::endl;
    }
  res.setup_time = time.wall_time();
  if (!short_output && opt.rank == 0) // benchmark.h:178-182 (one process per GPU: no min/avg/max split)
    std::cout << "Setup time:         " << res.setup_time << "s" << std::endl;

  double solver_time = 1e10;
  for (unsigned int t = 0; t < 4; ++t)
    {
      bp4_check(bp4_ctx_synchronize(problem.laplace_operator.context()));
      time.restart();
      res.n_iterations = problem.solve();
      bp4_check(bp4_ctx_synchronize(problem.laplace_operator.context()));
      solver_time = std::min(time.wall_time(), solver_time);
    }
  double matvec_time = 1e10;
  for (unsigned int t = 0; t < 2; ++t)
    {
      time.restart();
      for (unsigned int i = 0; i < 50; ++i) // argument order as in the reference (benchmark.h:209)
        problem.laplace_operator.vmult(problem.input, problem.output);
      bp4_check(bp4_ctx_synchronize(problem.laplace_operator.context()));
      matvec_time = std::min(time.wall_time() / 50, matvec_time);
    }
  res.solver_time = solver_time;
  res.matvec_time = matvec_time;
  if (opt.rank == 0 && short_output)
    std::cout << std::setw(2) << fe_degree << " | " << std::setw(2) << n_q_points       //
              << " |" << std::setw(10) << res.n_cells                                   //
              << " |" << std::setw(11) << res.n_dofs                                    //
              << " | " << std::setw(11) << solver_time / res.n_iterations               //
              << " | " << std::setw(11) << res.n_dofs / solver_time * res.n_iterations  //
              << " | " << std::setw(4) << res.n_iterations                              //
              << " | " << std::setw(11) << matvec_time << std::endl;
  return res;
}

// size sweep of do_test (benchmark.h:229-267)
template <int dim, int fe_degree, int n_q_points>
void do_test(const int s_in, const bool compact_output, const BenchmarkOptions &opt = BenchmarkOptions())
{
  if (s_in < 1)
    {
      unsigned int s = 1 + (unsigned int)std::log2((double)opt.n_ranks);
      if (opt.rank == 0)
        std::cout << " p |  q | n_element |     n_dofs |     time/it |   dofs/s/it | itCG | time/matvec" << std::endl;
      while (std::uint64_t(fe_degree + 1) * (fe_degree + 1) * (fe_degree + 1) * (1ULL << s) * n_components <
             6000000ULL * opt.n_ranks)
        {
          run_templated<dim, fe_degree, n_q_points>(s, compact_output, opt);
          ++s;
        }
      if (opt.rank == 0)
        std::cout << std::endl << std::endl;
    }
  else
    run_templated<dim, fe_degree, n_q_points>(s_in, compact_output, opt);
}

// CLI of the reference: bench <degree> [s] [compact_output]  (benchmark.h:270-318).
// Degrees 2..8 have device kernels; the reference also instantiates 1 and 9..11.
inline void run(int argc, char **argv)
{
  unsigned int degree = 2;
  int          s      = -1;
  bool         compact_output = true;
  if (argc > 1)
    degree = std::atoi(argv[1]);
  if (argc > 2)
    s = std::atoi(argv[2]);
  if (argc > 3)
    compact_output = std::atoi(argv[3]);
  BenchmarkOptions opt;
  if (const char *d = std::getenv("BP4_DEVICE"))
    opt.device = std::atoi(d);
  switch (degree)
    {
      case 2: do_test<dimension, 2, 4>(s, compact_output, opt); break;
      case 3: do_test<dimension, 3, 5>(s, compact_output, opt); break;
      case 4: do_test<dimension, 4, 6>(s, compact_output, opt); break;
      case 5: do_test<dimension, 5, 7>(s, compact_output, opt); break;
      case 6: do_test<dimension, 6, 8>(s, compact_output, opt); break;
      case 7: do_test<dimension, 7, 9>(s, compact_output, opt); break;
      case 8: do_test<dimension, 8, 10>(s, compact_output, opt); break;
      default: AssertThrow(false, ExcMessage("Only degrees 2 to 8 implemented on the device"));
    }
}
