// solver_control.h -- SolverControl / ReductionControl and the stock SolverCG of deal.II 9.3 as
// the reference instantiates them (benchmark_precond*/bench.cc:11-16), restated from the
// library's documented algorithm (SURVEY App. B3).  Vector operations go to the device
// through the vector stand-in.
#pragma once
#include <cmath>
#include <limits>
#include <stdexcept>
#include <vector>

namespace dealii
{
  class SolverControl
  {
  public:
    enum State { iterate = 0, success, failure };
    struct NoConvergence : public std::runtime_error
    {
      NoConvergence(unsigned int s, double r) : std::runtime_error("no convergence"), last_step(s), last_residual(r) {}
      unsigned int last_step;
      double       last_residual;
    };
    SolverControl(unsigned int n = 100, double tol = 1e-10) : maxsteps(n), tol(tol) {}
    virtual ~SolverControl() = default;
    virtual State check(const unsigned int step, const double check_value)
    {
      if (step == 0)
        initial_val = check_value;
      lstep  = step;
      lvalue = check_value;
      if (history_data_enabled)
        history_data.push_back(check_value);
      if (check_value <= tol)
        return lcheck = success;
      if (step >= maxsteps || std::isnan(check_value))
        return lcheck = failure;
      return lcheck = iterate;
    }
    unsigned int last_step() const { return lstep; }
    double       last_value() const { return lvalue; }
    double       initial_value() const { return initial_val; }
    State        last_check() const { return lcheck; }
    unsigned int max_steps() const { return maxsteps; }
    double       tolerance() const { return tol; }
    // every checked value, in check order (deal.II's enable_history_data / get_history_data)
    void                       enable_history_data() { history_data_enabled = true; }
    const std::vector<double> &get_history_data() const { return history_data; }

  protected:
    bool                history_data_enabled = false;
    std::vector<double> history_data;
    unsigned int maxsteps;
    double       tol, lvalue = 0, initial_val = 0;
    unsigned int lstep  = 0;
    State        lcheck = iterate;
  };

  // stop when the residual dropped below tol OR by the factor `reduce` relative to step 0
  class ReductionControl : public SolverControl
  {
  public:
    ReductionControl(unsigned int n = 100, double tol = 1e-10, double red = 1e-2)
      : SolverControl(n, tol), reduce(red)
    {}
    double reduction() const { return reduce; }
    State  check(const unsigned int step, const double check_value) override
    {
      if (step == 0)
        {
          initial_val = check_value;
          reduced_tol = check_value * reduce;
        }
      if (check_value < reduced_tol) // strict, as in deal.II's ReductionControl::check
        {
          lstep  = step;
          lvalue = check_value;
          if (history_data_enabled)
            history_data.push_back(check_value);
          return lcheck = success;
        }
      return SolverControl::check(step, check_value);
    }

  protected:
    double reduce, reduced_tol = 0;
  };

  template <typename VectorType>
  class SolverBase
  {
  public:
    explicit SolverBase(SolverControl &cn) : control(cn) {}
    SolverControl::State iteration_status(const unsigned int step, const double value, const VectorType &)
    {
      return control.check(step, value);
    }
    SolverControl &control;
  };

  // preconditioned CG, deal.II 9.3 SolverCG::solve
  template <typename VectorType>
  class SolverCG : public SolverBase<VectorType>
  {
  public:
    explicit SolverCG(SolverControl &cn) : SolverBase<VectorType>(cn) {}

    template <typename MatrixType, typename PreconditionerType>
    void solve(const MatrixType &A, VectorType &x, const VectorType &b, const PreconditionerType &preconditioner)
    {
      SolverControl::State conv = SolverControl::iterate;
      VectorType           g, d, h;
      g.reinit(x, true);
      d.reinit(x, true);
      h.reinit(x, true);
      int    it  = 0;
      double res = -std::numeric_limits<double>::max();
      if (!x.all_zero())
        {
          A.vmult(g, x);
          g.add(-1., b);
        }
      else
        g.equ(-1., b);
      res  = g.l2_norm();
      conv = this->iteration_status(0, res, x);
      if (conv != SolverControl::iterate)
        return;
      preconditioner.vmult(h, g);
      d.equ(-1., h);
      double gh = g * h;
      while (conv == SolverControl::iterate)
        {
          it++;
          A.vmult(h, d);
          double alpha = d * h; // deal.II asserts alpha != 0 in debug builds only
          alpha        = gh / alpha;
          x.add(alpha, d);
          res  = std::sqrt(std::abs(g.add_and_dot(alpha, h, g)));
          conv = this->iteration_status(it, res, x);
          if (conv != SolverControl::iterate)
            break;
          preconditioner.vmult(h, g);
          const double beta_den = gh;
          gh                    = g * h;
          d.sadd(gh / beta_den, -1., h);
        }
      if (conv != SolverControl::success)
        throw SolverControl::NoConvergence(it, res);
    }
  };
} // namespace dealii
