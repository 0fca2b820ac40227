// host_capi.cc -- C entry points over the host-side mirror (benchmark.h + one plugin), so
// that tests/ and bench.py can drive the SAME C++ path the CLI executables run: problem
// set-up (mesh, Renumber, LaplaceOperator::initialize), the run_cg_solver plugin and vmult.
// Built once per plugin: libbp4_host_plain.so / libbp4_host_merged.so and the device-resident
// solves libbp4_host_plain_device.so / libbp4_host_merged_device.so.
#define BP4_NO_MAIN
#if defined(BP4_PLUGIN_MERGED)
#  include "../benchmark_precond_merged/bench.cc"
#elif defined(BP4_PLUGIN_PLAIN_DEVICE)
#  include "../benchmark_precond_device/bench.cc"
#elif defined(BP4_PLUGIN_MERGED_DEVICE)
#  include "../benchmark_precond_merged_device/bench.cc"
#else
#  include "../benchmark_precond/bench.cc"
#endif

#include <cstring>

namespace
{
  thread_local std::string g_error;

  struct ProblemBase
  {
    virtual ~ProblemBase() = default;
    virtual unsigned int  solve()                                       = 0;
    virtual void          vmult()                                       = 0;
    virtual bp4_ctx      *ctx()                                         = 0;
    virtual const MatrixFree &mf()                                      = 0;
    virtual const DoFHandler &dh()                                      = 0;
    virtual const std::vector<unsigned int> &entity()                   = 0;
    virtual const std::vector<double>       &vertices()                 = 0;
    virtual const std::vector<double>       &coefficients()             = 0;
    virtual const std::vector<std::uint64_t> &range_cells()             = 0;
    virtual const std::vector<std::uint64_t> &range_private()           = 0;
    virtual LinearAlgebra::distributed::Vector<double> &input()         = 0;
    virtual LinearAlgebra::distributed::Vector<double> &output()        = 0;
    virtual LinearAlgebra::distributed::Vector<double> &diagonal()      = 0;
    double setup_seconds = 0;
  };

  template <int p>
  struct ProblemT : ProblemBase
  {
    ProblemT(unsigned int s, const BenchmarkOptions &opt) : prob(s, opt) {}
    unsigned int solve() override { return prob.solve(); }
    void         vmult() override { prob.laplace_operator.vmult(prob.output, prob.input); }
    bp4_ctx     *ctx() override { return prob.laplace_operator.context(); }
    const MatrixFree &mf() override { return *prob.matrix_free; }
    const DoFHandler &dh() override { return prob.dof_handler; }
    const std::vector<unsigned int> &entity() override { return prob.laplace_operator.get_compressed_dof_indices(); }
    const std::vector<double>       &vertices() override { return prob.laplace_operator.get_cell_vertices(); }
    const std::vector<double>       &coefficients() override { return prob.laplace_operator.get_cell_coefficients(); }
    const std::vector<std::uint64_t> &range_cells() override { return prob.laplace_operator.get_range_cell_offset(); }
    const std::vector<std::uint64_t> &range_private() override { return prob.laplace_operator.get_range_private_offset(); }
    LinearAlgebra::distributed::Vector<double> &input() override { return prob.input; }
    LinearAlgebra::distributed::Vector<double> &output() override { return prob.output; }
    LinearAlgebra::distributed::Vector<double> &diagonal() override { return prob.diag_mat.diagonal; }
    BenchmarkProblem<3, p, p + 2> prob;
  };

  template <typename F>
  int guarded(F &&f)
  {
    try
      {
        f();
        return 0;
      }
    catch (const std::exception &e)
      {
        g_error = e.what();
        return -1;
      }
  }
} // namespace

extern "C" {

const char *bp4h_last_error(void) { return g_error.c_str(); }
const char *bp4h_plugin(void)
{
#if defined(BP4_PLUGIN_MERGED)
  return "benchmark_precond_merged";
#elif defined(BP4_PLUGIN_PLAIN_DEVICE)
  return "benchmark_precond_device";
#elif defined(BP4_PLUGIN_MERGED_DEVICE)
  return "benchmark_precond_merged_device";
#else
  return "benchmark_precond";
#endif
}

// options: [n_ranks, rank, device, n_lanes, batches_per_range, renumber_a, renumber_r, renumber_g,
//           numbering_only, mapping_degree, deterministic]
int bp4h_create(int degree, int s, const int *options, const unsigned char *nccl_id, void **out)
{
  return guarded([&] {
    BenchmarkOptions opt;
    opt.nccl_id = nccl_id;
    if (options)
      {
        opt.n_ranks = options[0], opt.rank = options[1], opt.device = options[2];
        opt.n_lanes = options[3], opt.batches_per_range = options[4];
        opt.renumber_a = options[5], opt.renumber_r = options[6], opt.renumber_g = options[7];
        opt.numbering_only = options[8] != 0;
        opt.mapping_degree = options[9] > 0 ? options[9] : 1;
        opt.deterministic  = options[10] != 0;
      }
    Timer        t;
    ProblemBase *p = nullptr;
    switch (degree)
      {
        case 2: p = new ProblemT<2>(s, opt); break;
        case 3: p = new ProblemT<3>(s, opt); break;
        case 4: p = new ProblemT<4>(s, opt); break;
        case 5: p = new ProblemT<5>(s, opt); break;
        case 6: p = new ProblemT<6>(s, opt); break;
        case 7: p = new ProblemT<7>(s, opt); break;
        case 8: p = new ProblemT<8>(s, opt); break;
        default: throw std::runtime_error("Only degrees 2 to 8 implemented on the device");
      }
    p->setup_seconds = t.wall_time();
    *out             = p;
  });
}

int bp4h_destroy(void *h)
{
  return guarded([&] { delete static_cast<ProblemBase *>(h); });
}

// sizes: [n_cells_local, n_owned, n_ghost, n_dofs_global, n_cells_global, n_constrained, n_batches, n_ranges]
int bp4h_sizes(void *h, std::uint64_t *sizes)
{
  return guarded([&] {
    ProblemBase *p    = static_cast<ProblemBase *>(h);
    const auto  &part = *p->mf().get_dof_info().vector_partitioner;
    sizes[0]          = p->mf().n_physical_cells();
    sizes[1]          = part.locally_owned_size();
    sizes[2]          = part.n_ghost_indices();
    sizes[3]          = p->dh().n_dofs();
    sizes[4]          = p->dh().get_triangulation().n_global_active_cells();
    sizes[5]          = p->mf().get_constrained_dofs().size();
    sizes[6]          = p->mf().n_cell_batches();
    sizes[7]          = p->mf().get_task_info().cell_partition_data.size() - 1;
  });
}

void *bp4h_ctx(void *h) { return static_cast<ProblemBase *>(h)->ctx(); }
double bp4h_setup_seconds(void *h) { return static_cast<ProblemBase *>(h)->setup_seconds; }

int bp4h_get_entity_index(void *h, std::uint32_t *out)
{
  return guarded([&] {
    const auto &e = static_cast<ProblemBase *>(h)->entity();
    std::memcpy(out, e.data(), e.size() * sizeof(std::uint32_t));
  });
}
int bp4h_get_vertices(void *h, double *out)
{
  return guarded([&] {
    const auto &v = static_cast<ProblemBase *>(h)->vertices();
    std::memcpy(out, v.data(), v.size() * sizeof(double));
  });
}
// cell-batch ranges + private DoF runs handed to the device (bp4_desc::n_ranges): *n = number of
// table entries (n_ranges + 1, 0 when the numbering has no contiguous private runs); the
// tables are copied when the pointers are non-null
int bp4h_get_ranges(void *h, std::uint64_t *n, std::uint64_t *cell_offset, std::uint64_t *private_offset)
{
  return guarded([&] {
    ProblemBase *p = static_cast<ProblemBase *>(h);
    *n             = p->range_cells().size();
    if (cell_offset)
      std::copy(p->range_cells().begin(), p->range_cells().end(), cell_offset);
    if (private_offset)
      std::copy(p->range_private().begin(), p->range_private().end(), private_offset);
  });
}
// [n_cells][27][3] geometry coefficients of a quadratic mapping (*n = 0 for the tri-linear one)
int bp4h_get_coefficients(void *h, std::uint64_t *n, double *out)
{
  return guarded([&] {
    const auto &c = static_cast<ProblemBase *>(h)->coefficients();
    *n            = c.size();
    if (out)
      std::memcpy(out, c.data(), c.size() * sizeof(double));
  });
}
int bp4h_get_constrained(void *h, std::uint32_t *out)
{
  return guarded([&] {
    const auto &c = static_cast<ProblemBase *>(h)->mf().get_constrained_dofs();
    std::memcpy(out, c.data(), c.size() * sizeof(std::uint32_t));
  });
}
// lattice node id of every local node (owned in renumbered order, then ghosts): the DoF
// permutation in a labelling that does not depend on either implementation's internals
int bp4h_get_node_of_local(void *h, std::uint64_t *out)
{
  return guarded([&] {
    ProblemBase      *p    = static_cast<ProblemBase *>(h);
    const DoFHandler &dh   = p->dh();
    const auto       &part = *p->mf().get_dof_info().vector_partitioner;
    const std::uint64_t first = part.owned.first / 3, n_own = part.locally_owned_size() / 3;
    const unsigned int  rank  = p->mf().get_rank();
    for (std::uint64_t n = 0; n < dh.n_nodes; ++n)
      if (dh.owner[n] == rank)
        out[dh.node_number[n] - first] = n;
    if (!part.ghost_nodes.empty())
      {
        std::vector<std::uint64_t> lattice_of_number; // only for ghosts: search by number
        for (std::uint64_t n = 0; n < dh.n_nodes; ++n)
          if (dh.owner[n] != rank && dh.shared[n]) // ghosts are shared nodes; the others may carry
            {                                      // stale numbers (Renumber's neighbour shortcut)
              const auto it = std::lower_bound(part.ghost_nodes.begin(), part.ghost_nodes.end(), dh.node_number[n]);
              if (it != part.ghost_nodes.end() && *it == dh.node_number[n])
                out[n_own + (it - part.ghost_nodes.begin())] = n;
            }
      }
  });
}

// exchange plan: counts = [n_peers, n_export]; then peers[n_peers], import_offset[n_peers+1],
// export_offset[n_peers+1], export_index[n_export]
int bp4h_plan_sizes(void *h, std::uint64_t *counts)
{
  return guarded([&] {
    const auto &part = *static_cast<ProblemBase *>(h)->mf().get_dof_info().vector_partitioner;
    counts[0]        = part.peers.size();
    counts[1]        = part.export_index.size();
  });
}
int bp4h_get_plan(void *h, int *peers, std::uint64_t *import_offset, std::uint64_t *export_offset,
                  std::uint32_t *export_index)
{
  return guarded([&] {
    const auto &part = *static_cast<ProblemBase *>(h)->mf().get_dof_info().vector_partitioner;
    std::copy(part.peers.begin(), part.peers.end(), peers);
    std::copy(part.import_offset.begin(), part.import_offset.end(), import_offset);
    std::copy(part.export_offset.begin(), part.export_offset.end(), export_offset);
    std::copy(part.export_index.begin(), part.export_index.end(), export_index);
  });
}

int bp4h_set_solver(unsigned int max_steps, double abs_tol, double rel_tol)
{
  solver_settings().max_steps = max_steps;
  solver_settings().abs_tol   = abs_tol;
  solver_settings().rel_tol   = rel_tol;
  return 0;
}

// upload b (may be null: keep the default i % 8 right-hand side), run the plugin's
// run_cg_solver with x0 = 0, download x (may be null)
int bp4h_run_cg_solver(void *h, const double *b_host, double *x_host, unsigned int *iterations)
{
  return guarded([&] {
    ProblemBase *p = static_cast<ProblemBase *>(h);
    if (b_host)
      p->input().upload(b_host, p->input().local_size());
    *iterations = p->solve();
    if (x_host)
      p->output().download(x_host, p->output().local_size());
  });
}

// the residuals the last bp4h_run_cg_solver checked, steps 0 .. last_step: *n = their number;
// out (may be null) receives them
int bp4h_solver_history(double *out, unsigned int *n)
{
  const std::vector<double> &hist = last_solve_history();
  *n                              = (unsigned int)hist.size();
  if (out)
    std::copy(hist.begin(), hist.end(), out);
  return 0;
}

int bp4h_vmult(void *h, const double *src_host, double *dst_host)
{
  return guarded([&] {
    ProblemBase *p = static_cast<ProblemBase *>(h);
    if (src_host)
      p->input().upload(src_host, p->input().local_size());
    p->vmult();
    if (dst_host)
      p->output().download(dst_host, p->output().local_size());
  });
}

int bp4h_get_rhs(void *h, double *out)
{
  return guarded([&] {
    ProblemBase *p = static_cast<ProblemBase *>(h);
    p->input().download(out, p->input().local_size());
  });
}

int bp4h_get_diagonal(void *h, double *out)
{
  return guarded([&] {
    ProblemBase *p = static_cast<ProblemBase *>(h);
    p->diagonal().download(out, p->diagonal().local_size());
  });
}

} // extern "C"
