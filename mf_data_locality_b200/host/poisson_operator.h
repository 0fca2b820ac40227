// poisson_operator.h -- host-side mirror of the reference's Poisson::LaplaceOperator
// (poisson_operator.h:67-695): same template parameters, same public members
// (initialize, initialize_dof_vector, vmult, Tvmult, vmult_with_merged_sums,
// compute_inverse_diagonal, n_components, value_type, size_type).  All arithmetic runs on
// the B200 through the C ABI of include/bp4.h; this class only builds the two per-cell
// tables of LaplaceOperator::initialize -- the 27 compressed entity indices
// (poisson_operator.h:183-267) and the 8 vertices behind the tri-linear coefficients
// (:153-178) -- checks the "contiguous numbering" contract the renumbering must deliver,
// and hands them to bp4_ctx_create.
#pragma once
#include <array>
#include <memory>

#include "device_vector.h"
#include "diagonal_matrix_blocked.h"
#include "matrix_free_standin.h"

namespace Poisson
{
  using namespace dealii;

  // VectorizedArrayType is the reference's seventh parameter (poisson_operator.h:67-74): the SIMD
  // type of its CPU kernels.  Accepted and ignored so that reference call sites compile unchanged.
  template <int dim, int fe_degree, int n_q_points_1d = fe_degree + 1, int n_components_ = 1,
            typename Number = double, typename VectorType = LinearAlgebra::distributed::Vector<Number>,
            typename VectorizedArrayType = void>
  class LaplaceOperator
  {
  public:
    typedef Number                  value_type;
    typedef types::global_dof_index size_type;
    static constexpr unsigned int   n_components = n_components_;
    static_assert(dim == 3 && n_components_ == 3, "BP4: three components in three dimensions");

    LaplaceOperator() = default;
    LaplaceOperator(const LaplaceOperator &) = delete;
    ~LaplaceOperator()
    {
      if (ctx)
        bp4_ctx_destroy(ctx);
    }

    void initialize(std::shared_ptr<const MatrixFree> data_, const AffineConstraints &constraints,
                    const int device = 0, const bool deterministic = false)
    {
      data = data_;
      const DoFHandler &dh = data->get_dof_handler();
      AssertThrow(dh.get_fe().n_components() == n_components, "n_components mismatch");
      AssertThrow(dh.get_fe().degree == fe_degree, "fe_degree mismatch");
      const Utilities::MPI::Partitioner &part = *data->get_dof_info().vector_partitioner;
      const unsigned int                 n_cells = data->n_physical_cells();
      compressed_dof_indices.assign(std::size_t(27) * n_cells, numbers::invalid_unsigned_int);
      cell_vertices.resize(std::size_t(24) * n_cells);
      constexpr unsigned int p = fe_degree;
      const unsigned int lo[3] = {0, 1, p}, hi[3] = {1, p, p + 1};
      // cells in loop order (batch by batch, lane by lane); the per-cell work is independent
      parallel_chunks(n_cells, [&](const std::uint64_t c0, const std::uint64_t c1) {
        for (std::uint64_t cell_no = c0; cell_no < c1; ++cell_no)
          {
            const std::uint64_t cell = data->cell_order[cell_no];
            for (unsigned int v = 0; v < 8; ++v)
              {
                const Point3 x = dh.get_triangulation().vertex(cell, v);
                for (unsigned int d = 0; d < 3; ++d)
                  cell_vertices[24 * std::size_t(cell_no) + 3 * v + d] = x[d];
              }
            for (unsigned int a = 0; a < 27; ++a)
              {
                const unsigned int ex = a % 3, ey = (a / 3) % 3, ez = a / 9;
                const std::uint64_t n0 = dh.cell_node(cell, lo[ex], lo[ey], lo[ez]);
                if (constraints.node_is_constrained(n0))
                  continue; // entity stays invalid: read as 0, never written (:194, :205)
                const types::global_dof_index g0 = dh.dof_number(n0, 0);
                // contract of the renumbering: the entity's DoFs are contiguous, nodes
                // lexicographic, components interleaved (:197-199, :207-211, :224-239, :251-255)
                types::global_dof_index expect = g0;
                for (unsigned int k = lo[ez]; k < hi[ez]; ++k)
                  for (unsigned int j = lo[ey]; j < hi[ey]; ++j)
                    for (unsigned int i = lo[ex]; i < hi[ex]; ++i, expect += n_components)
                      AssertThrow(dh.dof_number(dh.cell_node(cell, i, j, k), 0) == expect,
                                  ExcMessage("Expected contiguous numbering"));
                compressed_dof_indices[27 * std::size_t(cell_no) + a] = part.global_to_local(g0);
              }
          }
      });

      compute_private_ranges(dh, constraints, part);
      // quadratic mapping: all 27 coefficient vectors v_{a+3b+9c} of X = sum v_m xi^a eta^b zeta^c
      // (cell_quadratic_coefficients, :690) from the 27 geometry nodes; per direction the
      // interpolant through t = 0, 1/2, 1 is f0 + (-3 f0 + 4 f1 - f2) t + (2 f0 - 4 f1 + 2 f2) t^2
      cell_coefficients.clear();
      if (data->get_additional_data().mapping_degree == 2)
        {
          cell_coefficients.resize(std::size_t(81) * n_cells);
          static const double T[3][3] = {{1., 0., 0.}, {-3., 4., -1.}, {2., -4., 2.}};
          parallel_chunks(n_cells, [&](const std::uint64_t c0, const std::uint64_t c1) {
            for (std::uint64_t cell_no = c0; cell_no < c1; ++cell_no)
              {
                const std::uint64_t cell = data->cell_order[cell_no];
                Point3              X[27];
                for (unsigned int k = 0; k < 3; ++k)
                  for (unsigned int j = 0; j < 3; ++j)
                    for (unsigned int i = 0; i < 3; ++i)
                      X[i + 3 * j + 9 * k] = dh.get_triangulation().point27(cell, i, j, k);
                for (unsigned int c = 0; c < 3; ++c)
                  for (unsigned int b = 0; b < 3; ++b)
                    for (unsigned int a = 0; a < 3; ++a)
                      for (unsigned int d = 0; d < 3; ++d)
                        {
                          double v = 0.;
                          for (unsigned int k = 0; k < 3; ++k)
                            for (unsigned int j = 0; j < 3; ++j)
                              for (unsigned int i = 0; i < 3; ++i)
                                v += T[c][k] * T[b][j] * T[a][i] * X[i + 3 * j + 9 * k][d];
                          cell_coefficients[81 * std::size_t(cell_no) + 3 * (a + 3 * b + 9 * c) + d] = v;
                        }
              }
          });
        }
      else
        AssertThrow(data->get_additional_data().mapping_degree == 1, "mapping degree 1 or 2");

      bp4_desc desc{};
      desc.n_ranges             = range_cell_offset.empty() ? 0 : range_cell_offset.size() - 1;
      desc.range_cell_offset    = range_cell_offset.data();
      desc.range_private_offset = range_private_offset.data();
      desc.coefficients         = cell_coefficients.empty() ? nullptr : cell_coefficients.data();
      desc.degree        = fe_degree;
      desc.device        = device;
      desc.n_cells       = n_cells;
      desc.n_owned       = part.locally_owned_size();
      desc.n_ghost       = part.n_ghost_indices();
      desc.entity_index  = compressed_dof_indices.data();
      desc.vertices      = cell_vertices.data();
      desc.n_constrained = data->get_constrained_dofs().size();
      desc.constrained   = data->get_constrained_dofs().data();
      desc.n_peers       = (int)part.peers.size();
      desc.peer_rank     = part.peers.data();
      desc.import_offset = part.import_offset.data();
      desc.export_offset = part.export_offset.data();
      desc.export_index  = part.export_index.data();
      desc.n_cells_before_comm = data->n_cells_before_comm;
      desc.n_cells_comm        = data->n_cells_comm;
      desc.deterministic       = deterministic ? 1 : 0;
      if (ctx)
        bp4_ctx_destroy(ctx);
      ctx = nullptr;
      if (device >= 0) // device < 0: tables only (host-side checks without a GPU)
        bp4_check(bp4_ctx_create(&desc, &ctx));
    }

    void initialize_dof_vector(VectorType &vec) const
    {
      const Utilities::MPI::Partitioner &part = *data->get_dof_info().vector_partitioner;
      vec.reinit(ctx, part.locally_owned_size(), part.n_ghost_indices(), data->get_dof_handler().n_dofs());
    }

    // dst = A src, identity on Dirichlet rows (poisson_operator.h:307-313)
    void vmult(VectorType &dst, const VectorType &src) const
    {
      bp4_check(bp4_vmult(ctx, dst.handle(), src.handle()));
    }
    void Tvmult(VectorType &dst, const VectorType &src) const { vmult(dst, src); }

    // pre-update of x, g, d, h; h = A d; the seven merged sums over all ranks
    // (poisson_operator.h:327-377; Tensor<1,7> becomes std::array<double,7>)
    std::array<Number, 7> vmult_with_merged_sums(VectorType &x, VectorType &g, VectorType &d, VectorType &h,
                                                 const DiagonalMatrixBlocked<n_components, Number> &prec,
                                                 const Number alpha, const Number beta,
                                                 const Number alpha_old, const Number beta_old) const
    {
      std::array<Number, 7> sums;
      bp4_check(bp4_vmult_merged(ctx, x.handle(), g.handle(), d.handle(), h.handle(),
                                 prec.diagonal.handle(), alpha, beta, alpha_old, beta_old, sums.data()));
      return sums;
    }

    // Inverse diagonal of the scalar Laplacian under the quadrature this operator was set up
    // with (the reference instantiates it with GLL(p+1), benchmark.h:128-140), returned the way
    // the reference returns it (poisson_operator.h:392-426): a DoF vector with 1/diag on the
    // first component of every node and 1 wherever the assembled value is 0.  The caller keeps
    // every n_components-th entry (benchmark.h:141-147).
    VectorType compute_inverse_diagonal() const
    {
      VectorType diag;
      initialize_dof_vector(diag);
      bp4_check(bp4_inverse_diagonal_vector(ctx, diag.handle()));
      return diag;
    }

    // cell-batch ranges of the loop and the owned DoFs private to each (bp4_desc::n_ranges)
    const std::vector<std::uint64_t> &get_range_cell_offset() const { return range_cell_offset; }
    const std::vector<std::uint64_t> &get_range_private_offset() const { return range_private_offset; }

    bp4_ctx                          *context() const { return ctx; }
    const std::vector<unsigned int>  &get_compressed_dof_indices() const { return compressed_dof_indices; }
    const std::vector<double>        &get_cell_vertices() const { return cell_vertices; }
    const std::vector<double>        &get_cell_coefficients() const { return cell_coefficients; }
    const MatrixFree                 &get_matrix_free() const { return *data; }

  private:
    // The DoF ranges MatrixFree::cell_loop hands to the pre/post hooks of vmult_with_merged_sums
    // right around a cell-batch range's own cells (poisson_operator.h:339-364) are the DoFs no
    // other range touches.  Renumber(*, *, 2) numbers exactly those first and range by range
    // (touch_count_cellbatch_range + touch_count_grouping, renumber_dofs_for_mf.h:556-590,
    // :622-671); here they are re-derived from the cell loop (same walk as the renumbering) and
    // handed to the device as one contiguous run per range.  If the numbering in use does not
    // deliver contiguous runs starting at DoF 0 (e.g. renumbering switched off), the tables stay
    // empty and the device streams the vector updates over the whole vector instead.
    void compute_private_ranges(const DoFHandler &dh, const AffineConstraints &constraints,
                                const Utilities::MPI::Partitioner &part)
    {
      range_cell_offset.clear();
      range_private_offset.clear();
      const auto         &ti      = data->get_task_info();
      const unsigned int  rank    = data->get_rank();
      const std::uint64_t first   = part.owned.first / n_components;
      const std::uint64_t n_nodes = part.locally_owned_size() / n_components;
      const unsigned int  n_ranges = (unsigned int)ti.cell_partition_data.size() - 1;
      if (n_ranges == 0)
        return;
      // per owned node: the one range around it, or invalid if there are several / it is shared
      // with another rank / Dirichlet (node by node from the lattice, in parallel)
      std::vector<std::uint32_t> only_range(n_nodes, numbers::invalid_unsigned_int);
      dh.parallel_rank_nodes(rank, [&](const std::uint64_t a, const std::uint64_t b) {
        for (std::uint64_t n = a; n < b; ++n)
          {
            if (dh.owner[n] != rank || dh.shared[n] || constraints.node_is_constrained(n))
              continue;
            std::uint32_t      ps[8];
            const unsigned int np = data->incident_positions(n, ps);
            bool               one = np > 0;
            for (unsigned int k = 1; k < np; ++k)
              one &= data->range_of_pos[ps[k]] == data->range_of_pos[ps[0]];
            if (one)
              only_range[dh.node_number[n] - first] = data->range_of_pos[ps[0]];
          }
      });
      // private = one range, not shared with another rank, not Dirichlet
      std::vector<std::uint64_t> n_private(n_ranges, 0), lo(n_ranges, ~std::uint64_t(0)), hi(n_ranges, 0);
      for (std::uint64_t i = 0; i < n_nodes; ++i)
        if (only_range[i] != numbers::invalid_unsigned_int)
          {
            const std::uint32_t r = only_range[i];
            ++n_private[r];
            lo[r] = std::min(lo[r], i);
            hi[r] = std::max(hi[r], i + 1);
          }
      std::vector<std::uint64_t> cell_off(n_ranges + 1, 0), priv_off(n_ranges + 1, 0);
      bool                       contiguous = true;
      for (unsigned int r = 0; r < n_ranges; ++r)
        {
          cell_off[r + 1] = data->batch_start[ti.cell_partition_data[r + 1]];
          priv_off[r + 1] = priv_off[r] + n_components * n_private[r];
          if (n_private[r] && (n_components * lo[r] != priv_off[r] || n_components * hi[r] != priv_off[r + 1]))
            contiguous = false;
        }
      if (!contiguous)
        return;
      range_cell_offset.swap(cell_off);
      range_private_offset.swap(priv_off);
    }

    std::vector<std::uint64_t>        range_cell_offset, range_private_offset;
    std::shared_ptr<const MatrixFree> data;
    std::vector<unsigned int>         compressed_dof_indices; // [cell][27], one lane per cell
    std::vector<double>               cell_vertices;          // [cell][8][3]
    std::vector<double>               cell_coefficients;      // [cell][27][3], quadratic mapping only
    bp4_ctx                          *ctx = nullptr;
  };
} // namespace Poisson
