// bp4_capi.cu -- implementation of the C ABI declared in include/bp4.h.
// Owns the device copies of the mesh data LaplaceOperator::initialize builds
// (poisson_operator.h:101-293), the vectors, the stream and the reduction scratch.
// There is no CPU fallback: every entry point needs a CUDA device.
#include <cuda.h>
#include <nccl.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <map>
#include <string>
#include <vector>

#include "../../include/bp4.h"
#include "bp4_launch.h"

namespace
{
  thread_local std::string g_err;

  int fail(int code, const char *fmt, ...)
  {
    char    buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
  }
} // namespace

#define CU(call)                                                                              \
  do                                                                                          \
    {                                                                                         \
      cudaError_t e_ = (call);                                                                \
      if (e_ != cudaSuccess)                                                                  \
        return fail(BP4_ERR_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #call,                  \
                    cudaGetErrorString(e_));                                                  \
    }                                                                                         \
  while (0)

#define NC(call)                                                                              \
  do                                                                                          \
    {                                                                                         \
      ncclResult_t r_ = (call);                                                               \
      if (r_ != ncclSuccess)                                                                  \
        return fail(BP4_ERR_NCCL, "%s:%d %s: %s", __FILE__, __LINE__, #call,                  \
                    ncclGetErrorString(r_));                                                  \
    }                                                                                         \
  while (0)

struct bp4_vec
{
  double  *buf = nullptr;
  uint64_t n   = 0;
  double  *p() const { return buf; }
};

struct ProfEvent
{
  cudaEvent_t a, b;
  int         id;
};

// instantiated graph of one device-resident solve (bp4_solve_cg / bp4_solve_cg_merged), keyed by
// the variant, the caller's x, b and prec buffers and the in-loop form; it owns the temporaries
// g, d, h so that their addresses, baked into the graph, stay valid
struct SolveGraph
{
  bool            merged = false;
  int             fused  = 0;
  const double   *x = nullptr, *b = nullptr, *prec = nullptr;
  double         *g = nullptr, *d = nullptr, *h = nullptr;
  cudaGraph_t     graph = nullptr;
  cudaGraphExec_t exec  = nullptr;
};

struct bp4_ctx
{
  int          degree = 0, device = 0, sms = 0;
  int          n_coef = 24; // geometry coefficients per cell: 24 (tri-linear) or 81 (all 27 vectors)
  uint64_t     n_cells = 0, n_owned = 0, n_ghost = 0, n_constrained = 0;
  uint64_t     n_before = 0, n_comm = 0; // cell partitions for the overlapped exchange
  cudaStream_t comm_stream = nullptr;
  cudaEvent_t  ev_a = nullptr, ev_b = nullptr;
  int          overlap = 1;
  cudaStream_t stream = nullptr;
  uint32_t    *d_entity = nullptr, *d_constrained = nullptr, *d_walk = nullptr;
  double      *d_coef = nullptr, *d_gll = nullptr;
  double      *d_acc  = nullptr; // [8] reduction scratch
  int         *d_flag = nullptr;
  uint32_t    *d_sched = nullptr; // [n_sched] unit counters of the cell-kernel launches of one loop
  uint32_t     n_sched = 4;       // 4, or one per colour in the deterministic mode
  double      *h_acc  = nullptr; // pinned [8] + sequence word (h_acc[8] reinterpreted), device-mapped
  unsigned long long pub_seq = 0;
  int         *h_flag = nullptr; // pinned
  // device-resident solves: the solver state, its pinned host images ([0] initial state read by
  // the graph, [1] final state written by it) and the cached graphs
  bp4::SolveState        *d_state = nullptr;
  bp4::SolveState        *h_state = nullptr;
  std::vector<SolveGraph> solves;
  // fused merged loop (vmult_with_merged_sums): units of whole cell-batch ranges, their batches
  // and the private DoF runs the vector updates are hooked to (bp4_kernels.cuh, BatchDesc)
  int             fused      = 0;      // 1: do_cg_update4b/3b on private DoFs inside the cell kernel
  bool            fused_pinned = false; // chosen by BP4_FUSED / bp4_debug_set_fused: comm_init keeps it
  uint64_t        n_private  = 0;      // [0, n_private) are private to one range, the rest is streamed
  uint32_t        unit_part[4] = {0, 0, 0, 0}; // first unit of the three cell partitions (+ end)
  bp4::BatchDesc *d_batch      = nullptr;
  uint32_t       *d_unit_batch = nullptr;
  // deterministic mode (DESIGN.md 4.6): cells stored colour by colour, colour k = stored cells
  // [color_off[k], color_off[k+1]); cell_color[i] = colour of the caller's cell i; the ordered
  // reductions' slots and ticket
  bool                  deterministic = false;
  uint32_t              n_colors      = 0;
  std::vector<uint64_t> color_off;
  std::vector<uint32_t> cell_color;
  bp4::DetSlots         det;
  // multi-GPU
  ncclComm_t            comm = nullptr;
  int                   rank = 0, n_ranks = 1;
  std::vector<int>      peer;
  std::vector<uint64_t> import_off, export_off;
  uint32_t             *d_export = nullptr;
  double               *d_sendbuf = nullptr, *d_recvbuf = nullptr;
  // Peer exchange without SMs (the USE_SHMEM analogue of benchmark.h:35, :105-108): every rank
  // owns one IPC-shared arena [flags | ghost_in[2] | contrib_in[2]]; owners push their exported
  // values into the peers' ghost_in with copy-engine peer copies, ghost holders push their
  // contributions into the owners' contrib_in, and arrival / release is signalled with stream
  // memory operations (cuStreamWriteValue64 / cuStreamWaitValue64) on the flag words -- nothing
  // of it needs an SM, so it runs next to the persistent cell kernel.
  struct P2P
  {
    bool                 on = false;
    char                *arena = nullptr;           // my arena (device)
    uint64_t             off_ghost[2] = {0, 0}, off_contrib[2] = {0, 0};
    std::vector<char *>  peer_arena;                // [n_peers] mapped base of peer k's arena
    std::vector<uint64_t> peer_off_ghost[2], peer_off_contrib[2]; // [n_peers] byte offsets there
    std::vector<uint64_t> peer_imp_off, peer_exp_off; // [n_peers] where MY data goes (doubles)
    uint64_t             epoch_fwd = 0, epoch_rev = 0;
    CUresult (*write64)(CUstream, CUdeviceptr, cuuint64_t, unsigned) = nullptr;
    CUresult (*wait64)(CUstream, CUdeviceptr, cuuint64_t, unsigned)  = nullptr;
  } p2p;
  // freed vector buffers kept for reuse, keyed by size: plays the role of deal.II's
  // GrowingVectorMemory pool behind SolverCGFullMerge's temporaries (solver_cg_optimized.h:201)
  std::multimap<uint64_t, double *> pool;
  // measurement
  bool                   profile = false;
  std::vector<ProfEvent> events;
  std::vector<cudaEvent_t> event_pool; // recycled timing events (creating one costs microseconds)
  double                 prof_ms[BP4_K_COUNT]  = {0};
  uint64_t               prof_cnt[BP4_K_COUNT] = {0};
  uint64_t               launches               = 0;
};

namespace
{
  bool capturing(cudaStream_t st)
  {
    cudaStreamCaptureStatus s = cudaStreamCaptureStatusNone;
    return cudaStreamIsCapturing(st, &s) == cudaSuccess && s != cudaStreamCaptureStatusNone;
  }

  // RAII: count a launch, and time it with events when profiling is on.  While the stream is
  // being captured into a graph the launch is counted but not timed (no events inside a graph).
  struct Timed
  {
    bp4_ctx *c;
    int      id;
    ProfEvent ev{};
    bool      on;
    Timed(bp4_ctx *c_, int id_, int n_launches = 1) : c(c_), id(id_), on(c_->profile && !capturing(c_->stream))
    {
      c->launches += n_launches;
      c->prof_cnt[id] += 1;
      if (on)
        {
          for (cudaEvent_t *e : {&ev.a, &ev.b})
            if (c->event_pool.empty())
              cudaEventCreate(e);
            else
              {
                *e = c->event_pool.back();
                c->event_pool.pop_back();
              }
          ev.id = id;
          cudaEventRecord(ev.a, c->stream);
        }
    }
    ~Timed()
    {
      if (on)
        {
          cudaEventRecord(ev.b, c->stream);
          c->events.push_back(ev);
        }
    }
  };

  int drain_events(bp4_ctx *c)
  {
    cudaError_t err = cudaSuccess;
    for (auto &ev : c->events) // every event pair is released, also after a failure
      {
        float ms = 0;
        if (err == cudaSuccess)
          err = cudaEventSynchronize(ev.b);
        if (err == cudaSuccess)
          err = cudaEventElapsedTime(&ms, ev.a, ev.b);
        if (err == cudaSuccess)
          c->prof_ms[ev.id] += ms;
        c->event_pool.push_back(ev.a);
        c->event_pool.push_back(ev.b);
      }
    c->events.clear();
    CU(err);
    return 0;
  }

  // buffer of n doubles, from the pool when one of that size is cached; zeroed on request only
  // (SolverCGFullMerge takes its temporaries with omit_zeroing_entries = true,
  // solver_cg_optimized.h:215-217)
  int pooled_alloc(bp4_ctx *c, uint64_t n, double **out, bool zero)
  {
    auto it = c->pool.find(n);
    if (it != c->pool.end())
      {
        *out = it->second;
        c->pool.erase(it);
      }
    else
      CU(cudaMalloc(out, sizeof(double) * (n + 2))); // + 2: the fused loop copies runs in 16-byte pieces, one element past either end
    if (zero)
      CU(cudaMemsetAsync(*out, 0, sizeof(double) * n, c->stream));
    return 0;
  }

  // n rows of `width` elements to the device, in the caller's order or, with `order`, row order[j]
  // as row j
  template <typename T>
  cudaError_t upload_rows(T *dst, const T *src, size_t width, uint64_t n, const std::vector<uint64_t> &order)
  {
    if (order.empty())
      return cudaMemcpy(dst, src, sizeof(T) * width * n, cudaMemcpyHostToDevice);
    std::vector<T> tmp(width * n);
    for (uint64_t j = 0; j < n; ++j)
      std::copy(src + width * order[j], src + width * (order[j] + 1), tmp.data() + width * j);
    return cudaMemcpy(dst, tmp.data(), sizeof(T) * tmp.size(), cudaMemcpyHostToDevice);
  }

  // sum of acc[0..k) over ranks, returned on the host
  int reduce_to_host(bp4_ctx *c, int k, double *out)
  {
    if (c->comm)
      NC(ncclAllReduce(c->d_acc, c->d_acc, k, ncclDouble, ncclSum, c->comm, c->stream));
    // the last kernel of the chain writes the values and then a sequence number into mapped
    // pinned memory; the host polls that word (and the stream, for errors, now and then)
    volatile unsigned long long *seq_word = reinterpret_cast<volatile unsigned long long *>(c->h_acc + 8);
    const unsigned long long     seq      = ++c->pub_seq;
    CU(bp4::launch_publish(c->d_acc, k, c->h_acc, const_cast<unsigned long long *>(seq_word), seq, c->stream));
    c->launches += 1;
    int idle = 0;
    for (unsigned long long spins = 1; *seq_word != seq; ++spins)
      if ((spins & 0xFFFF) == 0)
        {
          const cudaError_t q = cudaStreamQuery(c->stream);
          if (q != cudaSuccess && q != cudaErrorNotReady)
            CU(q);
          if (q == cudaSuccess && ++idle > 8) // stream drained, nothing published: cannot happen
            return fail(BP4_ERR_CUDA, "reduction result was not published");
        }
    for (int i = 0; i < k; ++i)
      out[i] = c->h_acc[i];
    return 0;
  }
} // namespace

extern "C" {
static void p2p_teardown(bp4_ctx *c);

const char *bp4_last_error(void) { return g_err.c_str(); }

int bp4_device_count(int *count)
{
  if (!count)
    return fail(BP4_ERR_ARG, "count is null");
  CU(cudaGetDeviceCount(count));
  return 0;
}

// cut the cell-batch ranges of one cell partition [pc0, pc1) into units (a few whole ranges,
// about `target` cells) and the units into batches of cpb cells; see BatchDesc
static void build_units(const std::vector<uint32_t> &range_cell, const std::vector<uint32_t> &range_priv,
                        size_t r0, size_t r1, uint32_t cpb, uint32_t target,
                        std::vector<bp4::BatchDesc> &batches, std::vector<uint32_t> &unit_batch)
{
  size_t r = r0;
  while (r < r1)
    {
      size_t re = r + 1;
      while (re < r1 && range_cell[re] - range_cell[r] < target)
        ++re;
      if (range_cell[r1] - range_cell[re] < target / 2) // a short remainder joins the last unit
        re = r1;
      unit_batch.push_back((uint32_t)batches.size());
      const uint32_t uc0 = range_cell[r], uc1 = range_cell[re];
      for (uint32_t cb = uc0; cb < uc1; cb += cpb)
        {
          const uint32_t  ce = std::min(cb + cpb, uc1);
          bp4::BatchDesc b{};
          b.cell0   = cb;
          b.n_cells = ce - cb;
          // ranges whose first cell lies in [cb, ce): pre; whose end lies in (cb, ce]: post
          size_t f0 = r, f1, l0, l1;
          while (f0 < re && range_cell[f0] < cb)
            ++f0;
          f1 = f0;
          while (f1 < re && range_cell[f1] < ce)
            ++f1;
          l0 = r;
          while (l0 < re && range_cell[l0 + 1] <= cb)
            ++l0;
          l1 = l0;
          while (l1 < re && range_cell[l1 + 1] <= ce)
            ++l1;
          b.pre_begin  = range_priv[f0];
          b.pre_end    = range_priv[f1];
          b.post_begin = range_priv[l0];
          b.post_end   = range_priv[l1];
          batches.push_back(b);
        }
      r = re;
    }
}

static uint32_t gcd_u32(uint32_t a, uint32_t b) { return b ? gcd_u32(b, a % b) : a; }

static int ctx_create_impl(const bp4_desc *d, bp4_ctx *c)
{
  c->degree  = d->degree;
  c->device  = d->device;
  c->n_cells = d->n_cells;
  c->n_owned = d->n_owned;
  c->n_ghost = d->n_ghost;
  c->n_constrained = d->n_constrained;
  c->n_before      = d->n_cells_before_comm;
  c->n_comm        = d->n_cells_comm;
  if (c->n_before + c->n_comm > c->n_cells)
    return fail(BP4_ERR_ARG, "cell partitions exceed n_cells");
  CU(cudaDeviceGetAttribute(&c->sms, cudaDevAttrMultiProcessorCount, d->device));
  CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&c->comm_stream, cudaStreamNonBlocking));
  CU(cudaEventCreateWithFlags(&c->ev_a, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&c->ev_b, cudaEventDisableTiming));

  std::vector<uint32_t> walk;
  CU(bp4::launch_init_degree(d->degree, walk));
  CU(cudaMalloc(&c->d_walk, sizeof(uint32_t) * walk.size()));
  CU(cudaMemcpy(c->d_walk, walk.data(), sizeof(uint32_t) * walk.size(), cudaMemcpyHostToDevice));

  // deterministic mode: colour the cells greedily in the given order -- a cell takes the lowest
  // colour that no earlier cell sharing one of its valid entities has -- and store them colour by
  // colour.  Within a colour no two cells touch the same DoF, so a launch per colour adds at most
  // once to every address.  One 64-bit colour mask per entity, keyed by its first DoF / 3.
  std::vector<uint64_t> order; // stored cell j = the caller's cell order[j]
  if (c->deterministic && d->n_cells)
    {
      const uint64_t        n_local = d->n_owned + d->n_ghost;
      std::vector<uint64_t> mask(n_local / 3, 0);
      c->cell_color.resize(d->n_cells);
      for (uint64_t i = 0; i < d->n_cells; ++i)
        {
          const uint32_t *e    = d->entity_index + 27 * i;
          uint64_t        used = 0;
          for (int a = 0; a < 27; ++a)
            if (e[a] != BP4_INVALID_INDEX)
              {
                if (e[a] >= n_local)
                  return fail(BP4_ERR_ARG, "entity_index[%llu][%d] = %u is not a local DoF", (unsigned long long)i,
                              a, e[a]);
                used |= mask[e[a] / 3];
              }
          if (~used == 0)
            return fail(BP4_ERR_ARG, "deterministic mode: cell %llu needs more than 64 colours",
                        (unsigned long long)i);
          const uint32_t col = (uint32_t)__builtin_ctzll(~used);
          for (int a = 0; a < 27; ++a)
            if (e[a] != BP4_INVALID_INDEX)
              mask[e[a] / 3] |= 1ull << col;
          c->cell_color[i] = col;
          c->n_colors      = std::max(c->n_colors, col + 1);
        }
      c->color_off.assign(c->n_colors + 1, 0);
      for (uint32_t col : c->cell_color)
        ++c->color_off[col + 1];
      for (uint32_t k = 0; k < c->n_colors; ++k)
        c->color_off[k + 1] += c->color_off[k];
      std::vector<uint64_t> next(c->color_off.begin(), c->color_off.end() - 1);
      order.resize(d->n_cells);
      for (uint64_t i = 0; i < d->n_cells; ++i)
        order[next[c->cell_color[i]]++] = i;
      c->n_sched = std::max<uint32_t>(c->n_sched, c->n_colors);
    }

  const size_t nc = d->n_cells ? d->n_cells : 1;
  c->n_coef       = d->coefficients ? 81 : 24;
  CU(cudaMalloc(&c->d_entity, sizeof(uint32_t) * 27 * nc));
  CU(cudaMalloc(&c->d_coef, sizeof(double) * c->n_coef * nc));
  if (d->n_cells)
    CU(upload_rows(c->d_entity, d->entity_index, 27, d->n_cells, order));
  if (d->n_cells && d->coefficients) // all 27 coefficient vectors of the reference's kernel, as given
    CU(upload_rows(c->d_coef, d->coefficients, 81, d->n_cells, order));
  else if (d->n_cells)
    {
      // tri-linear coefficients from the 8 vertices, poisson_operator.h:161-178
      std::vector<double> cf(24 * d->n_cells);
      for (uint64_t i = 0; i < d->n_cells; ++i)
        for (int k = 0; k < 3; ++k)
          {
            const double *v = d->vertices + 24 * i;
            double       *o = cf.data() + 24 * i;
            const double  v0 = v[0 + k], v1 = v[3 + k], v2 = v[6 + k], v3 = v[9 + k], v4 = v[12 + k],
                         v5 = v[15 + k], v6 = v[18 + k], v7 = v[21 + k];
            o[0 + k]  = v0;
            o[3 + k]  = v1 - v0;
            o[6 + k]  = v2 - v0;
            o[9 + k]  = v3 - v2 - (v1 - v0);
            o[12 + k] = v4 - v0;
            o[15 + k] = v5 - v4 - (v1 - v0);
            o[18 + k] = v6 - v4 - (v2 - v0);
            o[21 + k] = (v7 - v6 - (v5 - v4) - (v3 - v2 - (v1 - v0)));
          }
      CU(upload_rows(c->d_coef, cf.data(), 24, d->n_cells, order));
    }
  CU(cudaMalloc(&c->d_constrained, sizeof(uint32_t) * (d->n_constrained ? d->n_constrained : 1)));
  if (d->n_constrained)
    CU(cudaMemcpy(c->d_constrained, d->constrained, sizeof(uint32_t) * d->n_constrained,
                  cudaMemcpyHostToDevice));
  std::vector<double> gll;
  bp4::gll_table(d->degree, gll);
  CU(cudaMalloc(&c->d_gll, sizeof(double) * gll.size()));
  CU(cudaMemcpy(c->d_gll, gll.data(), sizeof(double) * gll.size(), cudaMemcpyHostToDevice));
  CU(cudaMalloc(&c->d_acc, sizeof(double) * 8));
  CU(cudaMemset(c->d_acc, 0, sizeof(double) * 8));
  CU(cudaMalloc(&c->d_flag, sizeof(int)));
  CU(cudaMalloc(&c->d_sched, sizeof(uint32_t) * c->n_sched));
  if (c->deterministic)
    {
      const size_t n_slot = (size_t)8 * 8 * c->sms; // K <= 7 partials of <= 8 * SMs blocks (stream_grid)
      CU(cudaMalloc(&c->det.slot, sizeof(double) * n_slot));
      CU(cudaMalloc(&c->det.ticket, sizeof(uint32_t)));
      CU(cudaMemset(c->det.ticket, 0, sizeof(uint32_t)));
    }
  CU(cudaMallocHost(&c->h_acc, sizeof(double) * 16)); // UVA: the pointer is valid on the device too
  memset(c->h_acc, 0, sizeof(double) * 16);
  CU(cudaMallocHost(&c->h_flag, sizeof(int)));
  CU(cudaMalloc(&c->d_state, sizeof(bp4::SolveState)));
  CU(cudaMallocHost(&c->h_state, 2 * sizeof(bp4::SolveState)));

  // cell-batch ranges and their private DoF runs -> units and batches of the fused merged loop
  if (d->n_ranges > 0)
    {
      if (!d->range_cell_offset || !d->range_private_offset)
        return fail(BP4_ERR_ARG, "range tables missing");
      std::vector<uint32_t> rc(d->n_ranges + 1), rp(d->n_ranges + 1);
      for (uint64_t r = 0; r <= d->n_ranges; ++r)
        {
          rc[r] = (uint32_t)d->range_cell_offset[r];
          rp[r] = (uint32_t)d->range_private_offset[r];
          if (r && (rc[r] <= rc[r - 1] || rp[r] < rp[r - 1]))
            return fail(BP4_ERR_ARG, "range tables must be increasing (range %llu)", (unsigned long long)r);
          if (rp[r] % 3)
            return fail(BP4_ERR_ARG, "private DoF runs must start at a node (multiple of 3)");
        }
      if (rc[0] != 0 || rc[d->n_ranges] != d->n_cells || rp[0] != 0 || rp[d->n_ranges] > d->n_owned)
        return fail(BP4_ERR_ARG, "range tables do not cover [0, n_cells) / exceed n_owned");
      // the three cell partitions of the overlapped exchange must fall on range boundaries
      const uint64_t cut[4] = {0, c->n_before, c->n_before + c->n_comm, c->n_cells};
      size_t         rcut[4];
      for (int k = 0; k < 4; ++k)
        {
          rcut[k] = std::lower_bound(rc.begin(), rc.end(), (uint32_t)cut[k]) - rc.begin();
          if (rc[rcut[k]] != cut[k])
            return fail(BP4_ERR_ARG, "a cell-batch range straddles a cell partition boundary");
        }
      bp4::FusedLoopCfg fl;
      CU(bp4::fused_loop_config(d->degree, fl));
      const uint32_t rsz = rc[1] - rc[0];
      uint32_t       target = fl.cpb / gcd_u32(fl.cpb, rsz) * rsz; // lcm: whole ranges in whole batches
      while (target > 64 && target > rsz)
        target -= rsz;
      std::vector<bp4::BatchDesc> batches;
      std::vector<uint32_t>       unit_batch;
      for (int k = 0; k < 3; ++k)
        {
          c->unit_part[k] = (uint32_t)unit_batch.size();
          build_units(rc, rp, rcut[k], rcut[k + 1], fl.cpb, target, batches, unit_batch);
        }
      c->unit_part[3] = (uint32_t)unit_batch.size();
      unit_batch.push_back((uint32_t)batches.size());
      CU(cudaMalloc(&c->d_batch, sizeof(bp4::BatchDesc) * (batches.size() ? batches.size() : 1)));
      CU(cudaMalloc(&c->d_unit_batch, sizeof(uint32_t) * unit_batch.size()));
      CU(cudaMemcpy(c->d_batch, batches.data(), sizeof(bp4::BatchDesc) * batches.size(), cudaMemcpyHostToDevice));
      CU(cudaMemcpy(c->d_unit_batch, unit_batch.data(), sizeof(uint32_t) * unit_batch.size(),
                    cudaMemcpyHostToDevice));
      c->n_private = c->n_coef == 24 ? rp[d->n_ranges] : 0; // in-loop updates: tri-linear kernel only
      // the staged fused loop takes a batch's private run in two jobs of its shared-memory rows
      for (const bp4::BatchDesc &b : batches) // run_limit 0: no fused kernel at this degree
        if (b.pre_end - b.pre_begin > fl.run_limit || b.post_end - b.post_begin > fl.run_limit)
          c->n_private = 0; // the updates of every DoF are streamed then
      c->fused     = fl.is_default && c->n_private > 0;
      if (const char *e = getenv("BP4_FUSED")) // developer knob: 0 = pre kernel + cells + post kernel
        {
          c->fused        = c->n_private > 0 && atoi(e) != 0;
          c->fused_pinned = true;
        }
    }
  if (c->deterministic) // the in-loop sums are per-block atomics, and ranges do not survive colouring
    c->fused = 0, c->n_private = 0;

  // ghost exchange plan
  if (d->n_peers > 0)
    {
      c->peer.assign(d->peer_rank, d->peer_rank + d->n_peers);
      c->import_off.assign(d->import_offset, d->import_offset + d->n_peers + 1);
      c->export_off.assign(d->export_offset, d->export_offset + d->n_peers + 1);
      const uint64_t ne = c->export_off.back();
      CU(cudaMalloc(&c->d_export, sizeof(uint32_t) * (ne ? ne : 1)));
      if (ne)
        CU(cudaMemcpy(c->d_export, d->export_index, sizeof(uint32_t) * ne, cudaMemcpyHostToDevice));
      CU(cudaMalloc(&c->d_sendbuf, sizeof(double) * (ne ? ne : 1)));
      CU(cudaMalloc(&c->d_recvbuf, sizeof(double) * (ne ? ne : 1)));
    }
  return 0;
}

int bp4_ctx_create(const bp4_desc *d, bp4_ctx **out)
{
  if (!d || !out)
    return fail(BP4_ERR_ARG, "null argument");
  if (d->degree < 2 || d->degree > 8)
    return fail(BP4_ERR_ARG, "degree %d not supported (2..8)", d->degree);
  if (d->n_owned % 3 || d->n_ghost % 3)
    return fail(BP4_ERR_ARG, "n_owned/n_ghost must be multiples of 3");
  if (d->n_owned + d->n_ghost >= 0xFFFFFFFFull)
    return fail(BP4_ERR_ARG, "local vector exceeds 32-bit local indices (poisson_operator.h:693)");
  if (d->n_cells && (!d->entity_index || (!d->vertices && !d->coefficients)))
    return fail(BP4_ERR_ARG, "entity_index/vertices missing");
  const char *det_env       = getenv("BP4_DETERMINISTIC");
  const bool  deterministic = d->deterministic != 0 || (det_env && atoi(det_env) != 0);
  if (deterministic && d->n_peers > 0)
    return fail(BP4_ERR_ARG, "the deterministic mode runs on one rank: the descriptor has a ghost-exchange plan");
  int ndev = 0;
  CU(cudaGetDeviceCount(&ndev));
  if (ndev == 0)
    return fail(BP4_ERR_CUDA, "no CUDA device: this library has no CPU fallback");
  CU(cudaSetDevice(d->device));
  bp4_ctx *c       = new bp4_ctx;
  c->deterministic = deterministic;
  if (int e = ctx_create_impl(d, c))
    {
      const std::string msg = g_err; // bp4_ctx_destroy must not clobber the message
      bp4_ctx_destroy(c);
      g_err = msg;
      return e;
    }
  *out = c;
  return 0;
}

int bp4_ctx_destroy(bp4_ctx *c)
{
  if (!c)
    return 0;
  cudaSetDevice(c->device);
  if (c->stream)
    cudaStreamSynchronize(c->stream);
  drain_events(c);
  for (cudaEvent_t e : c->event_pool)
    cudaEventDestroy(e);
  c->event_pool.clear();
  p2p_teardown(c);
  if (c->comm)
    ncclCommDestroy(c->comm);
  for (auto &kv : c->pool)
    cudaFree(kv.second);
  for (SolveGraph &sg : c->solves)
    {
      if (sg.exec)
        cudaGraphExecDestroy(sg.exec);
      if (sg.graph)
        cudaGraphDestroy(sg.graph);
      cudaFree(sg.g);
      cudaFree(sg.d);
      cudaFree(sg.h);
    }
  cudaFree(c->d_state);
  cudaFreeHost(c->h_state);
  cudaFree(c->d_entity);
  cudaFree(c->d_constrained);
  cudaFree(c->d_walk);
  cudaFree(c->d_coef);
  cudaFree(c->d_gll);
  cudaFree(c->d_acc);
  cudaFree(c->d_flag);
  cudaFree(c->d_sched);
  cudaFree(c->det.slot);
  cudaFree(c->det.ticket);
  cudaFree(c->d_batch);
  cudaFree(c->d_unit_batch);
  cudaFree(c->d_export);
  cudaFree(c->d_sendbuf);
  cudaFree(c->d_recvbuf);
  cudaFreeHost(c->h_acc);
  cudaFreeHost(c->h_flag);
  if (c->ev_a)
    cudaEventDestroy(c->ev_a);
  if (c->ev_b)
    cudaEventDestroy(c->ev_b);
  if (c->comm_stream)
    cudaStreamDestroy(c->comm_stream);
  if (c->stream)
    cudaStreamDestroy(c->stream);
  delete c;
  return 0;
}

int bp4_ctx_synchronize(bp4_ctx *c)
{
  if (!c)
    return fail(BP4_ERR_ARG, "null ctx");
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

int bp4_ctx_stream(bp4_ctx *c, void **stream)
{
  if (!c || !stream)
    return fail(BP4_ERR_ARG, "null argument");
  *stream = (void *)c->stream;
  return 0;
}

static int vec_alloc(bp4_ctx *c, uint64_t n, bp4_vec **out, bool zero)
{
  if (!c || !out)
    return fail(BP4_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  bp4_vec *v = new bp4_vec;
  v->n       = n;
  if (int e = pooled_alloc(c, n, &v->buf, zero))
    {
      delete v;
      return e;
    }
  *out = v;
  return 0;
}

int bp4_vec_alloc(bp4_ctx *c, uint64_t n, bp4_vec **out) { return vec_alloc(c, n, out, true); }
int bp4_vec_alloc_uninitialized(bp4_ctx *c, uint64_t n, bp4_vec **out) { return vec_alloc(c, n, out, false); }

int bp4_vec_free(bp4_ctx *c, bp4_vec *v)
{
  if (!v)
    return 0;
  if (v->buf)
    {
      if (c) // stream order makes reuse safe: the next user's work is queued behind ours
        c->pool.emplace(v->n, v->buf);
      else
        cudaFree(v->buf);
    }
  delete v;
  return 0;
}

int bp4_vec_size(const bp4_vec *v, uint64_t *n)
{
  if (!v || !n)
    return fail(BP4_ERR_ARG, "null argument");
  *n = v->n;
  return 0;
}

int bp4_vec_set_zero(bp4_ctx *c, bp4_vec *v)
{
  if (!c || !v)
    return fail(BP4_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  CU(cudaMemsetAsync(v->p(), 0, sizeof(double) * v->n, c->stream));
  return 0;
}

int bp4_vec_upload(bp4_ctx *c, bp4_vec *v, const double *host, uint64_t n)
{
  if (!c || !v || (!host && n))
    return fail(BP4_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  if (n > v->n)
    return fail(BP4_ERR_ARG, "upload of %llu > vector size %llu", (unsigned long long)n,
                (unsigned long long)v->n);
  CU(cudaMemcpyAsync(v->p(), host, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
  return 0;
}

int bp4_vec_download(bp4_ctx *c, const bp4_vec *v, double *host, uint64_t n)
{
  if (!c || !v || (!host && n))
    return fail(BP4_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  if (n > v->n)
    return fail(BP4_ERR_ARG, "download of %llu > vector size %llu", (unsigned long long)n,
                (unsigned long long)v->n);
  CU(cudaMemcpyAsync(host, v->p(), sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

int bp4_vec_device_ptr(bp4_ctx *c, bp4_vec *v, double **dev)
{
  if (!c || !v || !dev)
    return fail(BP4_ERR_ARG, "null argument");
  *dev = v->p();
  return 0;
}

static int check_len(const bp4_ctx *c, const bp4_vec *v, const char *name)
{
  if (!v)
    return fail(BP4_ERR_ARG, "%s is null", name);
  if (v->n < c->n_owned + c->n_ghost)
    return fail(BP4_ERR_ARG, "%s has %llu entries, need n_owned+n_ghost = %llu", name,
                (unsigned long long)v->n, (unsigned long long)(c->n_owned + c->n_ghost));
  return 0;
}

// BLAS-1 operands must hold at least the owned entries
static int check_owned(const bp4_ctx *c, const bp4_vec *v, const char *name)
{
  if (!v)
    return fail(BP4_ERR_ARG, "%s is null", name);
  if (v->n < c->n_owned)
    return fail(BP4_ERR_ARG, "%s has %llu entries, need n_owned = %llu", name, (unsigned long long)v->n,
                (unsigned long long)c->n_owned);
  return 0;
}

// BLAS-1 sweeps the owned entries, or the whole operand when it is shorter (the per-node
// diagonal holds n_owned/3 entries: diag_mat.diagonal.l2_norm(), benchmark.h:151)
static uint64_t sweep_len(const bp4_ctx *c, std::initializer_list<const bp4_vec *> vs)
{
  uint64_t n = c->n_owned;
  for (const bp4_vec *v : vs)
    n = std::min<uint64_t>(n, v->n);
  return n;
}

// scalars and vectors of one vmult_with_merged_sums call, for the fused cell loop
struct MergedCall
{
  double *x, *g, *d;
  const double *prec;
  double  alpha, beta, alpha_old, beta_old;
  const bp4::SolveState *state; // non-null: the scalars come from this solver state instead
};

// cell loop over the cell partition `part` (0..2, or -1 = all cells): dst += sum_cells A_cell src
// on the local vector; with `m` the private DoFs of the ranges get their do_cg_update4b/3b inside
static int cell_range(bp4_ctx *c, double *dst, const double *src, int part, const MergedCall *m)
{
  const uint64_t cut[4] = {0, c->n_before, c->n_before + c->n_comm, c->n_cells};
  const uint64_t begin = part < 0 ? 0 : cut[part], end = part < 0 ? c->n_cells : cut[part + 1];
  if (end <= begin)
    return 0;
  bp4::CellArgs a{};
  a.dtab  = c->d_walk;
  a.src   = src;
  a.dst   = dst;
  a.sched = c->d_sched + (part < 0 ? 0 : part);
  if (m)
    {
      const uint32_t u0 = part < 0 ? c->unit_part[0] : c->unit_part[part],
                     u1 = part < 0 ? c->unit_part[3] : c->unit_part[part + 1];
      a.entity_index = c->d_entity;
      a.coef         = c->d_coef;
      a.n_cells      = c->n_cells;
      a.batch        = c->d_batch;
      a.unit_batch   = c->d_unit_batch + u0;
      a.n_units      = u1 - u0;
      a.r            = m->g;
      a.p            = m->d;
      a.x            = m->x;
      a.prec         = m->prec;
      a.alpha        = m->alpha;
      a.beta         = m->beta;
      a.first        = m->alpha == 0. ? 1 : 0;
      a.update_x     = (m->alpha != 0. && m->alpha_old != 0.) ? 1 : 0;
      a.c1           = a.update_x ? m->alpha + m->alpha_old / m->beta_old : 0.;
      a.c2           = a.update_x ? m->alpha_old / m->beta_old : 0.;
      a.acc          = c->d_acc;
      a.state        = m->state;
      Timed t(c, BP4_K_MERGED);
      CU(bp4::launch_cell(c->degree, true, false, a, c->sms, c->stream));
    }
  else if (c->deterministic) // one launch per colour (single rank: part = -1), timed as one loop
    {
      Timed t(c, BP4_K_VMULT, (int)c->n_colors);
      for (uint32_t k = 0; k < c->n_colors; ++k)
        {
          const uint64_t c0 = c->color_off[k];
          a.entity_index    = c->d_entity + 27 * c0;
          a.coef            = c->d_coef + (uint64_t)c->n_coef * c0;
          a.n_cells         = c->color_off[k + 1] - c0;
          a.sched           = c->d_sched + k;
          CU(bp4::launch_cell(c->degree, false, c->n_coef == 81, a, c->sms, c->stream));
        }
    }
  else
    {
      a.entity_index = c->d_entity + 27 * begin;
      a.coef         = c->d_coef + (uint64_t)c->n_coef * begin;
      a.n_cells      = end - begin;
      Timed t(c, BP4_K_VMULT);
      CU(bp4::launch_cell(c->degree, false, c->n_coef == 81, a, c->sms, c->stream));
    }
  return 0;
}

static int exchange_ghosts_on(bp4_ctx *c, double *v, cudaStream_t st);
static int exchange_compress_on(bp4_ctx *c, double *v, cudaStream_t st);
static const double *contrib_buffer(const bp4_ctx *c);
static int compress_release(bp4_ctx *c, cudaStream_t st);


// MatrixFree::cell_loop (poisson_operator.h:310, :339) on one rank: update_ghost_values(src),
// cells, compress(add)(dst).  With a partitioned mesh the two exchanges run on a second stream
// while the cells that touch no ghost DoF are processed (SURVEY App. B1):
//   pack | interior part 1 || send/recv ghosts | ghost-touching cells | interior part 2 ||
//   send/recv contributions | unpack-add.
// dst must already be zero where the cells accumulate (owned and ghost slots).
static int cell_loop(bp4_ctx *c, double *dst, const double *src, const MergedCall *m)
{
  CU(cudaMemsetAsync(c->d_sched, 0, sizeof(uint32_t) * c->n_sched, c->stream));
  if (c->peer.empty())
    return cell_range(c, dst, src, -1, m);
  if (!c->comm)
    return fail(BP4_ERR_STATE, "ghost exchange not initialised (bp4_comm_init)");
  const uint64_t ne      = c->export_off.back();
  const bool     overlap = c->overlap && c->n_comm > 0;
  {
    Timed t(c, BP4_K_BLAS1);
    CU(bp4::launch_pack(ne, c->d_export, src, c->d_sendbuf, c->stream));
  }
  CU(cudaEventRecord(c->ev_a, c->stream));
  CU(cudaStreamWaitEvent(c->comm_stream, c->ev_a, 0));
  if (int e = exchange_ghosts_on(c, const_cast<double *>(src), c->comm_stream))
    return e;
  CU(cudaEventRecord(c->ev_b, c->comm_stream));
  if (overlap)
    if (int e = cell_range(c, dst, src, 0, m))
      return e;
  CU(cudaStreamWaitEvent(c->stream, c->ev_b, 0));
  if (overlap)
    {
      if (int e = cell_range(c, dst, src, 1, m))
        return e;
    }
  else if (int e = cell_range(c, dst, src, -1, m))
    return e;
  CU(cudaEventRecord(c->ev_a, c->stream));
  CU(cudaStreamWaitEvent(c->comm_stream, c->ev_a, 0));
  if (int e = exchange_compress_on(c, dst, c->comm_stream))
    return e;
  CU(cudaEventRecord(c->ev_b, c->comm_stream));
  if (overlap)
    if (int e = cell_range(c, dst, src, 2, m))
      return e;
  CU(cudaStreamWaitEvent(c->stream, c->ev_b, 0));
  {
    Timed t(c, BP4_K_BLAS1); // one launch for all peers: an owned entry may be exported to several (atomics)
    CU(bp4::launch_unpack_add(c->export_off.back(), c->d_export, contrib_buffer(c), dst, c->stream));
  }
  if (int e = compress_release(c, c->stream))
    return e;
  CU(cudaMemsetAsync(dst + c->n_owned, 0, sizeof(double) * c->n_ghost, c->stream));
  return 0;
}

// dst = A src on the context's stream (also captured into the plain device solve's loop body)
static int vmult_on(bp4_ctx *c, double *dst, const double *src)
{
  CU(cudaMemsetAsync(dst, 0, sizeof(double) * (c->n_owned + c->n_ghost), c->stream));
  if (int e = cell_loop(c, dst, src, nullptr))
    return e;
  Timed t(c, BP4_K_BLAS1);
  CU(bp4::launch_fixup(c->n_constrained, c->d_constrained, dst, src, c->stream));
  return 0;
}

int bp4_vmult(bp4_ctx *c, bp4_vec *dst, const bp4_vec *src)
{
  if (!c)
    return fail(BP4_ERR_ARG, "null ctx");
  if (int e = check_len(c, dst, "dst"))
    return e;
  if (int e = check_len(c, src, "src"))
    return e;
  if (dst == src)
    return fail(BP4_ERR_ARG, "vmult: dst aliases src");
  CU(cudaSetDevice(c->device));
  return vmult_on(c, dst->p(), src->p());
}

int bp4_debug_set_fused(bp4_ctx *c, int on)
{
  if (!c)
    return fail(BP4_ERR_ARG, "null ctx");
  if (on && c->deterministic)
    return fail(BP4_ERR_STATE, "the deterministic mode runs the streamed form only (the in-loop sums are "
                               "per-block atomics)");
  if (on && c->n_private == 0)
    return fail(BP4_ERR_STATE, "no private DoF runs: the context was created without range tables, with "
                               "quadratic geometry, at a degree without a fused kernel (> 4), or with runs "
                               "too long for its staging rows");
  c->fused        = on != 0;
  c->fused_pinned = true;
  return 0;
}

int bp4_fused_info(bp4_ctx *c, int *fused, uint64_t *n_private, uint64_t *n_units)
{
  if (!c)
    return fail(BP4_ERR_ARG, "null ctx");
  if (fused)
    *fused = c->fused;
  if (n_private)
    *n_private = c->n_private;
  if (n_units)
    *n_units = c->unit_part[3];
  return 0;
}

// vmult_with_merged_sums on the context's stream, the seven sums left in d_acc (also captured into
// the merged device solve's loop body, with the scalars from m.state)
static int merged_sweep(bp4_ctx *c, const MergedCall &m, double *h)
{
  const uint64_t n = c->n_owned;
  // DoFs private to one cell-batch range get do_cg_update4b / do_cg_update3b inside the cell
  // kernel; the rest of the vector -- shared between ranges or ranks, Dirichlet -- is streamed
  // before / after the loop (with the fused path off: everything)
  const uint64_t tail = c->fused ? c->n_private : 0;
  {
    Timed t(c, BP4_K_PRE);
    if (m.state)
      CU(bp4::launch_pre_dev(tail, n, h, m.x, m.g, m.d, m.prec, m.state, c->d_acc, c->sms, c->stream));
    else
      CU(bp4::launch_pre(tail, n, h, m.x, m.g, m.d, m.prec, m.alpha, m.beta, m.alpha_old, m.beta_old, c->d_acc,
                         c->sms, c->stream));
  }
  if (c->n_ghost)
    CU(cudaMemsetAsync(h + n, 0, sizeof(double) * c->n_ghost, c->stream));
  if (int e = cell_loop(c, h, m.d, c->fused ? &m : nullptr))
    return e;
  if (n > tail)
    {
      Timed t(c, BP4_K_POST);
      CU(bp4::launch_post(tail, n, m.g, m.d, h, m.prec, c->d_acc, c->det, c->sms, c->stream));
    }
  return 0;
}

int bp4_vmult_merged(bp4_ctx *c, bp4_vec *x, bp4_vec *g, bp4_vec *d, bp4_vec *h, const bp4_vec *prec,
                     double alpha, double beta, double alpha_old, double beta_old, double out[7])
{
  if (!c || !out)
    return fail(BP4_ERR_ARG, "null argument");
  for (auto pr : {std::make_pair((const bp4_vec *)x, "x"), std::make_pair((const bp4_vec *)g, "g"),
                  std::make_pair((const bp4_vec *)d, "d"), std::make_pair((const bp4_vec *)h, "h")})
    if (int e = check_len(c, pr.first, pr.second))
      return e;
  if (!prec || prec->n < c->n_owned / 3)
    return fail(BP4_ERR_ARG, "prec needs n_owned/3 entries");
  CU(cudaSetDevice(c->device));
  MergedCall m{x->p(), g->p(), d->p(), prec->p(), alpha, beta, alpha_old, beta_old, nullptr};
  if (int e = merged_sweep(c, m, h->p()))
    return e;
  return reduce_to_host(c, 7, out);
}

// the scalar GLL diagonal added into diag[3 * node]: one launch, or one per colour in the
// deterministic mode (every entry then gets at most one atomic add per launch); the launch count
// of the record includes the `more` launches of the caller that follow
static int assemble_diagonal(bp4_ctx *c, double *diag, int more)
{
  const uint32_t n_groups = c->deterministic ? c->n_colors : 1;
  Timed          t(c, BP4_K_BLAS1, (int)n_groups + more);
  for (uint32_t k = 0; k < n_groups; ++k)
    {
      const uint64_t c0 = c->deterministic ? c->color_off[k] : 0,
                     c1 = c->deterministic ? c->color_off[k + 1] : c->n_cells;
      CU(bp4::launch_diag_assemble(c->degree, c1 - c0, c->d_entity + 27 * c0, c->d_coef + (uint64_t)c->n_coef * c0,
                                   c->n_coef, c->d_gll, diag, 3, c->stream));
    }
  return 0;
}

int bp4_inverse_diagonal(bp4_ctx *c, bp4_vec *out)
{
  if (!c || !out)
    return fail(BP4_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  if (out->n < c->n_owned / 3)
    return fail(BP4_ERR_ARG, "diagonal vector needs n_owned/3 entries");
  // assemble DoF-wise into slot 3*node of a local vector so that the ordinary ghost
  // compress(add) (poisson_operator.h:419) can be reused, then keep one entry per owned node
  bp4_vec *tmp = nullptr;
  if (int e = bp4_vec_alloc(c, c->n_owned + c->n_ghost, &tmp))
    return e;
  if (int e = assemble_diagonal(c, tmp->p(), 2))
    return e;
  if (!c->peer.empty())
    if (int e = bp4_compress_add(c, tmp))
      return e;
  CU(bp4::launch_stride3(c->n_owned / 3, tmp->p(), out->p(), c->stream));
  CU(bp4::launch_diag_invert(c->n_owned / 3, out->p(), c->stream));
  return bp4_vec_free(c, tmp);
}

// the reference's own layout of the result (poisson_operator.h:392-426): a DoF vector whose
// component-0 entries hold 1/diag of the scalar operator and every other entry is 1 (0 -> 1)
int bp4_inverse_diagonal_vector(bp4_ctx *c, bp4_vec *out)
{
  if (!c)
    return fail(BP4_ERR_ARG, "null ctx");
  if (int e = check_len(c, out, "out"))
    return e;
  CU(cudaSetDevice(c->device));
  CU(cudaMemsetAsync(out->p(), 0, sizeof(double) * (c->n_owned + c->n_ghost), c->stream));
  if (int e = assemble_diagonal(c, out->p(), 1))
    return e;
  if (!c->peer.empty())
    if (int e = bp4_compress_add(c, out))
      return e;
  CU(bp4::launch_diag_invert(c->n_owned, out->p(), c->stream));
  return 0;
}

// dst[i] = src[n_components * i + component]: the extraction loop of benchmark.h:141-147
int bp4_extract_component(bp4_ctx *c, bp4_vec *dst, const bp4_vec *src, int n_components, int component)
{
  if (!c || !dst || !src)
    return fail(BP4_ERR_ARG, "null argument");
  if (n_components != 3 || component < 0 || component > 2)
    return fail(BP4_ERR_ARG, "three components per node");
  if (src->n < c->n_owned || dst->n < c->n_owned / 3)
    return fail(BP4_ERR_ARG, "Dimension mismatch %llu vs 3 x %llu", (unsigned long long)src->n,
                (unsigned long long)dst->n);
  CU(cudaSetDevice(c->device));
  Timed t(c, BP4_K_BLAS1);
  CU(bp4::launch_stride3(c->n_owned / 3, src->p() + component, dst->p(), c->stream));
  return 0;
}

int bp4_jacobi_vmult(bp4_ctx *c, bp4_vec *dst, const bp4_vec *src, const bp4_vec *diag)
{
  if (!c || !dst || !src || !diag)
    return fail(BP4_ERR_ARG, "null argument");
  if (dst->n < c->n_owned || src->n < c->n_owned || 3 * diag->n < c->n_owned)
    return fail(BP4_ERR_ARG, "Dimension mismatch %llu vs 3 x %llu", (unsigned long long)dst->n,
                (unsigned long long)diag->n);
  CU(cudaSetDevice(c->device));
  Timed t(c, BP4_K_BLAS1);
  CU(bp4::launch_jacobi(c->n_owned, dst->p(), src->p(), diag->p(), c->sms, c->stream));
  return 0;
}

int bp4_x_finalize_even(bp4_ctx *c, bp4_vec *x, const bp4_vec *d, const bp4_vec *g, const bp4_vec *prec,
                        double c1, double c2)
{
  if (!c || !x || !d || !g || !prec)
    return fail(BP4_ERR_ARG, "null argument");
  if (int e = check_owned(c, x, "x"))
    return e;
  if (int e = check_owned(c, d, "d"))
    return e;
  if (int e = check_owned(c, g, "g"))
    return e;
  if (3 * prec->n < c->n_owned)
    return fail(BP4_ERR_ARG, "prec needs n_owned/3 entries");
  CU(cudaSetDevice(c->device));
  Timed t(c, BP4_K_BLAS1);
  CU(bp4::launch_xfinal(c->n_owned, x->p(), d->p(), g->p(), prec->p(), c1, c2, c->sms, c->stream));
  return 0;
}

int bp4_equ(bp4_ctx *c, bp4_vec *dst, double a, const bp4_vec *src)
{
  if (!c || !dst || !src)
    return fail(BP4_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  Timed t(c, BP4_K_BLAS1);
  CU(bp4::launch_sadd(sweep_len(c, {dst, src}), dst->p(), 0., a, src->p(), c->sms, c->stream));
  return 0;
}

int bp4_add(bp4_ctx *c, bp4_vec *dst, double a, const bp4_vec *src)
{
  if (!c || !dst || !src)
    return fail(BP4_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  Timed t(c, BP4_K_BLAS1);
  CU(bp4::launch_sadd(sweep_len(c, {dst, src}), dst->p(), 1., a, src->p(), c->sms, c->stream));
  return 0;
}

int bp4_sadd(bp4_ctx *c, bp4_vec *dst, double s, double a, const bp4_vec *src)
{
  if (!c || !dst || !src)
    return fail(BP4_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  Timed t(c, BP4_K_BLAS1);
  CU(bp4::launch_sadd(sweep_len(c, {dst, src}), dst->p(), s, a, src->p(), c->sms, c->stream));
  return 0;
}

int bp4_dot(bp4_ctx *c, const bp4_vec *a, const bp4_vec *b, double *result)
{
  if (!c || !a || !b || !result)
    return fail(BP4_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  {
    Timed t(c, BP4_K_BLAS1);
    CU(bp4::launch_dot(sweep_len(c, {a, b}), a->p(), b->p(), c->d_acc, c->det, c->sms, c->stream));
  }
  return reduce_to_host(c, 1, result);
}

int bp4_add_and_dot(bp4_ctx *c, bp4_vec *g, double a, const bp4_vec *h, const bp4_vec *w, double *result)
{
  if (!c || !g || !h || !w || !result)
    return fail(BP4_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  {
    Timed t(c, BP4_K_BLAS1);
    CU(bp4::launch_add_and_dot(sweep_len(c, {g, h, w}), g->p(), a, h->p(), w->p(), c->d_acc, c->det, c->sms,
                               c->stream));
  }
  return reduce_to_host(c, 1, result);
}

int bp4_l2_norm(bp4_ctx *c, const bp4_vec *v, double *result)
{
  double s = 0;
  if (int e = bp4_dot(c, v, v, &s))
    return e;
  *result = std::sqrt(s);
  return 0;
}

int bp4_all_zero(bp4_ctx *c, const bp4_vec *v, int *result)
{
  if (!c || !v || !result)
    return fail(BP4_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  CU(cudaMemsetAsync(c->d_flag, 0, sizeof(int), c->stream));
  {
    Timed t(c, BP4_K_BLAS1);
    CU(bp4::launch_nonzero(sweep_len(c, {v}), v->p(), c->d_flag, c->sms, c->stream));
  }
  if (c->comm)
    NC(ncclAllReduce(c->d_flag, c->d_flag, 1, ncclInt, ncclMax, c->comm, c->stream));
  CU(cudaMemcpyAsync(c->h_flag, c->d_flag, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  *result = *c->h_flag ? 0 : 1;
  return 0;
}

// ---- whole solves on the device ----------------------------------------------------------
// Capture what `launch` enqueues on the context's stream into `graph`, after the nodes `deps`;
// `leaves` (optional) receives the nodes the next one must follow.  The capture is always ended,
// also when a launch fails, so that the stream stays usable.
extern "C++" {
template <typename F>
static int capture_into(bp4_ctx *c, cudaGraph_t graph, const cudaGraphNode_t *deps, size_t n_deps, F &&launch,
                        std::vector<cudaGraphNode_t> *leaves)
{
  CU(cudaStreamBeginCaptureToGraph(c->stream, graph, deps, nullptr, n_deps, cudaStreamCaptureModeThreadLocal));
  int e = launch();
  if (!e && leaves)
    {
      cudaStreamCaptureStatus st;
      const cudaGraphNode_t  *d = nullptr;
      size_t                  n = 0;
      const cudaError_t       q = cudaStreamGetCaptureInfo(c->stream, &st, nullptr, nullptr, &d, &n);
      if (q == cudaSuccess)
        leaves->assign(d, d + n);
      else
        e = fail(BP4_ERR_CUDA, "cudaStreamGetCaptureInfo: %s", cudaGetErrorString(q));
    }
  cudaGraph_t       out = nullptr;
  const cudaError_t q   = cudaStreamEndCapture(c->stream, &out);
  if (e)
    return e;
  CU(q);
  return 0;
}
} // extern "C++"

// One CUDA graph per solve:  initial state -> prologue -> WHILE { one iteration } -> epilogue ->
// final state to the host.  The loop body is captured from the launch code of the host-driven
// path (vmult_on, merged_sweep); the scalar kernels keep alpha, beta, ... in c->d_state and the
// last one of an iteration sets the loop condition.
static int build_solve_graph(bp4_ctx *c, SolveGraph &sg)
{
  const uint64_t n    = c->n_owned;
  double        *x    = const_cast<double *>(sg.x);
  const double  *prec = sg.prec;
  bp4::SolveState *st = c->d_state;
  double        *acc  = c->d_acc;
  CU(cudaGraphCreate(&sg.graph, 0));
  cudaGraphConditionalHandle loop;
  CU(cudaGraphConditionalHandleCreate(&loop, sg.graph, 1, cudaGraphCondAssignDefault));
  std::vector<cudaGraphNode_t> leaves;
  // initial state; plain: h = P g, d = -h, gh = g.h (SolverCG before its loop)
  auto prologue = [&]() -> int {
    CU(cudaMemcpyAsync(st, c->h_state, sizeof(bp4::SolveState), cudaMemcpyHostToDevice, c->stream));
    if (sg.merged)
      return 0;
    {
      Timed t(c, BP4_K_BLAS1);
      CU(bp4::launch_jacobi_dot(n, sg.h, sg.g, prec, acc + 2, c->det, c->sms, c->stream));
    }
    {
      Timed t(c, BP4_K_BLAS1);
      CU(bp4::launch_solve_scalar(bp4::kSolvePlainInit, st, acc, loop, c->stream));
    }
    Timed t(c, BP4_K_BLAS1);
    CU(bp4::launch_sadd(n, sg.d, 0., -1., sg.h, c->sms, c->stream));
    return 0;
  };
  if (int e = capture_into(c, sg.graph, nullptr, 0, prologue, &leaves))
    return e;
  cudaGraphNodeParams cp = {};
  cp.type                = cudaGraphNodeTypeConditional;
  cp.conditional.handle  = loop;
  cp.conditional.type    = cudaGraphCondTypeWhile;
  cp.conditional.size    = 1;
  cudaGraphNode_t cond;
  CU(cudaGraphAddNode(&cond, sg.graph, leaves.data(), leaves.size(), &cp));
  auto body = [&]() -> int {
    if (sg.merged)
      {
        const MergedCall m{x, sg.g, sg.d, prec, 0., 0., 0., 0., st};
        if (int e = merged_sweep(c, m, sg.h))
          return e;
        Timed t(c, BP4_K_BLAS1);
        CU(bp4::launch_solve_scalar(bp4::kSolveMergedStep, st, acc, loop, c->stream));
        return 0;
      }
    // SolverCG: h = A d; alpha = gh / d.h; x += alpha d; g += alpha h, |g|; check;
    // h = P g; beta = g.h / gh; d = beta d - h
    if (int e = vmult_on(c, sg.h, sg.d))
      return e;
    {
      Timed t(c, BP4_K_BLAS1);
      CU(bp4::launch_dot(n, sg.d, sg.h, acc, c->det, c->sms, c->stream));
    }
    {
      Timed t(c, BP4_K_BLAS1);
      CU(bp4::launch_solve_scalar(bp4::kSolvePlainAlpha, st, acc, loop, c->stream));
    }
    {
      Timed t(c, BP4_K_BLAS1);
      CU(bp4::launch_cg_xg(n, x, sg.g, sg.d, sg.h, st, acc + 1, c->det, c->sms, c->stream));
    }
    {
      Timed t(c, BP4_K_BLAS1);
      CU(bp4::launch_jacobi_dot(n, sg.h, sg.g, prec, acc + 2, c->det, c->sms, c->stream));
    }
    {
      Timed t(c, BP4_K_BLAS1);
      CU(bp4::launch_solve_scalar(bp4::kSolvePlainCheck, st, acc, loop, c->stream));
    }
    Timed t(c, BP4_K_BLAS1);
    CU(bp4::launch_sadd_dev(n, sg.d, &st->beta, -1., sg.h, c->sms, c->stream));
    return 0;
  };
  if (int e = capture_into(c, cp.conditional.phGraph_out[0], nullptr, 0, body, nullptr))
    return e;
  // merged: the pending x update; both: the final state to the host
  auto epilogue = [&]() -> int {
    if (sg.merged)
      {
        Timed t(c, BP4_K_BLAS1);
        CU(bp4::launch_solve_final(n, x, sg.d, sg.g, prec, st, c->deterministic, c->sms, c->stream));
      }
    CU(cudaMemcpyAsync(c->h_state + 1, st, sizeof(bp4::SolveState), cudaMemcpyDeviceToHost, c->stream));
    return 0;
  };
  if (int e = capture_into(c, sg.graph, &cond, 1, epilogue, nullptr))
    return e;
  CU(cudaGraphInstantiate(&sg.exec, sg.graph, 0));
  return 0;
}

static int solve_device(bp4_ctx *c, const bool merged, bp4_vec *x, const bp4_vec *b, const bp4_vec *prec,
                        const unsigned max_steps, const double tol, const double reduce, bp4_solve_result *out)
{
  if (!c || !out)
    return fail(BP4_ERR_ARG, "null argument");
  if (int e = check_len(c, x, "x"))
    return e;
  if (int e = check_len(c, b, "b"))
    return e;
  if (!prec || 3 * prec->n < c->n_owned)
    return fail(BP4_ERR_ARG, "prec needs n_owned/3 entries");
  if (x == b)
    return fail(BP4_ERR_ARG, "solve: x aliases b");
  if (!c->peer.empty() || c->n_ranks > 1)
    return fail(BP4_ERR_STATE, "the device solve runs on one rank: this context has a ghost-exchange plan or "
                               "a communicator over several ranks");
  CU(cudaSetDevice(c->device));
  SolveGraph *sg = nullptr;
  for (SolveGraph &e : c->solves)
    if (e.merged == merged && e.fused == c->fused && e.x == x->p() && e.b == b->p() && e.prec == prec->p())
      sg = &e;
  if (!sg)
    {
      c->solves.emplace_back();
      sg         = &c->solves.back();
      sg->merged = merged, sg->fused = c->fused, sg->x = x->p(), sg->b = b->p(), sg->prec = prec->p();
      const uint64_t nl = c->n_owned + c->n_ghost;
      for (double **v : {&sg->g, &sg->d, &sg->h})
        if (int e = pooled_alloc(c, nl, v, false))
          return e;
    }
  // step 0 on the host, with the entry points the host-driven solvers use: g = A x - b (-b for a
  // zero start vector), |g|, ReductionControl::check(0)
  bp4_vec g{sg->g, c->n_owned + c->n_ghost};
  int     zero = 0;
  if (int e = bp4_all_zero(c, x, &zero))
    return e;
  if (!zero)
    {
      if (int e = bp4_vmult(c, &g, x))
        return e;
      if (int e = bp4_add(c, &g, -1., b))
        return e;
    }
  else if (int e = bp4_equ(c, &g, -1., b))
    return e;
  double res = 0.;
  if (int e = bp4_l2_norm(c, &g, &res))
    return e;
  const double reduced_tol = res * reduce;
  const int    state0      = (res < reduced_tol || res <= tol) ? 1 : ((max_steps == 0 || std::isnan(res)) ? 2 : 0);
  *out                     = bp4_solve_result{state0, 0u, res, res};
  if (state0 != 0)
    return 0;
  if (!sg->exec)
    if (int e = build_solve_graph(c, *sg))
      {
        if (sg->graph) // a later call starts over
          cudaGraphDestroy(sg->graph);
        sg->graph = nullptr;
        return e;
      }
  bp4::SolveState &init = c->h_state[0];
  init                  = bp4::SolveState{};
  init.tol              = tol;
  init.reduced_tol      = reduced_tol;
  init.last_value       = res;
  init.initial_value    = res;
  init.max_steps        = max_steps;
  CU(cudaGraphLaunch(sg->exec, c->stream));
  c->launches += 1;
  CU(cudaStreamSynchronize(c->stream));
  const bp4::SolveState &fin = c->h_state[1];
  *out                       = bp4_solve_result{fin.state, fin.step, fin.last_value, res};
  return 0;
}

int bp4_solve_cg(bp4_ctx *c, bp4_vec *x, const bp4_vec *b, const bp4_vec *prec, unsigned max_steps, double tol,
                 double reduce, bp4_solve_result *out)
{
  return solve_device(c, false, x, b, prec, max_steps, tol, reduce, out);
}

int bp4_solve_cg_merged(bp4_ctx *c, bp4_vec *x, const bp4_vec *b, const bp4_vec *prec, unsigned max_steps,
                        double tol, double reduce, bp4_solve_result *out)
{
  return solve_device(c, true, x, b, prec, max_steps, tol, reduce, out);
}

// ---- multi-GPU ---------------------------------------------------------------------------
int bp4_comm_unique_id(unsigned char id[BP4_NCCL_ID_BYTES])
{
  static_assert(sizeof(ncclUniqueId) == BP4_NCCL_ID_BYTES, "ncclUniqueId size");
  ncclUniqueId u;
  NC(ncclGetUniqueId(&u));
  memcpy(id, &u, sizeof(u));
  return 0;
}

// ---- peer exchange over NVLink without SMs -------------------------------------------------
namespace
{
  constexpr int kP2PMaxRanks = 16;
  struct P2PCard // what every rank publishes about its arena
  {
    cudaIpcMemHandle_t handle;
    uint64_t           off_ghost[2], off_contrib[2];
    int64_t            imp_off_for[kP2PMaxRanks]; // my import offset (doubles) for owner r, or -1
    int64_t            exp_off_for[kP2PMaxRanks]; // my export offset (doubles) for ghost holder r, or -1
  };
  enum
  {
    kFlagDataFwd = 0, // [r] owner r's ghost values of exchange e have landed in my ghost_in[e & 1]
    kFlagAckFwd  = 1, // [r] ghost holder r has copied exchange e out of its ghost_in
    kFlagDataRev = 2, // [r] ghost holder r's contributions of exchange e have landed in my contrib_in[e & 1]
    kFlagAckRev  = 3  // [r] owner r has added exchange e into its vector
  };
  inline CUdeviceptr flag_addr(char *arena, int kind, int rank)
  {
    return (CUdeviceptr)(arena + sizeof(uint64_t) * (size_t)(kind * kP2PMaxRanks + rank));
  }
} // namespace

#define DRV(call)                                                                              \
  do                                                                                          \
    {                                                                                         \
      CUresult r_ = (call);                                                                   \
      if (r_ != CUDA_SUCCESS)                                                                 \
        return fail(BP4_ERR_CUDA, "%s:%d %s: driver error %d", __FILE__, __LINE__, #call, (int)r_); \
    }                                                                                         \
  while (0)

static int p2p_setup(bp4_ctx *c)
{
  if (c->peer.empty() || c->n_ranks > kP2PMaxRanks)
    return 0;
  if (const char *e = getenv("BP4_P2P"))
    if (atoi(e) == 0)
      return 0; // developer knob: NCCL send/recv exchange
  auto &p = c->p2p;
  cudaDriverEntryPointQueryResult qr;
  void *fw = nullptr, *fq = nullptr;
  if (cudaGetDriverEntryPoint("cuStreamWriteValue64", &fw, cudaEnableDefault, &qr) != cudaSuccess || !fw ||
      cudaGetDriverEntryPoint("cuStreamWaitValue64", &fq, cudaEnableDefault, &qr) != cudaSuccess || !fq)
    {
      cudaGetLastError();
      return 0; // no stream memory operations: stay on NCCL
    }
  p.write64 = reinterpret_cast<decltype(p.write64)>(fw);
  p.wait64  = reinterpret_cast<decltype(p.wait64)>(fq);
  const uint64_t ne = c->export_off.back(), ni = c->import_off.back();
  auto           up = [](uint64_t x) { return (x + 255) & ~uint64_t(255); };
  P2PCard        mine{};
  uint64_t       off = up(sizeof(uint64_t) * 4 * kP2PMaxRanks);
  for (int k = 0; k < 2; ++k)
    {
      mine.off_ghost[k] = off;
      off += up(sizeof(double) * (ni ? ni : 1));
    }
  for (int k = 0; k < 2; ++k)
    {
      mine.off_contrib[k] = off;
      off += up(sizeof(double) * (ne ? ne : 1));
    }
  CU(cudaMalloc(&p.arena, off));
  CU(cudaMemset(p.arena, 0, off));
  CU(cudaIpcGetMemHandle(&mine.handle, p.arena));
  for (int r = 0; r < kP2PMaxRanks; ++r)
    mine.imp_off_for[r] = mine.exp_off_for[r] = -1;
  for (size_t k = 0; k < c->peer.size(); ++k)
    {
      mine.imp_off_for[c->peer[k]] = (int64_t)c->import_off[k];
      mine.exp_off_for[c->peer[k]] = (int64_t)c->export_off[k];
    }
  for (int k = 0; k < 2; ++k)
    p.off_ghost[k] = mine.off_ghost[k], p.off_contrib[k] = mine.off_contrib[k];
  // all-gather the cards through NCCL (device staging buffers)
  P2PCard *d_mine = nullptr, *d_all = nullptr;
  CU(cudaMalloc(&d_mine, sizeof(P2PCard)));
  CU(cudaMalloc(&d_all, sizeof(P2PCard) * c->n_ranks));
  CU(cudaMemcpy(d_mine, &mine, sizeof(P2PCard), cudaMemcpyHostToDevice));
  NC(ncclAllGather(d_mine, d_all, sizeof(P2PCard), ncclChar, c->comm, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  std::vector<P2PCard> all(c->n_ranks);
  CU(cudaMemcpy(all.data(), d_all, sizeof(P2PCard) * c->n_ranks, cudaMemcpyDeviceToHost));
  CU(cudaFree(d_mine));
  CU(cudaFree(d_all));
  bool ok = true;
  for (size_t k = 0; k < c->peer.size() && ok; ++k)
    {
      const P2PCard &q = all[c->peer[k]];
      void          *base = nullptr;
      if (cudaIpcOpenMemHandle(&base, q.handle, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess)
        {
          cudaGetLastError();
          ok = false;
          break;
        }
      p.peer_arena.push_back((char *)base);
      for (int b = 0; b < 2; ++b)
        {
          p.peer_off_ghost[b].push_back(q.off_ghost[b]);
          p.peer_off_contrib[b].push_back(q.off_contrib[b]);
        }
      // my exports land in the peer's ghost block for me; my ghost contributions for that owner
      // land in its contribution block for me
      p.peer_imp_off.push_back((uint64_t)std::max<int64_t>(q.imp_off_for[c->rank], 0));
      p.peer_exp_off.push_back((uint64_t)std::max<int64_t>(q.exp_off_for[c->rank], 0));
    }
  // every rank must take the same path: agree on the outcome
  int *d_ok = nullptr, h_ok = ok ? 1 : 0;
  CU(cudaMalloc(&d_ok, sizeof(int)));
  CU(cudaMemcpy(d_ok, &h_ok, sizeof(int), cudaMemcpyHostToDevice));
  NC(ncclAllReduce(d_ok, d_ok, 1, ncclInt, ncclMin, c->comm, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  CU(cudaMemcpy(&h_ok, d_ok, sizeof(int), cudaMemcpyDeviceToHost));
  CU(cudaFree(d_ok));
  p.on = h_ok == 1;
  return 0;
}

static void p2p_teardown(bp4_ctx *c)
{
  for (char *b : c->p2p.peer_arena)
    cudaIpcCloseMemHandle(b);
  c->p2p.peer_arena.clear();
  cudaFree(c->p2p.arena);
  c->p2p.arena = nullptr;
  c->p2p.on    = false;
}

int bp4_comm_init(bp4_ctx *c, int rank, int n_ranks, const unsigned char id[BP4_NCCL_ID_BYTES])
{
  if (!c || !id)
    return fail(BP4_ERR_ARG, "null argument");
  if (c->deterministic && n_ranks > 1)
    return fail(BP4_ERR_STATE, "the deterministic mode runs on one rank");
  CU(cudaSetDevice(c->device));
  ncclUniqueId u;
  memcpy(&u, id, sizeof(u));
  NC(ncclCommInitRank(&c->comm, n_ranks, u, rank));
  c->rank    = rank;
  c->n_ranks = n_ranks;
  if (n_ranks > 1 && !c->fused_pinned)
    c->fused = 0; // see Cfg<P>::FUSED_DEFAULT
  return p2p_setup(c);
}

int bp4_comm_info(bp4_ctx *c, int *n_ranks, int *peer_copies)
{
  if (!c)
    return fail(BP4_ERR_ARG, "null ctx");
  if (n_ranks)
    *n_ranks = c->n_ranks;
  if (peer_copies)
    *peer_copies = c->p2p.on ? 1 : 0;
  return 0;
}

// update_ghost_values on stream st: the packed exports (d_sendbuf) go to the peers' ghost blocks.
// NCCL form: send/recv straight into the (contiguous, per-owner) ghost blocks of v.
// Peer-copy form: copy engine -> the peers' ghost_in[e & 1], flag; wait for my own ghosts, copy
// them from ghost_in into v, release the buffer to the owners.
static int exchange_ghosts_on(bp4_ctx *c, double *v, cudaStream_t st)
{
  auto &p = c->p2p;
  if (p.on)
    {
      const uint64_t e = ++p.epoch_fwd;
      const int      b = (int)(e & 1);
      for (size_t k = 0; k < c->peer.size(); ++k)
        {
          const uint64_t ns = c->export_off[k + 1] - c->export_off[k];
          if (!ns)
            continue;
          if (e > 2) // the peer has emptied this half of its ghost_in (exchange e - 2)
            DRV(p.wait64((CUstream)st, flag_addr(p.arena, kFlagAckFwd, c->peer[k]), e - 2, CU_STREAM_WAIT_VALUE_GEQ));
          CU(cudaMemcpyAsync(p.peer_arena[k] + p.peer_off_ghost[b][k] + sizeof(double) * p.peer_imp_off[k],
                             c->d_sendbuf + c->export_off[k], sizeof(double) * ns, cudaMemcpyDeviceToDevice, st));
          DRV(p.write64((CUstream)st, flag_addr(p.peer_arena[k], kFlagDataFwd, c->rank), e, CU_STREAM_WRITE_VALUE_DEFAULT));
        }
      for (size_t k = 0; k < c->peer.size(); ++k)
        {
          const uint64_t nr = c->import_off[k + 1] - c->import_off[k];
          if (!nr)
            continue;
          DRV(p.wait64((CUstream)st, flag_addr(p.arena, kFlagDataFwd, c->peer[k]), e, CU_STREAM_WAIT_VALUE_GEQ));
          CU(cudaMemcpyAsync(v + c->n_owned + c->import_off[k],
                             p.arena + p.off_ghost[b] + sizeof(double) * c->import_off[k], sizeof(double) * nr,
                             cudaMemcpyDeviceToDevice, st));
          DRV(p.write64((CUstream)st, flag_addr(p.peer_arena[k], kFlagAckFwd, c->rank), e, CU_STREAM_WRITE_VALUE_DEFAULT));
        }
      return 0;
    }
  NC(ncclGroupStart());
  for (size_t k = 0; k < c->peer.size(); ++k)
    {
      const uint64_t ns = c->export_off[k + 1] - c->export_off[k], nr = c->import_off[k + 1] - c->import_off[k];
      if (ns)
        NC(ncclSend(c->d_sendbuf + c->export_off[k], ns, ncclDouble, c->peer[k], c->comm, st));
      if (nr)
        NC(ncclRecv(v + c->n_owned + c->import_off[k], nr, ncclDouble, c->peer[k], c->comm, st));
    }
  NC(ncclGroupEnd());
  return 0;
}

// compress(add) on stream st: the ghost slots of v travel to their owners; the owner side ends
// with the contributions in contrib_buffer(c) ready for unpack_add (compress_release afterwards)
static int exchange_compress_on(bp4_ctx *c, double *v, cudaStream_t st)
{
  auto &p = c->p2p;
  if (p.on)
    {
      const uint64_t e = ++p.epoch_rev;
      const int      b = (int)(e & 1);
      for (size_t k = 0; k < c->peer.size(); ++k)
        {
          const uint64_t ns = c->import_off[k + 1] - c->import_off[k];
          if (!ns)
            continue;
          if (e > 2)
            DRV(p.wait64((CUstream)st, flag_addr(p.arena, kFlagAckRev, c->peer[k]), e - 2, CU_STREAM_WAIT_VALUE_GEQ));
          CU(cudaMemcpyAsync(p.peer_arena[k] + p.peer_off_contrib[b][k] + sizeof(double) * p.peer_exp_off[k],
                             v + c->n_owned + c->import_off[k], sizeof(double) * ns, cudaMemcpyDeviceToDevice, st));
          DRV(p.write64((CUstream)st, flag_addr(p.peer_arena[k], kFlagDataRev, c->rank), e, CU_STREAM_WRITE_VALUE_DEFAULT));
        }
      for (size_t k = 0; k < c->peer.size(); ++k)
        if (c->export_off[k + 1] > c->export_off[k])
          DRV(p.wait64((CUstream)st, flag_addr(p.arena, kFlagDataRev, c->peer[k]), e, CU_STREAM_WAIT_VALUE_GEQ));
      return 0;
    }
  NC(ncclGroupStart());
  for (size_t k = 0; k < c->peer.size(); ++k)
    {
      const uint64_t nr = c->export_off[k + 1] - c->export_off[k], ns = c->import_off[k + 1] - c->import_off[k];
      if (ns)
        NC(ncclSend(v + c->n_owned + c->import_off[k], ns, ncclDouble, c->peer[k], c->comm, st));
      if (nr)
        NC(ncclRecv(c->d_recvbuf + c->export_off[k], nr, ncclDouble, c->peer[k], c->comm, st));
    }
  NC(ncclGroupEnd());
  return 0;
}

// where the contributions of the last compress exchange wait for unpack_add
static const double *contrib_buffer(const bp4_ctx *c)
{
  return c->p2p.on ? reinterpret_cast<const double *>(c->p2p.arena + c->p2p.off_contrib[c->p2p.epoch_rev & 1])
                   : c->d_recvbuf;
}

// after unpack_add on stream st: hand this half of contrib_in back to the ghost holders
static int compress_release(bp4_ctx *c, cudaStream_t st)
{
  auto &p = c->p2p;
  if (p.on)
    for (size_t k = 0; k < c->peer.size(); ++k)
      if (c->export_off[k + 1] > c->export_off[k])
        DRV(p.write64((CUstream)st, flag_addr(p.peer_arena[k], kFlagAckRev, c->rank), p.epoch_rev,
                      CU_STREAM_WRITE_VALUE_DEFAULT));
  return 0;
}

// owners -> ghost copies (LA::distributed::Vector::update_ghost_values)
int bp4_update_ghost_values(bp4_ctx *c, bp4_vec *v)
{
  if (!c || !v)
    return fail(BP4_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  if (c->peer.empty())
    return 0;
  if (!c->comm)
    return fail(BP4_ERR_STATE, "ghost exchange not initialised (bp4_comm_init)");
  {
    Timed t(c, BP4_K_BLAS1);
    CU(bp4::launch_pack(c->export_off.back(), c->d_export, v->p(), c->d_sendbuf, c->stream));
  }
  return exchange_ghosts_on(c, v->p(), c->stream);
}

// ghost contributions -> owners, added (compress(VectorOperation::add)); ghost slots are zeroed
int bp4_compress_add(bp4_ctx *c, bp4_vec *v)
{
  if (!c || !v)
    return fail(BP4_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  if (c->peer.empty())
    return 0;
  if (!c->comm)
    return fail(BP4_ERR_STATE, "ghost exchange not initialised (bp4_comm_init)");
  if (int e = exchange_compress_on(c, v->p(), c->stream))
    return e;
  {
    Timed t(c, BP4_K_BLAS1); // one launch for all peers: an owned entry may be exported to several (atomics)
    CU(bp4::launch_unpack_add(c->export_off.back(), c->d_export, contrib_buffer(c), v->p(), c->stream));
  }
  if (int e = compress_release(c, c->stream))
    return e;
  CU(cudaMemsetAsync(v->p() + c->n_owned, 0, sizeof(double) * c->n_ghost, c->stream));
  return 0;
}

// ---- deterministic mode --------------------------------------------------------------------
int bp4_deterministic_info(bp4_ctx *c, int *on, uint32_t *n_colors, uint32_t *cell_color)
{
  if (!c)
    return fail(BP4_ERR_ARG, "null ctx");
  if (on)
    *on = c->deterministic ? 1 : 0;
  if (n_colors)
    *n_colors = c->n_colors;
  if (cell_color)
    std::copy(c->cell_color.begin(), c->cell_color.end(), cell_color);
  return 0;
}

// ---- measurement -------------------------------------------------------------------------
int bp4_profile_enable(bp4_ctx *c, int on)
{
  if (!c)
    return fail(BP4_ERR_ARG, "null ctx");
  if (!on)
    if (int e = drain_events(c))
      return e;
  c->profile = on != 0;
  return 0;
}

int bp4_profile_reset(bp4_ctx *c)
{
  if (!c)
    return fail(BP4_ERR_ARG, "null ctx");
  if (int e = drain_events(c))
    return e;
  for (int i = 0; i < BP4_K_COUNT; ++i)
    {
      c->prof_ms[i]  = 0;
      c->prof_cnt[i] = 0;
    }
  c->launches = 0;
  return 0;
}

int bp4_profile_get(bp4_ctx *c, int id, double *total_ms, uint64_t *launches)
{
  if (!c || id < 0 || id >= BP4_K_COUNT)
    return fail(BP4_ERR_ARG, "bad kernel id");
  if (int e = drain_events(c))
    return e;
  if (total_ms)
    *total_ms = c->prof_ms[id];
  if (launches)
    *launches = c->prof_cnt[id];
  return 0;
}

int bp4_launch_count(bp4_ctx *c, uint64_t *launches)
{
  if (!c || !launches)
    return fail(BP4_ERR_ARG, "null argument");
  *launches = c->launches;
  return 0;
}

} // extern "C"
