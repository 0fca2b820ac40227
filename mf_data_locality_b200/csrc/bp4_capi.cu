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
#include <list>
#include <map>
#include <memory>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/bp4.h"
#include "bp4_launch.h"
#include "bp4_vector_kernels.cuh"

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

// owning handles of CUDA and NCCL resources: std::unique_ptr with the matching release call
template <auto F>
struct Release
{
  template <typename P>
  void operator()(P p) const
  {
    F(p);
  }
};
template <typename T>
using dev_ptr = std::unique_ptr<T, Release<cudaFree>>;
template <typename T>
using host_ptr   = std::unique_ptr<T, Release<cudaFreeHost>>; // pinned
using stream_ptr = std::unique_ptr<CUstream_st, Release<cudaStreamDestroy>>;
using event_ptr  = std::unique_ptr<CUevent_st, Release<cudaEventDestroy>>;
using graph_ptr  = std::unique_ptr<CUgraph_st, Release<cudaGraphDestroy>>;
using exec_ptr   = std::unique_ptr<CUgraphExec_st, Release<cudaGraphExecDestroy>>;
using comm_ptr   = std::unique_ptr<ncclComm, Release<ncclCommDestroy>>;
using ipc_ptr    = std::unique_ptr<char, Release<cudaIpcCloseMemHandle>>; // a peer's mapped allocation

// n elements, at least one, into p: pinned host memory for a host_ptr, device memory otherwise
template <typename T, typename D>
cudaError_t allocate(std::unique_ptr<T, D> &p, size_t n)
{
  T           *q     = nullptr;
  const size_t bytes = sizeof(T) * std::max<size_t>(n, 1);
  cudaError_t  e;
  if constexpr (std::is_same_v<D, Release<cudaFreeHost>>)
    e = cudaMallocHost(&q, bytes);
  else
    e = cudaMalloc(&q, bytes);
  p.reset(q);
  return e;
}

// allocate, then copy n elements from the host
template <typename T>
cudaError_t upload(dev_ptr<T> &p, const T *src, size_t n)
{
  cudaError_t e = allocate(p, n);
  if (e == cudaSuccess && n)
    e = cudaMemcpy(p.get(), src, sizeof(T) * n, cudaMemcpyHostToDevice);
  return e;
}

// A vector owns its buffer (bp4_vec_alloc: n + 2 doubles, recycled through the context's pool)
// or views caller-owned memory (bp4_vec_wrap: exactly n doubles, never freed or pooled here).
struct bp4_vec
{
  dev_ptr<double> buf;
  bool            owned = true;
  uint64_t        n     = 0;
  double         *p() const { return buf.get(); }
  bp4_vec() = default;
  bp4_vec(bp4_vec &&) = default; // no move assignment: it would free a wrapped target's memory
  ~bp4_vec()
  {
    if (!owned)
      (void)buf.release();
  }
};

struct ProfEvent
{
  cudaEvent_t a, b;
  int         id;
};

// instantiated graph of one device-resident solve (bp4_solve_cg*, bp4_solve_cg*_async), keyed by
// the variant, the caller's x, b and prec buffers and the in-loop form; it owns the temporaries
// g, d, h so that their addresses, baked into the graph, stay valid.  Freeing a wrapped vector
// drops the entries that name its buffer (drop_solves_on).
struct SolveGraph
{
  bool          merged = false;
  int           fused  = 0;
  const double *x = nullptr, *b = nullptr, *prec = nullptr;
  bp4_vec       g, d, h;
  graph_ptr     graph;
  exec_ptr      exec;
  cudaGraphNode_t            begin = nullptr; // the solve_begin_kernel node: per-launch arguments
  cudaGraphConditionalHandle apply = 0;       // its IF node: g = A x for a non-zero x
};

// instantiated graph of one mixed-precision solve (bp4_solve_cg_mixed*), keyed by x, b and prec like
// SolveGraph; it owns the FP64 temporary g (= A x, then A x - b) and the FP32 residual, direction,
// product, correction and preconditioner of the inner solve
struct MixedGraph
{
  const double  *x = nullptr, *b = nullptr, *prec = nullptr;
  bp4_vec        g;
  dev_ptr<float> r32, d32, h32, e32, prec32;
  graph_ptr      graph;
  exec_ptr       exec;
  cudaGraphNode_t            begin = nullptr; // the mixed_begin_kernel node: per-launch arguments
  cudaGraphConditionalHandle apply = 0;       // its IF node: g = A x for a non-zero x
};

// Members are released in reverse declaration order, after ~bp4_ctx has waited for the context's
// work: the streams are declared first so that they are released last.
struct bp4_ctx
{
  stream_ptr   stream, comm_stream;
  cudaStream_t cur = nullptr; // the caller's stream (bp4_ctx_set_stream), null: the own `stream`
  cudaStream_t st() const { return cur ? cur : stream.get(); } // where all work of the context goes
  event_ptr    ev_a, ev_b;
  int          degree = 0, device = 0, sms = 0;
  int          n_coef = 24; // geometry coefficients per cell: 24 (tri-linear) or 81 (all 27 vectors)
  uint64_t     n_cells = 0, n_owned = 0, n_ghost = 0, n_constrained = 0;
  uint64_t     n_before = 0, n_comm = 0; // cell partitions for the overlapped exchange
  int          overlap = 1;
  dev_ptr<uint32_t> d_entity, d_constrained, d_walk;
  dev_ptr<double>   d_coef, d_gll;
  dev_ptr<double>   d_acc; // [8] reduction scratch
  dev_ptr<bp4::Update4b> d_update4b; // the scalars pre_kernel derives for the fused cell kernel
  dev_ptr<int>      d_flag;
  dev_ptr<uint32_t> d_sched;     // [n_sched] unit counters of the cell-kernel launches of one loop
  uint32_t          n_sched = 4; // 4, or one per colour in the deterministic mode
  host_ptr<double>  h_acc;       // pinned [8] + sequence word (h_acc[8] reinterpreted), device-mapped
  unsigned long long pub_seq = 0;
  host_ptr<int>      h_flag;
  // device-resident solves: the solver state, the pinned (device-mapped) result of the blocking
  // calls and the cached graphs
  dev_ptr<bp4::SolveState>   d_state;
  host_ptr<bp4_solve_result> h_result;
  std::list<SolveGraph>     solves; // a list: erasing an entry moves no other (bp4_vec has no move assignment)
  // mixed-precision solves (allocated on first use): the float copy of the geometry coefficients
  // for the FP32 cell kernel, the solver state, the pinned result of the blocking call, the graphs
  dev_ptr<float>             d_coef32;
  dev_ptr<bp4::MixedState>   d_mixed;
  host_ptr<bp4_mixed_result> h_mixed;
  std::list<MixedGraph>      mixed;
  // fused merged loop (vmult_with_merged_sums): units of whole cell-batch ranges, their batches
  // and the private DoF runs the vector updates are hooked to (bp4_kernels.cuh, BatchDesc)
  int             fused      = 0;      // 1: do_cg_update4b/3b on private DoFs inside the cell kernel
  bool            fused_pinned = false; // chosen by BP4_FUSED / bp4_debug_set_fused: comm_init keeps it
  uint64_t        n_private  = 0;      // [0, n_private) are private to one range, the rest is streamed
  uint32_t        unit_part[4] = {0, 0, 0, 0}; // first unit of the three cell partitions (+ end)
  dev_ptr<bp4::BatchDesc> d_batch;
  dev_ptr<uint32_t>       d_unit_batch;
  // deterministic mode (DESIGN.md 4.6): cells stored colour by colour, colour k = stored cells
  // [color_off[k], color_off[k+1]); cell_color[i] = colour of the caller's cell i; the ordered
  // reductions' slots and ticket (det views the two buffers)
  bool                  deterministic = false;
  uint32_t              n_colors      = 0;
  std::vector<uint64_t> color_off;
  std::vector<uint32_t> cell_color;
  dev_ptr<double>       det_slot;
  dev_ptr<uint32_t>     det_ticket;
  bp4::DetSlots         det;
  // multi-GPU
  comm_ptr              comm;
  int                   rank = 0, n_ranks = 1;
  std::vector<int>      peer;
  std::vector<uint64_t> import_off, export_off;
  dev_ptr<uint32_t>     d_export;
  dev_ptr<double>       d_sendbuf, d_recvbuf;
  // Peer exchange without SMs (the USE_SHMEM analogue of benchmark.h:35, :105-108): every rank
  // owns one IPC-shared arena [flags | ghost_in[2] | contrib_in[2]]; owners push their exported
  // values into the peers' ghost_in with copy-engine peer copies, ghost holders push their
  // contributions into the owners' contrib_in, and arrival / release is signalled with stream
  // memory operations (cuStreamWriteValue64 / cuStreamWaitValue64) on the flag words -- nothing
  // of it needs an SM, so it runs next to the persistent cell kernel.
  struct P2P
  {
    bool                 on = false;
    dev_ptr<char>        arena;                     // my arena (device)
    uint64_t             off_ghost[2] = {0, 0}, off_contrib[2] = {0, 0};
    std::vector<ipc_ptr> peer_arena;                // [n_peers] mapped base of peer k's arena
    std::vector<uint64_t> peer_off_ghost[2], peer_off_contrib[2]; // [n_peers] byte offsets there
    std::vector<uint64_t> peer_imp_off, peer_exp_off; // [n_peers] where MY data goes (doubles)
    uint64_t             epoch_fwd = 0, epoch_rev = 0;
    CUresult (*write64)(CUstream, CUdeviceptr, cuuint64_t, unsigned) = nullptr;
    CUresult (*wait64)(CUstream, CUdeviceptr, cuuint64_t, unsigned)  = nullptr;
  } p2p;
  // freed vector buffers kept for reuse, keyed by size: plays the role of deal.II's
  // GrowingVectorMemory pool behind SolverCGFullMerge's temporaries (solver_cg_optimized.h:201)
  std::multimap<uint64_t, dev_ptr<double>> pool;
  // measurement
  bool                   profile = false;
  std::vector<ProfEvent> events;
  std::vector<event_ptr> event_pool; // recycled timing events (creating one costs microseconds)
  double                 prof_ms[BP4_K_COUNT]  = {0};
  uint64_t               prof_cnt[BP4_K_COUNT] = {0};
  uint64_t               launches               = 0;

  ~bp4_ctx();
};

namespace
{
  bool capturing(cudaStream_t st)
  {
    cudaStreamCaptureStatus s = cudaStreamCaptureStatusNone;
    return cudaStreamIsCapturing(st, &s) == cudaSuccess && s != cudaStreamCaptureStatusNone;
  }

  // A call that waits on the host, allocates or builds a graph cannot run while the caller is
  // capturing the stream into a graph of its own: refuse it before anything is queued.
  int refuse_capture(const bp4_ctx *c, const char *call)
  {
    if (capturing(c->st()))
      return fail(BP4_ERR_STATE, "%s synchronises the stream or allocates, and the stream is being captured into a "
                                 "graph: call it before the capture begins or after it ends", call);
    return 0;
  }

  // RAII: count a launch, and time it with events when profiling is on.  While the stream is
  // being captured into a graph the launch is counted but not timed (no events inside a graph).
  struct Timed
  {
    bp4_ctx *c;
    int      id;
    ProfEvent ev{};
    bool      on;
    Timed(bp4_ctx *c_, int id_, int n_launches = 1) : c(c_), id(id_), on(c_->profile && !capturing(c_->st()))
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
                *e = c->event_pool.back().release();
                c->event_pool.pop_back();
              }
          ev.id = id;
          cudaEventRecord(ev.a, c->st());
        }
    }
    ~Timed()
    {
      if (on)
        {
          cudaEventRecord(ev.b, c->st());
          c->events.push_back(ev);
        }
    }
  };

  // collect the times of the recorded event pairs; returns the first error and sets no message, so
  // that ~bp4_ctx can drain without touching bp4_last_error
  cudaError_t drain_events(bp4_ctx *c)
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
        c->event_pool.emplace_back(ev.a);
        c->event_pool.emplace_back(ev.b);
      }
    c->events.clear();
    return err;
  }

  // The vector kernels (bp4_vector_kernels.cuh) are launched on the context's stream by one helper
  // per grid rule; nothing is launched for n == 0, a launch error becomes BP4_ERR_CUDA.
  int stream_grid(uint64_t n, int sms)
  {
    const uint64_t blocks = (n + 255) / 256;
    return (int)std::min<uint64_t>(std::max<uint64_t>(blocks, 1), (uint64_t)sms * 8);
  }

  // a grid-stride sweep over n elements: stream_grid(n) blocks of 256 threads, one Timed record of `id`
  template <typename... P, typename... A>
  int sweep(bp4_ctx *c, int id, uint64_t n, void (*kernel)(P...), A... args)
  {
    Timed t(c, id);
    if (n == 0)
      return 0;
    kernel<<<stream_grid(n, c->sms), 256, 0, c->st()>>>(args...);
    CU(cudaGetLastError());
    return 0;
  }

  // one thread per element: ceil(n / B) blocks of B threads, counted in the caller's Timed record
  template <int B = 256, typename... P, typename... A>
  int per_element(bp4_ctx *c, uint64_t n, void (*kernel)(P...), A... args)
  {
    if (n == 0)
      return 0;
    kernel<<<(unsigned)((n + B - 1) / B), B, 0, c->st()>>>(args...);
    CU(cudaGetLastError());
    return 0;
  }

  // v = n doubles, from the pool when a buffer of that size is cached; zeroed on request only
  // (SolverCGFullMerge takes its temporaries with omit_zeroing_entries = true,
  // solver_cg_optimized.h:215-217)
  int pooled_alloc(bp4_ctx *c, uint64_t n, bp4_vec &v, bool zero)
  {
    v.n     = n;
    auto it = c->pool.find(n);
    if (it != c->pool.end())
      {
        v.buf = std::move(it->second);
        c->pool.erase(it);
      }
    else
      CU(allocate(v.buf, n + 2)); // + 2: the fused loop copies runs in 16-byte pieces, one element past either end
    if (zero)
      CU(cudaMemsetAsync(v.p(), 0, sizeof(double) * n, c->st()));
    return 0;
  }

  // v's buffer back to the pool; stream order makes reuse safe: the next user's work is queued
  // behind ours.  A wrapped buffer is the caller's and stays out of the pool.
  void recycle(bp4_ctx *c, bp4_vec &v)
  {
    if (v.buf && v.owned)
      c->pool.emplace(v.n, std::move(v.buf));
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
      NC(ncclAllReduce(c->d_acc.get(), c->d_acc.get(), k, ncclDouble, ncclSum, c->comm.get(), c->st()));
    // the last kernel of the chain writes the values and then a sequence number into mapped
    // pinned memory; the host polls that word (and the stream, for errors, now and then)
    volatile unsigned long long *seq_word = reinterpret_cast<volatile unsigned long long *>(c->h_acc.get() + 8);
    const unsigned long long     seq      = ++c->pub_seq;
    bp4::publish_kernel<<<1, 32, 0, c->st()>>>(c->d_acc.get(), k, c->h_acc.get(), seq_word, seq);
    CU(cudaGetLastError());
    c->launches += 1;
    int idle = 0;
    for (unsigned long long spins = 1; *seq_word != seq; ++spins)
      if ((spins & 0xFFFF) == 0)
        {
          const cudaError_t q = cudaStreamQuery(c->st());
          if (q != cudaSuccess && q != cudaErrorNotReady)
            CU(q);
          if (q == cudaSuccess && ++idle > 8) // stream drained, nothing published: cannot happen
            return fail(BP4_ERR_CUDA, "reduction result was not published");
        }
    for (int i = 0; i < k; ++i)
      out[i] = c->h_acc.get()[i];
    return 0;
  }
} // namespace

// The caller's stream is not the context's to destroy or drain: an event recorded on it after the
// context's last call marks where the context's work ends there.
bp4_ctx::~bp4_ctx()
{
  cudaSetDevice(device);
  if (cur && ev_a && cudaEventRecord(ev_a.get(), cur) == cudaSuccess)
    cudaEventSynchronize(ev_a.get());
  if (stream)
    cudaStreamSynchronize(stream.get());
  drain_events(this);
}

extern "C" {
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
  for (stream_ptr *s : {&c->stream, &c->comm_stream})
    {
      cudaStream_t q;
      CU(cudaStreamCreateWithFlags(&q, cudaStreamNonBlocking));
      s->reset(q);
    }
  for (event_ptr *e : {&c->ev_a, &c->ev_b})
    {
      cudaEvent_t q;
      CU(cudaEventCreateWithFlags(&q, cudaEventDisableTiming));
      e->reset(q);
    }

  std::vector<uint32_t> walk;
  CU(bp4::launch_init_degree(d->degree, walk));
  CU(upload(c->d_walk, walk.data(), walk.size()));

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

  c->n_coef = d->coefficients ? 81 : 24;
  const uint64_t nc = std::max<uint64_t>(d->n_cells, 1);
  CU(allocate(c->d_entity, 27 * nc));
  CU(allocate(c->d_coef, c->n_coef * nc));
  if (d->n_cells)
    CU(upload_rows(c->d_entity.get(), d->entity_index, 27, d->n_cells, order));
  if (d->n_cells && d->coefficients) // all 27 coefficient vectors of the reference's kernel, as given
    CU(upload_rows(c->d_coef.get(), d->coefficients, 81, d->n_cells, order));
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
      CU(upload_rows(c->d_coef.get(), cf.data(), 24, d->n_cells, order));
    }
  CU(upload(c->d_constrained, d->constrained, d->n_constrained));
  std::vector<double> gll;
  bp4::gll_table(d->degree, gll);
  CU(upload(c->d_gll, gll.data(), gll.size()));
  CU(allocate(c->d_acc, 8));
  CU(cudaMemset(c->d_acc.get(), 0, sizeof(double) * 8));
  CU(allocate(c->d_update4b, 1));
  CU(allocate(c->d_flag, 1));
  CU(allocate(c->d_sched, c->n_sched));
  if (c->deterministic)
    {
      CU(allocate(c->det_slot, (size_t)8 * 8 * c->sms)); // K <= 7 partials of <= 8 * SMs blocks (stream_grid)
      CU(allocate(c->det_ticket, 1));
      CU(cudaMemset(c->det_ticket.get(), 0, sizeof(uint32_t)));
      c->det = {c->det_slot.get(), c->det_ticket.get()};
    }
  CU(allocate(c->h_acc, 16)); // UVA: the pointer is valid on the device too
  memset(c->h_acc.get(), 0, sizeof(double) * 16);
  CU(allocate(c->h_flag, 1));
  CU(allocate(c->d_state, 1));
  CU(allocate(c->h_result, 1));

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
      CU(upload(c->d_batch, batches.data(), batches.size()));
      CU(upload(c->d_unit_batch, unit_batch.data(), unit_batch.size()));
      c->n_private = c->n_coef == 24 ? rp[d->n_ranges] : 0; // in-loop updates: tri-linear kernel only
      // the staged fused loop takes a batch's private run in two jobs of its shared-memory rows
      for (const bp4::BatchDesc &b : batches) // run_limit 0: no fused kernel at this degree
        if (b.pre_end - b.pre_begin > fl.run_limit || b.post_end - b.post_begin > fl.run_limit)
          c->n_private = 0; // the updates of every DoF are streamed then
      // a job copies whole 16-byte pieces: a run ending at n_owned reads the element past the last
      // DoF (odd end) and the prec entry past the last node, which a wrapped vector does not have
      // (DESIGN.md 3).  Runs that end earlier stop at least one node before the end.
      if (rp[d->n_ranges] == d->n_owned)
        c->n_private = 0;
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
      CU(upload(c->d_export, d->export_index, ne));
      CU(allocate(c->d_sendbuf, ne));
      CU(allocate(c->d_recvbuf, ne));
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
  std::unique_ptr<bp4_ctx> c(new bp4_ctx);
  c->deterministic = deterministic;
  if (int e = ctx_create_impl(d, c.get()))
    return e;
  *out = c.release();
  return 0;
}

int bp4_ctx_destroy(bp4_ctx *c)
{
  delete c;
  return 0;
}

int bp4_ctx_synchronize(bp4_ctx *c)
{
  if (!c)
    return fail(BP4_ERR_ARG, "null ctx");
  if (int e = refuse_capture(c, "bp4_ctx_synchronize"))
    return e;
  CU(cudaStreamSynchronize(c->st()));
  return 0;
}

int bp4_ctx_stream(bp4_ctx *c, void **stream)
{
  if (!c || !stream)
    return fail(BP4_ERR_ARG, "null argument");
  *stream = (void *)c->st();
  return 0;
}

// The new stream waits for everything queued so far on the old one (an event, no host wait):
// pooled buffers, solve temporaries and the reduction scratch may still be in use there.
int bp4_ctx_set_stream(bp4_ctx *c, void *stream)
{
  if (!c)
    return fail(BP4_ERR_ARG, "null ctx");
  CU(cudaSetDevice(c->device));
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (s)
    {
      int dev = -1;
      if (cudaStreamGetDevice(s, &dev) != cudaSuccess)
        {
          cudaGetLastError();
          return fail(BP4_ERR_ARG, "set_stream: %p is not a stream", stream);
        }
      if (dev != c->device)
        return fail(BP4_ERR_ARG, "set_stream: stream %p belongs to device %d, the context runs on device %d", stream,
                    dev, c->device);
    }
  const cudaStream_t next = s ? s : c->stream.get();
  if (capturing(c->st()) || capturing(next))
    return fail(BP4_ERR_STATE, "set_stream: the old or the new stream is being captured into a graph: switch "
                               "streams outside a capture");
  if (next != c->st())
    {
      CU(cudaEventRecord(c->ev_a.get(), c->st()));
      CU(cudaStreamWaitEvent(next, c->ev_a.get(), 0));
    }
  c->cur = s;
  return 0;
}

static int vec_alloc(bp4_ctx *c, uint64_t n, bp4_vec **out, bool zero)
{
  if (!c || !out)
    return fail(BP4_ERR_ARG, "null argument");
  if (int e = refuse_capture(c, "bp4_vec_alloc"))
    return e;
  CU(cudaSetDevice(c->device));
  std::unique_ptr<bp4_vec> v(new bp4_vec);
  if (int e = pooled_alloc(c, n, *v, zero))
    return e;
  *out = v.release();
  return 0;
}

int bp4_vec_alloc(bp4_ctx *c, uint64_t n, bp4_vec **out) { return vec_alloc(c, n, out, true); }
int bp4_vec_alloc_uninitialized(bp4_ctx *c, uint64_t n, bp4_vec **out) { return vec_alloc(c, n, out, false); }

int bp4_vec_wrap(bp4_ctx *c, double *dev, uint64_t n, bp4_vec **out)
{
  if (!c || !out)
    return fail(BP4_ERR_ARG, "null argument");
  if (!dev || n == 0)
    return fail(BP4_ERR_ARG, "wrap: null pointer or empty vector");
  if (reinterpret_cast<uintptr_t>(dev) % 16)
    return fail(BP4_ERR_ARG, "wrap: %p is not 16-byte aligned", (void *)dev);
  CU(cudaSetDevice(c->device));
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, dev) != cudaSuccess)
    {
      cudaGetLastError();
      return fail(BP4_ERR_ARG, "wrap: %p is not device memory of device %d", (void *)dev, c->device);
    }
  if (at.type != cudaMemoryTypeDevice || at.device != c->device) // host, managed or another GPU's
    return fail(BP4_ERR_ARG, "wrap: %p is not device memory of device %d (memory type %d, device %d)", (void *)dev,
                c->device, (int)at.type, at.device);
  std::unique_ptr<bp4_vec> v(new bp4_vec);
  v->owned = false;
  v->n     = n;
  v->buf.reset(dev);
  *out = v.release();
  return 0;
}

// drop the cached solve graphs that name buf; their temporaries go back to the pool
static void drop_solves_on(bp4_ctx *c, const double *buf)
{
  for (auto it = c->solves.begin(); it != c->solves.end();)
    if (it->x == buf || it->b == buf || it->prec == buf)
      {
        for (bp4_vec *t : {&it->g, &it->d, &it->h})
          recycle(c, *t);
        it = c->solves.erase(it);
      }
    else
      ++it;
  for (auto it = c->mixed.begin(); it != c->mixed.end();)
    if (it->x == buf || it->b == buf || it->prec == buf)
      {
        recycle(c, it->g);
        it = c->mixed.erase(it);
      }
    else
      ++it;
}

int bp4_vec_free(bp4_ctx *c, bp4_vec *v)
{
  if (c && v)
    {
      if (v->owned)
        recycle(c, *v);
      else // the caller's next buffer has another address: without this the cache grew per solve
        {
          cudaSetDevice(c->device);
          drop_solves_on(c, v->p());
        }
    }
  delete v; // without a context an owned buffer is freed
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
  CU(cudaMemsetAsync(v->p(), 0, sizeof(double) * v->n, c->st()));
  return 0;
}

int bp4_vec_upload(bp4_ctx *c, bp4_vec *v, const double *host, uint64_t n)
{
  if (!c || !v || (!host && n))
    return fail(BP4_ERR_ARG, "null argument");
  if (int e = refuse_capture(c, "bp4_vec_upload"))
    return e;
  CU(cudaSetDevice(c->device));
  if (n > v->n)
    return fail(BP4_ERR_ARG, "upload of %llu > vector size %llu", (unsigned long long)n,
                (unsigned long long)v->n);
  CU(cudaMemcpyAsync(v->p(), host, sizeof(double) * n, cudaMemcpyHostToDevice, c->st()));
  return 0;
}

int bp4_vec_download(bp4_ctx *c, const bp4_vec *v, double *host, uint64_t n)
{
  if (!c || !v || (!host && n))
    return fail(BP4_ERR_ARG, "null argument");
  if (int e = refuse_capture(c, "bp4_vec_download"))
    return e;
  CU(cudaSetDevice(c->device));
  if (n > v->n)
    return fail(BP4_ERR_ARG, "download of %llu > vector size %llu", (unsigned long long)n,
                (unsigned long long)v->n);
  CU(cudaMemcpyAsync(host, v->p(), sizeof(double) * n, cudaMemcpyDeviceToHost, c->st()));
  CU(cudaStreamSynchronize(c->st()));
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

// vectors and scalars of one vmult_with_merged_sums call; the scalars go to pre_kernel, which
// derives those of do_cg_update4b for the streamed and the in-loop DoFs
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
  a.dtab  = c->d_walk.get();
  a.src   = src;
  a.dst   = dst;
  a.sched = c->d_sched.get() + (part < 0 ? 0 : part);
  if (m)
    {
      const uint32_t u0 = part < 0 ? c->unit_part[0] : c->unit_part[part],
                     u1 = part < 0 ? c->unit_part[3] : c->unit_part[part + 1];
      a.entity_index = c->d_entity.get();
      a.coef         = c->d_coef.get();
      a.n_cells      = c->n_cells;
      a.batch        = c->d_batch.get();
      a.unit_batch   = c->d_unit_batch.get() + u0;
      a.n_units      = u1 - u0;
      a.r            = m->g;
      a.p            = m->d;
      a.x            = m->x;
      a.prec         = m->prec;
      a.scalars      = c->d_update4b.get();
      a.acc          = c->d_acc.get();
      Timed t(c, BP4_K_MERGED);
      CU(bp4::launch_cell(c->degree, true, false, a, c->sms, c->st()));
    }
  else if (c->deterministic) // one launch per colour (single rank: part = -1), timed as one loop
    {
      Timed t(c, BP4_K_VMULT, (int)c->n_colors);
      for (uint32_t k = 0; k < c->n_colors; ++k)
        {
          const uint64_t c0 = c->color_off[k];
          a.entity_index    = c->d_entity.get() + 27 * c0;
          a.coef            = c->d_coef.get() + (uint64_t)c->n_coef * c0;
          a.n_cells         = c->color_off[k + 1] - c0;
          a.sched           = c->d_sched.get() + k;
          CU(bp4::launch_cell(c->degree, false, c->n_coef == 81, a, c->sms, c->st()));
        }
    }
  else
    {
      a.entity_index = c->d_entity.get() + 27 * begin;
      a.coef         = c->d_coef.get() + (uint64_t)c->n_coef * begin;
      a.n_cells      = end - begin;
      Timed t(c, BP4_K_VMULT);
      CU(bp4::launch_cell(c->degree, false, c->n_coef == 81, a, c->sms, c->st()));
    }
  return 0;
}

static int exchange_ghosts_on(bp4_ctx *c, double *v, cudaStream_t st);
static int exchange_compress_on(bp4_ctx *c, double *v, cudaStream_t st);
static int compress_finish(bp4_ctx *c, double *v);


// MatrixFree::cell_loop (poisson_operator.h:310, :339) on one rank: update_ghost_values(src),
// cells, compress(add)(dst).  With a partitioned mesh the two exchanges run on a second stream
// while the cells that touch no ghost DoF are processed (SURVEY App. B1):
//   pack | interior part 1 || send/recv ghosts | ghost-touching cells | interior part 2 ||
//   send/recv contributions | unpack-add.
// dst must already be zero where the cells accumulate (owned and ghost slots).
static int cell_loop(bp4_ctx *c, double *dst, const double *src, const MergedCall *m)
{
  CU(cudaMemsetAsync(c->d_sched.get(), 0, sizeof(uint32_t) * c->n_sched, c->st()));
  if (c->peer.empty())
    return cell_range(c, dst, src, -1, m);
  if (!c->comm)
    return fail(BP4_ERR_STATE, "ghost exchange not initialised (bp4_comm_init)");
  const uint64_t ne      = c->export_off.back();
  const bool     overlap = c->overlap && c->n_comm > 0;
  {
    Timed t(c, BP4_K_BLAS1);
    if (int e = per_element(c, ne, bp4::pack_kernel, ne, c->d_export.get(), src, c->d_sendbuf.get()))
      return e;
  }
  CU(cudaEventRecord(c->ev_a.get(), c->st()));
  CU(cudaStreamWaitEvent(c->comm_stream.get(), c->ev_a.get(), 0));
  if (int e = exchange_ghosts_on(c, const_cast<double *>(src), c->comm_stream.get()))
    return e;
  CU(cudaEventRecord(c->ev_b.get(), c->comm_stream.get()));
  if (overlap)
    if (int e = cell_range(c, dst, src, 0, m))
      return e;
  CU(cudaStreamWaitEvent(c->st(), c->ev_b.get(), 0));
  if (overlap)
    {
      if (int e = cell_range(c, dst, src, 1, m))
        return e;
    }
  else if (int e = cell_range(c, dst, src, -1, m))
    return e;
  CU(cudaEventRecord(c->ev_a.get(), c->st()));
  CU(cudaStreamWaitEvent(c->comm_stream.get(), c->ev_a.get(), 0));
  if (int e = exchange_compress_on(c, dst, c->comm_stream.get()))
    return e;
  CU(cudaEventRecord(c->ev_b.get(), c->comm_stream.get()));
  if (overlap)
    if (int e = cell_range(c, dst, src, 2, m))
      return e;
  CU(cudaStreamWaitEvent(c->st(), c->ev_b.get(), 0));
  return compress_finish(c, dst);
}

// dst = A src on the context's stream (also captured into the plain device solve's loop body)
static int vmult_on(bp4_ctx *c, double *dst, const double *src)
{
  CU(cudaMemsetAsync(dst, 0, sizeof(double) * (c->n_owned + c->n_ghost), c->st()));
  if (int e = cell_loop(c, dst, src, nullptr))
    return e;
  Timed t(c, BP4_K_BLAS1);
  return per_element(c, c->n_constrained, bp4::fixup_kernel<double>, c->n_constrained, c->d_constrained.get(), dst,
                     src);
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
  // one block at least: pre_kernel also clears the reduction scratch and publishes the scalars
  // the fused cell kernel reads
  if (int e = sweep(c, BP4_K_PRE, std::max<uint64_t>(n - tail, 1),
                    m.state ? bp4::pre_kernel<true> : bp4::pre_kernel<false>, tail, n, h, m.x, m.g, m.d, m.prec,
                    m.alpha, m.beta, m.alpha_old, m.beta_old, c->d_acc.get(), c->d_update4b.get(), m.state))
    return e;
  if (c->n_ghost)
    CU(cudaMemsetAsync(h + n, 0, sizeof(double) * c->n_ghost, c->st()));
  if (int e = cell_loop(c, h, m.d, c->fused ? &m : nullptr))
    return e;
  if (n > tail)
    return sweep(c, BP4_K_POST, n - tail, c->deterministic ? bp4::post_kernel<true> : bp4::post_kernel<false>, tail,
                 n, m.g, m.d, h, m.prec, c->d_acc.get(), c->det);
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
  if (int e = refuse_capture(c, "bp4_vmult_merged"))
    return e;
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
  const uint64_t n3       = (uint64_t)(c->degree + 1) * (c->degree + 1) * (c->degree + 1);
  Timed          t(c, BP4_K_BLAS1, (int)n_groups + more);
  for (uint32_t k = 0; k < n_groups; ++k)
    {
      const uint64_t c0 = c->deterministic ? c->color_off[k] : 0,
                     c1 = c->deterministic ? c->color_off[k + 1] : c->n_cells;
      if (int e = per_element<128>(c, (c1 - c0) * n3, bp4::diag_kernel, c->degree, c1 - c0, c->d_entity.get() + 27 * c0,
                                   c->d_coef.get() + (uint64_t)c->n_coef * c0, c->n_coef, c->d_gll.get(), diag, 3))
        return e;
    }
  return 0;
}

int bp4_inverse_diagonal(bp4_ctx *c, bp4_vec *out)
{
  if (!c || !out)
    return fail(BP4_ERR_ARG, "null argument");
  if (int e = refuse_capture(c, "bp4_inverse_diagonal"))
    return e;
  CU(cudaSetDevice(c->device));
  if (out->n < c->n_owned / 3)
    return fail(BP4_ERR_ARG, "diagonal vector needs n_owned/3 entries");
  // assemble DoF-wise into slot 3*node of a local vector so that the ordinary ghost
  // compress(add) (poisson_operator.h:419) can be reused, then keep one entry per owned node
  // (the temporary goes back to the pool on success and is freed on an error return)
  bp4_vec tmp;
  if (int e = pooled_alloc(c, c->n_owned + c->n_ghost, tmp, true))
    return e;
  if (int e = assemble_diagonal(c, tmp.p(), 2))
    return e;
  if (!c->peer.empty())
    if (int e = bp4_compress_add(c, &tmp))
      return e;
  const uint64_t n_nodes = c->n_owned / 3;
  if (int e = per_element(c, n_nodes, bp4::stride3_kernel, n_nodes, tmp.p(), out->p()))
    return e;
  if (int e = per_element(c, n_nodes, bp4::invert_diag_kernel, n_nodes, out->p()))
    return e;
  recycle(c, tmp);
  return 0;
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
  CU(cudaMemsetAsync(out->p(), 0, sizeof(double) * (c->n_owned + c->n_ghost), c->st()));
  if (int e = assemble_diagonal(c, out->p(), 1))
    return e;
  if (!c->peer.empty())
    if (int e = bp4_compress_add(c, out))
      return e;
  return per_element(c, c->n_owned, bp4::invert_diag_kernel, c->n_owned, out->p());
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
  return per_element(c, c->n_owned / 3, bp4::stride3_kernel, c->n_owned / 3, src->p() + component, dst->p());
}

int bp4_jacobi_vmult(bp4_ctx *c, bp4_vec *dst, const bp4_vec *src, const bp4_vec *diag)
{
  if (!c || !dst || !src || !diag)
    return fail(BP4_ERR_ARG, "null argument");
  if (dst->n < c->n_owned || src->n < c->n_owned || 3 * diag->n < c->n_owned)
    return fail(BP4_ERR_ARG, "Dimension mismatch %llu vs 3 x %llu", (unsigned long long)dst->n,
                (unsigned long long)diag->n);
  CU(cudaSetDevice(c->device));
  return sweep(c, BP4_K_BLAS1, c->n_owned, bp4::jacobi_kernel, c->n_owned, dst->p(), src->p(), diag->p());
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
  return sweep(c, BP4_K_BLAS1, c->n_owned, bp4::xfinal_kernel, c->n_owned, x->p(), d->p(), g->p(), prec->p(), c1,
               c2);
}

int bp4_sadd(bp4_ctx *c, bp4_vec *dst, double s, double a, const bp4_vec *src)
{
  if (!c || !dst || !src)
    return fail(BP4_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  const uint64_t n = sweep_len(c, {dst, src});
  return sweep(c, BP4_K_BLAS1, n, bp4::sadd_kernel<false>, n, dst->p(), s, a, src->p(), nullptr);
}

int bp4_equ(bp4_ctx *c, bp4_vec *dst, double a, const bp4_vec *src) { return bp4_sadd(c, dst, 0., a, src); }
int bp4_add(bp4_ctx *c, bp4_vec *dst, double a, const bp4_vec *src) { return bp4_sadd(c, dst, 1., a, src); }

int bp4_dot(bp4_ctx *c, const bp4_vec *a, const bp4_vec *b, double *result)
{
  if (!c || !a || !b || !result)
    return fail(BP4_ERR_ARG, "null argument");
  if (int e = refuse_capture(c, "bp4_dot"))
    return e;
  CU(cudaSetDevice(c->device));
  const uint64_t n = sweep_len(c, {a, b});
  if (int e = sweep(c, BP4_K_BLAS1, n, c->deterministic ? bp4::dot_kernel<true> : bp4::dot_kernel<false>, n, a->p(),
                    b->p(), c->d_acc.get(), c->det))
    return e;
  return reduce_to_host(c, 1, result);
}

int bp4_add_and_dot(bp4_ctx *c, bp4_vec *g, double a, const bp4_vec *h, const bp4_vec *w, double *result)
{
  if (!c || !g || !h || !w || !result)
    return fail(BP4_ERR_ARG, "null argument");
  if (int e = refuse_capture(c, "bp4_add_and_dot"))
    return e;
  CU(cudaSetDevice(c->device));
  const uint64_t n = sweep_len(c, {g, h, w});
  if (int e = sweep(c, BP4_K_BLAS1, n,
                    c->deterministic ? bp4::add_and_dot_kernel<true> : bp4::add_and_dot_kernel<false>, n, g->p(), a,
                    h->p(), w->p(), c->d_acc.get(), c->det))
    return e;
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
  if (int e = refuse_capture(c, "bp4_all_zero"))
    return e;
  CU(cudaSetDevice(c->device));
  CU(cudaMemsetAsync(c->d_flag.get(), 0, sizeof(int), c->st()));
  const uint64_t n = sweep_len(c, {v});
  if (int e = sweep(c, BP4_K_BLAS1, n, bp4::nonzero_kernel, n, v->p(), c->d_flag.get()))
    return e;
  if (c->comm)
    NC(ncclAllReduce(c->d_flag.get(), c->d_flag.get(), 1, ncclInt, ncclMax, c->comm.get(), c->st()));
  CU(cudaMemcpyAsync(c->h_flag.get(), c->d_flag.get(), sizeof(int), cudaMemcpyDeviceToHost, c->st()));
  CU(cudaStreamSynchronize(c->st()));
  *result = *c->h_flag ? 0 : 1;
  return 0;
}

// ---- whole solves on the device ----------------------------------------------------------
// Capture what `launch` enqueues into `graph`, after the nodes `deps`; `leaves` (optional)
// receives the nodes the next one must follow.  The capture runs on the context's own stream
// whichever stream is current (a caller's stream may be the legacy default stream, which cannot be
// captured) and is always ended, also when a launch fails, so that the stream stays usable.
extern "C++" {
template <typename F>
static int capture_into(bp4_ctx *c, cudaGraph_t graph, const cudaGraphNode_t *deps, size_t n_deps, F &&launch,
                        std::vector<cudaGraphNode_t> *leaves)
{
  const cudaStream_t cur = c->cur, own = c->stream.get();
  CU(cudaStreamBeginCaptureToGraph(own, graph, deps, nullptr, n_deps, cudaStreamCaptureModeThreadLocal));
  c->cur = nullptr;
  int e  = launch();
  c->cur = cur;
  if (!e && leaves)
    {
      cudaStreamCaptureStatus st;
      const cudaGraphNode_t  *d = nullptr;
      size_t                  n = 0;
      const cudaError_t       q = cudaStreamGetCaptureInfo(own, &st, nullptr, nullptr, &d, &n);
      if (q == cudaSuccess)
        leaves->assign(d, d + n);
      else
        e = fail(BP4_ERR_CUDA, "cudaStreamGetCaptureInfo: %s", cudaGetErrorString(q));
    }
  cudaGraph_t       out = nullptr;
  const cudaError_t q   = cudaStreamEndCapture(own, &out);
  if (e)
    return e;
  CU(q);
  return 0;
}
} // extern "C++"

// a conditional node (IF or WHILE on handle h) after `deps`; *body receives the graph it runs
static int add_conditional(cudaGraph_t graph, const std::vector<cudaGraphNode_t> &deps, cudaGraphConditionalHandle h,
                           cudaGraphConditionalNodeType type, cudaGraphNode_t *node, cudaGraph_t *body)
{
  cudaGraphNodeParams cp = {};
  cp.type                = cudaGraphNodeTypeConditional;
  cp.conditional.handle  = h;
  cp.conditional.type    = type;
  cp.conditional.size    = 1;
  CU(cudaGraphAddNode(node, graph, deps.data(), deps.size(), &cp));
  *body = cp.conditional.phGraph_out[0];
  return 0;
}

// the per-call arguments of a solve, as the parameters of its solve_begin_kernel node
struct SolveArgs
{
  bp4::SolveState           *st;
  const int                 *nonzero;
  uint32_t                   max_steps;
  double                     tol, reduce;
  double                    *history;
  void                      *result;
  cudaGraphConditionalHandle apply;
  void                      *ptr[8] = {&st, &nonzero, &max_steps, &tol, &reduce, &history, &result, &apply};
  SolveArgs(const SolveArgs &) = delete; // ptr points into this object
  SolveArgs(bp4::SolveState *st_, const int *nz, uint32_t ms, double t, double r, double *hi, void *re,
            cudaGraphConditionalHandle ap)
    : st(st_), nonzero(nz), max_steps(ms), tol(t), reduce(r), history(hi), result(re), apply(ap)
  {}
  cudaKernelNodeParams params()
  {
    cudaKernelNodeParams kp = {};
    kp.func                 = reinterpret_cast<void *>(bp4::solve_begin_kernel);
    kp.gridDim              = dim3(1);
    kp.blockDim             = dim3(32);
    kp.kernelParams         = ptr;
    return kp;
  }
};

// One CUDA graph per solve, every step of it on the device:
//   x != 0?  -> solve_begin (per-call arguments) -> IF x != 0 { g = A x } -> g = g_scale g - b,
//   |g|, check(0) -> [plain: h = P g, d = -h, gh] -> WHILE { one iteration }
//   -> [merged: IF iterated { pending x update }] -> result to the caller.
// The start residual and the loop body are captured from the launch code of the host-driven path
// (bp4_all_zero, vmult_on, bp4_add / bp4_equ, bp4_dot, merged_sweep); the scalar kernels keep
// alpha, beta, ... in c->d_state and set the loop condition.
static int build_solve_graph(bp4_ctx *c, SolveGraph &sg)
{
  const uint64_t n    = c->n_owned;
  double        *x    = const_cast<double *>(sg.x);
  const double  *prec = sg.prec;
  bp4::SolveState *st = c->d_state.get();
  double        *acc  = c->d_acc.get();
  double        *g = sg.g.p(), *d = sg.d.p(), *h = sg.h.p();
  cudaGraph_t    graph;
  CU(cudaGraphCreate(&graph, 0));
  sg.graph.reset(graph);
  // every handle needs its conditional node: the plain solve has no final x update, and its
  // step-0 kernel sets `loop` twice
  cudaGraphConditionalHandle loop, iterated;
  CU(cudaGraphConditionalHandleCreate(&sg.apply, graph, 0, cudaGraphCondAssignDefault));
  CU(cudaGraphConditionalHandleCreate(&loop, graph, 0, cudaGraphCondAssignDefault));
  iterated = loop;
  if (sg.merged)
    CU(cudaGraphConditionalHandleCreate(&iterated, graph, 0, cudaGraphCondAssignDefault));
  std::vector<cudaGraphNode_t> leaves;
  auto jacobi_dot = [&]() { // h = P g, g.h -> acc[2]
    return sweep(c, BP4_K_BLAS1, n, c->deterministic ? bp4::jacobi_dot_kernel<true> : bp4::jacobi_dot_kernel<false>,
                 n, h, g, prec, acc + 2, c->det);
  };
  auto scalar = [&](const int kind) -> int { // solve_scalar_kernel on one thread
    Timed t(c, BP4_K_BLAS1);
    bp4::solve_scalar_kernel<<<1, 32, 0, c->st()>>>(kind, st, acc, loop);
    CU(cudaGetLastError());
    return 0;
  };
  auto nonzero = [&]() -> int { // bp4_all_zero without the host round trip
    CU(cudaMemsetAsync(c->d_flag.get(), 0, sizeof(int), c->st()));
    return sweep(c, BP4_K_BLAS1, n, bp4::nonzero_kernel, n, (const double *)x, c->d_flag.get());
  };
  if (int e = capture_into(c, graph, nullptr, 0, nonzero, &leaves))
    return e;
  SolveArgs             a(st, c->d_flag.get(), 0u, 0., 0., nullptr, nullptr, sg.apply);
  cudaKernelNodeParams  kp = a.params();
  CU(cudaGraphAddKernelNode(&sg.begin, graph, leaves.data(), leaves.size(), &kp));
  c->launches += 1;
  cudaGraphNode_t apply_node;
  cudaGraph_t     apply_body;
  if (int e = add_conditional(graph, {sg.begin}, sg.apply, cudaGraphCondTypeIf, &apply_node, &apply_body))
    return e;
  if (int e = capture_into(c, apply_body, nullptr, 0, [&]() { return vmult_on(c, g, x); }, nullptr))
    return e;
  // g = 1 g - b or -b (bp4_add / bp4_equ), |g|^2 (bp4_dot), check(0); plain: h = P g, d = -h,
  // gh = g.h (SolverCG before its loop)
  auto step0 = [&]() -> int {
    if (int e = sweep(c, BP4_K_BLAS1, n, bp4::sadd_kernel<true>, n, g, 0., -1., sg.b, &st->g_scale))
      return e;
    if (int e = sweep(c, BP4_K_BLAS1, n, c->deterministic ? bp4::dot_kernel<true> : bp4::dot_kernel<false>, n,
                      (const double *)g, (const double *)g, acc, c->det))
      return e;
    {
      Timed t(c, BP4_K_BLAS1);
      bp4::solve_step0_kernel<<<1, 32, 0, c->st()>>>(st, acc, loop, iterated);
      CU(cudaGetLastError());
    }
    if (sg.merged)
      return 0;
    if (int e = jacobi_dot())
      return e;
    if (int e = scalar(bp4::kSolvePlainInit))
      return e;
    return sweep(c, BP4_K_BLAS1, n, bp4::sadd_kernel<false>, n, d, 0., -1., h, nullptr);
  };
  if (int e = capture_into(c, graph, &apply_node, 1, step0, &leaves))
    return e;
  cudaGraphNode_t cond;
  cudaGraph_t     loop_body;
  if (int e = add_conditional(graph, leaves, loop, cudaGraphCondTypeWhile, &cond, &loop_body))
    return e;
  auto body = [&]() -> int {
    if (sg.merged)
      {
        const MergedCall m{x, g, d, prec, 0., 0., 0., 0., st};
        if (int e = merged_sweep(c, m, h))
          return e;
        return scalar(bp4::kSolveMergedStep);
      }
    // SolverCG: h = A d; alpha = gh / d.h; x += alpha d; g += alpha h, |g|; check;
    // h = P g; beta = g.h / gh; d = beta d - h
    if (int e = vmult_on(c, h, d))
      return e;
    if (int e = sweep(c, BP4_K_BLAS1, n, c->deterministic ? bp4::dot_kernel<true> : bp4::dot_kernel<false>, n, d,
                      h, acc, c->det))
      return e;
    if (int e = scalar(bp4::kSolvePlainAlpha))
      return e;
    if (int e = sweep(c, BP4_K_BLAS1, n, c->deterministic ? bp4::cg_xg_kernel<true> : bp4::cg_xg_kernel<false>, n, x,
                      g, d, h, st, acc + 1, c->det))
      return e;
    if (int e = jacobi_dot())
      return e;
    if (int e = scalar(bp4::kSolvePlainCheck))
      return e;
    return sweep(c, BP4_K_BLAS1, n, bp4::sadd_kernel<true>, n, d, 0., -1., h, &st->beta);
  };
  if (int e = capture_into(c, loop_body, nullptr, 0, body, nullptr))
    return e;
  // merged: the pending x update, after at least one iteration
  cudaGraphNode_t last = cond;
  if (sg.merged)
    {
      cudaGraph_t fin_body;
      if (int e = add_conditional(graph, {cond}, iterated, cudaGraphCondTypeIf, &last, &fin_body))
        return e;
      auto fin = [&]() {
        return sweep(c, BP4_K_BLAS1, n, c->deterministic ? bp4::solve_final_kernel<true> : bp4::solve_final_kernel<false>,
                     n, x, d, g, prec, st);
      };
      if (int e = capture_into(c, fin_body, nullptr, 0, fin, nullptr))
        return e;
    }
  auto result = [&]() -> int {
    Timed t(c, BP4_K_BLAS1);
    bp4::solve_result_kernel<<<1, 32, 0, c->st()>>>(st);
    CU(cudaGetLastError());
    return 0;
  };
  if (int e = capture_into(c, graph, &last, 1, result, nullptr))
    return e;
  cudaGraphExec_t exec;
  CU(cudaGraphInstantiate(&exec, graph, 0));
  sg.exec.reset(exec);
  return 0;
}

// p must be readable and writable by the context's kernels: device memory of its device, or
// mapped pinned host memory (*dev receives its device address); 8-byte aligned
static int device_visible(const bp4_ctx *c, void *p, const char *name, void **dev)
{
  if (reinterpret_cast<uintptr_t>(p) % 8)
    return fail(BP4_ERR_ARG, "%s: %p is not 8-byte aligned", name, p);
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess)
    {
      cudaGetLastError();
      at.type = cudaMemoryTypeUnregistered;
    }
  if (at.type == cudaMemoryTypeDevice && at.device == c->device)
    *dev = p;
  else if (at.type == cudaMemoryTypeHost && at.devicePointer)
    *dev = at.devicePointer;
  else
    return fail(BP4_ERR_ARG, "%s: %p is neither device memory of device %d nor mapped pinned host memory (memory "
                             "type %d, device %d)", name, p, c->device, (int)at.type, at.device);
  return 0;
}

static int solve_async(bp4_ctx *c, const bool merged, bp4_vec *x, const bp4_vec *b, const bp4_vec *prec,
                       const unsigned max_steps, const double tol, const double reduce, bp4_solve_result *result,
                       double *history)
{
  if (!c || !result)
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
  if (int e = refuse_capture(c, merged ? "bp4_solve_cg_merged" : "bp4_solve_cg"))
    return e;
  void *res_dev = nullptr, *hist_dev = nullptr;
  if (int e = device_visible(c, result, "result", &res_dev))
    return e;
  if (history)
    if (int e = device_visible(c, history, "history", &hist_dev))
      return e;
  SolveGraph *sg = nullptr;
  for (SolveGraph &e : c->solves)
    if (e.merged == merged && e.fused == c->fused && e.x == x->p() && e.b == b->p() && e.prec == prec->p())
      sg = &e;
  if (!sg) // the entry goes into the cache once its temporaries are allocated
    {
      SolveGraph ns;
      ns.merged = merged, ns.fused = c->fused, ns.x = x->p(), ns.b = b->p(), ns.prec = prec->p();
      for (bp4_vec *v : {&ns.g, &ns.d, &ns.h})
        if (int e = pooled_alloc(c, c->n_owned + c->n_ghost, *v, false))
          return e;
      c->solves.push_back(std::move(ns));
      sg = &c->solves.back();
    }
  if (!sg->exec)
    if (int e = build_solve_graph(c, *sg))
      {
        sg->graph.reset(); // a later call starts over
        return e;
      }
  // this launch's arguments; launches queued before keep theirs
  SolveArgs            a(c->d_state.get(), c->d_flag.get(), max_steps, tol, reduce, static_cast<double *>(hist_dev),
                         res_dev, sg->apply);
  cudaKernelNodeParams kp = a.params();
  CU(cudaGraphExecKernelNodeSetParams(sg->exec.get(), sg->begin, &kp));
  CU(cudaGraphLaunch(sg->exec.get(), c->st()));
  c->launches += 1;
  return 0;
}

// the enqueued solve, then a wait for its result in the context's pinned result block
static int solve_blocking(bp4_ctx *c, const bool merged, bp4_vec *x, const bp4_vec *b, const bp4_vec *prec,
                          const unsigned max_steps, const double tol, const double reduce, bp4_solve_result *out)
{
  if (!c || !out)
    return fail(BP4_ERR_ARG, "null argument");
  if (int e = solve_async(c, merged, x, b, prec, max_steps, tol, reduce, c->h_result.get(), nullptr))
    return e;
  CU(cudaStreamSynchronize(c->st()));
  *out = *c->h_result;
  return 0;
}

int bp4_solve_cg(bp4_ctx *c, bp4_vec *x, const bp4_vec *b, const bp4_vec *prec, unsigned max_steps, double tol,
                 double reduce, bp4_solve_result *out)
{
  return solve_blocking(c, false, x, b, prec, max_steps, tol, reduce, out);
}

int bp4_solve_cg_merged(bp4_ctx *c, bp4_vec *x, const bp4_vec *b, const bp4_vec *prec, unsigned max_steps,
                        double tol, double reduce, bp4_solve_result *out)
{
  return solve_blocking(c, true, x, b, prec, max_steps, tol, reduce, out);
}

int bp4_solve_cg_async(bp4_ctx *c, bp4_vec *x, const bp4_vec *b, const bp4_vec *prec, unsigned max_steps, double tol,
                       double reduce, bp4_solve_result *result, double *history)
{
  return solve_async(c, false, x, b, prec, max_steps, tol, reduce, result, history);
}

int bp4_solve_cg_merged_async(bp4_ctx *c, bp4_vec *x, const bp4_vec *b, const bp4_vec *prec, unsigned max_steps,
                              double tol, double reduce, bp4_solve_result *result, double *history)
{
  return solve_async(c, true, x, b, prec, max_steps, tol, reduce, result, history);
}

// ---- mixed-precision solve ---------------------------------------------------------------
// The FP32 paths run on one rank outside the deterministic mode (no ghost exchange of float
// vectors, no ordered FP32 reductions)
static int refuse_f32(const bp4_ctx *c, const char *call)
{
  if (!c->peer.empty() || c->n_ranks > 1)
    return fail(BP4_ERR_STATE, "%s runs on one rank: this context has a ghost-exchange plan or a communicator over "
                               "several ranks", call);
  if (c->deterministic)
    return fail(BP4_ERR_STATE, "%s: the deterministic mode has no FP32 path (its ordered reductions are FP64 only)",
                call);
  return 0;
}

// the float copy of the geometry coefficients, made on first use
static int ensure_coef32(bp4_ctx *c)
{
  if (c->d_coef32)
    return 0;
  const uint64_t n = (uint64_t)c->n_coef * std::max<uint64_t>(c->n_cells, 1);
  CU(allocate(c->d_coef32, n));
  return sweep(c, BP4_K_BLAS1, n, bp4::narrow_kernel, n, (const double *)c->d_coef.get(), c->d_coef32.get());
}

// dst += sum_cells A_cell src with the FP32 cell kernel, all cells (one rank)
static int cell_loop_f32(bp4_ctx *c, float *dst, const float *src)
{
  CU(cudaMemsetAsync(c->d_sched.get(), 0, sizeof(uint32_t) * c->n_sched, c->st()));
  if (c->n_cells == 0)
    return 0;
  bp4::CellArgsT<float> a{};
  a.entity_index = c->d_entity.get();
  a.coef         = c->d_coef32.get();
  a.dtab         = c->d_walk.get();
  a.n_cells      = c->n_cells;
  a.src          = src;
  a.dst          = dst;
  a.sched        = c->d_sched.get();
  Timed t(c, BP4_K_VMULT);
  CU(bp4::launch_cell_f32(c->degree, c->n_coef == 81, a, c->sms, c->st()));
  return 0;
}

int bp4_debug_vmult_f32(bp4_ctx *c, bp4_vec *dst, const bp4_vec *src)
{
  if (!c)
    return fail(BP4_ERR_ARG, "null ctx");
  if (int e = check_len(c, dst, "dst"))
    return e;
  if (int e = check_len(c, src, "src"))
    return e;
  if (dst == src)
    return fail(BP4_ERR_ARG, "vmult: dst aliases src");
  if (int e = refuse_f32(c, "bp4_debug_vmult_f32"))
    return e;
  if (int e = refuse_capture(c, "bp4_debug_vmult_f32"))
    return e;
  CU(cudaSetDevice(c->device));
  if (int e = ensure_coef32(c))
    return e;
  const uint64_t n = c->n_owned + c->n_ghost;
  dev_ptr<float> s32, d32;
  CU(allocate(s32, n));
  CU(allocate(d32, n));
  if (int e = sweep(c, BP4_K_BLAS1, n, bp4::narrow_kernel, n, (const double *)src->p(), s32.get()))
    return e;
  CU(cudaMemsetAsync(d32.get(), 0, sizeof(float) * n, c->st()));
  if (int e = cell_loop_f32(c, d32.get(), s32.get()))
    return e;
  {
    Timed t(c, BP4_K_BLAS1);
    if (int e = per_element(c, c->n_constrained, bp4::fixup_kernel<float>, c->n_constrained, c->d_constrained.get(),
                            d32.get(), (const float *)s32.get()))
      return e;
  }
  if (int e = sweep(c, BP4_K_BLAS1, n, bp4::widen_kernel, n, (const float *)d32.get(), dst->p()))
    return e;
  CU(cudaStreamSynchronize(c->st())); // the float temporaries are freed on return
  return 0;
}

// the per-call arguments of a mixed solve, as the parameters of its mixed_begin_kernel node
struct MixedArgs
{
  bp4::MixedState           *st;
  const int                 *nonzero;
  uint32_t                   max_steps;
  double                     tol, reduce;
  double                    *history;
  void                      *result;
  cudaGraphConditionalHandle apply;
  void                      *ptr[8] = {&st, &nonzero, &max_steps, &tol, &reduce, &history, &result, &apply};
  MixedArgs(const MixedArgs &) = delete; // ptr points into this object
  MixedArgs(bp4::MixedState *st_, const int *nz, uint32_t ms, double t, double r, double *hi, void *re,
            cudaGraphConditionalHandle ap)
    : st(st_), nonzero(nz), max_steps(ms), tol(t), reduce(r), history(hi), result(re), apply(ap)
  {}
  cudaKernelNodeParams params()
  {
    cudaKernelNodeParams kp = {};
    kp.func                 = reinterpret_cast<void *>(bp4::mixed_begin_kernel);
    kp.gridDim              = dim3(1);
    kp.blockDim             = dim3(32);
    kp.kernelParams         = ptr;
    return kp;
  }
};

// One CUDA graph per mixed solve (conditional nodes nest: CUDA 12.4 and later allow conditional
// nodes in conditional bodies, and every handle is created on the top-level graph, the graph "or one
// of its children" that holds its node):
//   x != 0? -> mixed_begin -> IF apply { g = A x } -> prec32 = (float) prec
//   -> WHILE loop { g = g_scale g - b, |g|, check
//                   IF go { r32 = s g, e = 0, WHILE inner { FP32 merged iteration }, final e update,
//                           x += e / s, g = A x } }
//   -> result to the caller.
// The FP64 pieces are the kernels of the device-resident solves; the inner iteration is merged_sweep's
// streamed form on float vectors with the FP32 cell kernel, driven by solve_scalar_kernel on ms.inner.
static int build_mixed_graph(bp4_ctx *c, MixedGraph &mg)
{
  const uint64_t   n   = c->n_owned, nl = c->n_owned + c->n_ghost;
  double          *x   = const_cast<double *>(mg.x), *g = mg.g.p();
  bp4::MixedState *ms  = c->d_mixed.get();
  double          *acc = c->d_acc.get();
  float *r32 = mg.r32.get(), *d32 = mg.d32.get(), *h32 = mg.h32.get(), *e32 = mg.e32.get(), *p32 = mg.prec32.get();
  cudaGraph_t graph;
  CU(cudaGraphCreate(&graph, 0));
  mg.graph.reset(graph);
  cudaGraphConditionalHandle loop, go, inner;
  CU(cudaGraphConditionalHandleCreate(&mg.apply, graph, 0, cudaGraphCondAssignDefault));
  CU(cudaGraphConditionalHandleCreate(&loop, graph, 1, cudaGraphCondAssignDefault));
  CU(cudaGraphConditionalHandleCreate(&go, graph, 0, cudaGraphCondAssignDefault));
  CU(cudaGraphConditionalHandleCreate(&inner, graph, 0, cudaGraphCondAssignDefault));
  std::vector<cudaGraphNode_t> leaves;
  auto nonzero = [&]() -> int {
    CU(cudaMemsetAsync(c->d_flag.get(), 0, sizeof(int), c->st()));
    return sweep(c, BP4_K_BLAS1, n, bp4::nonzero_kernel, n, (const double *)x, c->d_flag.get());
  };
  if (int e = capture_into(c, graph, nullptr, 0, nonzero, &leaves))
    return e;
  MixedArgs            a(ms, c->d_flag.get(), 0u, 0., 0., nullptr, nullptr, mg.apply);
  cudaKernelNodeParams kp = a.params();
  CU(cudaGraphAddKernelNode(&mg.begin, graph, leaves.data(), leaves.size(), &kp));
  c->launches += 1;
  cudaGraphNode_t apply_node;
  cudaGraph_t     apply_body;
  if (int e = add_conditional(graph, {mg.begin}, mg.apply, cudaGraphCondTypeIf, &apply_node, &apply_body))
    return e;
  if (int e = capture_into(c, apply_body, nullptr, 0, [&]() { return vmult_on(c, g, x); }, nullptr))
    return e;
  auto narrow_prec = [&]() {
    return sweep(c, BP4_K_BLAS1, n / 3, bp4::narrow_kernel, n / 3, mg.prec, p32);
  };
  if (int e = capture_into(c, graph, &apply_node, 1, narrow_prec, &leaves))
    return e;
  cudaGraphNode_t loop_node;
  cudaGraph_t     loop_body;
  if (int e = add_conditional(graph, leaves, loop, cudaGraphCondTypeWhile, &loop_node, &loop_body))
    return e;
  // refinement step: the FP64 true residual and its check
  auto check = [&]() -> int {
    if (int e = sweep(c, BP4_K_BLAS1, n, bp4::sadd_kernel<true>, n, g, 0., -1., mg.b, &ms->outer.g_scale))
      return e;
    if (int e = sweep(c, BP4_K_BLAS1, n, bp4::dot_kernel<false>, n, (const double *)g, (const double *)g, acc, c->det))
      return e;
    Timed t(c, BP4_K_BLAS1);
    bp4::mixed_check_kernel<<<1, 32, 0, c->st()>>>(ms, acc, loop, go);
    CU(cudaGetLastError());
    return 0;
  };
  if (int e = capture_into(c, loop_body, nullptr, 0, check, &leaves))
    return e;
  cudaGraphNode_t go_node;
  cudaGraph_t     go_body;
  if (int e = add_conditional(loop_body, leaves, go, cudaGraphCondTypeIf, &go_node, &go_body))
    return e;
  auto start = [&]() -> int { // r32 = s (A x - b), e = 0; sets `inner`
    if (int e = sweep(c, BP4_K_BLAS1, n, bp4::mixed_residual_kernel, n, r32, (const double *)g,
                      (const bp4::MixedState *)ms, inner))
      return e;
    CU(cudaMemsetAsync(e32, 0, sizeof(float) * nl, c->st()));
    return 0;
  };
  if (int e = capture_into(c, go_body, nullptr, 0, start, &leaves))
    return e;
  cudaGraphNode_t inner_node;
  cudaGraph_t     inner_body;
  if (int e = add_conditional(go_body, leaves, inner, cudaGraphCondTypeWhile, &inner_node, &inner_body))
    return e;
  // one FP32 merged iteration: merged_sweep's streamed form (pre, cells, post) and the scalar step
  auto iteration = [&]() -> int {
    bp4::SolveState *in = &ms->inner;
    if (int e = sweep(c, BP4_K_PRE, std::max<uint64_t>(n, 1), bp4::pre_kernel<true, float>, (uint64_t)0, n, h32, e32,
                      r32, d32, (const float *)p32, 0., 0., 0., 0., acc, c->d_update4b.get(), (const bp4::SolveState *)in))
      return e;
    if (c->n_ghost)
      CU(cudaMemsetAsync(h32 + n, 0, sizeof(float) * c->n_ghost, c->st()));
    if (int e = cell_loop_f32(c, h32, d32))
      return e;
    if (n)
      if (int e = sweep(c, BP4_K_POST, n, bp4::post_kernel<false, float>, (uint64_t)0, n, (const float *)r32,
                        (const float *)d32, (const float *)h32, (const float *)p32, acc, c->det))
        return e;
    Timed t(c, BP4_K_BLAS1);
    bp4::solve_scalar_kernel<<<1, 32, 0, c->st()>>>(bp4::kSolveMergedStep, in, acc, inner);
    CU(cudaGetLastError());
    return 0;
  };
  if (int e = capture_into(c, inner_body, nullptr, 0, iteration, nullptr))
    return e;
  // the inner solve's pending e update, x += e / s, and A x for the next refinement step
  auto finish = [&]() -> int {
    if (int e = sweep(c, BP4_K_BLAS1, n, bp4::solve_final_kernel<false, float>, n, e32, (const float *)d32,
                      (const float *)r32, (const float *)p32, (const bp4::SolveState *)&ms->inner))
      return e;
    if (int e = sweep(c, BP4_K_BLAS1, n, bp4::mixed_update_kernel, n, x, (const float *)e32,
                      (const bp4::MixedState *)ms))
      return e;
    return vmult_on(c, g, x);
  };
  if (int e = capture_into(c, go_body, &inner_node, 1, finish, nullptr))
    return e;
  auto result = [&]() -> int {
    Timed t(c, BP4_K_BLAS1);
    bp4::mixed_result_kernel<<<1, 32, 0, c->st()>>>(ms);
    CU(cudaGetLastError());
    return 0;
  };
  if (int e = capture_into(c, graph, &loop_node, 1, result, nullptr))
    return e;
  cudaGraphExec_t exec;
  CU(cudaGraphInstantiate(&exec, graph, 0));
  mg.exec.reset(exec);
  return 0;
}

int bp4_solve_cg_mixed_async(bp4_ctx *c, bp4_vec *x, const bp4_vec *b, const bp4_vec *prec, unsigned max_steps,
                             double tol, double reduce, bp4_mixed_result *result, double *history)
{
  if (!c || !result)
    return fail(BP4_ERR_ARG, "null argument");
  if (int e = check_len(c, x, "x"))
    return e;
  if (int e = check_len(c, b, "b"))
    return e;
  if (!prec || 3 * prec->n < c->n_owned)
    return fail(BP4_ERR_ARG, "prec needs n_owned/3 entries");
  if (x == b)
    return fail(BP4_ERR_ARG, "solve: x aliases b");
  if (int e = refuse_f32(c, "bp4_solve_cg_mixed"))
    return e;
  CU(cudaSetDevice(c->device));
  if (int e = refuse_capture(c, "bp4_solve_cg_mixed"))
    return e;
  void *res_dev = nullptr, *hist_dev = nullptr;
  if (int e = device_visible(c, result, "result", &res_dev))
    return e;
  if (history)
    if (int e = device_visible(c, history, "history", &hist_dev))
      return e;
  if (!c->d_mixed)
    CU(allocate(c->d_mixed, 1));
  if (int e = ensure_coef32(c))
    return e;
  MixedGraph *mg = nullptr;
  for (MixedGraph &e : c->mixed)
    if (e.x == x->p() && e.b == b->p() && e.prec == prec->p())
      mg = &e;
  if (!mg) // the entry goes into the cache once its temporaries are allocated
    {
      const uint64_t nl = c->n_owned + c->n_ghost;
      MixedGraph     ns;
      ns.x = x->p(), ns.b = b->p(), ns.prec = prec->p();
      if (int e = pooled_alloc(c, nl, ns.g, false))
        return e;
      for (dev_ptr<float> *v : {&ns.r32, &ns.d32, &ns.h32, &ns.e32})
        CU(allocate(*v, nl));
      CU(allocate(ns.prec32, c->n_owned / 3));
      c->mixed.push_back(std::move(ns));
      mg = &c->mixed.back();
    }
  if (!mg->exec)
    if (int e = build_mixed_graph(c, *mg))
      {
        mg->graph.reset(); // a later call starts over
        return e;
      }
  MixedArgs            a(c->d_mixed.get(), c->d_flag.get(), max_steps, tol, reduce, static_cast<double *>(hist_dev),
                         res_dev, mg->apply);
  cudaKernelNodeParams kp = a.params();
  CU(cudaGraphExecKernelNodeSetParams(mg->exec.get(), mg->begin, &kp));
  CU(cudaGraphLaunch(mg->exec.get(), c->st()));
  c->launches += 1;
  return 0;
}

int bp4_solve_cg_mixed(bp4_ctx *c, bp4_vec *x, const bp4_vec *b, const bp4_vec *prec, unsigned max_steps, double tol,
                       double reduce, bp4_mixed_result *out)
{
  if (!c || !out)
    return fail(BP4_ERR_ARG, "null argument");
  if (!c->h_mixed)
    {
      if (int e = refuse_capture(c, "bp4_solve_cg_mixed"))
        return e;
      CU(cudaSetDevice(c->device));
      CU(allocate(c->h_mixed, 1));
    }
  if (int e = bp4_solve_cg_mixed_async(c, x, b, prec, max_steps, tol, reduce, c->h_mixed.get(), nullptr))
    return e;
  CU(cudaStreamSynchronize(c->st()));
  *out = *c->h_mixed;
  return 0;
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
  CU(allocate(p.arena, off));
  CU(cudaMemset(p.arena.get(), 0, off));
  CU(cudaIpcGetMemHandle(&mine.handle, p.arena.get()));
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
  dev_ptr<P2PCard> d_mine, d_all;
  CU(upload(d_mine, &mine, 1));
  CU(allocate(d_all, c->n_ranks));
  NC(ncclAllGather(d_mine.get(), d_all.get(), sizeof(P2PCard), ncclChar, c->comm.get(), c->st()));
  CU(cudaStreamSynchronize(c->st()));
  std::vector<P2PCard> all(c->n_ranks);
  CU(cudaMemcpy(all.data(), d_all.get(), sizeof(P2PCard) * c->n_ranks, cudaMemcpyDeviceToHost));
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
      p.peer_arena.emplace_back((char *)base);
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
  int          h_ok = ok ? 1 : 0;
  dev_ptr<int> d_ok;
  CU(upload(d_ok, &h_ok, 1));
  NC(ncclAllReduce(d_ok.get(), d_ok.get(), 1, ncclInt, ncclMin, c->comm.get(), c->st()));
  CU(cudaStreamSynchronize(c->st()));
  CU(cudaMemcpy(&h_ok, d_ok.get(), sizeof(int), cudaMemcpyDeviceToHost));
  p.on = h_ok == 1;
  return 0;
}

int bp4_comm_init(bp4_ctx *c, int rank, int n_ranks, const unsigned char id[BP4_NCCL_ID_BYTES])
{
  if (!c || !id)
    return fail(BP4_ERR_ARG, "null argument");
  if (int e = refuse_capture(c, "bp4_comm_init"))
    return e;
  if (c->deterministic && n_ranks > 1)
    return fail(BP4_ERR_STATE, "the deterministic mode runs on one rank");
  if (c->comm)
    return fail(BP4_ERR_STATE, "the communicator is already initialised (rank %d of %d): bp4_comm_init may be "
                               "called once per context", c->rank, c->n_ranks);
  CU(cudaSetDevice(c->device));
  ncclUniqueId u;
  memcpy(&u, id, sizeof(u));
  ncclComm_t comm;
  NC(ncclCommInitRank(&comm, n_ranks, u, rank));
  c->comm.reset(comm);
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
            DRV(p.wait64((CUstream)st, flag_addr(p.arena.get(), kFlagAckFwd, c->peer[k]), e - 2, CU_STREAM_WAIT_VALUE_GEQ));
          CU(cudaMemcpyAsync(p.peer_arena[k].get() + p.peer_off_ghost[b][k] + sizeof(double) * p.peer_imp_off[k],
                             c->d_sendbuf.get() + c->export_off[k], sizeof(double) * ns, cudaMemcpyDeviceToDevice, st));
          DRV(p.write64((CUstream)st, flag_addr(p.peer_arena[k].get(), kFlagDataFwd, c->rank), e, CU_STREAM_WRITE_VALUE_DEFAULT));
        }
      for (size_t k = 0; k < c->peer.size(); ++k)
        {
          const uint64_t nr = c->import_off[k + 1] - c->import_off[k];
          if (!nr)
            continue;
          DRV(p.wait64((CUstream)st, flag_addr(p.arena.get(), kFlagDataFwd, c->peer[k]), e, CU_STREAM_WAIT_VALUE_GEQ));
          CU(cudaMemcpyAsync(v + c->n_owned + c->import_off[k],
                             p.arena.get() + p.off_ghost[b] + sizeof(double) * c->import_off[k], sizeof(double) * nr,
                             cudaMemcpyDeviceToDevice, st));
          DRV(p.write64((CUstream)st, flag_addr(p.peer_arena[k].get(), kFlagAckFwd, c->rank), e, CU_STREAM_WRITE_VALUE_DEFAULT));
        }
      return 0;
    }
  NC(ncclGroupStart());
  for (size_t k = 0; k < c->peer.size(); ++k)
    {
      const uint64_t ns = c->export_off[k + 1] - c->export_off[k], nr = c->import_off[k + 1] - c->import_off[k];
      if (ns)
        NC(ncclSend(c->d_sendbuf.get() + c->export_off[k], ns, ncclDouble, c->peer[k], c->comm.get(), st));
      if (nr)
        NC(ncclRecv(v + c->n_owned + c->import_off[k], nr, ncclDouble, c->peer[k], c->comm.get(), st));
    }
  NC(ncclGroupEnd());
  return 0;
}

// compress(add) on stream st: the ghost slots of v travel to their owners; the owner side ends
// with the contributions in contrib_buffer(c) ready for compress_finish
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
            DRV(p.wait64((CUstream)st, flag_addr(p.arena.get(), kFlagAckRev, c->peer[k]), e - 2, CU_STREAM_WAIT_VALUE_GEQ));
          CU(cudaMemcpyAsync(p.peer_arena[k].get() + p.peer_off_contrib[b][k] + sizeof(double) * p.peer_exp_off[k],
                             v + c->n_owned + c->import_off[k], sizeof(double) * ns, cudaMemcpyDeviceToDevice, st));
          DRV(p.write64((CUstream)st, flag_addr(p.peer_arena[k].get(), kFlagDataRev, c->rank), e, CU_STREAM_WRITE_VALUE_DEFAULT));
        }
      for (size_t k = 0; k < c->peer.size(); ++k)
        if (c->export_off[k + 1] > c->export_off[k])
          DRV(p.wait64((CUstream)st, flag_addr(p.arena.get(), kFlagDataRev, c->peer[k]), e, CU_STREAM_WAIT_VALUE_GEQ));
      return 0;
    }
  NC(ncclGroupStart());
  for (size_t k = 0; k < c->peer.size(); ++k)
    {
      const uint64_t nr = c->export_off[k + 1] - c->export_off[k], ns = c->import_off[k + 1] - c->import_off[k];
      if (ns)
        NC(ncclSend(v + c->n_owned + c->import_off[k], ns, ncclDouble, c->peer[k], c->comm.get(), st));
      if (nr)
        NC(ncclRecv(c->d_recvbuf.get() + c->export_off[k], nr, ncclDouble, c->peer[k], c->comm.get(), st));
    }
  NC(ncclGroupEnd());
  return 0;
}

// where the contributions of the last compress exchange wait for unpack_add
static const double *contrib_buffer(const bp4_ctx *c)
{
  return c->p2p.on ? reinterpret_cast<const double *>(c->p2p.arena.get() + c->p2p.off_contrib[c->p2p.epoch_rev & 1])
                   : c->d_recvbuf.get();
}

// the end of compress(add) on the context's stream, once exchange_compress_on has delivered the
// contributions: add them into v, hand this half of contrib_in back to the ghost holders, zero the
// ghost slots of v
static int compress_finish(bp4_ctx *c, double *v)
{
  {
    // one launch for all peers: an owned entry may be exported to several (atomics)
    Timed          t(c, BP4_K_BLAS1);
    const uint64_t ne = c->export_off.back();
    if (int e = per_element(c, ne, bp4::unpack_add_kernel, ne, c->d_export.get(), contrib_buffer(c), v))
      return e;
  }
  auto &p = c->p2p;
  if (p.on)
    for (size_t k = 0; k < c->peer.size(); ++k)
      if (c->export_off[k + 1] > c->export_off[k])
        DRV(p.write64((CUstream)c->st(), flag_addr(p.peer_arena[k].get(), kFlagAckRev, c->rank), p.epoch_rev,
                      CU_STREAM_WRITE_VALUE_DEFAULT));
  CU(cudaMemsetAsync(v + c->n_owned, 0, sizeof(double) * c->n_ghost, c->st()));
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
    Timed          t(c, BP4_K_BLAS1);
    const uint64_t ne = c->export_off.back();
    if (int e = per_element(c, ne, bp4::pack_kernel, ne, c->d_export.get(), v->p(), c->d_sendbuf.get()))
      return e;
  }
  return exchange_ghosts_on(c, v->p(), c->st());
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
  if (int e = exchange_compress_on(c, v->p(), c->st()))
    return e;
  return compress_finish(c, v->p());
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
  if (int e = refuse_capture(c, "bp4_profile_enable"))
    return e;
  if (!on)
    CU(drain_events(c));
  c->profile = on != 0;
  return 0;
}

int bp4_profile_reset(bp4_ctx *c)
{
  if (!c)
    return fail(BP4_ERR_ARG, "null ctx");
  if (int e = refuse_capture(c, "bp4_profile_reset"))
    return e;
  CU(drain_events(c));
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
  if (int e = refuse_capture(c, "bp4_profile_get"))
    return e;
  CU(drain_events(c));
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
