// Raw (non-differentiable) data paths of the communicator: tensor -> backend
// routing, metadata exchange, plan construction.  The autograd layer
// (autograd_ops.cpp) wraps these.
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>

#include <nvtx3/nvToolsExt.h>

#include <algorithm>
#include <atomic>
#include <limits>
#include <numeric>

#include "../runtime/cuda_backend.h"
#include "communicator.h"

namespace m4t {

namespace {

DType to_dtype(at::ScalarType t) {
  switch (t) {
    case at::kByte: return DType::U8;
    case at::kChar: return DType::I8;
    case at::kShort: return DType::I16;
    case at::kInt: return DType::I32;
    case at::kLong: return DType::I64;
    case at::kFloat: return DType::F32;
    case at::kDouble: return DType::F64;
    case at::kBFloat16: return DType::BF16;
    case at::kHalf: return DType::F16;
    case at::kBool: return DType::BOOL;
    default: break;
  }
  throw std::invalid_argument(std::string("mpi4torch_b200: Failure to match torch::ScalarType ") +
                              c10::toString(t) + " to a transport dtype!");
}

ReduceOp to_op(int64_t op) {
  if (op < 0 || op >= static_cast<int64_t>(ReduceOp::kCount))
    throw std::invalid_argument("mpi4torch_b200: Collective operation not supported!");
  return static_cast<ReduceOp>(op);
}

// Decides which transport serves a tensor (reference MPIDeviceHelper,
// csrc/extension.cpp:61-104): CPU tensors -> shared-memory backend; CUDA
// tensors -> NVLink backend, or host staging when that is switched off.
struct Route {
  Backend* be = nullptr;
  void* stream = nullptr;
  bool staged = false;
  c10::Device device;
  c10::optional<c10::cuda::CUDAGuard> guard;

  Route(World& w, CommContext& cx, const Tensor& t) : device(t.device()) {
    if (t.is_cpu()) {
      be = &cx.host();
    } else if (t.is_cuda()) {
      if (!w.host_staging() && cx.cuda_ready()) {
        CudaBackend* cb = cx.cuda();
        TORCH_CHECK(t.device().index() == cb->device(), "mpi4torch_b200: tensor lives on cuda:",
                    static_cast<int>(t.device().index()), " but this rank's communicator is bound to cuda:", cb->device());
        guard.emplace(t.device());
        stream = c10::cuda::getCurrentCUDAStream(t.device().index()).stream();
        be = cb;
      } else {
        staged = true;
        be = &cx.host();
      }
    } else {
      TORCH_CHECK(false, "mpi4torch_b200: unsupported device ", t.device());
    }
  }
  Tensor to_comm(const Tensor& t) const {
    Tensor c = t.contiguous();
    return staged ? c.cpu() : c;
  }
  Tensor from_comm(const Tensor& t) const { return staged ? t.to(device) : t; }
};

// NVTX range per op (SURVEY 5.1): shows up in Nsight timelines / ncu range
// filters; costs nothing when no tool is attached.  M4T_NVTX=0 disables.
struct NvtxRange {
  bool on;
  explicit NvtxRange(const char* name) : on(nvtx_enabled()) {
    if (on) nvtxRangePushA(name);
  }
  ~NvtxRange() {
    if (on) nvtxRangePop();
  }
  static bool nvtx_enabled() {
    static const bool v = env_i64("M4T_NVTX", 1) != 0;
    return v;
  }
};

int64_t wrap_axis(int64_t axis, int64_t ndim, const char* what) {
  TORCH_CHECK(ndim > 0, "mpi4torch_b200: ", what, " needs a tensor with at least one dimension");
  TORCH_CHECK(axis >= -ndim && axis < ndim, "mpi4torch_b200: ", what, " axis ", axis, " out of range for a ", ndim,
              "-d tensor");
  return axis < 0 ? axis + ndim : axis;
}

// Largest per-rank staged payload one slab collective may move at once: the CUDA backend's staging half (every
// rank's share of a pull / reduce-scatter is staged there), unlimited on the shared-memory backend.
// M4T_SLAB_CHUNK_BYTES (read once) lowers it on any backend - used by the tests to drive the chunked paths.
std::atomic<int64_t> g_slab_chunked_calls{0};  // how often a slab collective had to be moved in pieces (introspection)

int64_t slab_limit_bytes(const Route& r, CommContext& cx) {
  static const int64_t forced = env_i64("M4T_SLAB_CHUNK_BYTES", 0);
  int64_t limit = std::numeric_limits<int64_t>::max();
  if (!r.staged && r.be != &cx.host() && cx.cuda_ready()) limit = cx.cuda()->half_bytes();
  if (forced > 0) limit = std::min(limit, forced);
  return limit;
}

// Suspends the AssumeUniformSizes promise for the pieces of a chunked call whose per-rank arguments differ
// (window pieces of a re-partition, placeholder tensors off the Scatter root).
struct UniformOff {
  bool& flag;
  bool saved;
  explicit UniformOff(bool& f) : flag(f), saved(f) { flag = false; }
  ~UniformOff() { flag = saved; }
};

uint32_t ptr_hash(const void* p) { return static_cast<uint32_t>(reinterpret_cast<uintptr_t>(p) & 0xffffffffu); }

}  // namespace

int64_t slab_chunked_calls() { return g_slab_chunked_calls.load(std::memory_order_relaxed); }

Communicator::Communicator() : world_(&World::instance()) {
  ctx_ = world_->ctx().get();
  rank_ = ctx_->rank();
  size_ = ctx_->size();
}

Communicator::Communicator(std::shared_ptr<CommContext> owned) : world_(&World::instance()), owned_(std::move(owned)) {
  is_world_ = false;
  ctx_ = owned_.get();
  rank_ = ctx_->rank();
  size_ = ctx_->size();
}

c10::intrusive_ptr<Communicator> Communicator::Split(int64_t color, int64_t key) {
  std::lock_guard<std::recursive_mutex> g(world_->mutex());
  // one metadata round: everybody learns everybody's (color, key)
  int64_t mine[2] = {color, key};
  std::vector<int64_t> all(static_cast<size_t>(size_) * 2);
  cx().allgather_i64(mine, 2, all.data());
  std::vector<std::pair<int64_t, int64_t>> members;  // (key, old rank)
  // a negative colour (MPI_UNDEFINED) still takes part in the exchange and gets
  // a communicator that contains only itself (MPI_COMM_SELF)
  for (int64_t p = 0; p < size_; ++p)
    if (color >= 0 ? all[p * 2] == color : p == rank_) members.emplace_back(all[p * 2 + 1], p);
  std::sort(members.begin(), members.end());
  int new_rank = -1;
  for (size_t i = 0; i < members.size(); ++i)
    if (members[i].second == rank_) new_rank = static_cast<int>(i);
  const uint64_t split_id = cx().next_split_id();  // identical on all ranks: Split is collective
  const std::string job = cx().job_id() + "_s" + std::to_string(split_id) +
                          (color >= 0 ? "c" + std::to_string(color) : "r" + std::to_string(rank_));
  std::shared_ptr<CommContext> child;
  if (cx().over_network()) {
    std::vector<int> world_ranks;
    for (const auto& m : members) world_ranks.push_back(cx().net()->members()[static_cast<size_t>(m.second)]);
    const int per_node = world_->ctx()->ranks_per_node();
    bool one_node = per_node > 0;
    for (int w : world_ranks) one_node = one_node && w / per_node == world_ranks[0] / per_node;
    if (one_node) {
      // all members live on one node: an ordinary shared-memory communicator - and, with a GPU per rank, the NVLink
      // backend (tensor parallelism inside the node, the world communicator across nodes)
      child = std::make_shared<CommContext>(new_rank, static_cast<int>(members.size()), job);
      if (world_->node_cuda_device() >= 0 && members.size() > 1)
        child->init_cuda(world_->node_cuda_device(), env_i64("M4T_SUB_STAGE_MB", 256), env_i64("M4T_SUB_SYMM_MB", 0));
    } else {
      // sub-communicator on the same TCP mesh: its own id keeps its frames apart from every other communicator's
      auto link = std::make_shared<NetLink>(cx().net()->engine_ptr(), net_comm_id(job), std::move(world_ranks), new_rank);
      child = std::make_shared<CommContext>(std::move(link), job);
    }
  } else {
    child = std::make_shared<CommContext>(new_rank, static_cast<int>(members.size()), job);
  }
  if (!cx().over_network() && cx().cuda_ready()) {
    // same device, smaller arenas than the world communicator's
    child->init_cuda(cx().cuda()->device(), env_i64("M4T_SUB_STAGE_MB", 256), env_i64("M4T_SUB_SYMM_MB", 0));
  }
  world_->register_child(child);
  return c10::make_intrusive<Communicator>(std::move(child));
}

void Communicator::Free() {
  TORCH_CHECK(!IsWorld(), "mpi4torch_b200: the world communicator cannot be freed");
  std::lock_guard<std::recursive_mutex> g(world_->mutex());
  if (!ctx_) return;
  world_->release_child(ctx_);
  ctx_ = nullptr;
  owned_.reset();  // the context's destructor performs the collective handshake
}

c10::intrusive_ptr<Communicator> comm_world() { return c10::make_intrusive<Communicator>(); }

void Communicator::Barrier() {
  std::lock_guard<std::recursive_mutex> g(world_->mutex());
  cx().barrier();
}

std::string Communicator::Describe() const {
  std::ostringstream o;
  o << "mpi4torch_b200 communicator rank " << rank_ << "/" << size_ << " job " << cx().job_id()
    << (cx().over_network() ? (cx().hierarchical() ? " | host: tcp mesh + shared memory inside the node (hierarchical Allreduce)"
                                                    : " | host: tcp mesh")
                            : " | cpu: posix-shm");
  if (cx().over_network()) o << " (job spans nodes; CUDA tensors are staged through host memory)";
  if (cx().cuda_ready()) o << " | " << cx().cuda()->describe();
  if (world_->host_staging()) o << " | host staging forced";
  return o.str();
}

Tensor Communicator::raw_allreduce(const Tensor& input, int64_t op_, double scale, bool has_scale,
                                   const c10::optional<Tensor>& accumulate) {
  NvtxRange nvtx_range_("m4t::Allreduce");
  const ReduceOp op = to_op(op_);
  const DType dt = to_dtype(input.scalar_type());
  check_op_dtype(op, dt);
  std::lock_guard<std::recursive_mutex> g(world_->mutex());
  Route r(*world_, cx(), input);
  Tensor in = r.to_comm(input);
  Tensor acc;
  Epilogue epi;
  epi.scale = scale;
  epi.has_scale = has_scale;
  if (accumulate.has_value() && accumulate->defined()) {
    TORCH_CHECK(accumulate->sizes() == input.sizes() && accumulate->scalar_type() == input.scalar_type() &&
                    accumulate->device() == input.device(),
                "mpi4torch_b200: accumulate tensor must match the input's shape, dtype and device");
    acc = r.to_comm(*accumulate);
    epi.accumulate = acc.data_ptr();
  }
  Tensor out = at::empty_like(in, at::MemoryFormat::Contiguous);
  r.be->allreduce(in.data_ptr(), out.data_ptr(), in.numel(), dt, op, epi, r.stream);
  return r.from_comm(out);
}

void Communicator::raw_allreduce_axpy_(Tensor& param, const Tensor& grad, double scale, int64_t max_blocks) {
  NvtxRange nvtx_range_("m4t::AllreduceAxpy");
  TORCH_CHECK(param.is_contiguous() && param.sizes() == grad.sizes() && param.scalar_type() == grad.scalar_type() &&
                  param.device() == grad.device(),
              "mpi4torch_b200: allreduce_axpy_ needs a contiguous parameter and a gradient of the same shape/dtype/device");
  const DType dt = to_dtype(param.scalar_type());
  std::lock_guard<std::recursive_mutex> g(world_->mutex());
  Route r(*world_, cx(), param);
  Tensor gin = r.to_comm(grad);
  Epilogue epi;
  epi.scale = scale;
  epi.has_scale = true;
  if (r.staged) {
    Tensor p = param.cpu();
    epi.accumulate = p.data_ptr();
    r.be->allreduce(gin.data_ptr(), p.data_ptr(), gin.numel(), dt, ReduceOp::SUM, epi, nullptr);
    param.copy_(p);
  } else {
    // out aliases accumulate: every element is read then written by the same thread
    epi.accumulate = param.data_ptr();
    CudaBackend* cb = dynamic_cast<CudaBackend*>(r.be);
    if (cb != nullptr && max_blocks > 0) {
      // small-footprint launch (few CTAs) so the collective can run under a GEMM
      // on another stream without evicting it; must be the same on every rank
      const int saved = cb->tuning().ar_blocks;
      cb->tuning().ar_blocks = static_cast<int>(max_blocks);
      try {
        r.be->allreduce(gin.data_ptr(), param.data_ptr(), gin.numel(), dt, ReduceOp::SUM, epi, r.stream);
      } catch (...) {
        cb->tuning().ar_blocks = saved;
        throw;
      }
      cb->tuning().ar_blocks = saved;
    } else {
      r.be->allreduce(gin.data_ptr(), param.data_ptr(), gin.numel(), dt, ReduceOp::SUM, epi, r.stream);
    }
  }
}

void Communicator::raw_bcast_(Tensor& work, int64_t root) {
  NvtxRange nvtx_range_("m4t::Bcast_");
  TORCH_CHECK(root >= 0 && root < size_, "mpi4torch_b200: Bcast_ root ", root, " out of range");
  const DType dt = to_dtype(work.scalar_type());
  std::lock_guard<std::recursive_mutex> g(world_->mutex());
  Route r(*world_, cx(), work);
  if (r.staged) {
    Tensor h = work.cpu();
    r.be->bcast(h.data_ptr(), h.numel(), dt, static_cast<int>(root), nullptr);
    work.copy_(h);
  } else {
    r.be->bcast(work.data_ptr(), work.numel(), dt, static_cast<int>(root), r.stream);
  }
}

void Communicator::raw_reduce_(Tensor& work, int64_t op_, int64_t root) {
  NvtxRange nvtx_range_("m4t::Reduce_");
  TORCH_CHECK(root >= 0 && root < size_, "mpi4torch_b200: Reduce_ root ", root, " out of range");
  const ReduceOp op = to_op(op_);
  const DType dt = to_dtype(work.scalar_type());
  check_op_dtype(op, dt);
  std::lock_guard<std::recursive_mutex> g(world_->mutex());
  Route r(*world_, cx(), work);
  if (r.staged) {
    Tensor h = work.cpu();
    r.be->reduce(h.data_ptr(), h.numel(), dt, op, static_cast<int>(root), nullptr);
    work.copy_(h);
  } else {
    r.be->reduce(work.data_ptr(), work.numel(), dt, op, static_cast<int>(root), r.stream);
  }
}

Tensor Communicator::raw_scan(const Tensor& input, int64_t op_, bool exclusive, bool reverse) {
  NvtxRange nvtx_range_(exclusive ? "m4t::Exscan" : "m4t::Scan");
  const ReduceOp op = to_op(op_);
  const DType dt = to_dtype(input.scalar_type());
  check_op_dtype(op, dt);
  std::lock_guard<std::recursive_mutex> g(world_->mutex());
  Route r(*world_, cx(), input);
  Tensor in = r.to_comm(input);
  Tensor out = at::empty_like(in, at::MemoryFormat::Contiguous);
  r.be->scan(in.data_ptr(), out.data_ptr(), in.numel(), dt, op, exclusive, reverse, r.stream);
  return r.from_comm(out);
}

void Communicator::exchange_meta(const int64_t* mine, int words, int64_t* all) {
  if (uniform_) {  // AssumeUniformSizes: every rank holds the same words, no host round
    for (int64_t p = 0; p < size_; ++p) std::copy(mine, mine + words, all + p * words);
    return;
  }
  cx().allgather_i64(mine, words, all);
}

Tensor Communicator::raw_gather(const Tensor& input, int64_t axis_, int64_t root, bool all) {
  NvtxRange nvtx_range_("m4t::Gather");
  TORCH_CHECK(all || (root >= 0 && root < size_), "mpi4torch_b200: Gather root ", root, " out of range");
  const DType dt = to_dtype(input.scalar_type());
  const int64_t axis = wrap_axis(axis_, input.dim(), all ? "Allgather" : "Gather");
  std::lock_guard<std::recursive_mutex> g(world_->mutex());
  Route r(*world_, cx(), input);
  Tensor in = r.to_comm(input);
  const auto shape = in.sizes().vec();
  const Axis3 a3 = split_axis(shape, axis);
  // one metadata round: [axis length, before, after]
  int64_t mine[3] = {a3.axis, a3.before, a3.after};
  std::vector<int64_t> allmeta(static_cast<size_t>(size_) * 3);
  exchange_meta(mine, 3, allmeta.data());
  std::vector<int64_t> lens(static_cast<size_t>(size_));
  for (int64_t p = 0; p < size_; ++p) {
    lens[p] = allmeta[p * 3];
    TORCH_CHECK(allmeta[p * 3 + 1] == a3.before && allmeta[p * 3 + 2] == a3.after,
                "mpi4torch_b200: ", all ? "Allgather" : "Gather", ": rank ", p,
                " has different non-gather dimensions than rank ", rank_);
  }
  const int rroot = all ? 0 : static_cast<int>(root);
  auto out_shape = shape;
  const bool i_receive = all || rank_ == root;
  // off-root the result has extent 0 along the gather axis (reference :538-554)
  const int64_t total_len = std::accumulate(lens.begin(), lens.end(), int64_t{0});
  out_shape[axis] = i_receive ? total_len : 0;
  // A rank's share larger than one staging half is moved in pieces (every rank sees the same lengths and the same
  // limit, so all ranks take the same decision): along `before` when whole rows fit, else along the gather axis.
  const int64_t es = static_cast<int64_t>(in.element_size());
  const int64_t max_len = *std::max_element(lens.begin(), lens.end());
  const int64_t limit = slab_limit_bytes(r, cx());
  if (a3.before * max_len * a3.after * es > limit && max_len > 0 && a3.after * es > limit && es <= limit) {
    // not even one row of the trailing dimensions fits: split those first, the pieces recurse into the splits below
    g_slab_chunked_calls.fetch_add(1, std::memory_order_relaxed);
    Tensor in3 = in.view({a3.before, a3.axis, a3.after});
    Tensor out = at::empty(out_shape, in.options());
    Tensor out3 = out.view({a3.before, i_receive ? total_len : 0, a3.after});
    const int64_t na = limit / es;
    for (int64_t c0 = 0; c0 < a3.after; c0 += na) {
      const int64_t n = std::min(na, a3.after - c0);
      Tensor part = raw_gather(in3.narrow(2, c0, n).contiguous(), 1, root, all);
      if (i_receive) out3.narrow(2, c0, n).copy_(part);
    }
    return r.from_comm(out);
  }
  if (a3.before * max_len * a3.after * es > limit && max_len > 0 && a3.after * es <= limit) {
    g_slab_chunked_calls.fetch_add(1, std::memory_order_relaxed);
    Tensor in3 = in.view({a3.before, a3.axis, a3.after});
    Tensor out = at::empty(out_shape, in.options());
    Tensor out3 = out.view({a3.before, i_receive ? total_len : 0, a3.after});
    const int64_t row_bytes = max_len * a3.after * es;  // one `before` row of the largest contributor
    if (a3.before > 1) {
      const int64_t nb = std::max<int64_t>(1, limit / std::max<int64_t>(row_bytes, 1));
      for (int64_t b0 = 0; b0 < a3.before; b0 += nb) {
        const int64_t n = std::min(nb, a3.before - b0);
        Tensor part = raw_gather(in3.narrow(0, b0, n), 1, root, all);  // recurses into the axis split if one row is too big
        if (i_receive) out3.narrow(0, b0, n).copy_(part);
      }
    } else {
      const int64_t nc = (row_bytes + limit - 1) / limit;
      std::vector<int64_t> displ(static_cast<size_t>(size_), 0);
      for (int64_t p = 1; p < size_; ++p) displ[p] = displ[p - 1] + lens[p - 1];
      for (int64_t k = 0; k < nc; ++k) {
        const int64_t r0 = a3.axis * k / nc, r1 = a3.axis * (k + 1) / nc;
        Tensor part = raw_gather(in3.narrow(1, r0, r1 - r0), 1, root, all);
        if (!i_receive) continue;
        int64_t toff = 0;
        for (int64_t p = 0; p < size_; ++p) {  // piece k of rank p goes to its place inside rank p's block
          const int64_t p0 = lens[p] * k / nc, p1 = lens[p] * (k + 1) / nc;
          if (p1 > p0) out3.narrow(1, displ[p] + p0, p1 - p0).copy_(part.narrow(1, toff, p1 - p0));
          toff += p1 - p0;
        }
      }
    }
    return r.from_comm(out);
  }
  PullPlan plan = plan_gather(static_cast<int>(rank_), static_cast<int>(size_), rroot, a3.before, a3.after, lens, all);
  Tensor out = at::empty(out_shape, in.options());
  r.be->pull(plan, in.data_ptr(), out.data_ptr(), dt, r.stream);
  return r.from_comm(out);
}

Tensor Communicator::raw_scatter(const Tensor& input, int64_t axis_, int64_t numelem, int64_t root) {
  NvtxRange nvtx_range_("m4t::Scatter");
  TORCH_CHECK(root >= 0 && root < size_, "mpi4torch_b200: Scatter root ", root, " out of range");
  TORCH_CHECK(numelem >= 0, "mpi4torch_b200: Scatter numelem must be non-negative");
  const DType dt = to_dtype(input.scalar_type());
  std::lock_guard<std::recursive_mutex> g(world_->mutex());
  Route r(*world_, cx(), input);
  Tensor in = r.to_comm(input);
  // one metadata round: [numelem, ndim, sizes...]; only root's shape matters
  // (off-root tensors are placeholders, reference :786-796).
  const int64_t nd = in.dim();
  TORCH_CHECK(nd + 2 <= kMetaWords, "mpi4torch_b200: tensor rank too large");
  std::vector<int64_t> mine(kMetaWords, 0);
  mine[0] = numelem;
  mine[1] = nd;
  for (int64_t i = 0; i < nd; ++i) mine[2 + i] = in.size(i);
  std::vector<int64_t> allmeta(static_cast<size_t>(size_) * kMetaWords);
  exchange_meta(mine.data(), kMetaWords, allmeta.data());
  const int64_t* rootmeta = allmeta.data() + root * kMetaWords;
  const int64_t rnd = rootmeta[1];
  std::vector<int64_t> rshape(rootmeta + 2, rootmeta + 2 + rnd);
  const int64_t axis = wrap_axis(axis_, rnd, "Scatter");
  std::vector<int64_t> counts(static_cast<size_t>(size_));
  int64_t total = 0;
  for (int64_t p = 0; p < size_; ++p) {
    counts[p] = allmeta[p * kMetaWords];
    total += counts[p];
  }
  // every rank sees the same numbers, so every rank raises (the reference only
  // raises on root, :835-837, leaving the others hanging)
  if (total != rshape[axis])
    throw std::invalid_argument("mpi4torch_b200: Scatter: sum of numelem (" + std::to_string(total) +
                                ") does not match the root tensor's axis length (" + std::to_string(rshape[axis]) + ")");
  const Axis3 a3 = split_axis(rshape, axis);
  auto out_shape = rshape;
  out_shape[axis] = numelem;
  {
    // root's whole tensor is staged: beyond a staging half it is moved in pieces - along `before` when whole rows fit,
    // else piece k of every destination's block (root concatenates them); off-root tensors stay placeholders
    const int64_t es = static_cast<int64_t>(in.element_size());
    const int64_t limit = slab_limit_bytes(r, cx());
    const int64_t row_bytes = a3.axis * a3.after * es;
    if (a3.before * row_bytes > limit && row_bytes > 0 && static_cast<int64_t>(size_) * a3.after * es > limit &&
        static_cast<int64_t>(size_) * es <= limit) {
      // one row per destination does not fit: split the trailing dimensions first
      g_slab_chunked_calls.fetch_add(1, std::memory_order_relaxed);
      UniformOff uniform_off(uniform_);  // off-root tensors are placeholders for the pieces
      const bool i_am_root = rank_ == root;
      Tensor in3 = i_am_root ? in.view({a3.before, a3.axis, a3.after}) : in;
      Tensor out = at::empty(out_shape, in.options());
      Tensor out3 = out.view({a3.before, numelem, a3.after});
      const int64_t na = limit / (es * static_cast<int64_t>(size_));
      for (int64_t c0 = 0; c0 < a3.after; c0 += na) {
        const int64_t n = std::min(na, a3.after - c0);
        Tensor part = raw_scatter(i_am_root ? in3.narrow(2, c0, n).contiguous() : in, 1, numelem, root);
        out3.narrow(2, c0, n).copy_(part.view({a3.before, numelem, n}));
      }
      return r.from_comm(out);
    }
    if (a3.before * row_bytes > limit && row_bytes > 0 && static_cast<int64_t>(size_) * a3.after * es <= limit) {
      g_slab_chunked_calls.fetch_add(1, std::memory_order_relaxed);
      UniformOff uniform_off(uniform_);  // off-root tensors are placeholders for the pieces
      const bool i_am_root = rank_ == root;
      Tensor in3 = i_am_root ? in.view({a3.before, a3.axis, a3.after}) : in;
      Tensor out = at::empty(out_shape, in.options());
      Tensor out3 = out.view({a3.before, numelem, a3.after});
      if (a3.before > 1) {
        const int64_t nb = std::max<int64_t>(1, limit / row_bytes);
        for (int64_t b0 = 0; b0 < a3.before; b0 += nb) {
          const int64_t n = std::min(nb, a3.before - b0);
          Tensor part = raw_scatter(i_am_root ? in3.narrow(0, b0, n) : in, 1, numelem, root);
          out3.narrow(0, b0, n).copy_(part.view({n, numelem, a3.after}));
        }
      } else {
        const int64_t nc = (row_bytes + limit - 1) / limit;
        std::vector<int64_t> displ(static_cast<size_t>(size_), 0);
        for (int64_t p = 1; p < size_; ++p) displ[p] = displ[p - 1] + counts[p - 1];
        for (int64_t k = 0; k < nc; ++k) {
          Tensor sub = in;
          if (i_am_root) {
            std::vector<Tensor> pieces;
            for (int64_t p = 0; p < size_; ++p) {
              const int64_t p0 = counts[p] * k / nc, p1 = counts[p] * (k + 1) / nc;
              pieces.push_back(in3.narrow(1, displ[p] + p0, p1 - p0));
            }
            sub = at::cat(pieces, 1);
          }
          const int64_t m0 = numelem * k / nc, m1 = numelem * (k + 1) / nc;
          Tensor part = raw_scatter(sub, 1, m1 - m0, root);
          if (m1 > m0) out3.narrow(1, m0, m1 - m0).copy_(part.view({1, m1 - m0, a3.after}));
        }
      }
      return r.from_comm(out);
    }
  }
  PullPlan plan = plan_scatter(static_cast<int>(rank_), static_cast<int>(size_), static_cast<int>(root), a3.before,
                               a3.after, counts);
  Tensor out = at::empty(out_shape, in.options());
  r.be->pull(plan, in.data_ptr(), out.data_ptr(), dt, r.stream);
  return r.from_comm(out);
}

Tensor Communicator::raw_alltoall(const Tensor& input, int64_t gatheraxis_, int64_t scatteraxis_, int64_t numelem) {
  NvtxRange nvtx_range_("m4t::Alltoall");
  TORCH_CHECK(numelem >= 0, "mpi4torch_b200: Alltoall numelem must be non-negative");
  const DType dt = to_dtype(input.scalar_type());
  const int64_t nd = input.dim();
  const int64_t gaxis = wrap_axis(gatheraxis_, nd, "Alltoall");
  const int64_t saxis = wrap_axis(scatteraxis_, nd, "Alltoall");
  std::lock_guard<std::recursive_mutex> g(world_->mutex());
  Route r(*world_, cx(), input);
  Tensor in = r.to_comm(input);
  const auto shape = in.sizes().vec();
  int64_t mine[2] = {numelem, shape[gaxis]};
  std::vector<int64_t> allmeta(static_cast<size_t>(size_) * 2);
  exchange_meta(mine, 2, allmeta.data());
  std::vector<int64_t> counts(static_cast<size_t>(size_)), glen(static_cast<size_t>(size_));
  for (int64_t p = 0; p < size_; ++p) {
    counts[p] = allmeta[p * 2];
    glen[p] = allmeta[p * 2 + 1];
  }
  PullPlan plan;
  auto out_shape = shape;
  if (gaxis == saxis) {
    const Axis3 a3 = split_axis(shape, gaxis);
    out_shape[gaxis] = numelem;
    {
      // re-partition of one global axis: beyond a staging half the global rows are exchanged window by window - every
      // rank contributes the rows it holds inside the window and asks for the rows it will own inside it
      const int64_t es = static_cast<int64_t>(in.element_size());
      const int64_t limit = slab_limit_bytes(r, cx());
      const int64_t row_bytes = a3.before * a3.after * es;  // one global row across `before`
      const int64_t max_len = *std::max_element(glen.begin(), glen.end());
      const int64_t total_rows = std::accumulate(glen.begin(), glen.end(), int64_t{0});
      const int64_t want_rows = std::accumulate(counts.begin(), counts.end(), int64_t{0});
      if (max_len * row_bytes > limit && row_bytes > 0 && row_bytes <= limit && total_rows == want_rows) {
        g_slab_chunked_calls.fetch_add(1, std::memory_order_relaxed);
        int64_t have0 = 0, own0 = 0;  // first global row I hold / I will own
        for (int64_t p = 0; p < rank_; ++p) {
          have0 += glen[p];
          own0 += counts[p];
        }
        const int64_t window = std::max<int64_t>(1, limit / row_bytes);
        Tensor out = at::empty(out_shape, in.options());
        // the pieces are not uniform across ranks even when the whole call is: the promise is suspended for them
        UniformOff uniform_off(uniform_);
        for (int64_t w0 = 0; w0 < total_rows; w0 += window) {
          const int64_t w1 = std::min(total_rows, w0 + window);
          const int64_t hlo = std::max(w0, have0), hhi = std::min(w1, have0 + glen[rank_]);
          const int64_t olo = std::max(w0, own0), ohi = std::min(w1, own0 + numelem);
          const int64_t hn = std::max<int64_t>(0, hhi - hlo), on = std::max<int64_t>(0, ohi - olo);
          Tensor sub = in.narrow(gaxis, hn > 0 ? hlo - have0 : 0, hn).contiguous();
          Tensor part = raw_alltoall(sub, gaxis, saxis, on);
          if (on > 0) out.narrow(gaxis, olo - own0, on).copy_(part);
        }
        return r.from_comm(out);
      }
    }
    plan = plan_repartition(static_cast<int>(rank_), static_cast<int>(size_), a3.before, a3.after, glen, counts);
  } else {
    const int64_t total = std::accumulate(counts.begin(), counts.end(), int64_t{0});
    if (total != shape[saxis])
      throw std::invalid_argument("mpi4torch_b200: Alltoall: sum of numelem (" + std::to_string(total) +
                                  ") does not match the scatter axis length (" + std::to_string(shape[saxis]) + ")");
    out_shape[gaxis] = std::accumulate(glen.begin(), glen.end(), int64_t{0});
    out_shape[saxis] = numelem;
    {
      // every rank's whole input is staged: beyond a staging half, rows [k/nc, (k+1)/nc) of every rank's gather axis
      // are exchanged per piece and land at their place inside that rank's block of the result
      const int64_t es = static_cast<int64_t>(in.element_size());
      const int64_t limit = slab_limit_bytes(r, cx());
      int64_t rest = es;  // bytes of one gather-axis row
      for (int64_t d = 0; d < nd; ++d)
        if (d != gaxis) rest *= shape[d];
      const int64_t max_len = *std::max_element(glen.begin(), glen.end());
      const int64_t per_dest = shape[saxis] > 0 ? rest / shape[saxis] * static_cast<int64_t>(size_) : 0;  // one scatter row per destination
      if (max_len * rest > limit && rest > limit && per_dest > 0 && per_dest <= limit) {
        // one gather-axis row does not fit: exchange piece k of every destination's block of the scatter axis
        g_slab_chunked_calls.fetch_add(1, std::memory_order_relaxed);
        const int64_t nc = (rest + limit - 1) / limit;
        std::vector<int64_t> sdispl(static_cast<size_t>(size_), 0);
        for (int64_t p = 1; p < size_; ++p) sdispl[p] = sdispl[p - 1] + counts[p - 1];
        Tensor out = at::empty(out_shape, in.options());
        for (int64_t k = 0; k < nc; ++k) {
          std::vector<Tensor> pieces;
          for (int64_t p = 0; p < size_; ++p) {
            const int64_t p0 = counts[p] * k / nc, p1 = counts[p] * (k + 1) / nc;
            pieces.push_back(in.narrow(saxis, sdispl[p] + p0, p1 - p0));
          }
          const int64_t m0 = numelem * k / nc, m1 = numelem * (k + 1) / nc;
          Tensor part = raw_alltoall(at::cat(pieces, saxis), gaxis, saxis, m1 - m0);
          if (m1 > m0) out.narrow(saxis, m0, m1 - m0).copy_(part);
        }
        return r.from_comm(out);
      }
      if (max_len * rest > limit && rest > 0 && rest <= limit) {
        g_slab_chunked_calls.fetch_add(1, std::memory_order_relaxed);
        const int64_t nc = (max_len * rest + limit - 1) / limit;
        std::vector<int64_t> displ(static_cast<size_t>(size_), 0);
        for (int64_t p = 1; p < size_; ++p) displ[p] = displ[p - 1] + glen[p - 1];
        Tensor out = at::empty(out_shape, in.options());
        for (int64_t k = 0; k < nc; ++k) {
          const int64_t r0 = shape[gaxis] * k / nc, r1 = shape[gaxis] * (k + 1) / nc;
          Tensor part = raw_alltoall(in.narrow(gaxis, r0, r1 - r0).contiguous(), gaxis, saxis, numelem);
          int64_t toff = 0;
          for (int64_t p = 0; p < size_; ++p) {
            const int64_t p0 = glen[p] * k / nc, p1 = glen[p] * (k + 1) / nc;
            if (p1 > p0) out.narrow(gaxis, displ[p] + p0, p1 - p0).copy_(part.narrow(gaxis, toff, p1 - p0));
            toff += p1 - p0;
          }
        }
        return r.from_comm(out);
      }
    }
    plan = plan_alltoall(static_cast<int>(rank_), static_cast<int>(size_), shape, gaxis, saxis, glen, counts);
  }
  Tensor out = at::empty(out_shape, in.options());
  r.be->pull(plan, in.data_ptr(), out.data_ptr(), dt, r.stream);
  return r.from_comm(out);
}

Tensor Communicator::raw_reduce_scatter(const Tensor& input, int64_t op_, int64_t axis_, int64_t numelem, double scale,
                                        bool has_scale, const c10::optional<Tensor>& accumulate) {
  NvtxRange nvtx_range_("m4t::Reduce_scatter");
  TORCH_CHECK(numelem >= 0, "mpi4torch_b200: Reduce_scatter numelem must be non-negative");
  const ReduceOp op = to_op(op_);
  const DType dt = to_dtype(input.scalar_type());
  check_op_dtype(op, dt);
  const int64_t axis = wrap_axis(axis_, input.dim(), "Reduce_scatter");
  std::lock_guard<std::recursive_mutex> g(world_->mutex());
  Route r(*world_, cx(), input);
  Tensor in = r.to_comm(input);
  const auto shape = in.sizes().vec();
  const Axis3 a3 = split_axis(shape, axis);
  int64_t mine[3] = {numelem, a3.before * a3.after, a3.axis};
  std::vector<int64_t> allmeta(static_cast<size_t>(size_) * 3);
  exchange_meta(mine, 3, allmeta.data());
  std::vector<int64_t> counts(static_cast<size_t>(size_));
  int64_t total = 0;
  for (int64_t p = 0; p < size_; ++p) {
    counts[p] = allmeta[p * 3];
    total += counts[p];
    TORCH_CHECK(allmeta[p * 3 + 1] == mine[1] && allmeta[p * 3 + 2] == mine[2],
                "mpi4torch_b200: Reduce_scatter needs identically shaped tensors on all ranks");
  }
  if (total != a3.axis)
    throw std::invalid_argument("mpi4torch_b200: Reduce_scatter: sum of numelem (" + std::to_string(total) +
                                ") does not match the scatter axis length (" + std::to_string(a3.axis) + ")");
  auto out_shape = shape;
  out_shape[axis] = numelem;
  {
    // the whole input of every rank is staged: larger than a staging half -> pieces along `before`, else along the
    // scatter axis (piece k of every destination's block, gathered into a temporary); same decision on all ranks
    const int64_t es = static_cast<int64_t>(in.element_size());
    const int64_t limit = slab_limit_bytes(r, cx());
    const int64_t in_bytes = in.numel() * es;
    if (in_bytes > limit && in.numel() > 0 && static_cast<int64_t>(size_) * a3.after * es > limit &&
        static_cast<int64_t>(size_) * es <= limit) {
      // one row per destination does not fit: split the trailing dimensions first
      g_slab_chunked_calls.fetch_add(1, std::memory_order_relaxed);
      Tensor in3 = in.view({a3.before, a3.axis, a3.after});
      Tensor out = at::empty(out_shape, in.options());
      Tensor out3 = out.view({a3.before, numelem, a3.after});
      const bool has_acc = accumulate.has_value() && accumulate->defined();
      Tensor acc3;
      if (has_acc) {
        TORCH_CHECK(accumulate->sizes().vec() == out_shape && accumulate->scalar_type() == input.scalar_type() &&
                        accumulate->device() == input.device(),
                    "mpi4torch_b200: Reduce_scatter: the accumulate tensor must have the result's shape, dtype and device");
        acc3 = r.to_comm(*accumulate).view({a3.before, numelem, a3.after});
      }
      const int64_t na = limit / (es * static_cast<int64_t>(size_));
      for (int64_t c0 = 0; c0 < a3.after; c0 += na) {
        const int64_t n = std::min(na, a3.after - c0);
        Tensor part = raw_reduce_scatter(in3.narrow(2, c0, n).contiguous(), op_, 1, numelem, scale, has_scale,
                                         has_acc ? c10::optional<Tensor>(acc3.narrow(2, c0, n).contiguous())
                                                 : c10::optional<Tensor>());
        out3.narrow(2, c0, n).copy_(part);
      }
      return r.from_comm(out);
    }
    if (in_bytes > limit && in.numel() > 0 && static_cast<int64_t>(size_) * a3.after * es <= limit) {
      g_slab_chunked_calls.fetch_add(1, std::memory_order_relaxed);
      Tensor in3 = in.view({a3.before, a3.axis, a3.after});
      Tensor out = at::empty(out_shape, in.options());
      Tensor out3 = out.view({a3.before, numelem, a3.after});
      Tensor acc3;
      const bool has_acc = accumulate.has_value() && accumulate->defined();
      if (has_acc) {
        TORCH_CHECK(accumulate->sizes().vec() == out_shape && accumulate->scalar_type() == input.scalar_type() &&
                        accumulate->device() == input.device(),
                    "mpi4torch_b200: Reduce_scatter: the accumulate tensor must have the result's shape, dtype and device");
        acc3 = r.to_comm(*accumulate).view({a3.before, numelem, a3.after});
      }
      auto acc_of = [&](const Tensor& piece) { return has_acc ? c10::optional<Tensor>(piece) : c10::optional<Tensor>(); };
      const int64_t row_bytes = a3.axis * a3.after * es;
      if (a3.before > 1) {
        const int64_t nb = std::max<int64_t>(1, limit / std::max<int64_t>(row_bytes, 1));
        for (int64_t b0 = 0; b0 < a3.before; b0 += nb) {
          const int64_t n = std::min(nb, a3.before - b0);
          Tensor part = raw_reduce_scatter(in3.narrow(0, b0, n), op_, 1, numelem, scale, has_scale,
                                           acc_of(has_acc ? acc3.narrow(0, b0, n) : Tensor()));
          out3.narrow(0, b0, n).copy_(part);
        }
      } else {
        const int64_t nc = (row_bytes + limit - 1) / limit;
        std::vector<int64_t> displ(static_cast<size_t>(size_), 0);
        for (int64_t p = 1; p < size_; ++p) displ[p] = displ[p - 1] + counts[p - 1];
        for (int64_t k = 0; k < nc; ++k) {
          std::vector<Tensor> pieces;
          for (int64_t p = 0; p < size_; ++p) {
            const int64_t p0 = counts[p] * k / nc, p1 = counts[p] * (k + 1) / nc;
            pieces.push_back(in3.narrow(1, displ[p] + p0, p1 - p0));
          }
          const int64_t m0 = numelem * k / nc, m1 = numelem * (k + 1) / nc;
          Tensor part = raw_reduce_scatter(at::cat(pieces, 1), op_, 1, m1 - m0, scale, has_scale,
                                           acc_of(has_acc ? acc3.narrow(1, m0, m1 - m0) : Tensor()));
          if (m1 > m0) out3.narrow(1, m0, m1 - m0).copy_(part);
        }
      }
      return r.from_comm(out);
    }
  }
  ReducePlan plan = plan_reduce_scatter(static_cast<int>(rank_), static_cast<int>(size_), a3.before, a3.after, counts);
  Tensor out = at::empty(out_shape, in.options());
  Epilogue epi;
  epi.scale = scale;
  epi.has_scale = has_scale;
  Tensor acc;
  if (accumulate.has_value() && accumulate->defined()) {
    TORCH_CHECK(accumulate->sizes().vec() == out_shape && accumulate->scalar_type() == input.scalar_type() &&
                    accumulate->device() == input.device(),
                "mpi4torch_b200: Reduce_scatter: the accumulate tensor must have the result's shape, dtype and device");
    acc = r.to_comm(*accumulate);
    epi.accumulate = acc.data_ptr();
  }
  r.be->reduce_pull(plan, in.data_ptr(), out.data_ptr(), dt, op, epi, r.stream);
  return r.from_comm(out);
}

// ---------------------------------------------------------------------------
// Non-blocking point-to-point.  The raw handle keeps the reference's layout
// (csrc/extension.cpp:1094-1107): [descriptor f64[7], comm buffer, original].
// descriptor = [request id, kind (0 send / 1 recv), peer, tag,
//               low 32 bits of the buffer address, device type, device index]
// ---------------------------------------------------------------------------
namespace {
Tensor make_descriptor(int64_t req, int kind, int64_t peer, int64_t tag, const Tensor& buf, const Tensor& orig) {
  Tensor d = at::empty({7}, at::TensorOptions().dtype(at::kDouble).device(at::kCPU));
  double* p = d.data_ptr<double>();
  p[0] = static_cast<double>(req);
  p[1] = static_cast<double>(kind);
  p[2] = static_cast<double>(peer);
  p[3] = static_cast<double>(tag);
  p[4] = static_cast<double>(ptr_hash(buf.data_ptr()));
  p[5] = static_cast<double>(static_cast<int>(orig.device().type()));
  p[6] = static_cast<double>(orig.device().index());
  return d;
}
}  // namespace

std::vector<Tensor> Communicator::raw_isend(const Tensor& input, int64_t dest, int64_t tag) {
  NvtxRange nvtx_range_("m4t::Isend");
  TORCH_CHECK(dest >= 0 && dest < size_, "mpi4torch_b200: Isend destination ", dest, " out of range");
  to_dtype(input.scalar_type());
  std::lock_guard<std::recursive_mutex> g(world_->mutex());
  Route r(*world_, cx(), input);
  Tensor buf = r.to_comm(input);
  if (buf.is_same(input)) buf = input.detach();  // own TensorImpl: the handle is an autograd output
  const int64_t req = r.be->isend(buf.data_ptr(), static_cast<int64_t>(buf.nbytes()), static_cast<int>(dest), tag, r.stream);
  return {make_descriptor(req, 0, dest, tag, buf, input), buf, input.detach()};
}

std::vector<Tensor> Communicator::raw_irecv(const Tensor& input, int64_t source, int64_t tag) {
  NvtxRange nvtx_range_("m4t::Irecv");
  TORCH_CHECK(source >= 0 && source < size_, "mpi4torch_b200: Irecv source ", source, " out of range");
  to_dtype(input.scalar_type());
  std::lock_guard<std::recursive_mutex> g(world_->mutex());
  Route r(*world_, cx(), input);
  // A non-contiguous (or host-staged) receive lands in a fresh buffer; callers
  // must use Wait's return value (same contract as the reference, :1256-1259).
  Tensor buf;
  if (r.staged) {
    buf = at::empty(input.sizes(), input.options().device(at::kCPU));
  } else {
    buf = input.is_contiguous() ? input.detach() : at::empty(input.sizes(), input.options());
  }
  const int64_t req = r.be->irecv(buf.data_ptr(), static_cast<int64_t>(buf.nbytes()), static_cast<int>(source), tag, r.stream);
  return {make_descriptor(req, 1, source, tag, buf, input), buf, input.detach()};
}

Tensor Communicator::raw_wait(const std::vector<Tensor>& handle) {
  NvtxRange nvtx_range_("m4t::Wait");
  TORCH_CHECK(handle.size() == 3, "mpi4torch_b200: a raw wait handle consists of exactly 3 tensors");
  const Tensor& desc = handle[0];
  TORCH_CHECK(desc.device().is_cpu() && desc.scalar_type() == at::kDouble && desc.numel() == 7,
              "mpi4torch_b200: malformed wait handle descriptor");
  const double* p = desc.data_ptr<double>();
  const int64_t req = static_cast<int64_t>(p[0]);
  const int kind = static_cast<int>(p[1]);
  const Tensor& buf = handle[1];
  // the in-flight transfer targets this exact buffer (reference :1231-1237)
  if (static_cast<uint32_t>(p[4]) != ptr_hash(buf.data_ptr()))
    throw std::runtime_error("mpi4torch_b200: Wait: the communication buffer of this handle was replaced "
                             "(handle bifurcation / gradient accumulation on a wait handle is not supported)");
  const c10::Device orig(static_cast<c10::DeviceType>(static_cast<int>(p[5])), static_cast<c10::DeviceIndex>(p[6]));
  std::lock_guard<std::recursive_mutex> g(world_->mutex());
  Backend* be;
  void* stream = nullptr;
  c10::optional<c10::cuda::CUDAGuard> guard;
  if (buf.is_cuda()) {
    TORCH_CHECK(cx().cuda_ready(), "mpi4torch_b200: CUDA wait handle without a CUDA backend");
    guard.emplace(buf.device());
    stream = c10::cuda::getCurrentCUDAStream(buf.device().index()).stream();
    be = cx().cuda();
  } else {
    be = &cx().host();
  }
  be->wait(req, stream);
  if (kind == 0) return handle[2];
  return buf.device() == orig ? buf : buf.to(orig);
}

}  // namespace m4t
