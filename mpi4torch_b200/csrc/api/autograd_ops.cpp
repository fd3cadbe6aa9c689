// Autograd layer: every communication op is a graph node whose backward is the
// adjoint communication (reference L2, csrc/extension.cpp:189-1265):
//
//   Allreduce(SUM)   <-> Allreduce(SUM)                 (:265-272)
//   Bcast_           <-> Reduce_(SUM)                   (:324-331, :381-393)
//   Gather           <-> Scatter                        (:483-495, :752-767)
//   Allgather        <-> Reduce_scatter                 (:616-631, implemented as the
//                                                         intended reduce-scatter, not the
//                                                         reference's literal-root-1 loop)
//   Alltoall(g,s)    <-> Alltoall(s,g)                  (:903-915)
//   Scan(SUM)        <-> reverse Scan(SUM)              (prefix sums from rank P-1 downwards)
//   Exscan(SUM)      <-> reverse Exscan(SUM)
//   Isend            <-> Irecv, started in WaitBackward (:1173-1218), tag + 10 (:1161)
//   JoinDummies      :   zero grads to the dummies      (:1013-1022)
//
// The backward functions call the *differentiable* entry points again, so
// higher-order derivatives work by construction.  Nodes keep the reference's
// names so autograd profiler / anomaly-mode output stays recognisable.
#include <torch/csrc/autograd/custom_function.h>
#include <torch/csrc/autograd/function.h>
#include <torch/csrc/autograd/functions/utils.h>
#include <torch/csrc/autograd/variable.h>

#include "communicator.h"

namespace m4t {

using torch::autograd::AutogradContext;
using torch::autograd::Function;
using torch::autograd::variable_list;

namespace {

constexpr int64_t kOpSum = static_cast<int64_t>(ReduceOp::SUM);
constexpr int64_t kBackwardTagOffset = 10;  // reference :1161

c10::intrusive_ptr<Communicator> comm_from(AutogradContext* ctx) {
  return ctx->saved_data["comm"].toCustomClass<Communicator>();
}

[[noreturn]] void unimplemented_backward() {
  // reference MPIUnimplementedNode (:194-202): raised only if backward actually runs
  throw std::runtime_error("This backward operation is currently unimplemented!");
}

// ---------------------------------------------------------------- Allreduce
// The latency-critical op (four tiny Allreduces per closure of the regression example, two scalar ones
// per step of the data-parallel layer) gets a hand-rolled graph node instead of a Function<>: no
// AutogradContext, no string-keyed saved_data, no output re-wrapping - about 10 us less per
// forward+backward pair on the shared-memory backend.
struct MPIAllreduceSumBackward : public torch::autograd::Node {
  c10::intrusive_ptr<Communicator> comm;
  int64_t op = kOpSum;
  double scale = 1.0;
  bool has_scale = false, has_acc = false;

  std::string name() const override { return "MPIAllreduceSumBackward"; }
  void release_variables() override {}  // nothing saved
  variable_list apply(variable_list&& grads) override {
    if (op != kOpSum) unimplemented_backward();
    variable_list out(has_acc ? 2 : 1);
    const Tensor& g = grads[0];
    if (!g.defined()) return out;
    if (task_should_compute_output(0))
      out[0] = has_scale ? comm->AllreduceFused(g, kOpSum, scale, c10::nullopt) : comm->Allreduce(g, kOpSum);
    if (has_acc && task_should_compute_output(1)) out[1] = g;
    return out;
  }
};

Tensor allreduce_with_node(Communicator* self, const Tensor& input, int64_t op, double scale, bool has_scale,
                           const c10::optional<Tensor>& accumulate) {
  const bool has_acc = accumulate.has_value() && accumulate->defined();
  auto node = std::shared_ptr<MPIAllreduceSumBackward>(new MPIAllreduceSumBackward(), torch::autograd::deleteNode);
  node->comm = c10::intrusive_ptr<Communicator>::reclaim_copy(self);
  node->op = op;
  node->scale = scale;
  node->has_scale = has_scale;
  node->has_acc = has_acc;
  if (has_acc) node->set_next_edges(torch::autograd::collect_next_edges(input, *accumulate));
  else node->set_next_edges(torch::autograd::collect_next_edges(input));
  Tensor result;
  {
    at::AutoDispatchBelowADInplaceOrView guard;  // the data path below never records history
    result = self->raw_allreduce(input, op, scale, has_scale, accumulate);
  }
  torch::autograd::set_history(result, node);
  return result;
}

// ------------------------------------------------------------------- Bcast_
struct MPIBcastInPlaceBackward : public Function<MPIBcastInPlaceBackward> {
  static Tensor forward(AutogradContext* ctx, const Tensor& input, c10::intrusive_ptr<Communicator> comm, int64_t root) {
    ctx->saved_data["comm"] = comm;
    ctx->saved_data["root"] = root;
    // shares storage with the input when it is already contiguous (:351)
    Tensor work = input.contiguous().detach();
    comm->raw_bcast_(work, root);
    return work;
  }
  static variable_list backward(AutogradContext* ctx, variable_list grads) {
    auto comm = comm_from(ctx);
    // Reduce_ is in place: never clobber a gradient that other nodes may still read
    Tensor g = grads[0].clone();
    return {comm->Reduce_(g, kOpSum, ctx->saved_data["root"].toInt()), Tensor(), Tensor()};
  }
};

// ------------------------------------------------------------------ Reduce_
struct MPIReduceSumInPlaceBackward : public Function<MPIReduceSumInPlaceBackward> {
  static Tensor forward(AutogradContext* ctx, const Tensor& input, c10::intrusive_ptr<Communicator> comm, int64_t op,
                        int64_t root) {
    ctx->saved_data["comm"] = comm;
    ctx->saved_data["op"] = op;
    ctx->saved_data["root"] = root;
    Tensor work = input.contiguous().detach();
    comm->raw_reduce_(work, op, root);
    return work;
  }
  static variable_list backward(AutogradContext* ctx, variable_list grads) {
    if (ctx->saved_data["op"].toInt() != kOpSum) unimplemented_backward();
    auto comm = comm_from(ctx);
    Tensor g = grads[0].clone();
    return {comm->Bcast_(g, ctx->saved_data["root"].toInt()), Tensor(), Tensor(), Tensor()};
  }
};

// Poison node installed on a non-leaf input consumed by an in-place op
// (reference MPINoInplaceBackward, :395-403 and :454-461).
struct MPINoInplaceBackward : public torch::autograd::Node {
  variable_list apply(variable_list&&) override {
    throw std::runtime_error("Reuse of variables passed to inplace MPI kernels not supported");
  }
  std::string name() const override { return "MPINoInplaceBackward"; }
};

// ------------------------------------------------------------------- Gather
struct MPIGatherBackward : public Function<MPIGatherBackward> {
  static Tensor forward(AutogradContext* ctx, const Tensor& input, c10::intrusive_ptr<Communicator> comm, int64_t axis,
                        int64_t root) {
    const int64_t ax = axis < 0 ? axis + input.dim() : axis;
    ctx->saved_data["comm"] = comm;
    ctx->saved_data["axis"] = ax;
    ctx->saved_data["root"] = root;
    ctx->saved_data["numelem"] = (ax >= 0 && ax < input.dim()) ? input.size(ax) : int64_t{0};
    return comm->raw_gather(input, axis, root, /*all=*/false);
  }
  static variable_list backward(AutogradContext* ctx, variable_list grads) {
    auto comm = comm_from(ctx);
    return {comm->Scatter(grads[0], ctx->saved_data["axis"].toInt(), ctx->saved_data["numelem"].toInt(),
                          ctx->saved_data["root"].toInt()),
            Tensor(), Tensor(), Tensor()};
  }
};

// ---------------------------------------------------------------- Allgather
struct MPIAllgatherBackward : public Function<MPIAllgatherBackward> {
  static Tensor forward(AutogradContext* ctx, const Tensor& input, c10::intrusive_ptr<Communicator> comm, int64_t axis) {
    const int64_t ax = axis < 0 ? axis + input.dim() : axis;
    ctx->saved_data["comm"] = comm;
    ctx->saved_data["axis"] = ax;
    ctx->saved_data["numelem"] = (ax >= 0 && ax < input.dim()) ? input.size(ax) : int64_t{0};
    return comm->raw_gather(input, axis, 0, /*all=*/true);
  }
  static variable_list backward(AutogradContext* ctx, variable_list grads) {
    auto comm = comm_from(ctx);
    // true reduce-scatter(v) of the gradient (survey 7.5: the reference's loop at
    // :626-628 scatters from the literal root 1)
    return {comm->Reduce_scatter(grads[0], kOpSum, ctx->saved_data["axis"].toInt(), ctx->saved_data["numelem"].toInt()),
            Tensor(), Tensor()};
  }
};

// ----------------------------------------------------------- Reduce_scatter
struct MPIReduceScatterBackward : public Function<MPIReduceScatterBackward> {
  static Tensor forward(AutogradContext* ctx, const Tensor& input, c10::intrusive_ptr<Communicator> comm, int64_t op,
                        int64_t axis, int64_t numelem, double scale, bool has_scale,
                        const c10::optional<Tensor>& accumulate) {
    const int64_t ax = axis < 0 ? axis + input.dim() : axis;
    ctx->saved_data["comm"] = comm;
    ctx->saved_data["op"] = op;
    ctx->saved_data["axis"] = ax;
    ctx->saved_data["scale"] = scale;
    ctx->saved_data["has_scale"] = has_scale;
    ctx->saved_data["has_acc"] = accumulate.has_value() && accumulate->defined();
    return comm->raw_reduce_scatter(input, op, axis, numelem, scale, has_scale, accumulate);
  }
  static variable_list backward(AutogradContext* ctx, variable_list grads) {
    if (ctx->saved_data["op"].toInt() != kOpSum) unimplemented_backward();
    auto comm = comm_from(ctx);
    Tensor g = grads[0];
    if (ctx->saved_data["has_scale"].toBool()) g = g * ctx->saved_data["scale"].toDouble();
    Tensor gacc = ctx->saved_data["has_acc"].toBool() ? grads[0] : Tensor();
    return {comm->Allgather(g, ctx->saved_data["axis"].toInt()), Tensor(), Tensor(), Tensor(), Tensor(), Tensor(), Tensor(),
            gacc};
  }
};

// ------------------------------------------------------------ Scan / Exscan
// d out_q / d x_p = 1 for every p at or before q in the fold, so the adjoint sums the gradients of the ranks at or
// after p: the same scan in the opposite direction (exclusive stays exclusive).
struct MPIScanSumBackward : public Function<MPIScanSumBackward> {
  static Tensor forward(AutogradContext* ctx, const Tensor& input, c10::intrusive_ptr<Communicator> comm, int64_t op,
                        bool reverse) {
    ctx->saved_data["comm"] = comm;
    ctx->saved_data["op"] = op;
    ctx->saved_data["reverse"] = reverse;
    return comm->raw_scan(input, op, /*exclusive=*/false, reverse);
  }
  static variable_list backward(AutogradContext* ctx, variable_list grads) {
    if (ctx->saved_data["op"].toInt() != kOpSum) unimplemented_backward();
    auto comm = comm_from(ctx);
    return {comm->scan_op(grads[0], kOpSum, false, !ctx->saved_data["reverse"].toBool()), Tensor(), Tensor(), Tensor()};
  }
};

struct MPIExscanSumBackward : public Function<MPIExscanSumBackward> {
  static Tensor forward(AutogradContext* ctx, const Tensor& input, c10::intrusive_ptr<Communicator> comm, int64_t op,
                        bool reverse) {
    ctx->saved_data["comm"] = comm;
    ctx->saved_data["op"] = op;
    ctx->saved_data["reverse"] = reverse;
    return comm->raw_scan(input, op, /*exclusive=*/true, reverse);
  }
  static variable_list backward(AutogradContext* ctx, variable_list grads) {
    if (ctx->saved_data["op"].toInt() != kOpSum) unimplemented_backward();
    auto comm = comm_from(ctx);
    return {comm->scan_op(grads[0], kOpSum, true, !ctx->saved_data["reverse"].toBool()), Tensor(), Tensor(), Tensor()};
  }
};

// ------------------------------------------------------------------ Scatter
struct MPIScatterBackward : public Function<MPIScatterBackward> {
  static Tensor forward(AutogradContext* ctx, const Tensor& input, c10::intrusive_ptr<Communicator> comm, int64_t axis,
                        int64_t numelem, int64_t root) {
    Tensor out = comm->raw_scatter(input, axis, numelem, root);
    ctx->saved_data["comm"] = comm;
    ctx->saved_data["axis"] = axis < 0 ? axis + out.dim() : axis;
    ctx->saved_data["root"] = root;
    ctx->saved_data["in_sizes"] = input.sizes().vec();
    ctx->saved_data["in_dtype"] = static_cast<int64_t>(input.scalar_type());
    ctx->saved_data["in_device_type"] = static_cast<int64_t>(input.device().type());
    ctx->saved_data["in_device_index"] = static_cast<int64_t>(input.device().index());
    return out;
  }
  static variable_list backward(AutogradContext* ctx, variable_list grads) {
    auto comm = comm_from(ctx);
    const int64_t root = ctx->saved_data["root"].toInt();
    Tensor gathered = comm->Gather(grads[0], ctx->saved_data["axis"].toInt(), root);
    if (comm->GetRank() == root) return {gathered, Tensor(), Tensor(), Tensor(), Tensor()};
    // off-root inputs are placeholders: zero gradient, but joined to the gather
    // so the communication stays on the (higher-order) graph (reference :752-767)
    const auto sizes = ctx->saved_data["in_sizes"].toIntVector();
    const auto opts = at::TensorOptions()
                          .dtype(static_cast<at::ScalarType>(ctx->saved_data["in_dtype"].toInt()))
                          .device(c10::Device(static_cast<c10::DeviceType>(ctx->saved_data["in_device_type"].toInt()),
                                              static_cast<c10::DeviceIndex>(ctx->saved_data["in_device_index"].toInt())));
    return {JoinDummies(at::zeros(sizes, opts), {gathered}), Tensor(), Tensor(), Tensor(), Tensor()};
  }
};

// ----------------------------------------------------------------- Alltoall
struct MPIAlltoallBackward : public Function<MPIAlltoallBackward> {
  static Tensor forward(AutogradContext* ctx, const Tensor& input, c10::intrusive_ptr<Communicator> comm,
                        int64_t gatheraxis, int64_t scatteraxis, int64_t numelem) {
    const int64_t nd = input.dim();
    const int64_t g = gatheraxis < 0 ? gatheraxis + nd : gatheraxis;
    const int64_t s = scatteraxis < 0 ? scatteraxis + nd : scatteraxis;
    ctx->saved_data["comm"] = comm;
    ctx->saved_data["gatheraxis"] = g;
    ctx->saved_data["scatteraxis"] = s;
    ctx->saved_data["numelem"] = (g >= 0 && g < nd) ? input.size(g) : int64_t{0};
    return comm->raw_alltoall(input, gatheraxis, scatteraxis, numelem);
  }
  static variable_list backward(AutogradContext* ctx, variable_list grads) {
    auto comm = comm_from(ctx);
    // same op with the axes swapped (:912)
    return {comm->Alltoall(grads[0], ctx->saved_data["scatteraxis"].toInt(), ctx->saved_data["gatheraxis"].toInt(),
                           ctx->saved_data["numelem"].toInt()),
            Tensor(), Tensor(), Tensor(), Tensor()};
  }
};

// -------------------------------------------------------------- JoinDummies
struct JoinDummiesBackward : public Function<JoinDummiesBackward> {
  static Tensor forward(AutogradContext* ctx, const Tensor& loopthrough, at::TensorList dummies) {
    // per-dummy metadata only (no tensors are kept alive): flat sizes + ranks
    std::vector<int64_t> sizes, ndims, dtypes, devtypes, devidx;
    for (const Tensor& d : dummies) {
      for (int64_t v : d.sizes()) sizes.push_back(v);
      ndims.push_back(d.dim());
      dtypes.push_back(static_cast<int64_t>(d.scalar_type()));
      devtypes.push_back(static_cast<int64_t>(d.device().type()));
      devidx.push_back(static_cast<int64_t>(d.device().index()));
    }
    ctx->saved_data["sizes"] = sizes;
    ctx->saved_data["ndims"] = ndims;
    ctx->saved_data["dtypes"] = dtypes;
    ctx->saved_data["devtypes"] = devtypes;
    ctx->saved_data["devidx"] = devidx;
    Tensor out = loopthrough.detach();  // shallow copy sharing storage (:1037)
    // the forward result is re-joined to every gradient in backward so that communication encoded
    // through this node stays on higher-order graphs (reference :1002-1022 keeps `loopthrough`)
    ctx->save_for_backward({out});
    return out;
  }
  static variable_list backward(AutogradContext* ctx, variable_list grads) {
    const auto sizes = ctx->saved_data["sizes"].toIntVector();
    const auto ndims = ctx->saved_data["ndims"].toIntVector();
    const auto dtypes = ctx->saved_data["dtypes"].toIntVector();
    const auto devtypes = ctx->saved_data["devtypes"].toIntVector();
    const auto devidx = ctx->saved_data["devidx"].toIntVector();
    // Under create_graph=True the forward result requires grad, so JoinDummies below records a node
    // whose edges lead back to this op's inputs; in a plain first-order backward grad mode is off and
    // JoinDummies is the identity.
    const variable_list saved = ctx->get_saved_variables();
    const std::vector<Tensor> fwd = {saved[0]};
    variable_list out;
    out.reserve(ndims.size() + 1);
    out.push_back(grads[0].defined() ? JoinDummies(grads[0], fwd) : grads[0]);
    size_t cursor = 0;
    for (size_t i = 0; i < ndims.size(); ++i) {
      const std::vector<int64_t> shape(sizes.begin() + cursor, sizes.begin() + cursor + ndims[i]);
      cursor += static_cast<size_t>(ndims[i]);
      const auto opts = at::TensorOptions()
                            .dtype(static_cast<at::ScalarType>(dtypes[i]))
                            .device(c10::Device(static_cast<c10::DeviceType>(devtypes[i]),
                                                static_cast<c10::DeviceIndex>(devidx[i])));
      out.push_back(JoinDummies(at::zeros(shape, opts), fwd));  // dummies receive zeros (:1002-1011)
    }
    return out;
  }
};

// ---------------------------------------------------- Isend / Irecv / Wait
struct MPINonBlockingBackward : public Function<MPINonBlockingBackward> {
  static variable_list forward(AutogradContext* ctx, const Tensor& input, c10::intrusive_ptr<Communicator> comm,
                               bool is_recv, int64_t peer, int64_t tag) {
    ctx->saved_data["comm"] = comm;
    return is_recv ? comm->raw_irecv(input, peer, tag) : comm->raw_isend(input, peer, tag);
  }
  static variable_list backward(AutogradContext* ctx, variable_list grads) {
    // the three incoming "gradients" ARE the wait handle of the reverse
    // transfer that MPIWaitBackward started (:1061-1069)
    auto comm = comm_from(ctx);
    TORCH_CHECK(grads.size() == 3 && grads[0].defined() && grads[1].defined() && grads[2].defined(),
                "mpi4torch_b200: a wait handle must be consumed by exactly one Wait "
                "(handle bifurcation is not supported)");
    return {comm->Wait({grads[0], grads[1], grads[2]}), Tensor(), Tensor(), Tensor(), Tensor()};
  }
};

struct MPIWaitBackward : public Function<MPIWaitBackward> {
  static Tensor forward(AutogradContext* ctx, at::TensorList handle, c10::intrusive_ptr<Communicator> comm) {
    const double* p = handle[0].data_ptr<double>();
    ctx->saved_data["comm"] = comm;
    ctx->saved_data["kind"] = static_cast<int64_t>(p[1]);
    ctx->saved_data["peer"] = static_cast<int64_t>(p[2]);
    ctx->saved_data["tag"] = static_cast<int64_t>(p[3]);
    return comm->raw_wait(handle.vec());
  }
  static variable_list backward(AutogradContext* ctx, variable_list grads) {
    auto comm = comm_from(ctx);
    const int64_t kind = ctx->saved_data["kind"].toInt();
    const int64_t peer = ctx->saved_data["peer"].toInt();
    const int64_t tag = ctx->saved_data["tag"].toInt() + kBackwardTagOffset;
    std::vector<Tensor> h;
    if (kind == 0) {
      // forward Isend -> backward Irecv of the gradient from `dest` (:1204-1208)
      h = comm->Irecv(at::zeros_like(grads[0]), peer, tag);
    } else {
      // forward Irecv -> backward Isend of the gradient to `source` (:1209-1212)
      h = comm->Isend(grads[0], peer, tag);
    }
    return {h[0], h[1], h[2], Tensor()};
  }
};

bool any_requires_grad(const std::vector<Tensor>& ts) {
  if (!at::GradMode::is_enabled()) return false;
  for (const Tensor& t : ts)
    if (t.defined() && t.requires_grad()) return true;
  return false;
}

}  // namespace

// ---------------------------------------------------------------------------
// differentiable entry points
// ---------------------------------------------------------------------------
// Every entry point skips the graph node when nothing can require a gradient (no_grad blocks, plain
// tensors, and - most often - the adjoint calls made from inside a first-order backward): the node's
// context and saved_data cost more than a small collective on the shared-memory backend.
Tensor Communicator::Allreduce(const Tensor& input, int64_t op) {
  if (!any_requires_grad({input})) return raw_allreduce(input, op, 1.0, false, c10::nullopt);
  return allreduce_with_node(this, input, op, 1.0, false, c10::nullopt);
}

Tensor Communicator::AllreduceFused(const Tensor& input, int64_t op, double scale,
                                    const c10::optional<Tensor>& accumulate) {
  if (!any_requires_grad({input, accumulate.has_value() ? *accumulate : Tensor()}))
    return raw_allreduce(input, op, scale, true, accumulate);
  return allreduce_with_node(this, input, op, scale, true, accumulate);
}

Tensor Communicator::Bcast_(const Tensor& input, int64_t root) {
  if (!any_requires_grad({input})) {
    Tensor work = input.contiguous().detach();
    raw_bcast_(work, root);
    return work;
  }
  return MPIBcastInPlaceBackward::apply(input, c10::intrusive_ptr<Communicator>::reclaim_copy(this), root);
}

Tensor Communicator::Reduce_(const Tensor& input, int64_t op, int64_t root) {
  if (!any_requires_grad({input})) {
    Tensor work = input.contiguous().detach();
    raw_reduce_(work, op, root);
    return work;
  }
  Tensor result = MPIReduceSumInPlaceBackward::apply(input, c10::intrusive_ptr<Communicator>::reclaim_copy(this), op, root);
  // Misuse guard (:454-461): a non-leaf input whose storage was just overwritten
  // must not feed any later op; leaves are exempt (AccumulateGrad needs them).
  if (at::GradMode::is_enabled() && input.requires_grad() && input.grad_fn()) {
    auto poison = std::shared_ptr<MPINoInplaceBackward>(new MPINoInplaceBackward(), torch::autograd::deleteNode);
    torch::autograd::set_history(input, poison);
  }
  return result;
}

Tensor Communicator::Gather(const Tensor& input, int64_t gatheraxis, int64_t root) {
  if (!any_requires_grad({input})) return raw_gather(input, gatheraxis, root, /*all=*/false);
  return MPIGatherBackward::apply(input, c10::intrusive_ptr<Communicator>::reclaim_copy(this), gatheraxis, root);
}

Tensor Communicator::Allgather(const Tensor& input, int64_t gatheraxis) {
  if (!any_requires_grad({input})) return raw_gather(input, gatheraxis, 0, /*all=*/true);
  return MPIAllgatherBackward::apply(input, c10::intrusive_ptr<Communicator>::reclaim_copy(this), gatheraxis);
}

Tensor Communicator::Scatter(const Tensor& input, int64_t scatteraxis, int64_t numelem, int64_t root) {
  if (!any_requires_grad({input})) return raw_scatter(input, scatteraxis, numelem, root);
  return MPIScatterBackward::apply(input, c10::intrusive_ptr<Communicator>::reclaim_copy(this), scatteraxis, numelem, root);
}

Tensor Communicator::Alltoall(const Tensor& input, int64_t gatheraxis, int64_t scatteraxis, int64_t numelem) {
  if (!any_requires_grad({input})) return raw_alltoall(input, gatheraxis, scatteraxis, numelem);
  return MPIAlltoallBackward::apply(input, c10::intrusive_ptr<Communicator>::reclaim_copy(this), gatheraxis, scatteraxis,
                                    numelem);
}

Tensor Communicator::Reduce_scatter(const Tensor& input, int64_t op, int64_t scatteraxis, int64_t numelem) {
  if (!any_requires_grad({input})) return raw_reduce_scatter(input, op, scatteraxis, numelem);
  return MPIReduceScatterBackward::apply(input, c10::intrusive_ptr<Communicator>::reclaim_copy(this), op, scatteraxis,
                                         numelem, 1.0, false, c10::optional<Tensor>());
}

Tensor Communicator::Reduce_scatterFused(const Tensor& input, int64_t op, int64_t scatteraxis, int64_t numelem, double scale,
                                         const c10::optional<Tensor>& accumulate) {
  if (!any_requires_grad({input, accumulate.has_value() ? *accumulate : Tensor()}))
    return raw_reduce_scatter(input, op, scatteraxis, numelem, scale, true, accumulate);
  return MPIReduceScatterBackward::apply(input, c10::intrusive_ptr<Communicator>::reclaim_copy(this), op, scatteraxis,
                                         numelem, scale, true, accumulate);
}

Tensor Communicator::Scan(const Tensor& input, int64_t op) { return scan_op(input, op, false, false); }

Tensor Communicator::Exscan(const Tensor& input, int64_t op) { return scan_op(input, op, true, false); }

Tensor Communicator::scan_op(const Tensor& input, int64_t op, bool exclusive, bool reverse) {
  if (!any_requires_grad({input})) return raw_scan(input, op, exclusive, reverse);
  auto self = c10::intrusive_ptr<Communicator>::reclaim_copy(this);
  if (exclusive) return MPIExscanSumBackward::apply(input, self, op, reverse);
  return MPIScanSumBackward::apply(input, self, op, reverse);
}

std::vector<Tensor> Communicator::Isend(const Tensor& input, int64_t dest, int64_t tag) {
  if (!any_requires_grad({input})) return raw_isend(input, dest, tag);
  return MPINonBlockingBackward::apply(input, c10::intrusive_ptr<Communicator>::reclaim_copy(this), false, dest, tag);
}

std::vector<Tensor> Communicator::Irecv(const Tensor& input, int64_t source, int64_t tag) {
  if (!any_requires_grad({input})) return raw_irecv(input, source, tag);
  return MPINonBlockingBackward::apply(input, c10::intrusive_ptr<Communicator>::reclaim_copy(this), true, source, tag);
}

Tensor Communicator::Wait(const std::vector<Tensor>& handle) {
  TORCH_CHECK(handle.size() == 3, "mpi4torch_b200: a raw wait handle consists of exactly 3 tensors");
  // MPIWaitBackward::forward reads the descriptor on the host: validate it first
  TORCH_CHECK(handle[0].defined() && handle[0].device().is_cpu() && handle[0].scalar_type() == at::kDouble &&
                  handle[0].numel() == 7 && handle[0].is_contiguous(),
              "mpi4torch_b200: malformed wait handle descriptor");
  // Bifurcation guard (:1183-1202): the buffer handed to Wait must come straight
  // from Isend/Irecv, otherwise autograd would sum two gradient handles and an
  // in-flight receive would write to freed memory.
  if (any_requires_grad(handle) && handle[1].grad_fn()) {
    const std::string n = handle[1].grad_fn()->name();
    if (n.find("MPINonBlockingBackward") == std::string::npos)
      throw std::runtime_error("mpi4torch_b200: Wait: handle element 1 must be produced directly by Isend/Irecv, "
                               "found " + n + " (wait handle bifurcation is not supported)");
  }
  if (!any_requires_grad(handle)) return raw_wait(handle);
  return MPIWaitBackward::apply(at::TensorList(handle), c10::intrusive_ptr<Communicator>::reclaim_copy(this));
}

Tensor JoinDummies(const Tensor& loopthrough, const std::vector<Tensor>& dummies) {
  // only the dummies decide (reference :1027-1033)
  if (!any_requires_grad(dummies)) return loopthrough;
  return JoinDummiesBackward::apply(loopthrough, at::TensorList(dummies));
}

}  // namespace m4t
