// Torch-facing communicator: the custom class exported to Python/TorchScript
// (reference MPI_Comm_Wrapper, csrc/extension.cpp:140-187) and the
// differentiable op entry points (reference L2, :254-1265).
#pragma once
#include <torch/custom_class.h>
#include <torch/torch.h>

#include <vector>

#include "../runtime/world.h"

namespace m4t {

using torch::Tensor;

struct Communicator : torch::CustomClassHolder {
  Communicator();  // the world communicator
  // a communicator over an existing context (created by Split)
  explicit Communicator(std::shared_ptr<CommContext> owned);

  // rank/size are cached at construction (the reference re-queries MPI on every
  // access, csrc/extension.cpp:175-187).
  int64_t GetRank() const { return rank_; }
  int64_t GetSize() const { return size_; }

  // ---- differentiable collectives ------------------------------------------
  Tensor Allreduce(const Tensor& input, int64_t op);
  // out = accumulate + scale * Allreduce(input): the scale / accumulate run in
  // the collective's epilogue, forward and backward.
  Tensor AllreduceFused(const Tensor& input, int64_t op, double scale, const c10::optional<Tensor>& accumulate);
  Tensor Bcast_(const Tensor& input, int64_t root);
  Tensor Reduce_(const Tensor& input, int64_t op, int64_t root);
  Tensor Gather(const Tensor& input, int64_t gatheraxis, int64_t root);
  Tensor Allgather(const Tensor& input, int64_t gatheraxis);
  Tensor Scatter(const Tensor& input, int64_t scatteraxis, int64_t numelem, int64_t root);
  Tensor Alltoall(const Tensor& input, int64_t gatheraxis, int64_t scatteraxis, int64_t numelem);
  Tensor Reduce_scatter(const Tensor& input, int64_t op, int64_t scatteraxis, int64_t numelem);
  // out = accumulate + scale * Reduce_scatter(input): scale / cast / accumulate run in the reducing kernel's
  // epilogue (the reference accumulates the scattered gradients with a separate `+=`, csrc/extension.cpp:616-631).
  // Backward: Allgather of (scale * grad); `accumulate` receives the incoming gradient unchanged.
  Tensor Reduce_scatterFused(const Tensor& input, int64_t op, int64_t scatteraxis, int64_t numelem, double scale,
                             const c10::optional<Tensor>& accumulate);
  // MPI_Scan / MPI_Exscan: the left fold of the inputs of ranks 0..r (Exscan: 0..r-1, zeros on rank 0) in
  // ascending rank order.  Backward (MPI_SUM only) is the reverse inclusive / exclusive scan of the gradient.
  Tensor Scan(const Tensor& input, int64_t op);
  Tensor Exscan(const Tensor& input, int64_t op);
  // Both directions as one differentiable entry point; `reverse` folds from rank P-1 downwards (the adjoint).
  Tensor scan_op(const Tensor& input, int64_t op, bool exclusive, bool reverse);

  // ---- differentiable non-blocking point-to-point ---------------------------
  std::vector<Tensor> Isend(const Tensor& input, int64_t dest, int64_t tag);
  std::vector<Tensor> Irecv(const Tensor& input, int64_t source, int64_t tag);
  Tensor Wait(const std::vector<Tensor>& handle);

  // ---- utilities --------------------------------------------------------------
  // MPI_Comm_split: ranks passing the same `color` (>= 0) form a new communicator,
  // ordered by (`key`, old rank); a negative colour yields a self-only communicator.
  // Collective over this communicator.  (The
  // reference gets sub-communicators from mpi4py, src/__init__.py:247-261.)
  c10::intrusive_ptr<Communicator> Split(int64_t color, int64_t key);
  bool IsWorld() const { return is_world_; }
  // Promise that every rank passes identically shaped tensors and the same `numelem` to the variable-size
  // ops (Gather / Allgather / Scatter / Alltoall / Reduce_scatter), as NCCL-style collectives require.  The
  // host-side size exchange is then skipped: the ops become pure stream work (CUDA-graph capturable).
  void AssumeUniformSizes(bool on) { uniform_ = on; }
  bool UniformSizes() const { return uniform_; }
  // MPI_Comm_free: collective over the communicator; releases its segments and symmetric heap.
  // Without it a sub-communicator's resources live until the process finalizes.
  void Free();
  void Barrier();
  std::string Describe() const;

  // ---- raw (non-differentiable) data paths, used by the autograd functions ---
  Tensor raw_allreduce(const Tensor& input, int64_t op, double scale, bool has_scale,
                       const c10::optional<Tensor>& accumulate);
  // param <- param + scale * Allreduce(grad, SUM), written in place (no autograd)
  void raw_allreduce_axpy_(Tensor& param, const Tensor& grad, double scale, int64_t max_blocks = 0);
  void raw_bcast_(Tensor& work, int64_t root);
  void raw_reduce_(Tensor& work, int64_t op, int64_t root);
  Tensor raw_scan(const Tensor& input, int64_t op, bool exclusive, bool reverse);
  Tensor raw_gather(const Tensor& input, int64_t axis, int64_t root, bool all);
  Tensor raw_scatter(const Tensor& input, int64_t axis, int64_t numelem, int64_t root);
  Tensor raw_alltoall(const Tensor& input, int64_t gatheraxis, int64_t scatteraxis, int64_t numelem);
  Tensor raw_reduce_scatter(const Tensor& input, int64_t op, int64_t axis, int64_t numelem, double scale = 1.0,
                            bool has_scale = false, const c10::optional<Tensor>& accumulate = c10::nullopt);
  std::vector<Tensor> raw_isend(const Tensor& input, int64_t dest, int64_t tag);
  std::vector<Tensor> raw_irecv(const Tensor& input, int64_t source, int64_t tag);
  Tensor raw_wait(const std::vector<Tensor>& handle);

  World& world() const { return *world_; }
  CommContext& context() const { return cx(); }

 private:
  CommContext& cx() const {
    TORCH_CHECK(ctx_ != nullptr && (is_world_ || ctx_->alive()), "mpi4torch_b200: this communicator has been freed");
    return *ctx_;
  }
  World* world_;
  bool is_world_ = true;
  CommContext* ctx_;                        // world context (owned by World) or owned_.get()
  std::shared_ptr<CommContext> owned_;      // non-null for communicators created by Split
  int64_t rank_, size_;
  bool uniform_ = false;
  // one metadata round over the control plane, or a local fill under AssumeUniformSizes
  void exchange_meta(const int64_t* mine, int words, int64_t* all);
};

// Differentiable dependency join (reference csrc/extension.cpp:1024-1046).
Tensor JoinDummies(const Tensor& loopthrough, const std::vector<Tensor>& dummies);

c10::intrusive_ptr<Communicator> comm_world();

// Number of Gather / Allgather / Reduce_scatter calls that were moved in pieces because one rank's share exceeded a
// staging half (or M4T_SLAB_CHUNK_BYTES); for tests and logs.
int64_t slab_chunked_calls();

}  // namespace m4t
