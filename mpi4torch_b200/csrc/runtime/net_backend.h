// Host backend over the TCP mesh (jobs that span nodes).  Same contract as CpuBackend, different transport:
//   Allreduce   small: every rank receives every contribution and reduces in rank order; large: ring reduce-scatter +
//               ring all-gather (each rank moves 2(P-1)/P of the message), epilogue applied to the finished vector
//   Bcast_      binomial tree from the root
//   Reduce_     binomial tree to the root, non-root buffers zero-filled
//   slab plans  request / response: a rank sends the box descriptors of its plan to the peers that hold the data, they
//               pack the rows and answer; the plans themselves (plan.cpp) are the ones the other backends execute
//   Isend/Irecv the engine's posted sends / receives with the user tag (FIFO per source and tag, unexpected messages
//               are buffered)
// Host-blocking like MPI on host buffers (reference csrc/extension.cpp:61-104); CUDA tensors reach it through the
// API layer's host staging.
#pragma once
#include <memory>
#include <unordered_map>
#include <vector>

#include "backend.h"
#include "net_link.h"

namespace m4t {

class NetBackend final : public Backend {
 public:
  explicit NetBackend(std::shared_ptr<NetLink> link) : link_(std::move(link)) {}

  const char* name() const override { return "tcp"; }
  int rank() const override { return link_->rank(); }
  int size() const override { return link_->size(); }

  void allreduce(const void* in, void* out, int64_t n, DType dt, ReduceOp op, const Epilogue& epi,
                 void* stream) override;
  void bcast(void* buf, int64_t n, DType dt, int root, void* stream) override;
  void reduce(void* buf, int64_t n, DType dt, ReduceOp op, int root, void* stream) override;
  // Scan / Exscan  small: every rank receives the contributions of the ranks before it in the fold; large: the owner of
  //                slice p receives slice p from every rank, folds it in order and returns each rank its prefix
  void scan(const void* in, void* out, int64_t n, DType dt, ReduceOp op, bool exclusive, bool reverse,
            void* stream) override;
  void pull(const PullPlan& plan, const void* in, void* out, DType dt, void* stream) override;
  void reduce_pull(const ReducePlan& plan, const void* in, void* out, DType dt, ReduceOp op, const Epilogue& epi,
                   void* stream) override;
  int64_t isend(const void* buf, int64_t bytes, int dest, int64_t tag, void* stream) override;
  int64_t irecv(void* buf, int64_t bytes, int source, int64_t tag, void* stream) override;
  void wait(int64_t request, void* stream) override;

 private:
  std::shared_ptr<NetLink> link_;
  std::unordered_map<int64_t, uint64_t> requests_;  // request id -> engine operation
  std::unordered_map<int64_t, void*> recv_bufs_;    // receive requests: where Wait copies the message
  int64_t next_request_ = 1;
  NetBuffer scratch_[3];  // grow-only temporaries of the large-message Allreduce and of Scan
};

// Host backend of a job that spans nodes with the same number of ranks on each: Allreduce is done in three steps -
// reduce-scatter inside the node through shared memory (local rank i ends up with slice i), Allreduce of that slice
// between the ranks that have the same local index on every node (one TCP "rail" per local rank, so all of a node's
// ranks drive the network at the same time and only 1/L of the message crosses it per rank), all-gather inside the
// node.  Every other operation goes to the flat mesh backend.  The same structure is what a device path would use
// (NVLink inside the node instead of shared memory).
class CpuBackend;
class HierBackend final : public Backend {
 public:
  HierBackend(CpuBackend& local, NetBackend& flat, std::shared_ptr<NetLink> rail)
      : local_(local), flat_(flat), rail_link_(std::move(rail)), rail_(rail_link_) {}

  const char* name() const override { return "shm+tcp"; }
  int rank() const override { return flat_.rank(); }
  int size() const override { return flat_.size(); }

  void allreduce(const void* in, void* out, int64_t n, DType dt, ReduceOp op, const Epilogue& epi,
                 void* stream) override;
  // rooted operations: along the root's rail between the nodes, through shared memory inside each node
  void bcast(void* buf, int64_t n, DType dt, int root, void* stream) override;
  void reduce(void* buf, int64_t n, DType dt, ReduceOp op, int root, void* stream) override;
  // Scan / Exscan: the flat mesh (one fold over all ranks, so 16-bit floats are rounded once)
  void scan(const void* in, void* out, int64_t n, DType dt, ReduceOp op, bool exclusive, bool reverse,
            void* stream) override {
    flat_.scan(in, out, n, dt, op, exclusive, reverse, stream);
  }
  // slab plans: boxes held by ranks of this node are read through the node's shared memory, the others over the mesh
  void pull(const PullPlan& plan, const void* in, void* out, DType dt, void* stream) override;
  // Reduce_scatter with the same count on every rank: the node first sums, through shared memory, the slices of the
  // destinations on each rail (local rank l collects those of ranks l, L+l, 2L+l, ...), then a reduce-scatter along the
  // rail finishes them; other shapes use the flat mesh
  void reduce_pull(const ReducePlan& plan, const void* in, void* out, DType dt, ReduceOp op, const Epilogue& epi,
                   void* stream) override;
  // point-to-point: a peer on this node is reached through the node's shared memory, any other through the mesh (a
  // given source always takes the same route, so per-source FIFO order holds); the low bit of the id says which
  int64_t isend(const void* buf, int64_t bytes, int dest, int64_t tag, void* stream) override;
  int64_t irecv(void* buf, int64_t bytes, int source, int64_t tag, void* stream) override;
  void wait(int64_t request, void* stream) override;

 private:
  CpuBackend& local_;
  NetBackend& flat_;
  std::shared_ptr<NetLink> rail_link_;
  NetBackend rail_;
  NetBuffer part_, land_, wide_in_, wide_out_;
};

}  // namespace m4t
