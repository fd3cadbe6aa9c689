// Abstract transport interface under the autograd layer.  Two implementations:
//   * CpuBackend  - POSIX shared memory + atomics (plumbing, local tests, the
//                   host-staged comparator; reference analogue: plain MPI on host
//                   buffers, csrc/extension.cpp:61-104),
//   * CudaBackend - symmetric heap over NVLink 5 / NVSwitch with hand-written
//                   sm_100a kernels (the product).
// All pointers are raw; `stream` is an opaque cudaStream_t for the CUDA backend
// and ignored by the CPU backend (whose calls are host-blocking like MPI).
#pragma once
#include <cstdint>

#include "common.h"
#include "plan.h"

namespace m4t {

class Backend {
 public:
  virtual ~Backend() = default;
  virtual const char* name() const = 0;
  virtual int rank() const = 0;
  virtual int size() const = 0;

  // out = epilogue(reduce_p in_p); in/out may alias.
  virtual void allreduce(const void* in, void* out, int64_t n, DType dt, ReduceOp op,
                         const Epilogue& epi, void* stream) = 0;
  // In place broadcast of root's buffer.
  virtual void bcast(void* buf, int64_t n, DType dt, int root, void* stream) = 0;
  // In place reduce to root; non-root buffers are zero-filled afterwards
  // (reference csrc/extension.cpp:443-447).
  virtual void reduce(void* buf, int64_t n, DType dt, ReduceOp op, int root, void* stream) = 0;
  // Prefix reduction across ranks (Scan / Exscan).  out = left fold of `in` over the ranks in
  // ascending order up to and including me (exclusive: up to the rank before me, zeros on rank 0);
  // `reverse` folds from rank P-1 downwards instead (the adjoint of a SUM scan).  16-bit floats fold
  // in fp32 and are rounded once; every backend gives the same bits.
  virtual void scan(const void* in, void* out, int64_t n, DType dt, ReduceOp op, bool exclusive, bool reverse,
                    void* stream) = 0;
  // Strided box pulls (Gather / Allgather / Scatter / Alltoall).
  virtual void pull(const PullPlan& plan, const void* in, void* out, DType dt, void* stream) = 0;
  // Reduce-scatter along an axis (Allgather's adjoint).
  virtual void reduce_pull(const ReducePlan& plan, const void* in, void* out, DType dt, ReduceOp op,
                           const Epilogue& epi, void* stream) = 0;

  // Non-blocking point-to-point.  Returns a request id (> 0).
  virtual int64_t isend(const void* buf, int64_t bytes, int dest, int64_t tag, void* stream) = 0;
  virtual int64_t irecv(void* buf, int64_t bytes, int source, int64_t tag, void* stream) = 0;
  // Completes a request; throws if the id is unknown (already waited on).
  virtual void wait(int64_t request, void* stream) = 0;
};

}  // namespace m4t
