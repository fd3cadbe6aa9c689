// CPU shared-memory backend: every rank publishes its contribution in a
// growable POSIX-shm arena, a flag barrier orders publication, peers read
// straight out of each other's arenas.  Two arenas per rank alternate by op
// parity, so each collective needs exactly one barrier (two for the
// large-message two-phase allreduce).
#pragma once
#include <list>
#include <string>
#include <unordered_map>
#include <vector>

#include "backend.h"
#include "control.h"

namespace m4t {

class CpuBackend final : public Backend {
 public:
  explicit CpuBackend(Control& ctl);
  ~CpuBackend() override;

  const char* name() const override { return "cpu-shm"; }
  int rank() const override { return ctl_.rank(); }
  int size() const override { return ctl_.size(); }

  void allreduce(const void* in, void* out, int64_t n, DType dt, ReduceOp op, const Epilogue& epi,
                 void* stream) override;
  void bcast(void* buf, int64_t n, DType dt, int root, void* stream) override;
  void reduce(void* buf, int64_t n, DType dt, ReduceOp op, int root, void* stream) override;
  // Scan / Exscan: small messages fold the peers' staged copies in order; from kTwoPhaseBytes the owner of slice p
  // writes every rank's prefix of slice p into that rank's result half (two barriers)
  void scan(const void* in, void* out, int64_t n, DType dt, ReduceOp op, bool exclusive, bool reverse,
            void* stream) override;
  void pull(const PullPlan& plan, const void* in, void* out, DType dt, void* stream) override;
  void reduce_pull(const ReducePlan& plan, const void* in, void* out, DType dt, ReduceOp op,
                   const Epilogue& epi, void* stream) override;
  int64_t isend(const void* buf, int64_t bytes, int dest, int64_t tag, void* stream) override;
  int64_t irecv(void* buf, int64_t bytes, int source, int64_t tag, void* stream) override;
  void wait(int64_t request, void* stream) override;

 private:
  struct Mapping {
    char* ptr = nullptr;
    size_t cap = 0;
    uint64_t gen = 0;
  };
  struct Request {
    bool is_recv = false;
    void* buf = nullptr;
    int64_t bytes = 0;
    int peer = 0;
    int64_t tag = 0;
  };

  std::string arena_name(int rank, int par, uint64_t gen) const;
  char* stage(int par, size_t bytes);           // own arena with at least `bytes`
  const char* peer_arena(int peer, int par);    // valid after the op's barrier
  void deliver(const MsgDesc& d, int source, Request& rq);
  std::string msg_name(int src, int dst, uint64_t seq) const;

  Control& ctl_;
  Mapping own_[2];
  Mapping peers_[kMaxRanks][2];
  uint64_t op_seq_ = 0;

  std::unordered_map<int64_t, Request> requests_;
  int64_t next_request_ = 1;
  uint64_t send_seq_[kMaxRanks] = {};
  std::list<MsgDesc> unexpected_[kMaxRanks];
};

}  // namespace m4t
