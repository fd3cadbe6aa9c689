// CUDA backend: the symmetric heap + kernel launch policy for one rank.
// All collectives are stream-ordered on the caller's stream (no host blocking);
// consecutive collectives issued on different streams are chained with events so
// the device-side flag protocol always sees one total order per rank.
#pragma once
#include <cuda_runtime.h>

#include <list>
#include <memory>
#include <unordered_map>
#include <vector>

#include "../kernels/kernels.h"
#include "backend.h"
#include "control.h"
#include "symm_heap.h"

namespace m4t {

struct CudaTuning {
  int64_t oneshot_max_bytes;   // M4T_ONESHOT_MAX_KB: bound on bytes x (P-1) for the one-shot path
  int64_t chunk_bytes;         // M4T_CHUNK_KB   (0 = auto: one chunk, or bytes/8 when pipelined)
  int64_t pipe_min_bytes;      // M4T_PIPE_MIN_MB: messages >= this use the role-split pipelined kernel
  int nvls_min_ranks;          // M4T_NVLS_MIN_RANKS: in-switch reduction only pays off from this world size
  int ar_blocks;               // M4T_AR_BLOCKS  (two-shot / NVLS grid)
  int oneshot_blocks;          // M4T_ONESHOT_BLOCKS
  int slab_blocks;             // M4T_SLAB_BLOCKS
  int p2p_blocks;              // M4T_P2P_BLOCKS
  int force_algo;              // M4T_ALLREDUCE_ALGO: 0 auto, 1 oneshot, 2 twoshot, 3 nvls
};

class CudaBackend final : public Backend {
 public:
  // stage_mb / symm_mb < 0: take M4T_STAGE_MB / M4T_SYMM_MB (sub-communicators pass smaller arenas)
  CudaBackend(Control& ctl, int device, int64_t stage_mb = -1, int64_t symm_mb = -1);
  ~CudaBackend() override;

  const char* name() const override { return "cuda-nvlink"; }
  int rank() const override { return ctl_.rank(); }
  int size() const override { return ctl_.size(); }
  int device() const { return device_; }
  const SymmHeap& heap() const { return *heap_; }
  const DeviceComm& device_comm() const { return dc_; }
  CudaTuning& tuning() { return tune_; }
  bool has_nvls() const { return dc_.mc_heap != nullptr; }
  std::string describe() const;

  void allreduce(const void* in, void* out, int64_t n, DType dt, ReduceOp op, const Epilogue& epi,
                 void* stream) override;
  void bcast(void* buf, int64_t n, DType dt, int root, void* stream) override;
  void reduce(void* buf, int64_t n, DType dt, ReduceOp op, int root, void* stream) override;
  void scan(const void* in, void* out, int64_t n, DType dt, ReduceOp op, bool exclusive, bool reverse,
            void* stream) override;
  void pull(const PullPlan& plan, const void* in, void* out, DType dt, void* stream) override;
  void reduce_pull(const ReducePlan& plan, const void* in, void* out, DType dt, ReduceOp op,
                   const Epilogue& epi, void* stream) override;
  int64_t isend(const void* buf, int64_t bytes, int dest, int64_t tag, void* stream) override;
  int64_t irecv(void* buf, int64_t bytes, int source, int64_t tag, void* stream) override;
  void wait(int64_t request, void* stream) override;

  // Explicit algorithm choice (benchmarks / tests).
  void allreduce_algo(const void* in, void* out, int64_t n, DType dt, ReduceOp op, const Epilogue& epi,
                      ArAlgo algo, int blocks, int64_t chunk_bytes, cudaStream_t stream);
  ArAlgo pick_algo(int64_t bytes, DType dt, ReduceOp op) const;

  // ---- tensor-core paths -------------------------------------------------------
  // Collective-order bump allocation inside the heap's persistent user arena
  // (every rank must call it with the same sizes in the same order).
  int64_t symm_alloc(int64_t bytes);
  char* symm_ptr(int64_t off) const { return dc_.heap[dc_.sync.rank] + off; }
  bool fused_linear_available(int64_t N, int64_t K) const;
  // y[M,N] = x[M,K] @ (scale * sum_ranks w[N,K])^T; returns the address of the
  // averaged weight (valid until the call after next).
  const void* fused_allreduce_linear(const void* x, const void* w, void* y, int64_t M, int64_t N, int64_t K,
                                     int64_t ldx, int64_t ldy, float scale, cudaStream_t stream,
                                     const MseEpilogue* mse = nullptr);
  void gemm_bf16_tn(const void* A, const void* B, void* C, int64_t M, int64_t N, int64_t K, int64_t lda, int64_t ldb,
                    int64_t ldc, cudaStream_t stream, const MseEpilogue* mse = nullptr);
  // Experimental: w[N,K] += scale * sum_ranks (dy[Mb,N]^T x[Mb,K]) in one kernel (wgrad GEMM +
  // in-switch reduce-scatter + SGD update + multicast of the new weights).  `w` must come from
  // symmetric_alloc() and be replicated across ranks.
  bool fused_wgrad_available(const void* w, int64_t Mb, int64_t N, int64_t K) const;
  bool fused_wgrad_multicast() const;  // in-switch reduction (true) or peer loads/stores (false)
  // prefetch_avg: also all-reduce the updated weights (x 1/size) into a symmetric buffer whose
  // address is returned - the next forward can then run as a plain local GEMM.
  const void* fused_wgrad_update(void* w, const void* dy, const void* x, int64_t Mb, int64_t N, int64_t K, int64_t ldy,
                                 int64_t ldx, float scale, cudaStream_t stream, bool prefetch_avg = false,
                                 const float* gscale = nullptr);

  // Throws if a device-side wait timed out since the last check.
  void check_device_error();
  // Symmetric scratch for fused kernels (e.g. Allreduce->GEMM): bytes inside the current staging half.
  int64_t half_bytes() const { return dc_.half_bytes; }

 private:
  struct Request {
    bool is_recv = false;
    bool matched = false;
    void* buf = nullptr;
    int64_t bytes = 0;
    int peer = 0;
    int64_t tag = 0;
    cudaEvent_t ready = nullptr;  // recv: buffer may be overwritten after this event
    cudaEvent_t done = nullptr;   // transfer complete
  };
  struct Unexpected {
    int64_t tag;
    int64_t bytes;
    void* temp;
    cudaEvent_t done;
  };

  void chain(cudaStream_t s);  // serialise collectives across streams
  cudaEvent_t new_event();
  void free_event(cudaEvent_t e);
  cudaStream_t send_stream(int peer);
  cudaStream_t recv_stream(int peer);
  P2pChannel send_channel(int dest) const;
  P2pChannel recv_channel(int source) const;
  void launch_recv(const MsgDesc& d, int source, void* dst, cudaEvent_t ready, cudaEvent_t done);
  // Pops one descriptor from source's ring (blocking or not) and matches it; returns false if none available.
  bool progress_source(int source, bool blocking);
  void complete_from_unexpected(Request& rq, Unexpected& u);

  Control& ctl_;
  int device_;
  std::unique_ptr<SymmHeap> heap_;
  DeviceComm dc_{};
  CudaTuning tune_{};
  unsigned long long* d_counters_ = nullptr;
  unsigned int* d_done_ = nullptr;
  int* h_err_ = nullptr;  // pinned + mapped
  int* d_err_ = nullptr;

  cudaStream_t last_stream_ = nullptr;
  bool have_last_ = false;
  cudaEvent_t chain_event_ = nullptr;

  int64_t p2p_off_ = 0, p2p_head_off_ = 0, p2p_tail_off_ = 0;
  int64_t slot_bytes_ = 0;
  int nslots_ = 0;
  bool p2p_push_ = false;  // ring in the receiver's heap (sender pushes) instead of the sender's (receiver pulls)
  std::vector<cudaStream_t> send_streams_, recv_streams_;
  std::vector<unsigned long long> send_chunks_, recv_chunks_;
  std::vector<uint64_t> send_seq_;
  std::unordered_map<int64_t, Request> requests_;
  std::vector<std::list<int64_t>> posted_;          // per source: unmatched irecv ids in post order
  std::vector<std::list<Unexpected>> unexpected_;   // per source
  int64_t next_request_ = 1;
  std::vector<cudaEvent_t> event_pool_;

  struct FusedLinearState {
    int64_t w_off = 0, wavg_off[2] = {0, 0}, flags_off = 0;
    uint64_t calls = 0;
  };
  std::unordered_map<int64_t, FusedLinearState> fused_;  // key = N << 32 | K
  struct FusedWgradState {
    int64_t stage_off = 0, stage_stride = 0, src_stride = 0, cnt_off = 0, done_off = 0, wavg_off = -1, epoch_off = -1;
    int ksplit = 1;
    uint64_t calls = 0;
  };
  std::unordered_map<int64_t, FusedWgradState> wgrad_;  // key = N << 32 | K
  int64_t symm_off_ = 0, symm_cursor_ = 0, symm_bytes_ = 0;
  int64_t p2p_ce_min_bytes_ = 2 << 20;  // copy-engine path threshold (M4T_P2P_CE_MIN_KB)
  bool gemm_2cta_default_ = true;  // CTA-pair kernel validated on B200: 1521 vs 1390 TFLOP/s (cuBLAS 1552)
};

}  // namespace m4t
