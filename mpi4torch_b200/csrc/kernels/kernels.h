// Host-callable launchers of the sm_100a kernels.  Torch-free; the CUDA backend
// (runtime/cuda_backend.cpp) fills a DeviceComm once and passes it by value.
#pragma once
#include <string>
#include <utility>
#include <vector>
#include <cuda_runtime.h>

#include "../runtime/common.h"
#include "../runtime/plan.h"
#include "device_sync.cuh"

namespace m4t {

// Symmetric-heap layout (identical on every rank):
//   [0, kPadBytes)                       barrier flag pads + p2p flags
//   [p2p_off, p2p_off + p2p_bytes)       p2p FIFO slots
//   [stage_off, stage_off + 2*half)      staging halves (op parity)
constexpr int64_t kBarrierPadBytes = static_cast<int64_t>(kMaxChannels) * kMaxGpuPeers * 4;  // 32 KiB

struct DeviceComm {
  SyncCtx sync;
  char* heap[kMaxGpuPeers];  // unicast mappings of every rank's heap (heap[rank] is local)
  char* mc_heap;             // multicast mapping of the heap, or nullptr
  int64_t stage_off;         // byte offset of staging half 0
  int64_t half_bytes;        // bytes per staging half
  int sm_count;
};

// Number of kernels this library has launched in this process (bench.py's
// "gpu_launches" evidence).
unsigned long long kernel_launch_count();
void note_kernel_launch();
// Same, and additionally tallied under `name` (bench.py reports which code paths really ran).
void note_kernel_launch(const char* name);
std::vector<std::pair<std::string, unsigned long long>> kernel_launch_table();

enum class ArAlgo : int { AUTO = 0, ONESHOT = 1, TWOSHOT = 2, NVLS = 3, LOCAL = 4 };

// True if the (dtype, op) pair has an in-switch multimem.ld_reduce form we emit.
bool nvls_supported(DType dt, ReduceOp op);

// Bytes of staging (per half) an allreduce of n elements needs with `algo`.
int64_t allreduce_stage_bytes(int64_t n, DType dt, ArAlgo algo, int size);

// out = epilogue(reduce over ranks of in).  One launch.
// sym_in_off >= 0: `in` is this rank's instance of a symmetric tensor at that heap offset (the
// same on every rank); two-shot / NVLS kernels then read it in place instead of staging it.
void launch_allreduce(const DeviceComm& dc, const void* in, void* out, int64_t n, DType dt, ReduceOp op,
                      const Epilogue& epi, ArAlgo algo, int blocks, int64_t chunk_bytes, cudaStream_t stream,
                      int64_t sym_in_off = -1);

// World-size-1 / local form: out = epilogue(normalise(in)); also the copy kernel.
void launch_local_epilogue(const void* in, void* out, int64_t n, DType dt, ReduceOp op, const Epilogue& epi,
                           int sm_count, cudaStream_t stream);

// Bytes of staging (per half) a scan of n elements needs with `algo` (ONESHOT or TWOSHOT).
int64_t scan_stage_bytes(int64_t n, DType dt, ArAlgo algo, int size);
// out = fold of `in` over the ranks before me in ascending rank order (scan.cu): inclusive (Scan)
// or exclusive (Exscan, zeros on the first rank of the order); `reverse` folds from rank P-1 down.
// One launch; the message must fit one staging half (scan_stage_bytes).
void launch_scan(const DeviceComm& dc, const void* in, void* out, int64_t n, DType dt, ReduceOp op, bool exclusive,
                 bool reverse, ArAlgo algo, int blocks, cudaStream_t stream);

// Broadcast root's private buffer in place (NVLS push when mc_heap, else peer pull).
void launch_bcast(const DeviceComm& dc, void* buf, int64_t n, DType dt, int root, int blocks,
                  cudaStream_t stream);
// Reduce to root in place, zero-fill non-roots.
void launch_reduce(const DeviceComm& dc, void* buf, int64_t n, DType dt, ReduceOp op, int root, int blocks,
                   cudaStream_t stream);

// Copies `bytes` of a private buffer into this rank's staging half (current parity).
void launch_stage_in(const DeviceComm& dc, const void* in, int64_t bytes, int sm_count, cudaStream_t stream);
// Barrier + strided box pulls from peers' staging (Gather/Allgather/Scatter/Alltoall).
void launch_slab_pull(const DeviceComm& dc, const PullPlan& plan, const void* in, void* out, DType dt,
                      int blocks, cudaStream_t stream);
// Experimental Allgather by multicast push (slab_push.cu); false = not eligible, nothing launched.
bool launch_allgather_push(const DeviceComm& dc, const PullPlan& plan, const void* in, void* out, DType dt, int blocks,
                           cudaStream_t stream);
// Barrier + reduce-scatter box (Allgather adjoint) with fused epilogue.
void launch_slab_reduce(const DeviceComm& dc, const ReducePlan& plan, const void* in, void* out, DType dt,
                        ReduceOp op, const Epilogue& epi, bool use_nvls, int blocks, cudaStream_t stream);
// Local strided box copy (world size 1).
void launch_slab_local(const PullPlan& plan, const void* in, void* out, DType dt, int sm_count,
                       cudaStream_t stream);

// ---- point-to-point FIFO (one directed pair) --------------------------------
// As seen from the launching side: `slots` is the sender's ring (local pointer
// on the sender, peer mapping on the receiver); head flags live in the
// RECEIVER's pad (sender writes them remotely), tail flags in the SENDER's pad.
struct P2pChannel {
  char* slots;
  uint32_t* head_flags;  // [nslots], value = chunk index + 1 once the slot holds that chunk
  uint32_t* tail_flags;  // [nslots], value = chunk index + 1 once that chunk has been consumed
  int64_t slot_bytes;
  int nslots;
};
// Forces both p2p kernels to be loaded (lazy module loading hazard, see p2p.cu).
void preload_p2p_kernels();
// Chunks a message of `bytes` occupies in the ring (>= 1: empty messages carry a flag).
int64_t p2p_num_chunks(int64_t bytes, int64_t slot_bytes);
// Sender: copies `bytes` from `src` into the ring, chunk by chunk, publishing head flags.
void launch_p2p_send(const SyncCtx& sync, const P2pChannel& ch, const void* src, int64_t bytes,
                     unsigned long long first_chunk, int blocks, cudaStream_t stream);
// Receiver: pulls chunks out of the sender's ring into `dst`, acknowledging tail flags.
void launch_p2p_recv(const SyncCtx& sync, const P2pChannel& ch, void* dst, int64_t bytes,
                     unsigned long long first_chunk, int blocks, cudaStream_t stream);
// Copy-engine variants for large messages: same ring / flags / chunk numbering, payload moved by
// cudaMemcpyAsync (no SM copies a byte), flags handled by one-warp kernels between the copies.
void launch_p2p_send_ce(const SyncCtx& sync, const P2pChannel& ch, const void* src, int64_t bytes,
                        unsigned long long first_chunk, cudaStream_t stream);
void launch_p2p_recv_ce(const SyncCtx& sync, const P2pChannel& ch, void* dst, int64_t bytes,
                        unsigned long long first_chunk, cudaStream_t stream);

// ---- tcgen05 GEMM + fused Allreduce->GEMM (gemm_tcgen05.cu) --------------------
bool gemm_bf16_tn_supported(int64_t M, int64_t N, int64_t K, const void* A, const void* B, const void* C, int64_t lda,
                            int64_t ldb, int64_t ldc);
// Optional fused MSE epilogue: instead of y the kernel stores dL/dy =
// grad_scale * (y - target) and adds loss_scale * sum((y - target)^2) to *loss_acc.
struct MseEpilogue {
  const void* target;
  int64_t ldt;
  float* loss_acc;
  float loss_scale, grad_scale;
};
// C[M,N] = A[M,K] * B[N,K]^T, bf16 in / fp32 accumulate (TMEM) / bf16 out.
void launch_gemm_bf16_tn(const void* A, const void* B, void* C, int64_t M, int64_t N, int64_t K, int64_t lda,
                         int64_t ldb, int64_t ldc, int sm_count, cudaStream_t stream, const MseEpilogue* mse = nullptr);
// Same contract on CTA pairs (cta_group::2, 256x256 cluster tiles, 6-stage TMA ring).
void launch_gemm_bf16_tn_2cta(const void* A, const void* B, void* C, int64_t M, int64_t N, int64_t K, int64_t lda,
                              int64_t ldb, int64_t ldc, int sm_count, cudaStream_t stream, const MseEpilogue* mse = nullptr);
// y = x @ (scale * sum_ranks W)^T in one kernel; W staged at heap offset w_off on every rank.
void launch_fused_allreduce_gemm(const DeviceComm& dc, const void* x, void* y, int64_t M, int64_t N, int64_t K,
                                 int64_t ldx, int64_t ldy, int64_t w_off, int64_t wavg_off, int64_t flags_off,
                                 uint32_t panel_target, float scale, cudaStream_t stream, const MseEpilogue* mse = nullptr);
void launch_fused_allreduce_gemm_2cta(const DeviceComm& dc, const void* x, void* y, int64_t M, int64_t N, int64_t K,
                                      int64_t ldx, int64_t ldy, int64_t w_off, int64_t wavg_off, int64_t flags_off,
                                      uint32_t panel_target, float scale, cudaStream_t stream,
                                      const MseEpilogue* mse = nullptr);
int fused_gemm_grid(const DeviceComm& dc);

// ---- weight gradient (wgrad_tcgen05_2cta.cu), experimental -------------------------
// G[N,K] = dY[Mb,N]^T * X[Mb,K]: both operands MN-major, no transposed copies.
bool wgrad_bf16_supported(int64_t Mb, int64_t N, int64_t K, const void* dy, const void* x, const void* g, int64_t ldy,
                          int64_t ldx, int64_t ldg);
// C[M,N] = A[M,K] * B[K,N], both row-major bf16 (dgrad: gy @ W): the CTA-pair kernel with an MN-major B operand.
bool gemm_bf16_nn_supported(int64_t M, int64_t N, int64_t K, const void* A, const void* B, const void* C, int64_t lda,
                            int64_t ldb, int64_t ldc);
void launch_gemm_bf16_nn_2cta(const void* A, const void* B, void* C, int64_t M, int64_t N, int64_t K, int64_t lda,
                              int64_t ldb, int64_t ldc, int sm_count, cudaStream_t stream);
void launch_wgrad_bf16(const void* dy, const void* x, void* g, int64_t Mb, int64_t N, int64_t K, int64_t ldy,
                       int64_t ldx, int64_t ldg, int sm_count, cudaStream_t stream, const float* gscale = nullptr,
                       float axpy = 0.0f);
// gscale: optional device scalar folded into the epilogue; axpy != 0: g <- g + axpy * gscale * (dy^T x)
// (the single-rank SGD step as the GEMM's own epilogue).
// wgrad GEMM -> reduce-scatter through the switch -> W += scale * sum -> multicast of the new
// weights, ONE kernel.  W (bf16 [N,K] contiguous) lives at heap offset w_off on every rank and
// must be replicated (identical on all ranks), as it is under data-parallel SGD.
void set_wgrad_debug(int mask);  // timing experiments (see WgradComm::debug)
int64_t fused_wgrad_tiles(int64_t N, int64_t K);
int fused_wgrad_signals_per_unit();   // signals on a tile counter per work unit and rank
int fused_wgrad_max_unicast_ranks();  // largest world the peer-load (no multicast) mode supports
void launch_fused_wgrad_update(const DeviceComm& dc, const void* dy, const void* x, int64_t Mb, int64_t N, int64_t K,
                               int64_t ldy, int64_t ldx, int64_t w_off, int64_t stage_off, int64_t stage_stride,
                               int64_t cnt_off, int64_t done_off, int ksplit, uint32_t tile_target,
                               uint32_t done_target, float scale, int64_t wavg_off, cudaStream_t stream,
                               int64_t epoch_off = -1, const float* gscale = nullptr, bool use_multicast = true,
                               int64_t src_stride = 0);
// src_stride (peer-store mode): the staging area holds one copy per SOURCE rank, src_stride bytes apart.
// tile_target = signals per WORK UNIT summed over ranks (the kernel multiplies by the tile's number of units).
// epoch_off >= 0: tile_target / done_target are PER-CALL increments and the call index lives in the local
// device word at that heap offset (advanced by the kernel): no host-side step state, graph-capturable.
// wavg_off >= 0: additionally leaves (1/P) * sum_ranks W_new in the bf16 [N,K] buffer at that heap
// offset on every rank (the parameter all-reduce of the NEXT forward, run under this GEMM).
// Plain device copy into the heap (used to stage the weight for the fused kernel).
void launch_copy_bytes(void* dst, const void* src, int64_t bytes, int sm_count, cudaStream_t stream);

// Fills `n` bytes with zero (used for non-root results / backward recv buffers).
void launch_zero(void* p, int64_t bytes, int sm_count, cudaStream_t stream);

}  // namespace m4t
