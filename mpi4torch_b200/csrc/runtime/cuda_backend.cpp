#include "cuda_backend.h"

#include <algorithm>
#include <cstring>
#include <sstream>

namespace m4t {

#define M4T_CUDA(expr)                                                                   \
  do {                                                                                   \
    cudaError_t m4t_e_ = (expr);                                                         \
    M4T_CHECK(m4t_e_ == cudaSuccess, #expr << " failed: " << cudaGetErrorString(m4t_e_)); \
  } while (0)

namespace {
int64_t round_up64(int64_t v, int64_t a) { return (v + a - 1) / a * a; }
constexpr int64_t kP2pHeadOff = 32 * 1024;  // after the 32 KiB barrier pad
constexpr int64_t kP2pTailOff = 48 * 1024;
constexpr int64_t kP2pRingOff = 1 << 20;
constexpr int kMaxSlots = 64;
}  // namespace

CudaBackend::CudaBackend(Control& ctl, int device, int64_t stage_mb, int64_t symm_mb) : ctl_(ctl), device_(device) {
  const int P = ctl.size();
  M4T_CHECK(P <= kMaxGpuPeers, "the NVLink backend supports up to " << kMaxGpuPeers << " ranks (got " << P << ")");
  M4T_CUDA(cudaSetDevice(device_));
  tune_.oneshot_max_bytes = env_i64("M4T_ONESHOT_MAX_KB", 2048) * 1024;
  tune_.chunk_bytes = env_i64("M4T_CHUNK_KB", 0) * 1024;
  tune_.pipe_min_bytes = env_i64("M4T_PIPE_MIN_MB", 512) << 20;
  tune_.nvls_min_ranks = static_cast<int>(env_i64("M4T_NVLS_MIN_RANKS", 4));
  tune_.ar_blocks = static_cast<int>(env_i64("M4T_AR_BLOCKS", 148));
  tune_.oneshot_blocks = static_cast<int>(env_i64("M4T_ONESHOT_BLOCKS", 32));
  tune_.slab_blocks = static_cast<int>(env_i64("M4T_SLAB_BLOCKS", 128));
  tune_.p2p_blocks = static_cast<int>(env_i64("M4T_P2P_BLOCKS", 32));
  tune_.force_algo = static_cast<int>(env_i64("M4T_ALLREDUCE_ALGO", 0));

  // 1 MiB slots; the copy-engine path moves half a ring per DMA, so a deeper ring means fewer, larger copies
  // (64 MiB ring: 0.46 ms for a 64 MiB fwd+bwd exchange on 8 GPUs, 16 MiB ring: 0.64 ms).  Rings are per peer:
  // the default keeps their total at 512 MiB per rank.
  const int64_t default_slots = std::max<int64_t>(16, std::min<int64_t>(64, 512 / std::max(1, P)));
  nslots_ = static_cast<int>(std::min<int64_t>(kMaxSlots, std::max<int64_t>(2, env_i64("M4T_P2P_SLOTS", default_slots))));
  slot_bytes_ = round_up64(std::max<int64_t>(4096, env_i64("M4T_P2P_SLOT_KB", 1024) * 1024), 128);
  p2p_push_ = env_i64("M4T_P2P_PUSH", 0) != 0;
  // messages of at least this many bytes move on the copy engines (-1: never); both ends decide from the
  // message size alone, so they always agree
  p2p_ce_min_bytes_ = env_i64("M4T_P2P_CE_MIN_KB", 2048) < 0 ? -1 : env_i64("M4T_P2P_CE_MIN_KB", 2048) * 1024;
  p2p_head_off_ = kP2pHeadOff;
  p2p_tail_off_ = kP2pTailOff;
  p2p_off_ = kP2pRingOff;
  const int64_t p2p_bytes = static_cast<int64_t>(P) * nslots_ * slot_bytes_;
  const int64_t stage_off = round_up64(p2p_off_ + p2p_bytes, 2 << 20);
  const int64_t half = P > 1 ? round_up64((stage_mb >= 0 ? stage_mb : env_i64("M4T_STAGE_MB", 2176)) << 20, 2 << 20) : 0;
  symm_off_ = stage_off + 2 * half;
  symm_bytes_ = P > 1 ? round_up64((symm_mb >= 0 ? symm_mb : env_i64("M4T_SYMM_MB", 512)) << 20, 2 << 20) : 0;
  symm_cursor_ = 0;
  heap_ = std::make_unique<SymmHeap>(ctl_, device_, static_cast<size_t>(symm_off_ + symm_bytes_));

  M4T_CUDA(cudaMalloc(&d_counters_, 2 * sizeof(unsigned long long)));
  M4T_CUDA(cudaMemset(d_counters_, 0, 2 * sizeof(unsigned long long)));
  M4T_CUDA(cudaMalloc(&d_done_, sizeof(unsigned int)));
  M4T_CUDA(cudaMemset(d_done_, 0, sizeof(unsigned int)));
  M4T_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&h_err_), sizeof(int), cudaHostAllocMapped));
  *h_err_ = 0;
  M4T_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&d_err_), h_err_, 0));
  M4T_CUDA(cudaEventCreateWithFlags(&chain_event_, cudaEventDisableTiming));

  cudaDeviceProp prop;
  M4T_CUDA(cudaGetDeviceProperties(&prop, device_));
  std::memset(&dc_, 0, sizeof(dc_));
  for (int p = 0; p < P; ++p) {
    dc_.heap[p] = heap_->peer(p);
    dc_.sync.pads[p] = reinterpret_cast<uint32_t*>(heap_->peer(p));
  }
  dc_.mc_heap = heap_->multicast();
  dc_.sync.counters = d_counters_;
  dc_.sync.done_ctr = d_done_;
  dc_.sync.err_flag = d_err_;
  dc_.sync.timeout_ns = static_cast<unsigned long long>(env_i64("M4T_DEVICE_TIMEOUT_S", 20)) * 1000000000ull;
  dc_.sync.rank = ctl.rank();
  dc_.sync.size = P;
  dc_.stage_off = stage_off;
  dc_.half_bytes = half;
  dc_.sm_count = prop.multiProcessorCount;

  send_streams_.assign(static_cast<size_t>(P), nullptr);
  recv_streams_.assign(static_cast<size_t>(P), nullptr);
  // Create every side stream and a pool of events NOW: resource creation can
  // synchronise the device, and doing it lazily between an Isend (whose kernel
  // may be spinning on a full ring) and the matching Irecv would stall the
  // very kernel that is waiting for that receive.
  for (int p = 0; p < P; ++p) {
    M4T_CUDA(cudaStreamCreateWithFlags(&send_streams_[p], cudaStreamNonBlocking));
    M4T_CUDA(cudaStreamCreateWithFlags(&recv_streams_[p], cudaStreamNonBlocking));
  }
  preload_p2p_kernels();
  for (int i = 0; i < 64; ++i) {
    cudaEvent_t e;
    M4T_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    event_pool_.push_back(e);
  }
  send_chunks_.assign(static_cast<size_t>(P), 0ull);
  recv_chunks_.assign(static_cast<size_t>(P), 0ull);
  send_seq_.assign(static_cast<size_t>(P), 0ull);
  posted_.resize(static_cast<size_t>(P));
  unexpected_.resize(static_cast<size_t>(P));
  M4T_CUDA(cudaDeviceSynchronize());
  ctl_.barrier();
}

CudaBackend::~CudaBackend() {
  cudaSetDevice(device_);
  cudaDeviceSynchronize();
  for (auto s : send_streams_)
    if (s) cudaStreamDestroy(s);
  for (auto s : recv_streams_)
    if (s) cudaStreamDestroy(s);
  for (auto e : event_pool_) cudaEventDestroy(e);
  if (chain_event_) cudaEventDestroy(chain_event_);
  if (d_counters_) cudaFree(d_counters_);
  if (d_done_) cudaFree(d_done_);
  if (h_err_) cudaFreeHost(h_err_);
  heap_.reset();
}

std::string CudaBackend::describe() const {
  std::ostringstream o;
  o << "cuda-nvlink rank " << rank() << "/" << size() << " dev " << device_ << " heap " << heap_->describe()
    << " staging " << (dc_.half_bytes >> 20) << " MiB x2 nvls=" << (has_nvls() ? 1 : 0);
  return o.str();
}

void CudaBackend::check_device_error() {
  if (h_err_ && *reinterpret_cast<volatile int*>(h_err_) != 0) {
    const int code = *h_err_;
    *h_err_ = 0;
    ctl_.signal_abort();
    M4T_CHECK(false, "device-side wait timed out (code " << code << ") on rank " << rank()
                         << ": a peer never reached the matching collective / transfer "
                            "(mismatched collective order across ranks?)");
  }
}

void CudaBackend::chain(cudaStream_t s) {
  // Inside a CUDA-graph capture the graph orders its own nodes, and a capturing stream must not
  // wait on events recorded outside the capture.  The collective kernels themselves are
  // capturable: flag values and staging parity come from device-resident counters.
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(s, &cap) != cudaSuccess) {
    cudaGetLastError();  // e.g. legacy stream while another stream captures: treat as "not capturing"
  } else if (cap != cudaStreamCaptureStatusNone) {
    return;
  }
  if (have_last_ && last_stream_ != s) {
    // the previous stream may have been destroyed by its owner in the meantime: its work has then been
    // completed or abandoned, and there is nothing left to order against
    if (cudaEventRecord(chain_event_, last_stream_) == cudaSuccess) {
      M4T_CUDA(cudaStreamWaitEvent(s, chain_event_, 0));
    } else {
      cudaGetLastError();
    }
  }
  last_stream_ = s;
  have_last_ = true;
}

cudaEvent_t CudaBackend::new_event() {
  if (!event_pool_.empty()) {
    cudaEvent_t e = event_pool_.back();
    event_pool_.pop_back();
    return e;
  }
  cudaEvent_t e;
  M4T_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  return e;
}

void CudaBackend::free_event(cudaEvent_t e) {
  if (e) event_pool_.push_back(e);
}

ArAlgo CudaBackend::pick_algo(int64_t bytes, DType dt, ReduceOp op) const {
  if (size() == 1) return ArAlgo::LOCAL;
  const bool nvls_ok = has_nvls() && nvls_supported(dt, op);
  const bool nvls_pays = nvls_ok && size() >= tune_.nvls_min_ranks;
  if (tune_.force_algo == 1) return ArAlgo::ONESHOT;
  if (tune_.force_algo == 2) return ArAlgo::TWOSHOT;
  if (tune_.force_algo == 3 && nvls_ok) return ArAlgo::NVLS;
  const int64_t oneshot_cap = dc_.half_bytes / size() - 128;
  // one-shot ingress is (P-1) x bytes: bound that product (2 MiB by default),
  // i.e. 2 MiB messages at P=2 but ~292 KiB at P=8
  if (bytes * (size() - 1) <= tune_.oneshot_max_bytes && bytes <= oneshot_cap) return ArAlgo::ONESHOT;
  return nvls_pays ? ArAlgo::NVLS : ArAlgo::TWOSHOT;
}

void CudaBackend::allreduce_algo(const void* in, void* out, int64_t n, DType dt, ReduceOp op, const Epilogue& epi,
                                 ArAlgo algo, int blocks, int64_t chunk_bytes, cudaStream_t stream) {
  check_device_error();
  check_op_dtype(op, dt);
  if (n == 0) return;
  M4T_CUDA(cudaSetDevice(device_));
  if (size() == 1 || algo == ArAlgo::LOCAL) {
    launch_local_epilogue(in, out, n, dt, op, epi, dc_.sm_count, stream);
    return;
  }
  chain(stream);
  const int64_t es = dtype_size(dt);
  if (algo == ArAlgo::NVLS) M4T_CHECK(has_nvls() && nvls_supported(dt, op), "NVLS unavailable for " << dtype_name(dt) << "/" << op_name(op));
  if (algo == ArAlgo::ONESHOT) {
    M4T_CHECK(allreduce_stage_bytes(n, dt, algo, size()) <= dc_.half_bytes, "one-shot allreduce too large for staging");
    launch_allreduce(dc_, in, out, n, dt, op, epi, algo, blocks, chunk_bytes, stream);
    return;
  }
  // split so that [in copy | reduced out] fits one staging half
  const int64_t max_bytes = (dc_.half_bytes / 2 - 256) / 128 * 128;
  const int64_t max_elems = std::max<int64_t>(16, max_bytes / es);
  for (int64_t off = 0; off < n; off += max_elems) {
    const int64_t cnt = std::min(max_elems, n - off);
    Epilogue e = epi;
    if (e.accumulate) e.accumulate = static_cast<const char*>(e.accumulate) + off * es;
    // experimental (M4T_ZERO_COPY_IN=1): an input inside the symmetric user arena is read in place.
    // Contract: if one rank passes a symmetric tensor, every rank passes its instance of the same one.
    static const bool zero_copy = env_i64("M4T_ZERO_COPY_IN", 0) != 0;
    int64_t sym_off = -1;
    if (zero_copy) {
      const char* ib = static_cast<const char*>(in) + off * es;
      const char* arena = dc_.heap[dc_.sync.rank] + symm_off_;
      if (ib >= arena && ib + round_up64(cnt * es, 16) <= arena + symm_bytes_) sym_off = ib - dc_.heap[dc_.sync.rank];
    }
    launch_allreduce(dc_, static_cast<const char*>(in) + off * es, static_cast<char*>(out) + off * es, cnt, dt, op, e,
                     algo, blocks, chunk_bytes, stream, sym_off);
  }
}

void CudaBackend::allreduce(const void* in, void* out, int64_t n, DType dt, ReduceOp op, const Epilogue& epi,
                            void* stream) {
  const int64_t bytes = n * dtype_size(dt);
  const ArAlgo algo = pick_algo(bytes, dt, op);
  const int blocks = algo == ArAlgo::ONESHOT ? tune_.oneshot_blocks : tune_.ar_blocks;
  // Every cross-rank barrier costs several microseconds, so mid-size messages
  // run as ONE chunk (two barriers); large ones are cut into ~8 chunks for the
  // role-split kernel whose flags are off the critical path.
  int64_t chunk = tune_.chunk_bytes;
  if (chunk <= 0) chunk = bytes >= tune_.pipe_min_bytes ? ((bytes / 8 + (1 << 20) - 1) >> 20 << 20) : (int64_t{1} << 40);
  allreduce_algo(in, out, n, dt, op, epi, algo, blocks, chunk, static_cast<cudaStream_t>(stream));
}

void CudaBackend::bcast(void* buf, int64_t n, DType dt, int root, void* stream) {
  check_device_error();
  M4T_CHECK(root >= 0 && root < size(), "Bcast_: root " << root << " out of range");
  if (size() == 1 || n == 0) return;
  M4T_CUDA(cudaSetDevice(device_));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  chain(s);
  const int64_t es = dtype_size(dt);
  const int64_t max_elems = std::max<int64_t>(16, ((dc_.half_bytes - 256) / 128 * 128) / es);
  for (int64_t off = 0; off < n; off += max_elems)
    launch_bcast(dc_, static_cast<char*>(buf) + off * es, std::min(max_elems, n - off), dt, root, tune_.ar_blocks, s);
}

void CudaBackend::reduce(void* buf, int64_t n, DType dt, ReduceOp op, int root, void* stream) {
  check_device_error();
  check_op_dtype(op, dt);
  M4T_CHECK(root >= 0 && root < size(), "Reduce_: root " << root << " out of range");
  if (n == 0) return;
  M4T_CUDA(cudaSetDevice(device_));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (size() == 1) {
    launch_local_epilogue(buf, buf, n, dt, op, Epilogue{}, dc_.sm_count, s);
    return;
  }
  chain(s);
  const int64_t es = dtype_size(dt);
  const int64_t max_elems = std::max<int64_t>(16, ((dc_.half_bytes - 256) / 128 * 128) / es);
  for (int64_t off = 0; off < n; off += max_elems)
    launch_reduce(dc_, static_cast<char*>(buf) + off * es, std::min(max_elems, n - off), dt, op, root, tune_.ar_blocks, s);
}

void CudaBackend::scan(const void* in, void* out, int64_t n, DType dt, ReduceOp op, bool exclusive, bool reverse,
                       void* stream) {
  check_device_error();
  check_op_dtype(op, dt);
  if (n == 0) return;
  M4T_CUDA(cudaSetDevice(device_));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t es = dtype_size(dt);
  if (size() == 1) {
    if (exclusive) launch_zero(out, n * es, dc_.sm_count, s);
    else launch_local_epilogue(in, out, n, dt, op, Epilogue{}, dc_.sm_count, s);
    return;
  }
  chain(s);
  // the Allreduce's choice, with two-shot where it would take NVLS (the switch only returns full reductions, never
  // prefixes)
  ArAlgo algo = pick_algo(n * es, dt, op);
  if (algo == ArAlgo::NVLS) algo = ArAlgo::TWOSHOT;
  const int blocks = algo == ArAlgo::ONESHOT ? tune_.oneshot_blocks : tune_.ar_blocks;
  // pieces that fit one staging half: P slots (one-shot) or [in copy | result] (two-shot); multiples of
  // 128 bytes, so every piece keeps the alignment of the whole tensor
  const int64_t max_bytes = algo == ArAlgo::ONESHOT ? (dc_.half_bytes / size()) / 128 * 128 - 128
                                                    : (dc_.half_bytes / 2 - 256) / 128 * 128;
  const int64_t max_elems = std::max<int64_t>(16, max_bytes / es);
  for (int64_t off = 0; off < n; off += max_elems)
    launch_scan(dc_, static_cast<const char*>(in) + off * es, static_cast<char*>(out) + off * es,
                std::min(max_elems, n - off), dt, op, exclusive, reverse, algo, blocks, s);
  check_device_error();
}

namespace {
int grid_for(int64_t max_elems, int64_t es, int cap) {
  const int64_t vecs = (max_elems * es + 15) / 16;
  const int64_t want = (vecs + 512 * 4 - 1) / (512 * 4);
  return static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(cap, want)));
}
}  // namespace

void CudaBackend::pull(const PullPlan& plan, const void* in, void* out, DType dt, void* stream) {
  check_device_error();
  M4T_CUDA(cudaSetDevice(device_));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (size() == 1) {
    launch_slab_local(plan, in, out, dt, dc_.sm_count, s);
    return;
  }
  const int64_t es = dtype_size(dt);
  M4T_CHECK(plan.max_stage_elems * es <= dc_.half_bytes,
            "collective stages " << plan.max_stage_elems * es << " B per rank but the staging half is "
                                 << dc_.half_bytes << " B; raise M4T_STAGE_MB (M4T_SUB_STAGE_MB for communicators created by Split)");
  chain(s);
  // Allgather as an NVSwitch multicast push (each rank's shard leaves its GPU once, the switch replicates it)
  // for shards up to 32 MiB, where it measured at or ahead of the pull kernel on 8 GPUs (0.51 vs 1.06 ms at
  // 16 MiB per rank); larger shards pull (1.79 vs 1.91 ms at 64 MiB).  M4T_AG_PUSH=0/1 forces.  The
  // eligibility test only looks at rank-independent quantities.
  static const int64_t ag_push_mode = env_i64("M4T_AG_PUSH", -1);  // read once
  const bool ag_push = ag_push_mode > 0 || (ag_push_mode < 0 && has_nvls() && plan.max_stage_elems * es <= (32ll << 20));
  if (ag_push && plan.replicated_output &&
      launch_allgather_push(dc_, plan, in, out, dt, grid_for(plan.max_out_elems, es, tune_.slab_blocks), s))
    return;
  if (plan.stage_elems > 0) launch_stage_in(dc_, in, plan.stage_elems * es, dc_.sm_count, s);
  launch_slab_pull(dc_, plan, in, out, dt, grid_for(plan.max_out_elems, es, tune_.slab_blocks), s);
}

void CudaBackend::reduce_pull(const ReducePlan& plan, const void* in, void* out, DType dt, ReduceOp op,
                              const Epilogue& epi, void* stream) {
  check_device_error();
  check_op_dtype(op, dt);
  M4T_CUDA(cudaSetDevice(device_));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t es = dtype_size(dt);
  if (size() > 1) {
    M4T_CHECK(plan.stage_elems * es <= dc_.half_bytes,
              "Reduce_scatter stages " << plan.stage_elems * es << " B but the staging half is " << dc_.half_bytes
                                       << " B; raise M4T_STAGE_MB (M4T_SUB_STAGE_MB for communicators created by Split)");
    chain(s);
    if (plan.stage_elems > 0) launch_stage_in(dc_, in, plan.stage_elems * es, dc_.sm_count, s);
  }
  launch_slab_reduce(dc_, plan, in, out, dt, op, epi, has_nvls(), grid_for(plan.max_out_elems, es, tune_.slab_blocks), s);
}

// ---------------------------------------------------------------------------
// tensor-core paths
// ---------------------------------------------------------------------------
int64_t CudaBackend::symm_alloc(int64_t bytes) {
  const int64_t need = round_up64(std::max<int64_t>(bytes, 16), 1024);
  M4T_CHECK(symm_cursor_ + need <= symm_bytes_, "symmetric user arena exhausted (" << symm_bytes_
                                                    << " B); raise M4T_SYMM_MB");
  const int64_t off = symm_off_ + symm_cursor_;
  symm_cursor_ += need;
  return off;
}

bool CudaBackend::fused_linear_available(int64_t N, int64_t K) const {
  if (size() <= 1 || !has_nvls()) return false;
  static const int64_t fused_linear_mode = env_i64("M4T_FUSED_LINEAR", 1);  // read once
  if (fused_linear_mode == 0) return false;
  // in-switch reduction only pays off from ~4 ranks (measured: at P=2 the
  // separate peer-load allreduce + GEMM is as fast as the fused kernel)
  if (size() < tune_.nvls_min_ranks && fused_linear_mode != 2) return false;
  if (N % 256 != 0 || 256 % size() != 0 || K % 64 != 0) return false;
  const int64_t need = 3 * N * K * 2 + 4096;
  return fused_.count((N << 32) | K) > 0 || symm_cursor_ + need + 4096 <= symm_bytes_;
}

void CudaBackend::gemm_bf16_tn(const void* A, const void* B, void* C, int64_t M, int64_t N, int64_t K, int64_t lda,
                               int64_t ldb, int64_t ldc, cudaStream_t stream, const MseEpilogue* mse) {
  M4T_CUDA(cudaSetDevice(device_));
  // CTA-pair kernel for anything big enough to fill the pairs; M4T_GEMM_2CTA=0/1 forces.
  static const int64_t mode = env_i64("M4T_GEMM_2CTA", -1);
  const bool big = M >= 512 && N >= 512;
  if (mode == 1 || (mode < 0 && big && gemm_2cta_default_)) {
    launch_gemm_bf16_tn_2cta(A, B, C, M, N, K, lda, ldb, ldc, dc_.sm_count, stream, mse);
  } else {
    launch_gemm_bf16_tn(A, B, C, M, N, K, lda, ldb, ldc, dc_.sm_count, stream, mse);
  }
}

const void* CudaBackend::fused_allreduce_linear(const void* x, const void* w, void* y, int64_t M, int64_t N, int64_t K,
                                                int64_t ldx, int64_t ldy, float scale, cudaStream_t stream,
                                                const MseEpilogue* mse) {
  check_device_error();
  M4T_CHECK(fused_linear_available(N, K), "fused Allreduce->GEMM unavailable for N=" << N << " K=" << K);
  M4T_CUDA(cudaSetDevice(device_));
  const int64_t key = (N << 32) | K;
  auto it = fused_.find(key);
  if (it == fused_.end()) {
    FusedLinearState st;
    st.w_off = symm_alloc(N * K * 2);
    st.wavg_off[0] = symm_alloc(N * K * 2);
    st.wavg_off[1] = symm_alloc(N * K * 2);
    st.flags_off = symm_alloc((N / 256) * 4);
    it = fused_.emplace(key, st).first;
  }
  FusedLinearState& st = it->second;
  chain(stream);
  // The switch reads every rank's weight at ONE heap offset.  A weight that was
  // allocated with symmetric_alloc() is used in place (zero copy); any other
  // tensor is staged first.
  int64_t w_off = st.w_off;
  const char* wb = static_cast<const char*>(w);
  const char* arena = dc_.heap[dc_.sync.rank] + symm_off_;
  if (wb >= arena && wb + N * K * 2 <= arena + symm_bytes_) {
    w_off = wb - dc_.heap[dc_.sync.rank];
  } else {
    launch_copy_bytes(symm_ptr(st.w_off), w, N * K * 2, dc_.sm_count, stream);
  }
  const int par = static_cast<int>(st.calls & 1);
  st.calls += 1;
  const uint32_t target = static_cast<uint32_t>(st.calls * static_cast<uint64_t>(size()) * fused_gemm_grid(dc_));
  static const int64_t fused_2cta = env_i64("M4T_FUSED_2CTA", 1);
  if (fused_2cta) {
    launch_fused_allreduce_gemm_2cta(dc_, x, y, M, N, K, ldx, ldy, w_off, st.wavg_off[par], st.flags_off, target,
                                     scale, stream, mse);
  } else {
    launch_fused_allreduce_gemm(dc_, x, y, M, N, K, ldx, ldy, w_off, st.wavg_off[par], st.flags_off, target, scale,
                                stream, mse);
  }
  return symm_ptr(st.wavg_off[par]);
}

bool CudaBackend::fused_wgrad_multicast() const { return has_nvls() && size() >= tune_.nvls_min_ranks; }

bool CudaBackend::fused_wgrad_available(const void* w, int64_t Mb, int64_t N, int64_t K) const {
  if (size() <= 1) return false;
  // in-switch reduction from nvls_min_ranks ranks up, peer loads / peer stores below that
  if (!fused_wgrad_multicast() && size() > fused_wgrad_max_unicast_ranks()) return false;
  static const int64_t mode = env_i64("M4T_FUSED_WGRAD", 1);  // read once; 0 disables the fused backward
  if (mode == 0) return false;
  if (N % 256 != 0 || K % 256 != 0 || Mb % 128 != 0) return false;
  const char* wb = static_cast<const char*>(w);
  const char* arena = dc_.heap[dc_.sync.rank] + symm_off_;
  if (!(wb >= arena && wb + N * K * 2 <= arena + symm_bytes_)) return false;  // must be switch-visible in place
  // 2 partial buffers (per source rank in peer-store mode) + W_avg prefetch
  const int64_t need = (2 * (fused_wgrad_multicast() ? 1 : size()) + 1) * N * K * 2 + fused_wgrad_tiles(N, K) * 4 + 8192;
  return wgrad_.count((N << 32) | K) > 0 || symm_cursor_ + need <= symm_bytes_;
}

const void* CudaBackend::fused_wgrad_update(void* w, const void* dy, const void* x, int64_t Mb, int64_t N, int64_t K,
                                            int64_t ldy, int64_t ldx, float scale, cudaStream_t stream,
                                            bool prefetch_avg, const float* gscale) {
  check_device_error();
  M4T_CHECK(fused_wgrad_available(w, Mb, N, K), "fused wgrad->Allreduce->SGD unavailable for N=" << N << " K=" << K
                                                    << " (needs a weight from symmetric_empty(), N % 256 == K % 256 == batch % 128 == 0, M4T_FUSED_WGRAD != 0)");
  M4T_CUDA(cudaSetDevice(device_));
  const int64_t key = (N << 32) | K;
  auto it = wgrad_.find(key);
  if (it == wgrad_.end()) {
    FusedWgradState st;
    // two work units per tile even out the last wave on 74 CTA pairs (M4T_WGRAD_KSPLIT=1 disables)
    static const int64_t ksplit_env = env_i64("M4T_WGRAD_KSPLIT", 2);  // read once
    st.ksplit = (ksplit_env >= 2 && (Mb / 64) % 2 == 0) ? 2 : 1;
    st.stage_stride = N * K * 2;  // dense: the peer-store epilogue addresses [ksplit * N, K] through one tensor map
    // multicast mode: one staging area per rank (own partials, pulled through the switch by the owners);
    // peer-store mode: one area per SOURCE rank in every heap (the epilogues push to the owner)
    st.src_stride = st.stage_stride * st.ksplit;
    st.stage_off = symm_alloc(st.src_stride * (fused_wgrad_multicast() ? 1 : size()));
    st.cnt_off = symm_alloc(fused_wgrad_tiles(N, K) * 4);
    st.done_off = symm_alloc(16);
    st.epoch_off = symm_alloc(16);  // call index, kept on the device (graph-capturable launches)
    it = wgrad_.emplace(key, st).first;  // the arena is zero-initialised: counters start at 0
  }
  FusedWgradState& st = it->second;
  if (prefetch_avg && st.wavg_off < 0) st.wavg_off = symm_alloc(N * K * 2);  // same call sequence on every rank
  chain(stream);
  const int64_t w_off = static_cast<const char*>(w) - dc_.heap[dc_.sync.rank];
  st.calls += 1;
  // per-call increments of the monotonic counters; the kernel multiplies by (device call index + 1)
  const uint32_t tile_target = static_cast<uint32_t>(fused_wgrad_signals_per_unit() * size());
  const uint32_t done_target = static_cast<uint32_t>(size() * fused_gemm_grid(dc_));
  launch_fused_wgrad_update(dc_, dy, x, Mb, N, K, ldy, ldx, w_off, st.stage_off, st.stage_stride, st.cnt_off,
                            st.done_off, st.ksplit, tile_target, done_target, scale, prefetch_avg ? st.wavg_off : -1,
                            stream, st.epoch_off, gscale, fused_wgrad_multicast(), st.src_stride);
  return prefetch_avg ? symm_ptr(st.wavg_off) : nullptr;
}

// ---------------------------------------------------------------------------
// point-to-point
// ---------------------------------------------------------------------------
cudaStream_t CudaBackend::send_stream(int peer) {
  if (!send_streams_[peer]) M4T_CUDA(cudaStreamCreateWithFlags(&send_streams_[peer], cudaStreamNonBlocking));
  return send_streams_[peer];
}
cudaStream_t CudaBackend::recv_stream(int peer) {
  if (!recv_streams_[peer]) M4T_CUDA(cudaStreamCreateWithFlags(&recv_streams_[peer], cudaStreamNonBlocking));
  return recv_streams_[peer];
}

P2pChannel CudaBackend::send_channel(int dest) const {
  P2pChannel ch;
  const int r = rank();
  // default: ring in the SENDER's heap (local copy-in, receiver pulls over NVLink).  With
  // M4T_P2P_PUSH=1 (experimental, every rank must agree) the ring for the pair lives in the
  // RECEIVER's heap, indexed by the source: the sender's stores cross NVLink as posted
  // writes (no round trip) and the receiver's copy-out is local.
  ch.slots = p2p_push_ ? heap_->peer(dest) + p2p_off_ + static_cast<int64_t>(r) * nslots_ * slot_bytes_
                       : heap_->peer(r) + p2p_off_ + static_cast<int64_t>(dest) * nslots_ * slot_bytes_;
  // head flags live in the receiver's pad, indexed by the source rank (me)
  ch.head_flags = reinterpret_cast<uint32_t*>(heap_->peer(dest) + p2p_head_off_) + static_cast<int64_t>(r) * kMaxSlots;
  // tail flags live in my pad, indexed by the destination
  ch.tail_flags = reinterpret_cast<uint32_t*>(heap_->peer(r) + p2p_tail_off_) + static_cast<int64_t>(dest) * kMaxSlots;
  ch.slot_bytes = slot_bytes_;
  ch.nslots = nslots_;
  return ch;
}

P2pChannel CudaBackend::recv_channel(int source) const {
  P2pChannel ch;
  const int r = rank();
  ch.slots = p2p_push_ ? heap_->peer(r) + p2p_off_ + static_cast<int64_t>(source) * nslots_ * slot_bytes_
                       : heap_->peer(source) + p2p_off_ + static_cast<int64_t>(r) * nslots_ * slot_bytes_;
  ch.head_flags = reinterpret_cast<uint32_t*>(heap_->peer(r) + p2p_head_off_) + static_cast<int64_t>(source) * kMaxSlots;
  ch.tail_flags = reinterpret_cast<uint32_t*>(heap_->peer(source) + p2p_tail_off_) + static_cast<int64_t>(r) * kMaxSlots;
  ch.slot_bytes = slot_bytes_;
  ch.nslots = nslots_;
  return ch;
}

int64_t CudaBackend::isend(const void* buf, int64_t bytes, int dest, int64_t tag, void* stream) {
  check_device_error();
  M4T_CHECK(dest >= 0 && dest < size(), "Isend: destination rank " << dest << " out of range");
  M4T_CUDA(cudaSetDevice(device_));
  cudaStream_t user = static_cast<cudaStream_t>(stream);
  cudaStream_t ss = send_stream(dest);
  // the payload is produced on the user's stream
  cudaEvent_t ready = new_event();
  M4T_CUDA(cudaEventRecord(ready, user));
  M4T_CUDA(cudaStreamWaitEvent(ss, ready, 0));
  free_event(ready);
  const unsigned long long first = send_chunks_[dest];
  M4T_LOG("rank %d isend -> %d tag %ld bytes %ld first_chunk %llu stream %p", rank(), dest, (long)tag, (long)bytes, first, (void*)user);
  if (p2p_ce_min_bytes_ >= 0 && bytes >= p2p_ce_min_bytes_) launch_p2p_send_ce(dc_.sync, send_channel(dest), buf, bytes, first, ss);
  else launch_p2p_send(dc_.sync, send_channel(dest), buf, bytes, first, tune_.p2p_blocks, ss);
  send_chunks_[dest] += static_cast<unsigned long long>(p2p_num_chunks(bytes, slot_bytes_));
  Request rq;
  rq.is_recv = false;
  rq.matched = true;
  rq.peer = dest;
  rq.tag = tag;
  rq.bytes = bytes;
  rq.done = new_event();
  M4T_CUDA(cudaEventRecord(rq.done, ss));
  // publish the descriptor so the receiver can match (src, tag) on the host
  PairRing& ring = ctl_.block()->rings[rank()][dest];
  MsgDesc d{};
  d.seq = ++send_seq_[dest];
  d.tag = tag;
  d.bytes = static_cast<uint64_t>(bytes);
  d.kind = 2;
  std::memcpy(d.inline_data, &first, sizeof(first));
  const uint64_t head = ring.head.load(std::memory_order_relaxed);
  ctl_.wait_until([&] { return head - ring.tail.load(std::memory_order_acquire) < kMailboxDepth; },
                  "space in the send ring");
  ring.entries[head % kMailboxDepth] = d;
  ring.head.store(head + 1, std::memory_order_release);
  const int64_t id = next_request_++;
  requests_[id] = rq;
  return id;
}

void CudaBackend::launch_recv(const MsgDesc& d, int source, void* dst, cudaEvent_t ready, cudaEvent_t done) {
  cudaStream_t rs = recv_stream(source);
  if (ready) M4T_CUDA(cudaStreamWaitEvent(rs, ready, 0));
  unsigned long long first = 0;
  std::memcpy(&first, d.inline_data, sizeof(first));
  M4T_CHECK(first == recv_chunks_[source], "p2p FIFO out of sync with rank " << source << " (expected chunk "
                                               << recv_chunks_[source] << ", message starts at " << first << ")");
  M4T_LOG("rank %d launch_recv <- %d tag %ld bytes %ld first_chunk %llu dst %p ready %p", rank(), source, (long)d.tag,
          (long)d.bytes, first, dst, (void*)ready);
  if (p2p_ce_min_bytes_ >= 0 && static_cast<int64_t>(d.bytes) >= p2p_ce_min_bytes_)
    launch_p2p_recv_ce(dc_.sync, recv_channel(source), dst, static_cast<int64_t>(d.bytes), first, rs);
  else
    launch_p2p_recv(dc_.sync, recv_channel(source), dst, static_cast<int64_t>(d.bytes), first, tune_.p2p_blocks, rs);
  recv_chunks_[source] += static_cast<unsigned long long>(p2p_num_chunks(static_cast<int64_t>(d.bytes), slot_bytes_));
  M4T_CUDA(cudaEventRecord(done, rs));
}

bool CudaBackend::progress_source(int source, bool blocking) {
  PairRing& ring = ctl_.block()->rings[source][rank()];
  const uint64_t tail = ring.tail.load(std::memory_order_relaxed);
  if (ring.head.load(std::memory_order_acquire) <= tail) {
    if (!blocking) return false;
    ctl_.wait_until([&] { return ring.head.load(std::memory_order_acquire) > tail; }, "a matching message");
  }
  MsgDesc d = ring.entries[tail % kMailboxDepth];
  ring.tail.store(tail + 1, std::memory_order_release);
  M4T_CHECK(d.kind == 2, "host-memory message from rank " << source << " received by the CUDA backend");
  // the device FIFO is strictly ordered: this message must be drained now
  for (auto it = posted_[source].begin(); it != posted_[source].end(); ++it) {
    Request& rq = requests_.at(*it);
    if (rq.tag != d.tag) continue;
    M4T_CHECK(static_cast<int64_t>(d.bytes) <= rq.bytes,
              "message truncated: " << d.bytes << " bytes sent by rank " << source << " (tag " << d.tag
                                    << ") into a " << rq.bytes << "-byte receive buffer");
    rq.done = new_event();
    launch_recv(d, source, rq.buf, rq.ready, rq.done);
    rq.matched = true;
    posted_[source].erase(it);
    return true;
  }
  Unexpected u;
  u.tag = d.tag;
  u.bytes = static_cast<int64_t>(d.bytes);
  u.temp = nullptr;
  // stream-ordered allocation: a plain cudaMalloc could synchronise with the
  // sender's spinning kernel
  if (u.bytes > 0) M4T_CUDA(cudaMallocAsync(&u.temp, static_cast<size_t>(u.bytes), recv_stream(source)));
  u.done = new_event();
  launch_recv(d, source, u.temp, nullptr, u.done);
  unexpected_[source].push_back(u);
  return true;
}

void CudaBackend::complete_from_unexpected(Request& rq, Unexpected& u) {
  M4T_CHECK(u.bytes <= rq.bytes, "message truncated: " << u.bytes << " bytes (tag " << u.tag << ") into a "
                                                       << rq.bytes << "-byte receive buffer");
  cudaStream_t rs = recv_stream(rq.peer);
  if (rq.ready) M4T_CUDA(cudaStreamWaitEvent(rs, rq.ready, 0));
  M4T_CUDA(cudaStreamWaitEvent(rs, u.done, 0));
  if (u.bytes > 0) M4T_CUDA(cudaMemcpyAsync(rq.buf, u.temp, static_cast<size_t>(u.bytes), cudaMemcpyDeviceToDevice, rs));
  rq.done = new_event();
  M4T_CUDA(cudaEventRecord(rq.done, rs));
  if (u.temp) M4T_CUDA(cudaFreeAsync(u.temp, rs));
  free_event(u.done);
  rq.matched = true;
}

int64_t CudaBackend::irecv(void* buf, int64_t bytes, int source, int64_t tag, void* stream) {
  check_device_error();
  M4T_CHECK(source >= 0 && source < size(), "Irecv: source rank " << source << " out of range");
  M4T_CUDA(cudaSetDevice(device_));
  Request rq;
  rq.is_recv = true;
  rq.buf = buf;
  rq.bytes = bytes;
  rq.peer = source;
  rq.tag = tag;
  rq.ready = new_event();
  M4T_CUDA(cudaEventRecord(rq.ready, static_cast<cudaStream_t>(stream)));
  const int64_t id = next_request_++;
  M4T_LOG("rank %d irecv <- %d tag %ld bytes %ld req %ld buf %p stream %p", rank(), source, (long)tag, (long)bytes, (long)id, buf, stream);
  // an earlier unexpected message with this tag?
  auto& ux = unexpected_[source];
  for (auto it = ux.begin(); it != ux.end(); ++it) {
    if (it->tag == tag) {
      complete_from_unexpected(rq, *it);
      ux.erase(it);
      requests_[id] = rq;
      return id;
    }
  }
  requests_[id] = rq;
  posted_[source].push_back(id);
  // opportunistic early match so the pull overlaps whatever the caller does next
  while (!requests_.at(id).matched && progress_source(source, false)) {
  }
  return id;
}

void CudaBackend::wait(int64_t request, void* stream) {
  auto it = requests_.find(request);
  M4T_CHECK(it != requests_.end(), "Wait: unknown or already completed request " << request
                                       << " (a WaitHandle may only be waited on once)");
  M4T_CUDA(cudaSetDevice(device_));
  if (it->second.is_recv) {
    const int src = it->second.peer;
    while (!requests_.at(request).matched) progress_source(src, true);
    it = requests_.find(request);
  }
  Request rq = it->second;
  requests_.erase(it);
  M4T_LOG("rank %d wait req %ld (%s peer %d tag %ld) stream %p", rank(), (long)request, rq.is_recv ? "recv" : "send", rq.peer,
          (long)rq.tag, stream);
  M4T_CUDA(cudaStreamWaitEvent(static_cast<cudaStream_t>(stream), rq.done, 0));
  free_event(rq.done);
  free_event(rq.ready);
  check_device_error();
}

}  // namespace m4t
