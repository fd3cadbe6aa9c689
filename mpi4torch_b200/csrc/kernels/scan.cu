// Scan / Exscan (prefix reductions across ranks) over NVLink 5 / NVSwitch, one launch per call.
//
// Fold order is the contract: rank r's result is the left fold of the inputs in ascending rank
// order, ((x_0 op x_1) op x_2) ... op x_r (Exscan: up to x_{r-1}, zeros on rank 0).  With
// `reverse` (the adjoint of a SUM scan, used by backward) the order is P-1, P-2, ... downwards.
// Both algorithms below run exactly that fold per element, so they produce identical bits, and the
// same bits as the host backends (runtime/host_kernels.h CpuScanRange).
//
//   ONESHOT  push my vector into slot[rank] of the staging half of every rank that needs it,
//            one barrier, fold the needed slots locally in order.  Latency path.
//   TWOSHOT  stage -> barrier -> the owner of shard s walks the ranks in fold order with one
//            accumulator and stores every rank's prefix of shard s straight into that rank's
//            result region over NVLink -> barrier -> copy my result region out.  Every rank
//            moves (P-1)/P of the message in and out, the traffic of the two-shot Allreduce.
//
// There is no NVLS form: the switch's multimem.ld_reduce returns the full reduction only, never a
// prefix.  `exclusive` / `reverse` are uniform runtime flags (not template parameters), so the
// instantiations stay at dtype x op.  Flag values and staging parity come from the device counters
// (device_sync.cuh), so a Scan inside a captured CUDA graph replays correctly.
#include <algorithm>

#include "kernels.h"
#include "vec_ops.cuh"

namespace m4t {

namespace {

constexpr int kThreads = 512;
constexpr int kUnroll = 4;

struct ScanArgs {
  SyncCtx sync;
  char* heap[kMaxGpuPeers];
  const void* in;
  void* out;
  int64_t stage_off;
  int64_t half_bytes;
  int64_t n;           // elements
  int64_t nvec;        // 16-byte vectors covering n
  int64_t slot_bytes;  // bytes per rank slot (ONESHOT) / per region (TWOSHOT)
  int aligned;         // in/out 16-byte aligned
  int exclusive;
  int reverse;
};

// rank at position k of the fold, and the position of rank p
__device__ __forceinline__ int fold_rank(int k, int P, bool rev) { return rev ? P - 1 - k : k; }
__device__ __forceinline__ int fold_pos(int p, int P, bool rev) { return rev ? P - 1 - p : p; }

template <DType DT, ReduceOp OP>
__global__ void __launch_bounds__(kThreads) scan_oneshot_kernel(const ScanArgs a) {
  using V = VecOf<DT>;
  const SyncCtx& c = a.sync;
  const unsigned long long fb = read_flag_base(c);
  const int par = static_cast<int>(read_op_count(c) & 1ull);
  const int64_t half = a.stage_off + static_cast<int64_t>(par) * a.half_bytes;
  const int P = c.size, r = c.rank;
  const bool rev = a.reverse != 0, excl = a.exclusive != 0, al = a.aligned != 0;
  const int me = fold_pos(r, P, rev);
  const int64_t stride = static_cast<int64_t>(gridDim.x) * kThreads;
  const int64_t first = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x;

  // push my contribution into slot[r] of every rank whose prefix contains it (my own included for Scan)
  const int lo = excl ? me + 1 : me;
  for (int64_t i = first; i < a.nvec; i += stride) {
    const Vec16 v = load_private<DT>(a.in, i, a.n, al);
    const int64_t off = half + static_cast<int64_t>(r) * a.slot_bytes + i * 16;
#pragma unroll 1
    for (int k = lo; k < P; ++k) st_vec(a.heap[fold_rank(k, P, rev)] + off, v);
  }
  block_barrier_all(c, fb, 0);
  // fold the slots of positions 0 .. cnt-1 that landed in my own HBM
  const int cnt = excl ? me : me + 1;
  const char* mine = a.heap[r] + half;
  for (int64_t i = first; i < a.nvec; i += stride) {
    Vec16 res = {};
    if (cnt > 0) {
      typename V::A acc[V::N];
      init_from<DT, OP>(acc, ld_vec_sys(mine + static_cast<int64_t>(fold_rank(0, P, rev)) * a.slot_bytes + i * 16));
#pragma unroll 1
      for (int k = 1; k < cnt; ++k)
        combine_into<DT, OP>(acc, ld_vec_sys(mine + static_cast<int64_t>(fold_rank(k, P, rev)) * a.slot_bytes + i * 16));
      res = V::pack(acc);
    }
    store_private<DT>(a.out, i, a.n, al, res);
  }
  finish_op(c, 1);
}

template <DType DT, ReduceOp OP>
__global__ void __launch_bounds__(kThreads) scan_twoshot_kernel(const ScanArgs a) {
  using V = VecOf<DT>;
  const SyncCtx& c = a.sync;
  const unsigned long long fb = read_flag_base(c);
  const int par = static_cast<int>(read_op_count(c) & 1ull);
  const int P = c.size, r = c.rank;
  const bool rev = a.reverse != 0, excl = a.exclusive != 0, al = a.aligned != 0;
  // staging half: [ in copy : slot_bytes ][ my prefix, written by the shard owners : slot_bytes ]
  const int64_t in_off = a.stage_off + static_cast<int64_t>(par) * a.half_bytes;
  const int64_t out_off = in_off + a.slot_bytes;
  char* my_in = a.heap[r] + in_off;
  const char* my_out = a.heap[r] + out_off;
  const int64_t gstride = static_cast<int64_t>(gridDim.x) * kThreads;
  const int64_t first = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x;
  const int64_t L = (a.nvec + P - 1) / P;  // shard length
  // Block b touches the same pattern of every shard in all three phases: the barriers pair block b
  // of every rank only, so whatever block b reads after a barrier was written by block b.
  const int64_t nw = first < L ? (L - first + gstride - 1) / gstride : 0;
  const int64_t nitems = nw * P;

  // ---- phase A: stage my part of every shard
  for (int64_t j0 = 0; j0 < nitems; j0 += kUnroll) {
    Vec16 v[kUnroll];
    int64_t idx[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int64_t j = j0 + u;
      const int64_t i = (j % P) * L + first + (j / P) * gstride;
      idx[u] = (j < nitems && i < a.nvec) ? i : -1;
      if (idx[u] >= 0) v[u] = load_private<DT>(a.in, idx[u], a.n, al);
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u)
      if (idx[u] >= 0) st_vec(my_in + idx[u] * 16, v[u]);
  }
  block_barrier_all(c, fb, 0);
  // ---- phase B: running fold of shard r over the ranks in fold order; rank p's prefix goes to p's result region
  for (int64_t w0 = 0; w0 < nw; w0 += kUnroll) {
    int64_t off[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int64_t i = static_cast<int64_t>(r) * L + first + (w0 + u) * gstride;
      off[u] = (w0 + u < nw && i < a.nvec) ? i * 16 : -1;
    }
    typename V::A acc[kUnroll][V::N];
#pragma unroll 1
    for (int k = 0; k < P; ++k) {
      char* peer = a.heap[fold_rank(k, P, rev)];
      if (excl) {
        // prefix before x_p; x of the last position is never needed
#pragma unroll
        for (int u = 0; u < kUnroll; ++u)
          if (off[u] >= 0) st_vec(peer + out_off + off[u], k == 0 ? Vec16{} : V::pack(acc[u]));
        if (k == P - 1) break;
      }
      Vec16 v[kUnroll];
#pragma unroll
      for (int u = 0; u < kUnroll; ++u)
        if (off[u] >= 0) v[u] = ld_vec_sys(peer + in_off + off[u]);
#pragma unroll
      for (int u = 0; u < kUnroll; ++u) {
        if (off[u] < 0) continue;
        if (k == 0) init_from<DT, OP>(acc[u], v[u]);
        else combine_into<DT, OP>(acc[u], v[u]);
        if (!excl) st_vec(peer + out_off + off[u], V::pack(acc[u]));
      }
    }
  }
  block_barrier_all(c, fb, 1);
  // ---- phase C: my prefixes of every shard are in my HBM
  for (int64_t j0 = 0; j0 < nitems; j0 += kUnroll) {
    Vec16 v[kUnroll];
    int64_t idx[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int64_t j = j0 + u;
      const int64_t i = (j % P) * L + first + (j / P) * gstride;
      idx[u] = (j < nitems && i < a.nvec) ? i : -1;
      if (idx[u] >= 0) v[u] = ld_vec_sys(my_out + idx[u] * 16);
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u)
      if (idx[u] >= 0) store_private<DT>(a.out, idx[u], a.n, al, v[u]);
  }
  finish_op(c, 2);
}

template <DType DT, ReduceOp OP> struct LaunchScanOneshot {
  static void run(const ScanArgs& a, int blocks, cudaStream_t s) { scan_oneshot_kernel<DT, OP><<<blocks, kThreads, 0, s>>>(a); }
};
template <DType DT, ReduceOp OP> struct LaunchScanTwoshot {
  static void run(const ScanArgs& a, int blocks, cudaStream_t s) { scan_twoshot_kernel<DT, OP><<<blocks, kThreads, 0, s>>>(a); }
};

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace

int64_t scan_stage_bytes(int64_t n, DType dt, ArAlgo algo, int size) {
  const int64_t span = ((n * dtype_size(dt) + 15) / 16 * 16 + 127) / 128 * 128;
  return algo == ArAlgo::ONESHOT ? span * size : 2 * span;
}

void launch_scan(const DeviceComm& dc, const void* in, void* out, int64_t n, DType dt, ReduceOp op, bool exclusive,
                 bool reverse, ArAlgo algo, int blocks, cudaStream_t stream) {
  check_op_dtype(op, dt);
  M4T_CHECK(algo == ArAlgo::ONESHOT || algo == ArAlgo::TWOSHOT, "launch_scan needs the one-shot or two-shot algorithm");
  M4T_CHECK(scan_stage_bytes(n, dt, algo, dc.sync.size) <= dc.half_bytes,
            "scan of " << n << " elements does not fit the staging half (" << dc.half_bytes << " B)");
  ScanArgs a;
  a.sync = dc.sync;
  for (int p = 0; p < kMaxGpuPeers; ++p) a.heap[p] = dc.heap[p];
  a.in = in;
  a.out = out;
  a.stage_off = dc.stage_off;
  a.half_bytes = dc.half_bytes;
  a.n = n;
  a.nvec = (n * dtype_size(dt) + 15) / 16;
  a.slot_bytes = ((a.nvec * 16 + 127) / 128) * 128;
  a.aligned = aligned16(in) && aligned16(out);
  a.exclusive = exclusive ? 1 : 0;
  a.reverse = reverse ? 1 : 0;
  blocks = std::max(1, std::min(blocks, kMaxChannels));
  const int P = dc.sync.size;
  // the grid depends on n and P only, so it is the same on every rank (barriers pair block b with block b)
  const int64_t per_block = algo == ArAlgo::ONESHOT ? a.nvec : (a.nvec + P - 1) / P;
  blocks = static_cast<int>(std::min<int64_t>(blocks, std::max<int64_t>(1, (per_block + kThreads - 1) / kThreads)));
  cudaError_t e;
  if (algo == ArAlgo::ONESHOT) {
    M4T_DISPATCH_DTYPE_OP(dt, op, LaunchScanOneshot, a, blocks, stream);
    e = cudaGetLastError();
    M4T_CHECK(e == cudaSuccess, "scan_oneshot launch failed: " << cudaGetErrorString(e));
    note_kernel_launch("scan_oneshot");
  } else {
    M4T_DISPATCH_DTYPE_OP(dt, op, LaunchScanTwoshot, a, blocks, stream);
    e = cudaGetLastError();
    M4T_CHECK(e == cudaSuccess, "scan_twoshot launch failed: " << cudaGetErrorString(e));
    note_kernel_launch("scan_twoshot");
  }
}

}  // namespace m4t
