// Host-side copy / reduction kernels shared by the host backends (POSIX shared memory: cpu_backend.cpp, TCP:
// net_backend.cpp): OpenMP-parallel memcpy, the element-wise reduction over P sources with the fused epilogue, and the
// strided box variants the slab plans use.
#pragma once
#include <algorithm>
#include <cstring>

#include <omp.h>

#include "backend.h"
#include "control.h"
#include "plan.h"
#include "reduce_ops.h"

namespace m4t {

// Large copies / reductions are memory-bound; a rank may use the OpenMP threads the launcher
// left it (OMP_NUM_THREADS = cores / ranks).  Below the threshold one thread is faster.
constexpr size_t kParallelBytes = 1u << 20;

inline void par_memcpy(void* dst, const void* src, size_t bytes) {
  if (bytes < kParallelBytes || omp_get_max_threads() <= 1 || omp_in_parallel()) {
    std::memcpy(dst, src, bytes);
    return;
  }
  constexpr size_t kChunk = 256u << 10;
  const int64_t chunks = static_cast<int64_t>((bytes + kChunk - 1) / kChunk);
#pragma omp parallel for schedule(static)
  for (int64_t c = 0; c < chunks; ++c) {
    const size_t off = static_cast<size_t>(c) * kChunk;
    std::memcpy(static_cast<char*>(dst) + off, static_cast<const char*>(src) + off, std::min(kChunk, bytes - off));
  }
}

template <typename A> inline A scale_acc(A v, double s) {
  return static_cast<A>(static_cast<double>(v) * s);
}
template <> inline float scale_acc<float>(float v, double s) { return v * static_cast<float>(s); }

// out[i] = epi(combine_k srcs[k][i]) for i in [lo, hi).  Sources are combined in index order
// k = 0..nsrc-1 per element (identical result on every rank); the loops are blocked so that
// the inner ones run over contiguous elements of ONE source and vectorise.
template <DType DT, ReduceOp OP> struct CpuReduceRange {
  using E = Elem<DT>;
  using S = typename E::storage;
  using A = typename E::acc;
  using C = Combine<OP, A, E::is_float>;

  static void run_serial(const void* const* srcs, int nsrc, S* o, const S* accp, bool scaled, double s, int64_t lo,
                         int64_t hi) {
    constexpr int kBlock = 512;
    A buf[kBlock];
    for (int64_t b0 = lo; b0 < hi; b0 += kBlock) {
      const int n = static_cast<int>(std::min<int64_t>(kBlock, hi - b0));
      const S* s0 = static_cast<const S*>(srcs[0]) + b0;
      for (int j = 0; j < n; ++j) buf[j] = normalise_single<OP, A>(E::load(s0[j]));
      for (int k = 1; k < nsrc; ++k) {
        const S* sk = static_cast<const S*>(srcs[k]) + b0;
        for (int j = 0; j < n; ++j) buf[j] = C::apply(buf[j], E::load(sk[j]));
      }
      if (scaled)
        for (int j = 0; j < n; ++j) buf[j] = scale_acc<A>(buf[j], s);
      if (accp)
        for (int j = 0; j < n; ++j) buf[j] = buf[j] + E::load(accp[b0 + j]);
      for (int j = 0; j < n; ++j) o[b0 + j] = E::store(buf[j]);
    }
  }

  static void run(const void* const* srcs, int nsrc, void* out, int64_t lo, int64_t hi,
                  const Epilogue* epi) {
    S* o = static_cast<S*>(out);
    const S* accp = (epi && epi->accumulate) ? static_cast<const S*>(epi->accumulate) : nullptr;
    const bool scaled = epi && epi->has_scale;
    const double s = epi ? epi->scale : 1.0;
    const int64_t n = hi - lo;
    const int threads = omp_get_max_threads();
    if (n <= 0) return;
    if (static_cast<size_t>(n) * sizeof(S) < kParallelBytes || threads <= 1 || omp_in_parallel()) {
      run_serial(srcs, nsrc, o, accp, scaled, s, lo, hi);
      return;
    }
    const int64_t per = ((n + threads - 1) / threads + 511) / 512 * 512;
#pragma omp parallel for schedule(static)
    for (int t = 0; t < threads; ++t) {
      const int64_t a = lo + static_cast<int64_t>(t) * per;
      const int64_t b = std::min(hi, a + per);
      if (a < b) run_serial(srcs, nsrc, o, accp, scaled, s, a, b);
    }
  }
};

// Running fold for Scan / Exscan: dsts[k][i] = combine of srcs[0..k][i] (exclusive: of srcs[0..k-1][i], zero for
// k = 0) for i in [lo, hi).  Per element this is exactly CpuReduceRange's fold over the first sources, so a rank that
// folds its own prefix and a slice owner that writes everybody's prefixes produce the same bits.
template <DType DT, ReduceOp OP> struct CpuScanRange {
  using E = Elem<DT>;
  using S = typename E::storage;
  using A = typename E::acc;
  using C = Combine<OP, A, E::is_float>;

  static void run_serial(const void* const* srcs, void* const* dsts, int nsrc, bool exclusive, int64_t lo, int64_t hi) {
    constexpr int kBlock = 512;
    A buf[kBlock];
    for (int64_t b0 = lo; b0 < hi; b0 += kBlock) {
      const int n = static_cast<int>(std::min<int64_t>(kBlock, hi - b0));
      for (int k = 0; k < nsrc; ++k) {
        S* d = static_cast<S*>(dsts[k]) + b0;
        if (exclusive) {
          if (k == 0) std::memset(d, 0, static_cast<size_t>(n) * sizeof(S));
          else for (int j = 0; j < n; ++j) d[j] = E::store(buf[j]);
          if (k == nsrc - 1) break;
        }
        const S* sk = static_cast<const S*>(srcs[k]) + b0;
        if (k == 0) for (int j = 0; j < n; ++j) buf[j] = normalise_single<OP, A>(E::load(sk[j]));
        else for (int j = 0; j < n; ++j) buf[j] = C::apply(buf[j], E::load(sk[j]));
        if (!exclusive) for (int j = 0; j < n; ++j) d[j] = E::store(buf[j]);
      }
    }
  }

  static void run(const void* const* srcs, void* const* dsts, int nsrc, bool exclusive, int64_t lo, int64_t hi) {
    const int64_t n = hi - lo;
    const int threads = omp_get_max_threads();
    if (n <= 0) return;
    if (static_cast<size_t>(n) * sizeof(S) < kParallelBytes || threads <= 1 || omp_in_parallel()) {
      run_serial(srcs, dsts, nsrc, exclusive, lo, hi);
      return;
    }
    const int64_t per = ((n + threads - 1) / threads + 511) / 512 * 512;
#pragma omp parallel for schedule(static)
    for (int t = 0; t < threads; ++t) {
      const int64_t a = lo + static_cast<int64_t>(t) * per;
      const int64_t b = std::min(hi, a + per);
      if (a < b) run_serial(srcs, dsts, nsrc, exclusive, a, b);
    }
  }
};

// dst[i] = acc[i] + src[i]  (phase-2 epilogue of the two-phase allreduce)
template <DType DT, ReduceOp OP> struct CpuAccumulateCopy {
  static void run(const void* src, const void* acc, void* dst, int64_t lo, int64_t hi) {
    using E = Elem<DT>;
    using S = typename E::storage;
    const S* s = static_cast<const S*>(src);
    const S* a = static_cast<const S*>(acc);
    S* d = static_cast<S*>(dst);
    for (int64_t i = lo; i < hi; ++i) d[i] = E::store(E::load(a[i]) + E::load(s[i]));
  }
};

inline void copy_rows(const SlabJob& j, const char* src, char* dst, int64_t es) {
  const size_t run_bytes = static_cast<size_t>(j.run * es);
  for (int64_t i0 = 0; i0 < j.n[0]; ++i0)
    for (int64_t i1 = 0; i1 < j.n[1]; ++i1)
      for (int64_t i2 = 0; i2 < j.n[2]; ++i2) {
        const int64_t so = j.src_off + i0 * j.ss[0] + i1 * j.ss[1] + i2 * j.ss[2];
        const int64_t d_o = j.dst_off + i0 * j.ds[0] + i1 * j.ds[1] + i2 * j.ds[2];
        std::memcpy(dst + d_o * es, src + so * es, run_bytes);
      }
}

template <DType DT, ReduceOp OP> struct CpuReduceBox {
  static void run(const SlabJob& j, const char* const* srcs, int nsrc, char* out, const Epilogue* epi) {
    const int64_t es = dtype_size(DT);
    for (int64_t i0 = 0; i0 < j.n[0]; ++i0)
      for (int64_t i1 = 0; i1 < j.n[1]; ++i1)
        for (int64_t i2 = 0; i2 < j.n[2]; ++i2) {
          const int64_t so = j.src_off + i0 * j.ss[0] + i1 * j.ss[1] + i2 * j.ss[2];
          const int64_t d_o = j.dst_off + i0 * j.ds[0] + i1 * j.ds[1] + i2 * j.ds[2];
          const void* row_srcs[kMaxRanks];
          for (int k = 0; k < nsrc; ++k) row_srcs[k] = srcs[k] + so * es;
          Epilogue e;
          if (epi) {
            e = *epi;
            if (e.accumulate) e.accumulate = static_cast<const char*>(e.accumulate) + d_o * es;
          }
          CpuReduceRange<DT, OP>::run(row_srcs, nsrc, out + d_o * es, 0, j.run, epi ? &e : nullptr);
        }
  }
};

}  // namespace m4t
