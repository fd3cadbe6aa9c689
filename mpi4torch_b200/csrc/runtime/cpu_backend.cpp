#include "cpu_backend.h"

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <cerrno>
#include <cstring>

#include <omp.h>

#include "host_kernels.h"
#include "reduce_ops.h"

namespace m4t {

namespace {

constexpr size_t kMinArena = 1u << 20;
constexpr int64_t kTwoPhaseBytes = 256 * 1024;
constexpr int64_t kPieceBytes = 8 << 20;  // larger Allreduces are done in pieces of this size

size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace

CpuBackend::CpuBackend(Control& ctl) : ctl_(ctl) {}

CpuBackend::~CpuBackend() {
  for (int par = 0; par < 2; ++par) {
    if (own_[par].ptr) {
      munmap(own_[par].ptr, own_[par].cap);
      shm_unlink(arena_name(ctl_.rank(), par, own_[par].gen).c_str());
    }
    for (int p = 0; p < kMaxRanks; ++p)
      if (peers_[p][par].ptr) munmap(peers_[p][par].ptr, peers_[p][par].cap);
  }
  // drop payload segments of messages that were never received
  for (int s = 0; s < kMaxRanks; ++s)
    for (auto& d : unexpected_[s])
      if (d.kind == 1) shm_unlink(msg_name(s, ctl_.rank(), d.seq).c_str());
}

std::string CpuBackend::arena_name(int rank, int par, uint64_t gen) const {
  return ctl_.seg_name("a" + std::to_string(rank) + "_" + std::to_string(par) + "_" + std::to_string(gen));
}

std::string CpuBackend::msg_name(int src, int dst, uint64_t seq) const {
  return ctl_.seg_name("m" + std::to_string(src) + "_" + std::to_string(dst) + "_" + std::to_string(seq));
}

char* CpuBackend::stage(int par, size_t bytes) {
  Mapping& m = own_[par];
  if (bytes <= m.cap) return m.ptr;
  const size_t newcap = round_up(std::max({bytes, 2 * m.cap, kMinArena}), 4096);
  const uint64_t newgen = m.gen + 1;
  const std::string name = arena_name(ctl_.rank(), par, newgen);
  shm_unlink(name.c_str());
  int fd = shm_open(name.c_str(), O_CREAT | O_EXCL | O_RDWR, 0600);
  M4T_CHECK(fd >= 0, "shm_open(" << name << ") failed: " << std::strerror(errno));
  M4T_CHECK(ftruncate(fd, static_cast<off_t>(newcap)) == 0,
            "ftruncate(" << newcap << ") failed: " << std::strerror(errno) << " (is /dev/shm large enough?)");
  void* p = mmap(nullptr, newcap, PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
  close(fd);
  M4T_CHECK(p != MAP_FAILED, "mmap of arena failed: " << std::strerror(errno));
  if (m.ptr) {
    // Safe: by the parity argument no peer can still be reading the arena that
    // served the op two steps ago.
    munmap(m.ptr, m.cap);
    shm_unlink(arena_name(ctl_.rank(), par, m.gen).c_str());
  }
  m.ptr = static_cast<char*>(p);
  m.cap = newcap;
  m.gen = newgen;
  auto& slot = ctl_.block()->slots[ctl_.rank()];
  slot.arena_cap[par].store(newcap, std::memory_order_relaxed);
  slot.arena_gen[par].store(newgen, std::memory_order_release);
  return m.ptr;
}

const char* CpuBackend::peer_arena(int peer, int par) {
  if (peer == ctl_.rank()) return own_[par].ptr;
  auto& slot = ctl_.block()->slots[peer];
  const uint64_t gen = slot.arena_gen[par].load(std::memory_order_acquire);
  Mapping& m = peers_[peer][par];
  if (gen != m.gen) {
    if (m.ptr) munmap(m.ptr, m.cap);
    m = Mapping{};
    const size_t cap = slot.arena_cap[par].load(std::memory_order_relaxed);
    const std::string name = arena_name(peer, par, gen);
    int fd = shm_open(name.c_str(), O_RDWR, 0600);
    M4T_CHECK(fd >= 0, "shm_open(" << name << ") failed: " << std::strerror(errno));
    void* p = mmap(nullptr, cap, PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
    close(fd);
    M4T_CHECK(p != MAP_FAILED, "mmap of peer arena failed: " << std::strerror(errno));
    m.ptr = static_cast<char*>(p);
    m.cap = cap;
    m.gen = gen;
  }
  return m.ptr;
}

void CpuBackend::allreduce(const void* in, void* out, int64_t n, DType dt, ReduceOp op,
                           const Epilogue& epi, void*) {
  check_op_dtype(op, dt);
  const int P = ctl_.size(), r = ctl_.rank();
  const int64_t es = dtype_size(dt);
  const size_t bytes = static_cast<size_t>(n * es);
  if (P == 1) {
    const void* srcs[1] = {in};
    M4T_DISPATCH_DTYPE_OP(dt, op, CpuReduceRange, srcs, 1, out, 0, n, &epi);
    return;
  }
  if (static_cast<int64_t>(bytes) > kPieceBytes) {
    // cache-sized pieces: the staged copy of a piece is still in the last-level cache when the peers reduce it and when
    // the result is copied out (64 MiB at 4 ranks: 46 ms in one piece, a third of that in 8 MiB pieces)
    const int64_t step = kPieceBytes / es;
    for (int64_t off = 0; off < n; off += step) {
      const int64_t len = std::min(step, n - off);
      Epilogue e = epi;
      if (e.accumulate) e.accumulate = static_cast<const char*>(e.accumulate) + off * es;
      allreduce(static_cast<const char*>(in) + off * es, static_cast<char*>(out) + off * es, len, dt, op, e, nullptr);
    }
    return;
  }
  const int par = static_cast<int>(op_seq_++ & 1);
  const bool two_phase = static_cast<int64_t>(bytes) >= kTwoPhaseBytes;
  char* mine = stage(par, two_phase ? 2 * bytes : bytes);
  if (bytes) par_memcpy(mine, in, bytes);
  ctl_.barrier();
  const void* srcs[kMaxRanks];
  for (int p = 0; p < P; ++p) srcs[p] = peer_arena(p, par);
  if (!two_phase) {
    M4T_DISPATCH_DTYPE_OP(dt, op, CpuReduceRange, srcs, P, out, 0, n, &epi);
    return;
  }
  // phase 1: reduce my slice into the result half of my arena (scale fused)
  Epilogue e1;
  e1.scale = epi.scale;
  e1.has_scale = epi.has_scale;
  const int64_t lo = n * r / P, hi = n * (r + 1) / P;
  M4T_DISPATCH_DTYPE_OP(dt, op, CpuReduceRange, srcs, P, mine + bytes, lo, hi, &e1);
  ctl_.barrier();
  // phase 2: collect every owner's slice (accumulate fused)
  for (int p = 0; p < P; ++p) {
    const int64_t plo = n * p / P, phi = n * (p + 1) / P;
    const char* res = peer_arena(p, par) + bytes;
    if (epi.accumulate) {
      M4T_DISPATCH_DTYPE_OP(dt, ReduceOp::SUM, CpuAccumulateCopy, res, epi.accumulate, out, plo, phi);
    } else {
      par_memcpy(static_cast<char*>(out) + plo * es, res + plo * es, static_cast<size_t>((phi - plo) * es));
    }
  }
}

void CpuBackend::bcast(void* buf, int64_t n, DType dt, int root, void*) {
  const int P = ctl_.size(), r = ctl_.rank();
  M4T_CHECK(root >= 0 && root < P, "Bcast_: root " << root << " out of range");
  if (P == 1) return;
  const size_t bytes = static_cast<size_t>(n * dtype_size(dt));
  const int par = static_cast<int>(op_seq_++ & 1);
  if (r == root) {
    char* mine = stage(par, bytes);
    if (bytes) par_memcpy(mine, buf, bytes);
  }
  ctl_.barrier();
  if (r != root && bytes) par_memcpy(buf, peer_arena(root, par), bytes);
}

void CpuBackend::reduce(void* buf, int64_t n, DType dt, ReduceOp op, int root, void*) {
  check_op_dtype(op, dt);
  const int P = ctl_.size(), r = ctl_.rank();
  M4T_CHECK(root >= 0 && root < P, "Reduce_: root " << root << " out of range");
  const size_t bytes = static_cast<size_t>(n * dtype_size(dt));
  if (P == 1) {
    const void* srcs[1] = {buf};
    M4T_DISPATCH_DTYPE_OP(dt, op, CpuReduceRange, srcs, 1, buf, 0, n, nullptr);
    return;
  }
  const int par = static_cast<int>(op_seq_++ & 1);
  char* mine = stage(par, bytes);
  if (bytes) par_memcpy(mine, buf, bytes);
  ctl_.barrier();
  if (r == root) {
    const void* srcs[kMaxRanks];
    for (int p = 0; p < P; ++p) srcs[p] = peer_arena(p, par);
    M4T_DISPATCH_DTYPE_OP(dt, op, CpuReduceRange, srcs, P, buf, 0, n, nullptr);
  } else if (bytes) {
    std::memset(buf, 0, bytes);
  }
}

void CpuBackend::scan(const void* in, void* out, int64_t n, DType dt, ReduceOp op, bool exclusive, bool reverse, void*) {
  check_op_dtype(op, dt);
  const int P = ctl_.size(), r = ctl_.rank();
  const int64_t es = dtype_size(dt);
  const size_t bytes = static_cast<size_t>(n * es);
  if (n == 0) return;
  if (P == 1) {
    if (exclusive) {
      std::memset(out, 0, bytes);
    } else {
      const void* srcs[1] = {in};
      M4T_DISPATCH_DTYPE_OP(dt, op, CpuReduceRange, srcs, 1, out, 0, n, nullptr);
    }
    return;
  }
  if (static_cast<int64_t>(bytes) > kPieceBytes) {  // cache-sized pieces, as in allreduce
    const int64_t step = kPieceBytes / es;
    for (int64_t off = 0; off < n; off += step)
      scan(static_cast<const char*>(in) + off * es, static_cast<char*>(out) + off * es, std::min(step, n - off), dt, op,
           exclusive, reverse, nullptr);
    return;
  }
  auto fold_rank = [&](int k) { return reverse ? P - 1 - k : k; };  // rank at position k of the fold
  const int me = reverse ? P - 1 - r : r;
  const int par = static_cast<int>(op_seq_++ & 1);
  const bool two_phase = static_cast<int64_t>(bytes) >= kTwoPhaseBytes;
  char* mine = stage(par, two_phase ? 2 * bytes : bytes);
  par_memcpy(mine, in, bytes);
  ctl_.barrier();
  const void* srcs[kMaxRanks];
  for (int k = 0; k < P; ++k) srcs[k] = peer_arena(fold_rank(k), par);
  if (!two_phase) {
    const int cnt = exclusive ? me : me + 1;
    if (cnt == 0) {
      std::memset(out, 0, bytes);
      return;
    }
    M4T_DISPATCH_DTYPE_OP(dt, op, CpuReduceRange, srcs, cnt, out, 0, n, nullptr);
    return;
  }
  // phase 1: the owner of slice r writes every rank's prefix of it into that rank's result half
  void* dsts[kMaxRanks];
  for (int k = 0; k < P; ++k) dsts[k] = const_cast<char*>(static_cast<const char*>(srcs[k])) + bytes;
  M4T_DISPATCH_DTYPE_OP(dt, op, CpuScanRange, srcs, dsts, P, exclusive, n * r / P, n * (r + 1) / P);
  ctl_.barrier();
  // phase 2: my prefixes of all slices are in my own result half
  par_memcpy(out, mine + bytes, bytes);
}

void CpuBackend::pull(const PullPlan& plan, const void* in, void* out, DType dt, void*) {
  const int P = ctl_.size(), r = ctl_.rank();
  const int64_t es = dtype_size(dt);
  if (P == 1) {
    for (const auto& j : plan.jobs) copy_rows(j, static_cast<const char*>(in), static_cast<char*>(out), es);
    return;
  }
  const int par = static_cast<int>(op_seq_++ & 1);
  if (plan.stage_elems > 0) {
    const size_t bytes = static_cast<size_t>(plan.stage_elems * es);
    char* mine = stage(par, bytes);
    par_memcpy(mine, in, bytes);
  }
  ctl_.barrier();
  for (const auto& j : plan.jobs) {
    const char* src = (j.peer == r) ? static_cast<const char*>(in) : peer_arena(j.peer, par);
    copy_rows(j, src, static_cast<char*>(out), es);
  }
}

void CpuBackend::reduce_pull(const ReducePlan& plan, const void* in, void* out, DType dt, ReduceOp op,
                             const Epilogue& epi, void*) {
  check_op_dtype(op, dt);
  const int P = ctl_.size(), r = ctl_.rank();
  const int64_t es = dtype_size(dt);
  const char* srcs[kMaxRanks];
  if (P == 1) {
    srcs[0] = static_cast<const char*>(in);
    if (plan.out_elems > 0) {
      M4T_DISPATCH_DTYPE_OP(dt, op, CpuReduceBox, plan.box, srcs, 1, static_cast<char*>(out), &epi);
    }
    return;
  }
  const int par = static_cast<int>(op_seq_++ & 1);
  const size_t bytes = static_cast<size_t>(plan.stage_elems * es);
  char* mine = stage(par, bytes);
  if (bytes) par_memcpy(mine, in, bytes);
  ctl_.barrier();
  if (plan.out_elems == 0) return;
  for (int p = 0; p < P; ++p) srcs[p] = (p == r) ? static_cast<const char*>(in) : peer_arena(p, par);
  M4T_DISPATCH_DTYPE_OP(dt, op, CpuReduceBox, plan.box, srcs, P, static_cast<char*>(out), &epi);
}

// ---------------------------------------------------------------------------
// point-to-point: eager, buffered sends through per-pair descriptor rings
// ---------------------------------------------------------------------------
int64_t CpuBackend::isend(const void* buf, int64_t bytes, int dest, int64_t tag, void*) {
  const int P = ctl_.size(), r = ctl_.rank();
  M4T_CHECK(dest >= 0 && dest < P, "Isend: destination rank " << dest << " out of range");
  PairRing& ring = ctl_.block()->rings[r][dest];
  MsgDesc d{};
  d.seq = ++send_seq_[dest];
  d.tag = tag;
  d.bytes = static_cast<uint64_t>(bytes);
  if (bytes <= kInlineBytes) {
    d.kind = 0;
    if (bytes) std::memcpy(d.inline_data, buf, static_cast<size_t>(bytes));
  } else {
    d.kind = 1;
    const std::string name = msg_name(r, dest, d.seq);
    shm_unlink(name.c_str());
    int fd = shm_open(name.c_str(), O_CREAT | O_EXCL | O_RDWR, 0600);
    M4T_CHECK(fd >= 0, "shm_open(" << name << ") failed: " << std::strerror(errno));
    M4T_CHECK(ftruncate(fd, static_cast<off_t>(bytes)) == 0,
              "ftruncate(" << bytes << ") failed: " << std::strerror(errno));
    void* p = mmap(nullptr, static_cast<size_t>(bytes), PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
    close(fd);
    M4T_CHECK(p != MAP_FAILED, "mmap of message segment failed: " << std::strerror(errno));
    par_memcpy(p, buf, static_cast<size_t>(bytes));
    munmap(p, static_cast<size_t>(bytes));
  }
  const uint64_t head = ring.head.load(std::memory_order_relaxed);
  ctl_.wait_until([&] { return head - ring.tail.load(std::memory_order_acquire) < kMailboxDepth; },
                  "space in the send ring");
  ring.entries[head % kMailboxDepth] = d;
  ring.head.store(head + 1, std::memory_order_release);
  const int64_t id = next_request_++;
  Request rq;
  rq.is_recv = false;
  rq.peer = dest;
  rq.tag = tag;
  rq.bytes = bytes;
  requests_[id] = rq;
  return id;
}

int64_t CpuBackend::irecv(void* buf, int64_t bytes, int source, int64_t tag, void*) {
  const int P = ctl_.size();
  M4T_CHECK(source >= 0 && source < P, "Irecv: source rank " << source << " out of range");
  const int64_t id = next_request_++;
  Request rq;
  rq.is_recv = true;
  rq.buf = buf;
  rq.bytes = bytes;
  rq.peer = source;
  rq.tag = tag;
  requests_[id] = rq;
  return id;
}

void CpuBackend::deliver(const MsgDesc& d, int source, Request& rq) {
  M4T_CHECK(static_cast<int64_t>(d.bytes) <= rq.bytes,
            "message truncated: " << d.bytes << " bytes sent by rank " << source << " (tag " << d.tag
                                  << ") into a " << rq.bytes << "-byte receive buffer");
  if (d.kind == 0) {
    if (d.bytes) std::memcpy(rq.buf, d.inline_data, d.bytes);
    return;
  }
  const std::string name = msg_name(source, ctl_.rank(), d.seq);
  int fd = shm_open(name.c_str(), O_RDWR, 0600);
  M4T_CHECK(fd >= 0, "shm_open(" << name << ") failed: " << std::strerror(errno));
  void* p = mmap(nullptr, d.bytes, PROT_READ, MAP_SHARED, fd, 0);
  close(fd);
  M4T_CHECK(p != MAP_FAILED, "mmap of message segment failed: " << std::strerror(errno));
  par_memcpy(rq.buf, p, d.bytes);
  munmap(p, d.bytes);
  shm_unlink(name.c_str());
}

void CpuBackend::wait(int64_t request, void*) {
  auto it = requests_.find(request);
  M4T_CHECK(it != requests_.end(), "Wait: unknown or already completed request " << request
                                       << " (a WaitHandle may only be waited on once)");
  Request rq = it->second;
  requests_.erase(it);
  if (!rq.is_recv) return;  // sends are buffered: complete at post time
  const int src = rq.peer;
  auto& pending = unexpected_[src];
  for (auto u = pending.begin(); u != pending.end(); ++u) {
    if (u->tag == rq.tag) {
      deliver(*u, src, rq);
      pending.erase(u);
      return;
    }
  }
  PairRing& ring = ctl_.block()->rings[src][ctl_.rank()];
  for (;;) {
    const uint64_t tail = ring.tail.load(std::memory_order_relaxed);
    ctl_.wait_until([&] { return ring.head.load(std::memory_order_acquire) > tail; }, "a matching message");
    MsgDesc d = ring.entries[tail % kMailboxDepth];
    ring.tail.store(tail + 1, std::memory_order_release);
    if (d.tag == rq.tag) {
      deliver(d, src, rq);
      return;
    }
    pending.push_back(d);
  }
}

}  // namespace m4t
