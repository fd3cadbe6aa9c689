#include "net_backend.h"

#include <cstring>

#include "cpu_backend.h"
#include "host_kernels.h"

namespace m4t {

namespace {
// grow-only scratch: large collectives reuse the same pages instead of faulting fresh ones in on every call
void grow(NetBuffer& b, size_t n) {
  if (b.size() < n) b.allocate(n + n / 4);
}

constexpr int64_t kDirectBytes = 64 * 1024;  // below: every rank receives every contribution
constexpr int kDescWords = 8;                // src_off, n[3], ss[3], run

void push_desc(std::vector<int64_t>& v, const SlabJob& j) {
  v.push_back(j.src_off);
  for (int i = 0; i < 3; ++i) v.push_back(j.n[i]);
  for (int i = 0; i < 3; ++i) v.push_back(j.ss[i]);
  v.push_back(j.run);
}

SlabJob read_desc(const int64_t* w) {
  SlabJob j;
  j.src_off = w[0];
  for (int i = 0; i < 3; ++i) j.n[i] = w[1 + i];
  for (int i = 0; i < 3; ++i) j.ss[i] = w[4 + i];
  j.run = w[7];
  return j;
}

// rows of a box, packed contiguously in loop order (i0, i1, i2)
void pack_box(const SlabJob& j, const char* src, char* dst, int64_t es) {
  const size_t run_bytes = static_cast<size_t>(j.run * es);
  for (int64_t i0 = 0; i0 < j.n[0]; ++i0)
    for (int64_t i1 = 0; i1 < j.n[1]; ++i1)
      for (int64_t i2 = 0; i2 < j.n[2]; ++i2) {
        std::memcpy(dst, src + (j.src_off + i0 * j.ss[0] + i1 * j.ss[1] + i2 * j.ss[2]) * es, run_bytes);
        dst += run_bytes;
      }
}

void unpack_box(const SlabJob& j, const char* src, char* dst, int64_t es) {
  const size_t run_bytes = static_cast<size_t>(j.run * es);
  for (int64_t i0 = 0; i0 < j.n[0]; ++i0)
    for (int64_t i1 = 0; i1 < j.n[1]; ++i1)
      for (int64_t i2 = 0; i2 < j.n[2]; ++i2) {
        std::memcpy(dst + (j.dst_off + i0 * j.ds[0] + i1 * j.ds[1] + i2 * j.ds[2]) * es, src, run_bytes);
        src += run_bytes;
      }
}

// Serves the box requests of every peer out of `in` and returns the packed answers (kept alive by the caller until
// the sends are complete).  reqs[p] = descriptor words received from p.
void serve_requests(NetLink& link, int64_t data_tag, const std::vector<NetBuffer>& reqs, const char* in, int64_t es,
                    std::vector<NetBuffer>& answers, std::vector<uint64_t>& ops) {
  const int P = link.size(), r = link.rank();
  answers.clear();
  answers.resize(static_cast<size_t>(P));
  for (int p = 0; p < P; ++p) {
    if (p == r || reqs[static_cast<size_t>(p)].empty()) continue;
    const auto* w = reinterpret_cast<const int64_t*>(reqs[static_cast<size_t>(p)].data());
    const size_t njobs = reqs[static_cast<size_t>(p)].size() / (kDescWords * sizeof(int64_t));
    if (njobs == 1) {
      const SlabJob j = read_desc(w);
      if (j.rows() == 1) {  // one contiguous run: straight out of the input, no packing
        ops.push_back(link.send(p, kNetColl, data_tag, in + j.src_off * es, static_cast<size_t>(j.run * es)));
        continue;
      }
    }
    size_t total = 0;
    for (size_t k = 0; k < njobs; ++k) total += static_cast<size_t>(read_desc(w + k * kDescWords).elems() * es);
    auto& buf = answers[static_cast<size_t>(p)];
    buf.allocate(total);
    char* dst = buf.data();
    for (size_t k = 0; k < njobs; ++k) {
      const SlabJob j = read_desc(w + k * kDescWords);
      pack_box(j, in, dst, es);
      dst += j.elems() * es;
    }
    ops.push_back(link.send(p, kNetColl, data_tag, buf.data(), buf.size()));
  }
}
}  // namespace

void NetBackend::allreduce(const void* in, void* out, int64_t n, DType dt, ReduceOp op, const Epilogue& epi, void*) {
  check_op_dtype(op, dt);
  const int P = size(), r = rank();
  const int64_t es = dtype_size(dt);
  const size_t bytes = static_cast<size_t>(n * es);
  if (P == 1) {
    const void* srcs[1] = {in};
    M4T_DISPATCH_DTYPE_OP(dt, op, CpuReduceRange, srcs, 1, out, 0, n, &epi);
    return;
  }
  const int64_t tag = link_->next_seq() * 4;
  NetEngine& eng = link_->engine();
  const void* srcs[kMaxRanks];
  std::vector<uint64_t> ops;
  if (static_cast<int64_t>(bytes) <= kDirectBytes || n < P) {
    NetBuffer tmp;
    tmp.allocate(bytes * static_cast<size_t>(P - 1));
    for (int p = 0, k = 0; p < P; ++p) {
      if (p == r) {
        srcs[p] = in;
        continue;
      }
      char* slot = tmp.data() + bytes * static_cast<size_t>(k++);
      srcs[p] = slot;
      ops.push_back(link_->recv(p, kNetColl, tag, slot, bytes));
    }
    for (int p = 0; p < P; ++p)
      if (p != r) ops.push_back(link_->send(p, kNetColl, tag, in, bytes));
    eng.wait_all(ops);
    M4T_DISPATCH_DTYPE_OP(dt, op, CpuReduceRange, srcs, P, out, 0, n, &epi);
    return;
  }
  // reduce-scatter by direct exchange (rank p reduces slice p, sources in rank order exactly like the shared-memory
  // backend), then all-gather of the finished slices; every rank sends and receives (P-1)/P of the message twice
  auto lo = [&](int p) { return n * p / P; };
  const int64_t mylo = lo(r), mylen = lo(r + 1) - lo(r);
  NetBuffer& tmp = scratch_[0];
  NetBuffer& res = scratch_[1];
  grow(tmp, static_cast<size_t>(mylen * es) * static_cast<size_t>(P - 1));
  grow(res, static_cast<size_t>(mylen * es));
  const size_t res_bytes = static_cast<size_t>(mylen * es);
  for (int p = 0, k = 0; p < P; ++p) {
    if (p == r) {
      srcs[p] = static_cast<const char*>(in) + mylo * es;
      continue;
    }
    char* slot = tmp.data() + static_cast<size_t>(mylen * es) * static_cast<size_t>(k++);
    srcs[p] = slot;
    ops.push_back(link_->recv(p, kNetColl, tag, slot, static_cast<size_t>(mylen * es)));
  }
  for (int p = 0; p < P; ++p)
    if (p != r)
      ops.push_back(link_->send(p, kNetColl, tag, static_cast<const char*>(in) + lo(p) * es,
                                static_cast<size_t>((lo(p + 1) - lo(p)) * es)));
  eng.wait_all(ops);
  ops.clear();
  Epilogue e1;
  e1.scale = epi.scale;
  e1.has_scale = epi.has_scale;
  M4T_DISPATCH_DTYPE_OP(dt, op, CpuReduceRange, srcs, P, res.data(), 0, mylen, &e1);
  // phase 2 (accumulate fused while the slices land)
  NetBuffer& land = scratch_[2];
  if (epi.accumulate) grow(land, bytes);
  char* dst = epi.accumulate ? land.data() : static_cast<char*>(out);
  for (int p = 0; p < P; ++p)
    if (p != r) ops.push_back(link_->recv(p, kNetColl, tag + 1, dst + lo(p) * es, static_cast<size_t>((lo(p + 1) - lo(p)) * es)));
  for (int p = 0; p < P; ++p)
    if (p != r) ops.push_back(link_->send(p, kNetColl, tag + 1, res.data(), res_bytes));
  if (mylen) std::memcpy(dst + mylo * es, res.data(), res_bytes);
  eng.wait_all(ops);
  if (epi.accumulate) {
    M4T_DISPATCH_DTYPE_OP(dt, ReduceOp::SUM, CpuAccumulateCopy, land.data(), epi.accumulate, out, 0, n);
  }
}

void NetBackend::bcast(void* buf, int64_t n, DType dt, int root, void*) {
  const int P = size(), r = rank();
  M4T_CHECK(root >= 0 && root < P, "Bcast_: root " << root << " out of range");
  if (P == 1) return;
  const size_t bytes = static_cast<size_t>(n * dtype_size(dt));
  const int64_t tag = link_->next_seq() * 4;
  NetEngine& eng = link_->engine();
  const int v = (r - root + P) % P;  // binomial tree on ranks relative to the root
  int mask = 1;
  while (mask < P) {
    if (v & mask) {
      eng.wait(link_->recv((v - mask + root) % P, kNetColl, tag, buf, bytes));
      break;
    }
    mask <<= 1;
  }
  mask >>= 1;
  std::vector<uint64_t> ops;
  while (mask > 0) {
    if (v + mask < P) ops.push_back(link_->send((v + mask + root) % P, kNetColl, tag, buf, bytes));
    mask >>= 1;
  }
  eng.wait_all(ops);
}

void NetBackend::reduce(void* buf, int64_t n, DType dt, ReduceOp op, int root, void*) {
  check_op_dtype(op, dt);
  const int P = size(), r = rank();
  M4T_CHECK(root >= 0 && root < P, "Reduce_: root " << root << " out of range");
  const size_t bytes = static_cast<size_t>(n * dtype_size(dt));
  if (P == 1) {
    const void* srcs[1] = {buf};
    M4T_DISPATCH_DTYPE_OP(dt, op, CpuReduceRange, srcs, 1, buf, 0, n, nullptr);
    return;
  }
  const int64_t tag = link_->next_seq() * 4;
  NetEngine& eng = link_->engine();
  if (r != root) {
    eng.wait(link_->send(root, kNetColl, tag, buf, bytes));
    if (bytes) std::memset(buf, 0, bytes);  // reference csrc/extension.cpp:443-447
    return;
  }
  // the root combines the contributions in rank order (same result as the shared-memory backend)
  NetBuffer tmp;
  tmp.allocate(bytes * static_cast<size_t>(P - 1));
  const void* srcs[kMaxRanks];
  std::vector<uint64_t> ops;
  for (int p = 0, k = 0; p < P; ++p) {
    if (p == r) {
      srcs[p] = buf;
      continue;
    }
    char* slot = tmp.data() + bytes * static_cast<size_t>(k++);
    srcs[p] = slot;
    ops.push_back(link_->recv(p, kNetColl, tag, slot, bytes));
  }
  eng.wait_all(ops);
  M4T_DISPATCH_DTYPE_OP(dt, op, CpuReduceRange, srcs, P, buf, 0, n, nullptr);
}

void NetBackend::scan(const void* in, void* out, int64_t n, DType dt, ReduceOp op, bool exclusive, bool reverse, void*) {
  check_op_dtype(op, dt);
  const int P = size(), r = rank();
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
  auto fold_rank = [&](int k) { return reverse ? P - 1 - k : k; };  // rank at position k of the fold
  auto fold_pos = [&](int p) { return reverse ? P - 1 - p : p; };
  const int me = fold_pos(r);
  const int64_t tag = link_->next_seq() * 4;
  NetEngine& eng = link_->engine();
  const void* srcs[kMaxRanks];
  std::vector<uint64_t> ops;
  if (static_cast<int64_t>(bytes) <= kDirectBytes || n < P) {
    // my vector goes to the ranks after me in the fold; I receive the ones before me and fold them in order
    NetBuffer& tmp = scratch_[0];
    grow(tmp, bytes * static_cast<size_t>(me));
    for (int k = 0; k < me; ++k) {
      char* slot = tmp.data() + bytes * static_cast<size_t>(k);
      srcs[k] = slot;
      ops.push_back(link_->recv(fold_rank(k), kNetColl, tag, slot, bytes));
    }
    for (int k = me + 1; k < P; ++k) ops.push_back(link_->send(fold_rank(k), kNetColl, tag, in, bytes));
    eng.wait_all(ops);
    srcs[me] = in;
    const int cnt = exclusive ? me : me + 1;
    if (cnt == 0) std::memset(out, 0, bytes);
    else M4T_DISPATCH_DTYPE_OP(dt, op, CpuReduceRange, srcs, cnt, out, 0, n, nullptr);
    return;
  }
  // the owner of slice p receives that slice from every rank, folds it in order and sends rank q its prefix of it:
  // every rank sends and receives (P-1)/P of the message twice, as in the Allreduce
  auto lo = [&](int p) { return n * p / P; };
  const int64_t mylo = lo(r), mylen = lo(r + 1) - lo(r);
  const size_t slice_bytes = static_cast<size_t>(mylen * es);
  NetBuffer& tmp = scratch_[0];
  NetBuffer& res = scratch_[1];
  grow(tmp, slice_bytes * static_cast<size_t>(P));
  grow(res, slice_bytes * static_cast<size_t>(P));
  void* dsts[kMaxRanks];
  for (int k = 0; k < P; ++k) {
    const int p = fold_rank(k);
    dsts[k] = p == r ? static_cast<char*>(out) + mylo * es : res.data() + slice_bytes * static_cast<size_t>(k);
    if (p == r) {
      srcs[k] = static_cast<const char*>(in) + mylo * es;
      continue;
    }
    char* slot = tmp.data() + slice_bytes * static_cast<size_t>(k);
    srcs[k] = slot;
    ops.push_back(link_->recv(p, kNetColl, tag, slot, slice_bytes));
  }
  for (int p = 0; p < P; ++p)
    if (p != r)
      ops.push_back(link_->send(p, kNetColl, tag, static_cast<const char*>(in) + lo(p) * es,
                                static_cast<size_t>((lo(p + 1) - lo(p)) * es)));
  eng.wait_all(ops);
  ops.clear();
  M4T_DISPATCH_DTYPE_OP(dt, op, CpuScanRange, srcs, dsts, P, exclusive, 0, mylen);
  for (int p = 0; p < P; ++p)
    if (p != r)
      ops.push_back(link_->recv(p, kNetColl, tag + 1, static_cast<char*>(out) + lo(p) * es,
                                static_cast<size_t>((lo(p + 1) - lo(p)) * es)));
  for (int k = 0; k < P; ++k)
    if (fold_rank(k) != r) ops.push_back(link_->send(fold_rank(k), kNetColl, tag + 1, dsts[k], slice_bytes));
  eng.wait_all(ops);
}

void NetBackend::pull(const PullPlan& plan, const void* in, void* out, DType dt, void*) {
  const int P = size(), r = rank();
  const int64_t es = dtype_size(dt);
  const char* cin = static_cast<const char*>(in);
  char* cout = static_cast<char*>(out);
  if (P == 1) {
    for (const auto& j : plan.jobs) copy_rows(j, cin, cout, es);
    return;
  }
  const int64_t seq = link_->next_seq();
  const int64_t req_tag = seq * 4, data_tag = seq * 4 + 1;
  NetEngine& eng = link_->engine();
  // what I want from whom
  std::vector<std::vector<int64_t>> want(static_cast<size_t>(P));
  std::vector<std::vector<const SlabJob*>> mine(static_cast<size_t>(P));
  for (const auto& j : plan.jobs) {
    if (j.peer == r) continue;
    push_desc(want[static_cast<size_t>(j.peer)], j);
    mine[static_cast<size_t>(j.peer)].push_back(&j);
  }
  std::vector<uint64_t> req_recv(static_cast<size_t>(P), 0), sends;
  for (int p = 0; p < P; ++p)
    if (p != r) req_recv[static_cast<size_t>(p)] = link_->recv(p, kNetColl, req_tag, nullptr, SIZE_MAX);
  for (int p = 0; p < P; ++p)
    if (p != r)
      sends.push_back(link_->send(p, kNetColl, req_tag, want[static_cast<size_t>(p)].data(),
                                  want[static_cast<size_t>(p)].size() * sizeof(int64_t)));
  // answers I expect
  std::vector<NetBuffer> got(static_cast<size_t>(P));
  std::vector<uint64_t> data_recv(static_cast<size_t>(P), 0);
  std::vector<bool> direct(static_cast<size_t>(P), false);
  for (int p = 0; p < P; ++p) {
    if (p == r || mine[static_cast<size_t>(p)].empty()) continue;
    const auto& js = mine[static_cast<size_t>(p)];
    if (js.size() == 1 && js[0]->rows() == 1) {  // one contiguous run: straight into the output
      data_recv[static_cast<size_t>(p)] =
          link_->recv(p, kNetColl, data_tag, cout + js[0]->dst_off * es, static_cast<size_t>(js[0]->run * es));
      direct[static_cast<size_t>(p)] = true;
      continue;
    }
    size_t total = 0;
    for (const SlabJob* j : js) total += static_cast<size_t>(j->elems() * es);
    got[static_cast<size_t>(p)].allocate(total);
    data_recv[static_cast<size_t>(p)] = link_->recv(p, kNetColl, data_tag, got[static_cast<size_t>(p)].data(), total);
  }
  for (const auto& j : plan.jobs)
    if (j.peer == r) copy_rows(j, cin, cout, es);
  std::vector<NetBuffer> reqs(static_cast<size_t>(P));
  for (int p = 0; p < P; ++p)
    if (p != r) eng.wait(req_recv[static_cast<size_t>(p)], &reqs[static_cast<size_t>(p)]);
  std::vector<NetBuffer> answers;
  serve_requests(*link_, data_tag, reqs, cin, es, answers, sends);
  for (int p = 0; p < P; ++p) {
    if (!data_recv[static_cast<size_t>(p)]) continue;
    eng.wait(data_recv[static_cast<size_t>(p)]);
    if (direct[static_cast<size_t>(p)]) continue;
    const char* src = got[static_cast<size_t>(p)].data();
    for (const SlabJob* j : mine[static_cast<size_t>(p)]) {
      unpack_box(*j, src, cout, es);
      src += j->elems() * es;
    }
  }
  eng.wait_all(sends);
}

void NetBackend::reduce_pull(const ReducePlan& plan, const void* in, void* out, DType dt, ReduceOp op, const Epilogue& epi,
                             void*) {
  check_op_dtype(op, dt);
  const int P = size(), r = rank();
  const int64_t es = dtype_size(dt);
  const char* cin = static_cast<const char*>(in);
  const char* srcs[kMaxRanks];
  if (P == 1) {
    srcs[0] = cin;
    if (plan.out_elems > 0) {
      M4T_DISPATCH_DTYPE_OP(dt, op, CpuReduceBox, plan.box, srcs, 1, static_cast<char*>(out), &epi);
    }
    return;
  }
  const int64_t seq = link_->next_seq();
  const int64_t req_tag = seq * 4, data_tag = seq * 4 + 1;
  NetEngine& eng = link_->engine();
  std::vector<int64_t> want;
  if (plan.out_elems > 0) push_desc(want, plan.box);
  std::vector<uint64_t> req_recv(static_cast<size_t>(P), 0), sends;
  for (int p = 0; p < P; ++p)
    if (p != r) req_recv[static_cast<size_t>(p)] = link_->recv(p, kNetColl, req_tag, nullptr, SIZE_MAX);
  for (int p = 0; p < P; ++p)
    if (p != r) sends.push_back(link_->send(p, kNetColl, req_tag, want.data(), want.size() * sizeof(int64_t)));
  const size_t box_bytes = plan.out_elems > 0 ? static_cast<size_t>(plan.box.elems() * es) : 0;
  std::vector<NetBuffer> got(static_cast<size_t>(P));
  std::vector<uint64_t> data_recv(static_cast<size_t>(P), 0);
  if (box_bytes) {
    for (int p = 0; p < P; ++p) {
      got[static_cast<size_t>(p)].allocate(box_bytes);
      if (p != r) data_recv[static_cast<size_t>(p)] = link_->recv(p, kNetColl, data_tag, got[static_cast<size_t>(p)].data(), box_bytes);
    }
    pack_box(plan.box, cin, got[static_cast<size_t>(r)].data(), es);
  }
  std::vector<NetBuffer> reqs(static_cast<size_t>(P));
  for (int p = 0; p < P; ++p)
    if (p != r) eng.wait(req_recv[static_cast<size_t>(p)], &reqs[static_cast<size_t>(p)]);
  std::vector<NetBuffer> answers;
  serve_requests(*link_, data_tag, reqs, cin, es, answers, sends);
  if (box_bytes) {
    for (int p = 0; p < P; ++p) {
      if (p != r) eng.wait(data_recv[static_cast<size_t>(p)]);
      srcs[p] = got[static_cast<size_t>(p)].data();
    }
    SlabJob packed = plan.box;  // sources are the packed answers, the destination keeps the plan's strides
    packed.src_off = 0;
    packed.ss[2] = packed.run;
    packed.ss[1] = packed.n[2] * packed.run;
    packed.ss[0] = packed.n[1] * packed.n[2] * packed.run;
    M4T_DISPATCH_DTYPE_OP(dt, op, CpuReduceBox, packed, srcs, P, static_cast<char*>(out), &epi);
  }
  eng.wait_all(sends);
}

int64_t NetBackend::isend(const void* buf, int64_t bytes, int dest, int64_t tag, void*) {
  M4T_CHECK(dest >= 0 && dest < size(), "Isend: destination rank " << dest << " out of range");
  // buffered (the engine keeps a copy): a handle that is dropped without Wait must not leave the engine reading
  // freed memory, and like the shared-memory backend the send then completes locally
  const uint64_t op = link_->engine().post_send(link_->members()[static_cast<size_t>(dest)], link_->comm_id(), kNetP2p, tag,
                                                buf, static_cast<size_t>(bytes), /*copy=*/true);
  const int64_t id = next_request_++;
  requests_[id] = op;
  return id;
}

int64_t NetBackend::irecv(void* buf, int64_t bytes, int source, int64_t tag, void*) {
  M4T_CHECK(source >= 0 && source < size(), "Irecv: source rank " << source << " out of range");
  // received into an engine buffer and copied out by Wait (a dropped handle never leaves a dangling target)
  const uint64_t op = link_->recv(source, kNetP2p, tag, nullptr, static_cast<size_t>(bytes));
  const int64_t id = next_request_++;
  requests_[id] = op;
  recv_bufs_[id] = buf;
  return id;
}

void NetBackend::wait(int64_t request, void*) {
  auto it = requests_.find(request);
  M4T_CHECK(it != requests_.end(), "Wait: unknown or already completed request " << request
                                       << " (a WaitHandle may only be waited on once)");
  const uint64_t op = it->second;
  requests_.erase(it);
  auto rb = recv_bufs_.find(request);
  if (rb == recv_bufs_.end()) {
    link_->engine().wait(op);
    return;
  }
  void* dst = rb->second;
  recv_bufs_.erase(rb);
  NetBuffer data;
  const size_t n = link_->engine().wait(op, &data);
  if (n) std::memcpy(dst, data.data(), n);
}

// ---------------------------------------------------------------------------------------------------------------------

namespace {
template <DType DT> void widen_to_f32(const void* src, float* dst, int64_t n) {
  using E = Elem<DT>;
  const auto* s = static_cast<const typename E::storage*>(src);
  for (int64_t i = 0; i < n; ++i) dst[i] = E::load(s[i]);
}
// out = round(val [+ acc]): the one rounding of the 16-bit float contract
template <DType DT> void narrow_from_f32(const float* val, const void* acc, void* out, int64_t n) {
  using E = Elem<DT>;
  const auto* a = static_cast<const typename E::storage*>(acc);
  auto* o = static_cast<typename E::storage*>(out);
  if (a)
    for (int64_t i = 0; i < n; ++i) o[i] = E::store(val[i] + E::load(a[i]));
  else
    for (int64_t i = 0; i < n; ++i) o[i] = E::store(val[i]);
}
}  // namespace

void HierBackend::pull(const PullPlan& plan, const void* in, void* out, DType dt, void* stream) {
  const int L = local_.size(), node = rank() / L;
  const int P = size(), N = P / L, l = local_.rank();
  bool uniform_allgather = plan.replicated_output && static_cast<int>(plan.axis_len.size()) == P && plan.axis_len[0] > 0 &&
                           plan.before > 0 && plan.after > 0;
  for (int p = 1; uniform_allgather && p < P; ++p) uniform_allgather = plan.axis_len[static_cast<size_t>(p)] == plan.axis_len[0];
  if (uniform_allgather) {
    // Allgather with the same length on every rank: along the rail first (each rank fetches N-1 slices over the network
    // instead of (N-1) L), then the node's ranks exchange what their rails brought through shared memory
    const int64_t c = plan.axis_len[0], before = plan.before, after = plan.after, es = dtype_size(dt);
    const PullPlan far = plan_gather(node, N, 0, before, after, std::vector<int64_t>(static_cast<size_t>(N), c), /*all=*/true);
    grow(part_, static_cast<size_t>(before * c * N * after * es));
    rail_.pull(far, in, part_.data(), dt, nullptr);  // [before, N*c, after]: slice k = rank (k, l)
    PullPlan near;
    near.stage_elems = near.max_stage_elems = before * c * N * after;
    near.out_elems = near.max_out_elems = before * c * P * after;
    near.replicated_output = true;
    for (int q = 0; q < L; ++q) {
      SlabJob j;  // local rank q's rail buffer: slice k goes to global rank k*L + q
      j.peer = (l + q) % L;
      const int src = j.peer;
      j.src_off = 0;
      j.dst_off = static_cast<int64_t>(src) * c * after;
      j.n[1] = before;
      j.ss[1] = c * N * after;
      j.ds[1] = c * P * after;
      j.n[2] = N;
      j.ss[2] = c * after;
      j.ds[2] = static_cast<int64_t>(L) * c * after;
      j.run = c * after;
      near.jobs.push_back(j);
    }
    local_.pull(near, part_.data(), out, dt, nullptr);
    return;
  }
  PullPlan near = plan, far = plan;  // same sizes, disjoint job lists (they fill disjoint parts of the output)
  near.jobs.clear();
  far.jobs.clear();
  for (const auto& j : plan.jobs) {
    if (j.peer / L == node) {
      near.jobs.push_back(j);
      near.jobs.back().peer = j.peer % L;
    } else {
      far.jobs.push_back(j);
    }
  }
  local_.pull(near, in, out, dt, stream);
  flat_.pull(far, in, out, dt, stream);
}

void HierBackend::reduce_pull(const ReducePlan& plan, const void* in, void* out, DType dt, ReduceOp op, const Epilogue& epi,
                              void* stream) {
  check_op_dtype(op, dt);
  const int L = local_.size(), l = local_.rank(), P = size(), N = P / L, node = rank() / L;
  bool uniform = static_cast<int>(plan.numelem.size()) == P && plan.numelem[0] > 0;
  for (int p = 1; uniform && p < P; ++p) uniform = plan.numelem[static_cast<size_t>(p)] == plan.numelem[0];
  if (!uniform) {
    flat_.reduce_pull(plan, in, out, dt, op, epi, stream);
    return;
  }
  const int64_t c = plan.numelem[0], before = plan.before, after = plan.after;
  if (dt == DType::BF16 || dt == DType::F16) {
    // two reduction levels: on an fp32 copy, rounded once (together with the accumulate operand)
    const int64_t n_in = before * c * P * after, n_out = before * c * after;
    grow(wide_in_, static_cast<size_t>(n_in) * sizeof(float));
    grow(wide_out_, static_cast<size_t>(n_out) * sizeof(float));
    auto* wi = reinterpret_cast<float*>(wide_in_.data());
    auto* wo = reinterpret_cast<float*>(wide_out_.data());
    if (dt == DType::BF16) widen_to_f32<DType::BF16>(in, wi, n_in);
    else widen_to_f32<DType::F16>(in, wi, n_in);
    Epilogue e32;
    e32.scale = epi.scale;
    e32.has_scale = epi.has_scale;
    reduce_pull(plan, wi, wo, DType::F32, op, e32, nullptr);
    if (dt == DType::BF16) narrow_from_f32<DType::BF16>(wo, epi.accumulate, out, n_out);
    else narrow_from_f32<DType::F16>(wo, epi.accumulate, out, n_out);
    return;
  }
  const int64_t es = dtype_size(dt);
  // 1. inside the node: local rank l gets the node's sums of the slices of ranks l, L+l, ... as [before, N*c, after]
  ReducePlan near;
  near.stage_elems = before * c * P * after;
  near.out_elems = near.max_out_elems = before * c * N * after;
  near.box.peer = -1;
  near.box.src_off = static_cast<int64_t>(l) * c * after;
  near.box.n[1] = before;
  near.box.ss[1] = c * P * after;
  near.box.ds[1] = c * N * after;
  near.box.n[2] = N;
  near.box.ss[2] = static_cast<int64_t>(L) * c * after;
  near.box.ds[2] = c * after;
  near.box.run = c * after;
  grow(part_, static_cast<size_t>(near.out_elems * es));
  local_.reduce_pull(near, in, part_.data(), dt, op, Epilogue{}, nullptr);
  // 2. along the rail: reduce-scatter of those N slices, node k keeps slice k (scale / accumulate fused)
  const ReducePlan far = plan_reduce_scatter(node, N, before, after, std::vector<int64_t>(static_cast<size_t>(N), c));
  rail_.reduce_pull(far, part_.data(), out, dt, op, epi, nullptr);
}

int64_t HierBackend::isend(const void* buf, int64_t bytes, int dest, int64_t tag, void* stream) {
  M4T_CHECK(dest >= 0 && dest < size(), "Isend: destination rank " << dest << " out of range");
  const int L = local_.size(), node = rank() / L;
  if (dest / L == node) return (local_.isend(buf, bytes, dest % L, tag, stream) << 1) | 1;
  return flat_.isend(buf, bytes, dest, tag, stream) << 1;
}

int64_t HierBackend::irecv(void* buf, int64_t bytes, int source, int64_t tag, void* stream) {
  M4T_CHECK(source >= 0 && source < size(), "Irecv: source rank " << source << " out of range");
  const int L = local_.size(), node = rank() / L;
  if (source / L == node) return (local_.irecv(buf, bytes, source % L, tag, stream) << 1) | 1;
  return flat_.irecv(buf, bytes, source, tag, stream) << 1;
}

void HierBackend::wait(int64_t request, void* stream) {
  if (request & 1) local_.wait(request >> 1, stream);
  else flat_.wait(request >> 1, stream);
}

void HierBackend::bcast(void* buf, int64_t n, DType dt, int root, void*) {
  M4T_CHECK(root >= 0 && root < size(), "Bcast_: root " << root << " out of range");
  const int L = local_.size(), l = local_.rank();
  // the root's rail carries the buffer to one rank per node, shared memory spreads it inside each node
  if (l == root % L) rail_.bcast(buf, n, dt, root / L, nullptr);
  local_.bcast(buf, n, dt, root % L, nullptr);
}

void HierBackend::reduce(void* buf, int64_t n, DType dt, ReduceOp op, int root, void*) {
  check_op_dtype(op, dt);
  M4T_CHECK(root >= 0 && root < size(), "Reduce_: root " << root << " out of range");
  const int L = local_.size(), l = local_.rank();
  if (dt == DType::BF16 || dt == DType::F16) {
    // two reduction levels: run them on an fp32 copy so that the result is rounded once
    grow(wide_in_, static_cast<size_t>(n) * sizeof(float));
    auto* w = reinterpret_cast<float*>(wide_in_.data());
    if (dt == DType::BF16) widen_to_f32<DType::BF16>(buf, w, n);
    else widen_to_f32<DType::F16>(buf, w, n);
    reduce(w, n, DType::F32, op, root, nullptr);
    if (dt == DType::BF16) narrow_from_f32<DType::BF16>(w, nullptr, buf, n);
    else narrow_from_f32<DType::F16>(w, nullptr, buf, n);
    return;
  }
  // inside the node to the rank on the root's rail (the others are zero-filled), then along that rail to the root
  local_.reduce(buf, n, dt, op, root % L, nullptr);
  if (l == root % L) rail_.reduce(buf, n, dt, op, root / L, nullptr);
}

void HierBackend::allreduce(const void* in, void* out, int64_t n, DType dt, ReduceOp op, const Epilogue& epi, void*) {
  check_op_dtype(op, dt);
  const int L = local_.size(), l = local_.rank();
  if (dt == DType::BF16 || dt == DType::F16) {
    // 16-bit floats accumulate in fp32 and are rounded ONCE (the contract of every backend): the three steps run on an
    // fp32 copy, the result is narrowed at the end together with the accumulate operand
    grow(wide_in_, static_cast<size_t>(n) * sizeof(float));
    grow(wide_out_, static_cast<size_t>(n) * sizeof(float));
    auto* wi = reinterpret_cast<float*>(wide_in_.data());
    auto* wo = reinterpret_cast<float*>(wide_out_.data());
    if (dt == DType::BF16) widen_to_f32<DType::BF16>(in, wi, n);
    else widen_to_f32<DType::F16>(in, wi, n);
    Epilogue e32;
    e32.scale = epi.scale;
    e32.has_scale = epi.has_scale;
    allreduce(wi, wo, n, DType::F32, op, e32, nullptr);
    if (dt == DType::BF16) narrow_from_f32<DType::BF16>(wo, epi.accumulate, out, n);
    else narrow_from_f32<DType::F16>(wo, epi.accumulate, out, n);
    return;
  }
  const int64_t es = dtype_size(dt);
  Epilogue scale_only;
  scale_only.scale = epi.scale;
  scale_only.has_scale = epi.has_scale;
  if (n < 4 * L || n * es <= 4096) {
    // latency-bound: one shared-memory Allreduce, then every rank reduces the (tiny) vector along its rail
    grow(part_, static_cast<size_t>(n * es));
    local_.allreduce(in, part_.data(), n, dt, op, Epilogue{}, nullptr);
    rail_.allreduce(part_.data(), out, n, dt, op, epi, nullptr);
    return;
  }
  std::vector<int64_t> counts(static_cast<size_t>(L));
  for (int i = 0; i < L; ++i) counts[static_cast<size_t>(i)] = n * (i + 1) / L - n * i / L;
  const int64_t mine = counts[static_cast<size_t>(l)];
  grow(part_, static_cast<size_t>(mine * es));
  // 1. inside the node: local rank i receives the node's sum of slice i
  const ReducePlan rs = plan_reduce_scatter(l, L, 1, 1, counts);
  local_.reduce_pull(rs, in, part_.data(), dt, op, Epilogue{}, nullptr);
  // 2. between the nodes: the ranks with the same local index combine their slices (scale fused)
  rail_.allreduce(part_.data(), part_.data(), mine, dt, op, scale_only, nullptr);
  // 3. inside the node: every local rank collects all finished slices (accumulate fused afterwards)
  const PullPlan ag = plan_gather(l, L, 0, 1, 1, counts, /*all=*/true);
  if (epi.accumulate) {
    grow(land_, static_cast<size_t>(n * es));
    local_.pull(ag, part_.data(), land_.data(), dt, nullptr);
    M4T_DISPATCH_DTYPE_OP(dt, ReduceOp::SUM, CpuAccumulateCopy, land_.data(), epi.accumulate, out, 0, n);
  } else {
    local_.pull(ag, part_.data(), out, dt, nullptr);
  }
}

}  // namespace m4t
