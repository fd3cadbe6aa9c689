// Registration: TORCH_LIBRARY custom class + ops (reference csrc/extension.cpp:
// 1270-1304 uses the legacy torch::RegisterOperators API) and the pybind module
// that bootstraps the world at import (reference :1396-1436).
#include <execinfo.h>
#include <signal.h>
#include <torch/extension.h>
#include <torch/library.h>
#include <unistd.h>

#include "../runtime/cuda_backend.h"
#include "communicator.h"

namespace m4t {

namespace {

// M4T_DEBUG_SEGV=1: print a native backtrace on SIGSEGV/SIGABRT (no gdb in the image).
void segv_handler(int sig) {
  void* frames[64];
  const int n = backtrace(frames, 64);
  const char msg[] = "[m4t] fatal signal, native backtrace:\n";
  (void)!write(2, msg, sizeof(msg) - 1);
  backtrace_symbols_fd(frames, n, 2);
  signal(sig, SIG_DFL);
  raise(sig);
}

void maybe_install_segv_handler() {
  if (env_i64("M4T_DEBUG_SEGV", 0)) {
    signal(SIGSEGV, segv_handler);
    signal(SIGABRT, segv_handler);
  }
}

void init_world(bool want_cuda, int64_t device) {
  maybe_install_segv_handler();
  World& w = World::instance();
  if (want_cuda && !w.cuda_ready()) {
    w.init_cuda(static_cast<int>(device));
  }
}

// Multi-node start-up, driven from Python (mpi4torch_b200/__init__.py::_bootstrap): every rank opens its listening
// socket, the addresses travel through the launcher's store, then the mesh is connected.
int g_listen_fd = -1;

int64_t net_listen() {
  int port = 0;
  g_listen_fd = NetEngine::listen_any(&port);
  return port;
}

void net_connect(int64_t rank, int64_t size, const std::vector<std::string>& addrs, const std::string& job) {
  M4T_CHECK(g_listen_fd >= 0, "net_connect() without net_listen()");
  const double timeout_s = static_cast<double>(env_i64("M4T_TIMEOUT_S", 300));
  auto engine = std::make_shared<NetEngine>(static_cast<int>(rank), static_cast<int>(size), g_listen_fd, addrs, timeout_s,
                                            net_comm_id(job));
  g_listen_fd = -1;
  World::set_network(std::move(engine));
}

void deactivate_cuda_aware_mpi_support() {
  // Reference :54-59 forces host staging for CUDA tensors; same effect here.
  World::instance().set_host_staging(true);
}

void activate_nvlink_transport() { World::instance().set_host_staging(false); }

}  // namespace

TORCH_LIBRARY(mpi4torch_b200, m) {
  m.class_<Communicator>("Communicator")
      .def("GetRank", &Communicator::GetRank)
      .def("GetSize", &Communicator::GetSize)
      .def("Allreduce", &Communicator::Allreduce)
      .def("AllreduceFused", &Communicator::AllreduceFused)
      .def("Bcast_", &Communicator::Bcast_)
      .def("Reduce_", &Communicator::Reduce_)
      .def("Gather", &Communicator::Gather)
      .def("Allgather", &Communicator::Allgather)
      .def("Scatter", &Communicator::Scatter)
      .def("Alltoall", &Communicator::Alltoall)
      .def("Reduce_scatter", &Communicator::Reduce_scatter)
      .def("Reduce_scatterFused", &Communicator::Reduce_scatterFused)
      .def("Scan", &Communicator::Scan)
      .def("Exscan", &Communicator::Exscan)
      .def("AssumeUniformSizes", &Communicator::AssumeUniformSizes)
      .def("UniformSizes", &Communicator::UniformSizes)
      .def("Isend", &Communicator::Isend)
      .def("Irecv", &Communicator::Irecv)
      .def("Wait", &Communicator::Wait)
      .def("Split", &Communicator::Split)
      .def("IsWorld", &Communicator::IsWorld)
      .def("Free", &Communicator::Free)
      .def("Barrier", &Communicator::Barrier)
      .def("Describe", &Communicator::Describe)
      // Only the world communicator exists, so pickling round-trips it by name
      // (the reference's unpickle test is inverted and always throws, :1292-1294).
      .def_pickle([](const c10::intrusive_ptr<Communicator>& self) -> std::string {
                    TORCH_CHECK(self->IsWorld(), "mpi4torch_b200: only the world communicator can be pickled");
                    return "MPI_COMM_WORLD";
                  },
                  [](std::string state) -> c10::intrusive_ptr<Communicator> {
                    TORCH_CHECK(state == "MPI_COMM_WORLD", "mpi4torch_b200: unknown pickled communicator '", state, "'");
                    return comm_world();
                  });
  m.def("COMM_WORLD", &comm_world);
  // The reference converts an MPI Fortran handle (csrc/extension.cpp:165-172).  There is no MPI
  // here, hence no handle space: the op exists for API parity and returns the world communicator.
  m.def("comm_from_fortran", [](int64_t) { return comm_world(); });
  m.def("JoinDummies(Tensor loopthrough, Tensor[] dummies) -> Tensor",
        [](const Tensor& loopthrough, std::vector<Tensor> dummies) { return JoinDummies(loopthrough, dummies); });
}

}  // namespace m4t

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  using namespace m4t;
  m.doc() = "mpi4torch_b200 native core: shared-memory control plane, CPU backend, NVLink/NVSwitch CUDA backend";
  m.def("init_world", &init_world, py::arg("want_cuda"), py::arg("device") = 0,
        "Attach to the job (collective) and optionally bring up the CUDA backend on `device`.");
  m.def("finalize", [] { World::finalize(); });
  m.def("net_listen", &net_listen, "Opens this rank's listening socket for the multi-node TCP mesh; returns the port");
  m.def("net_connect", &net_connect, py::arg("rank"), py::arg("size"), py::arg("addrs"), py::arg("job") = "",
        "Connects the TCP mesh (addrs[p] = 'host:port' of rank p); the world communicator is then created on it");
  m.def("over_network", [] { return World::instance().ctx()->over_network(); });
  m.def("set_node_cuda_device", [](int64_t device) { World::instance().set_node_cuda_device(static_cast<int>(device)); },
        "Job that spans nodes: the device node-local sub-communicators bind their NVLink backend to");
  m.def("world_initialised", [] { return World::initialised(); });
  m.def("deactivate_cuda_aware_mpi_support", &deactivate_cuda_aware_mpi_support);
  m.def("activate_nvlink_transport", &activate_nvlink_transport);
  m.def("cuda_backend_ready", [] { return World::instance().cuda_ready(); });
  m.def("has_nvls", [] { return World::instance().cuda_ready() && World::instance().cuda()->has_nvls(); });
  m.def("heap_mode", [] {
    World& w = World::instance();
    if (!w.cuda_ready()) return std::string("none");
    switch (w.cuda()->heap().mode()) {
      case HeapMode::VMM_MULTICAST: return std::string("vmm+multicast");
      case HeapMode::VMM: return std::string("vmm");
      default: return std::string("cudaIpc");
    }
  });
  m.def("set_tuning", [](const std::string& key, int64_t value) {
    World& w = World::instance();
    TORCH_CHECK(w.cuda_ready(), "CUDA backend not initialised");
    CudaTuning& t = w.cuda()->tuning();
    if (key == "oneshot_max_bytes") t.oneshot_max_bytes = value;
    else if (key == "chunk_bytes") t.chunk_bytes = value;
    else if (key == "ar_blocks") t.ar_blocks = static_cast<int>(value);
    else if (key == "pipe_min_bytes") t.pipe_min_bytes = value;
    else if (key == "nvls_min_ranks") t.nvls_min_ranks = static_cast<int>(value);
    else if (key == "oneshot_blocks") t.oneshot_blocks = static_cast<int>(value);
    else if (key == "slab_blocks") t.slab_blocks = static_cast<int>(value);
    else if (key == "p2p_blocks") t.p2p_blocks = static_cast<int>(value);
    else if (key == "force_algo") t.force_algo = static_cast<int>(value);
    else if (key == "wgrad_debug") set_wgrad_debug(static_cast<int>(value));
    else TORCH_CHECK(false, "unknown tuning key ", key);
  });
  m.def("slab_chunked_calls", [] { return slab_chunked_calls(); },
        "Gather / Allgather / Reduce_scatter calls moved in pieces (share larger than a staging half).");
  m.def("kernel_launch_table", [] {
    py::dict d;
    for (const auto& kv : kernel_launch_table()) d[py::str(kv.first)] = static_cast<int64_t>(kv.second);
    return d;
  }, "Launch counts of the named (tensor-core / fused) kernels in this process.");
  m.def("kernel_launch_count", [] { return static_cast<int64_t>(kernel_launch_count()); },
        "Kernels launched by this library in this process.");
  // Slab-plan introspection (tests): every job as a dict of plain integers.
  auto jobs_to_py = [](const std::vector<SlabJob>& jobs) {
    py::list out;
    for (const SlabJob& j : jobs) {
      py::dict d;
      d["peer"] = j.peer;
      d["src_off"] = j.src_off;
      d["dst_off"] = j.dst_off;
      d["n"] = py::make_tuple(j.n[0], j.n[1], j.n[2]);
      d["ss"] = py::make_tuple(j.ss[0], j.ss[1], j.ss[2]);
      d["ds"] = py::make_tuple(j.ds[0], j.ds[1], j.ds[2]);
      d["run"] = j.run;
      out.append(d);
    }
    return out;
  };
  m.def("plan_gather", [jobs_to_py](int rank, int size, int root, int64_t before, int64_t after,
                                     std::vector<int64_t> lens, bool all) {
    PullPlan p = plan_gather(rank, size, root, before, after, lens, all);
    return py::make_tuple(jobs_to_py(p.jobs), p.stage_elems, p.out_elems);
  });
  m.def("plan_scatter", [jobs_to_py](int rank, int size, int root, int64_t before, int64_t after,
                                      std::vector<int64_t> counts) {
    PullPlan p = plan_scatter(rank, size, root, before, after, counts);
    return py::make_tuple(jobs_to_py(p.jobs), p.stage_elems, p.out_elems);
  });
  m.def("plan_alltoall", [jobs_to_py](int rank, int size, std::vector<int64_t> shape, int64_t g, int64_t s_,
                                       std::vector<int64_t> glen, std::vector<int64_t> counts) {
    PullPlan p = plan_alltoall(rank, size, shape, g, s_, glen, counts);
    return py::make_tuple(jobs_to_py(p.jobs), p.stage_elems, p.out_elems);
  });
  m.def("plan_repartition", [jobs_to_py](int rank, int size, int64_t before, int64_t after, std::vector<int64_t> cur,
                                          std::vector<int64_t> nw) {
    PullPlan p = plan_repartition(rank, size, before, after, cur, nw);
    return py::make_tuple(jobs_to_py(p.jobs), p.stage_elems, p.out_elems);
  });
  m.def("check_device_error", [] {
    World& w = World::instance();
    if (w.cuda_ready()) w.cuda()->check_device_error();
  });
  // the reference's 12 integer op constants (csrc/extension.cpp:1424-1435)
  m.attr("MPI_MAX") = py::int_(static_cast<int>(ReduceOp::MAX));
  m.attr("MPI_MIN") = py::int_(static_cast<int>(ReduceOp::MIN));
  m.attr("MPI_SUM") = py::int_(static_cast<int>(ReduceOp::SUM));
  m.attr("MPI_PROD") = py::int_(static_cast<int>(ReduceOp::PROD));
  m.attr("MPI_LAND") = py::int_(static_cast<int>(ReduceOp::LAND));
  m.attr("MPI_BAND") = py::int_(static_cast<int>(ReduceOp::BAND));
  m.attr("MPI_LOR") = py::int_(static_cast<int>(ReduceOp::LOR));
  m.attr("MPI_BOR") = py::int_(static_cast<int>(ReduceOp::BOR));
  m.attr("MPI_LXOR") = py::int_(static_cast<int>(ReduceOp::LXOR));
  m.attr("MPI_BXOR") = py::int_(static_cast<int>(ReduceOp::BXOR));
  m.attr("MPI_MINLOC") = py::int_(static_cast<int>(ReduceOp::MINLOC));
  m.attr("MPI_MAXLOC") = py::int_(static_cast<int>(ReduceOp::MAXLOC));
}
