// Python extension `hpc_patterns_b200._C`: thin pybind11 layer over the native
// launchers (csrc/kernels/api.h), peer memory (csrc/common/peer_mem.h), topology
// (csrc/p2p/topology_core.hpp) and the concurrency driver (csrc/concurency).
//
// Pointers and streams cross the boundary as integers: a device pointer is
// `tensor.data_ptr()` or the value returned by alloc(); a stream is
// `torch.cuda.current_stream().cuda_stream`.  That is the whole interop
// contract (see hpc_patterns_b200/models/interop.py), so the extension needs no
// torch headers and imports on a GPU-less machine.
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <cstring>
#include <iostream>
#include <sstream>
#include <type_traits>

#include "common/cuda_check.h"
#include "common/driver_api.h"
#include "common/dtype_traits.h"
#include "common/peer_mem.h"
#include "common/signal_layout.h"
#include "concurency/bench.hpp"
#include "concurency/driver.hpp"
#include "kernels/api.h"
#include "kernels/ring_order.h"
#include "kernels/tile_order.h"
#include "p2p/topology_core.hpp"

namespace py = pybind11;
using namespace hpcp;

namespace {

template <typename T>
T* as_ptr(uintptr_t p) {
  return reinterpret_cast<T*>(p);
}
cudaStream_t as_stream(uintptr_t s) { return reinterpret_cast<cudaStream_t>(s); }

CopyEngine engine_from(const std::string& s) {
  if (s == "ldst") return CopyEngine::kLdSt;
  if (s == "tma") return CopyEngine::kTma;
  throw std::invalid_argument("engine must be 'ldst' or 'tma'");
}

ElemType elem_from(const std::string& s) {
  ElemType t;
  if (elem_type_from_name(s, &t)) return t;
  throw std::invalid_argument("dtype must be one of float int uint double long ulong short ushort uchar");
}

CopyTuning tuning_from(const py::dict& d) {
  CopyTuning t;
  if (d.contains("ctas")) t.ctas = d["ctas"].cast<int>();
  if (d.contains("threads")) t.threads = d["threads"].cast<int>();
  if (d.contains("unroll")) t.unroll = d["unroll"].cast<int>();
  if (d.contains("stage_kb")) t.stage_kb = d["stage_kb"].cast<int>();
  if (d.contains("stages")) t.stages = d["stages"].cast<int>();
  if (d.contains("vec_bytes")) t.vec_bytes = d["vec_bytes"].cast<int>();
  if (d.contains("blocked")) t.blocked = d["blocked"].cast<int>();
  if (d.contains("halo_ctas")) t.halo_ctas = d["halo_ctas"].cast<int>();
  if (d.contains("l2_hint")) t.l2_hint = d["l2_hint"].cast<int>();
  return t;
}

HaloMode halo_mode_from(const std::string& s) {
  if (s == "none") return HaloMode::kNone;
  if (s == "pull") return HaloMode::kPull;
  if (s == "push") return HaloMode::kPush;
  throw std::invalid_argument("halo mode must be 'pull', 'push' or 'none'");
}

HaloTuning halo_tuning_from(const py::dict& d) {
  HaloTuning t;
  if (d.contains("ctas")) t.ctas = d["ctas"].cast<int>();
  if (d.contains("tile_kb")) t.tile_kb = d["tile_kb"].cast<int>();
  if (d.contains("stages")) t.stages = d["stages"].cast<int>();
  if (d.contains("l2_hint")) t.l2_hint = d["l2_hint"].cast<int>();
  if (d.contains("depth")) t.depth = d["depth"].cast<int>();
  return t;
}

SyncOps sync_from(const py::dict& d) {
  SyncOps s;
  if (d.contains("wait_flag")) s.wait_flag = as_ptr<const uint32_t>(d["wait_flag"].cast<uintptr_t>());
  if (d.contains("wait_epoch")) s.wait_epoch = d["wait_epoch"].cast<uint32_t>();
  if (d.contains("signal_flag")) s.signal_flag = as_ptr<uint32_t>(d["signal_flag"].cast<uintptr_t>());
  if (d.contains("signal_epoch")) s.signal_epoch = d["signal_epoch"].cast<uint32_t>();
  if (d.contains("ticket")) s.ticket = as_ptr<uint32_t>(d["ticket"].cast<uintptr_t>());
  if (d.contains("ticket_base")) s.ticket_base = d["ticket_base"].cast<uint32_t>();
  if (d.contains("timeout_ns")) s.timeout_ns = d["timeout_ns"].cast<uint64_t>();
  if (d.contains("status")) s.status = as_ptr<uint32_t>(d["status"].cast<uintptr_t>());
  return s;
}

std::unique_ptr<con::Backend> backend_from(const std::string& choice) {
  if (choice.rfind("fake:", 0) == 0) return con::make_fake_backend(choice.substr(5));
  if (choice == "cpu") return con::make_cpu_backend();
  std::string why;
  auto b = con::make_cuda_backend(&why);
  if (!b) {
    if (choice == "cuda") throw std::runtime_error("CUDA backend unavailable: " + why);
    return con::make_cpu_backend();
  }
  return b;
}

}  // namespace

PYBIND11_MODULE(_C, m) {
  m.doc() = "hpc-patterns-b200 native extension (sm_100a kernels + peer memory + topology)";

  // ------------------------------------------------------------ constants ----
  m.attr("PAD_WORDS") = kPadWords;
  m.attr("PAD_BARRIER") = kPadBarrier;
  m.attr("PAD_READY") = kPadReady;
  m.attr("PAD_DONE") = kPadDone;
  m.attr("PAD_ACK") = kPadAck;
  m.attr("PAD_LOCAL") = kPadLocal;
  m.attr("PAD_TAIL_WORDS") = kPadTailWords;
  m.attr("STATUS_OK") = static_cast<uint32_t>(kStatusOk);
  m.attr("STATUS_TIMEOUT") = static_cast<uint32_t>(kStatusTimeout);
  m.attr("STATUS_MISMATCH") = static_cast<uint32_t>(kStatusMismatch);
  m.attr("IPC_HANDLE_BYTES") = static_cast<int>(kIpcHandleBytes);
  m.attr("REFERENCE_MESSAGE_BYTES") = 1179648ull * 40 * 4;

  // --------------------------------------------------------------- device ----
  m.def("device_count", [] {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
      (void)cudaGetLastError();
      return 0;
    }
    return n;
  });
  m.def("sm_count", &device_sm_count, py::arg("device"));
  m.def("driver_api_available", [] { return DriverApi::available(); });
  m.def("multicast_supported", [](int device) { return NodeMemory::multicast_supported(device); });

  // --------------------------------------------------------------- memory ----
  m.def(
      "alloc",
      [](size_t bytes, const std::string& kind, int device, bool zero) {
        HPCP_REQUIRE(kind.size() == 1, "kind must be one of D H S M");
        return reinterpret_cast<uintptr_t>(alloc_bytes(bytes, alloc_kind_from_letter(kind[0]), device, zero));
      },
      py::arg("bytes"), py::arg("kind") = "D", py::arg("device") = 0, py::arg("zero") = true,
      "Allocate memory of kind D(evice) H(pinned) S(managed) M(alloc); returns the address.");
  m.def(
      "free",
      [](uintptr_t p, const std::string& kind) {
        free_bytes(as_ptr<void>(p), alloc_kind_from_letter(kind.at(0)));
      },
      py::arg("ptr"), py::arg("kind") = "D");
  m.def("enable_peer_access", [](const std::vector<int>& devices) { enable_peer_access(devices); });
  m.def("peer_access_problem", [](const std::vector<int>& devices) { return peer_access_problem(devices); });
  m.def("ipc_export", [](uintptr_t p) {
    unsigned char h[kIpcHandleBytes];
    ipc_export(as_ptr<void>(p), h);
    return py::bytes(reinterpret_cast<const char*>(h), kIpcHandleBytes);
  });
  m.def("ipc_open", [](const py::bytes& handle) {
    const std::string s = handle;
    HPCP_REQUIRE(s.size() == kIpcHandleBytes, "IPC handle must be 64 bytes");
    return reinterpret_cast<uintptr_t>(ipc_open(reinterpret_cast<const unsigned char*>(s.data())));
  });
  m.def("ipc_close", [](uintptr_t p) { ipc_close(as_ptr<void>(p)); });
  m.def("memset_async", [](uintptr_t p, int value, size_t bytes, uintptr_t stream) {
    HPCP_CUDA(cudaMemsetAsync(as_ptr<void>(p), value, bytes, as_stream(stream)));
  });
  m.def("memcpy_async", [](uintptr_t dst, uintptr_t src, size_t bytes, uintptr_t stream) {
    HPCP_CUDA(cudaMemcpyAsync(as_ptr<void>(dst), as_ptr<const void>(src), bytes, cudaMemcpyDefault,
                              as_stream(stream)));
  });
  m.def("memcpy_peer_async",
        [](uintptr_t dst, int dst_dev, uintptr_t src, int src_dev, size_t bytes, uintptr_t stream) {
          HPCP_CUDA(cudaMemcpyPeerAsync(as_ptr<void>(dst), dst_dev, as_ptr<const void>(src), src_dev,
                                        bytes, as_stream(stream)));
        });
  m.def("read_u32", [](uintptr_t p) {
    uint32_t v = 0;
    HPCP_CUDA(cudaMemcpy(&v, as_ptr<const void>(p), sizeof v, cudaMemcpyDefault));
    return v;
  });
  m.def("read_u64", [](uintptr_t p) {
    unsigned long long v = 0;
    HPCP_CUDA(cudaMemcpy(&v, as_ptr<const void>(p), sizeof v, cudaMemcpyDefault));
    return v;
  });
  m.def("write_u32", [](uintptr_t p, uint32_t v) {
    HPCP_CUDA(cudaMemcpy(as_ptr<void>(p), &v, sizeof v, cudaMemcpyDefault));
  });

  // -------------------------------------------------------------- streams ----
  m.def("stream_create", [](int device, bool non_blocking) {
    int prev = 0;
    HPCP_CUDA(cudaGetDevice(&prev));
    HPCP_CUDA(cudaSetDevice(device));
    cudaStream_t s;
    HPCP_CUDA(cudaStreamCreateWithFlags(&s, non_blocking ? cudaStreamNonBlocking : cudaStreamDefault));
    HPCP_CUDA(cudaSetDevice(prev));
    return reinterpret_cast<uintptr_t>(s);
  }, py::arg("device") = 0, py::arg("non_blocking") = true,
  "Create a raw CUDA stream owned by this extension (wrap it with torch.cuda.ExternalStream).");
  m.def("stream_destroy", [](uintptr_t s) { HPCP_CUDA(cudaStreamDestroy(as_stream(s))); });
  m.def("stream_synchronize", [](uintptr_t s) {
    py::gil_scoped_release release;
    HPCP_CUDA(cudaStreamSynchronize(as_stream(s)));
  });
  m.def("device_native_info", [](int device) {
    // Native (driver-level) handles underneath the runtime ordinal — see csrc/interop/device_table.h.
    const DriverApi& d = DriverApi::get();
    int prev = 0;
    HPCP_CUDA(cudaGetDevice(&prev));
    HPCP_CUDA(cudaSetDevice(device));
    HPCP_CUDA(cudaFree(nullptr));
    CUdevice cu_dev;
    HPCP_CU(d.cuDeviceGet(&cu_dev, device));
    CUcontext current = nullptr;
    HPCP_CU(d.cuCtxGetCurrent(&current));
    HPCP_CUDA(cudaSetDevice(prev));
    py::dict out;
    out["ordinal"] = device;
    out["cu_device"] = static_cast<int>(cu_dev);
    out["cu_context"] = reinterpret_cast<uintptr_t>(current);
    return out;
  });
  m.def("stream_context", [](uintptr_t stream) {
    const DriverApi& d = DriverApi::get();
    CUcontext ctx = nullptr;
    CUgreenCtx green = nullptr;
    HPCP_CU(d.cuStreamGetCtx(reinterpret_cast<CUstream>(stream), &ctx, &green));
    return reinterpret_cast<uintptr_t>(ctx);
  });

  // -------------------------------------------------------------- signals ----
  m.def("signal", [](uintptr_t flag, uint32_t epoch, uintptr_t stream) {
    launch_signal(as_ptr<uint32_t>(flag), epoch, as_stream(stream));
  });
  m.def("wait",
        [](uintptr_t flag, uint32_t epoch, uint64_t timeout_ns, uintptr_t status, uintptr_t stream) {
          launch_wait(as_ptr<const uint32_t>(flag), epoch, timeout_ns, as_ptr<uint32_t>(status),
                      as_stream(stream));
        });
  m.def("barrier_all", [](const std::vector<uintptr_t>& pads, int rank, uint32_t epoch,
                          uint64_t timeout_ns, uintptr_t status, uintptr_t stream) {
    std::vector<uint32_t*> p;
    for (auto x : pads) p.push_back(as_ptr<uint32_t>(x));
    launch_barrier_all(p.data(), rank, static_cast<int>(p.size()), epoch, timeout_ns,
                       as_ptr<uint32_t>(status), as_stream(stream));
  });

  // ------------------------------------------------------------------ p2p ----
  m.def(
      "copy",
      [](uintptr_t dst, uintptr_t src, size_t bytes, bool src_is_peer, const std::string& engine,
         const py::dict& tune, const py::dict& sync, int device, uintptr_t stream) {
        return launch_copy(as_ptr<void>(dst), as_ptr<const void>(src), bytes, src_is_peer,
                           engine_from(engine), tuning_from(tune), sync_from(sync), device,
                           as_stream(stream));
      },
      py::arg("dst"), py::arg("src"), py::arg("bytes"), py::arg("src_is_peer") = false,
      py::arg("engine") = "ldst", py::arg("tune") = py::dict(), py::arg("sync") = py::dict(),
      py::arg("device") = 0, py::arg("stream") = 0,
      "dst[0:bytes] = src[0:bytes] with an sm_100a kernel; either side may be a peer pointer. "
      "Returns the number of CTAs launched (advance the ticket counter by it).");
  m.def("fill_pattern", [](uintptr_t dst, size_t n_words, uint32_t seed, uintptr_t stream) {
    launch_fill_pattern(as_ptr<uint32_t>(dst), n_words, seed, as_stream(stream));
  });
  m.def(
      "verify_pattern",
      [](uintptr_t data, size_t n_words, uint32_t seed, uintptr_t mismatch, uintptr_t word_sum,
         uintptr_t wait_flag, uint32_t wait_epoch, uint64_t timeout_ns, uintptr_t status,
         uintptr_t stream) {
        launch_verify_pattern(as_ptr<const uint32_t>(data), n_words, seed,
                              as_ptr<unsigned long long>(mismatch),
                              as_ptr<unsigned long long>(word_sum), as_ptr<const uint32_t>(wait_flag),
                              wait_epoch, timeout_ns, as_ptr<uint32_t>(status), as_stream(stream));
      },
      py::arg("data"), py::arg("n_words"), py::arg("seed"), py::arg("mismatch"),
      py::arg("word_sum") = 0, py::arg("wait_flag") = 0, py::arg("wait_epoch") = 0,
      py::arg("timeout_ns") = 0, py::arg("status") = 0, py::arg("stream") = 0);

  // ------------------------------------------------------- fused triad+put ----
  m.def(
      "triad_put",
      [](uintptr_t a_local, uintptr_t a_peer, uintptr_t b, uintptr_t c, float s, size_t n,
         const std::string& engine, const py::dict& tune, const py::dict& sync, uintptr_t arrive_flag,
         uint32_t arrive_epoch, int device, uintptr_t stream, size_t n_put) {
        TriadPutArgs t;
        t.a_local = as_ptr<float>(a_local);
        t.a_peer = as_ptr<float>(a_peer);
        t.b = as_ptr<const float>(b);
        t.c = as_ptr<const float>(c);
        t.s = s;
        t.n = n;
        t.n_put = n_put;
        return launch_triad_put(t, engine_from(engine), tuning_from(tune), sync_from(sync),
                                as_ptr<const uint32_t>(arrive_flag), arrive_epoch, device,
                                as_stream(stream));
      },
      py::arg("a_local"), py::arg("a_peer"), py::arg("b"), py::arg("c"), py::arg("s"), py::arg("n"),
      py::arg("engine") = "ldst", py::arg("tune") = py::dict(), py::arg("sync") = py::dict(),
      py::arg("arrive_flag") = 0, py::arg("arrive_epoch") = 0, py::arg("device") = 0,
      py::arg("stream") = 0, py::arg("n_put") = 0,
      "Fused a = b + s*c written to a_local AND the peer-mapped a_peer (0 = no put), then signal. "
      "n_put < n: halo mode, only a[0:n_put) is put to the peer.");
  m.def("fill_triad_inputs", [](uintptr_t b, uintptr_t c, size_t n, int rank, uintptr_t stream) {
    launch_fill_triad_inputs(as_ptr<float>(b), as_ptr<float>(c), n, rank, as_stream(stream));
  });
  m.def("verify_triad",
        [](uintptr_t a, size_t n, int src_rank, float s, uintptr_t mismatch, uintptr_t stream) {
          launch_verify_triad(as_ptr<const float>(a), n, src_rank, s,
                              as_ptr<unsigned long long>(mismatch), as_stream(stream));
        });

  // --------------------------------------------- fused stencil + halo exchange ----
  m.attr("HALO_FLAG_BYTES") = static_cast<size_t>(kHaloFlagBytes);
  m.attr("HALO_FLAG_SETS") = kHaloFlagSets;
  m.attr("HALO_MAX_CTAS") = kHaloMaxCtas;
  m.attr("HALO_DEFAULT_DEPTH") = kHaloDefaultDepth;
  m.def(
      "halo_sweep_depth",
      [](int rows, const std::string& mode, const py::dict& tune) {
        return halo_sweep_depth(rows, halo_mode_from(mode), halo_tuning_from(tune));
      },
      py::arg("rows"), py::arg("mode") = "pull", py::arg("tune") = py::dict(),
      "Deepest sweep (steps per pass over the slab) a multi-step launch takes with these settings.");
  m.def("halo_sweep_schedule", &halo_sweep_schedule, py::arg("steps"), py::arg("depth"),
        "Sweep sizes of a `steps`-step launch whose deepest sweep is `depth`.");
  m.def(
      "halo_stencil_ctas",
      [](size_t row_elems, const std::string& mode, const py::dict& tune, int device) {
        return halo_stencil_ctas(row_elems, halo_tuning_from(tune), halo_mode_from(mode), device);
      },
      py::arg("row_elems"), py::arg("mode") = "pull", py::arg("tune") = py::dict(), py::arg("device") = 0);
  m.def(
      "halo_stencil",
      [](const py::dict& d, const std::string& mode, const py::dict& tune, int device, uintptr_t stream) {
        HaloStencilArgs a;
        auto pair = [&](const char* key, auto& dst) {
          if (!d.contains(key)) return;
          const auto v = d[key].cast<std::vector<uintptr_t>>();
          HPCP_REQUIRE(v.size() == 2, std::string("halo_stencil: '") + key + "' must hold two addresses");
          for (int q = 0; q < 2; ++q) dst[q] = as_ptr<std::remove_pointer_t<std::decay_t<decltype(dst[0])>>>(v[q]);
        };
        pair("u", a.u);
        pair("left_u", a.left_u);
        pair("right_u", a.right_u);
        pair("halo_lo", a.halo_lo);
        pair("halo_hi", a.halo_hi);
        pair("left_halo_hi", a.left_halo_hi);
        pair("right_halo_lo", a.right_halo_lo);
        if (d.contains("flags_local")) a.flags_local = as_ptr<uint32_t>(d["flags_local"].cast<uintptr_t>());
        if (d.contains("flags_left")) a.flags_left = as_ptr<uint32_t>(d["flags_left"].cast<uintptr_t>());
        if (d.contains("flags_right")) a.flags_right = as_ptr<uint32_t>(d["flags_right"].cast<uintptr_t>());
        if (d.contains("flag_set")) a.flag_set = d["flag_set"].cast<int>();
        a.rows = d["rows"].cast<int>();
        a.row_elems = d["row_elems"].cast<size_t>();
        if (d.contains("tile_begin")) a.tile_begin = d["tile_begin"].cast<size_t>();
        if (d.contains("tile_end")) a.tile_end = d["tile_end"].cast<size_t>();
        if (d.contains("alpha")) a.alpha = d["alpha"].cast<float>();
        if (d.contains("s")) a.s = d["s"].cast<float>();
        if (d.contains("step_base")) a.step_base = d["step_base"].cast<uint32_t>();
        if (d.contains("steps")) a.steps = d["steps"].cast<int>();
        if (d.contains("timeout_ns")) a.timeout_ns = d["timeout_ns"].cast<uint64_t>();
        if (d.contains("status")) a.status = as_ptr<uint32_t>(d["status"].cast<uintptr_t>());
        return launch_halo_stencil(a, halo_mode_from(mode), halo_tuning_from(tune), device, as_stream(stream));
      },
      py::arg("args"), py::arg("mode") = "pull", py::arg("tune") = py::dict(), py::arg("device") = 0,
      py::arg("stream") = 0,
      "Fused 3-point slab stencil + halo exchange with both ring neighbours (pull / push / none); `steps` steps in one "
      "persistent launch.  Returns the number of CTAs.");
  m.def("halo_init", [](uintptr_t u, uintptr_t halo_lo, uintptr_t halo_hi, int rows, size_t row_elems, int rank,
                        int world, uintptr_t stream) {
    launch_halo_init(as_ptr<float>(u), as_ptr<float>(halo_lo), as_ptr<float>(halo_hi), rows, row_elems, rank, world,
                     as_stream(stream));
  });
  m.def("halo_verify_from_init", [](uintptr_t u, int rows, size_t row_elems, int rank, int world, uint32_t steps,
                                    float alpha, float s, uintptr_t mismatch, uintptr_t stream) {
    launch_halo_verify_from_init(as_ptr<const float>(u), rows, row_elems, rank, world, steps, alpha, s,
                                 as_ptr<unsigned long long>(mismatch), as_stream(stream));
  });
  m.def("halo_verify_step", [](uintptr_t u_new, uintptr_t u_old, uintptr_t up_row, uintptr_t dn_row, int rows,
                               size_t row_elems, float alpha, float s, uintptr_t mismatch, uintptr_t stream) {
    launch_halo_verify_step(as_ptr<const float>(u_new), as_ptr<const float>(u_old), as_ptr<const float>(up_row),
                            as_ptr<const float>(dn_row), rows, row_elems, alpha, s,
                            as_ptr<unsigned long long>(mismatch), as_stream(stream));
  });

  // ------------------------------------------------- concurrency payloads ----
  m.def("busy_wait", [](uintptr_t out, size_t n_items, size_t tripcount, uintptr_t stream) {
    launch_busy_wait(as_ptr<float>(out), n_items, tripcount, as_stream(stream));
  });
  m.def(
      "fused_bench",
      [](const std::vector<py::dict>& cmds, const std::string& engine, const py::dict& tune, int device,
         uintptr_t stream) {
        std::vector<FusedCommand> v;
        for (const auto& d : cmds) {
          FusedCommand f;
          const std::string kind = d["kind"].cast<std::string>();
          f.kind = kind == "busy" ? FusedKind::kBusy : kind == "triad" ? FusedKind::kTriad : FusedKind::kCopy;
          if (d.contains("n")) f.n = d["n"].cast<size_t>();
          if (d.contains("tripcount")) f.tripcount = d["tripcount"].cast<size_t>();
          if (d.contains("dst")) f.dst = as_ptr<void>(d["dst"].cast<uintptr_t>());
          if (d.contains("src")) f.src = as_ptr<const void>(d["src"].cast<uintptr_t>());
          if (d.contains("a")) f.a = as_ptr<float>(d["a"].cast<uintptr_t>());
          if (d.contains("b")) f.b = as_ptr<const float>(d["b"].cast<uintptr_t>());
          if (d.contains("c")) f.c = as_ptr<const float>(d["c"].cast<uintptr_t>());
          if (d.contains("s")) f.s = d["s"].cast<float>();
          if (d.contains("ctas")) f.ctas = d["ctas"].cast<int>();
          v.push_back(f);
        }
        return launch_fused_bench(v.data(), static_cast<int>(v.size()), engine_from(engine),
                                  tuning_from(tune), device, as_stream(stream));
      },
      py::arg("commands"), py::arg("engine") = "tma", py::arg("tune") = py::dict(),
      py::arg("device") = 0, py::arg("stream") = 0);

  m.def("tc_busy_operand_bytes", &tc_busy_operand_bytes);
  m.def("tc_busy_out_elems_per_cta", &tc_busy_out_elems_per_cta);
  m.def("tc_fill_operands", [](uintptr_t operands, uintptr_t stream) {
    launch_tc_fill_operands(as_ptr<void>(operands), as_stream(stream));
  });
  m.def("tc_busy", [](uintptr_t operands, uintptr_t out, int ctas, uint32_t tripcount, uintptr_t stream,
                      int cluster) {
    launch_tc_busy(as_ptr<const void>(operands), as_ptr<float>(out), ctas, tripcount, as_stream(stream), cluster);
  }, py::arg("operands"), py::arg("out"), py::arg("ctas"), py::arg("tripcount"), py::arg("stream") = 0,
  py::arg("cluster") = 1,
  "tcgen05 tile loop: out[cta] = tripcount * (A[128x64] . B[256x64]^T), operands via TMA, accumulator in TMEM.");

  m.def(
      "gemm_put",
      [](uintptr_t a, uintptr_t b, uintptr_t c_local, uintptr_t c_peer, int m_, int n, int k, bool out_bf16,
         const py::dict& sync, int ctas, int device, uintptr_t stream, int cluster, bool tma_epilogue) {
        return launch_gemm_put(as_ptr<const void>(a), as_ptr<const void>(b), as_ptr<void>(c_local),
                               as_ptr<void>(c_peer), m_, n, k, out_bf16, sync_from(sync), ctas, device,
                               as_stream(stream), cluster, tma_epilogue);
      },
      py::arg("a"), py::arg("b"), py::arg("c_local"), py::arg("c_peer"), py::arg("m"), py::arg("n"), py::arg("k"),
      py::arg("out_bf16") = false, py::arg("sync") = py::dict(), py::arg("ctas") = 0, py::arg("device") = 0,
      py::arg("stream") = 0, py::arg("cluster") = 0, py::arg("tma_epilogue") = false,
      "tcgen05 GEMM C = A . B^T (bf16 in, fp32 out) whose epilogue stores to c_local and/or the peer-mapped c_peer.");

  m.def(
      "gemm_reduce_scatter",
      [](uintptr_t a, uintptr_t b, const std::vector<uintptr_t>& shards, const std::vector<uintptr_t>& done_flags,
         uint32_t done_epoch, uintptr_t ticket, uint32_t ticket_base, int rank, int m_, int n, int k, int ctas,
         int device, uintptr_t stream, int cluster, uintptr_t c_multicast, bool out_bf16, bool tma_epilogue) {
        GemmRsArgs args;
        args.tma_epilogue = tma_epilogue;
        args.c_multicast = as_ptr<float>(c_multicast);
        args.out_bf16 = out_bf16;
        if (shards.empty() || shards.size() > static_cast<size_t>(kApiMaxRanks))
          throw std::invalid_argument("gemm_reduce_scatter: 1..16 shard pointers");
        if (!done_flags.empty() && done_flags.size() != shards.size())
          throw std::invalid_argument("gemm_reduce_scatter: done_flags must be empty or one per rank");
        args.a = as_ptr<const void>(a);
        args.b = as_ptr<const void>(b);
        args.world = static_cast<int>(shards.size());
        for (int q = 0; q < args.world; ++q) {
          args.shard[q] = as_ptr<void>(shards[q]);
          args.done_flag[q] = done_flags.empty() ? nullptr : as_ptr<uint32_t>(done_flags[q]);
        }
        args.done_epoch = done_epoch;
        args.ticket = as_ptr<uint32_t>(ticket);
        args.ticket_base = ticket_base;
        args.rank = rank;
        args.m = m_;
        args.n = n;
        args.k = k;
        return launch_gemm_reduce_scatter(args, ctas, device, as_stream(stream), cluster);
      },
      py::arg("a"), py::arg("b"), py::arg("shards"), py::arg("done_flags") = std::vector<uintptr_t>(),
      py::arg("done_epoch") = 0, py::arg("ticket") = 0, py::arg("ticket_base") = 0, py::arg("rank") = 0, py::arg("m"),
      py::arg("n"), py::arg("k"), py::arg("ctas") = 0, py::arg("device") = 0, py::arg("stream") = 0,
      py::arg("cluster") = 0, py::arg("c_multicast") = 0, py::arg("out_bf16") = false,
      py::arg("tma_epilogue") = false,
      "tcgen05 GEMM whose epilogue adds every tile into the owner's fp32 shard over NVLink (GEMM -> reduce-scatter), "
      "or, with c_multicast, into every rank's copy through the NVSwitch (GEMM -> all-reduce).");
  m.def(
      "gemm_all_to_all",
      [](uintptr_t a, uintptr_t b, const std::vector<uintptr_t>& recv, bool out_bf16,
         const std::vector<uintptr_t>& done_flags, uint32_t done_epoch, uintptr_t ticket, uint32_t ticket_base, int rank,
         int m_, int n, int k, int ctas, int device, uintptr_t stream, int cluster) {
        GemmA2aArgs args;
        if (recv.empty() || recv.size() > static_cast<size_t>(kApiMaxRanks))
          throw std::invalid_argument("gemm_all_to_all: 1..16 receive buffers");
        if (!done_flags.empty() && done_flags.size() != recv.size())
          throw std::invalid_argument("gemm_all_to_all: done_flags must be empty or one per rank");
        args.a = as_ptr<const void>(a);
        args.b = as_ptr<const void>(b);
        args.world = static_cast<int>(recv.size());
        for (int q = 0; q < args.world; ++q) {
          args.recv[q] = as_ptr<void>(recv[q]);
          args.done_flag[q] = done_flags.empty() ? nullptr : as_ptr<uint32_t>(done_flags[q]);
        }
        args.out_bf16 = out_bf16;
        args.done_epoch = done_epoch;
        args.ticket = as_ptr<uint32_t>(ticket);
        args.ticket_base = ticket_base;
        args.rank = rank;
        args.m = m_;
        args.n = n;
        args.k = k;
        return launch_gemm_all_to_all(args, ctas, device, as_stream(stream), cluster);
      },
      py::arg("a"), py::arg("b"), py::arg("recv"), py::arg("out_bf16") = false,
      py::arg("done_flags") = std::vector<uintptr_t>(), py::arg("done_epoch") = 0, py::arg("ticket") = 0,
      py::arg("ticket_base") = 0, py::arg("rank") = 0, py::arg("m"), py::arg("n"), py::arg("k"), py::arg("ctas") = 0,
      py::arg("device") = 0, py::arg("stream") = 0, py::arg("cluster") = 0,
      "tcgen05 GEMM whose epilogue stores row block q of the result into rank q's receive buffer (GEMM -> all-to-all).");
  // Tile / gather orderings of the tensor-core kernels (kernels/tile_order.h), exposed for the CPU tests.
  m.def("gemm_tile_coords", [](int tile, int tiles_m, int tiles_n) {
    int mb = 0, nb = 0;
    umma::tile_coords(tile, tiles_m, tiles_n, &mb, &nb);
    return std::make_pair(mb, nb);
  });
  m.def("gemm_shard_coords", [](int tile, int rank, int world, int first, int shard_tiles_m, int tiles_n) {
    int mb = 0, nb = 0;
    umma::shard_coords(tile, rank, world, first, shard_tiles_m, tiles_n, &mb, &nb);
    return std::make_pair(mb, nb);
  });
  m.def("gemm_gather_piece", [](size_t c, int rank, int world, int shard_tiles_m, uint32_t chunks_per_block,
                                uint32_t chunk_bytes, size_t block_bytes) {
    const umma::GatherPiece p = umma::gather_piece(c, rank, world, shard_tiles_m, chunks_per_block, chunk_bytes,
                                                   block_bytes);
    return py::make_tuple(p.peer, p.m_blk, p.src_off, p.dst_off);
  });
  m.def("allgather_gemm_chunks_per_block", &allgather_gemm_chunks_per_block, py::arg("k"), py::arg("chunk_bytes") = 0);
  m.def(
      "allgather_gemm",
      [](uintptr_t a_full, const std::vector<uintptr_t>& a_src, uintptr_t b, uintptr_t c, bool out_bf16,
         uintptr_t ready, uint32_t ready_base, int chunk_bytes, const std::vector<uintptr_t>& done_flags,
         uint32_t done_epoch, uintptr_t ticket, uint32_t ticket_base, uint64_t timeout_ns, uintptr_t status, int rank,
         int m_, int n, int k, int ctas, int device, uintptr_t stream, int cluster, int activation) {
        AgGemmArgs args;
        args.activation = activation;
        if (a_src.empty() || a_src.size() > static_cast<size_t>(kApiMaxRanks))
          throw std::invalid_argument("allgather_gemm: 1..16 row-block pointers");
        if (!done_flags.empty() && done_flags.size() != a_src.size())
          throw std::invalid_argument("allgather_gemm: done_flags must be empty or one per rank");
        args.a_full = as_ptr<void>(a_full);
        args.world = static_cast<int>(a_src.size());
        for (int q = 0; q < args.world; ++q) {
          args.a_src[q] = as_ptr<const void>(a_src[q]);
          args.done_flag[q] = done_flags.empty() ? nullptr : as_ptr<uint32_t>(done_flags[q]);
        }
        args.b = as_ptr<const void>(b);
        args.c = as_ptr<void>(c);
        args.out_bf16 = out_bf16;
        args.ready = as_ptr<uint32_t>(ready);
        args.ready_base = ready_base;
        args.chunk_bytes = chunk_bytes;
        args.done_epoch = done_epoch;
        args.ticket = as_ptr<uint32_t>(ticket);
        args.ticket_base = ticket_base;
        args.timeout_ns = timeout_ns;
        args.status = as_ptr<uint32_t>(status);
        args.rank = rank;
        args.m = m_;
        args.n = n;
        args.k = k;
        return launch_allgather_gemm(args, ctas, device, as_stream(stream), cluster);
      },
      py::arg("a_full"), py::arg("a_src"), py::arg("b"), py::arg("c"), py::arg("out_bf16") = false, py::arg("ready") = 0,
      py::arg("ready_base") = 0, py::arg("chunk_bytes") = 0, py::arg("done_flags") = std::vector<uintptr_t>(),
      py::arg("done_epoch") = 0, py::arg("ticket") = 0, py::arg("ticket_base") = 0, py::arg("timeout_ns") = 0,
      py::arg("status") = 0, py::arg("rank") = 0, py::arg("m"), py::arg("n"), py::arg("k"), py::arg("ctas") = 0,
      py::arg("device") = 0, py::arg("stream") = 0, py::arg("cluster") = 0, py::arg("activation") = 0,
      "tcgen05 GEMM over row-sharded A: one gather thread per CTA pulls the peers' rows (TMA bulk, NVLink) while "
      "the tiles of the rows that are already here are computed (all-gather -> GEMM).");
  m.def(
      "wait_flags",
      [](uintptr_t flags, int count, uint32_t epoch, uint64_t timeout_ns, uintptr_t status, uintptr_t stream) {
        launch_wait_flags(as_ptr<const uint32_t>(flags), count, epoch, timeout_ns, as_ptr<uint32_t>(status),
                          as_stream(stream));
      },
      py::arg("flags"), py::arg("count"), py::arg("epoch"), py::arg("timeout_ns") = 0, py::arg("status") = 0,
      py::arg("stream") = 0);

  // ------------------------------------------------------------ allreduce ----
  m.def("init3", [](uintptr_t va, uintptr_t vb, uintptr_t vc, size_t n, double a, double b, double c,
                    const std::string& dtype, uintptr_t stream) {
    launch_init3(as_ptr<void>(va), as_ptr<void>(vb), as_ptr<void>(vc), n, a, b, c, elem_from(dtype),
                 as_stream(stream));
  });
  m.def("accumulate", [](uintptr_t va, uintptr_t vc, size_t n, const std::string& dtype, uintptr_t stream) {
    launch_accumulate(as_ptr<const void>(va), as_ptr<void>(vc), n, elem_from(dtype), as_stream(stream));
  });
  m.def("count_mismatch", [](uintptr_t v, size_t n, double expected, const std::string& dtype,
                             uintptr_t count, uintptr_t stream) {
    launch_count_mismatch(as_ptr<const void>(v), n, expected, elem_from(dtype),
                          as_ptr<unsigned long long>(count), as_stream(stream));
  });
  // Slot / flow-control rules of the fused ring (kernels/ring_order.h), exposed for the CPU protocol model.
  m.def("ring_src_slot", &ring_src_slot);
  m.def("ring_fwd_slot", &ring_fwd_slot);
  m.def("ring_forwards", &ring_forwards);
  m.def("ring_waits_for_ack", &ring_waits_for_ack);
  m.def("ring_publishes_ack", &ring_publishes_ack);
  m.def("ring_pull_keeps_copy", &ring_pull_keeps_copy);
  m.def("ring_pull_copy_slot", &ring_pull_copy_slot);
  m.def("ring_pull_src_slot", &ring_pull_src_slot);
  m.def("ring_pull_waits_for_ack", &ring_pull_waits_for_ack);
  m.def("ring_pull_publishes_ack", &ring_pull_publishes_ack);
  m.def("ring_num_chunks", &ring_num_chunks, py::arg("n"), py::arg("chunk_elems") = 0, py::arg("elem_bytes") = 4);
  m.def("elem_size", [](const std::string& dtype) { return elem_size(elem_from(dtype)); });
  m.def(
      "ring_allreduce",
      [](uintptr_t va, uintptr_t vc, uintptr_t slots_local, uintptr_t slots_right,
         uintptr_t arrived_local, uintptr_t arrived_right, int world, size_t n, size_t chunk_elems,
         uint32_t epoch_base, uint64_t timeout_ns, uintptr_t status, const std::string& dtype, int ctas,
         int device, uintptr_t stream, int n_slots, uintptr_t ack_local, uintptr_t ack_left, bool pull,
         uintptr_t va_left, uintptr_t slots_left) {
        RingArgs a;
        a.pull = pull;
        a.va_left = as_ptr<const void>(va_left);
        a.slots_left = as_ptr<const void>(slots_left);
        a.n_slots = n_slots;
        a.ack_local = as_ptr<uint32_t>(ack_local);
        a.ack_left = as_ptr<uint32_t>(ack_left);
        a.va = as_ptr<const void>(va);
        a.vc = as_ptr<void>(vc);
        a.slots_local = as_ptr<void>(slots_local);
        a.slots_right = as_ptr<void>(slots_right);
        a.arrived_local = as_ptr<uint32_t>(arrived_local);
        a.arrived_right = as_ptr<uint32_t>(arrived_right);
        a.world = world;
        a.n = n;
        a.chunk_elems = chunk_elems;
        a.epoch_base = epoch_base;
        a.timeout_ns = timeout_ns;
        a.status = as_ptr<uint32_t>(status);
        launch_ring_allreduce(a, elem_from(dtype), ctas, device, as_stream(stream));
      },
      py::arg("va"), py::arg("vc"), py::arg("slots_local"), py::arg("slots_right"),
      py::arg("arrived_local"), py::arg("arrived_right"), py::arg("world"), py::arg("n"),
      py::arg("chunk_elems") = 0, py::arg("epoch_base") = 0, py::arg("timeout_ns") = 0,
      py::arg("status") = 0, py::arg("dtype") = "float", py::arg("ctas") = 0, py::arg("device") = 0,
      py::arg("stream") = 0, py::arg("n_slots") = 0, py::arg("ack_local") = 0, py::arg("ack_left") = 0,
      py::arg("pull") = false, py::arg("va_left") = 0, py::arg("slots_left") = 0);
  m.def(
      "allreduce_two_shot",
      [](const std::vector<uintptr_t>& va, const std::vector<uintptr_t>& vc,
         const std::vector<uintptr_t>& pads, uintptr_t ticket, uint32_t ticket_base, int rank, size_t n,
         uint32_t barrier_epoch, uint64_t timeout_ns, uintptr_t status, const std::string& dtype,
         int ctas, int device, uintptr_t stream) {
        TwoShotArgs a;
        a.world = static_cast<int>(va.size());
        HPCP_REQUIRE(a.world <= kApiMaxRanks && vc.size() == va.size() && pads.size() == va.size(),
                     "two-shot: inconsistent rank lists");
        for (int r = 0; r < a.world; ++r) {
          a.va[r] = as_ptr<const void>(va[r]);
          a.vc[r] = as_ptr<void>(vc[r]);
          a.pads[r] = as_ptr<uint32_t>(pads[r]);
        }
        a.ticket = as_ptr<uint32_t>(ticket);
        a.ticket_base = ticket_base;
        a.rank = rank;
        a.n = n;
        a.barrier_epoch = barrier_epoch;
        a.timeout_ns = timeout_ns;
        a.status = as_ptr<uint32_t>(status);
        return launch_allreduce_two_shot(a, elem_from(dtype), ctas, device, as_stream(stream));
      },
      py::arg("va"), py::arg("vc"), py::arg("pads"), py::arg("ticket"), py::arg("ticket_base"),
      py::arg("rank"), py::arg("n"), py::arg("barrier_epoch"), py::arg("timeout_ns") = 0,
      py::arg("status") = 0, py::arg("dtype") = "float", py::arg("ctas") = 0, py::arg("device") = 0,
      py::arg("stream") = 0);
  m.def(
      "allreduce_nvls",
      [](uintptr_t va_mc, uintptr_t vc_mc, const std::vector<uintptr_t>& pads, uintptr_t ticket,
         uint32_t ticket_base, int rank, size_t n, uint32_t barrier_epoch, uint64_t timeout_ns,
         uintptr_t status, const std::string& dtype, int ctas, int device, uintptr_t stream) {
        NvlsArgs a;
        a.world = static_cast<int>(pads.size());
        HPCP_REQUIRE(a.world <= kApiMaxRanks, "nvls: too many ranks");
        a.va_mc = as_ptr<const void>(va_mc);
        a.vc_mc = as_ptr<void>(vc_mc);
        for (int r = 0; r < a.world; ++r) a.pads[r] = as_ptr<uint32_t>(pads[r]);
        a.ticket = as_ptr<uint32_t>(ticket);
        a.ticket_base = ticket_base;
        a.rank = rank;
        a.n = n;
        a.barrier_epoch = barrier_epoch;
        a.timeout_ns = timeout_ns;
        a.status = as_ptr<uint32_t>(status);
        return launch_allreduce_nvls(a, elem_from(dtype), ctas, device, as_stream(stream));
      },
      py::arg("va_mc"), py::arg("vc_mc"), py::arg("pads"), py::arg("ticket"), py::arg("ticket_base"),
      py::arg("rank"), py::arg("n"), py::arg("barrier_epoch"), py::arg("timeout_ns") = 0,
      py::arg("status") = 0, py::arg("dtype") = "float", py::arg("ctas") = 0, py::arg("device") = 0,
      py::arg("stream") = 0);

  // ------------------------------------------------------------- topology ----
  m.def("topology_merge_planes", [](int n_gpus, const std::vector<std::vector<std::string>>& links) {
    std::vector<topo::LinkSet> ls;
    for (const auto& l : links) ls.emplace_back(l.begin(), l.end());
    return topo::merge_planes(n_gpus, ls);
  });
  m.def("topology_device_for_rank",
        [](const std::string& policy, int local_rank, int n_devices,
           const std::vector<std::vector<int>>& planes, int n_domains) {
          return topo::device_for_rank(policy, local_rank, n_devices, planes, n_domains);
        },
        py::arg("policy"), py::arg("local_rank"), py::arg("n_devices"),
        py::arg("planes") = std::vector<std::vector<int>>{}, py::arg("n_domains") = 2);
  m.def("topology_discover", [](const std::string& fake_spec) {
    topo::Fabric f;
    std::string why;
    bool ok = fake_spec.empty() ? topo::discover_fabric(&f, &why) : topo::fabric_from_fake(fake_spec, &f, &why);
    if (!ok) throw std::runtime_error("no fabric information: " + why);
    const auto planes = topo::merge_planes(static_cast<int>(f.gpus.size()), f.links);
    return topo::to_json(f, planes);
  }, py::arg("fake_spec") = "");

  // ---------------------------------------------------------- concurrency ----
  m.def(
      "concurency_main",
      [](const std::vector<std::string>& argv, const std::string& backend) {
        auto b = backend_from(backend);
        std::ostringstream out, err;
        int rc;
        {
          py::gil_scoped_release release;
          rc = con::run(argv, *b, out, err, "concurency");
        }
        return py::make_tuple(rc, out.str(), err.str());
      },
      py::arg("argv"), py::arg("backend") = "auto",
      "Run the concurrency benchmark driver in-process; returns (exit_status, stdout, stderr).");
  m.def(
      "concurency_bench",
      [](const std::string& backend, const std::string& mode, const std::vector<std::string>& commands,
         const std::unordered_map<std::string, size_t>& params, bool enable_profiling, int n_queues,
         int n_repetitions, bool verbose) {
        auto b = backend_from(backend);
        con::BenchRequest req;
        req.mode = mode;
        req.commands = commands;
        req.params = params;
        req.enable_profiling = enable_profiling;
        req.n_queues = n_queues;
        req.n_repetitions = n_repetitions;
        req.verbose = verbose;
        con::BenchResult r;
        {
          py::gil_scoped_release release;
          r = b->run(req);
        }
        py::dict d;
        d["total_us"] = r.total_us;
        d["per_command_us"] = r.per_command_us;
        d["device_us"] = r.device_us;
        d["device_total_us"] = r.device_total_us;
        return d;
      },
      py::arg("backend"), py::arg("mode"), py::arg("commands"), py::arg("params"),
      py::arg("enable_profiling") = false, py::arg("n_queues") = -1, py::arg("n_repetitions") = 10,
      py::arg("verbose") = false,
      "bench(mode, commands, params, ...) -> {total_us, per_command_us} (↔ bench<T>() of the reference).");
  m.def("concurency_judge", [](double max_speedup, double speedup, double gbps, double min_bw,
                               unsigned long long bytes) {
    return con::verdict_text(con::judge(max_speedup, speedup, gbps, min_bw, bytes));
  });
  m.def("strip_twos", &con::strip_twos);
}
