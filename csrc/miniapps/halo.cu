// halo: the miniapp loop as a time-stepping halo exchange — native CLI of the suite's flagship kernel.
//
// The reference's miniapp alternates a kernel with a blocking exchange of a full block with both ring
// neighbours and a host wait after each (allreduce-mpi-sycl.cpp:167-181: Accumulate().wait();
// SendRecvRing(VA -> right, VB <- left); swap; Accumulate().wait()).  This program runs the same
// dependency structure as a slab stencil whose exchange lives INSIDE the kernel
// (csrc/kernels/halo_stencil.cu): `-n` ranks (one host thread + one GPU each, more ranks than GPUs are
// placed round-robin like devices.hpp:46-47), a periodic field of ranks x rows rows of `--bytes` each,
// `--steps` time steps per timed iteration in ONE persistent launch per rank (or one launch per step
// with --per-step), exact verification of every element against the closed-form field advanced on the
// fly by an independent kernel, and the reference-style report: "Passed <rank>" per rank, then the
// elapsed time (max over ranks, min over iterations) and the P2P bus bandwidth.
//
//   halo -n 8                       # 8 GPUs, pull mode, 8 rows of 188 743 680 B, 20 steps per iteration
//   halo -n 2 --mode push --rows 1  # NVLink-bound: every computed row is exchanged
//   halo -n 4 --stock memcpy        # the stock shape instead: kernel, wait, cudaMemcpyAsync to peers, wait
#include <getopt.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <iostream>
#include <limits>
#include <string>
#include <vector>

#include "../common/cuda_check.h"
#include "../common/nvtx.h"
#include "../common/peer_mem.h"
#include "../common/rank_runtime.h"
#include "../common/signal_layout.h"
#include "../kernels/api.h"
#include "devices.hpp"

namespace {
using namespace hpcp;

struct Config {
  int ranks = 0;
  int rows = 8;
  size_t bytes = 1179648ull * 40 * 4;   // one row = one message of p2p/peer2pear.cpp:115-116
  int steps = 20;
  int iters = 5;
  int warmup = 1;
  std::string mode = "pull";
  std::string stock;                     // "" | "memcpy": kernel -> wait -> library copies -> wait per step
  bool per_step = false;
  HaloTuning tune;
  uint64_t timeout_ns = 30ull * 1000 * 1000 * 1000;
  std::string json_path;
  bool cpu = false;                      // host-only plumbing run: ranks are threads, rows live in host vectors
  std::string dump_path;                 // --cpu only: the final field, rank after rank, raw fp32
};

void print_help() {
  std::cout << "Usage: halo [options]\n"
               " -n N          ranks (one host thread + one GPU each; default: all GPUs; more ranks than GPUs share)\n"
               " --rows R      rows per rank (default 8: HBM time ~ NVLink time)\n"
               " --bytes B     bytes per row (one row = one message)\n"
               " --steps K     time steps per timed iteration (default 20); --iters N  --warmup N\n"
               " --mode pull|push   neighbours' rows are LOADED from their fields / new boundary rows are STORED into\n"
               "                    their halo buffers — both from inside the stencil kernel\n"
               " --per-step    one launch per step instead of one persistent K-step launch\n"
               " --stock memcpy     the reference's shape through stock calls: kernel; wait; copies; wait\n"
               " --ctas N --tile-kb N --stages N   kernel geometry\n"
               " --l2-hint             evict_first L2 policy on the slab's own streaming loads / stores\n"
               " --depth D     pull: most steps one sweep of the slab advances (0: default, 1: one step per sweep)\n"
               " --json FILE   append one JSON row\n"
               " --cpu         no GPU: ranks are host threads, the exchange is a memcpy into (push) or a read out of\n"
               "               (pull) the neighbours' arrays, one barrier per step: options, ring order, verification\n"
               "               and output of the program on a machine without a device (default 4 ranks)\n"
               " --dump FILE   with --cpu: the final field (rank after rank, raw fp32), for comparison with an\n"
               "               independent implementation\n";
}

struct Shared {
  Config cfg;
  NodeMemory* mem = nullptr;
  SymmetricBuffer field, halo, flags, pads;
  double best_ms = 0;
  unsigned long long total_bad = 0;
  int ctas = 0;
};

// HPCP_TRACE=1: one stderr line per rank per milestone (which call a stuck rank never returned from).
void trace(int rank, const char* what, int it = -1, int k = -1) {
  static const bool on = std::getenv("HPCP_TRACE") != nullptr;
  if (on) std::fprintf(stderr, "[halo trace] rank %d %s it=%d step=%d\n", rank, what, it, k);
}

void rank_main(RankCtx& ctx, Shared& sh) {
  const Config& cfg = sh.cfg;
  const int me = ctx.rank, P = ctx.world;
  const int dev = sh.mem->device(me);
  HPCP_CUDA(cudaSetDevice(dev));
  cudaStream_t stream;
  HPCP_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  const int left = (me - 1 + P) % P, right = (me + 1) % P;
  const size_t row_elems = cfg.bytes / 4, slab = static_cast<size_t>(cfg.rows) * cfg.bytes;
  auto u = [&](int r, int parity) {
    return reinterpret_cast<float*>(static_cast<char*>(sh.field.ptr[r]) + parity * slab);
  };
  auto halo = [&](int r, int side, int parity) {
    return reinterpret_cast<float*>(static_cast<char*>(sh.halo.ptr[r]) + (side * 2 + parity) * cfg.bytes);
  };
  uint32_t* my_pad = static_cast<uint32_t*>(sh.pads.ptr[me]);
  uint32_t* status = my_pad + kPadWords;
  std::vector<uint32_t*> pad_list;
  for (int r = 0; r < P; ++r) pad_list.push_back(static_cast<uint32_t*>(sh.pads.ptr[r]));
  const HaloMode mode = !cfg.stock.empty() ? HaloMode::kNone : cfg.mode == "push" ? HaloMode::kPush : HaloMode::kPull;

  HaloStencilArgs a;
  for (int q = 0; q < 2; ++q) {
    a.u[q] = u(me, q);
    a.left_u[q] = u(left, q);
    a.right_u[q] = u(right, q);
    a.halo_lo[q] = halo(me, 0, q);
    a.halo_hi[q] = halo(me, 1, q);
    a.left_halo_hi[q] = halo(left, 1, q);
    a.right_halo_lo[q] = halo(right, 0, q);
  }
  a.flags_local = static_cast<uint32_t*>(sh.flags.ptr[me]);
  a.flags_left = static_cast<uint32_t*>(sh.flags.ptr[left]);
  a.flags_right = static_cast<uint32_t*>(sh.flags.ptr[right]);
  a.rows = cfg.rows;
  a.row_elems = row_elems;
  a.timeout_ns = cfg.timeout_ns;
  a.status = status;

  launch_halo_init(u(me, 0), halo(me, 0, 0), halo(me, 1, 0), cfg.rows, row_elems, me, P, stream);
  HPCP_CUDA(cudaStreamSynchronize(stream));
  ctx.barrier();

  uint32_t g = 0, barrier_epoch = 0;
  cudaEvent_t e0, e1;
  HPCP_CUDA(cudaEventCreate(&e0));
  HPCP_CUDA(cudaEventCreate(&e1));
  double best_ms = std::numeric_limits<double>::max();
  for (int it = 0; it < cfg.warmup + cfg.iters; ++it) {
    NvtxRange range(it < cfg.warmup ? "halo warm-up" : "halo timed");
    HPCP_CUDA(cudaStreamSynchronize(stream));
    trace(me, "before host barrier", it);
    ctx.barrier();
    launch_barrier_all(pad_list.data(), me, P, ++barrier_epoch, cfg.timeout_ns, status, stream);
    HPCP_CUDA(cudaEventRecord(e0, stream));
    trace(me, "device barrier enqueued", it);
    if (!cfg.stock.empty()) {
      for (int k = 0; k < cfg.steps; ++k, ++g) {
        const int out = (g + 1) & 1;
        a.step_base = g;
        a.steps = 1;
        launch_halo_stencil(a, HaloMode::kNone, cfg.tune, dev, stream);
        HPCP_CUDA(cudaStreamSynchronize(stream));                                   // Accumulate(...).wait()
        trace(me, "kernel done", it, k);
        HPCP_CUDA(cudaMemcpyAsync(halo(left, 1, out), u(me, out), cfg.bytes, cudaMemcpyDefault, stream));
        HPCP_CUDA(cudaMemcpyAsync(halo(right, 0, out), u(me, out) + static_cast<size_t>(cfg.rows - 1) * row_elems,
                                  cfg.bytes, cudaMemcpyDefault, stream));
        HPCP_CUDA(cudaStreamSynchronize(stream));                                   // the blocking Send/Recv pair
        trace(me, "copies done", it, k);
        ctx.barrier();                                                              // ... of every rank
      }
    } else if (cfg.per_step) {
      for (int k = 0; k < cfg.steps; ++k, ++g) {
        a.step_base = g;
        a.steps = 1;
        launch_halo_stencil(a, mode, cfg.tune, dev, stream);
      }
    } else {
      a.step_base = g;
      a.steps = cfg.steps;
      sh.ctas = launch_halo_stencil(a, mode, cfg.tune, dev, stream);
      g += static_cast<uint32_t>(cfg.steps);
    }
    HPCP_CUDA(cudaEventRecord(e1, stream));
    HPCP_CUDA(cudaStreamSynchronize(stream));
    uint32_t st = 0;
    HPCP_CUDA(cudaMemcpy(&st, status, sizeof st, cudaMemcpyDefault));
    HPCP_REQUIRE(st == kStatusOk, "rank " + std::to_string(me) + ": device-side wait timed out");
    float ms = 0;
    HPCP_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    const double t = ctx.max(ms);
    if (it >= cfg.warmup) best_ms = std::min(best_ms, t);
  }

  // Verify every element of this rank's slab against the closed-form field advanced g steps.
  unsigned long long* count = nullptr;
  HPCP_CUDA(cudaMalloc(&count, sizeof *count));
  HPCP_CUDA(cudaMemsetAsync(count, 0, sizeof *count, stream));
  launch_halo_verify_from_init(u(me, g & 1), cfg.rows, row_elems, me, P, g, a.alpha, a.s, count, stream);
  unsigned long long bad = 0;
  HPCP_CUDA(cudaMemcpyAsync(&bad, count, sizeof bad, cudaMemcpyDeviceToHost, stream));
  HPCP_CUDA(cudaStreamSynchronize(stream));
  (void)cudaFree(count);
  const double total_bad = ctx.sum(static_cast<double>(bad));
  if (bad == 0)
    std::cout << "Passed " << me << std::endl;
  else
    std::cout << "FAILED " << me << ": " << bad << " wrong elements" << std::endl;
  if (me == 0) {
    sh.best_ms = best_ms;
    sh.total_bad = static_cast<unsigned long long>(total_bad);
  }
  (void)cudaEventDestroy(e0);
  (void)cudaEventDestroy(e1);
  (void)cudaStreamDestroy(stream);
}

// ---------------------------------------------------------------- host-only path ----
// The same program without a device, like `allreduce --cpu` / `peer2pear --cpu`: ranks are threads of the rank
// runtime, a slab is a host vector, "pull" reads the neighbours' boundary rows in place, "push" copies the new boundary
// rows into the neighbours' halo arrays, and one barrier per step stands in for the step words.  Exists to test the
// program logic (options, slab decomposition, ring order, parity double-buffering, verification, output) on a machine
// without a GPU; the verification advances the closed-form initial field of the WHOLE ring column by column, exactly as
// halo_verify_init_kernel does.
__attribute__((noinline)) float host_stencil1(float prev, float cur, float next, float alpha, float s) {
  const float sum = prev + next;
  const float side = s * sum;
  const float mid = alpha * cur;
  return mid + side;
}

float host_u0(uint32_t grow, uint64_t j) {  // halo_u0 of kernels/halo_stencil.cu
  const uint32_t jl = static_cast<uint32_t>(j);
  const uint32_t h = (grow * 2654435761u) ^ (jl * 40503u + (jl >> 11));
  return static_cast<float>(static_cast<int>(h & 0xFFFFu) - 32768) * (1.0f / 1024.0f);
}

int run_on_host(const Config& cfg) {
  const int P = cfg.ranks > 0 ? cfg.ranks : 4;
  HPCP_REQUIRE(P >= 1 && P <= kMaxRanks, "ranks out of range");
  const int R = cfg.rows;
  const size_t n = cfg.bytes / 4;
  const bool push = cfg.mode == "push" || !cfg.stock.empty();  // the stock shape is a push with host waits
  const float alpha = HaloStencilArgs{}.alpha, sc = HaloStencilArgs{}.s;
  std::vector<std::vector<float>> u[2], lo[2], hi[2];
  for (int q = 0; q < 2; ++q) {
    u[q].resize(P);
    lo[q].resize(P);
    hi[q].resize(P);
  }
  double best_ms = 0;
  unsigned long long total_bad = 0;
  int final_parity = 0;
  run_ranks(P, [&](RankCtx& ctx) {
    const int me = ctx.rank, left = (me - 1 + P) % P, right = (me + 1) % P;
    const uint32_t G = static_cast<uint32_t>(P) * R, first = static_cast<uint32_t>(me) * R;
    for (int q = 0; q < 2; ++q) {
      u[q][me].assign(static_cast<size_t>(R) * n, 0.f);
      lo[q][me].assign(n, 0.f);
      hi[q][me].assign(n, 0.f);
    }
    for (size_t j = 0; j < n; ++j) {
      for (int r = 0; r < R; ++r) u[0][me][static_cast<size_t>(r) * n + j] = host_u0(first + r, j);
      lo[0][me][j] = host_u0((first + G - 1) % G, j);
      hi[0][me][j] = host_u0((first + R) % G, j);
    }
    uint32_t g = 0;
    double best = std::numeric_limits<double>::max();
    for (int it = 0; it < cfg.warmup + cfg.iters; ++it) {
      ctx.barrier();
      const auto t0 = std::chrono::steady_clock::now();
      for (int k = 0; k < cfg.steps; ++k, ++g) {
        const int in = g & 1, out = in ^ 1;
        ctx.barrier();  // every rank finished step g-1: its rows (pull) / my halo arrays (push) hold step g's inputs
        const float* below = push ? lo[in][me].data() : u[in][left].data() + static_cast<size_t>(R - 1) * n;
        const float* above = push ? hi[in][me].data() : u[in][right].data();
        const float* src = u[in][me].data();
        float* dst = u[out][me].data();
        for (int r = 0; r < R; ++r) {
          const float* dn = r == 0 ? below : src + static_cast<size_t>(r - 1) * n;
          const float* up = r == R - 1 ? above : src + static_cast<size_t>(r + 1) * n;
          const float* ce = src + static_cast<size_t>(r) * n;
          float* o = dst + static_cast<size_t>(r) * n;
          for (size_t j = 0; j < n; ++j) o[j] = host_stencil1(dn[j], ce[j], up[j], alpha, sc);
        }
        if (push) {  // my new first row is the left neighbour's upper halo, my new last row the right one's lower halo
          std::copy(dst, dst + n, hi[out][left].begin());
          std::copy(dst + static_cast<size_t>(R - 1) * n, dst + static_cast<size_t>(R) * n, lo[out][right].begin());
        }
      }
      ctx.barrier();
      const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
      const double t = ctx.max(ms);
      if (it >= cfg.warmup) best = std::min(best, t);
    }
    // every column of the whole ring from the closed form, advanced g steps; compare this rank's rows exactly
    unsigned long long bad = 0;
    std::vector<float> v(G), w(G);
    const float* mine = u[g & 1][me].data();
    for (size_t j = 0; j < n; ++j) {
      for (uint32_t q = 0; q < G; ++q) v[q] = host_u0(q, j);
      for (uint32_t k = 0; k < g; ++k) {
        for (uint32_t q = 0; q < G; ++q) w[q] = host_stencil1(v[(q + G - 1) % G], v[q], v[(q + 1) % G], alpha, sc);
        v.swap(w);
      }
      for (int r = 0; r < R; ++r) bad += mine[static_cast<size_t>(r) * n + j] != v[first + r];
    }
    const double all_bad = ctx.sum(static_cast<double>(bad));
    if (bad == 0)
      std::cout << "Passed " << me << std::endl;
    else
      std::cout << "FAILED " << me << ": " << bad << " wrong elements" << std::endl;
    if (me == 0) {
      best_ms = best;
      total_bad = static_cast<unsigned long long>(all_bad);
      final_parity = static_cast<int>(g & 1);
    }
  });
  if (!cfg.dump_path.empty()) {
    FILE* f = std::fopen(cfg.dump_path.c_str(), "wb");
    HPCP_REQUIRE(f != nullptr, "cannot open --dump file");
    for (int r = 0; r < P; ++r) std::fwrite(u[final_parity][r].data(), sizeof(float), u[final_parity][r].size(), f);
    std::fclose(f);
  }
  const double ms_per_step = best_ms / cfg.steps;
  const double bus = static_cast<double>(P) * 2.0 * static_cast<double>(cfg.bytes) / (ms_per_step * 1e6);
  const std::string what = std::string(!cfg.stock.empty() ? "stock-" + cfg.stock : cfg.mode) + "/host-threads";
  std::cout << "Elapsed (max over ranks, min of " << cfg.iters << "): " << best_ms << " ms for " << cfg.steps
            << " steps = " << ms_per_step << " ms/step | halo " << what << " P=" << P << " rows=" << R
            << " bytes=" << cfg.bytes << " ctas=0 | " << bus << " GB/s P2P bus (aggregate), " << bus / P / 2.0
            << " GB/s per GPU per direction" << std::endl;
  if (!cfg.json_path.empty()) {
    if (FILE* f = std::fopen(cfg.json_path.c_str(), "a")) {
      std::fprintf(f,
                   "{\"pattern\":\"halo\",\"variant\":\"%s\",\"ranks\":%d,\"rows\":%d,\"bytes\":%zu,\"steps\":%d,"
                   "\"ms_per_step\":%.6f,\"bus_GBps\":%.3f,\"per_gpu_per_dir_GBps\":%.3f,\"ctas\":0,"
                   "\"mismatches\":%llu}\n",
                   what.c_str(), P, R, cfg.bytes, cfg.steps, ms_per_step, bus, bus / P / 2.0, total_bad);
      std::fclose(f);
    }
  }
  return total_bad == 0 ? 0 : 1;
}

}  // namespace

int main(int argc, char** argv) {
  hpcp::prefer_eager_module_loading();  // spin-waiting kernels + lazy module loading can deadlock (cuda_check.h)
  try {
    Config cfg;
    static const option long_opts[] = {
        {"rows", required_argument, nullptr, 1}, {"bytes", required_argument, nullptr, 2},
        {"steps", required_argument, nullptr, 3}, {"iters", required_argument, nullptr, 4},
        {"warmup", required_argument, nullptr, 5}, {"mode", required_argument, nullptr, 6},
        {"per-step", no_argument, nullptr, 7}, {"stock", required_argument, nullptr, 8},
        {"ctas", required_argument, nullptr, 9}, {"tile-kb", required_argument, nullptr, 10},
        {"stages", required_argument, nullptr, 11}, {"json", required_argument, nullptr, 12},
        {"l2-hint", no_argument, nullptr, 13}, {"cpu", no_argument, nullptr, 14},
        {"dump", required_argument, nullptr, 15}, {"depth", required_argument, nullptr, 16},
        {"help", no_argument, nullptr, 'h'}, {nullptr, 0, nullptr, 0}};
    int opt;
    while ((opt = getopt_long(argc, argv, "hn:", long_opts, nullptr)) != -1) {
      switch (opt) {
        case 'h': print_help(); return 1;
        case 'n': cfg.ranks = std::atoi(optarg); break;
        case 1: cfg.rows = std::atoi(optarg); break;
        case 2: cfg.bytes = static_cast<size_t>(std::atoll(optarg)); break;
        case 3: cfg.steps = std::max(1, std::atoi(optarg)); break;
        case 4: cfg.iters = std::max(1, std::atoi(optarg)); break;
        case 5: cfg.warmup = std::max(0, std::atoi(optarg)); break;
        case 6: cfg.mode = optarg; break;
        case 7: cfg.per_step = true; break;
        case 8: cfg.stock = optarg; break;
        case 9: cfg.tune.ctas = std::atoi(optarg); break;
        case 10: cfg.tune.tile_kb = std::atoi(optarg); break;
        case 11: cfg.tune.stages = std::atoi(optarg); break;
        case 12: cfg.json_path = optarg; break;
        case 13: cfg.tune.l2_hint = 1; break;
        case 14: cfg.cpu = true; break;
        case 15: cfg.dump_path = optarg; break;
        case 16: cfg.tune.depth = std::max(0, std::atoi(optarg)); break;
        default: print_help(); return 1;
      }
    }
    HPCP_REQUIRE(cfg.mode == "pull" || cfg.mode == "push", "--mode must be pull or push");
    HPCP_REQUIRE(cfg.stock.empty() || cfg.stock == "memcpy", "--stock accepts memcpy");
    HPCP_REQUIRE(cfg.rows >= 1 && cfg.bytes >= 16 && cfg.bytes % 16 == 0, "--rows >= 1, --bytes a multiple of 16");
    HPCP_REQUIRE(cfg.dump_path.empty() || cfg.cpu, "--dump belongs to --cpu");
    if (cfg.cpu) return run_on_host(cfg);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
      (void)cudaGetLastError();
      std::cerr << "Error: No devices" << std::endl;
      return 1;
    }
    const int P = cfg.ranks > 0 ? cfg.ranks : ndev;
    HPCP_REQUIRE(P >= 1 && P <= kMaxRanks, "ranks out of range");
    HPCP_REQUIRE(P * cfg.rows <= 128, "ranks x rows must not exceed 128 (verification kernel)");
    std::vector<int> devices;
    for (int r = 0; r < P; ++r) devices.push_back(primary_device(r, P, ndev));
    const int ranks_per_dev = (P + ndev - 1) / ndev;
    const HaloMode geo_mode = cfg.mode == "push" ? HaloMode::kPush : HaloMode::kPull;
    if (ranks_per_dev > 1) {  // co-residency of the spinning persistent kernels that share a GPU
      HaloTuning all = cfg.tune;
      all.ctas = 0;
      const int full = halo_stencil_ctas(cfg.bytes / 4, all, geo_mode, devices[0]);
      const int share = std::max(1, full / ranks_per_dev);
      cfg.tune.ctas = cfg.tune.ctas > 0 ? std::min(cfg.tune.ctas, share) : share;
    }
    // the same grid on every rank and in every launch: the step words are indexed by CTA
    cfg.tune.ctas = halo_stencil_ctas(cfg.bytes / 4, cfg.tune, geo_mode, devices[0]);

    Shared sh;
    sh.cfg = cfg;
    NodeMemory mem(devices);
    sh.mem = &mem;
    sh.field = mem.alloc(2 * static_cast<size_t>(cfg.rows) * cfg.bytes, AllocKind::kDevice, /*zero=*/false);
    sh.halo = mem.alloc(4 * cfg.bytes, AllocKind::kDevice, /*zero=*/false);
    sh.flags = mem.alloc(kHaloFlagBytes, AllocKind::kDevice, /*zero=*/true);
    sh.pads = mem.alloc_pads(0);
    sh.ctas = cfg.tune.ctas;

    run_ranks(P, [&](RankCtx& ctx) { rank_main(ctx, sh); });

    const double ms_per_step = sh.best_ms / cfg.steps;
    const double bus = static_cast<double>(P) * 2.0 * static_cast<double>(cfg.bytes) / (ms_per_step * 1e6);
    const std::string what =
        !cfg.stock.empty() ? "stock-" + cfg.stock : cfg.mode + (cfg.per_step ? "/per-step" : "/persistent");
    std::cout << "Elapsed (max over ranks, min of " << cfg.iters << "): " << sh.best_ms << " ms for " << cfg.steps
              << " steps = " << ms_per_step << " ms/step | halo " << what << " P=" << P << " rows=" << cfg.rows
              << " bytes=" << cfg.bytes << " ctas=" << sh.ctas << " | " << bus << " GB/s P2P bus (aggregate), "
              << bus / P / 2.0 << " GB/s per GPU per direction" << std::endl;
    if (!cfg.json_path.empty()) {
      if (FILE* f = std::fopen(cfg.json_path.c_str(), "a")) {
        std::fprintf(f,
                     "{\"pattern\":\"halo\",\"variant\":\"%s\",\"ranks\":%d,\"rows\":%d,\"bytes\":%zu,\"steps\":%d,"
                     "\"ms_per_step\":%.6f,\"bus_GBps\":%.3f,\"per_gpu_per_dir_GBps\":%.3f,\"ctas\":%d,"
                     "\"mismatches\":%llu}\n",
                     what.c_str(), P, cfg.rows, cfg.bytes, cfg.steps, ms_per_step, bus, bus / P / 2.0, sh.ctas,
                     sh.total_bad);
        std::fclose(f);
      }
    }
    mem.free(sh.field);
    mem.free(sh.halo);
    mem.free(sh.flags);
    mem.free(sh.pads);
    return sh.total_bad == 0 ? 0 : 1;
  } catch (const std::exception& e) {
    std::cerr << "Error: " << e.what() << std::endl;
    return 1;
  }
}
