// Host-callable launchers for every sm_100a kernel in the suite.
//
// Plain C++ (no torch, no MPI): raw device pointers + a cudaStream_t.  Both
// front ends use exactly these entry points:
//   * the native CLIs (csrc/p2p, csrc/concurency, csrc/miniapps) through the
//     thread-per-rank runtime in csrc/common/rank_runtime.h, and
//   * the PyTorch extension (csrc/bindings.cpp) for one-process-per-GPU runs
//     launched by torchrun, where peer pointers come from CUDA IPC handles.
//
// Pointers named *_peer may be NVLink peer-mapped addresses; *_mc are NVSwitch
// multicast addresses.  Every launcher returns after enqueueing on `stream`.
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <vector>

namespace hpcp {

constexpr int kApiMaxRanks = 16;

// How the bytes move inside a copy kernel.
enum class CopyEngine : int {
  kLdSt = 0,  // 128-bit ld.global / st.global from every thread of the grid
  kTma = 1,   // one elected thread per CTA drives cp.async.bulk (TMA) through smem stages
};

struct CopyTuning {
  int ctas = 0;      // 0 -> heuristic (multiple of the SM count)
  int threads = 0;   // 0 -> heuristic
  int unroll = 0;    // LdSt: 16-byte loads in flight per thread (1,2,4,8); 0 -> 4
  int stage_kb = 0;  // Tma: smem stage size in KiB; 0 -> 16
  int stages = 0;    // Tma: number of smem stages; 0 -> 8
  int vec_bytes = 0; // LdSt: 16 (LDG/STG.128) or 32 (sm_100 LDG/STG.256); 0 -> 16
  int blocked = 0;   // LdSt: 1 = each CTA owns one contiguous region instead of a grid-stride
  int l2_hint = 0;   // triad_put, TMA engine, EXPERIMENTAL: 1 = L2 evict_first policy on the bulk loads of b, c and
                     // the local bulk store of a (streamed once); the peer store keeps the default policy
  int halo_ctas = 0; // triad_put halo mode, TMA engine, EXPERIMENTAL: > 0 dedicates that many CTAs to the
                     // halo (NVLink-bound) tiles and the rest to the interior instead of interleaving
};

// Optional prologue wait + epilogue signal attached to a data-moving kernel so a
// whole "rendezvous send" (wait for receiver, move, tell receiver) is ONE launch.
struct SyncOps {
  const uint32_t* wait_flag = nullptr;  // local word to wait on before moving (may be null)
  uint32_t wait_epoch = 0;
  uint32_t* signal_flag = nullptr;      // word (usually on the peer) to publish after moving
  uint32_t signal_epoch = 0;
  uint32_t* ticket = nullptr;           // rank-local CTA ticket counter (needed iff signal_flag)
  uint32_t ticket_base = 0;             // value of *ticket before this launch
  uint64_t timeout_ns = 0;              // 0 = wait forever
  uint32_t* status = nullptr;           // rank-local status word (see signal.cuh)
};

int device_sm_count(int device);

// ---------------------------------------------------------------- signals ----
void launch_signal(uint32_t* flag, uint32_t epoch, cudaStream_t stream);
void launch_wait(const uint32_t* flag, uint32_t epoch, uint64_t timeout_ns, uint32_t* status,
                 cudaStream_t stream);
// In-kernel barrier across `world` GPUs: writes `epoch` into slot [rank] of every
// peer's barrier section, then waits until all slots of the local pad reach it.
void launch_barrier_all(uint32_t* const* pads /*[world], peer-mapped*/, int rank, int world,
                        uint32_t epoch, uint64_t timeout_ns, uint32_t* status,
                        cudaStream_t stream);

// ------------------------------------------------------------------- p2p ----
// dst[0:bytes) = src[0:bytes).  Either side may be a peer-mapped pointer:
// put = local src -> peer dst, get = peer src -> local dst.  Returns the number
// of CTAs launched (the caller advances its ticket counter by it).
int launch_copy(void* dst, const void* src, size_t bytes, bool src_is_peer, CopyEngine engine,
                const CopyTuning& tune, const SyncOps& sync, int device, cudaStream_t stream);

// Payload: word[i] = mix32(i*2654435761 ^ seed) — a seeded bijection of the index,
// generated on the device (↔ fill_randomly, p2p/peer2pear.cpp:8-17).
void launch_fill_pattern(uint32_t* dst, size_t n_words, uint32_t seed, cudaStream_t stream);
// Exact receiver-side check (↔ sorted-sum check p2p/peer2pear.cpp:55-63, made exact):
// counts mismatching words into *mismatch_count and accumulates the 64-bit word sum.
// If wait_flag != null each CTA first waits for the arrival epoch (fused wait+verify).
void launch_verify_pattern(const uint32_t* data, size_t n_words, uint32_t seed,
                           unsigned long long* mismatch_count, unsigned long long* word_sum,
                           const uint32_t* wait_flag, uint32_t wait_epoch, uint64_t timeout_ns,
                           uint32_t* status, cudaStream_t stream);

// ------------------------------------------------ fused triad + P2P put ----
// a = b + s*c computed once and written BOTH to a_local and (over NVLink) to
// a_peer, then the arrival epoch is published on the peer and (optionally) the
// local arrival word is awaited — compute, put and sync in one launch.
struct TriadPutArgs {
  float* a_local = nullptr;
  float* a_peer = nullptr;  // may equal nullptr -> plain triad (the unfused compute)
  const float* b = nullptr;
  const float* c = nullptr;
  float s = 0.f;
  size_t n = 0;             // elements the triad runs over, multiple of 4
  size_t n_put = 0;         // halo: only a[0:n_put) also goes to the peer; 0 -> n.  n % n_put == 0 and
                            // (when n_put < n) n_put * 4 a multiple of the 16 KiB tile
};
int launch_triad_put(const TriadPutArgs& args, CopyEngine engine, const CopyTuning& tune,
                     const SyncOps& sync, const uint32_t* arrive_flag, uint32_t arrive_epoch,
                     int device, cudaStream_t stream);
void launch_fill_triad_inputs(float* b, float* c, size_t n, int rank, cudaStream_t stream);
void launch_verify_triad(const float* a, size_t n, int src_rank, float s,
                         unsigned long long* mismatch_count, cudaStream_t stream);

// ------------------------------------- fused stencil + halo exchange (flagship) ----
// One step: u'[r][j] = alpha*u[r][j] + s*(u[r-1][j] + u[r+1][j]) over this rank's slab [rows][row_elems] of a field
// that is periodic in r and split over the ring of ranks; rows -1 / `rows` are the neighbours' boundary rows.
// kPull reads them out of the neighbours' fields over NVLink inside the kernel, kPush stores the new boundary rows
// into the neighbours' halo buffers from inside the kernel, kNone only reads local halo buffers (the compute kernel of
// the stock kernel -> library transfer -> wait arm).  `steps` steps run in ONE persistent launch; neighbouring CTAs of
// the same index synchronise through monotonic step words (no grid barrier, no host sync).  See halo_stencil.cu.
enum class HaloMode : int { kNone = 0, kPull = 1, kPush = 2 };
constexpr int kHaloFlagWords = 8;    // one 32-byte sector per flag word
constexpr int kHaloMaxCtas = 1024;   // flag words per side
constexpr int kHaloFlagSets = 16;    // independent flag sets (chunked launches of one step use one set per chunk)
constexpr size_t kHaloFlagBytes = static_cast<size_t>(kHaloFlagSets) * 2 * kHaloMaxCtas * kHaloFlagWords * 4;
struct HaloTuning {
  int ctas = 0;     // 0 -> every resident CTA slot (SMs x occupancy); always clamped to it
  int tile_kb = 0;  // bytes of a row per shared-memory stage in KiB; 0 -> 16
  int stages = 0;   // shared-memory stages (>= 6); 0 -> 6 (two CTAs per SM with 16 KiB tiles)
  int l2_hint = 0;  // 1: L2 evict_first policy on the streaming loads / stores of the slab's own rows
  int depth = 0;    // pull: most steps one sweep of the slab may advance (deep halos); 0 -> kHaloDefaultDepth, 1 -> one
                    // step per sweep (halo_stencil_kernel only)
};
constexpr int kHaloDefaultDepth = 3;  // measured: see docs/halo.md, "Deep sweeps"
struct HaloStencilArgs {
  float* u[2] = {nullptr, nullptr};                 // local field, ping-pong: step g reads u[g&1], writes u[(g+1)&1]
  const float* left_u[2] = {nullptr, nullptr};      // pull: the left / right neighbour's u[0], u[1] (peer-mapped)
  const float* right_u[2] = {nullptr, nullptr};
  float* halo_lo[2] = {nullptr, nullptr};           // push / none: local halo rows by step parity (from the left ...
  float* halo_hi[2] = {nullptr, nullptr};           // ... and from the right neighbour)
  float* left_halo_hi[2] = {nullptr, nullptr};      // push: the left neighbour's halo_hi (receives my new row 0)
  float* right_halo_lo[2] = {nullptr, nullptr};     // push: the right neighbour's halo_lo (receives my new last row)
  uint32_t* flags_local = nullptr;                  // kHaloFlagBytes of zeroed words on every rank
  uint32_t* flags_left = nullptr;                   // the neighbours' flag buffers (peer-mapped)
  uint32_t* flags_right = nullptr;
  int flag_set = 0;
  int rows = 0;
  size_t row_elems = 0;                             // multiple of 4
  size_t tile_begin = 0, tile_end = 0;              // column tiles of a row to process; end 0 -> all
  float alpha = 0.5f, s = 0.25f;
  uint32_t step_base = 0;                           // global index of the first step of this launch
  int steps = 1;
  uint64_t timeout_ns = 0;
  uint32_t* status = nullptr;
};
// CTAs a launch with this geometry uses (identical on every rank; the flag words are indexed by it).
int halo_stencil_ctas(size_t row_elems, const HaloTuning& tune, HaloMode mode, int device);
// Deepest sweep a multi-step launch takes with these settings (1: every step is its own sweep).
int halo_sweep_depth(int rows, HaloMode mode, const HaloTuning& tune);
// Sweep sizes of a `steps`-step launch with maximum depth `depth`: greedy, the largest odd size <= min(depth, remaining
// - 1), so every sweep is odd and the last one is a single step (identical on every rank).
std::vector<int> halo_sweep_schedule(int steps, int depth);
int launch_halo_stencil(const HaloStencilArgs& args, HaloMode mode, const HaloTuning& tune, int device,
                        cudaStream_t stream);
// u[r][j] = u0(rank*rows + r, j); halo_lo / halo_hi (may be null) = the neighbours' boundary rows of the initial field.
void launch_halo_init(float* u, float* halo_lo, float* halo_hi, int rows, size_t row_elems, int rank, int world,
                      cudaStream_t stream);
// Exact check of this rank's rows after `steps` steps against the closed-form initial field (world*rows <= 128).
void launch_halo_verify_from_init(const float* u, int rows, size_t row_elems, int rank, int world, uint32_t steps,
                                  float alpha, float s, unsigned long long* mismatch_count, cudaStream_t stream);
// Exact check of one step: u_new against the stencil of u_old with the given boundary rows (any may be peer-mapped).
void launch_halo_verify_step(const float* u_new, const float* u_old, const float* up_row, const float* dn_row,
                             int rows, size_t row_elems, float alpha, float s, unsigned long long* mismatch_count,
                             cudaStream_t stream);

// ------------------------------------------- fused concurrency "megakernel" ----
// One persistent launch that executes a whole command group of the concurrency
// benchmark: CTAs are partitioned between the commands, so compute and copies
// overlap by construction instead of by the runtime's stream scheduling.
enum class FusedKind : int { kBusy = 0, kTriad = 1, kCopy = 2 };
struct FusedCommand {
  FusedKind kind = FusedKind::kBusy;
  size_t n = 0;              // work-items (busy) / elements (triad, copy)
  size_t tripcount = 0;      // busy only
  void* dst = nullptr;       // copy: destination (device, peer, pinned-host or managed)
  const void* src = nullptr; // copy: source
  float* a = nullptr;        // busy: output; triad: a
  const float* b = nullptr;
  const float* c = nullptr;
  float s = 3.0f;
  int ctas = 0;              // 0 -> heuristic share of the SMs
};
constexpr int kFusedMaxCommands = 8;
// Returns the total number of CTAs launched.
int launch_fused_bench(const FusedCommand* cmds, int n_cmds, CopyEngine engine,
                       const CopyTuning& tune, int device, cudaStream_t stream);
// The stand-alone busy-wait command (N work-items x 64*tripcount dependent FMAs).
void launch_busy_wait(float* out, size_t n_items, size_t tripcount, cudaStream_t stream);

// --------------------------------------------- tensor-core compute command ----
// `T`: per-CTA bf16 tile D[128x256] += A[128x64] . B[256x64]^T repeated `tripcount` times with
// tcgen05.mma (TMEM accumulator), operands fetched once by TMA.  `operands` holds A then B
// (tc_busy_operand_bytes()), `out` receives ctas * 128 * 256 floats = tripcount * (A . B^T).
size_t tc_busy_operand_bytes();
size_t tc_busy_out_elems_per_cta();
void launch_tc_fill_operands(void* operands, cudaStream_t stream);
// cluster = 2 launches thread-block clusters of two CTAs that share the B tile through TMA multicast.
void launch_tc_busy(const void* operands, float* out, int ctas, uint32_t tripcount,
                    cudaStream_t stream, int cluster = 1);

// ------------------------------------------------- tensor-core GEMM -> put ----
// C[M,N] fp32 = A[M,K] . B[N,K]^T (bf16, K-major) with tcgen05/TMEM/TMA; the epilogue writes the tile to
// c_local and/or straight into c_peer over NVLink, then publishes sync.signal_flag.  M % 128 == N % 256 ==
// K % 64 == 0.  Returns the number of CTAs launched.
// out_bf16: C is stored as bf16 (half the NVLink bytes) instead of fp32.
// cluster: 0 = auto (CTA pairs sharing the B tile by TMA multicast when the shape allows), 1 = off, 2 = force,
// 3 = 2-SM UMMA (tcgen05.mma.cta_group::2, one 256x256 tile per CTA pair; opt-in).
// tma_epilogue (opt-in): the C tile leaves through the TMA unit (swizzled smem pieces + cp.async.bulk.tensor.2d stores)
// instead of st.global from the epilogue warps.
int launch_gemm_put(const void* a_bf16, const void* b_bf16, void* c_local, void* c_peer, int m, int n,
                    int k, bool out_bf16, const SyncOps& sync, int ctas, int device, cudaStream_t stream,
                    int cluster = 0, bool tma_epilogue = false);

// ------------------------------------- tensor-core GEMM fused with a collective ----
// GEMM -> reduce-scatter (tensor-parallel row-parallel layer): C_r = A_r[M,K_r] . B_r[N,K_r]^T is this rank's
// partial sum; the epilogue ADDS every tile into the fp32 shard [M/world, N] of the rank that owns those rows
// (red.global.add.v4.f32 over NVLink), then the last CTA publishes done_epoch on every rank's done_flag.
// The owner zeroes its shard before the step and reads it after all `world` flags arrived (launch_wait_flags).
// fp32 atomics: the summation order is not fixed.  M % (128*world) == N % 256 == K % 64 == 0.
struct GemmRsArgs {
  const void* a = nullptr;                          // bf16 [M, K_r], K-major
  const void* b = nullptr;                          // bf16 [N, K_r], K-major
  void* shard[kApiMaxRanks] = {nullptr};            // peer-mapped: every rank's [M/world, N], fp32 (bf16 if out_bf16)
  // true: the additions are issued by the TMA unit — each epilogue warp stages 32 x 32 fp32 pieces in swizzled shared
  // memory and one cp.reduce.async.bulk.tensor.2d (UTMAREDG.2D.ADD) adds 4 KiB — instead of REDG requests from the
  // LSU (fp32 shards only).  Same result; which one is faster is a measurement.
  bool tma_epilogue = false;
  // bf16 shards: REDG.E.ADD.BF16x8 — half the NVLink bytes, but each of the P additions rounds to bf16.
  bool out_bf16 = false;
  // GEMM -> all-reduce through the switch instead: when set, `shard` is ignored and every tile is added with
  // multimem.red.add.v4.f32 into this NVLS multicast mapping of a full fp32 [M, N] buffer that exists (zeroed) on
  // every rank — each rank's partial product leaves its GPU exactly once and all ranks end up with the whole sum.
  float* c_multicast = nullptr;
  uint32_t* done_flag[kApiMaxRanks] = {nullptr};    // word on rank q written by THIS rank (may be null)
  uint32_t done_epoch = 0;
  uint32_t* ticket = nullptr;                       // rank-local CTA ticket counter (needed iff any done_flag)
  uint32_t ticket_base = 0;
  int rank = 0, world = 1;
  int m = 0, n = 0, k = 0;
};
int launch_gemm_reduce_scatter(const GemmRsArgs& args, int ctas, int device, cudaStream_t stream, int cluster = 0);

// GEMM -> all-to-all: C_r = A_r[M,K] . B_r[N,K]^T, row block q of C_r goes to rank q: every tile is stored (fp32 or
// bf16) straight into slot `rank` of rank q's receive buffer [world, M/world, N]; done flags as above.
struct GemmA2aArgs {
  const void* a = nullptr;
  const void* b = nullptr;
  void* recv[kApiMaxRanks] = {nullptr};             // peer-mapped: every rank's receive buffer
  bool out_bf16 = false;
  uint32_t* done_flag[kApiMaxRanks] = {nullptr};
  uint32_t done_epoch = 0;
  uint32_t* ticket = nullptr;
  uint32_t ticket_base = 0;
  int rank = 0, world = 1;
  int m = 0, n = 0, k = 0;
};
int launch_gemm_all_to_all(const GemmA2aArgs& args, int ctas, int device, cudaStream_t stream, int cluster = 0);

// All-gather -> GEMM (column-parallel layer on row-sharded activations): C[M,N] = A[M,K] . B_r[N,K]^T where rank q
// holds rows [q*M/world, (q+1)*M/world) of A.  One gather thread per CTA pulls the peers' row blocks over NVLink
// with TMA bulk copies into a_full and counts arrivals per 128-row block in `ready`; a tile's loads wait for its
// block, the local block needs no wait.  `ready` counts up forever: a launch adds
// allgather_gemm_chunks_per_block(k, chunk_bytes) to the counter of every remote block, ready_base is the value
// before the launch.  The peers' blocks must be final before the launch (barrier) and done_flag tells them when
// this rank has finished reading.
struct AgGemmArgs {
  void* a_full = nullptr;                           // local bf16 [M, K]; this rank's rows already in place
  const void* a_src[kApiMaxRanks] = {nullptr};      // peer-mapped: rank q's row block [M/world, K]
  const void* b = nullptr;                          // bf16 [N, K]
  void* c = nullptr;                                // fp32 (or bf16 when out_bf16) [M, N]
  bool out_bf16 = false;
  int activation = 0;                               // fused into the epilogue: 0 none, 1 relu, 2 gelu (tanh form), 3 silu
  uint32_t* ready = nullptr;                        // local [M/128] arrival counters
  uint32_t ready_base = 0;
  int chunk_bytes = 0;                              // gather granularity; 0 -> 4096
  uint32_t* done_flag[kApiMaxRanks] = {nullptr};
  uint32_t done_epoch = 0;
  uint32_t* ticket = nullptr;
  uint32_t ticket_base = 0;
  uint64_t timeout_ns = 0;
  uint32_t* status = nullptr;
  int rank = 0, world = 1;
  int m = 0, n = 0, k = 0;
};
uint32_t allgather_gemm_chunks_per_block(int k, int chunk_bytes);
int launch_allgather_gemm(const AgGemmArgs& args, int ctas, int device, cudaStream_t stream, int cluster = 0);
// Waits until `count` (<= 32) consecutive words all reached `epoch` (the receiving side of the two kernels above).
void launch_wait_flags(const uint32_t* flags, int count, uint32_t epoch, uint64_t timeout_ns, uint32_t* status,
                       cudaStream_t stream);

// ------------------------------------------------------ allreduce miniapp ----
// Element types of the miniapp's arrays (↔ mpi::get_datatype<T>(), mpi_datatype.hpp:28-51: every one of them is usable
// with MPI_SUM upstream).  Kernels are instantiated per ADDITION CLASS: signed and unsigned integers of one width share
// the two's-complement add.
enum class ElemType : int {
  kFloat = 0, kInt = 1, kUInt = 2, kDouble = 3, kLong = 4, kULong = 5, kShort = 6, kUShort = 7, kUChar = 8
};
constexpr size_t elem_size(ElemType t) {
  return t == ElemType::kDouble || t == ElemType::kLong || t == ElemType::kULong ? 8
         : t == ElemType::kShort || t == ElemType::kUShort                       ? 2
         : t == ElemType::kUChar                                                 ? 1
                                                                                 : 4;
}

// VA = a, VB = b, VC = c (↔ Initialize, allreduce-mpi-sycl.cpp:33-41). Any pointer may be null.
void launch_init3(void* va, void* vb, void* vc, size_t n, double a, double b, double c,
                  ElemType type, cudaStream_t stream);
// VC += VA, the unfused kernel of the reference pattern (↔ Accumulate, :26-31).
void launch_accumulate(const void* va, void* vc, size_t n, ElemType type, cudaStream_t stream);
// Counts elements with |v - expected| >= 1e-6 (↔ the assert loop, :192-204).
void launch_count_mismatch(const void* v, size_t n, double expected, ElemType type,
                           unsigned long long* count, cudaStream_t stream);

// Fused ring "rotate + accumulate" allreduce: all P-1 exchange steps and all P
// accumulations in ONE launch per rank.  Hop t of chunk c is read once, added
// into VC and forwarded to the right neighbour's slot over NVLink; arrival is
// signalled per chunk, so communication, accumulation and forwarding pipeline
// across the ring without any host involvement.  Launches that reuse the same slots must be separated by a
// cross-rank barrier (launch_barrier_all): flow control covers the hops of ONE launch.
struct RingArgs {
  const void* va = nullptr;       // local input block (hop 0)
  void* vc = nullptr;             // local accumulator (VC += every hop)
  void* slots_local = nullptr;    // (world-1) * n elements, written by the left neighbour
  void* slots_right = nullptr;    // peer-mapped: the right neighbour's slots
  uint32_t* arrived_local = nullptr;  // n_chunks words, written by the left neighbour
  uint32_t* arrived_right = nullptr;  // peer-mapped: right neighbour's arrival words
  int world = 0;
  size_t n = 0;                   // elements per rank; n * elem_size a multiple of 16 bytes
  size_t chunk_elems = 0;         // 0 -> 128 KiB worth of elements; chunk bytes a multiple of 16
  uint32_t epoch_base = 0;        // arrival words count up: base + hop
  uint64_t timeout_ns = 0;
  uint32_t* status = nullptr;
  // Receive-slot policy.  0 (default) = world-1 slots, no flow control.  2 = the reference's VA/VB double
  // buffer: slots hold 2 * n elements, hop t lands in slot (t-1) % 2, and per-chunk ack words (n_chunks words,
  // written by the right neighbour into ack_local; ack_left = the left neighbour's, peer-mapped) keep a sender
  // from overwriting a chunk its neighbour has not consumed yet.  Ack epochs share epoch_base with the arrivals.
  int n_slots = 0;
  uint32_t* ack_local = nullptr;
  uint32_t* ack_left = nullptr;
  // Pull variant: the receiver LOADS every block from its left neighbour's memory (va_left for hop 1, slots_left for
  // the later hops; both peer-mapped) and keeps a local copy in slots_local for its own right neighbour;
  // slots_right is not used.  Same arrival / ack words, same slot policies.
  bool pull = false;
  const void* va_left = nullptr;
  const void* slots_left = nullptr;
};
size_t ring_num_chunks(size_t n, size_t chunk_elems, size_t elem_bytes = 4);
void launch_ring_allreduce(const RingArgs& args, ElemType type, int ctas, int device,
                           cudaStream_t stream);

// One-kernel "collective" allreduce (the miniapp's -a path, ↔ MPI_Allreduce :61-67).
// two-shot over peer mappings: rank r reduces slice r by loading it from every
// rank's VA and stores the sum into every rank's VC, then a cross-GPU barrier.
struct TwoShotArgs {
  const void* va[kApiMaxRanks] = {nullptr};  // peer-mapped inputs of every rank
  void* vc[kApiMaxRanks] = {nullptr};        // peer-mapped outputs of every rank
  uint32_t* pads[kApiMaxRanks] = {nullptr};  // signal pads of every rank
  uint32_t* ticket = nullptr;
  uint32_t ticket_base = 0;
  int rank = 0;
  int world = 0;
  size_t n = 0;                              // elements; n * elem_size a multiple of 16 * world bytes
  uint32_t barrier_epoch = 0;
  uint64_t timeout_ns = 0;
  uint32_t* status = nullptr;
};
int launch_allreduce_two_shot(const TwoShotArgs& args, ElemType type, int ctas, int device,
                              cudaStream_t stream);
// NVLS: multimem.ld_reduce over the multicast mapping of VA for slice `rank`,
// multimem.st of the sum into the multicast mapping of VC (in-switch reduce + broadcast).
struct NvlsArgs {
  const void* va_mc = nullptr;
  void* vc_mc = nullptr;
  uint32_t* pads[kApiMaxRanks] = {nullptr};
  uint32_t* ticket = nullptr;
  uint32_t ticket_base = 0;
  int rank = 0;
  int world = 0;
  size_t n = 0;
  uint32_t barrier_epoch = 0;
  uint64_t timeout_ns = 0;
  uint32_t* status = nullptr;
};
int launch_allreduce_nvls(const NvlsArgs& args, ElemType type, int ctas, int device,
                          cudaStream_t stream);

}  // namespace hpcp
