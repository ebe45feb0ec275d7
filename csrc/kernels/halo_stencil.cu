// K-halo: slab-decomposed 3-point stencil fused with its halo exchange — the suite's flagship.
//
// The reference's only communication loop is "kernel; wait; MPI_Send/Recv with both ring
// neighbours; wait; swap; kernel" (allreduce-mpi-sycl.cpp:167-181: Accumulate().wait(),
// SendRecvRing(VA -> right, VB <- left), swap, Accumulate().wait()): every step's compute
// consumes what the previous step received, and nothing overlaps.  K-halo is that dependency
// structure as a B200 kernel.  The global field is [world * rows][row_elems] floats, periodic in
// the row dimension and split into slabs of `rows` rows per GPU (one row = one message of the
// p2p benchmark, 188 743 680 B by default, p2p/peer2pear.cpp:115-116).  One step is the stream
// triad  a = b + s * c  with  b = alpha * u[r],  c = u[r-1] + u[r+1]:
//
//     u'[r][j] = alpha * u[r][j] + s * (u[r-1][j] + u[r+1][j])
//
// Row -1 is the left neighbour's last row and row `rows` the right neighbour's first row of the
// SAME step's input: the halo.  Two forms of the exchange, both inside the stencil kernel:
//   pull  the kernel reads the neighbours' boundary rows straight out of their field over NVLink
//         (cp.async.bulk global -> shared on a peer-mapped address).  No halo buffer exists, the
//         halo costs no HBM write and no HBM read on the consumer.
//   push  the kernel stores its freshly computed boundary rows into halo buffers on the neighbours
//         (cp.async.bulk shared -> peer global) next to the local store, from the same smem tile.
// `none` reads local halo buffers and talks to nobody: the compute kernel of the stock arm
// (kernel -> cudaMemcpyAsync / NCCL send+recv -> host wait), which models/halo.py times next to it.
//
// Work split.  A CTA owns column tiles j = blockIdx.x + k * gridDim.x of EVERY row and marches down
// the rows of a column tile, so each input tile is fetched from HBM once and used three times from
// shared memory (as u[r+1], u[r], u[r-1]); the result of row r overwrites the tile of row r-1 in
// place and leaves through the TMA unit.  Because a column tile is owned by the same CTA index on
// every rank and in every step, the only cross-CTA dependency of step g+1 is "CTA c of my two
// neighbours finished step g".  That is one monotonic word per (neighbour, CTA):
//   * RAW  my step g reads the neighbour's u_g boundary tile / my halo[g&1]: written in its step g-1;
//   * WAR  my step g overwrites u[(g+1)&1] / the neighbour's halo[(g+1)&1]: last read in its step g-1.
// Both are "neighbour's CTA c completed step g-1", i.e. flag >= g.  So K steps run in ONE launch
// with no grid barrier, no host sync and no per-step launch (`steps` > 1), or one launch per step
// (`steps` == 1) with the same words carrying the dependency across launches.
//
// Warp roles (TMA engine, one or two CTAs per SM):
//   warp 0 / lane 0   DMA thread: waits for the two neighbour words, streams tiles global -> smem
//                     (mbarrier complete_tx), stores finished tiles smem -> global (+ peers), publishes.
//   warps 1..4        math: wait full[up|centre|down], stencil in place, fence.proxy.async, arrive.
#include "api.h"

#include <algorithm>
#include <mutex>
#include <vector>

#include "../common/cuda_check.h"
#include "../common/signal.cuh"

namespace hpcp {

namespace {

constexpr int kHaloMathWarps = 4;
constexpr int kHaloThreads = 32 * (1 + kHaloMathWarps);

struct HaloParams {
  unsigned char* u[2];
  const unsigned char* up_src[2];   // row -1 of step parity p: pull = left neighbour's last row, else halo_lo[p]
  const unsigned char* dn_src[2];   // row `rows`:              pull = right neighbour's row 0,   else halo_hi[p]
  unsigned char* put_first[2];      // push: where my new row 0 goes on the left neighbour (its halo_hi[p])
  unsigned char* put_last[2];       // push: where my new last row goes on the right neighbour (its halo_lo[p])
  // Flag arrays, one 32-byte sector per CTA (index blockIdx.x * kHaloFlagWords):
  const uint32_t* wait_lo;          // local, written by the left neighbour's CTAs
  const uint32_t* wait_hi;          // local, written by the right neighbour's CTAs
  uint32_t* signal_lo;              // on the left neighbour (its wait_hi array)
  uint32_t* signal_hi;              // on the right neighbour (its wait_lo array)
  int rows;
  size_t row_bytes;
  size_t tile_begin, tile_end;      // column tiles [begin, end) of a row handled by this launch
  uint32_t tile_bytes;
  int stages;
  int l2_hint;                      // 1: L2 evict_first policy on the local streaming loads and stores (used once)
  float alpha, s;
  uint32_t step_base;
  int steps;
  uint64_t timeout_ns;
  uint32_t* status;
};

__device__ __forceinline__ float stencil1(float up, float ce, float dn, float alpha, float s) {
  // Explicitly rounded, never contracted: bit-identical to `alpha * u + s * (up + dn)` evaluated
  // operation by operation in fp32 (the PyTorch reference of the tests).
  return __fadd_rn(__fmul_rn(alpha, ce), __fmul_rn(s, __fadd_rn(up, dn)));
}
__device__ __forceinline__ float4 stencil4(const float4& up, const float4& ce, const float4& dn, float alpha,
                                           float s) {
  return make_float4(stencil1(up.x, ce.x, dn.x, alpha, s), stencil1(up.y, ce.y, dn.y, alpha, s),
                     stencil1(up.z, ce.z, dn.z, alpha, s), stencil1(up.w, ce.w, dn.w, alpha, s));
}

// Cursor into a ring of S mbarrier-guarded slots: slot index + the phase parity of its current use.
struct Ring {
  int slot;
  uint32_t phase;
  __device__ __forceinline__ void advance(int n, int S) {  // n < S
    slot += n;
    if (slot >= S) {
      slot -= S;
      phase ^= 1u;
    }
  }
  __device__ __forceinline__ Ring at(int n, int S) const {
    Ring r = *this;
    r.advance(n, S);
    return r;
  }
};

// mbarrier wait that gives up when the DMA thread reported a dead peer.
__device__ __forceinline__ bool mbar_wait_or_abort(uint64_t* bar, uint32_t parity, const volatile int* abort_w) {
  while (!ptx::mbar_try_wait(bar, parity)) {
    if (*abort_w != 0) return false;
  }
  return true;
}

// kMode: 0 none, 1 pull, 2 push.
template <int kMode>
__global__ void __launch_bounds__(kHaloThreads) halo_stencil_kernel(const HaloParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  const uint32_t T = p.tile_bytes;
  const int S = p.stages;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + static_cast<size_t>(S) * T);
  uint64_t* computed = full + S;
  volatile int* abort_w = reinterpret_cast<volatile int*>(computed + S);

  if (threadIdx.x == 0) {
    for (int i = 0; i < S; ++i) {
      ptx::mbar_init(&full[i], 1);
      ptx::mbar_init(&computed[i], kHaloMathWarps);
    }
    *abort_w = 0;
    ptx::fence_mbar_init();
  }
  __syncthreads();

  const int R = p.rows;
  const size_t n_tiles = p.tile_end - p.tile_begin;
  const size_t ncols = n_tiles > blockIdx.x ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  if (ncols == 0) return;  // same geometry on every rank: nobody waits for this CTA index
  const uint64_t loads_per_step = ncols * static_cast<uint64_t>(R + 2);
  const uint64_t comps_per_step = ncols * static_cast<uint64_t>(R);
  auto col_off = [&](size_t jj) { return (p.tile_begin + blockIdx.x + jj * gridDim.x) * static_cast<size_t>(T); };
  auto col_len = [&](size_t off) {
    return static_cast<uint32_t>(p.row_bytes - off < T ? p.row_bytes - off : T);
  };

  const int warp = threadIdx.x >> 5;
  if (warp == 0) {
    if (threadIdx.x != 0) return;
    // ------------------------------------------------------------------ DMA thread ----
    const uint64_t policy = p.l2_hint ? ptx::l2_policy_evict_first() : 0;
    Ring ld{0, 0};    // next tile to load
    Ring st{0, 0};    // tile the next finished row overwrote (= the next one to store)
    Ring done{0, 0};  // next `computed` barrier to consume
    for (int si = 0; si < p.steps; ++si) {
      const uint32_t g = p.step_base + static_cast<uint32_t>(si);
      const int in = static_cast<int>(g & 1u), out = in ^ 1;
      if (kMode != 0) {
        const bool ok = wait_epoch(p.wait_lo + blockIdx.x * kHaloFlagWords, g, p.timeout_ns, p.status) &&
                        wait_epoch(p.wait_hi + blockIdx.x * kHaloFlagWords, g, p.timeout_ns, p.status);
        if (!ok) {
          *abort_w = 1;
          return;
        }
        asm volatile("fence.proxy.async;" ::: "memory");  // acquired peer data -> visible to the bulk loads
      }
      const unsigned char* uin = p.u[in];
      unsigned char* uout = p.u[out];
      const unsigned char* up_src = p.up_src[in];
      const unsigned char* dn_src = p.dn_src[in];
      uint64_t issued = 0, retired = 0;  // tiles of THIS step, in load order
      size_t jj_l = 0;                   // load cursor: column tile, row slot m = row + 1
      int m_l = 0;
      auto issue_next = [&]() {
        const size_t off = col_off(jj_l);
        const uint32_t len = col_len(off);
        const unsigned char* src = m_l == 0       ? up_src + off
                                   : m_l == R + 1 ? dn_src + off
                                                  : uin + static_cast<size_t>(m_l - 1) * p.row_bytes + off;
        ptx::mbar_arrive_expect_tx(&full[ld.slot], len);
        if (p.l2_hint && m_l != 0 && m_l != R + 1)  // own rows: streamed once, never re-read through L2
          ptx::bulk_g2s_hint(smem + static_cast<size_t>(ld.slot) * T, src, len, &full[ld.slot], policy);
        else
          ptx::bulk_g2s(smem + static_cast<size_t>(ld.slot) * T, src, len, &full[ld.slot]);
        ld.advance(1, S);
        ++issued;
        if (++m_l == R + 2) {
          m_l = 0;
          ++jj_l;
        }
      };
      size_t jj_c = 0;  // compute cursor
      int r = 0;
      uint64_t i0 = 0;  // tile (in load order) that row r of column jj_c overwrites
      for (uint64_t c = 0; c < comps_per_step; ++c) {
        while (issued < loads_per_step && issued < retired + static_cast<uint64_t>(S)) issue_next();
        if (!mbar_wait_or_abort(&computed[done.slot], done.phase, abort_w)) return;
        done.advance(1, S);
        const size_t off = col_off(jj_c);
        const uint32_t len = col_len(off);
        const unsigned char* sa = smem + static_cast<size_t>(st.slot) * T;
        // interior rows are not read again before the next step has streamed the whole slab through L2; the boundary
        // rows are what the neighbours pull, leave them to the default policy
        if (p.l2_hint && r != 0 && r != R - 1)
          ptx::bulk_s2g_hint(uout + static_cast<size_t>(r) * p.row_bytes + off, sa, len, policy);
        else
          ptx::bulk_s2g(uout + static_cast<size_t>(r) * p.row_bytes + off, sa, len);
        if (kMode == 2) {
          if (r == 0) ptx::bulk_s2g(p.put_first[out] + off, sa, len);
          if (r == R - 1) ptx::bulk_s2g(p.put_last[out] + off, sa, len);
        }
        ptx::bulk_commit();
        ptx::bulk_wait_read<1>();  // every store but the newest has left shared memory
        retired = i0;              // tiles [0, i0) are free (incl. the two never-stored tiles of a finished column)
        if (++r == R) {            // next column: skip the centre-last and down-halo tiles
          r = 0;
          ++jj_c;
          i0 += 3;
          st.advance(3, S);
        } else {
          i0 += 1;
          st.advance(1, S);
        }
      }
      ptx::bulk_wait<0>();  // this step's stores are performed (local field and, in push mode, the peers' halos)
      asm volatile("fence.proxy.async;" ::: "memory");
      if (kMode != 0) {
        ptx::fence_acq_rel_sys();
        ptx::st_release_sys(p.signal_hi + blockIdx.x * kHaloFlagWords, g + 1u);
        ptx::st_release_sys(p.signal_lo + blockIdx.x * kHaloFlagWords, g + 1u);
      }
    }
  } else {
    // ------------------------------------------------------------------ math warps ----
    const int mt = static_cast<int>(threadIdx.x) - 32;
    const float alpha = p.alpha, s = p.s;
    Ring up_t{0, 0};  // tile of row r-1 (overwritten with the result of row r)
    Ring done{0, 0};
    for (int si = 0; si < p.steps; ++si) {
      size_t jj = 0;
      int r = 0;
      for (uint64_t c = 0; c < comps_per_step; ++c) {
        const Ring ce_t = up_t.at(1, S), dn_t = up_t.at(2, S);
        if (r == 0) {
          if (!mbar_wait_or_abort(&full[up_t.slot], up_t.phase, abort_w)) return;
          if (!mbar_wait_or_abort(&full[ce_t.slot], ce_t.phase, abort_w)) return;
        }
        if (!mbar_wait_or_abort(&full[dn_t.slot], dn_t.phase, abort_w)) return;
        float4* up = reinterpret_cast<float4*>(smem + static_cast<size_t>(up_t.slot) * T);
        const float4* ce = reinterpret_cast<const float4*>(smem + static_cast<size_t>(ce_t.slot) * T);
        const float4* dn = reinterpret_cast<const float4*>(smem + static_cast<size_t>(dn_t.slot) * T);
        const uint32_t nv = col_len(col_off(jj)) / 16;
#pragma unroll 4
        for (uint32_t v = mt; v < nv; v += 32 * kHaloMathWarps) up[v] = stencil4(up[v], ce[v], dn[v], alpha, s);
        ptx::fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the TMA store
        __syncwarp();
        if ((threadIdx.x & 31) == 0) ptx::mbar_arrive(&computed[done.slot]);
        done.advance(1, S);
        if (++r == R) {
          r = 0;
          ++jj;
          up_t.advance(3, S);
        } else {
          up_t.advance(1, S);
        }
      }
    }
  }
}

// ------------------------------------------------------------------ deep sweeps ----
// halo_sweep_kernel<D> (pull only): one pass over the slab advances a column tile by up to D steps.  Columns are
// independent and CTA c owns the same column tiles on every rank in every step, so a sweep of depth d starting at step
// g loads the R + 2d input tiles of a column (rows -d .. R+d-1 of u[g&1]: the left neighbour's last d rows, its own R
// rows, the right neighbour's first d rows), keeps the intermediate time levels on chip and stores only level d of rows
// 0 .. R-1 into u[(g+d)&1].  HBM traffic per step falls from ~2R rows to ~2R/d; NVLink bytes per step stay the same.
//
// Schedule (halo_sweep_schedule, identical on every rank): greedy sweeps of the largest ODD size <= min(D, remaining-1),
// so u[(g+d)&1] = u[(g+1)&1] keeps every parity-addressed buffer of the single-step kernel right, and the launch ends
// with a one-step sweep: u[(g-1)&1] holds step g-1 afterwards, what verify_last_step() recomputes from.  The step words
// are those of halo_stencil_kernel: wait for both neighbour words >= g at the start of a sweep, publish g+d at its end.
// RAW: the neighbours' rows of step g are complete.  WAR: u[(g+d)&1] was last read by the neighbours' previous sweep
// (odd length, same boundaries on every rank), which ended at g.
//
// On-chip wavefront.  Input tile i of a column (row m = i - d) arrives; for i >= 2 the math warps compute level 1 at
// row m-1 from the three input tiles i-2, i-1, i (read from shared memory), then level L at row m-L from level L-1's
// rows m-L-1, m-L (registers) and m-L+1 (just computed), L = 2 .. d.  Level L is valid from arrival 2L on, so arrivals
// 2d .. R+2d-1 produce level d of rows 0 .. R-1, written IN PLACE over input tile i-2 (read only by this arrival and the
// two before it).  Every thread owns fixed float4 positions of the tile: levels 1 .. D-1 keep two rows each in
// registers.  Every arrival i >= 2 is one `computed` event of its slot i-2, stored or not.
//
// Slot rules (Ring cursors, S stages):
//   * loads: tiles of a column in consecutive slots, R + 2d per column, at most S ahead of `retired`;
//   * events: slot i-2 for arrival i = 2 .. R+2d-1; the cursor moves by 1 per event and by 2 more at the end of a
//     column (the last two input tiles are never an event slot): +3 from the last event of a column to the next column's
//     first, as in halo_stencil_kernel;
//   * a stored event (i >= 2d) frees the tiles below it once bulk_wait_read<1> says the older stores have read their
//     slots (`retired = t`, as halo_stencil_kernel); an unstored event (i < 2d, the first 2d-2 of a column) frees its
//     own tile too, after bulk_wait_read<0> if a store is still pending (`retired = t + 1`) -- without that, the 2d + 1
//     tiles a column needs before its first store would not fit a 6-slot ring for d >= 3.
// tests/test_halo_sweep.py runs these rules as an executable model.
// Three math warps: 4 warps per CTA, two CTAs = 2 warps per SM sub-partition, which leaves each thread up to 255
// registers for the 2 x (D-1) x 11 float4 of wavefront state (D = 3: 247, no spills).  Eight math warps (9 warps per CTA,
// up to 5 per sub-partition) cap a thread at 96 registers and spill.
constexpr int kSweepMathWarps = 3;
constexpr int kSweepThreads = 32 * (1 + kSweepMathWarps);
constexpr uint32_t kSweepMaxTileBytes = 16 * 1024;  // register state is sized for 16 KiB tiles

struct SweepParams {
  unsigned char* u[2];
  const unsigned char* left_u[2];   // the left neighbour's u[p] (row 0); a sweep of depth d pulls its rows R-d .. R-1
  const unsigned char* right_u[2];  // the right neighbour's u[p]; a sweep of depth d pulls its rows 0 .. d-1
  const uint32_t* wait_lo;
  const uint32_t* wait_hi;
  uint32_t* signal_lo;
  uint32_t* signal_hi;
  int rows;
  size_t row_bytes;
  size_t tile_begin, tile_end;
  uint32_t tile_bytes;
  int stages;
  float alpha, s;
  uint32_t step_base;
  int steps;
  uint64_t timeout_ns;
  uint32_t* status;
};

__host__ __device__ __forceinline__ int sweep_depth(int remaining, int D) {
  const int x = remaining - 1 < D ? remaining - 1 : D;
  return x <= 1 ? 1 : x - 1 + (x & 1);  // largest odd <= x
}

template <int D>
__global__ void __launch_bounds__(kSweepThreads, 2) halo_sweep_kernel(const SweepParams p) {
  static_assert(D >= 3 && (D & 1) == 1, "deep sweeps have odd depth >= 3");
  extern __shared__ __align__(128) unsigned char smem[];
  const uint32_t T = p.tile_bytes;
  const int S = p.stages;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + static_cast<size_t>(S) * T);
  uint64_t* computed = full + S;
  volatile int* abort_w = reinterpret_cast<volatile int*>(computed + S);

  if (threadIdx.x == 0) {
    for (int i = 0; i < S; ++i) {
      ptx::mbar_init(&full[i], 1);
      ptx::mbar_init(&computed[i], kSweepMathWarps);
    }
    *abort_w = 0;
    ptx::fence_mbar_init();
  }
  __syncthreads();

  const int R = p.rows;
  const size_t n_tiles = p.tile_end - p.tile_begin;
  const size_t ncols = n_tiles > blockIdx.x ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  if (ncols == 0) return;  // same geometry on every rank: nobody waits for this CTA index
  auto col_off = [&](size_t jj) { return (p.tile_begin + blockIdx.x + jj * gridDim.x) * static_cast<size_t>(T); };
  auto col_len = [&](size_t off) {
    return static_cast<uint32_t>(p.row_bytes - off < T ? p.row_bytes - off : T);
  };

  const int warp = threadIdx.x >> 5;
  if (warp == 0) {
    if (threadIdx.x != 0) return;
    // ------------------------------------------------------------------ DMA thread ----
    Ring ld{0, 0};    // next tile to load
    Ring ev{0, 0};    // slot of the next event (input tile i-2 of arrival i)
    Ring done{0, 0};  // next `computed` barrier to consume
    for (int k = 0; k < p.steps;) {
      const int d = sweep_depth(p.steps - k, D);
      const uint32_t g = p.step_base + static_cast<uint32_t>(k);
      const int in = static_cast<int>(g & 1u), out = in ^ 1;  // d is odd
      const bool ok = wait_epoch(p.wait_lo + blockIdx.x * kHaloFlagWords, g, p.timeout_ns, p.status) &&
                      wait_epoch(p.wait_hi + blockIdx.x * kHaloFlagWords, g, p.timeout_ns, p.status);
      if (!ok) {
        *abort_w = 1;
        return;
      }
      asm volatile("fence.proxy.async;" ::: "memory");  // acquired peer data -> visible to the bulk loads
      const unsigned char* uin = p.u[in];
      unsigned char* uout = p.u[out];
      const unsigned char* lo_src = p.left_u[in] + static_cast<size_t>(R - d) * p.row_bytes;
      const unsigned char* hi_src = p.right_u[in];
      const int n_in = R + 2 * d;  // input tiles of a column
      const uint64_t loads = ncols * static_cast<uint64_t>(n_in);
      const uint64_t events = ncols * static_cast<uint64_t>(n_in - 2);
      uint64_t issued = 0, retired = 0;  // tiles of THIS sweep, in load order
      size_t jj_l = 0;                   // load cursor: column tile, input tile m_l (row m_l - d)
      int m_l = 0;
      auto issue_next = [&]() {
        const size_t off = col_off(jj_l);
        const uint32_t len = col_len(off);
        const unsigned char* src = m_l < d       ? lo_src + static_cast<size_t>(m_l) * p.row_bytes + off
                                   : m_l < R + d ? uin + static_cast<size_t>(m_l - d) * p.row_bytes + off
                                                 : hi_src + static_cast<size_t>(m_l - R - d) * p.row_bytes + off;
        ptx::mbar_arrive_expect_tx(&full[ld.slot], len);
        ptx::bulk_g2s(smem + static_cast<size_t>(ld.slot) * T, src, len, &full[ld.slot]);
        ld.advance(1, S);
        ++issued;
        if (++m_l == n_in) {
          m_l = 0;
          ++jj_l;
        }
      };
      size_t jj_c = 0;     // event cursor: column tile, arrival i
      int i = 2;
      uint64_t t = 0;      // tile (in load order) of the current event
      bool pending = false;  // a store newer than the last bulk_wait_read<0> may still read its slot
      for (uint64_t e = 0; e < events; ++e) {
        while (issued < loads && issued < retired + static_cast<uint64_t>(S)) issue_next();
        if (!mbar_wait_or_abort(&computed[done.slot], done.phase, abort_w)) return;
        done.advance(1, S);
        if (i >= 2 * d) {
          const size_t off = col_off(jj_c);
          ptx::bulk_s2g(uout + static_cast<size_t>(i - 2 * d) * p.row_bytes + off,
                        smem + static_cast<size_t>(ev.slot) * T, col_len(off));
          ptx::bulk_commit();
          ptx::bulk_wait_read<1>();  // every store but the newest has left shared memory
          retired = t;
          pending = true;
        } else {
          if (pending) ptx::bulk_wait_read<0>();
          pending = false;
          retired = t + 1;
        }
        ++t;
        ev.advance(1, S);
        if (++i == n_in) {  // next column: the last two input tiles are no event slot
          i = 2;
          ++jj_c;
          t += 2;
          ev.advance(2, S);
        }
      }
      ptx::bulk_wait<0>();  // this sweep's stores are performed
      asm volatile("fence.proxy.async;" ::: "memory");
      ptx::fence_acq_rel_sys();
      ptx::st_release_sys(p.signal_hi + blockIdx.x * kHaloFlagWords, g + static_cast<uint32_t>(d));
      ptx::st_release_sys(p.signal_lo + blockIdx.x * kHaloFlagWords, g + static_cast<uint32_t>(d));
      k += d;
    }
  } else {
    // ------------------------------------------------------------------ math warps ----
    constexpr int P = (kSweepMaxTileBytes / 16 + 32 * kSweepMathWarps - 1) / (32 * kSweepMathWarps);  // float4 / thread
    const uint32_t mt = threadIdx.x - 32;
    const float alpha = p.alpha, s = p.s;
    // lv[L-1][0|1][k]: rows q-1, q of level L (the two newest) at position k, L = 1 .. D-1
    float4 lv[D - 1][2][P];
#pragma unroll
    for (int L = 0; L < D - 1; ++L)
#pragma unroll
      for (int k = 0; k < P; ++k) lv[L][0][k] = lv[L][1][k] = make_float4(0.f, 0.f, 0.f, 0.f);
    Ring up_t{0, 0};  // input tile i-2 of arrival i (overwritten with level d of row i-2d)
    Ring done{0, 0};
    for (int ks = 0; ks < p.steps;) {
      const int d = sweep_depth(p.steps - ks, D);
      const int n_in = R + 2 * d;
      for (size_t jj = 0; jj < ncols; ++jj) {
        const uint32_t nv = col_len(col_off(jj)) / 16;
        for (int i = 2; i < n_in; ++i) {
          const Ring ce_t = up_t.at(1, S), dn_t = up_t.at(2, S);
          if (i == 2) {
            if (!mbar_wait_or_abort(&full[up_t.slot], up_t.phase, abort_w)) return;
            if (!mbar_wait_or_abort(&full[ce_t.slot], ce_t.phase, abort_w)) return;
          }
          if (!mbar_wait_or_abort(&full[dn_t.slot], dn_t.phase, abort_w)) return;
          float4* up = reinterpret_cast<float4*>(smem + static_cast<size_t>(up_t.slot) * T);
          const float4* ce = reinterpret_cast<const float4*>(smem + static_cast<size_t>(ce_t.slot) * T);
          const float4* dn = reinterpret_cast<const float4*>(smem + static_cast<size_t>(dn_t.slot) * T);
          const bool store = i >= 2 * d;
#pragma unroll
          for (int k = 0; k < P; ++k) {
            const uint32_t v = mt + static_cast<uint32_t>(k) * 32 * kSweepMathWarps;
            if (v < nv) {
              float4 x = stencil4(up[v], ce[v], dn[v], alpha, s);  // level 1, row i-d-1
#pragma unroll
              for (int L = 2; L <= D; ++L) {
                if (L <= d) {
                  float4 y = x;  // not valid before arrival 2L, and then only feeds levels that are not valid either
                  if (i >= 2 * L) y = stencil4(lv[L - 2][0][k], lv[L - 2][1][k], x, alpha, s);  // level L, row i-d-L
                  lv[L - 2][0][k] = lv[L - 2][1][k];
                  lv[L - 2][1][k] = x;
                  x = y;
                }
              }
              if (store) up[v] = x;
            }
          }
          if (store) ptx::fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the TMA store
          __syncwarp();
          if ((threadIdx.x & 31) == 0) ptx::mbar_arrive(&computed[done.slot]);
          done.advance(1, S);
          up_t.advance(1, S);
        }
        up_t.advance(2, S);
      }
      ks += d;
    }
  }
}

// ------------------------------------------------------------- field values ----
// u0(global row, column): a hash folded to [-32, 32) with 10 fractional bits, reproducible on the host
// (models/halo.py::initial_field).
__device__ __forceinline__ float halo_u0(uint32_t grow, uint64_t j) {
  const uint32_t jl = static_cast<uint32_t>(j);
  const uint32_t h = (grow * 2654435761u) ^ (jl * 40503u + (jl >> 11));
  return static_cast<float>(static_cast<int>(h & 0xFFFFu) - 32768) * (1.0f / 1024.0f);
}

__global__ void halo_init_kernel(float* __restrict__ u, float* __restrict__ halo_lo, float* __restrict__ halo_hi,
                                 int rows, size_t row_elems, int rank, int world) {
  const uint32_t grows = static_cast<uint32_t>(rows) * world;
  const uint32_t first = static_cast<uint32_t>(rank) * rows;
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (size_t j = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; j < row_elems; j += stride) {
    for (int r = 0; r < rows; ++r) u[static_cast<size_t>(r) * row_elems + j] = halo_u0(first + r, j);
    if (halo_lo != nullptr) halo_lo[j] = halo_u0((first + grows - 1) % grows, j);
    if (halo_hi != nullptr) halo_hi[j] = halo_u0((first + rows) % grows, j);
  }
}

// Independent check from the closed-form initial field: every thread owns one column of the GLOBAL
// field (all world * rows rows), advances it `steps` times with the periodic stencil in the kernel's
// operation order and compares this rank's rows exactly.
constexpr int kHaloMaxGlobalRows = 128;
__global__ void halo_verify_init_kernel(const float* __restrict__ u, int rows, size_t row_elems, int rank, int world,
                                        uint32_t steps, float alpha, float s, unsigned long long* mismatch_count) {
  const int G = rows * world;
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  unsigned long long bad = 0;
  float v[kHaloMaxGlobalRows];
  for (size_t j = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; j < row_elems; j += stride) {
    for (int g = 0; g < G; ++g) v[g] = halo_u0(static_cast<uint32_t>(g), j);
    for (uint32_t k = 0; k < steps; ++k) {
      const float first = v[0];
      float prev = v[G - 1];
      for (int g = 0; g < G; ++g) {
        const float cur = v[g];
        const float next = g + 1 < G ? v[g + 1] : first;
        v[g] = stencil1(prev, cur, next, alpha, s);
        prev = cur;
      }
    }
    for (int r = 0; r < rows; ++r) bad += (__ldcg(u + static_cast<size_t>(r) * row_elems + j) != v[rank * rows + r]);
  }
  for (int off = 16; off > 0; off >>= 1) bad += __shfl_xor_sync(0xffffffffu, bad, off);
  if ((threadIdx.x & 31) == 0 && bad) atomicAdd(mismatch_count, bad);
}

// Check of ONE step through an independent data path: plain (coherent) vector loads of the step's input,
// including the neighbours' boundary rows wherever they live (peer-mapped field or local halo buffer).
__global__ void halo_verify_step_kernel(const float* __restrict__ u_new, const float* __restrict__ u_old,
                                        const float* __restrict__ up_row, const float* __restrict__ dn_row, int rows,
                                        size_t row_elems, float alpha, float s, unsigned long long* mismatch_count) {
  const size_t nvec = row_elems / 4;
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  unsigned long long bad = 0;
  auto ld = [](const float* base, size_t v) {
    const uint4 w = ptx::ld_peer_v4(reinterpret_cast<const uint4*>(base) + v);
    return make_float4(__uint_as_float(w.x), __uint_as_float(w.y), __uint_as_float(w.z), __uint_as_float(w.w));
  };
  for (size_t v = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; v < nvec; v += stride) {
    float4 up = ld(up_row, v);
    float4 ce = ld(u_old, v);
    for (int r = 0; r < rows; ++r) {
      const float4 dn = r + 1 < rows ? ld(u_old + static_cast<size_t>(r + 1) * row_elems, v) : ld(dn_row, v);
      const float4 want = stencil4(up, ce, dn, alpha, s);
      const float4 got = ld(u_new + static_cast<size_t>(r) * row_elems, v);
      bad += (got.x != want.x) + (got.y != want.y) + (got.z != want.z) + (got.w != want.w);
      up = ce;
      ce = dn;
    }
  }
  for (int off = 16; off > 0; off >>= 1) bad += __shfl_xor_sync(0xffffffffu, bad, off);
  if ((threadIdx.x & 31) == 0 && bad) atomicAdd(mismatch_count, bad);
}

struct HaloGeometry {
  uint32_t tile_bytes;
  int stages;
  size_t smem;
  int ctas;
};

template <auto kKernel, int kThreads>
int occupancy_of(size_t smem) {
  // One attribute + occupancy query per (kernel, smem, device), not per launch (per-step launches come here K times).
  // The dynamic shared-memory limit of the function is only ever RAISED: instances with different stage counts coexist.
  struct Entry {
    size_t smem;
    int device, per_sm;
  };
  static std::mutex mu;
  static std::vector<Entry> cache;
  static size_t limit_set[64] = {0};
  int device = 0;
  HPCP_CUDA(cudaGetDevice(&device));
  std::lock_guard<std::mutex> lk(mu);
  if (device >= 0 && device < 64 && smem > limit_set[device]) {
    HPCP_ENABLE_SMEM(kKernel, smem);
    limit_set[device] = smem;
  }
  for (const Entry& e : cache)
    if (e.smem == smem && e.device == device) return e.per_sm;
  int per_sm = 0;
  HPCP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kKernel, kThreads, smem));
  cache.push_back({smem, device, per_sm});
  return per_sm;
}

// Deep sweeps need pull mode, tiles of at most 16 KiB (the register state of the wavefront) and the default L2 policy
// (the evict_first hint exists only in halo_stencil_kernel); rows do not matter here, so the grid does not depend on
// them.
bool sweeps_allowed(HaloMode mode, const HaloTuning& tune) {
  const int tile_kb = tune.tile_kb > 0 ? tune.tile_kb : 16;
  return mode == HaloMode::kPull && tune.depth != 1 && tile_kb * 1024u <= kSweepMaxTileBytes && tune.l2_hint == 0;
}

HaloGeometry halo_geometry(size_t row_bytes, const HaloTuning& tune, HaloMode mode, int device) {
  HaloGeometry g;
  g.tile_bytes = static_cast<uint32_t>((tune.tile_kb > 0 ? tune.tile_kb : 16) * 1024);
  g.stages = tune.stages > 0 ? tune.stages : 6;  // 6 x 16 KiB: two CTAs per SM (measured best, profiles/r2c1)
  HPCP_REQUIRE(g.stages >= 6, "halo_stencil: needs >= 6 shared-memory stages");
  g.smem = static_cast<size_t>(g.stages) * g.tile_bytes + static_cast<size_t>(g.stages) * 16 + 16;
  HPCP_REQUIRE(g.smem <= 227 * 1024, "halo_stencil: stages * tile exceed 227 KiB of shared memory");
  const int sms = device_sm_count(device);
  int per_sm = 1;
  // Co-residency: a persistent multi-step launch spins on neighbour words, so every CTA must be resident.
  switch (mode) {
    case HaloMode::kNone: per_sm = occupancy_of<halo_stencil_kernel<0>, kHaloThreads>(g.smem); break;
    case HaloMode::kPull: per_sm = occupancy_of<halo_stencil_kernel<1>, kHaloThreads>(g.smem); break;
    case HaloMode::kPush: per_sm = occupancy_of<halo_stencil_kernel<2>, kHaloThreads>(g.smem); break;
  }
  // A time series mixes single-step and deep launches with the same step words (indexed by CTA): one grid that both
  // kernels keep fully resident.
  if (sweeps_allowed(mode, tune))
    per_sm = std::min(per_sm, occupancy_of<halo_sweep_kernel<3>, kSweepThreads>(g.smem));
  HPCP_REQUIRE(per_sm >= 1, "halo_stencil: kernel does not fit on an SM");
  const size_t tiles = (row_bytes + g.tile_bytes - 1) / g.tile_bytes;
  const int resident = std::min(sms * per_sm, kHaloMaxCtas);  // one step word per CTA and side
  const int want = tune.ctas > 0 ? std::min(tune.ctas, resident) : resident;
  g.ctas = static_cast<int>(std::max<size_t>(1, std::min<size_t>(tiles, static_cast<size_t>(want))));
  HPCP_REQUIRE(g.ctas <= kHaloMaxCtas, "halo_stencil: more CTAs than flag words");
  return g;
}

}  // namespace

int halo_stencil_ctas(size_t row_elems, const HaloTuning& tune, HaloMode mode, int device) {
  return halo_geometry(row_elems * sizeof(float), tune, mode, device).ctas;
}

int halo_sweep_depth(int rows, HaloMode mode, const HaloTuning& tune) {
  HPCP_REQUIRE(tune.depth >= 0, "halo_stencil: depth >= 0");
  if (!sweeps_allowed(mode, tune)) return 1;
  // Halo rows come only from the immediate neighbours: depth <= rows.  Depth 3 is the only instantiation: depth 5 keeps
  // 2 x 4 x 11 float4 = 352 registers of wavefront state per thread, more than two CTAs per SM can hold.
  const int want = std::min(tune.depth > 0 ? tune.depth : kHaloDefaultDepth, rows);
  return want >= 3 ? 3 : 1;
}

std::vector<int> halo_sweep_schedule(int steps, int depth) {
  std::vector<int> out;
  for (int k = 0; k < steps;) {
    out.push_back(sweep_depth(steps - k, depth));
    k += out.back();
  }
  return out;
}

int launch_halo_stencil(const HaloStencilArgs& a, HaloMode mode, const HaloTuning& tune, int device,
                        cudaStream_t stream) {
  HPCP_REQUIRE(a.rows >= 1 && a.row_elems > 0 && a.row_elems % 4 == 0,
               "halo_stencil: rows >= 1 and row_elems a positive multiple of 4");
  HPCP_REQUIRE(a.steps >= 1, "halo_stencil: steps >= 1");
  HPCP_REQUIRE(a.u[0] != nullptr && a.u[1] != nullptr, "halo_stencil: both field buffers are needed");
  const size_t row_bytes = a.row_elems * sizeof(float);
  const HaloGeometry g = halo_geometry(row_bytes, tune, mode, device);
  const int ctas = g.ctas;
  const size_t tiles_per_row = (row_bytes + g.tile_bytes - 1) / g.tile_bytes;
  HaloParams p{};
  for (int q = 0; q < 2; ++q) {
    p.u[q] = reinterpret_cast<unsigned char*>(a.u[q]);
    if (mode == HaloMode::kPull) {
      HPCP_REQUIRE(a.left_u[q] != nullptr && a.right_u[q] != nullptr, "halo_stencil: pull needs the neighbours' fields");
      p.up_src[q] = reinterpret_cast<const unsigned char*>(a.left_u[q]) + static_cast<size_t>(a.rows - 1) * row_bytes;
      p.dn_src[q] = reinterpret_cast<const unsigned char*>(a.right_u[q]);
    } else {
      HPCP_REQUIRE(a.halo_lo[q] != nullptr && a.halo_hi[q] != nullptr, "halo_stencil: halo buffers are needed");
      p.up_src[q] = reinterpret_cast<const unsigned char*>(a.halo_lo[q]);
      p.dn_src[q] = reinterpret_cast<const unsigned char*>(a.halo_hi[q]);
    }
    if (mode == HaloMode::kPush) {
      HPCP_REQUIRE(a.left_halo_hi[q] != nullptr && a.right_halo_lo[q] != nullptr,
                   "halo_stencil: push needs the neighbours' halo buffers");
      p.put_first[q] = reinterpret_cast<unsigned char*>(a.left_halo_hi[q]);
      p.put_last[q] = reinterpret_cast<unsigned char*>(a.right_halo_lo[q]);
    }
  }
  if (mode != HaloMode::kNone) {
    HPCP_REQUIRE(a.flags_local != nullptr && a.flags_left != nullptr && a.flags_right != nullptr,
                 "halo_stencil: neighbour flag words are needed");
    HPCP_REQUIRE(a.flag_set >= 0 && a.flag_set < kHaloFlagSets, "halo_stencil: flag_set out of range");
  }
  p.rows = a.rows;
  p.row_bytes = row_bytes;
  p.tile_begin = a.tile_begin;
  p.tile_end = a.tile_end == 0 ? tiles_per_row : a.tile_end;
  HPCP_REQUIRE(p.tile_begin < p.tile_end && p.tile_end <= tiles_per_row, "halo_stencil: bad column-tile range");
  p.tile_bytes = g.tile_bytes;
  p.stages = g.stages;
  p.l2_hint = tune.l2_hint;
  p.alpha = a.alpha;
  p.s = a.s;
  p.step_base = a.step_base;
  p.steps = a.steps;
  p.timeout_ns = a.timeout_ns;
  p.status = a.status;
  // Flag words: one 32-byte sector per (flag set, side, CTA); the kernel adds blockIdx.x * kHaloFlagWords.
  const size_t set_words = static_cast<size_t>(a.flag_set) * 2 * kHaloMaxCtas * kHaloFlagWords;
  const size_t side_words = static_cast<size_t>(kHaloMaxCtas) * kHaloFlagWords;
  auto launch = [&](auto kernel) {  // the shared-memory attribute was set when the geometry was computed
    kernel<<<ctas, kHaloThreads, g.smem, stream>>>(p);
  };
  if (mode != HaloMode::kNone) {
    p.wait_lo = a.flags_local + set_words;
    p.wait_hi = a.flags_local + set_words + side_words;
    p.signal_lo = a.flags_left + set_words + side_words;  // I am the right neighbour of my left neighbour
    p.signal_hi = a.flags_right + set_words;              // and the left neighbour of my right neighbour
  }
  const int depth = halo_sweep_depth(a.rows, mode, tune);
  if (depth > 1 && sweep_depth(a.steps, depth) > 1) {  // at least one deep sweep: K >= 4
    SweepParams q{};
    for (int r = 0; r < 2; ++r) {
      q.u[r] = p.u[r];
      q.left_u[r] = reinterpret_cast<const unsigned char*>(a.left_u[r]);
      q.right_u[r] = reinterpret_cast<const unsigned char*>(a.right_u[r]);
    }
    q.wait_lo = p.wait_lo;
    q.wait_hi = p.wait_hi;
    q.signal_lo = p.signal_lo;
    q.signal_hi = p.signal_hi;
    q.rows = p.rows;
    q.row_bytes = p.row_bytes;
    q.tile_begin = p.tile_begin;
    q.tile_end = p.tile_end;
    q.tile_bytes = p.tile_bytes;
    q.stages = p.stages;
    q.alpha = p.alpha;
    q.s = p.s;
    q.step_base = p.step_base;
    q.steps = p.steps;
    q.timeout_ns = p.timeout_ns;
    q.status = p.status;
    halo_sweep_kernel<3><<<ctas, kSweepThreads, g.smem, stream>>>(q);
    HPCP_CUDA(cudaGetLastError());
    return ctas;
  }
  switch (mode) {
    case HaloMode::kNone: launch(halo_stencil_kernel<0>); break;
    case HaloMode::kPull: launch(halo_stencil_kernel<1>); break;
    case HaloMode::kPush: launch(halo_stencil_kernel<2>); break;
  }
  HPCP_CUDA(cudaGetLastError());
  return ctas;
}

void launch_halo_init(float* u, float* halo_lo, float* halo_hi, int rows, size_t row_elems, int rank, int world,
                      cudaStream_t stream) {
  const int threads = 256;
  const int ctas = static_cast<int>(std::min<size_t>((row_elems + threads - 1) / threads, 148 * 8));
  halo_init_kernel<<<std::max(ctas, 1), threads, 0, stream>>>(u, halo_lo, halo_hi, rows, row_elems, rank, world);
  HPCP_CUDA(cudaGetLastError());
}

void launch_halo_verify_from_init(const float* u, int rows, size_t row_elems, int rank, int world, uint32_t steps,
                                  float alpha, float s, unsigned long long* mismatch_count, cudaStream_t stream) {
  HPCP_REQUIRE(rows * world <= kHaloMaxGlobalRows, "halo verify: world * rows exceeds 128 global rows");
  const int threads = 128;
  const int ctas = static_cast<int>(std::min<size_t>((row_elems + threads - 1) / threads, 148 * 16));
  halo_verify_init_kernel<<<std::max(ctas, 1), threads, 0, stream>>>(u, rows, row_elems, rank, world, steps, alpha, s,
                                                                    mismatch_count);
  HPCP_CUDA(cudaGetLastError());
}

void launch_halo_verify_step(const float* u_new, const float* u_old, const float* up_row, const float* dn_row,
                             int rows, size_t row_elems, float alpha, float s, unsigned long long* mismatch_count,
                             cudaStream_t stream) {
  const int threads = 256;
  const int ctas = static_cast<int>(std::min<size_t>((row_elems / 4 + threads - 1) / threads, 148 * 8));
  halo_verify_step_kernel<<<std::max(ctas, 1), threads, 0, stream>>>(u_new, u_old, up_row, dn_row, rows, row_elems,
                                                                    alpha, s, mismatch_count);
  HPCP_CUDA(cudaGetLastError());
}

}  // namespace hpcp
