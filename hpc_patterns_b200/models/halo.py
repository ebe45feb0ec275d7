"""Halo exchange fused into a slab stencil: the flagship pattern of this suite.

The reference's one communication loop is the miniapp's ring: compute, wait, exchange a
full block with BOTH ring neighbours (``MPI_Send`` to the right, ``MPI_Recv`` from the
left), wait, swap, compute on what arrived (allreduce-mpi-sycl.cpp:167-181) — a 1-D
periodic neighbour exchange with a true step-to-step dependency and no overlap at all.
``HaloStencil`` is that loop as a time-stepping stencil on B200s:

* the global field ``[world * rows][row_elems]`` is periodic in the row dimension and
  split into slabs of ``rows`` rows per GPU; one row is one message (188 743 680 B by
  default, the size of p2p/peer2pear.cpp:115-116);
* a step is ``u' = alpha*u + s*(u[r-1] + u[r+1])`` (the stream triad ``a = b + s*c`` with
  a neighbour sum for ``c``); rows -1 / ``rows`` are the neighbours' boundary rows of the
  same step, so step g+1 consumes what step g produced on the neighbours;
* the exchange happens INSIDE the stencil kernel (csrc/kernels/halo_stencil.cu): ``pull``
  reads the boundary rows out of the neighbours' fields over NVLink with TMA bulk loads,
  ``push`` stores the new boundary rows into the neighbours' halo buffers with TMA bulk
  stores; per-CTA step words keep it RAW/WAR safe without any barrier or host sync, and
  ``step(k)`` runs k steps in one persistent launch;
* in pull mode a k-step launch advances the slab by up to ``depth`` steps per pass over it
  (deep halos: ``depth`` rows pulled from each neighbour, the intermediate time levels kept
  on chip), so HBM moves ~2*rows/depth rows per step instead of ~2*rows; the sweep sizes
  follow ``sweep_schedule`` and the result is bit-identical to one step per pass.

``stock_step`` is the reference's shape through library calls (the thing to beat):
compute kernel, host wait, ``cudaMemcpyAsync`` to the peers or NCCL send/recv, host wait.
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional

import torch

from .. import native
from ..parallel.comm import Comm
from ..parallel.symmetric import SignalPads, SymmetricBuffer, tensor_from_ptr

REFERENCE_MESSAGE_BYTES = 1179648 * 40 * 4  # 188 743 680, p2p/peer2pear.cpp:115-116
DEFAULT_ROWS = 8
MODES = ("pull", "push", "none")


def balanced_rows(hbm_gbs: float = 6567.4, nvlink_gbs: float = 706.1) -> int:
    """Rows per slab for which the step's HBM time equals its NVLink time.

    The reference's concurrency benchmark tunes its commands to equal duration before it
    overlaps them (concurency/main.cpp:219-258); the same rule here: a step streams
    (2*rows + 2) rows through HBM in pull mode (rows reads + rows writes + the two boundary
    rows the neighbours read) and moves 2 rows over NVLink in EACH direction at once.
    Denominators are stock measurements, not this kernel's: the driver's copy peak
    (MEASURED_PEAKS.json hbm_gbs) and the copy engines' rate with both directions of a pair
    busy — 1412.2 GB/s per pair = 706.1 per direction (profiles/r2_call3_2gpu/p2p_tune.jsonl;
    one direction alone reaches 717-770).  -> 8 rows.
    """
    rows = (2.0 * hbm_gbs / nvlink_gbs - 2.0) / 2.0
    return max(1, int(rows))


DEFAULT_SWEEP_DEPTH = 3       # kHaloDefaultDepth (csrc/kernels/api.h)
SWEEP_MAX_TILE_KB = 16        # the deep kernel's register state is sized for 16 KiB tiles


def sweep_depth(rows: int, mode: str, tune: Optional[dict] = None) -> int:
    """Deepest sweep a multi-step launch takes (halo_sweep_depth in halo_stencil.cu): deep sweeps need pull mode, tiles
    of at most 16 KiB and the default L2 policy; tune ``depth`` 0 / missing is the default, 1 one step per sweep; the
    depth is at most ``rows`` (halo rows come from the immediate neighbours only) and 3 is the one instantiation."""
    tune = tune or {}
    depth = int(tune.get("depth") or 0)
    if depth < 0:
        raise ValueError("depth >= 0")
    allowed = (mode == "pull" and depth != 1 and int(tune.get("tile_kb") or 16) <= SWEEP_MAX_TILE_KB
               and not tune.get("l2_hint"))
    return 3 if allowed and min(depth or DEFAULT_SWEEP_DEPTH, rows) >= 3 else 1


def sweep_schedule(steps: int, depth: int) -> List[int]:
    """Sweep sizes of a ``steps``-step launch whose deepest sweep is ``depth`` (halo_sweep_schedule in
    halo_stencil.cu): greedy, the largest odd size <= min(depth, remaining - 1).  Odd sizes keep the ping-pong parity
    of every step; the last sweep is one step, so the buffer of step g-1 holds it after the launch."""
    out: List[int] = []
    k = 0
    while k < steps:
        x = min(depth, steps - k - 1)
        out.append(1 if x <= 1 else x - 1 + (x & 1))
        k += out[-1]
    return out


def initial_field(world: int, rows: int, row_elems: int) -> torch.Tensor:
    """The closed-form initial field of the kernels (halo_u0 in halo_stencil.cu), fp32 [world*rows, row_elems]."""
    g = torch.arange(world * rows, dtype=torch.int64).unsqueeze(1)
    j = torch.arange(row_elems, dtype=torch.int64).unsqueeze(0)
    h = ((g * 2654435761) & 0xFFFFFFFF) ^ ((j * 40503 + (j >> 11)) & 0xFFFFFFFF)
    return (((h & 0xFFFF) - 32768).to(torch.float32)) * (1.0 / 1024.0)


def reference_steps(field: torch.Tensor, steps: int, alpha: float = 0.5, s: float = 0.25) -> torch.Tensor:
    """Plain PyTorch fp32 reference of the whole (undecomposed) periodic stencil, operation by operation."""
    u = field.clone()
    a = torch.tensor(alpha, dtype=torch.float32)
    b = torch.tensor(s, dtype=torch.float32)
    for _ in range(steps):
        u = a * u + b * (torch.roll(u, 1, 0) + torch.roll(u, -1, 0))
    return u


class HaloStencil:
    """One rank's slab of the periodic field + the fused step.  One instance per process (torchrun) or
    several in one process on one GPU (``VirtualRing`` below: the protocol tests of a 1-GPU box)."""

    def __init__(self, comm: Comm, device: int, message_bytes: int = REFERENCE_MESSAGE_BYTES,
                 rows: int = DEFAULT_ROWS, mode: str = "pull", alpha: float = 0.5, s: float = 0.25,
                 tune: Optional[dict] = None, timeout_s: float = 30.0, _shared: Optional[dict] = None):
        if mode not in MODES:
            raise ValueError(f"mode must be one of {MODES}")
        if message_bytes % 16 or message_bytes <= 0:
            raise ValueError("message size (one row) must be a positive multiple of 16 bytes")
        if rows < 1:
            raise ValueError("rows must be >= 1")
        self.C = native()
        self.comm, self.device = comm, device
        self.rank, self.world = comm.rank, comm.world
        self.mode, self.alpha, self.s = mode, float(alpha), float(s)
        self.rows, self.row_bytes, self.row_elems = int(rows), int(message_bytes), int(message_bytes) // 4
        self.tune = dict(tune or {})
        if "depth" not in self.tune and os.environ.get("HPCP_HALO_DEPTH"):
            self.tune["depth"] = int(os.environ["HPCP_HALO_DEPTH"])
        self.left = (self.rank - 1) % self.world
        self.right = (self.rank + 1) % self.world
        torch.cuda.set_device(device)
        slab = self.rows * self.row_bytes
        if _shared is not None:         # virtual ranks of one process (VirtualRing): buffers made by the group
            self.pads, self.field, self.halo, self.flags = (_shared[k] for k in ("pads", "field", "halo", "flags"))
        else:
            self.pads = SignalPads(comm, device, timeout_s=timeout_s)
            self.field = SymmetricBuffer(comm, 2 * slab, device, zero=False)        # u[0] | u[1]
            self.halo = SymmetricBuffer(comm, 4 * self.row_bytes, device, zero=False)  # lo[0] lo[1] hi[0] hi[1]
            self.flags = SymmetricBuffer(comm, self.C.HALO_FLAG_BYTES, device, zero=True)
        self.ctas = self.C.halo_stencil_ctas(self.row_elems, "pull" if mode == "none" else mode, self.tune, device)
        if "ctas" in self.tune:
            self.ctas = min(self.ctas, int(self.tune["ctas"]))
        self.tune["ctas"] = self.ctas   # identical grid in every launch: flag words are indexed by CTA
        # deepest sweep of a multi-step launch (1 in push / none mode, with rows < 3 or tune depth 1)
        self.depth = sweep_depth(self.rows, mode, self.tune)
        self.last_schedule: List[int] = [1]   # sweep sizes of the most recent multi-step launch
        self._flag_layout: Optional[int] = None   # None until the first step; 1 = whole rows, n = n column chunks
        self.g = 0                      # global step counter (monotonic; the flag words count with it)
        self.launches = 0
        self._counter = torch.zeros(1, dtype=torch.int64, device=torch.device("cuda", device))
        self._streams: Dict[str, torch.cuda.Stream] = {}
        self.reset()

    # ---- addresses -------------------------------------------------------------------
    def u_ptr(self, rank: int, parity: int, row: int = 0) -> int:
        return self.field.ptrs[rank] + (parity * self.rows + row) * self.row_bytes

    def halo_ptr(self, rank: int, side: str, parity: int) -> int:
        return self.halo.ptrs[rank] + ((0 if side == "lo" else 2) + parity) * self.row_bytes

    def u_tensor(self, parity: Optional[int] = None) -> torch.Tensor:
        """This rank's current field (or the given parity) as a [rows, row_elems] fp32 view."""
        parity = self.g & 1 if parity is None else parity
        return tensor_from_ptr(self.u_ptr(self.rank, parity), self.rows * self.row_bytes, self.device,
                               torch.float32).view(self.rows, self.row_elems)

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _args(self, steps: int, flag_set: int = 0, tile_begin: int = 0, tile_end: int = 0) -> dict:
        me, le, ri = self.rank, self.left, self.right
        return {
            "u": [self.u_ptr(me, 0), self.u_ptr(me, 1)],
            "left_u": [self.u_ptr(le, 0), self.u_ptr(le, 1)],
            "right_u": [self.u_ptr(ri, 0), self.u_ptr(ri, 1)],
            "halo_lo": [self.halo_ptr(me, "lo", 0), self.halo_ptr(me, "lo", 1)],
            "halo_hi": [self.halo_ptr(me, "hi", 0), self.halo_ptr(me, "hi", 1)],
            "left_halo_hi": [self.halo_ptr(le, "hi", 0), self.halo_ptr(le, "hi", 1)],
            "right_halo_lo": [self.halo_ptr(ri, "lo", 0), self.halo_ptr(ri, "lo", 1)],
            "flags_local": self.flags.ptrs[me], "flags_left": self.flags.ptrs[le],
            "flags_right": self.flags.ptrs[ri], "flag_set": flag_set,
            "rows": self.rows, "row_elems": self.row_elems, "tile_begin": tile_begin, "tile_end": tile_end,
            "alpha": self.alpha, "s": self.s, "step_base": self.g & 0xFFFFFFFF, "steps": steps,
            "timeout_ns": self.pads.timeout_ns, "status": self.pads.status_ptr,
        }

    # ---- state -----------------------------------------------------------------------
    def reset(self) -> None:
        """Back to step 0: the closed-form initial field, halo buffers of step 0, zeroed step words."""
        torch.cuda.synchronize(self.device)
        self.comm.barrier()
        st = self._stream()
        self.C.memset_async(self.flags.local_ptr, 0, self.C.HALO_FLAG_BYTES, st)
        self.C.halo_init(self.u_ptr(self.rank, 0), self.halo_ptr(self.rank, "lo", 0),
                         self.halo_ptr(self.rank, "hi", 0), self.rows, self.row_elems, self.rank, self.world, st)
        self.g = 0
        self._flag_layout = None
        torch.cuda.synchronize(self.device)
        self.comm.barrier()

    def _use_layout(self, chunks: int) -> None:
        """A time series is stepped ONE way: whole-row fused steps (1), column-chunked host steps (n chunks, one word
        set per chunk) or stock steps (0: they exchange through library calls and never touch the step words, so a
        fused step after them would wait for words nobody advanced).  reset() starts a new series."""
        if self._flag_layout is None:
            self._flag_layout = chunks
        elif self._flag_layout != chunks:
            raise RuntimeError("fused steps, chunked host steps and stock steps keep different step words: "
                               "reset() between them")

    # ---- the fused step ----------------------------------------------------------------
    def step(self, steps: int = 1) -> None:
        """``steps`` time steps, exchange included, in ONE kernel launch on the current stream."""
        self._use_layout(1)
        self.C.halo_stencil(self._args(steps), self.mode, self.tune, self.device, self._stream())
        if steps > 1:   # per-step launches (timed as a side row) leave the traffic model of the persistent launch
            self.last_schedule = sweep_schedule(steps, self.depth)
        self.g += steps
        self.launches += 1

    # ---- unfused pieces (overlap %, stock arm) --------------------------------------------
    def compute_only(self) -> None:
        """The stencil kernel alone: reads the local halo buffers, exchanges nothing, does not advance the step
        counter (timing only: the field is no longer a valid time series afterwards — reset() before verifying)."""
        self.C.halo_stencil(self._args(1), "none", self.tune, self.device, self._stream())
        self.launches += 1

    def exchange_only(self, engine: str = "tma") -> None:
        """The two boundary rows put to the neighbours' halo buffers with the stand-alone K-p2p kernel (no compute),
        then wait for both arrivals — the transfer half of one step."""
        C, pads, st = self.C, self.pads, self._stream()
        self._xepoch = getattr(self, "_xepoch", 0) + 1
        par = (self.g + 1) & 1
        # message "to the left" is announced in the PAD_DONE section, "to the right" in PAD_ACK (two distinct words
        # even when both neighbours are the same rank, or this rank itself)
        for dst_rank, row, dst, section in ((self.left, 0, self.halo_ptr(self.left, "hi", par), C.PAD_DONE),
                                            (self.right, self.rows - 1, self.halo_ptr(self.right, "lo", par), C.PAD_ACK)):
            sync = pads.sync_ops(signal_rank=dst_rank, signal_section=section, epoch=self._xepoch)
            pads.advance_tickets(C.copy(dst, self.u_ptr(self.rank, par, row), self.row_bytes, False, engine, {},
                                        sync, self.device, st))
        # my right neighbour signalled PAD_DONE (I am its left), my left neighbour PAD_ACK
        C.wait(pads.word(self.rank, C.PAD_DONE + self.right), self._xepoch, pads.timeout_ns, pads.status_ptr, st)
        C.wait(pads.word(self.rank, C.PAD_ACK + self.left), self._xepoch, pads.timeout_ns, pads.status_ptr, st)
        self.launches += 4

    def stock_step(self, how: str = "memcpy", host_wait: bool = True) -> None:
        """The reference's loop shape through stock calls: kernel, wait, library transfer to both neighbours, wait
        (allreduce-mpi-sycl.cpp:176-181).  Numerically the same time series as ``step`` (the transfers fill the
        halo buffers the next kernel reads)."""
        C, pads = self.C, self.pads
        self._use_layout(0)
        stream = torch.cuda.current_stream(self.device)
        st = stream.cuda_stream
        out = (self.g + 1) & 1
        C.halo_stencil(self._args(1), "none", self.tune, self.device, st)
        self.launches += 1
        if host_wait:
            stream.synchronize()                                       # Accumulate(...).wait()
        first, last = self.u_ptr(self.rank, out, 0), self.u_ptr(self.rank, out, self.rows - 1)
        if how == "memcpy":
            self._sepoch = getattr(self, "_sepoch", 0) + 1
            C.memcpy_async(self.halo_ptr(self.left, "hi", out), first, self.row_bytes, st)
            C.memcpy_async(self.halo_ptr(self.right, "lo", out), last, self.row_bytes, st)
            C.signal(pads.word(self.left, C.PAD_READY + self.rank), self._sepoch, st)
            if self.right != self.left:
                C.signal(pads.word(self.right, C.PAD_READY + self.rank), self._sepoch, st)
            C.wait(pads.word(self.rank, C.PAD_READY + self.left), self._sepoch, pads.timeout_ns, pads.status_ptr, st)
            C.wait(pads.word(self.rank, C.PAD_READY + self.right), self._sepoch, pads.timeout_ns, pads.status_ptr, st)
        elif how == "nccl":
            import torch.distributed as dist
            row = self.row_bytes
            t_first = tensor_from_ptr(first, row, self.device, torch.float32)
            t_last = tensor_from_ptr(last, row, self.device, torch.float32)
            r_lo = tensor_from_ptr(self.halo_ptr(self.rank, "lo", out), row, self.device, torch.float32)
            r_hi = tensor_from_ptr(self.halo_ptr(self.rank, "hi", out), row, self.device, torch.float32)
            if self.world == 1:
                r_hi.copy_(t_first)
                r_lo.copy_(t_last)
            else:
                # tags keep the two messages of a 2-rank ring apart (both go to the same peer)
                ops = [dist.P2POp(dist.isend, t_last, self.right, tag=0), dist.P2POp(dist.irecv, r_lo, self.left, tag=0),
                       dist.P2POp(dist.isend, t_first, self.left, tag=1), dist.P2POp(dist.irecv, r_hi, self.right, tag=1)]
                for w in dist.batch_isend_irecv(ops):
                    w.wait()
        else:
            raise ValueError(how)
        if host_wait:
            stream.synchronize()                                       # the blocking MPI_Send/Recv pair
        self.g += 1

    # ---- checking -------------------------------------------------------------------------
    def _count(self) -> int:
        torch.cuda.synchronize(self.device)
        return int(self._counter.item())

    def verify_from_init(self) -> int:
        """Wrong words in this rank's slab against the closed-form field advanced ``g`` steps (exact)."""
        self._counter.zero_()
        self.C.halo_verify_from_init(self.u_ptr(self.rank, self.g & 1), self.rows, self.row_elems, self.rank,
                                     self.world, self.g & 0xFFFFFFFF, self.alpha, self.s,
                                     self._counter.data_ptr(), self._stream())
        return self._count()

    def verify_last_step(self) -> int:
        """Wrong words of the most recent step, recomputed through plain loads of its input — the neighbours'
        boundary rows are read straight from their fields (every rank must be idle: call after a barrier)."""
        if self.g == 0:
            return 0
        new, old = self.g & 1, (self.g - 1) & 1
        self._counter.zero_()
        self.C.halo_verify_step(self.u_ptr(self.rank, new), self.u_ptr(self.rank, old),
                                self.u_ptr(self.left, old, self.rows - 1), self.u_ptr(self.right, old, 0),
                                self.rows, self.row_elems, self.alpha, self.s, self._counter.data_ptr(),
                                self._stream())
        return self._count()

    def check(self) -> None:
        self.pads.check()

    # ---- end to end through host memory ------------------------------------------------------
    def make_host_buffers(self) -> List[torch.Tensor]:
        """Two pinned host fields [rows, row_elems]; [0] holds this rank's slab of the current step."""
        bufs = [torch.empty(self.rows, self.row_elems, dtype=torch.float32).pin_memory() for _ in range(2)]
        bufs[0].copy_(self.u_tensor())
        torch.cuda.synchronize(self.device)
        return bufs

    def step_from_host(self, host_in: torch.Tensor, host_out: torch.Tensor, chunks: int = 16) -> None:
        """Out-of-core time step, the public end-to-end call: the slab lives in pinned host memory; this uploads ALL of
        it (every input the step consumes), runs the fused step with the NVLink exchange, and downloads ALL of the new
        slab.  Column chunks pipeline H2D, kernel and D2H on three streams; the neighbours' halos never touch the host
        (push mode: they arrive in the halo buffers during the previous step).  Returns after the result is on the host.
        """
        if self.mode != "push":
            raise RuntimeError("step_from_host needs mode='push' (a pulled neighbour row would race with its upload)")
        C = self.C
        main = torch.cuda.current_stream(self.device)
        for name in ("h2d", "d2h"):
            if name not in self._streams:
                self._streams[name] = torch.cuda.Stream(self.device)
        h2d, d2h = self._streams["h2d"], self._streams["d2h"]
        tile = (self.tune.get("tile_kb") or 16) * 1024
        tiles = (self.row_bytes + tile - 1) // tile
        chunks = max(1, min(chunks, tiles, C.HALO_FLAG_SETS))
        per = (tiles + chunks - 1) // chunks
        self._use_layout(chunks if chunks > 1 else 1)
        inp, out = self.g & 1, (self.g + 1) & 1
        h2d.wait_stream(main)          # the previous step's kernels and downloads precede this upload
        h2d.wait_stream(d2h)
        for k in range(chunks):
            t0, t1 = k * per, min(tiles, (k + 1) * per)
            if t0 >= t1:
                break
            b0, b1 = t0 * tile, min(self.row_bytes, t1 * tile)
            for r in range(self.rows):
                C.memcpy_async(self.u_ptr(self.rank, inp, r) + b0, host_in[r].data_ptr() + b0, b1 - b0,
                               h2d.cuda_stream)
            up = torch.cuda.Event()
            up.record(h2d)
            main.wait_event(up)
            C.halo_stencil(self._args(1, flag_set=k, tile_begin=t0, tile_end=t1), self.mode, self.tune, self.device,
                           main.cuda_stream)
            self.launches += 1
            done = torch.cuda.Event()
            done.record(main)
            d2h.wait_event(done)
            for r in range(self.rows):
                C.memcpy_async(host_out[r].data_ptr() + b0, self.u_ptr(self.rank, out, r) + b0, b1 - b0,
                               d2h.cuda_stream)
        self.g += 1
        d2h.synchronize()
        main.synchronize()

    @property
    def h2d_bytes_per_step(self) -> int:
        return self.rows * self.row_bytes

    @property
    def d2h_bytes_per_step(self) -> int:
        return self.rows * self.row_bytes

    # ---- traffic model (roofline rows) ------------------------------------------------------
    def hbm_bytes_per_step(self) -> int:
        """Bytes this GPU's HBM serves per step: rows reads + rows writes of the slab, + the halo traffic.  Pull mode
        averages over the sweeps of the most recent ``step(k)`` with k > 1 (one step per sweep before any): a sweep of
        depth d reads and writes the slab once and serves the d boundary rows on each side that the neighbours pull."""
        r, b = self.rows, self.row_bytes
        if self.mode == "pull":
            sweeps = self.last_schedule
            return sum((2 * r + 2 * d) * b for d in sweeps) // sum(sweeps)
        return (2 * r + 4) * b              # + two halo rows read here + two halo rows the neighbours write here

    def nvlink_bytes_per_step(self) -> int:
        """Bytes per direction per GPU per step: one row to (or from) each neighbour."""
        return 2 * self.row_bytes

    def close(self) -> None:
        torch.cuda.synchronize(self.device)
        self.flags.close()
        self.halo.close()
        self.field.close()
        self.pads.close()


class VirtualRing:
    """``world`` HaloStencil ranks driven by ONE process: virtual ranks sharing a GPU (the cross-GPU protocol on a
    1-GPU box) or one rank per GPU of a node (single-process profiling).  ``step(k)`` enqueues k steps on every rank;
    a rank only ever waits for steps its neighbours have already been handed, so one host thread can drive them all:
    per-step launches in rank order, or — ``persistent=True`` — one k-step launch per rank on its own stream with the
    grids sized so that every CTA of every rank sharing a GPU is resident."""

    def __init__(self, world: int, message_bytes: int, rows: int, mode: str = "pull", devices: Optional[List[int]] = None,
                 alpha: float = 0.5, s: float = 0.25, tune: Optional[dict] = None, timeout_s: float = 20.0):
        from ..parallel.local import LocalGroup

        self.group = LocalGroup(world, devices)
        C = native()
        tune = dict(tune or {})
        share = max(self.group.ranks_on(d) for d in set(self.group.devices))
        if share > 1:   # co-residency of the spinning persistent kernels that share a GPU
            kind, dev = "pull" if mode == "none" else mode, self.group.devices[0]
            if tune.get("ctas"):   # a requested grid stays as long as the CTAs of every rank fit on the GPU at once
                tile_elems = (tune.get("tile_kb") or 16) * 256    # rows of HALO_MAX_CTAS tiles: the resident count
                resident = C.halo_stencil_ctas(C.HALO_MAX_CTAS * tile_elems, kind, {**tune, "ctas": 0}, dev)
                tune["ctas"] = max(1, min(tune["ctas"], resident // share))
            else:
                tune["ctas"] = max(1, C.halo_stencil_ctas(message_bytes // 4, kind, tune, dev) // share)
        fields = self.group.symmetric(2 * rows * message_bytes, zero=False)
        halos = self.group.symmetric(4 * message_bytes, zero=False)
        flags = self.group.symmetric(C.HALO_FLAG_BYTES, zero=True)
        pads = self.group.pads(timeout_s=timeout_s)
        self.ranks: List[HaloStencil] = []
        for r in range(world):
            dev = self.group.devices[r]
            with torch.cuda.device(dev):
                self.ranks.append(HaloStencil(self.group.comms[r], dev, message_bytes, rows, mode, alpha, s, tune,
                                              timeout_s, _shared={"pads": pads[r], "field": fields[r],
                                                                  "halo": halos[r], "flags": flags[r]}))
        self.streams = [torch.cuda.Stream(self.group.devices[r]) for r in range(world)]

    def step(self, steps: int = 1, persistent: bool = False) -> None:
        if persistent:
            for hs, st in zip(self.ranks, self.streams):
                with torch.cuda.device(hs.device), torch.cuda.stream(st):
                    hs.step(steps)
        else:
            for _ in range(steps):
                for hs, st in zip(self.ranks, self.streams):
                    with torch.cuda.device(hs.device), torch.cuda.stream(st):
                        hs.step(1)

    def synchronize(self) -> None:
        for st in self.streams:
            st.synchronize()
        for hs in self.ranks:
            hs.check()

    def gather(self) -> torch.Tensor:
        """The whole field [world*rows, row_elems] on the host."""
        self.synchronize()
        return torch.cat([hs.u_tensor().cpu() for hs in self.ranks], 0)

    def close(self) -> None:
        for hs in self.ranks:
            hs.close()


def main(argv: Optional[List[str]] = None) -> int:
    """``torchrun --nproc-per-node N -m hpc_patterns_b200 halo [--rows R] [--bytes B] [--steps K] [--mode pull|push]``
    — process-per-GPU twin of ``bin/halo``: same report lines (``Passed <rank>``, elapsed, bus GB/s)."""
    import argparse
    import json

    from ..utils.timing import BlockTimer

    ap = argparse.ArgumentParser(prog="halo")
    ap.add_argument("--rows", type=int, default=balanced_rows())
    ap.add_argument("--bytes", type=int, default=REFERENCE_MESSAGE_BYTES)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--mode", default="pull", choices=("pull", "push"))
    ap.add_argument("--per-step", action="store_true", help="one launch per step instead of one persistent launch")
    ap.add_argument("--stock", default=None, choices=("memcpy", "nccl"),
                    help="the reference's shape through stock calls instead: kernel; wait; library transfer; wait")
    ap.add_argument("--tile-kb", type=int, default=0)
    ap.add_argument("--stages", type=int, default=0)
    ap.add_argument("--ctas", type=int, default=0)
    ap.add_argument("--l2-hint", action="store_true", help="evict_first L2 policy on the slab's own streaming traffic")
    ap.add_argument("--depth", type=int, default=0,
                    help="pull: most steps one sweep of the slab advances (0: HPCP_HALO_DEPTH or the measured default, "
                         "1: one step per sweep)")
    ap.add_argument("--json", default=None)
    args = ap.parse_args(argv)
    comm = Comm()
    dev = comm.device
    torch.cuda.set_device(dev)
    tune = {k: v for k, v in (("tile_kb", args.tile_kb), ("stages", args.stages), ("ctas", args.ctas),
                              ("l2_hint", int(args.l2_hint)), ("depth", args.depth)) if v}
    hs = HaloStencil(comm, dev, args.bytes, args.rows, args.mode, tune=tune)
    if args.stock:
        enqueue = lambda: [hs.stock_step(args.stock) for _ in range(args.steps)]      # noqa: E731
    elif args.per_step:
        enqueue = lambda: [hs.step(1) for _ in range(args.steps)]                      # noqa: E731
    else:
        enqueue = lambda: hs.step(args.steps)                                          # noqa: E731
    m = BlockTimer(comm, hs.pads, dev).measure(enqueue, args.steps, blocks=args.iters, preheat_ms=100.0)
    bad = hs.verify_from_init()
    print(f"{'Passed' if bad == 0 else 'FAILED'} {comm.rank}" + ("" if bad == 0 else f": {bad} wrong elements"), flush=True)
    total_bad = int(comm.sum(bad))
    comm.barrier()
    if comm.rank == 0:
        bus = comm.world * 2 * args.bytes / (m["ms"] * 1e6)
        what = f"stock-{args.stock}" if args.stock else args.mode + ("/per-step" if args.per_step else "/persistent")
        print(f"Elapsed (max over ranks, min of {args.iters}): {m['ms'] * args.steps:.4f} ms for {args.steps} steps = "
              f"{m['ms']:.5f} ms/step | halo {what} P={comm.world} rows={args.rows} bytes={args.bytes} ctas={hs.ctas} "
              f"depth={hs.depth} | "
              f"{bus:.1f} GB/s P2P bus (aggregate), {bus / comm.world / 2:.1f} GB/s per GPU per direction", flush=True)
        if args.json:
            with open(args.json, "a") as f:
                f.write(json.dumps({"pattern": "halo", "variant": what, "ranks": comm.world, "rows": args.rows,
                                    "bytes": args.bytes, "steps": args.steps, "depth": hs.depth, "ms_per_step": m["ms"],
                                    "bus_GBps": bus, "per_gpu_per_dir_GBps": bus / comm.world / 2, "ctas": hs.ctas,
                                    "mismatches": total_bad}) + "\n")
    hs.close()
    comm.close()
    return 0 if total_bad == 0 else 1


if __name__ == "__main__":
    raise SystemExit(main())
