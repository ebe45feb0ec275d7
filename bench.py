#!/usr/bin/env python
"""Flagship benchmark: slab stencil fused with its halo exchange over NVLink, ring of N B200s.

Metric (BASELINE.json): P2P bus GB/s at the reference's message size (188 743 680 B = 47 185 920 floats,
p2p/peer2pear.cpp:115-116) and compute/comm overlap %, device-timed, max over ranks, whole-job aggregate.

One step, on every rank (hpc_patterns_b200/models/halo.py, csrc/kernels/halo_stencil.cu):
    u'[r] = alpha*u[r] + s*(u[r-1] + u[r+1])      over the rank's slab of `rows` rows of one message each,
where rows -1 and `rows` are the two ring neighbours' boundary rows of the SAME step — so every step consumes what
the previous step produced on the neighbours, the dependency structure of the reference's miniapp loop
(compute; Send/Recv with both ring neighbours; swap; compute — allreduce-mpi-sycl.cpp:167-181).  The exchange is
inside the stencil kernel (pull: TMA bulk loads from the neighbours' fields; push: TMA bulk stores into their halo
buffers), K steps are ONE persistent launch, no NCCL / cudaMemcpy / host sync on the path.  Per step a rank moves one
message to (or from) each neighbour: value = N x 2 x message / time.  `rows` balances the step's HBM time against its
NVLink time, the rule of the reference's autotuner (concurency/main.cpp:219-258).  N=1: the rank is its own neighbour.

Contract: `python bench.py --gpus N --steps K --warmup W [--dump-outputs DIR]`; for N>1 launched by torchrun (one rank
per GPU).  `--dump-outputs` writes the field the timed call computes (see dump_field) for comparing two builds.
Rank 0 prints ONE JSON line.  Timing: W>=3 untimed warm-up steps, a time-based pre-heat, then `--blocks` blocks of
EXACTLY K steps, each behind an in-kernel cross-GPU barrier, CUDA events on the launching stream, max over ranks;
`value` is the best block (the reference reports the minimum over 10 iterations, peer2pear.cpp:23,52), all blocks are
listed.  `--impl reference`: the reference's GPU programs cannot be built here (no SYCL / Level-Zero / MPI) -> prints
{"impl": "reference", "unavailable": ...}; `--config cpu_concurency` runs the one part that does build (its OpenMP
concurrency bench, unmodified, baseline/reference_arm.py) for either impl.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

REFERENCE_UNAVAILABLE = ("argonne-lcf/HPC-Patterns is C++17 SYCL/OpenMP-offload/Level-Zero/MPI source with no "
                         "setup.py or pyproject.toml (pip: 'not installable'); its GPU programs need icpx + Level-Zero + "
                         "GPU-aware MPICH, none of which exists in this image.  Only its host OpenMP concurrency bench "
                         "builds (g++ -fopenmp): see the cpu_concurency field / --config cpu_concurency")
MESSAGE_BYTES = 1179648 * 40 * 4
HBM_GBS_MEASURED = 6567.4     # MEASURED_PEAKS.json hbm_gbs (copy, read+write bytes)
NVLINK_GBS_MEASURED = 770.0   # measured peer copy, ONE direction busy (B200_PROFILING.md); 900 nominal
NVLINK_BIDIR_GBS_MEASURED = 706.1   # copy engines with BOTH directions of a pair busy: 1412.2 GB/s per pair
                                    # (profiles/r2_call3_2gpu/p2p_tune.jsonl) — what a neighbour exchange can get


def measured_hbm_gbs() -> float:
    """Roofline denominator: the driver-written copy bandwidth of THIS box generation (MEASURED_PEAKS.json), the
    committed value when the file is missing or unreadable.  `rows` keeps using the committed constant so that the
    benchmark's configuration does not move with a re-measurement."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            v = float(json.load(f)["hbm_gbs"])
        return v if v > 0 else HBM_GBS_MEASURED
    except Exception:
        return HBM_GBS_MEASURED


def env_int(name: str, default: int) -> int:
    return int(os.environ.get(name, str(default)))


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=("ours", "reference"))
    ap.add_argument("--config", default="halo", choices=("halo", "cpu_concurency"))
    ap.add_argument("--bytes", type=int, default=MESSAGE_BYTES, help="one message = one row of the slab")
    ap.add_argument("--rows", type=int, default=env_int("HPCP_BENCH_ROWS", 0),
                    help="rows per slab; 0 -> balanced (HBM time = NVLink time at the measured peaks)")
    ap.add_argument("--mode", default=os.environ.get("HPCP_BENCH_MODE", "pull"), choices=("pull", "push"))
    ap.add_argument("--ctas", type=int, default=env_int("HPCP_BENCH_CTAS", 0))
    ap.add_argument("--tile-kb", type=int, default=env_int("HPCP_BENCH_TILE_KB", 0))
    ap.add_argument("--stages", type=int, default=env_int("HPCP_BENCH_STAGES", 0))
    ap.add_argument("--blocks", type=int, default=env_int("HPCP_BENCH_BLOCKS", 5))
    ap.add_argument("--preheat-ms", type=float, default=float(os.environ.get("HPCP_BENCH_PREHEAT_MS", "300")))
    ap.add_argument("--e2e-steps", type=int, default=4)
    ap.add_argument("--no-extras", action="store_true", help="skip the unfused / stock / legacy comparison runs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the field the timed call computes as DIR/field_rank<r>.npy "
                         "(float32, a fixed sample of columns when larger than DUMP_ELEMS over all ranks)")
    args = ap.parse_args()
    if args.steps < 1 or args.blocks < 1:
        ap.error("--steps and --blocks must be >= 1")
    return args


DUMP_ELEMS = 8 << 20        # float32 words over all ranks: 32 MB per dump


def dump_columns(row_elems: int, ncols: int):
    """The columns a dump keeps: the same ones in every run with the same --bytes / --gpus (seeded, sorted)."""
    import numpy as np

    if ncols >= row_elems:
        return None
    return np.sort(np.random.default_rng(0).choice(row_elems, ncols, replace=False))


def dump_field(hs, steps: int, out_dir: str) -> None:
    """What a caller of the timed path receives: this rank's slab after one ``hs.step(steps)`` call.  The call is
    replayed from the closed-form initial field (reset()), because how many steps the timed series ran depends on the
    time-based pre-heat; so runs with the same arguments get the same input and two builds compare word for word."""
    import numpy as np
    import torch

    hs.reset()
    hs.step(steps)
    u = hs.u_tensor()
    cols = dump_columns(hs.row_elems, max(1, DUMP_ELEMS // hs.world // hs.rows))
    if cols is not None:
        u = u[:, torch.from_numpy(cols).to(u.device)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"field_rank{hs.rank}.npy"), u.cpu().numpy())


def cpu_concurency(impl: str) -> dict:
    from baseline import reference_arm

    return reference_arm.run_cpu_concurency(impl)


def main() -> int:
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    if args.config == "cpu_concurency":
        if rank == 0:
            print(json.dumps(cpu_concurency(args.impl)), flush=True)
        return 0
    if args.impl == "reference":
        if rank == 0:
            out = {"impl": "reference", "unavailable": REFERENCE_UNAVAILABLE}
            try:
                out["cpu_concurency"] = cpu_concurency("reference")
            except Exception as e:  # the CPU arm is a side dish: never fail the line over it
                out["cpu_concurency"] = {"unavailable": repr(e)[:200]}
            print(json.dumps(out), flush=True)
        return 0

    import torch

    from hpc_patterns_b200.models.halo import HaloStencil, balanced_rows
    from hpc_patterns_b200.parallel.comm import Comm
    from hpc_patterns_b200.utils.clocks import ClockSampler
    from hpc_patterns_b200.utils.timing import BlockTimer

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: bench.py measures sm_100a kernels"}))
        return 1

    comm = Comm()
    world, device = comm.world, comm.device
    if world != args.gpus and comm.rank == 0:
        print(f"# note: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE", file=sys.stderr)
    torch.cuda.set_device(device)

    # Clock sampler: all the slow NVML work happens HERE, long before any timed region; it samples only while
    # resumed (a flag), and only on rank 0.
    sampler = None
    if comm.rank == 0:
        try:
            uuid = "GPU-" + str(torch.cuda.get_device_properties(device).uuid)
        except Exception:
            uuid = None
        sampler = ClockSampler(gpu_index=device, period_ms=1.0, uuid=uuid).start(paused=True)

    rows = args.rows if args.rows > 0 else balanced_rows(HBM_GBS_MEASURED, NVLINK_BIDIR_GBS_MEASURED)
    tune = {k: v for k, v in (("ctas", args.ctas), ("tile_kb", args.tile_kb), ("stages", args.stages)) if v}
    K, W = args.steps, max(args.warmup, 3)
    hs = HaloStencil(comm, device, args.bytes, rows, args.mode, tune=tune)
    timer = BlockTimer(comm, hs.pads, device)

    # ---- correctness first: W steps from the closed-form initial field, every word of the slab checked ----------
    hs.step(W)
    wrong_init = int(comm.sum(hs.verify_from_init()))
    hs.check()

    # ---- the headline: K steps = ONE persistent launch, exchange inside -----------------------------------------
    if sampler is not None:
        sampler.resume()
    launches0 = hs.launches
    fused = timer.measure(lambda: hs.step(K), K, blocks=args.blocks, preheat_ms=args.preheat_ms,
                          warmup=lambda: hs.step(W))
    if sampler is not None:
        sampler.pause()
    gpu_launches_per_block = 1          # ONE persistent K-halo launch runs all K steps of a timed block (the in-kernel
                                        # barrier is enqueued before the start event, i.e. outside the region)
    total_fused_launches = hs.launches - launches0
    wrong_last = int(comm.sum(hs.verify_last_step()))
    if args.dump_outputs:
        dump_field(hs, K, args.dump_outputs)
    ms_per_step = fused["ms"]
    msg = args.bytes
    value = world * 2 * msg / (ms_per_step * 1e-3) / 1e9          # aggregate GB/s over all GPUs, both neighbours
    per_gpu_dir = msg * 2 / (ms_per_step * 1e-3) / 1e9            # per GPU per direction
    hbm_peak = measured_hbm_gbs()
    hbm_ms = hs.hbm_bytes_per_step() / hbm_peak / 1e6
    nvl_ms = (hs.nvlink_bytes_per_step() / NVLINK_BIDIR_GBS_MEASURED / 1e6) if world > 1 else 0.0
    roof_ms = max(hbm_ms, nvl_ms)

    extras = {}
    if not args.no_extras:
        pre = min(args.preheat_ms, 150.0)
        k = max(5, min(K, 20))
        # one launch per step (same kernel, the step words carry the dependency across launches)
        per_launch = timer.measure(lambda: [hs.step(1) for _ in range(k)], k, blocks=3, preheat_ms=pre)
        # the stencil kernel alone (no exchange) and the exchange alone (stand-alone put kernels + arrival waits)
        t_compute = timer.measure(lambda: [hs.compute_only() for _ in range(k)], k, blocks=3, preheat_ms=pre)
        t_xchg = timer.measure(lambda: [hs.exchange_only() for _ in range(k)], k, blocks=3, preheat_ms=pre)
        # the reference's loop shape through stock calls — first-class numbers, same harness
        hs.reset()
        stock_mc = timer.measure(lambda: [hs.stock_step("memcpy") for _ in range(k)], k, blocks=args.blocks,
                                 preheat_ms=pre)
        wrong_stock = int(comm.sum(hs.verify_last_step()))
        stock_nccl = None
        if world > 1:
            try:
                stock_nccl = timer.measure(lambda: [hs.stock_step("nccl") for _ in range(k)], k, blocks=args.blocks,
                                           preheat_ms=pre)
                wrong_stock += int(comm.sum(hs.verify_last_step()))
            except Exception as e:  # NCCL is only a comparison row
                extras["nccl_error"] = repr(e)[:200]
        stock_nowait = timer.measure(lambda: [hs.stock_step("memcpy", host_wait=False) for _ in range(k)], k, blocks=3,
                                     preheat_ms=0)
        # share of the shorter piece that the fused step hides; the raw value exceeds 100 when the fused kernel is also
        # faster than the LONGER piece run alone (N=8: the stand-alone exchange to two different peers takes 0.71 ms)
        overlap_raw = (t_compute["ms"] + t_xchg["ms"] - ms_per_step) / min(t_compute["ms"], t_xchg["ms"]) * 100.0
        overlap = min(overlap_raw, 100.0)
        extras.update({
            "overlap_pct": round(overlap, 1), "overlap_pct_uncapped": round(overlap_raw, 1),
            "unfused_compute_ms": round(t_compute["ms"], 4), "unfused_exchange_ms": round(t_xchg["ms"], 4),
            "one_launch_per_step_ms": round(per_launch["ms"], 4),
            "stock": {
                "shape": "stencil kernel; host wait; library transfer of both boundary rows; host wait "
                         "(allreduce-mpi-sycl.cpp:176-181)",
                "memcpy_ms": round(stock_mc["ms"], 4), "memcpy_blocks_ms": stock_mc["blocks_ms"],
                "nccl_sendrecv_ms": None if stock_nccl is None else round(stock_nccl["ms"], 4),
                "nccl_blocks_ms": None if stock_nccl is None else stock_nccl["blocks_ms"],
                "memcpy_no_host_wait_ms": round(stock_nowait["ms"], 4),
                "preheat_ms": stock_mc["preheat_ms"], "wrong_words": wrong_stock,
            },
            "speedup_vs_stock_memcpy": round(stock_mc["ms"] / ms_per_step, 3),
            "speedup_vs_stock_nccl": None if stock_nccl is None else round(stock_nccl["ms"] / ms_per_step, 3),
        })
        # rows = 1: everything that is computed is exchanged -> NVLink-bound at N >= 2 (the wire-rate number)
        if rows != 1:
            hs1 = HaloStencil(comm, device, args.bytes, 1, args.mode, tune=tune)
            t1 = BlockTimer(comm, hs1.pads, device).measure(lambda: hs1.step(K), K, blocks=3, preheat_ms=pre)
            bad1 = int(comm.sum(hs1.verify_last_step()))
            extras["rows_1"] = {"ms_per_step": round(t1["ms"], 5),
                                "per_gpu_per_direction_GBps": round(2 * msg / (t1["ms"] * 1e-3) / 1e9, 1),
                                "frac_of_nvlink_770_measured": round(2 * msg / (t1["ms"] * 1e-3) / 1e9 / 770.0, 3)
                                if world > 1 else None,
                                "wrong_words": bad1}
            hs1.close()
        # round-1 flagship (unidirectional ring put of a triad, no dependency between steps) under THIS harness
        try:
            from hpc_patterns_b200.models.peer2pear import FusedTriadExchange

            legacy = {}
            for ratio in (3, 1):
                ex = FusedTriadExchange(comm, device, args.bytes, s=3.0, engine="tma", compute_ratio=ratio)
                tl = BlockTimer(comm, ex.pads, device).measure(lambda: [ex.step() for _ in range(k)], k, blocks=3,
                                                               preheat_ms=pre)
                legacy[f"ratio_{ratio}"] = {"ms_per_step": round(tl["ms"], 5), "blocks_ms": tl["blocks_ms"],
                                            "wrong_words": int(comm.sum(ex.verify()))}
                ex.close()
            extras["legacy_triad_ring_put"] = legacy
        except Exception as e:
            extras["legacy_error"] = repr(e)[:200]

    clocks = sampler.stop() if sampler is not None else None
    hs.close()

    # ---- end to end through the public API: the slab lives in pinned host memory --------------------------------
    he = HaloStencil(comm, device, args.bytes, rows, "push", tune=tune)
    bufs = he.make_host_buffers()
    for i in range(2):
        he.step_from_host(bufs[i & 1], bufs[(i + 1) & 1])
    torch.cuda.synchronize(device)
    comm.barrier()
    t0 = time.perf_counter()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    stream = torch.cuda.current_stream(device)
    e0.record(stream)
    for i in range(args.e2e_steps):
        he.step_from_host(bufs[i & 1], bufs[(i + 1) & 1])      # returns when the new slab is in host memory
    e1.record(stream)
    torch.cuda.synchronize(device)
    comm.barrier()
    e2e_wall_ms = comm.max((time.perf_counter() - t0) * 1e3)
    e2e_ms = max(comm.max(e0.elapsed_time(e1)), e2e_wall_ms) / max(args.e2e_steps, 1)
    e2e_value = world * 2 * msg / (e2e_ms * 1e-3) / 1e9
    e2e_bad = he.verify_from_init()
    host_final = bufs[args.e2e_steps & 1]
    e2e_bad += int((host_final != he.u_tensor().cpu()).sum().item())    # what the caller holds == the device field
    e2e_bad = int(comm.sum(e2e_bad))
    he.check()
    h2d, d2h = he.h2d_bytes_per_step, he.d2h_bytes_per_step
    he.close()

    if comm.rank == 0:
        out = {
            "impl": "ours",
            "metric": "p2p_bus_GBps (slab stencil fused with its halo exchange: one 188743680 B message to/from each "
                      "ring neighbour per step, aggregate over GPUs)",
            "value": round(value, 2), "unit": "GB/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": round(ms_per_step, 5),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp32", "data": "synthetic",
            "config": {
                "model": "aurora.mpich miniapp loop as a halo exchange: 3-point slab stencil + exchange with both "
                         "ring neighbours, fused (K-halo)",
                "global_batch": world, "seq_len": msg // 4, "parallelism": f"ring{world}",
                "message_bytes": msg, "messages_per_step_per_gpu": 2, "rows": rows, "mode": args.mode,
                "ctas": hs.ctas, "steps_per_launch": K,
                "rows_rule": "rows such that the step's HBM time ~ its NVLink time at stock measured rates (HBM copy "
                             "6567 GB/s; copy engines with both directions busy 706 GB/s/dir) — the balancing rule of "
                             "the reference's autotuner",
                "peer": "self (no NVLink at N=1)" if world == 1 else "rank-1 and rank+1 over NVLink/NVSwitch",
                "l2": f"inputs larger than L2: {(2 * rows + 2)} x 180 MiB streamed per step, no reuse between steps",
                "timing": "in-kernel cross-GPU barrier, then cuda events on the launching stream; max over ranks; "
                          "best of `blocks` blocks of exactly `steps` steps after a time-based pre-heat",
                "note": "fp32 is the reference's dtype (APP_DATA_TYPE float); bytes moved, not FLOPs, are the metric",
            },
            "blocks_ms_per_step": fused["blocks_ms"], "median_ms_per_step": round(fused["median_ms"], 5),
            "spread_pct": fused["spread_pct"], "preheat_ms": fused["preheat_ms"],
            "clocks": clocks or {"sm_mhz": None, "sm_max_mhz": None, "reasons": []},
            "e2e": {"value": round(e2e_value, 2), "unit": "GB/s", "ms_per_step": round(e2e_ms, 4),
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "pcie_GBps_per_gpu_each_way": round(h2d / (e2e_ms * 1e-3) / 1e9, 1),
                    "steps": args.e2e_steps, "wrong_words": e2e_bad, "mode": "push",
                    "what": "out-of-core step: the WHOLE slab is uploaded from pinned host memory, stepped with the "
                            "NVLink exchange, and the WHOLE new slab is downloaded, every step",
                    "api": "hpc_patterns_b200.models.halo.HaloStencil.step_from_host"},
            "gpu_launches": gpu_launches_per_block, "gpu_launches_all_blocks": total_fused_launches,
            "gpu_launches_note": "halo_stencil_kernel<pull|push>: K steps per launch (config.steps_per_launch); "
                                 "one_launch_per_step_ms is the same kernel launched K times",
            "wrong_words": wrong_init + wrong_last,
            "per_gpu_per_direction_GBps": round(per_gpu_dir, 1),
            "frac_of_nvlink_706_measured_bidirectional": round(per_gpu_dir / NVLINK_BIDIR_GBS_MEASURED, 3) if world > 1 else None,
            "frac_of_nvlink_770_measured": round(per_gpu_dir / 770.0, 3) if world > 1 else None,
            "frac_of_nvlink_900_nominal": round(per_gpu_dir / 900.0, 3) if world > 1 else None,
            "hbm_traffic_GBps": round(hs.hbm_bytes_per_step() / (ms_per_step * 1e-3) / 1e9, 1),
            "roofline": {"hbm_ms": round(hbm_ms, 4), "nvlink_ms": round(nvl_ms, 4), "bound_ms": round(roof_ms, 4),
                         "frac": round(roof_ms / ms_per_step, 3),
                         "hbm_gbs": hbm_peak, "nvlink_gbs_per_dir": NVLINK_BIDIR_GBS_MEASURED,
                         "of": "max(HBM bytes / MEASURED_PEAKS.json hbm_gbs (copy peak), NVLink bytes per direction / "
                               "706.1 GB/s measured with both directions busy)"},
            **extras,
        }
        if not args.no_extras:
            try:
                out["cpu_concurency"] = cpu_concurency("ours")
            except Exception as e:
                out["cpu_concurency"] = {"unavailable": repr(e)[:200]}
        print(json.dumps(out), flush=True)
    comm.close()
    return 0 if (wrong_init + wrong_last == 0 and e2e_bad == 0) else 1


if __name__ == "__main__":
    sys.exit(main())
