#!/usr/bin/env python
"""Sweep the K-halo kernel's geometry (mode x tile x stages x CTAs x sweep depth) at the benchmark's shape; one JSON row
per point.

    python scripts/halo_tune.py --out gpurun_out/halo_tune.jsonl            # 1 GPU (loop-back)
    torchrun --nproc-per-node 2 scripts/halo_tune.py --out ...              # over NVLink
"""
from __future__ import annotations

import argparse
import itertools
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from hpc_patterns_b200.models.halo import REFERENCE_MESSAGE_BYTES, HaloStencil  # noqa: E402
from hpc_patterns_b200.parallel.comm import Comm  # noqa: E402
from hpc_patterns_b200.utils.timing import BlockTimer  # noqa: E402


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="gpurun_out/halo_tune.jsonl")
    ap.add_argument("--rows", type=int, nargs="+", default=[8])
    ap.add_argument("--modes", nargs="+", default=["pull", "push"])
    ap.add_argument("--geometry", nargs="+", default=["16x12", "16x8", "8x12", "8x24", "32x6", "8x13", "16x6", "4x24"],
                    help="tile_kb x stages")
    ap.add_argument("--ctas", type=int, nargs="+", default=[0])
    ap.add_argument("--l2-hint", type=int, nargs="+", default=[0], help="0: default L2 policy, 1: evict_first streaming")
    ap.add_argument("--depth", type=int, nargs="+", default=[0],
                    help="pull: most steps per sweep of the slab (0: the default, 1: one step per sweep)")
    ap.add_argument("--bytes", type=int, default=REFERENCE_MESSAGE_BYTES)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--preheat-ms", type=float, default=100.0)
    args = ap.parse_args()
    comm = Comm()
    dev = comm.device
    torch.cuda.set_device(dev)
    rows_out = []
    for rows, mode, geo, ctas, hint, depth in itertools.product(args.rows, args.modes, args.geometry, args.ctas,
                                                                 args.l2_hint, args.depth):
        tile_kb, stages = (int(x) for x in geo.split("x"))
        tune = {"tile_kb": tile_kb, "stages": stages, "l2_hint": hint, "depth": depth}
        if ctas:
            tune["ctas"] = ctas
        try:
            hs = HaloStencil(comm, dev, args.bytes, rows, mode, tune=tune)
        except Exception as e:
            if comm.rank == 0:
                print(f"skip {mode} {geo}: {e}", flush=True)
            continue
        timer = BlockTimer(comm, hs.pads, dev)
        m = timer.measure(lambda: hs.step(args.steps), args.steps, blocks=3, preheat_ms=args.preheat_ms)
        m1 = timer.measure(lambda: [hs.step(1) for _ in range(args.steps)], args.steps, blocks=3, preheat_ms=0)
        bad = int(comm.sum(hs.verify_last_step()))
        row = {"world": comm.world, "rows": rows, "mode": mode, "tile_kb": tile_kb, "stages": stages, "l2_hint": hint, "ctas": hs.ctas,
               "depth": hs.depth,
               "ms_per_step": round(m["ms"], 5), "blocks": m["blocks_ms"], "per_step_launch_ms": round(m1["ms"], 5),
               "hbm_GBps": round(hs.hbm_bytes_per_step() / m["ms"] / 1e6, 1),
               "nvlink_GBps_per_dir": round(hs.nvlink_bytes_per_step() / m["ms"] / 1e6, 1), "wrong_words": bad}
        hs.close()
        if comm.rank == 0:
            print(json.dumps(row), flush=True)
            rows_out.append(row)
    if comm.rank == 0:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "a") as f:
            for r in rows_out:
                f.write(json.dumps(r) + "\n")
    comm.close()
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
