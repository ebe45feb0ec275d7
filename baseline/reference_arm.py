"""The one part of the reference that builds in this image, run UNMODIFIED: its OpenMP concurrency bench.

argonne-lcf/HPC-Patterns has no Python package (no setup.py nor pyproject.toml), its GPU programs need icpx/SYCL,
Level-Zero and a GPU-aware MPICH, none of which a CUDA machine has — so the GPU headline has no reference arm
(``bench.py --impl reference`` says so).  What does build is BASELINE.json's config #1, "concurency/bench
compute+copy overlap on CPU host (OpenMP, no GPU)": ``concurency/main.cpp`` + ``concurency/bench_omp.cpp`` with plain
``g++ -fopenmp``, compiled from an unmodified checkout (HPCP_REFERENCE) into ``oracle/_ref`` by oracle/reference_omp.py
(``__graft_entry__.build()`` runs it when HPCP_REFERENCE is set; the binaries are git-ignored).  The run of the
reference's nowait build on ``concurency_args()`` is recorded in tests/golden/ (oracle/make_golden.py), so the tests
check this arm against it where no build of the reference exists.

Both arms run the reference's five command groups (run_omp.sh:9) through each program's stock ``main()`` and
report the same numbers, parsed from the same stdout contract (main.cpp:284-319).
"""
from __future__ import annotations

import math
import os
import re
import subprocess
from typing import Dict, List, Optional

from oracle import reference_omp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GROUPS = ["C C", "C M2D", "C D2M", "M2D D2M", "H2D D2H"]          # concurency/run_omp.sh:9
MODES = reference_omp.MODES                                        # run_omp.sh:6-7


def build_reference(mode: str = "nowait") -> Optional[str]:
    """The reference's bench for `mode`: from HPCP_REFERENCE_BIN (a directory of prebuilt omp_<mode>) if set, else
    built by build() into oracle/_ref, or built now from HPCP_REFERENCE."""
    if mode not in MODES:
        return None
    if os.environ.get("HPCP_REFERENCE_BIN"):
        exe = reference_omp.binary(mode, os.environ["HPCP_REFERENCE_BIN"])
        return exe if os.path.exists(exe) else None
    exe = reference_omp.binary(mode)
    if not os.path.exists(exe):
        tree = reference_omp.reference_tree()
        if tree is None:
            return None
        try:
            reference_omp.build(tree)
        except (OSError, subprocess.SubprocessError):
            return None
    return exe


def concurency_args(mode: str = "nowait", repetitions: int = 5, elements: int = 8_000_000,
                    tripcount: int = 40000) -> List[str]:
    """The command line (after the program name) both arms run: the five groups, every size given explicitly."""
    args = [mode, "--repetitions", str(repetitions), "--tripcount_C", str(tripcount)]
    for c in ("MD", "DM", "HD", "DH"):
        args += [f"--globalsize_{c}", str(elements)]
    for g in GROUPS:
        args += ["--commands"] + g.split()
    return args


def ours_binary() -> Optional[str]:
    exe = os.path.join(ROOT, "bin", "omp_con")
    return exe if os.path.exists(exe) else None


def _num(text: str) -> float:
    try:
        return float(text.rstrip("x"))
    except ValueError:     # "-nan", "inf": a 0 us measurement divided by itself (both programs print it)
        return float("nan")


def parse_concurency(text: str) -> List[Dict]:
    """One dict per command group from the stdout contract both programs share."""
    groups: List[Dict] = []
    cur: Dict = {}
    for line in text.splitlines():
        m = re.match(r"# (\S+) \| (.*) \| Starting Benchmarking", line)
        if m:
            cur = {"mode": m.group(1), "commands": m.group(2).strip()}
            groups.append(cur)
            continue
        m = re.search(r"Minimum Measured Total Time Serial: (\S+?)us", line)
        if m and cur is not None:
            cur["serial_us"] = _num(m.group(1))
        m = re.search(r"Minimum Measured Total Time //: (\S+?)us", line)
        if m:
            cur["concurrent_us"] = _num(m.group(1))
        m = re.search(r"Maximum Theoretical Speedup: (\S+)", line)
        if m:
            cur["max_speedup"] = _num(m.group(1))
        m = re.search(r"Speedup Relative to Serial: (\S+)", line)
        if m:
            cur["speedup"] = _num(m.group(1))
        m = re.match(r"## (\S+) \| (.*) \| (SUCCESS|FAILURE)", line)
        if m and groups:
            groups[-1]["verdict"] = m.group(3)
    return [g for g in groups if "speedup" in g]


def run_cpu_concurency(impl: str, mode: str = "nowait", repetitions: int = 5, elements: int = 8_000_000,
                       tripcount: int = 40000, threads: Optional[int] = None) -> Dict:
    """Run the five reference command groups through the stock main() of `impl` ('reference' or 'ours').

    Every tunable is given on the command line (``--tripcount_C``, ``--globalsize_<copy>``: public flags of both
    programs, main.cpp:143-196) so that neither program autotunes: on a host-only build the reference's copies
    (``#pragma omp target update``, bench_omp.cpp:83-95) are no-ops that take 0 us, its autotuner then scales every
    size to zero and the program aborts on ``omp_target_alloc(0)`` ("Wrong Allocation").  For the same reason only the
    ``C C`` group does real work in the reference arm; it is the headline of this config, the other groups are listed.
    """
    exe = build_reference(mode) if impl == "reference" else ours_binary()
    if exe is None:
        return {"impl": impl, "unavailable": "reference tree / binary not present"}
    cmd = [exe] + concurency_args(mode, repetitions, elements, tripcount)
    env = dict(os.environ)
    env["OMP_NUM_THREADS"] = str(threads or min(os.cpu_count() or 1, 8))
    env.pop("OMP_PROC_BIND", None)
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    groups = parse_concurency(p.stdout)
    cc = next((g for g in groups if g["commands"].split() == ["C", "C"]), None)
    if cc is None:
        return {"impl": impl, "unavailable": f"unexpected output (rc {p.returncode}): {p.stdout[-300:]} {p.stderr[-300:]}"}

    def num(x):
        return None if x is None or x != x or x in (float("inf"), float("-inf")) else x

    return {
        "impl": impl, "config": "cpu_concurency", "mode": mode,
        "metric": "concurency 'C C' speedup relative to serial (CPU host OpenMP; two busy-wait kernels of "
                  f"{tripcount} x 64 dependent FMAs)",
        "value": num(cc["speedup"]), "unit": "x", "higher_is_better": True,
        "cc_concurrent_us": num(cc.get("concurrent_us")), "cc_serial_us": num(cc.get("serial_us")),
        "cc_verdict": cc.get("verdict"),
        "successes": sum(1 for g in groups if g.get("verdict") == "SUCCESS"), "groups": len(groups),
        "per_group": [{"commands": g["commands"], "speedup": num(g["speedup"]),
                       "concurrent_us": num(g.get("concurrent_us")), "verdict": g.get("verdict")} for g in groups],
        "note": "host-only build: the reference's copy commands are no-op target updates (0 us), so only 'C C' "
                "compares like with like; ours executes real host memcpys for M/D/H",
        "omp_threads": int(env["OMP_NUM_THREADS"]), "repetitions": repetitions, "elements": elements,
        "binary": os.path.relpath(exe, ROOT), "rc": p.returncode,
    }
