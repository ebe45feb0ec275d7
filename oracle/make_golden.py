"""Record the reference's concurrency bench and log parser as tests/golden/reference_concurency.json.gz.

    python oracle/make_golden.py PATH_TO_HPC_PATTERNS [--out FILE]

Needs a checkout of argonne-lcf/HPC-Patterns, g++ with OpenMP, ``tabulate``, and this project built (``bin/omp_con``
is run for the "ours" log of the parser check).  The reference's OpenMP bench is compiled from its unmodified sources
into a temporary directory by oracle/reference_omp.py.  Every
command line and log that tests/test_reference_parity.py replays is run through it and through the reference's
``concurency/parse.py``; exit status and stdout are stored.  Random command lines and logs are drawn from a fixed seed.
The run of the reference arm of bench.py (baseline/reference_arm.py: concurency_args) is stored the same way.
"""
from __future__ import annotations

import argparse
import gzip
import json
import os
import random
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from baseline.reference_arm import concurency_args  # noqa: E402
from oracle.reference_omp import MODES, build  # noqa: E402
from tests.test_reference_parity import ARGS, EXTRAS, GOLDEN, USAGE_ARGVS, run_key  # noqa: E402

SEED = 20260917
RANDOM_RUNS = 160
RANDOM_LOGS = 60

# command-line alphabet of the random runs
TOKENS = ["C", "M2D", "D2M", "MD", "DM", "H2D", "D2H", "HD", "DH", "C2", "2C", "M2D2", "HM", "MH", "X", "M2X"]
FLAGS = [["--verbose"], ["--enable_profiling"], ["--queues", "1"], ["--queues", "2"], ["--repetitions", "1"],
         ["--min_bandwidth", "0.000001"], ["--bogus"], ["-x"], ["--tripcount_C", "7"], ["--globalsize_C", "2"]]
RUN_MODES = ["nowait", "host_threads", "serial", "in_order", ""]

# line alphabet of the random logs
LOG_MODES = ["nowait", "host_threads", "in_order", "out_of_order", "fused", "serial"]
LOG_CMDS = ["C", "MD", "DM", "HD", "DH", "DP", "A", "T"]
VERDICTS = ["SUCCESS: Close from Theoretical Speedup", "FAILURE: Far from Theoretical Speedup",
            "FAILURE: Minimun Bandwish not reached"]
EXPORTS = ["CUDA_VISIBLE_DEVICES=0", "HPCP_FUSED_COPY_ENGINE=1", "OMP_PROC_BIND=false", "CUDA_DEVICE_MAX_CONNECTIONS=32",
           "A=1 B=2"]
NOISE = ["# nowait | C MD | Starting Benchmarking...", "Minimum Measured Total Time Serial: 12us",
         "  Minimum Time Command 0 (  C): 7us", "Speedup Relative to Serial: 1.9x", "", "Parameters used:",
         "  tripcount_C: 40000", "+ ./omp_con nowait --commands C M2D"]


def random_argv(rng: random.Random) -> list:
    mode = rng.choice(RUN_MODES)
    argv = [mode] if mode else []
    for _ in range(rng.randint(0, 3)):
        argv += rng.choice(FLAGS)
    argv += ["--globalsize_default_memory", "2000", "--tripcount_C", "50", "--repetitions", "2"]
    for cmd in ("MD", "DM", "HD", "DH"):       # explicit sizes: no autotuning, whose result depends on 0 us timings
        argv += ["--globalsize_" + cmd, "2000"]
    for _ in range(rng.randint(0, 3)):
        argv += ["--commands"] + [rng.choice(TOKENS) for _ in range(rng.randint(0, 3))]
    return argv


def random_log_line(rng: random.Random) -> str:
    kind = rng.choice(["verdict", "verdict", "export", "noise"])
    if kind == "verdict":
        cmds = " ".join(rng.choice(LOG_CMDS) for _ in range(rng.randint(1, 3)))
        return f"## {rng.choice(LOG_MODES)} | {cmds} | {rng.choice(VERDICTS)}"
    if kind == "export":
        return "+ export " + " ".join(rng.choice(EXPORTS) for _ in range(rng.randint(1, 2)))
    return rng.choice(NOISE)


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("reference", help="checkout of argonne-lcf/HPC-Patterns")
    ap.add_argument("--out", default=GOLDEN)
    args = ap.parse_args()
    parse_py = os.path.join(args.reference, "concurency", "parse.py")
    ours = os.path.join(ROOT, "bin", "omp_con")
    tmp = tempfile.mkdtemp(prefix="hpcp_golden_")
    try:
        bins = build(args.reference, tmp)

        def run(binary, argv):
            p = subprocess.run([bins[binary]] + argv, capture_output=True, text=True, timeout=300)
            return {"rc": p.returncode, "stdout": p.stdout}

        def ref_parse(log, fmt=None):
            path = os.path.join(tmp, "in.log")
            with open(path, "w") as f:
                f.write(log)
            p = subprocess.run([sys.executable, parse_py, path] + ([fmt] if fmt else []), capture_output=True,
                               text=True, timeout=60, check=True)
            return p.stdout

        runs = {}
        for mode in MODES:
            for extra in EXTRAS:
                argv = [mode] + extra + ARGS
                runs[run_key(mode, argv)] = run(mode, argv)
        for argv in USAGE_ARGVS:
            runs[run_key("nowait", argv)] = run("nowait", argv)

        # what bench.py --impl reference --config cpu_concurency runs (baseline/reference_arm.py)
        cpu_concurency = {"argv": concurency_args(), **run("nowait", concurency_args())}

        parse_logs = []
        for who in ("ref", "ours"):
            log = "+ export OMP_PROC_BIND=false\n"
            for mode in ("nowait", "host_threads"):
                exe = bins[mode] if who == "ref" else ours
                log += subprocess.run([exe, mode] + ARGS, capture_output=True, text=True, timeout=300).stdout
            parse_logs.append({"who": who, "log": log, "stdout": ref_parse(log)})

        rng = random.Random(SEED)
        random_runs = []
        for _ in range(RANDOM_RUNS):
            argv = random_argv(rng)
            binary = argv[0] if argv and argv[0] in MODES else "nowait"
            random_runs.append({"argv": argv, **run(binary, argv)})
        random_logs = []
        for _ in range(RANDOM_LOGS):
            log = "\n".join(random_log_line(rng) for _ in range(rng.randint(0, 25))) + "\n"
            fmt = rng.choice(["simple", "github", "plain"])
            random_logs.append({"log": log, "fmt": fmt, "stdout": ref_parse(log, fmt)})
    finally:
        shutil.rmtree(tmp, ignore_errors=True)

    golden = {"about": "argonne-lcf/HPC-Patterns concurency: OpenMP bench (host build) and parse.py, recorded by "
                       "oracle/make_golden.py",
              "runs": runs, "cpu_concurency": cpu_concurency, "parse_logs": parse_logs, "random_runs": random_runs, "random_logs": random_logs}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with gzip.GzipFile(args.out, "wb", mtime=0) as f:       # mtime 0: the same records give the same bytes
        f.write(json.dumps(golden, indent=0, sort_keys=True).encode() + b"\n")
    print(f"wrote {args.out}: {len(runs)} runs, {len(random_runs)} random runs, {len(random_logs)} random logs")
    return 0


if __name__ == "__main__":
    sys.exit(main())
