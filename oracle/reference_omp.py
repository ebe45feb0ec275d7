"""The reference's OpenMP concurrency bench as binaries under oracle/_ref/ (git-ignored; no source is copied).

    HPCP_REFERENCE=PATH_TO_HPC_PATTERNS python oracle/reference_omp.py     (__graft_entry__.build() does the same)

argonne-lcf/HPC-Patterns' GPU programs need icpx/SYCL, Level-Zero and a GPU-aware MPICH; what builds with plain
``g++ -fopenmp`` is ``concurency/main.cpp`` + ``concurency/bench_omp.cpp`` (target regions fall back to the host),
once the Intel extension ``omp_target_alloc_host`` is mapped to the standard ``omp_target_alloc`` on the command line.
The sources are compiled where they are, unmodified, in the same two builds as concurency/run_omp.sh:6-7.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from typing import Dict, Optional

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "oracle", "_ref")
MODES = {"nowait": "NOWAIT", "host_threads": "HOST_THREADS"}


def host_cxx() -> str:
    return os.environ.get("HOSTCXX") or ("/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++"))


def reference_tree() -> Optional[str]:
    """The checkout named by HPCP_REFERENCE, if it is one."""
    ref = os.environ.get("HPCP_REFERENCE")
    return ref if ref and os.path.exists(os.path.join(ref, "concurency", "main.cpp")) else None


def binary(mode: str, out: str = OUT) -> str:
    return os.path.join(out, f"omp_{mode}")


def build(ref: str, out: str = OUT) -> Dict[str, str]:
    """Compile both builds of the bench from the checkout `ref` into `out`; {mode: executable}."""
    os.makedirs(out, exist_ok=True)
    con = os.path.join(ref, "concurency")
    for mode, flag in MODES.items():
        subprocess.run([host_cxx(), "-O2", "-std=c++17", "-fopenmp", f"-D{flag}",
                        "-Domp_target_alloc_host=omp_target_alloc", os.path.join(con, "main.cpp"),
                        os.path.join(con, "bench_omp.cpp"), "-o", binary(mode, out)], check=True, timeout=900)
    return {mode: binary(mode, out) for mode in MODES}


if __name__ == "__main__":
    tree = reference_tree()
    if tree is None:
        sys.exit("set HPCP_REFERENCE to a checkout of argonne-lcf/HPC-Patterns")
    print(build(tree))
