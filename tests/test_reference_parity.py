"""Drop-in parity against the REAL reference program, through its recorded behaviour.

The reference's OpenMP backend (concurency/bench_omp.cpp + main.cpp) compiles with plain ``g++ -fopenmp``
(target regions fall back to the host) once the Intel-only ``omp_target_alloc_host`` is mapped to
``omp_target_alloc`` on the command line, sources unmodified.  ``oracle/make_golden.py`` runs that build and the
reference's ``parse.py`` on the command lines and logs below and stores exit status and stdout in
``tests/golden/reference_concurency.json.gz``; these tests replay them against ours (SURVEY.md §2.2-A):

* our binary and the reference binary print the same sequence of line shapes for the same arguments;
* the reference's own ``parse.py`` and ours render the same tables from the same logs.
"""
import gzip
import json
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_concurency.json.gz")

ARGS = ["--tripcount_C", "3000", "--commands", "C", "C"]
EXTRAS = [[], ["--verbose", "--repetitions", "3"], ["--min_bandwidth", "100000"],
          ["--queues", "1", "--verbose", "--repetitions", "2"]]
USAGE_ARGVS = [[], ["bogus_mode", "--commands", "C", "C"], ["nowait", "--bogus"], ["nowait", "--commands", "C", "X"],
               ["nowait", "--commands", "C", "H2M"]]


def run_key(binary: str, argv) -> str:
    """Key of one recorded reference run: which of its two builds (nowait / host_threads), and the argv."""
    return json.dumps([binary, list(argv)])


@pytest.fixture(scope="module")
def golden():
    with gzip.open(GOLDEN, "rt") as f:
        return json.load(f)


def _ref(golden, binary, argv):
    r = golden["runs"][run_key(binary, argv)]
    return r["rc"], r["stdout"]


def _shape(text: str):
    """Line shapes: numbers -> N, verdict text kept up to the colon (the result itself is timing-dependent)."""
    out = []
    for line in text.splitlines():
        if line.startswith("# CUDA backend unavailable"):     # our one informational extra line ('#' = comment)
            continue
        if "WARNING: Large Unbalance" in line:                 # timing-dependent in both programs
            continue
        line = re.sub(r"-?nan|\binf", "N", line)       # a 0 us measurement divides by zero in both programs
        line = re.sub(r"\d+(\.\d+)?(e[+-]?\d+)?", "N", line)
        line = re.sub(r"(SUCCESS|FAILURE): .*", "VERDICT", line)
        out.append(line)
    return out


@pytest.mark.parametrize("extra", EXTRAS)
@pytest.mark.parametrize("mode", ["host_threads", "nowait"])
def test_same_stdout_shape_as_the_reference_binary(golden, bin_dir, mode, extra):
    ref_rc, ref_out = _ref(golden, mode, [mode] + extra + ARGS)
    ours = subprocess.run([os.path.join(bin_dir, "omp_con"), mode] + extra + ARGS, capture_output=True, text=True,
                          timeout=300)
    assert "## " + mode + " | C C | " in ref_out, ref_out
    assert _shape(ours.stdout) == _shape(ref_out)
    assert ref_rc in (0, 1) and ours.returncode in (0, 1)      # 1 = some group FAILED (same rule)


def test_usage_and_exit_status_match(golden, bin_dir):
    ref_rc, ref_out = _ref(golden, "nowait", [])
    ours = subprocess.run([os.path.join(bin_dir, "omp_con")], capture_output=True, text=True)
    assert ref_rc == ours.returncode == 1
    for flag in ("--commands", "--repetitions", "--min_bandwidth", "--queues", "--enable_profiling"):
        assert flag in ref_out and flag in ours.stdout
    for bad in USAGE_ARGVS[1:4]:
        r_rc, r_out = _ref(golden, "nowait", bad)
        o = subprocess.run([os.path.join(bin_dir, "omp_con")] + bad, capture_output=True, text=True)
        assert r_rc == o.returncode == 1
        assert r_out.splitlines()[0] == o.stdout.splitlines()[0]          # same ERROR line, then the usage text
        assert r_out.splitlines()[0].startswith("ERROR: ")
    bad_rc, _ = _ref(golden, "nowait", USAGE_ARGVS[4])
    bad_ours = subprocess.run([os.path.join(bin_dir, "omp_con"), "nowait", "--commands", "C", "H2M"],
                              capture_output=True, text=True)
    assert bad_rc == bad_ours.returncode == 1              # HM / MH are rejected by both


def _our_parse(tmp_path, log: str, fmt=None):
    path = tmp_path / "in.log"
    path.write_text(log)
    mine = subprocess.run([sys.executable, "-m", "hpc_patterns_b200.utils.parse", str(path)] + ([fmt] if fmt else []),
                          capture_output=True, text=True, env=dict(os.environ, PYTHONPATH=ROOT), timeout=60)
    assert mine.returncode == 0, mine.stderr
    return mine.stdout


def test_parsers_are_interchangeable(golden, tmp_path):
    """Logs of both programs ("+ export OMP_PROC_BIND=false", then the nowait and host_threads runs of ARGS) through
    the reference's parse.py and ours."""
    assert {c["who"] for c in golden["parse_logs"]} == {"ref", "ours"}
    for case in golden["parse_logs"]:
        mine = _our_parse(tmp_path, case["log"])
        assert mine == case["stdout"] and "OMP_PROC_BIND=false" in mine, case["who"]


def test_random_command_lines_behave_like_the_reference(golden, bin_dir):
    """Random argv (valid and invalid; drawn once, with a fixed seed, by oracle/make_golden.py) through the reference
    binary and ours: same exit status, same usage-or-run decision, same sequence of line shapes.  Sizes are tiny, the
    verdict text itself is normalised away.

    Not in the alphabet on purpose: two-letter tokens with a `C` ("CC", "CM", ...) and the empty token.  The reference
    accepts them (its check is "letters from CMDH, not HM / MH", main.cpp:186-191) and then times a meaningless copy
    "from C to C" with globalsize_CC = 1, or a nameless command; here they are usage errors (DESIGN.md §6)."""
    cases = golden["random_runs"]
    assert len(cases) >= 60
    for case in cases:
        argv, ref_rc, ref_out = case["argv"], case["rc"], case["stdout"]
        ours = subprocess.run([os.path.join(bin_dir, "omp_con")] + argv, capture_output=True, text=True, timeout=120)
        ref_usage = "--commands" in ref_out and "## " not in ref_out and ref_rc == 1
        ours_usage = "--commands" in ours.stdout and "## " not in ours.stdout and ours.returncode == 1
        assert ours.returncode in (0, 1), (argv, ours.returncode, ours.stderr[-300:])                 # we never crash
        if ref_rc < 0:
            # the reference's offload allocator aborts ("Wrong Allocation") for device buffers when g++ has no offload
            # device to fall back to — an artefact of building it for the host; nothing to compare with
            continue
        assert ref_usage == ours_usage, (argv, ref_out[-300:], ours.stdout[-300:])
        if not ref_usage:
            assert (ref_rc in (0, 1)) and (ours.returncode in (0, 1)), (argv, ref_rc, ours.returncode)
            assert _shape(ours.stdout) == _shape(ref_out), (argv, ref_out, ours.stdout)


def test_random_logs_render_like_the_reference_parser(golden, tmp_path):
    """The reference's parse.py and ours print the same tables for any log a sweep script can produce (random logs
    drawn once, with a fixed seed, by oracle/make_golden.py)."""
    cases = golden["random_logs"]
    assert len(cases) >= 40
    for case in cases:
        assert _our_parse(tmp_path, case["log"], case["fmt"]) == case["stdout"], (case["log"], case["stdout"])
