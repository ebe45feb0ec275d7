"""Host-side logic of the halo-exchange flagship (no GPU): field closed form, decomposition, the step-word
protocol as a randomly scheduled model, the bench's reference arm and JSON contract."""
import json
import os
import random
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_balanced_rows_rule():
    from hpc_patterns_b200.models.halo import balanced_rows

    # pull mode: (2R + 2) rows through HBM vs 2 rows per direction over NVLink
    assert balanced_rows(6567.4, 770.0) == 7          # one direction busy
    r = balanced_rows()                               # both directions busy (what a neighbour exchange gets): default
    assert r == 8
    hbm = (2 * r + 2) / 6567.4
    nvl = 2 / 706.1
    assert abs(hbm - nvl) / nvl < 0.1
    assert balanced_rows(100.0, 1000.0) == 1            # never below one row


def test_slab_decomposition_equals_global_stencil():
    """Stepping every slab with its neighbours' boundary rows as halos IS the global periodic stencil (exactly)."""
    from hpc_patterns_b200.models.halo import initial_field, reference_steps

    world, rows, n = 3, 2, 64
    u = initial_field(world, rows, n)
    assert u.shape == (world * rows, n) and u.dtype == torch.float32
    assert float(u.min()) >= -32.0 and float(u.max()) < 32.0
    want = reference_steps(u, 4)
    slabs = [u[r * rows:(r + 1) * rows].clone() for r in range(world)]
    a, s = torch.tensor(0.5), torch.tensor(0.25)
    for _ in range(4):
        new = []
        for r in range(world):
            lo = slabs[(r - 1) % world][-1:]
            hi = slabs[(r + 1) % world][:1]
            ext = torch.cat([lo, slabs[r], hi], 0)
            new.append(a * ext[1:-1] + s * (ext[:-2] + ext[2:]))
        slabs = new
    assert torch.equal(torch.cat(slabs, 0), want)


@pytest.mark.parametrize("world,ctas,mode", [(1, 2, "pull"), (2, 3, "pull"), (4, 2, "pull"), (2, 2, "push"), (5, 1, "push")])
def test_step_word_protocol_model(world, ctas, mode):
    """Random interleaving of the kernel's rules (csrc/kernels/halo_stencil.cu): a CTA starts step g when both
    neighbour words are >= g, reads its inputs, writes its outputs, then publishes g+1 on both neighbours.
    Every read must see exactly the version the step needs, under every schedule."""
    rnd = random.Random(1234 + world * 10 + ctas)
    steps = 6
    # version of (rank, cta, parity) boundary data; in push mode the halo buffers hold the versions
    field = {(p, c, 0): 0 for p in range(world) for c in range(ctas)}
    field.update({(p, c, 1): -1 for p in range(world) for c in range(ctas)})
    halo = {(p, c, side, 0): 0 for p in range(world) for c in range(ctas) for side in ("lo", "hi")}
    halo.update({(p, c, side, 1): -1 for p in range(world) for c in range(ctas) for side in ("lo", "hi")})
    flags = {(p, side, c): 0 for p in range(world) for side in ("lo", "hi") for c in range(ctas)}
    # each CTA is a little state machine: (step, phase) with phases wait -> read -> write -> publish
    state = {(p, c): [0, "wait"] for p in range(world) for c in range(ctas)}
    reading = {}      # (rank, cta) -> set of resources currently being read
    done = 0
    guard = 0
    while done < world * ctas:
        guard += 1
        assert guard < 200000, "model deadlocked"
        p, c = rnd.randrange(world), rnd.randrange(ctas)
        g, ph = state[(p, c)]
        if g == steps:
            continue
        left, right = (p - 1) % world, (p + 1) % world
        par, out = g & 1, (g + 1) & 1
        if ph == "wait":
            if flags[(p, "lo", c)] >= g and flags[(p, "hi", c)] >= g:
                state[(p, c)][1] = "read"
        elif ph == "read":
            if mode == "pull":
                res = [("f", left, c, par), ("f", right, c, par), ("f", p, c, par)]
                for kind, q, cc, pp in res:
                    assert field[(q, cc, pp)] == g, f"rank {p} cta {c} step {g} read version {field[(q, cc, pp)]}"
            else:
                res = [("h", p, c, "lo", par), ("h", p, c, "hi", par), ("f", p, c, par)]
                assert halo[(p, c, "lo", par)] == g and halo[(p, c, "hi", par)] == g and field[(p, c, par)] == g
            reading[(p, c)] = set(res)
            state[(p, c)][1] = "write"
        elif ph == "write":
            # the writes of this step must not hit anything a neighbour is still reading
            targets = [("f", p, c, out)]
            if mode == "push":
                targets += [("h", left, c, "hi", out), ("h", right, c, "lo", out)]
            for other, rs in reading.items():
                if other != (p, c):
                    assert not (rs & set(targets)), f"WAR: rank {p} cta {c} step {g} overwrites data in use by {other}"
            field[(p, c, out)] = g + 1
            if mode == "push":
                halo[(left, c, "hi", out)] = g + 1
                halo[(right, c, "lo", out)] = g + 1
            reading.pop((p, c), None)
            state[(p, c)][1] = "publish"
        else:
            flags[(right, "lo", c)] = g + 1     # I am the left neighbour of my right neighbour
            flags[(left, "hi", c)] = g + 1
            state[(p, c)] = [g + 1, "wait"]
            if g + 1 == steps:
                done += 1
    assert all(v == steps for v in flags.values())


# Stand-in for the reference's nowait build where none exists: it accepts only the command line the reference arm was
# recorded with (tests/golden, oracle/make_golden.py) and replays that run's stdout and exit status.
_REPLAY = """import gzip, json, sys
rec = json.load(gzip.open({golden!r}, "rt"))["cpu_concurency"]
if sys.argv[1:] != rec["argv"]:
    sys.exit("not the recorded command line: %r" % sys.argv[1:])
sys.stdout.write(rec["stdout"])
sys.exit(rec["rc"])
"""


def _reference_arm_env(tmp_path):
    """Environment for bench.py's reference arm and the binary it must report: the reference's own build when there
    is one (HPCP_REFERENCE_BIN, oracle/_ref or HPCP_REFERENCE), else the recorded run."""
    from oracle import reference_omp

    env = dict(os.environ)
    if env.get("HPCP_REFERENCE_BIN"):
        return env, reference_omp.binary("nowait", env["HPCP_REFERENCE_BIN"])
    if os.path.exists(reference_omp.binary("nowait")) or reference_omp.reference_tree() is not None:
        return env, reference_omp.binary("nowait")
    stand_in = tmp_path / "omp_nowait"
    stand_in.write_text(f"#!{sys.executable}\n" +
                        _REPLAY.format(golden=os.path.join(ROOT, "tests", "golden", "reference_concurency.json.gz")))
    stand_in.chmod(0o755)
    env["HPCP_REFERENCE_BIN"] = str(tmp_path)
    return env, str(stand_in)


def test_bench_reference_arm_prints_unavailable_and_cpu_numbers(tmp_path):
    env, exe = _reference_arm_env(tmp_path)
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "2",
                        "--warmup", "1"], capture_output=True, text=True, timeout=900, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads(p.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and "unavailable" in d
    cc = d["cpu_concurency"]
    assert cc["impl"] == "reference" and cc["config"] == "cpu_concurency" and cc["groups"] == 5, cc
    assert cc["binary"] == os.path.relpath(exe, ROOT)


@pytest.mark.parametrize("impl", ["reference", "ours"])
def test_bench_cpu_concurency_config(impl, bin_dir, tmp_path):
    env = _reference_arm_env(tmp_path)[0] if impl == "reference" else None
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", impl, "--config", "cpu_concurency"],
                       capture_output=True, text=True, timeout=900, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads(p.stdout.strip().splitlines()[-1])
    assert d["impl"] == impl and d["value"] is not None and d["value"] > 0, d
    assert [g["commands"] for g in d["per_group"]] == ["C C", "C MD", "C DM", "MD DM", "HD DH"]


def test_block_timer_preheat_count_is_rank_independent():
    """The number of pre-heat blocks comes from a reduced time, so every rank enqueues the same count."""
    from hpc_patterns_b200.utils import timing

    class FakeComm:
        def barrier(self):
            pass

        def max(self, v):
            return max(v, 7.0)        # some other rank was slower

    class FakePads:
        def device_barrier(self, stream):
            pass

        def check(self):
            pass

    calls = []
    t = timing.BlockTimer.__new__(timing.BlockTimer)
    t.comm, t.pads, t.device, t.stream = FakeComm(), FakePads(), 0, None
    t.block_ms = lambda enqueue, after=None: (enqueue(), 2.0)[1]
    import unittest.mock as mock
    with mock.patch.object(timing.torch.cuda, "synchronize", lambda *_: None):
        info = t.preheat(lambda: calls.append(1), min_ms=10.0)
    assert info["blocks"] == len(calls) == 1 + 8          # (10 - 2) / 2 -> max(4, 7) -> 7 + 1


@pytest.mark.parametrize("mode", ["pull", "push"])
@pytest.mark.parametrize("ranks,rows,row_bytes,steps", [(1, 1, 64, 3), (3, 2, 4096, 5), (4, 5, 1040, 4)])
def test_native_halo_host_path_matches_torch(bin_dir, tmp_path, mode, ranks, rows, row_bytes, steps):
    """`halo --cpu`: the native program's slab decomposition, ring order and parity double-buffering without a GPU.
    Its final field (--dump) must equal a plain PyTorch fp32 run of the undecomposed periodic stencil bit for bit —
    which also pins the C++ closed-form initial field to models/halo.py::initial_field."""
    import numpy as np
    import torch
    from hpc_patterns_b200.models.halo import initial_field, reference_steps

    dump = tmp_path / "field.f32"
    iters, warmup = 2, 1
    p = subprocess.run([os.path.join(bin_dir, "halo"), "--cpu", "-n", str(ranks), "--rows", str(rows), "--bytes",
                        str(row_bytes), "--steps", str(steps), "--iters", str(iters), "--warmup", str(warmup),
                        "--mode", mode, "--dump", str(dump)], capture_output=True, text=True, timeout=120)
    assert p.returncode == 0, p.stdout + p.stderr
    assert p.stdout.count("Passed") == ranks and f"halo {mode}/host-threads P={ranks} rows={rows}" in p.stdout
    got = torch.from_numpy(np.fromfile(dump, dtype=np.float32)).reshape(ranks * rows, row_bytes // 4)
    want = reference_steps(initial_field(ranks, rows, row_bytes // 4), steps * (iters + warmup))
    assert torch.equal(got, want), float((got - want).abs().max())


def test_block_timer_order_of_operations_and_statistics(monkeypatch):
    """What made round 1's driver numbers wrong was host work between the cross-rank barrier and the start event.  The
    order in which a timed block touches the world is therefore a contract: synchronize, host barrier, DEVICE barrier
    enqueued, start event, the work, stop event, synchronize, host barrier, status check — nothing else in between;
    a measurement is the minimum over the blocks, every block is reported."""
    from hpc_patterns_b200.utils import timing

    log = []
    times = iter([8.0, 50.0, 44.0, 40.0, 42.0, 41.0])       # pre-heat block, then five timed blocks (ms per block)

    class Event:
        made = 0

        def __init__(self, enable_timing=False):
            self.name = "e0" if Event.made % 2 == 0 else "e1"      # block_ms creates the start event, then the stop event
            Event.made += 1

        def record(self, stream):
            log.append(self.name)

        def elapsed_time(self, other):
            assert (self.name, other.name) == ("e0", "e1")
            return next(times)

    class Comm:
        def barrier(self):
            log.append("host_barrier")

        def max(self, v):
            return v

    class Pads:
        def device_barrier(self, stream):
            log.append("device_barrier")

        def check(self):
            log.append("check")

    monkeypatch.setattr(timing.torch.cuda, "Event", Event)
    monkeypatch.setattr(timing.torch.cuda, "synchronize", lambda d=None: log.append("sync"))
    t = timing.BlockTimer.__new__(timing.BlockTimer)
    t.comm, t.pads, t.device = Comm(), Pads(), 0
    t.stream = type("S", (), {"cuda_stream": 0})()
    m = t.measure(lambda: log.append("work"), units=20, blocks=5, preheat_ms=4.0)
    block = ["sync", "host_barrier", "device_barrier", "e0", "work", "e1", "sync", "host_barrier", "check"]
    assert log[:len(block)] == block                                   # the pre-heat block (8 ms >= 4 ms: no repeats)
    assert log[len(block):len(block) + 3] == ["sync", "host_barrier", "check"]   # end of the pre-heat
    timed = log[len(block) + 3:]
    assert timed == block * 5
    assert m["ms"] == 2.0 and m["max_ms"] == 2.5 and m["median_ms"] == 2.1
    assert m["blocks_ms"] == [2.5, 2.2, 2.0, 2.1, 2.05] and m["spread_pct"] == 25.0
