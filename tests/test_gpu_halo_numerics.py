"""K-halo numerics where a wrong kernel could still match the plain fp32 reference (csrc/kernels/halo_stencil.cu).

Every fused step must equal ``reference_steps`` (PyTorch fp32, one rounding per operation) bit for bit.  At the
suite's usual coefficients (alpha = 0.5, s = 0.25) the products ``alpha*u`` and ``s*(up + dn)`` are exact, so an FMA
contraction of either product, or ``s*up + s*dn``, gives the same bits as the correct expression.  The cases here run
at ALPHA, S instead, where every one of those forms changes many words (checked on the CPU below).  They cover the
three kernels (pull at depth 3 and 1, push), CTAs that own several column tiles next to real neighbours, the deep
kernel at edge geometries, every sweep schedule up to 12 steps, and the two device checkers, which must count exactly
what is wrong.

CPU cases: the coefficient sensitivity, and the executable model of the deep kernel's shared-memory ring
(tests/test_halo_sweep.py) over every deep geometry below, so that a slot-rule error shows up as a ProtocolError here
and not as a stalled CTA on a GPU.  The GPU cases use one B200 and virtual ranks (VirtualRing).
"""
from __future__ import annotations

import functools
import json
import os
import subprocess
import sys
from typing import NamedTuple

import pytest
import torch

from hpc_patterns_b200.models.halo import initial_field, reference_steps, sweep_depth, sweep_schedule
from tests.test_halo_sweep import simulate

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

ALPHA, S = 0.3, 0.35          # neither is a power of two: alpha*u and s*(up + dn) round; alpha + 2s = 1 keeps it bounded
KB = 1024
TILE = 16 * KB
RAGGED = 4 * TILE + 1040      # five 16 KiB column tiles, the last one 65 float4: fewer than the 96 math threads
TWELVE = 11 * TILE + 16       # twelve column tiles, the last one a single float4
SWEEP_DEPTH = 3               # the one deep instantiation, halo_sweep_kernel<3>


class Geometry(NamedTuple):
    world: int
    rows: int
    message: int              # bytes of one row
    tile_kb: int = 16
    stages: int = 6
    ctas: int = 0             # 0: VirtualRing's default grid

    @property
    def tune(self) -> dict:
        tune = {"tile_kb": self.tile_kb, "stages": self.stages, "depth": 0}   # depth 0: the default, whatever the env
        return {**tune, "ctas": self.ctas} if self.ctas else tune

    @property
    def tiles(self) -> int:
        return -(-self.message // (self.tile_kb * KB))

    @property
    def grid(self) -> int:
        """CTAs per rank.  Every geometry here has at most 148 tiles, and every SM holds at least one CTA, so residency
        never binds: one rank gets one CTA per tile; ranks sharing the GPU split the tiles unless a grid is requested."""
        if self.ctas:
            return min(self.ctas, self.tiles)
        return self.tiles if self.world == 1 else max(1, self.tiles // self.world)

    @property
    def columns(self) -> int:
        """Most column tiles one CTA owns."""
        return -(-self.tiles // self.grid)

    @property
    def depth(self) -> int:
        """Deepest sweep of a persistent pull launch."""
        return sweep_depth(self.rows, "pull", self.tune)

    def __str__(self) -> str:
        extra = f"-ctas{self.ctas}" if self.ctas else ""
        return f"w{self.world}-r{self.rows}-{self.message}B-t{self.tile_kb}-s{self.stages}{extra}"


# ---- the table: every geometry and launch the GPU cases run --------------------------------------------------------

KERNELS = {"pull": ("pull", {}), "pull-depth1": ("pull", {"depth": 1}), "push": ("push", {})}
SERIES = ((1, False), (7, True), (1, False), (4, True))      # (steps, persistent): per-step, deep, per-step, deep

# 1. the three kernels at rounding coefficients
ROUNDING = [Geometry(1, 3, RAGGED), Geometry(2, 4, RAGGED), Geometry(3, 5, RAGGED), Geometry(4, 8, RAGGED)]
# 2. several column tiles per CTA with neighbours; 5 CTAs over 12 tiles own 3 or 2 columns
MULTI_COLUMN = [Geometry(w, 5, TWELVE, ctas=c) for w in (2, 3, 4) for c in (1, 2, 5)]
# 3. deep-kernel geometry, (geometry, K): each runs persistent step(K), step(1), persistent step(K).  Messages: one
#    float4, shorter than a tile, n tiles, n tiles + 16 B, n tiles + 1 KiB (64 float4 in the last tile for 4, 12 and
#    16 KiB tiles).  12 KiB tiles are not a power of two; 32 KiB tiles fall back to depth 1.
DEEP = [
    (Geometry(1, 8, 16), 4),
    (Geometry(3, 16, 16, stages=7), 7),
    (Geometry(1, 32, 16, tile_kb=4, stages=13), 13),
    (Geometry(3, 3, 16, tile_kb=12), 8),
    (Geometry(1, 3, 4 * KB), 5),
    (Geometry(3, 3, 4 * KB, tile_kb=4), 20),
    (Geometry(1, 16, 4 * KB, tile_kb=12, stages=13), 9),
    (Geometry(3, 32, 4 * KB), 6),
    (Geometry(1, 3, 2 * TILE), 11),
    (Geometry(3, 16, 2 * TILE, tile_kb=12, stages=7), 4),
    (Geometry(1, 32, 5 * TILE, tile_kb=4, stages=7), 8),
    (Geometry(3, 3, 5 * TILE, stages=13), 12),
    (Geometry(1, 3, 3 * TILE + 16, stages=7), 10),
    (Geometry(3, 16, 3 * TILE + 16, tile_kb=4, stages=13), 7),
    (Geometry(1, 16, 5 * TILE + 16, tile_kb=12, ctas=2), 20),
    (Geometry(3, 32, 2 * TILE + 16), 5),
    (Geometry(1, 3, 3 * TILE + KB, tile_kb=12), 4),
    (Geometry(3, 3, 3 * TILE + KB), 13),
    (Geometry(1, 16, 3 * TILE + KB, stages=13), 6),
    (Geometry(3, 16, 3 * TILE + KB, tile_kb=4, ctas=5), 9),
    (Geometry(1, 32, 3 * TILE + KB, stages=7), 20),
    (Geometry(3, 32, 3 * TILE + KB, tile_kb=12, stages=13), 11),
    (Geometry(3, 3, 7 * TILE + KB, stages=7, ctas=3), 16),
    (Geometry(1, 8, 3 * TILE + KB, tile_kb=32), 7),
    (Geometry(3, 4, 4 * TILE + 16, tile_kb=32), 5),
]
# 4. every schedule, 5. the checkers: an odd ring, a ragged row
SCHEDULE = Geometry(3, 4, RAGGED)
SCHEDULE_STEPS = range(1, 13)
CHECKER = Geometry(3, 4, RAGGED)
CHECKER_ROW_LIMIT = Geometry(2, 64, 2 * TILE + 16)            # world * rows = 128, the limit of verify_from_init
# 6. bench.py's own run: 24 MiB + 16 B rows, 8 rows, 20 steps, at its grid of 2 CTAs on each of 148 SMs
BENCH_ARGS = ["--bytes", "25165840", "--rows", "8", "--steps", "20", "--warmup", "3", "--no-extras", "--e2e-steps", "1",
              "--blocks", "1", "--preheat-ms", "20"]
BENCH = Geometry(1, 8, 25165840)
BENCH_COLUMNS = -(-BENCH.tiles // (2 * 148))


def deep_launches() -> list:
    """(rows, stages, most columns per CTA, K) of every persistent launch above that runs halo_sweep_kernel."""
    launches = set()
    for g in ROUNDING + MULTI_COLUMN:
        launches.update((g.rows, g.stages, g.columns, k) for k, persistent in SERIES if persistent)
    launches.update((g.rows, g.stages, g.columns, k) for g, k in DEEP if g.depth == SWEEP_DEPTH)
    launches.update((SCHEDULE.rows, SCHEDULE.stages, SCHEDULE.columns, k) for k in SCHEDULE_STEPS)
    launches.update([(CHECKER.rows, CHECKER.stages, CHECKER.columns, 7),
                     (CHECKER_ROW_LIMIT.rows, CHECKER_ROW_LIMIT.stages, CHECKER_ROW_LIMIT.columns, 7),
                     (BENCH.rows, BENCH.stages, BENCH_COLUMNS, 20)])
    return sorted(launch for launch in launches if max(sweep_schedule(launch[3], SWEEP_DEPTH)) > 1)


def compared_fields() -> list:
    """(world, rows, row_elems, steps) of every field a GPU case compares with the reference at rounding coefficients."""
    fields = set()

    def series(g, calls):
        done = 0
        for k in calls:
            done += k
            fields.add((g.world, g.rows, g.message // 4, done))

    for g in ROUNDING + MULTI_COLUMN:
        series(g, [k for k, _ in SERIES])
    for g, k in DEEP:
        series(g, [k, 1, k])
    for k in SCHEDULE_STEPS:
        series(SCHEDULE, [k])
        series(SCHEDULE, [1, k])
    series(CHECKER, [7])
    series(CHECKER_ROW_LIMIT, [7])
    return sorted(fields)


# ---- CPU: the coefficients must expose a wrong rounding ------------------------------------------------------------

def wrong_stencils(alpha: float, s: float) -> dict:
    """Four plausible ways to compile the step wrongly.  FMAs are emulated in fp64: the product of two floats is exact
    there, so only the final rounding to fp32 differs from a true FMA (and only in rare double-rounding ties)."""
    a = torch.tensor(alpha, dtype=torch.float32)
    b = torch.tensor(s, dtype=torch.float32)

    def fma(x, y, z):
        return (x.double() * y.double() + z.double()).float()

    return {
        "fma(alpha, u, s*(up+dn))": lambda u, up, dn: fma(a, u, b * (up + dn)),
        "fma(s, up+dn, alpha*u)": lambda u, up, dn: fma(b, up + dn, a * u),
        "alpha*u + (s*up + s*dn)": lambda u, up, dn: a * u + (b * up + b * dn),
        "(alpha*u + s*up) + s*dn": lambda u, up, dn: (a * u + b * up) + b * dn,
    }


def run_stencil(step, field: torch.Tensor, steps: int) -> torch.Tensor:
    u = field.clone()
    for _ in range(steps):
        u = step(u, torch.roll(u, 1, 0), torch.roll(u, -1, 0))
    return u


def test_power_of_two_coefficients_hide_contraction():
    """Why the cases here do not run at the usual 0.5 / 0.25: there, both FMA contractions and the split product give
    the correct bits on every word (world 2, 4 rows, 4096 columns, 20 steps); only re-associating the sum shows."""
    field = initial_field(2, 4, 4096)
    want = reference_steps(field, 20, 0.5, 0.25)
    wrong = {name: int((run_stencil(step, field, 20) != want).sum()) for name, step in wrong_stencils(0.5, 0.25).items()}
    assert wrong == {"fma(alpha, u, s*(up+dn))": 0, "fma(s, up+dn, alpha*u)": 0, "alpha*u + (s*up + s*dn)": 0,
                     "(alpha*u + s*up) + s*dn": 15896}


@pytest.mark.parametrize("world,rows,row_elems", sorted({f[:3] for f in compared_fields()}))
def test_rounding_coefficients_expose_every_wrong_form(world, rows, row_elems):
    """At ALPHA, S every wrong form changes many words of every field a GPU case compares, at every step count."""
    steps = sorted(f[3] for f in compared_fields() if f[:3] == (world, rows, row_elems))
    field = initial_field(world, rows, row_elems)
    for name, step in wrong_stencils(ALPHA, S).items():
        want, got, done = field, field, 0
        for k in steps:
            want = reference_steps(want, k - done, ALPHA, S)
            got = run_stencil(step, got, k - done)
            done = k
            wrong = int((got != want).sum())
            assert wrong >= field.numel() // 5, (name, k, wrong, field.numel())


# ---- CPU: the ring model over every deep geometry ------------------------------------------------------------------

@functools.lru_cache(maxsize=None)
def model_passes(rows: int, stages: int, columns: int, steps: int, seeds: int = 1) -> bool:
    """The sweep kernel's slot rules (tests/test_halo_sweep.py) for this geometry: raises ProtocolError on a rule
    error, under random completion orders with and without slow stores."""
    schedule = sweep_schedule(steps, SWEEP_DEPTH)
    for seed in range(seeds):
        for store_delay in (0, 3):
            assert simulate(stages, rows, columns, schedule, seed, store_delay=store_delay) == \
                len(schedule) * rows * columns
    return True


def test_tables_reach_every_edge():
    """The deep table reaches every edge it is meant to: message shapes, tiles, stages, rows, worlds, several columns
    per CTA, and one global row-count limit."""
    deep = [g for g, _ in DEEP]
    assert {g.tile_kb for g in deep} == {4, 12, 16, 32} and {g.stages for g in deep} == {6, 7, 13}
    assert {g.rows for g in deep} >= {3, 16, 32} and {g.world for g in deep} == {1, 3}
    assert all(g.world * g.rows <= 128 for g in deep) and all(g.tiles <= 148 for g in deep)
    tails = {(g.message % (g.tile_kb * KB)) or g.tile_kb * KB for g in deep if g.tile_kb <= 16}
    assert {16, 4 * KB, KB} <= tails and 16 in {g.message for g in deep}
    assert any(g.message < g.tile_kb * KB for g in deep if g.message > 16)
    assert any(g.columns > 1 and g.world > 1 for g in deep) and any(g.columns > 1 and g.world == 1 for g in deep)
    assert all(g.depth == (1 if g.tile_kb > 16 else SWEEP_DEPTH) for g in deep)
    assert {g.columns for g in MULTI_COLUMN} >= {12, 6, 3} and CHECKER_ROW_LIMIT.world * CHECKER_ROW_LIMIT.rows == 128


@pytest.mark.parametrize("rows,stages,columns,steps", deep_launches())
def test_ring_model_accepts_every_deep_launch(rows, stages, columns, steps):
    assert model_passes(rows, stages, columns, steps, seeds=3)


def test_virtual_ring_keeps_the_grids_of_the_table(native, monkeypatch):
    """Every geometry above gets the grid the GPU cases assert.  The emulated device takes the native grid rule
    (one CTA per column tile, at most the resident count: 2 CTAs on each of 148 SMs); a requested grid is only cut
    to what lets every rank sharing the GPU stay resident, not divided by the number of ranks."""
    from hpc_patterns_b200.models import halo as halo_mod
    from tests.emu_device import EmuNative, install

    resident = 2 * 148

    class GridRule(EmuNative):
        def halo_stencil_ctas(self, row_elems, mode="pull", tune=None, device=0):
            tune = tune or {}
            tiles = -(-row_elems * 4 // ((tune.get("tile_kb") or 16) * KB))
            return max(1, min(tiles, tune.get("ctas") or resident, resident))

    install(monkeypatch.setattr, GridRule())
    for g in ROUNDING + MULTI_COLUMN + [g for g, _ in DEEP] + [SCHEDULE, CHECKER, CHECKER_ROW_LIMIT]:
        ring = halo_mod.VirtualRing(g.world, g.message, g.rows, "pull", devices=[0] * g.world, tune=g.tune)
        assert [hs.ctas for hs in ring.ranks] == [g.grid] * g.world, g
    g = Geometry(4, 3, 100 * TILE, ctas=100)                   # 4 x 100 CTAs would not all be resident
    ring = halo_mod.VirtualRing(g.world, g.message, g.rows, "pull", devices=[0] * g.world, tune=g.tune)
    assert [hs.ctas for hs in ring.ranks] == [resident // 4] * 4


# ---- GPU helpers ---------------------------------------------------------------------------------------------------

def _ring(g: Geometry, mode: str = "pull", tune: dict | None = None):
    from hpc_patterns_b200.models.halo import VirtualRing

    ring = VirtualRing(g.world, g.message, g.rows, mode, devices=[0] * g.world, alpha=ALPHA, s=S,
                       tune={**g.tune, **(tune or {})})
    assert all(hs.ctas == g.grid for hs in ring.ranks), ([hs.ctas for hs in ring.ranks], g.grid)
    return ring


def _run(ring, g: Geometry, calls) -> None:
    """``calls`` of (steps, persistent) on a fresh ring; the gathered field must equal the reference after each."""
    want = initial_field(g.world, g.rows, g.message // 4)
    done = 0
    for steps, persistent in calls:
        if persistent and ring.ranks[0].depth > 1:           # never launch a deep geometry the slot model rejects
            model_passes(g.rows, g.stages, g.columns, steps)
        ring.step(steps, persistent=persistent)
        done += steps
        want = reference_steps(want, steps, ALPHA, S)
        got = ring.gather()
        assert torch.equal(got, want), (done, int((got != want).sum()))


def _checkers_pass(ring) -> None:
    for hs in ring.ranks:
        assert (hs.verify_from_init(), hs.verify_last_step()) == (0, 0), hs.rank


# ---- GPU 1-4: exact at rounding coefficients -----------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("kernel", list(KERNELS))
@pytest.mark.parametrize("g", ROUNDING, ids=str)
def test_rounding_coefficients_through_every_kernel(native, g, kernel):
    mode, tune = KERNELS[kernel]
    ring = _ring(g, mode, tune)
    try:
        assert all(hs.depth == (SWEEP_DEPTH if kernel == "pull" else 1) for hs in ring.ranks)
        _run(ring, g, SERIES)
        _checkers_pass(ring)
    finally:
        ring.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", list(KERNELS))
@pytest.mark.parametrize("g", MULTI_COLUMN, ids=str)
def test_several_columns_per_cta_with_neighbours(native, g, kernel):
    """Step words are per CTA and a CTA publishes once per sweep, after all its columns; the deep kernel carries its
    register wavefront from one column into the next."""
    mode, tune = KERNELS[kernel]
    ring = _ring(g, mode, tune)
    try:
        assert all(hs.ctas == g.ctas for hs in ring.ranks)
        _run(ring, g, SERIES)
        _checkers_pass(ring)
    finally:
        ring.close()


@pytest.mark.gpu
@pytest.mark.parametrize("g,steps", DEEP, ids=str)
def test_deep_kernel_geometry(native, g, steps):
    ring = _ring(g)
    try:
        assert all(hs.depth == (1 if g.tile_kb > 16 else SWEEP_DEPTH) for hs in ring.ranks)
        _run(ring, g, ((steps, True), (1, False), (steps, True)))
        _checkers_pass(ring)
    finally:
        ring.close()


@pytest.mark.gpu
@pytest.mark.parametrize("first", [0, 1], ids=["from-g0", "after-step1"])
@pytest.mark.parametrize("steps", SCHEDULE_STEPS)
def test_every_schedule(native, steps, first):
    """A persistent launch of every length up to 12, from g = 0 and from g = 1, so that deep sweeps also start at odd
    steps; the sweeps it ran are the schedule rule's."""
    g = SCHEDULE
    ring = _ring(g)
    try:
        _run(ring, g, ((1, False),) * first + ((steps, True),))
        want = sweep_schedule(steps, SWEEP_DEPTH)
        assert list(native.halo_sweep_schedule(steps, SWEEP_DEPTH)) == want
        assert all(hs.depth == SWEEP_DEPTH and hs.last_schedule == want for hs in ring.ranks)
        _checkers_pass(ring)
    finally:
        ring.close()


# ---- GPU 5: the checkers count what is wrong -----------------------------------------------------------------------

def _counts(ring) -> list:
    return [(hs.verify_from_init(), hs.verify_last_step()) for hs in ring.ranks]


@pytest.mark.gpu
def test_checkers_count_one_flipped_bit(native):
    g = CHECKER
    R, n = g.rows, g.message // 4
    ring = _ring(g)
    try:
        _run(ring, g, ((7, True),))
        for r in range(g.world):
            for row, col in ((0, 1000), (R - 1, 1000), (1, 1000), (2, 0), (R - 1, n - 1), (0, n - 3)):
                words = ring.ranks[r].u_tensor().view(torch.int32)
                words[row, col] ^= 1                          # lowest mantissa bit of one word of the current field
                want = [(1, 1) if q == r else (0, 0) for q in range(g.world)]
                assert _counts(ring) == want, (r, row, col)
                words[row, col] ^= 1
                assert _counts(ring) == [(0, 0)] * g.world, (r, row, col)
    finally:
        ring.close()


@pytest.mark.gpu
def test_last_step_checker_counts_what_a_corrupted_input_changes(native):
    """One word of rank q's previous field at its last row feeds rows R-2, R-1 of rank q and row 0 of rank q+1; the
    counts of verify_last_step() must be what a torch step of the corrupted previous field says, rank by rank."""
    g = CHECKER
    R, n = g.rows, g.message // 4
    ring = _ring(g)
    try:
        _run(ring, g, ((7, True),))
        current = ring.gather()
        for q in range(g.world):
            for col in (0, 517, n - 1):
                prev = ring.ranks[q].u_tensor((ring.ranks[q].g - 1) & 1)
                prev[R - 1, col] += 1.0
                torch.cuda.synchronize()
                previous = torch.cat([hs.u_tensor((hs.g - 1) & 1).cpu() for hs in ring.ranks], 0)
                wrong = (current != reference_steps(previous, 1, ALPHA, S)).view(g.world, R, n).sum((1, 2)).tolist()
                assert wrong[q] >= 1 and sum(wrong) >= 2, wrong
                assert [hs.verify_last_step() for hs in ring.ranks] == wrong, (q, col)
                assert [hs.verify_from_init() for hs in ring.ranks] == [0] * g.world
                prev[R - 1, col] -= 1.0
                assert _counts(ring) == [(0, 0)] * g.world, (q, col)
    finally:
        ring.close()


@pytest.mark.gpu
def test_verify_from_init_at_its_global_row_limit(native):
    g = CHECKER_ROW_LIMIT
    ring = _ring(g)
    try:
        _run(ring, g, ((7, True),))
        _checkers_pass(ring)
    finally:
        ring.close()
    over = Geometry(3, 43, 16)                                  # 129 global rows
    ring = _ring(over)
    try:
        with pytest.raises(RuntimeError, match="128"):
            ring.ranks[0].verify_from_init()
    finally:
        ring.close()


# ---- GPU 6: the benchmark computes the reference -------------------------------------------------------------------

@pytest.mark.gpu
def test_bench_outputs_equal_the_reference(native, tmp_path):
    """bench.py's timed call at the default depth and at depth 1 (HPCP_HALO_DEPTH=1): zero wrong words, identical
    dumps, and the dumped columns equal the reference.  bench.py runs at alpha = 0.5, s = 0.25, where contraction
    does not show; what this guards is the deep kernel at the benchmark's geometry and the dump path."""
    import numpy as np

    from bench import DUMP_ELEMS, dump_columns

    dumps = {}
    for depth in ("", "1"):
        out = tmp_path / f"depth{depth or 'default'}"
        env = {k: v for k, v in os.environ.items() if k not in ("HPCP_HALO_DEPTH", "RANK", "WORLD_SIZE", "LOCAL_RANK")}
        if depth:
            env["HPCP_HALO_DEPTH"] = depth
        proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", *BENCH_ARGS,
                               "--dump-outputs", str(out)], env=env, capture_output=True, text=True, timeout=900)
        assert proc.returncode == 0, proc.stderr[-3000:]
        line = json.loads([ln for ln in proc.stdout.splitlines() if ln.startswith("{")][-1])
        assert line["wrong_words"] == 0 and line["e2e"]["wrong_words"] == 0, line
        dumps[depth] = np.load(out / "field_rank0.npy")
    assert np.array_equal(dumps[""].view(np.uint32), dumps["1"].view(np.uint32))
    g = BENCH
    cols = torch.from_numpy(dump_columns(g.message // 4, DUMP_ELEMS // g.rows))
    want = reference_steps(initial_field(g.world, g.rows, g.message // 4)[:, cols], 20)
    assert torch.equal(torch.from_numpy(dumps[""]), want)
