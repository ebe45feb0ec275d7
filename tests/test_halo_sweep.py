"""Deep sweeps of K-halo (halo_sweep_kernel<D> in csrc/kernels/halo_stencil.cu), on the CPU: the sweep schedule, and an
executable model of the kernel's shared-memory ring and register wavefront.

A sweep of depth d streams the R + 2d input tiles of a column tile (rows -d .. R+d-1) through a ring of S slots.  Arrival
i >= 2 computes level 1 of row i-d-1 from the input tiles i-2, i-1, i and level L of row i-d-L from level L-1 (two rows
in registers + the one just computed); arrivals i >= 2d write level d of row i-2d over input tile i-2 and the DMA thread
stores it.  Every arrival is one `computed` event of slot i-2; a stored event frees the tiles below it after
`bulk_wait_read<1>` (`retired = t`), an unstored one (the first 2d-2 of a column) frees its own tile after
`bulk_wait_read<0>` (`retired = t + 1`); the event cursor moves by 2 more at the end of a column.  The model restates
those rules, runs the DMA thread and the math warps as coroutines under a random scheduler that delays every bulk load
and store completion, and checks: no deadlock, no load lands in a slot that a store or the wavefront still reads, every
level reads the rows it is meant to, every store sends level d of the row it is meant to.  Mutated rules must be caught.
"""
import random

import pytest

from hpc_patterns_b200.models.halo import DEFAULT_SWEEP_DEPTH, sweep_depth, sweep_schedule
from tests.test_halo_pipeline_model import Cursor
from tests.test_umma_pipeline_model import MBar, ProtocolError, run

MATH_WARPS = 3


@pytest.mark.parametrize("depth", [1, 3, 5, 7])
@pytest.mark.parametrize("steps", list(range(1, 42)))
def test_schedule_rule(steps, depth):
    sweeps = sweep_schedule(steps, depth)
    assert sum(sweeps) == steps
    assert all(d % 2 == 1 and 1 <= d <= depth for d in sweeps)
    assert sweeps[-1] == 1
    # greedy: every sweep is the largest odd size that leaves at least one step for the closing one-step sweep
    k = 0
    for d in sweeps[:-1]:
        x = min(depth, steps - k - 1)
        assert d == (x if x % 2 else x - 1) or (x <= 1 and d == 1)
        k += d


def test_schedule_of_the_benchmark():
    assert sweep_schedule(20, 3) == [3] * 6 + [1, 1]
    assert sweep_schedule(20, 5) == [5, 5, 5, 3, 1, 1]
    assert sweep_schedule(20, 1) == [1] * 20
    assert sweep_schedule(3, 3) == [1, 1, 1]      # no deep sweep: the single-step kernel runs
    assert sweep_schedule(4, 3) == [3, 1]


def test_native_schedule_and_depth_match_the_mirror(native):
    for steps in range(1, 30):
        for depth in (1, 3, 5):
            assert list(native.halo_sweep_schedule(steps, depth)) == sweep_schedule(steps, depth)
    assert native.HALO_DEFAULT_DEPTH == 3
    assert native.halo_sweep_depth(8, "pull", {}) == 3
    assert native.halo_sweep_depth(8, "pull", {"depth": 1}) == 1
    assert native.halo_sweep_depth(8, "pull", {"depth": 7}) == 3      # deepest instantiation
    assert native.halo_sweep_depth(2, "pull", {}) == 1                # halo rows come from the neighbours only
    assert native.halo_sweep_depth(3, "pull", {}) == 3
    assert native.halo_sweep_depth(8, "push", {}) == 1
    assert native.halo_sweep_depth(8, "pull", {"tile_kb": 32}) == 1   # wavefront registers sized for 16 KiB tiles
    assert native.halo_sweep_depth(8, "pull", {"l2_hint": 1}) == 1


def test_python_depth_rule_matches_native(native):
    """HaloStencil.depth (the traffic model, reports) comes from the Python mirror; the launch uses the native rule."""
    assert DEFAULT_SWEEP_DEPTH == native.HALO_DEFAULT_DEPTH
    for rows in (1, 2, 3, 4, 8):
        for mode in ("pull", "push", "none"):
            for tune in ({}, {"depth": 0}, {"depth": 1}, {"depth": 2}, {"depth": 3}, {"depth": 5}, {"tile_kb": 8},
                         {"tile_kb": 16}, {"tile_kb": 32}, {"l2_hint": 1}, {"depth": 3, "tile_kb": 4}):
                assert sweep_depth(rows, mode, tune) == native.halo_sweep_depth(rows, mode, tune), (rows, mode, tune)


def simulate(stages, rows, ncols, schedule, seed, free_extra=0, end_skip=2, wait_unstored=True, retire_unstored=True,
             store_delay=0):
    """free_extra: tiles freed beyond the rules; end_skip: extra event-cursor advance at the end of a column;
    wait_unstored: bulk_wait_read<0> before an unstored event frees its tile; retire_unstored: whether it does;
    store_delay: a store cannot read its slot before the DMA thread consumed this many more events or waits for it
    (slow stores: a legal schedule that the uniform random scheduler rarely picks)."""
    rng = random.Random(seed)
    S, R, W = stages, rows, MATH_WARPS
    full = [MBar(f"full[{i}]", 1) for i in range(S)]
    computed = [MBar(f"computed[{i}]", W) for i in range(S)]
    content = [None] * S          # ("in", sweep, col, m) input tile m, ("out", sweep, col, (level, row)) a result
    busy_store = [0] * S
    needed_by_math = [0] * S
    writes = [0] * S
    load_q, store_q = [], []
    parked = []                   # [events still to consume, completion] of delayed stores
    stored = []

    def release(until=None):
        """One more event consumed (until=None), or the DMA thread waits for the store of `until`: it and every older
        store become able to complete."""
        if until is not None:
            while any(item[2] is until for item in parked):
                store_q.append(parked.pop(0)[1])
            return
        for item in list(parked):
            item[0] -= 1
            if item[0] <= 0:
                parked.remove(item)
                store_q.append(item[1])

    def dma():
        ld, ev, done = Cursor(S), Cursor(S), Cursor(S)
        for sw, d in enumerate(schedule):
            n_in = R + 2 * d
            loads, events = ncols * n_in, ncols * (n_in - 2)
            issued = retired = 0
            jj_l = m_l = 0
            jj_c, i, t = 0, 2, 0
            outstanding = []
            for _ in range(events):
                while issued < loads and issued < retired + S + free_extra:
                    slot = ld.slot
                    full[slot].arrive(expect_tx=1)
                    # arrivals m, m+1, m+2 read input tile m (as down, centre, up); arrivals run from 2 to n_in - 1
                    readers = sum(1 for a in (m_l, m_l + 1, m_l + 2) if 2 <= a < n_in)

                    def landed(slot=slot, tile=("in", sw, jj_l, m_l), readers=readers):
                        if busy_store[slot]:
                            raise ProtocolError(f"load of {tile} landed in slot {slot} while a store still reads it")
                        if needed_by_math[slot]:
                            raise ProtocolError(f"load of {tile} landed in slot {slot}: {content[slot]} is still needed")
                        content[slot] = tile
                        needed_by_math[slot] = readers * W
                        full[slot].complete_tx(1)

                    load_q.append(landed)
                    ld.advance(1)
                    issued += 1
                    m_l += 1
                    if m_l == n_in:
                        m_l, jj_l = 0, jj_l + 1
                yield lambda s=done.slot, p=done.phase: computed[s].done(p)
                done.advance(1)
                release()
                if i >= 2 * d:
                    slot = ev.slot
                    busy_store[slot] += 1
                    token = [False]

                    def read_out(slot=slot, want=("out", sw, jj_c, (d, i - 2 * d)), token=token):
                        if content[slot] != want:
                            raise ProtocolError(f"store of {want} read {content[slot]} from slot {slot}")
                        stored.append(want)
                        busy_store[slot] -= 1
                        token[0] = True

                    if store_delay:
                        parked.append([store_delay, read_out, token])
                    else:
                        store_q.append(read_out)
                    outstanding.append(token)
                    while len(outstanding) > 1:                  # bulk_wait_read<1>
                        oldest = outstanding.pop(0)
                        release(until=oldest)
                        yield lambda tk=oldest: tk[0]
                    retired = t
                else:
                    if wait_unstored:                            # bulk_wait_read<0>
                        for tk in outstanding:
                            release(until=tk)
                            yield lambda tk=tk: tk[0]
                        outstanding = []
                    if retire_unstored:
                        retired = t + 1
                t += 1
                ev.advance(1)
                i += 1
                if i == n_in:
                    i, jj_c, t = 2, jj_c + 1, t + 2
                    ev.advance(end_skip)
            for tk in outstanding:                               # bulk_wait<0> at the end of the sweep
                release(until=tk)
                yield lambda tk=tk: tk[0]

    def math(warp):
        up_t, done = Cursor(S), Cursor(S)
        for sw, d in enumerate(schedule):
            n_in = R + 2 * d
            for jj in range(ncols):
                lv = {}                                          # level -> its two newest rows, (level, row) tuples
                for i in range(2, n_in):
                    ce_t, dn_t = up_t.at(1), up_t.at(2)
                    if i == 2:
                        yield lambda c=up_t: full[c.slot].done(c.phase)
                        yield lambda c=ce_t: full[c.slot].done(c.phase)
                    yield lambda c=dn_t: full[c.slot].done(c.phase)
                    want = tuple(("in", sw, jj, i - 2 + k) for k in range(3))
                    got = (content[up_t.slot], content[ce_t.slot], content[dn_t.slot])
                    if got != want:
                        raise ProtocolError(f"level 1 of sweep {sw} col {jj} arrival {i} (warp {warp}) read {got}")
                    for c in (up_t, ce_t, dn_t):
                        needed_by_math[c.slot] -= 1
                    x = (1, i - d - 1)
                    for L in range(2, d + 1):
                        y = x
                        if i >= 2 * L:
                            pair = lv.get(L - 1)
                            if pair != [(L - 1, i - d - L - 1), (L - 1, i - d - L)] or x != (L - 1, i - d - L + 1):
                                raise ProtocolError(f"level {L} at arrival {i}: registers {pair}, new {x}")
                            y = (L, i - d - L)
                        lv[L - 1] = (lv.get(L - 1) or [None, None])[1:] + [x]
                        x = y
                    if i >= 2 * d:
                        writes[up_t.slot] += 1
                        if writes[up_t.slot] == W:
                            writes[up_t.slot] = 0
                            content[up_t.slot] = ("out", sw, jj, x)
                    yield None
                    computed[done.slot].arrive()
                    done.advance(1)
                    up_t.advance(1)
                up_t.advance(2)

    agents = [dma()] + [math(w) for w in range(MATH_WARPS)]
    run(agents, [load_q, store_q], rng)
    want = [("out", sw, c, (d, r)) for sw, d in enumerate(schedule) for c in range(ncols) for r in range(R)]
    if sorted(stored) != sorted(want):
        raise ProtocolError("not every result tile was stored exactly once")
    return len(stored)


@pytest.mark.parametrize("stages", [6, 7, 12])
@pytest.mark.parametrize("rows,ncols", [(3, 3), (4, 2), (8, 2), (9, 1)])
@pytest.mark.parametrize("steps", [4, 7, 20])
def test_sweep_rules_are_safe_under_random_schedules(stages, rows, ncols, steps):
    schedule = sweep_schedule(steps, 3)
    for seed in range(10):
        for store_delay in (0, 3):
            assert simulate(stages, rows, ncols, schedule, seed, store_delay=store_delay) == len(schedule) * rows * ncols


def test_deeper_sweeps_keep_the_rules():
    """The rules do not depend on D: depth 5 and 7 (not instantiated for register reasons) pass the model too."""
    for depth, rows in ((5, 5), (7, 8)):
        schedule = sweep_schedule(2 * depth + 1, depth)
        for seed in range(10):
            assert simulate(6, rows, 2, schedule, seed) == len(schedule) * rows * 2


def test_loads_running_too_far_ahead_are_caught():
    with pytest.raises(ProtocolError):
        for seed in range(200):
            simulate(6, 3, 3, [3, 1], seed, free_extra=1)


def test_wrong_end_of_column_skip_is_caught():
    with pytest.raises(ProtocolError):
        for seed in range(50):
            simulate(6, 3, 3, [3, 1], seed, end_skip=1)


def test_freeing_an_unstored_tile_without_waiting_for_the_stores_is_caught():
    """`retired = t + 1` with the previous column's last store still reading its slot: a load can land on it."""
    with pytest.raises(ProtocolError, match="store still reads"):
        for seed in range(100):
            simulate(6, 3, 4, [3, 1], seed, wait_unstored=False, store_delay=4)


def test_unstored_events_must_free_their_tile():
    """Without `retired = t + 1` the 2d + 1 = 7 tiles a column needs before its first store do not fit 6 slots."""
    with pytest.raises(ProtocolError, match="deadlock"):
        simulate(6, 3, 3, [3, 1], seed=0, retire_unstored=False)


def test_emulated_deep_launches_and_traffic_model(monkeypatch):
    """The Python layer on the emulated device (which steps one step at a time, the result a deep launch must equal):
    HaloStencil picks depth 3, the field and verify_last_step() hold, and the byte model follows the sweeps of the last
    multi-step launch."""
    import torch

    from hpc_patterns_b200.models import halo as halo_mod
    from hpc_patterns_b200.models.halo import initial_field, reference_steps
    from tests.emu_device import EmuNative, install

    emu = EmuNative()
    install(monkeypatch.setattr, emu)
    n, rows = 3000, 8
    hs = halo_mod.VirtualRing(1, 4 * n, rows, "pull", devices=[0], tune={"tile_kb": 4}).ranks[0]
    assert hs.depth == 3
    b = hs.row_bytes
    assert hs.hbm_bytes_per_step() == (2 * rows + 2) * b
    hs.step(20)
    assert torch.equal(hs.u_tensor(), reference_steps(initial_field(1, rows, n), 20))
    assert hs.verify_last_step() == 0 and hs.verify_from_init() == 0
    assert hs.hbm_bytes_per_step() == (6 * (2 * rows + 6) + 2 * (2 * rows + 2)) * b // 20
    hs.step(1)                                       # a per-step launch keeps the model of the persistent one
    assert hs.hbm_bytes_per_step() == (6 * (2 * rows + 6) + 2 * (2 * rows + 2)) * b // 20
    monkeypatch.setenv("HPCP_HALO_DEPTH", "1")
    one = halo_mod.VirtualRing(1, 4 * n, rows, "pull", devices=[0], tune={"tile_kb": 4}).ranks[0]
    assert one.depth == 1
    one.step(20)
    assert one.hbm_bytes_per_step() == (2 * rows + 2) * b
