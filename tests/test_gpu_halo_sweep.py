"""GPU tests of the deep K-halo sweeps (halo_sweep_kernel in csrc/kernels/halo_stencil.cu): multi-step pull launches that
advance the slab up to 3 steps per pass must compute exactly what one step per pass computes, the plain PyTorch fp32
run of the whole undecomposed field."""
import pytest
import torch

pytestmark = pytest.mark.gpu

MESSAGE = 5 * 16384 + 2048      # six column tiles of 16 KiB, the last one partial


def _ring(world, rows, tune=None, message_bytes=MESSAGE):
    from hpc_patterns_b200.models.halo import VirtualRing

    return VirtualRing(world, message_bytes, rows, "pull", devices=[0] * world, tune=dict(tune or {}))


def _want(world, rows, row_elems, steps):
    from hpc_patterns_b200.models.halo import initial_field, reference_steps

    return reference_steps(initial_field(world, rows, row_elems), steps)


@pytest.mark.parametrize("world", [1, 2, 4])
@pytest.mark.parametrize("rows", [3, 4, 5, 6, 7, 8, 9])
def test_persistent_deep_launches_are_exact(native, world, rows):
    ring = _ring(world, rows)
    try:
        assert all(hs.depth == 3 for hs in ring.ranks)
        done = 0
        for k in (2, 3, 5, 13, 20):
            ring.step(k, persistent=True)
            done += k
            got = ring.gather()
            want = _want(world, rows, MESSAGE // 4, done)
            assert torch.equal(got, want), (k, float((got - want).abs().max()))
        for hs in ring.ranks:
            assert hs.verify_from_init() == 0 and hs.verify_last_step() == 0
    finally:
        ring.close()


@pytest.mark.parametrize("world,rows", [(1, 8), (2, 3), (4, 5)])
def test_mixed_series(native, world, rows):
    """step(1) / step(K) / step(1): the single-step and the deep kernel share the grid and the step words."""
    ring = _ring(world, rows, tune={"tile_kb": 8, "stages": 8})
    try:
        ring.step(1)
        ring.step(11, persistent=True)
        ring.step(1)
        ring.step(4, persistent=True)
        ring.step(2)
        assert torch.equal(ring.gather(), _want(world, rows, MESSAGE // 4, 19))
    finally:
        ring.close()


def test_depth_one_and_default_depth_agree_at_a_24_mib_row(native):
    """Default geometry (16 KiB x 6 stages, two CTAs per SM) at a 24 MiB row: the deep launch keeps the grid of the
    single-step kernel, verify_last_step() holds after it, and the field is bit-identical to depth 1."""
    from hpc_patterns_b200.models.halo import HaloStencil
    from hpc_patterns_b200.parallel.comm import Comm

    fields, ctas = {}, {}
    for depth in (1, 0):
        hs = HaloStencil(Comm(), 0, message_bytes=24 << 20, rows=8, mode="pull", tune={"depth": depth} if depth else {})
        try:
            assert hs.depth == (3 if depth == 0 else 1)
            hs.step(20)
            torch.cuda.synchronize()
            hs.check()
            assert hs.verify_from_init() == 0 and hs.verify_last_step() == 0
            fields[depth] = hs.u_tensor().clone()
            ctas[depth] = hs.ctas
            assert hs.ctas >= 148
        finally:
            hs.close()
    assert ctas[0] == ctas[1]
    assert torch.equal(fields[0], fields[1])
