"""CPU tests of the launch order of a batch's tiles (af_debug_tile_order): CTA c of a fused launch over n_ctas CTAs runs
the tiles at positions c, c + n_ctas, ...; the order must be a permutation that evens out the CTAs' step counts."""
import ctypes as C

import numpy as np
import pytest

SMS = 148       # B200


def _order(steps, n_ctas):
    import audioflow
    L = audioflow.load_library()
    s = np.ascontiguousarray(steps, np.uint32)
    o = np.full(len(s), 0xFFFFFFFF, np.uint32)
    u32p = C.POINTER(C.c_uint32)
    mx = L.af_debug_tile_order(s.ctypes.data_as(u32p), len(s), n_ctas, o.ctypes.data_as(u32p))
    return o, int(mx)


def _loads(steps, order, n_ctas):
    loads = np.zeros(n_ctas, np.int64)
    np.add.at(loads, np.arange(len(order)) % n_ctas, np.asarray(steps, np.int64)[order])
    return loads


def _stream_tiles(frames):
    """steps of each tile of a stream with `frames` STFT frames (128 frames per tile, 32 per step)"""
    n_tiles = max(1, -(-frames // 128))
    return [min(4, -(-min(128, frames - 128 * t) // 32)) if frames > 128 * t else 1 for t in range(n_tiles)]


def _check(steps, n_ctas):
    order, mx = _order(steps, n_ctas)
    assert sorted(order.tolist()) == list(range(len(steps))), "not a permutation"
    loads = _loads(steps, order, n_ctas)
    assert mx == loads.max()
    ident = _loads(steps, np.arange(len(steps)), n_ctas).max()
    assert mx <= ident
    assert mx >= -(-int(np.sum(steps)) // n_ctas)
    return order, mx, ident


def test_cfg2_shape_reaches_the_bound():
    """256 streams of 30 s: 23 tiles of 4 steps and one of 2 each.  Round robin gives the busiest CTA 168 steps; every
    tile costs 2 or 4, so no whole-tile assignment does better than 164."""
    steps = [4] * 23 + [2]
    steps = steps * 256
    _, mx, ident = _check(steps, SMS)
    assert ident == 168
    assert mx == 164


def test_fewer_tiles_than_ctas_keep_their_order():
    steps = [4, 2, 3, 1, 4]
    order, mx = _order(steps, len(steps))
    assert order.tolist() == list(range(len(steps))) and mx == 4


@pytest.mark.parametrize("seed", range(6))
def test_ragged_batches(seed):
    rng = np.random.default_rng(seed)
    n_streams = int(rng.integers(1, 400))
    steps = []
    for f in rng.integers(0, 6000, n_streams):
        steps += _stream_tiles(int(f))
    n_ctas = min(len(steps), SMS)
    _, mx, _ = _check(steps, n_ctas)
    # longest first to the least loaded CTA: within one tile (4 steps) of the mean when the positions allow it
    if len(steps) >= 4 * n_ctas:
        assert mx <= -(-sum(steps) // n_ctas) + 4


@pytest.mark.parametrize("n_tiles", [149, 150, 200, 295, 297])
def test_just_over_one_tile_per_cta(n_tiles):
    rng = np.random.default_rng(n_tiles)
    steps = rng.integers(1, 5, n_tiles).tolist()
    _check(steps, SMS)
