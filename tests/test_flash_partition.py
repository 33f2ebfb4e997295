"""CPU: the tile partition of the sharded FlashVDM decoder (hy3dgeo.parallel.flash_partition) and the host image of the
level-0 layout sizes (flash_minigrid_sizes; checked against the kernel in tests/test_gpu_sharded_flash.py)."""
import random

import pytest

from hy3dgeo.parallel import _tile_queries, flash_minigrid_sizes, flash_partition


def _check(tiles, world):
    parts = flash_partition(tiles, world)
    total = sum(tiles)
    assert len(parts) == world
    owner = []                                     # group of every tile, in list order
    for g, k in enumerate(tiles):
        owner += [g] * k
    nxt = 0
    for t0, t1, g0, g1 in parts:
        assert t0 == nxt and t1 >= t0              # contiguous, ordered, every tile owned exactly once
        nxt = t1
        if t1 == t0:
            assert g0 == g1                        # no tiles: empty group range
        else:
            # the range runs from the first tile's group to the last tile's; the groups inside it that hold tiles are
            # exactly the groups these tiles use (groups without tiles may lie between them)
            assert owner[t0] == g0 and owner[t1 - 1] == g1 - 1
            assert {g for g in range(g0, g1) if tiles[g]} == set(owner[t0:t1])
    assert nxt == total
    sizes = [t1 - t0 for t0, t1, _, _ in parts]
    assert max(sizes) - min(sizes) <= 1
    return parts


@pytest.mark.parametrize("world", [1, 2, 3, 8, 300])
def test_random_tile_counts(world):
    rng = random.Random(world)
    for _ in range(200):
        G = rng.choice([1, 2, 64, 216])
        tiles = [rng.choice([0, 0, 1, 2, 5, 108, rng.randrange(0, 300)]) for _ in range(G)]
        _check(tiles, world)


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_empty_and_degenerate_lists(world):
    for tiles in ([], [0], [0] * 216, [0, 0, 1, 0], [3] + [0] * 215, [0] * 215 + [1]):
        parts = _check(tiles, world)
        if sum(tiles) == 0:
            assert all(t0 == t1 and g0 == g1 for t0, t1, g0, g1 in parts)


def test_more_ranks_than_tiles():
    parts = _check([0, 2, 0, 1], 8)
    assert sum(1 for t0, t1, _, _ in parts if t1 > t0) == 3
    assert [(g0, g1) for t0, t1, g0, g1 in parts if t1 > t0] == [(1, 2), (1, 2), (3, 4)]


def test_level0_over_three_ranks_splits_groups():
    counts, soff = flash_minigrid_sizes(96, 4, 100)           # octree 384: 64 mini-grids of 24^3 = 108 tiles
    tiles = [-(-c // 128) for c in counts]
    assert tiles == [108] * 64 and soff == [g * 139 for g in range(65)]
    parts = _check(tiles, 3)
    assert [t1 - t0 for t0, t1, _, _ in parts] == [2304] * 3
    assert parts[0][3] == 22 and parts[1][2] == 21              # mini-grid 21 is cut: selected by ranks 0 and 1


@pytest.mark.parametrize("N,m,stride", [(96, 4, 100), (16, 4, 100), (15, 3, 7), (64, 8, 100), (8, 2, 1)])
def test_minigrid_sizes(N, m, stride):
    counts, soff = flash_minigrid_sizes(N, m, stride)
    s3 = (N // m) ** 3
    assert counts == [s3] * m ** 3 and len(soff) == m ** 3 + 1
    assert soff[0] == 0 and all(b - a == len(range(0, s3, stride)) for a, b in zip(soff, soff[1:]))


def test_tile_queries_sum_to_the_list():
    rng = random.Random(7)
    for world in (1, 2, 3, 8, 50):
        counts = [rng.choice([0, 1, 127, 128, 129, rng.randrange(0, 2000)]) for _ in range(216)]
        parts = flash_partition([-(-c // 128) for c in counts], world)
        q = [_tile_queries(counts, t0, t1) for t0, t1, _, _ in parts]
        assert sum(q) == sum(counts) and all(v <= 128 * (t1 - t0) for v, (t0, t1, _, _) in zip(q, parts))
