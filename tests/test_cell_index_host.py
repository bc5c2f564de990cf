"""CPU: the cell index of a map (BCG_BATCH_CELL_INDEX trailer) as a NumPy reference, and the property the sparse
egocentric kernel rests on: the cells of tile columns c0 .. c1 - 1 of band ty are cells[prefix[ty tx + c0] ..
prefix[ty tx + c1])."""
import numpy as np
import pytest


def cell_index_reference(data):
    """(prefix, cells) of a uint8 [H, W] costmap: exclusive counts of cells != 0 per 32 x 16 tile (row-major tile order,
    tiles_y * tiles_x + 1 entries), and every such cell as x | y << 16, grouped by tile, row-major inside a tile."""
    h, w = data.shape
    tiles_x, tiles_y = (w + 31) // 32, (h + 15) // 16
    occ = np.zeros((tiles_y * 16, tiles_x * 32), dtype=bool)
    occ[:h, :w] = data != 0
    tiles = occ.reshape(tiles_y, 16, tiles_x, 32).transpose(0, 2, 1, 3).reshape(tiles_y * tiles_x, 16, 32)
    prefix = np.r_[0, np.cumsum(tiles.reshape(len(tiles), -1).sum(axis=1))].astype(np.uint32)
    t, r, bit = np.nonzero(tiles)
    x = (t % tiles_x) * 32 + bit
    y = (t // tiles_x) * 16 + r
    return prefix, (x | (y << 16)).astype(np.uint32)


def _random_map(rng, h, w, density):
    data = np.zeros((h, w), dtype=np.uint8)
    mask = rng.random_sample((h, w)) < density
    data[mask] = rng.choice([254, 99, 1], size=int(mask.sum()))
    return data


@pytest.mark.parametrize("shape", [(1, 1), (16, 32), (17, 33), (100, 75), (250, 301)])
@pytest.mark.parametrize("density", [0.0, 0.01, 0.05])
def test_reference_lists_every_occupied_cell_once_grouped_by_tile(shape, density):
    rng = np.random.RandomState(shape[0] * 1000 + shape[1] + int(density * 100))
    data = _random_map(rng, *shape, density)
    prefix, cells = cell_index_reference(data)
    tiles_x = (shape[1] + 31) // 32
    assert prefix[0] == 0 and prefix[-1] == len(cells) == np.count_nonzero(data)
    x, y = cells & 0xffff, cells >> 16
    assert np.all(data[y, x] != 0)
    assert len(set(cells.tolist())) == len(cells)
    tile = (y // 16) * tiles_x + x // 32
    assert np.all(np.diff(tile) >= 0)
    for t in range(len(prefix) - 1):                     # a tile's cells sit in [prefix[t], prefix[t + 1]), row-major
        seg = cells[prefix[t]:prefix[t + 1]]
        assert np.all(tile[prefix[t]:prefix[t + 1]] == t)
        key = (seg >> 16).astype(np.int64) * 65536 + (seg & 0xffff)
        assert np.all(np.diff(key) > 0)


def test_band_column_range_is_one_contiguous_slice():
    rng = np.random.RandomState(3)
    data = _random_map(rng, 203, 290, 0.03)
    prefix, cells = cell_index_reference(data)
    tiles_x, tiles_y = (290 + 31) // 32, (203 + 15) // 16
    x, y = cells & 0xffff, cells >> 16
    for _ in range(200):
        ty = rng.randint(tiles_y)
        c0 = rng.randint(tiles_x + 1)
        c1 = rng.randint(c0, tiles_x + 1)
        got = cells[prefix[ty * tiles_x + c0]:prefix[ty * tiles_x + c1]]
        want = cells[(y // 16 == ty) & (x // 32 >= c0) & (x // 32 < c1)]
        assert np.array_equal(np.sort(got), np.sort(want))
