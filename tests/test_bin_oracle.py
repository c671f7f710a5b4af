"""CPU: the restatement of tile binning (oracle/bin_oracle.py) against lists worked out by hand, a loop-by-loop restatement and its
own invariants, before it is used to check the GPU binning bit for bit (tests/test_binning_gpu.py)."""
import numpy as np
import pytest

from oracle import bin_oracle as B

EMPTY = (1, 1, 0, 0)


def _entry(mask, sid):
    return (mask << 32) | sid


def _lists_by_loops(rects, order, width, height, rank=0, world=1):
    """The same definition, one draw rank and one fine tile at a time: {coarse tile id: [entries in draw order]}."""
    g = B.geometry(width, height)
    lists = {}
    for p, sid in enumerate(reversed([int(s) for s in order])):
        x0, y0, x1, y1 = (int(v) for v in rects[sid])
        masks = {}
        for fy in range(y0, y1 + 1):
            for fx in range(x0, x1 + 1):
                cx, cy = fx // 8, fy // 4
                masks[(cx, cy)] = masks.get((cx, cy), 0) | (1 << (8 * (fy % 4) + fx % 8))
        for (cx, cy), m in masks.items():
            if world > 1 and (cx + cy) % world != rank:
                continue
            lists.setdefault(cy * g.coarse_x + cx, []).append((p, _entry(m, sid)))
    return {t: [e for _, e in sorted(v)] for t, v in lists.items()}


def _random_rects(rng, n, g, empty_frac=0.2, big_frac=0.05):
    x0 = rng.integers(0, g.tiles_x, n)
    y0 = rng.integers(0, g.tiles_y, n)
    span = np.where(rng.uniform(size=n) < big_frac, rng.integers(8, 80, n), rng.integers(0, 4, n))
    x1 = np.minimum(x0 + span, g.tiles_x - 1)
    y1 = np.minimum(y0 + rng.integers(0, 3, n) + span // 2, g.tiles_y - 1)
    r = np.stack([x0, y0, x1, y1], 1).astype(np.uint16)
    r[rng.uniform(size=n) < empty_frac] = EMPTY
    r[rng.integers(0, n, max(1, n // 100))] = (0, 0, g.tiles_x - 1, g.tiles_y - 1)      # whole-screen splats
    return r


@pytest.mark.parametrize("w,h,px,ncoarse,path", [
    (320, 200, 16, 12, B.COUNTING), (1920, 1080, 16, 255, B.COUNTING), (1921, 1080, 32, 72, B.COUNTING),
    (3840, 2160, 32, 255, B.COUNTING), (4096, 2160, 32, 272, B.RADIX), (7680, 4320, 32, 1020, B.RADIX),
    (4096, 256, 16, 128, B.COUNTING), (8192, 256, 16, 256, B.COUNTING), (256, 8192, 16, 256, B.COUNTING), (24576, 64, 16, 192, B.COUNTING)])
def test_geometry_and_path(w, h, px, ncoarse, path):
    g = B.geometry(w, h)
    assert (g.tile_px, g.ncoarse) == (px, ncoarse)
    assert B.binning_path(w, h) == path
    assert B.binning_path(w, h, bin_version=1) == B.RADIX


def test_hand_built_rects():
    # 320 x 200 at 16 px: 20 x 13 fine tiles, 3 x 4 coarse tiles (ids cy * 3 + cx)
    rects = np.array([
        (5, 6, 5, 6),        # splat 0: one fine tile, (5, 6) -> coarse (0, 1), fine (5, 2) inside it: bit 21
        (7, 3, 8, 4),        # splat 1: the four fine tiles around the corner shared by coarse tiles 0, 1, 3, 4
        (0, 0, 19, 12),      # splat 2: the whole screen, incl. the partial last coarse column (4 fine tiles) and row (1)
        EMPTY,               # splat 3: not drawn
    ], np.uint16)
    order = np.array([3, 2, 1, 0], np.uint32)       # draw ranks 0, 1, 2, 3 = splats 0, 1, 2, 3
    b = B.bin_frame(rects, order, 320, 200)
    full, col4, row1, corner = 0xFFFFFFFF, 0x0F0F0F0F, 0xFF, 0x0F
    want = {
        0: [_entry(1 << 31, 1), _entry(full, 2)],
        1: [_entry(1 << 24, 1), _entry(full, 2)],
        2: [_entry(col4, 2)],
        3: [_entry(1 << 21, 0), _entry(1 << 7, 1), _entry(full, 2)],
        4: [_entry(1 << 0, 1), _entry(full, 2)],
        5: [_entry(col4, 2)],
        6: [_entry(full, 2)], 7: [_entry(full, 2)], 8: [_entry(col4, 2)],
        9: [_entry(row1, 2)], 10: [_entry(row1, 2)], 11: [_entry(corner, 2)],
    }
    for t in range(12):
        assert b.list_of(t).tolist() == want[t], t
    assert b.total == 1 + 4 + 12
    counts = [2, 2, 1, 3, 2, 1, 1, 1, 1, 1, 1, 1]
    ends = np.cumsum(counts)
    assert b.ranges(B.COUNTING).tolist() == [[int(e - c), int(e)] for e, c in zip(ends, counts)]
    assert b.ranges(B.RADIX).tolist() == b.ranges(B.COUNTING).tolist()      # no empty tile here
    assert b.tile_order(B.COUNTING).tolist() == [3, 0, 1, 4, 2, 5, 6, 7, 8, 9, 10, 11]
    assert b.tile_order(B.RADIX).tolist() == list(range(12))
    # only the single pixel: the empty tiles' encodings differ between the paths
    one = B.bin_frame(rects, np.array([0], np.uint32), 320, 200)
    assert one.ranges(B.COUNTING).tolist() == [[0, 0]] * 3 + [[0, 1]] + [[1, 1]] * 8
    assert one.ranges(B.RADIX).tolist() == [list(B.EMPTY_RANGE)] * 3 + [[0, 1]] + [list(B.EMPTY_RANGE)] * 8
    assert one.tile_order(B.COUNTING).tolist() == [3, 0, 1, 2, 4, 5, 6, 7, 8, 9, 10, 11]
    # overflow: both ends clamped to the capacity
    assert b.ranges(B.COUNTING, capacity=5).tolist() == [[0, 2], [2, 4], [4, 5]] + [[5, 5]] * 9
    # nothing drawn
    none = B.bin_frame(rects, np.array([3], np.uint32), 320, 200)
    assert none.total == 0 and none.entries.size == 0


@pytest.mark.parametrize("w,h,seed", [(320, 200, 1), (801, 455, 2), (4112, 256, 3), (256, 1024, 4), (4096, 2160, 5)])
def test_matches_loop_restatement(w, h, seed):
    rng = np.random.default_rng(seed)
    g = B.geometry(w, h)
    n = 600
    rects = _random_rects(rng, n, g)
    order = rng.permutation(n)[: n - 37].astype(np.uint32)      # render_count below the splat count
    for world in (1, 3):
        for rank in range(world):
            b = B.bin_frame(rects, order, w, h, rank, world)
            want = _lists_by_loops(rects, order, w, h, rank, world)
            for t in range(g.ncoarse):
                assert b.list_of(t).tolist() == want.get(t, []), (world, rank, t)


@pytest.mark.parametrize("w,h", [(801, 455), (1921, 1080), (7680, 4320), (8192, 256)])
def test_invariants(w, h):
    rng = np.random.default_rng(w + h)
    g = B.geometry(w, h)
    n = 5000
    rects = _random_rects(rng, n, g)
    order = rng.permutation(n).astype(np.uint32)
    b = B.bin_frame(rects, order, w, h)
    x0, y0, x1, y1 = rects.astype(np.int64).T
    drawn = (x1 >= x0) & (y1 >= y0)
    # the total is the number of coarse tiles each drawn rect reaches
    per = ((x1 // 8 - x0 // 8 + 1) * (y1 // 4 - y0 // 4 + 1))[drawn]
    assert b.total == per.sum() == b.entries.size
    # every (tile, splat) instance appears exactly once, and every fine tile of every rect exactly once
    sid = (b.entries & np.uint64(0xFFFFFFFF)).astype(np.int64)
    mask = (b.entries >> np.uint64(32)).astype(np.int64)
    assert np.unique(b.tiles.astype(np.int64) * n + sid).size == b.total
    assert (mask != 0).all()
    bits = np.array([bin(int(m)).count("1") for m in mask])
    assert np.bincount(sid, weights=bits, minlength=n)[drawn].astype(np.int64).tolist() == ((x1 - x0 + 1) * (y1 - y0 + 1))[drawn].tolist()
    assert not np.isin(np.nonzero(~drawn)[0], sid).any()
    # lists are contiguous in tile-id order, each in draw order
    assert (np.diff(b.tiles.astype(np.int64)) >= 0).all()
    draw_rank = np.empty(n, np.int64)
    draw_rank[order[::-1]] = np.arange(n)
    r = draw_rank[sid]
    same = np.diff(b.tiles.astype(np.int64)) == 0
    assert (np.diff(r)[same] > 0).all()
    ranges = b.ranges(B.COUNTING)
    assert ranges[0, 0] == 0 and ranges[-1, 1] == b.total and (ranges[1:, 0] == ranges[:-1, 1]).all()
    order_t = b.tile_order(B.COUNTING)
    assert sorted(order_t.tolist()) == list(range(g.ncoarse))
    assert (np.diff(b.counts[order_t].astype(np.int64)) <= 0).all()


@pytest.mark.parametrize("world", [2, 3, 8])
def test_ranks_partition_the_single_rank_lists(world):
    w, h = 1921, 1080
    rng = np.random.default_rng(world)
    g = B.geometry(w, h)
    rects = _random_rects(rng, 3000, g)
    order = rng.permutation(3000).astype(np.uint32)
    whole = B.bin_frame(rects, order, w, h)
    parts = [B.bin_frame(rects, order, w, h, r, world) for r in range(world)]
    assert sum(p.total for p in parts) == whole.total
    for t in range(g.ncoarse):
        cx, cy = t % g.coarse_x, t // g.coarse_x
        for r, p in enumerate(parts):
            if (cx + cy) % world == r:
                assert np.array_equal(p.list_of(t), whole.list_of(t)), (t, r)
            else:
                assert p.counts[t] == 0, (t, r)
