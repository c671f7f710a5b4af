"""Plain restatement of tile binning (DESIGN.md sections 4 and 6), for exact comparison with the engine's binning state.

Binning turns each drawn splat's fine-tile rect into per-coarse-tile lists of {fine mask, splat id} in draw order.  This module
states what those lists are from the definitions alone, in numpy, with no knowledge of how the kernels compute them:

* Tile geometry.  The fine-tile edge is 16 px while that gives at most 256 coarse tiles, otherwise 32 px.  A coarse tile is 8 x 4
  fine tiles; coarse tile (cx, cy) has id cy * coarse_x + cx.
* Path.  Frames of at most 256 coarse tiles are binned by a counting sort (GS_BIN >= 2, the default), all others by emitting the
  instances and radix-sorting them by tile id.  Both must produce the same lists.
* Lists.  Draw rank p (p = 0 first) draws splat order[render_count - 1 - p].  The list of a coarse tile holds, in increasing p, every
  draw rank whose non-empty rect reaches the tile; an entry is (fine mask << 32) | splat id, where bit 8 * fy + fx stands for fine
  tile (fx, fy) of the coarse tile.
* Sharding.  With world > 1 a rank keeps the coarse tiles with (cx + cy) % world == rank only.  Its lists are the GLOBAL draw order
  filtered this way, also when the rank sorted only its own subset of the splats.
* Derived values.  The lists are stored one after another in tile-id order, so `ranges` is the exclusive prefix sum of the list
  lengths and `total` their sum.  The two paths encode an EMPTY tile differently: the counting sort writes (start, start) like any
  other tile, the radix path leaves the initial (0xffffffff, 0).  The counting-sort path also schedules the blend by list length,
  longest first, ties to the lower tile id; the radix path keeps the identity schedule.
* Overflow.  Entries past the instance capacity are not stored; the counting-sort path clamps both ends of every range to the
  capacity (`ranges(..., capacity=)`), so a blend reads stored entries only.

Test infrastructure only: nothing under gaussiansplats3d_b200/ imports it, and it imports nothing from there.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

FINE_TILE_PX = (16, 32)
COARSE_W, COARSE_H = 8, 4                   # fine tiles per coarse tile
COUNTING_SORT_MAX_COARSE = 256
COUNTING, RADIX = 2, 1                      # binning paths, numbered like the engine's GS_BIN generations
EMPTY_RANGE = (0xFFFFFFFF, 0)               # the radix path's encoding of a tile without instances


@dataclass(frozen=True)
class Geometry:
    width: int
    height: int
    tile_px: int
    tiles_x: int
    tiles_y: int
    coarse_x: int
    coarse_y: int

    @property
    def ncoarse(self) -> int:
        return self.coarse_x * self.coarse_y

    @property
    def max_diagonal(self) -> int:
        return self.coarse_x - 1 + self.coarse_y - 1


def _ceil_div(a: int, b: int) -> int:
    return -(-a // b)


def geometry(width: int, height: int) -> Geometry:
    for px in FINE_TILE_PX:
        tx, ty = _ceil_div(width, px), _ceil_div(height, px)
        g = Geometry(width, height, px, tx, ty, _ceil_div(tx, COARSE_W), _ceil_div(ty, COARSE_H))
        if g.ncoarse <= COUNTING_SORT_MAX_COARSE:
            return g
    return g                                # 32 px: the largest fine tile, whatever the count


def binning_path(width: int, height: int, bin_version: int = 2) -> int:
    return COUNTING if bin_version >= 2 and geometry(width, height).ncoarse <= COUNTING_SORT_MAX_COARSE else RADIX


@dataclass
class Binning:
    geometry: Geometry
    tiles: np.ndarray       # u32 per instance, in list order
    entries: np.ndarray     # u64 per instance, in list order: (fine mask << 32) | splat id
    counts: np.ndarray      # u64 per coarse tile: list lengths

    @property
    def total(self) -> int:
        return int(self.counts.sum())

    def starts(self) -> np.ndarray:
        return np.cumsum(self.counts) - self.counts

    def ranges(self, path: int, capacity: int | None = None) -> np.ndarray:
        """u32 [ncoarse, 2] as the engine stores them after this frame."""
        start = self.starts()
        end = start + self.counts
        if capacity is not None:
            start, end = np.minimum(start, capacity), np.minimum(end, capacity)
        r = np.stack([start, end], 1).astype(np.uint32)
        if path == RADIX:
            r[self.counts == 0] = EMPTY_RANGE
        return r

    def tile_order(self, path: int) -> np.ndarray:
        ids = np.arange(self.geometry.ncoarse, dtype=np.int64)
        if path == RADIX:
            return ids.astype(np.uint32)
        return np.lexsort((ids, -self.counts.astype(np.int64))).astype(np.uint32)

    def list_of(self, tile: int) -> np.ndarray:
        s = int(self.starts()[tile])
        return self.entries[s:s + int(self.counts[tile])]


def fine_mask(fx0, fy0, fx1, fy1) -> np.ndarray:
    """Mask of the fine tiles [fx0, fx1] x [fy0, fy1] (coordinates inside one coarse tile): bit 8 * fy + fx."""
    fx0, fy0, fx1, fy1 = (np.asarray(a, np.int64) for a in (fx0, fy0, fx1, fy1))
    row = ((np.int64(1) << (fx1 - fx0 + 1)) - 1) << fx0
    mask = np.zeros(np.broadcast(fx0, fy0).shape, np.int64)
    for fy in range(COARSE_H):
        mask |= np.where((fy0 <= fy) & (fy <= fy1), row << (COARSE_W * fy), 0)
    return mask.astype(np.uint64)


def bin_frame(rects, order, width: int, height: int, rank: int = 0, world: int = 1) -> Binning:
    """The coarse-tile lists of one frame.  `rects`: u16 [n, 4] inclusive fine-tile rects {x0, y0, x1, y1} per splat (x1 < x0 or
    y1 < y0: not drawn); `order`: the draw order (its LAST element is drawn first), render_count = len(order)."""
    g = geometry(width, height)
    rects = np.asarray(rects).reshape(-1, 4).astype(np.int64)
    order = np.asarray(order, np.int64).reshape(-1)
    sid = order[::-1]                                    # sid[p] = splat of draw rank p
    rank_of = np.arange(sid.size, dtype=np.int64)
    x0, y0, x1, y1 = rects[sid].T
    drawn = (x1 >= x0) & (y1 >= y0)
    sid, rank_of, x0, y0, x1, y1 = sid[drawn], rank_of[drawn], x0[drawn], y0[drawn], x1[drawn], y1[drawn]
    # every coarse tile of every rect
    cx0, cx1, cy0, cy1 = x0 // COARSE_W, x1 // COARSE_W, y0 // COARSE_H, y1 // COARSE_H
    cw = cx1 - cx0 + 1
    per = cw * (cy1 - cy0 + 1)
    owner = np.repeat(np.arange(sid.size), per)
    k = np.arange(int(per.sum()), dtype=np.int64) - np.repeat(np.cumsum(per) - per, per)
    cx = cx0[owner] + k % cw[owner]
    cy = cy0[owner] + k // cw[owner]
    if world > 1:
        mine = (cx + cy) % world == rank
        owner, cx, cy = owner[mine], cx[mine], cy[mine]
    # the part of the rect inside each coarse tile, in that tile's fine coordinates
    bx, by = cx * COARSE_W, cy * COARSE_H
    mask = fine_mask(np.maximum(x0[owner], bx) - bx, np.maximum(y0[owner], by) - by,
                     np.minimum(x1[owner], bx + COARSE_W - 1) - bx, np.minimum(y1[owner], by + COARSE_H - 1) - by)
    tile = cy * g.coarse_x + cx
    at = np.lexsort((rank_of[owner], tile))              # by tile id, then draw rank
    tiles = tile[at].astype(np.uint32)
    entries = (mask[at] << np.uint64(32)) | sid[owner][at].astype(np.uint64)
    counts = np.bincount(tiles, minlength=g.ncoarse).astype(np.uint64)
    return Binning(g, tiles, entries, counts)
