"""CPU model of how k_raster (csrc/nr_raster.cu) lays its warp blocks over a tile and stages a face's pixel box.

A warp owns an 8x8 block (two pixels per lane: (l & 7, l >> 3) and four rows below) or, when the work is
small, an 8x4 block (the upper half only).  Two pieces of integer arithmetic decide which pixels a warp
evaluates, and no parity case reaches all of their corners:
  * the work item -> (tile, sub-block) -> block origin mapping (nr_raster.cu:140, :186-193): every pixel of
    every tile must be covered exactly once, for 16x16 and 8x8 tiles and both block heights;
  * the pixel-box bit masks (nr_raster.cu:250-256): one 32-bit word per 8x4 half, bit = lane.  The bits
    must be exactly the pixels of the box inside the block, and a half's word is zero iff the box misses
    that half (phase 1 skips the edge functions of that half on that condition).
The kernel itself is checked against the oracle on the GPU (test_gpu_raster_blocks.py)."""
import itertools

import pytest

BLK, HALF_H = 8, 4
M32 = 0xffffffff


def block_origins(tsz, tall):
    """nr_raster.cu:140, :186-191 -> [(tile item, sub, wx0, wy0)] of one tile at (0, 0)."""
    fine = tsz == 8
    bh = BLK if tall else HALF_H
    blk_shift = (0 if fine else 2) + (0 if tall else 1)
    out = []
    for item in range(1 << blk_shift):           # the items of tile 0
        sub = item & ((1 << blk_shift) - 1)
        wx0 = 0 if fine else (sub & 1) * BLK
        wy0 = (sub if fine else sub >> 1) * bh
        out.append((item >> blk_shift, sub, wx0, wy0))
    return out, bh


def lane_pixels(wx0, wy0, tall):
    """nr_raster.cu:193,195 and the epilogue (:337-338): the pixels lane l writes."""
    px = []
    for lane in range(32):
        xi, yi = wx0 + (lane & 7), wy0 + (lane >> 3)
        px.append((xi, yi))
        if tall:
            px.append((xi, yi + HALF_H))
    return px


@pytest.mark.parametrize("tsz,tall", list(itertools.product([16, 8], [True, False])))
def test_every_pixel_of_a_tile_is_one_lanes(tsz, tall):
    blocks, bh = block_origins(tsz, tall)
    assert len(blocks) == (tsz // BLK) * (tsz // bh)
    assert all(t == 0 for t, _, _, _ in blocks)
    seen = []
    for _, _, wx0, wy0 in blocks:
        seen += lane_pixels(wx0, wy0, tall)
    assert sorted(seen) == sorted((x, y) for x in range(tsz) for y in range(tsz))


def box_masks(bx0, bx1, by0, by1, bh):
    """nr_raster.cu:250-256 for a box given relative to the block origin (32-bit unsigned arithmetic)."""
    c0, c1 = max(bx0, 0), min(bx1, BLK - 1)
    r0, r1 = max(by0, 0), min(by1, bh - 1)
    cols = ((2 << c1) - 1) & ~((1 << c0) - 1) & M32
    rows = ((2 << r1) - 1) & ~((1 << r0) - 1) & M32
    upper = (cols * ((((rows & 15) * 0x00204081) & M32) & 0x01010101)) & M32
    lower = (cols * ((((rows >> 4) * 0x00204081) & M32) & 0x01010101)) & M32
    return upper, lower


@pytest.mark.parametrize("bh", [BLK, HALF_H])
def test_box_masks_are_exactly_the_box(bh):
    """Every box that survives the pixel-box cull (nr_raster.cu:226-227), corners up to two pixels outside
    the block on every side."""
    span = range(-2, BLK + 2)
    n = 0
    for bx0, bx1, by0, by1 in itertools.product(span, span, span, span):
        if bx0 > bx1 or by0 > by1 or bx0 > BLK - 1 or bx1 < 0 or by0 > bh - 1 or by1 < 0:
            continue
        upper, lower = box_masks(bx0, bx1, by0, by1, bh)
        want_u = want_l = 0
        for lane in range(32):
            x, y = lane & 7, lane >> 3
            inx = bx0 <= x <= bx1
            if inx and by0 <= y <= by1:
                want_u |= 1 << lane
            if inx and bh == BLK and by0 <= y + HALF_H <= by1:
                want_l |= 1 << lane
        assert (upper, lower) == (want_u, want_l), (bx0, bx1, by0, by1, bh)
        assert (upper == 0) == (by0 > HALF_H - 1)
        assert (lower == 0) == (bh == HALF_H or by1 < HALF_H)
        n += 1
    assert n == (sum(1 for a in span for b in span if a <= b and a <= BLK - 1 and b >= 0) *
                 sum(1 for a in span for b in span if a <= b and a <= bh - 1 and b >= 0))
