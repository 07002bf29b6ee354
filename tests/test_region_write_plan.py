"""Region writes (``region.write_plan``, ``region.check_disjoint`` and the host-side checks of
``cae_tiles_paste_u8``): no device."""
import ctypes

import numpy as np
import pytest

from cnn_autoencoder_b200 import _cabi as C
from cnn_autoencoder_b200.region import check_disjoint, write_plan


def _disjoint_boxes(rng, H, W, bh, bw, n):
    """Up to ``n`` random non-overlapping boxes (rejection sampling)."""
    taken = np.zeros((H, W), dtype=bool)
    boxes = []
    for _ in range(20 * n):
        y, x = int(rng.integers(0, H - bh + 1)), int(rng.integers(0, W - bw + 1))
        if not taken[y:y + bh, x:x + bw].any():
            taken[y:y + bh, x:x + bw] = True
            boxes.append((y, x))
            if len(boxes) == n:
                break
    return boxes


def _check_write_plan(shape, chunks, boxes, bh, bw):
    """Brute-force pixel map of every touched chunk: each pixel is exactly one of written from
    box b at the right offset, zero padding, or kept from the old tile."""
    H, W = shape[:2]
    cy, cx = chunks[:2]
    chunk_yx, pieces, full, fill = write_plan(shape, chunks, boxes, bh, bw)
    assert pieces.dtype == np.int32 and fill.dtype == np.int32 and full.dtype == bool
    assert fill.shape[1] == 8 and (fill[:, 1] == -1).all() and (pieces[:, 1] >= 0).all()
    K = len(chunk_yx)
    hits = np.zeros((K, cy, cx), dtype=np.int32)
    src = np.full((K, cy, cx, 3), -1)                # (box, y, x) each tile pixel is written from
    for k, b, sy, sx, dy, dx, h, w in pieces.tolist():
        hits[k, sy:sy + h, sx:sx + w] += 1
        src[k, sy:sy + h, sx:sx + w, 0] = b
        src[k, sy:sy + h, sx:sx + w, 1] = (dy + np.arange(h))[:, None]
        src[k, sy:sy + h, sx:sx + w, 2] = (dx + np.arange(w))[None, :]
    for k, b, sy, sx, dy, dx, h, w in fill.tolist():
        assert 0 <= k < K and h > 0 and w > 0
        assert 0 <= sy and sy + h <= cy and 0 <= sx and sx + w <= cx
        hits[k, sy:sy + h, sx:sx + w] += 1
    assert hits.max() <= 1                                    # pieces are disjoint
    boxes_a = np.asarray(boxes)
    for k, (iy, ix) in enumerate(chunk_yx.tolist()):
        gy = iy * cy + np.arange(cy)[:, None]                 # array coordinates of the tile
        gx = ix * cx + np.arange(cx)[None, :]
        inside = (gy < H) & (gx < W)
        # padding is exactly what lies beyond the array edge, and it is zero-filled
        assert (hits[k][~inside] == 1).all() and (src[k, ..., 0][~inside] == -1).all()
        written = np.zeros((cy, cx), dtype=bool)
        for b, (y, x) in enumerate(boxes_a.tolist()):
            m = inside & (gy >= y) & (gy < y + bh) & (gx >= x) & (gx < x + bw)
            written |= m
            assert (src[k, ..., 0][m] == b).all()
            assert (src[k, ..., 1][m] == (gy - y + 0 * gx)[m]).all()
            assert (src[k, ..., 2][m] == (gx - x + 0 * gy)[m]).all()
        assert (hits[k][inside & ~written] == 0).all()        # kept from the old tile
        assert written.any()
        assert full[k] == (written == inside).all()
    return chunk_yx, pieces, full, fill


@pytest.mark.parametrize('seed', range(8))
def test_write_plan_pixel_map(seed):
    rng = np.random.default_rng(seed)
    ps = int(rng.choice([16, 32]))
    H = int(rng.integers(1, 7)) * ps + int(rng.integers(0, ps))             # ragged or exact
    W = int(rng.integers(1, 7)) * ps + int(rng.integers(0, ps))
    bh, bw = int(rng.integers(1, min(H, 2 * ps) + 1)), int(rng.integers(1, min(W, 2 * ps) + 1))
    boxes = _disjoint_boxes(rng, H, W, bh, bw, int(rng.integers(1, 12)))
    _check_write_plan((H, W, 3), (ps, ps, 3), boxes, bh, bw)


def test_write_plan_full_and_partial():
    # 100 x 70 in 32^2 chunks: 4 x 3 chunks, the last row 4 px tall, the last column 6 px wide
    chunk_yx, _, full, fill = _check_write_plan((100, 70, 3), (32, 32, 3), [(0, 0)], 100, 70)
    assert full.all() and len(chunk_yx) == 12
    # edge chunks: 3 below-the-edge pieces (bottom row) + 4 right-of-the-edge pieces (right column)
    assert len(fill) == 3 + 4
    assert [9, -1, 4, 0, 0, 0, 28, 32] in fill.tolist()                   # chunk (3, 0)
    assert [11, -1, 0, 6, 0, 0, 4, 26] in fill.tolist()                   # chunk (3, 2)
    # a strip of whole chunk rows: full; a window inside one chunk: partial
    _, _, full, _ = _check_write_plan((100, 70, 3), (32, 32, 3), [(32, 0)], 64, 70)
    assert full.all()
    chunk_yx, _, full, fill = _check_write_plan((100, 70, 3), (32, 32, 3), [(33, 40)], 10, 20)
    assert chunk_yx.tolist() == [[1, 1]] and full.tolist() == [False] and len(fill) == 0
    # the edge chunk (3, 2) is full once its 4 x 6 in-array pixels are written
    chunk_yx, _, full, fill = _check_write_plan((100, 70, 3), (32, 32, 3), [(96, 64)], 4, 6)
    assert chunk_yx.tolist() == [[3, 2]] and full.tolist() == [True] and len(fill) == 2
    # several boxes together cover a chunk
    _, _, full, _ = _check_write_plan((100, 70, 3), (32, 32, 3), [(0, 0), (16, 0), (0, 16), (16, 16)],
                                      16, 16)
    assert full.tolist() == [True]


@pytest.mark.parametrize('boxes, bh, bw', [
    ([(0, 0), (0, 0)], 4, 4),                  # the same box twice
    ([(0, 0), (3, 3)], 4, 4),                  # one corner pixel shared
    ([(10, 0), (0, 5), (13, 2)], 4, 4),
    ([(0, 0), (50, 60), (0, 9), (2, 10)], 3, 10),
])
def test_overlapping_boxes_are_refused(boxes, bh, bw):
    with pytest.raises(ValueError, match='overlap'):
        check_disjoint(boxes, bh, bw)
    with pytest.raises(ValueError, match='overlap'):
        write_plan((100, 70, 3), (32, 32, 3), boxes, bh, bw)


def test_touching_boxes_are_accepted():
    check_disjoint([(0, 0), (0, 4), (4, 0), (4, 4)], 4, 4)
    rng = np.random.default_rng(5)
    boxes = _disjoint_boxes(rng, 300, 300, 7, 9, 200)
    check_disjoint(boxes, 7, 9)
    # against a brute-force pairwise check
    for _ in range(20):
        bx = [(int(rng.integers(0, 40)), int(rng.integers(0, 40))) for _ in range(12)]
        a = np.asarray(bx)
        clash = any(abs(a[i, 0] - a[j, 0]) < 5 and abs(a[i, 1] - a[j, 1]) < 6
                    for i in range(len(a)) for j in range(i))
        if clash:
            with pytest.raises(ValueError):
                check_disjoint(bx, 5, 6)
        else:
            check_disjoint(bx, 5, 6)


# ---- cae_tiles_paste_u8: a bad piece table is refused on the host, before any copy or launch ----
# (the pointers below are never dereferenced: every call here fails its checks first)
_FAKE = ctypes.c_void_p(1 << 20)


def _paste(pieces, tiles=_FAKE, n_tiles=2, ps=16, c=3, pieces_dev=_FAKE, boxes=_FAKE, n_boxes=2,
           box_h=10, box_w=12):
    p = np.ascontiguousarray(np.asarray(pieces, dtype=np.int32).reshape(-1, 8))
    rc = C.lib().cae_tiles_paste_u8(tiles, n_tiles, ps, c, p.ctypes.data if len(p) else None,
                                    len(p), pieces_dev, boxes, n_boxes, box_h, box_w, None)
    return rc, C.lib().cae_last_error().decode()


GOOD = [0, 1, 2, 3, 0, 0, 10, 12]


@pytest.mark.parametrize('bad, what', [
    ([2, 0, 0, 0, 0, 0, 4, 4], 'tile 2 of 2'),               # tile index >= n_tiles
    ([-1, 0, 0, 0, 0, 0, 4, 4], 'tile -1'),                  # a paste always names a tile
    ([0, 2, 0, 0, 0, 0, 4, 4], 'box 2 of 2'),
    ([0, -2, 0, 0, 0, 0, 4, 4], 'box -2'),
    ([0, 0, 10, 0, 0, 0, 7, 4], 'outside its 16^2 tile'),     # rows 10..17 of a 16-row tile
    ([0, 0, 0, 13, 0, 0, 4, 4], 'outside its 16^2 tile'),
    ([0, 0, -1, 0, 0, 0, 4, 4], 'outside its 16^2 tile'),
    ([0, 0, 0, 0, 0, 0, 0, 4], 'outside its 16^2 tile'),      # empty piece
    ([0, -1, 0, 10, 0, 0, 4, 7], 'outside its 16^2 tile'),    # fill pieces are checked in the tile
    ([0, 0, 0, 0, 7, 0, 4, 4], 'outside its 10 x 12 box'),
    ([0, 0, 0, 0, 0, 9, 4, 4], 'outside its 10 x 12 box'),
    ([0, 0, 0, 0, -1, 0, 4, 4], 'outside its 10 x 12 box'),
])
def test_paste_refuses_a_bad_piece(bad, what):
    rc, msg = _paste([GOOD, bad])
    assert rc == 2 and 'cae_tiles_paste_u8' in msg and 'piece 1' in msg and what in msg, msg


def test_paste_fill_pieces_need_no_box():
    # a fill piece larger than the boxes passes its checks (it reads no box): the error names
    # the bad second piece
    rc, msg = _paste([[0, -1, 0, 0, 0, 0, 16, 16], [0, 0, 0, 0, 0, 0, 0, 1]])
    assert rc == 2 and 'piece 1' in msg, msg


def test_paste_refuses_null_pointers():
    for kw in (dict(tiles=None), dict(pieces_dev=None), dict(boxes=None)):
        rc, msg = _paste([GOOD], **kw)
        assert rc == 2 and 'null pointer' in msg, (kw, msg)
    rc = C.lib().cae_tiles_paste_u8(_FAKE, 2, 16, 3, None, 1, _FAKE, _FAKE, 2, 10, 12, None)
    assert rc == 2 and 'null pointer' in C.lib().cae_last_error().decode()
    rc, msg = _paste([GOOD], pieces_dev=ctypes.c_void_p((1 << 20) + 4))
    assert rc == 2 and 'aligned' in msg
    rc, msg = _paste([GOOD], ps=0)
    assert rc == 2 and 'bad argument' in msg
