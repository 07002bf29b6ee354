"""Region reads (``region.plan`` and the host-side checks of ``cae_tiles_crop_u8``): no device."""
import ctypes

import numpy as np
import pytest

from cnn_autoencoder_b200 import _cabi as C
from cnn_autoencoder_b200.region import plan


def _check_plan(shape, chunks, boxes, bh, bw):
    H, W = shape[:2]
    cy, cx = chunks[:2]
    chunk_yx, pieces = plan(shape, chunks, boxes, bh, bw)
    assert pieces.dtype == np.int32 and pieces.shape[1] == 8
    # distinct chunks in row-major order, pieces sorted by chunk
    lin = chunk_yx[:, 0] * (-(-W // cx)) + chunk_yx[:, 1]
    assert (np.diff(lin) > 0).all()
    assert (np.diff(pieces[:, 0]) >= 0).all()
    assert set(pieces[:, 0].tolist()) == set(range(len(chunk_yx)))
    # brute-force pixel map: every pixel of every box covered by exactly one piece, with the
    # right source pixel
    cover = np.zeros((len(boxes), bh, bw), dtype=np.int32)
    src_y = np.full((len(boxes), bh, bw), -1)
    src_x = np.full((len(boxes), bh, bw), -1)
    for k, b, sy, sx, dy, dx, h, w in pieces.tolist():
        iy, ix = chunk_yx[k]
        assert h > 0 and w > 0
        assert 0 <= sy and sy + h <= cy and 0 <= sx and sx + w <= cx          # inside its chunk
        assert iy * cy + sy + h <= H and ix * cx + sx + w <= W                # inside the array
        assert 0 <= dy and dy + h <= bh and 0 <= dx and dx + w <= bw          # inside its box
        cover[b, dy:dy + h, dx:dx + w] += 1
        src_y[b, dy:dy + h, dx:dx + w] = (iy * cy + sy + np.arange(h))[:, None]
        src_x[b, dy:dy + h, dx:dx + w] = (ix * cx + sx + np.arange(w))[None, :]
    assert (cover == 1).all()
    for b, (y, x) in enumerate(boxes):
        assert (src_y[b] == y + np.arange(bh)[:, None]).all()
        assert (src_x[b] == x + np.arange(bw)[None, :]).all()
    # the chunks listed are the ones the boxes touch
    touched = {(iy, ix) for (y, x) in boxes for iy in range(y // cy, (y + bh - 1) // cy + 1)
               for ix in range(x // cx, (x + bw - 1) // cx + 1)}
    assert touched == {tuple(t) for t in chunk_yx.tolist()}
    return chunk_yx, pieces


@pytest.mark.parametrize('seed', range(6))
def test_plan_covers_every_box_pixel_once(seed):
    rng = np.random.default_rng(seed)
    ps = int(rng.choice([16, 32, 64]))
    H = int(rng.integers(1, 9)) * ps + int(rng.integers(1, ps))              # ragged edges
    W = int(rng.integers(1, 9)) * ps + int(rng.integers(1, ps))
    bh, bw = int(rng.integers(1, min(H, 3 * ps))), int(rng.integers(1, min(W, 3 * ps)))
    n = int(rng.integers(1, 30))
    boxes = [(int(rng.integers(0, H - bh + 1)), int(rng.integers(0, W - bw + 1))) for _ in range(n)]
    boxes.append((H - bh, W - bw))                                            # the bottom-right edge
    chunk_yx, _ = _check_plan((H, W, 3), (ps, ps, 3), boxes, bh, bw)
    assert len(chunk_yx) == len({tuple(t) for t in chunk_yx.tolist()})


def test_plan_whole_array_and_single_chunk():
    chunk_yx, pieces = _check_plan((100, 70, 3), (32, 32, 3), [(0, 0)], 100, 70)
    assert len(chunk_yx) == 4 * 3 and len(pieces) == 12
    assert pieces[-1].tolist() == [11, 0, 0, 0, 96, 64, 4, 6]               # edge chunk: 4 x 6 px
    chunk_yx, pieces = _check_plan((100, 70, 3), (32, 32, 3), [(33, 40), (33, 40)], 10, 20)
    assert chunk_yx.tolist() == [[1, 1]] and pieces[:, 1].tolist() == [0, 1]


@pytest.mark.parametrize('box', [(-1, 0), (0, -1), (91, 0), (0, 61), (100, 70)])
def test_plan_refuses_boxes_outside_the_array(box):
    with pytest.raises(ValueError):
        plan((100, 70, 3), (32, 32, 3), [(0, 0), box], 10, 10)


def test_plan_refuses_empty_boxes():
    with pytest.raises(ValueError):
        plan((100, 70, 3), (32, 32, 3), [(0, 0)], 0, 10)
    with pytest.raises(ValueError):
        plan((100, 70, 3), (32, 32, 3), np.zeros((0, 2)), 4, 4)


# ---- cae_tiles_crop_u8: a bad piece table is refused on the host, before any copy or launch ----
# (the pointers below are never dereferenced: every call here fails its checks first)
_FAKE = ctypes.c_void_p(1 << 20)


def _crop(pieces, tiles=_FAKE, n_tiles=2, ps=16, c=3, pieces_dev=_FAKE, out=_FAKE, n_boxes=2,
          box_h=10, box_w=12):
    p = np.ascontiguousarray(np.asarray(pieces, dtype=np.int32).reshape(-1, 8))
    rc = C.lib().cae_tiles_crop_u8(tiles, n_tiles, ps, c, p.ctypes.data if len(p) else None,
                                   len(p), pieces_dev, out, n_boxes, box_h, box_w, None)
    return rc, C.lib().cae_last_error().decode()


GOOD = [0, 1, 2, 3, 0, 0, 10, 12]


@pytest.mark.parametrize('bad, what', [
    ([2, 0, 0, 0, 0, 0, 4, 4], 'tile 2 of 2'),               # tile index >= n_tiles
    ([-2, 0, 0, 0, 0, 0, 4, 4], 'tile -2'),
    ([0, 2, 0, 0, 0, 0, 4, 4], 'box 2 of 2'),
    ([0, 0, 10, 0, 0, 0, 7, 4], 'outside its 16^2 tile'),     # rows 10..17 of a 16-row tile
    ([0, 0, 0, 13, 0, 0, 4, 4], 'outside its 16^2 tile'),
    ([0, 0, -1, 0, 0, 0, 4, 4], 'outside its 16^2 tile'),
    ([0, 0, 0, 0, 0, 0, 0, 4], 'outside its 16^2 tile'),      # empty piece
    ([0, 0, 0, 0, 7, 0, 4, 4], 'outside its 10 x 12 box'),
    ([0, 0, 0, 0, 0, 9, 4, 4], 'outside its 10 x 12 box'),
    ([-1, 0, 0, 0, 0, -1, 4, 4], 'outside its 10 x 12 box'),  # fill pieces are checked too
])
def test_crop_refuses_a_bad_piece(bad, what):
    rc, msg = _crop([GOOD, bad])
    assert rc == 2 and 'piece 1' in msg and what in msg, msg


def test_crop_refuses_null_pointers():
    for kw in (dict(tiles=None), dict(pieces_dev=None), dict(out=None)):
        rc, msg = _crop([GOOD], **kw)
        assert rc == 2 and 'null pointer' in msg, (kw, msg)
    rc = C.lib().cae_tiles_crop_u8(_FAKE, 2, 16, 3, None, 1, _FAKE, _FAKE, 2, 10, 12, None)
    assert rc == 2 and 'null pointer' in C.lib().cae_last_error().decode()
    rc, msg = _crop([GOOD], pieces_dev=ctypes.c_void_p((1 << 20) + 4))
    assert rc == 2 and 'aligned' in msg
    rc, msg = _crop([GOOD], ps=0)
    assert rc == 2 and 'bad argument' in msg
