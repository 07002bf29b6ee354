"""Reduced-resolution region reads (``region.reduce_plan``, the level geometry, the reduction's
oracles and the host-side checks of ``cae_tiles_crop_reduce_u8``): no device."""
import ctypes

import numpy as np
import pytest
from PIL import Image

from cnn_autoencoder_b200 import _cabi as C
from cnn_autoencoder_b200.region import check_factor, level_shape, plan, reduce_plan


def reduce_ref(img, f):
    """The level-``f`` image of ``img`` (Y x X x c uint8): block means over the pixels inside
    the array, rounded half up."""
    Y, X, c = img.shape
    ly, lx = -(-Y // f), -(-X // f)
    pad = np.zeros((ly * f, lx * f, c), dtype=np.int64)
    pad[:Y, :X] = img
    s = pad.reshape(ly, f, lx, f, c).sum(axis=(1, 3))
    n = (np.minimum(f, Y - f * np.arange(ly))[:, None] * np.minimum(f, X - f * np.arange(lx)))[..., None]
    return ((s + n // 2) // n).astype(np.uint8)


def _definition(img, f):
    """The definition, pixel by pixel."""
    Y, X, c = img.shape
    out = np.zeros((-(-Y // f), -(-X // f), c), dtype=np.uint8)
    for i in range(out.shape[0]):
        for j in range(out.shape[1]):
            blk = img[i * f:min((i + 1) * f, Y), j * f:min((j + 1) * f, X)].astype(np.int64)
            n = blk.shape[0] * blk.shape[1]
            out[i, j] = (blk.sum(axis=(0, 1)) + n // 2) // n
    return out


# ---- level geometry ----
@pytest.mark.parametrize('seed', range(8))
def test_level_plan_names_the_level0_chunks(seed):
    rng = np.random.default_rng(seed)
    ps = int(rng.choice([16, 32, 64]))
    f = int(rng.choice([f for f in (1, 2, 4, 8, 16, 32, 64) if f <= ps]))
    # ragged edges: neither Y nor X a multiple of f (when f > 1) or of ps
    Y = int(rng.integers(1, 7)) * ps + int(rng.integers(1, ps))
    X = int(rng.integers(1, 7)) * ps + int(rng.integers(1, ps))
    if f > 1:
        Y += 1 if Y % f == 0 else 0
        X += 1 if X % f == 0 else 0
    shape = (Y, X, 3)
    ly, lx, c = level_shape(shape, f)
    assert (ly, lx, c) == (-(-Y // f), -(-X // f), 3)
    lc = ps // f
    # the level image in chunks of ps/f has the level-0 chunk grid
    assert (-(-ly // lc), -(-lx // lc)) == (-(-Y // ps), -(-X // ps))
    bh, bw = int(rng.integers(1, ly + 1)), int(rng.integers(1, lx + 1))
    boxes = [(int(rng.integers(0, ly - bh + 1)), int(rng.integers(0, lx - bw + 1))) for _ in range(12)]
    boxes.append((ly - bh, lx - bw))                                         # the ragged corner
    chunk_yx, pieces = reduce_plan(shape, ps, f, boxes, bh, bw)
    assert pieces.dtype == np.int32 and pieces.shape[1] == 12
    # the chunks are the level-0 chunks under the boxes' level-0 footprints (clipped to the array)
    want = {(iy, ix) for y, x in boxes
            for iy in range(y * f // ps, (min((y + bh) * f, Y) - 1) // ps + 1)
            for ix in range(x * f // ps, (min((x + bw) * f, X) - 1) // ps + 1)}
    assert {tuple(t) for t in chunk_yx.tolist()} == want
    # the first 8 columns are plan's in level pixels; then the chunk's in-array extent
    c8, p8 = plan((ly, lx, 3), (lc, lc, 3), boxes, bh, bw)
    assert np.array_equal(c8, chunk_yx) and np.array_equal(pieces[:, :8], p8)
    iy, ix = chunk_yx[pieces[:, 0], 0], chunk_yx[pieces[:, 0], 1]
    assert np.array_equal(pieces[:, 8], np.minimum(ps, Y - iy * ps))
    assert np.array_equal(pieces[:, 9], np.minimum(ps, X - ix * ps))
    assert not pieces[:, 10:].any()
    k, b, sy, sx, dy, dx, h, w, vh, vw = pieces[:, :10].T.astype(np.int64)
    # every piece lies in its chunk's level grid and starts inside the in-array part
    assert (sy + h <= lc).all() and (sx + w <= lc).all()
    assert ((sy + h - 1) * f < vh).all() and ((sx + w - 1) * f < vw).all()


def test_level_shapes_and_one_chunk_per_level_pixel():
    assert level_shape((100, 70, 3), 1) == (100, 70, 3)
    assert level_shape((100, 70, 3), 4) == (25, 18, 3)
    assert level_shape((100, 70, 1), 64) == (2, 2, 1)
    chunk_yx, pieces = reduce_plan((100, 70, 3), 32, 4, [(0, 0)], 25, 18)
    assert len(chunk_yx) == 4 * 3
    # the bottom-right chunk holds 4 x 6 level-0 pixels: 1 x 2 level pixels, partly covered blocks
    assert pieces[-1].tolist() == [11, 0, 0, 0, 24, 16, 1, 2, 4, 6, 0, 0]


@pytest.mark.parametrize('f, ps', [(3, 64), (0, 64), (-2, 64), (6, 48), (128, 64), (32, 48),
                                   (1.0, 64), (True, 64), ('2', 64)])
def test_bad_factors_are_refused(f, ps):
    with pytest.raises(ValueError):
        check_factor(f, ps)
    with pytest.raises(ValueError):
        reduce_plan((100, 70, 3), ps, f, [(0, 0)], 1, 1)


def test_boxes_outside_the_level_image_are_refused():
    with pytest.raises(ValueError):
        reduce_plan((100, 70, 3), 32, 4, [(0, 0)], 26, 18)
    with pytest.raises(ValueError):
        reduce_plan((100, 70, 3), 32, 4, [(24, 17)], 1, 2)


# ---- oracles ----
@pytest.mark.parametrize('c', [1, 3])
def test_numpy_reduction_is_the_definition_and_agrees_with_pil(c):
    rng = np.random.default_rng(40 + c)
    for f in (1, 2, 4, 8, 16, 32, 64):
        Y, X = 3 * f + int(rng.integers(1, f + 1)), 2 * f + int(rng.integers(1, f + 1))
        img = rng.integers(0, 256, size=(Y, X, c), dtype=np.uint8)
        want = reduce_ref(img, f)
        assert np.array_equal(want, _definition(img, f)), f
        pil = np.asarray(Image.fromarray(img[..., 0] if c == 1 else img).reduce(f))
        pil = pil.reshape(want.shape)
        full_y, full_x = Y // f, X // f
        # exact on every full block, within 1 on the partial edge blocks
        assert np.array_equal(pil[:full_y, :full_x], want[:full_y, :full_x]), f
        assert np.abs(pil.astype(int) - want).max() <= 1, f


def test_rounding_is_half_up():
    img = np.array([[[1], [2]], [[2], [2]]], dtype=np.uint8)       # 7 / 4 = 1.75 -> 2
    assert reduce_ref(img, 2).ravel().tolist() == [2]
    img = np.array([[[1], [2]]], dtype=np.uint8)                   # 3 / 2 = 1.5 -> 2
    assert reduce_ref(img, 2).ravel().tolist() == [2]
    img = np.array([[[0], [1]], [[0], [0]]], dtype=np.uint8)       # 1 / 4 -> 0
    assert reduce_ref(img, 2).ravel().tolist() == [0]


# ---- cae_tiles_crop_reduce_u8: a bad call is refused on the host, before any copy or launch ----
# (the pointers below are never dereferenced: every call here fails its checks first)
_FAKE = ctypes.c_void_p(1 << 20)


def _reduce(pieces, tiles=_FAKE, n_tiles=2, ps=16, c=3, f=2, pieces_dev=_FAKE, out=_FAKE, n_boxes=2,
            box_h=6, box_w=7):
    p = np.ascontiguousarray(np.asarray(pieces, dtype=np.int32).reshape(-1, 12))
    rc = C.lib().cae_tiles_crop_reduce_u8(tiles, n_tiles, ps, c, f, p.ctypes.data if len(p) else None,
                                          len(p), pieces_dev, out, n_boxes, box_h, box_w, None)
    return rc, C.lib().cae_last_error().decode()


# rows 2..6 x columns 3..7 of tile 0's 8 x 8 level grid (ps 16, f 2) to (0, 0) of box 1 (6 x 7)
GOOD = [0, 1, 2, 3, 0, 0, 5, 5, 16, 16, 0, 0]


@pytest.mark.parametrize('f, ps', [(3, 16), (0, 16), (-2, 16), (32, 16), (16, 24), (1024, 1024)])
def test_reduce_refuses_a_bad_factor(f, ps):
    rc, msg = _reduce([GOOD], f=f, ps=ps)
    assert rc == 2 and 'cae_tiles_crop_reduce_u8' in msg and 'factor %d' % f in msg, msg


@pytest.mark.parametrize('bad, what', [
    ([2, 0, 0, 0, 0, 0, 4, 4, 16, 16, 0, 0], 'tile 2 of 2'),
    ([-2, 0, 0, 0, 0, 0, 4, 4, 16, 16, 0, 0], 'tile -2'),
    ([0, 2, 0, 0, 0, 0, 4, 4, 16, 16, 0, 0], 'box 2 of 2'),
    ([0, -1, 0, 0, 0, 0, 4, 4, 16, 16, 0, 0], 'box -1'),
    ([0, 0, 5, 0, 0, 0, 4, 4, 16, 16, 0, 0], 'outside its 8^2 level tile'),   # level rows 5..8
    ([0, 0, 0, 6, 0, 0, 4, 4, 16, 16, 0, 0], 'outside its 8^2 level tile'),
    ([0, 0, 0, 0, 0, 0, 0, 4, 16, 16, 0, 0], 'outside its 8^2 level tile'),   # empty piece
    ([0, 0, 0, 0, 0, 0, 4, 4, 17, 16, 0, 0], 'in-array extent 17 x 16'),     # vh > ps
    ([0, 0, 0, 0, 0, 0, 4, 4, 16, 0, 0, 0], 'in-array extent 16 x 0'),
    ([0, 0, 0, 0, 0, 0, 4, 4, 6, 16, 0, 0], 'past the in-array part 6 x 16'),  # level row 3 = rows 6, 7
    ([0, 0, 0, 2, 0, 0, 2, 3, 16, 8, 0, 0], 'past the in-array part 16 x 8'),  # level column 4 = 8, 9
    ([-1, 0, 0, 0, 0, 0, 4, 4, 6, 16, 0, 0], 'past the in-array part'),       # fill pieces too
    ([0, 0, 0, 0, 3, 0, 4, 4, 16, 16, 0, 0], 'outside its 6 x 7 box'),
    ([0, 0, 0, 0, 0, 4, 4, 4, 16, 16, 0, 0], 'outside its 6 x 7 box'),
    ([0, 0, 0, 0, -1, 0, 4, 4, 16, 16, 0, 0], 'outside its 6 x 7 box'),
])
def test_reduce_refuses_a_bad_piece(bad, what):
    rc, msg = _reduce([GOOD, bad])
    assert rc == 2 and 'cae_tiles_crop_reduce_u8' in msg and 'piece 1' in msg and what in msg, msg


def test_reduce_accepts_a_partial_last_block():
    # level row 2 of a chunk with 5 in-array rows covers row 4 only: valid; the call then fails
    # on the next piece, which proves the first passed its checks
    rc, msg = _reduce([[0, 0, 0, 0, 0, 0, 3, 3, 5, 5, 0, 0], [0, 0, 0, 0, 0, 0, 0, 1, 16, 16, 0, 0]])
    assert rc == 2 and 'piece 1' in msg, msg


def test_reduce_refuses_null_pointers_misalignment_and_wide_pixels():
    for kw in (dict(tiles=None), dict(pieces_dev=None), dict(out=None)):
        rc, msg = _reduce([GOOD], **kw)
        assert rc == 2 and 'null pointer' in msg, (kw, msg)
    rc = C.lib().cae_tiles_crop_reduce_u8(_FAKE, 2, 16, 3, 2, None, 1, _FAKE, _FAKE, 2, 6, 7, None)
    assert rc == 2 and 'null pointer' in C.lib().cae_last_error().decode()
    rc, msg = _reduce([GOOD], pieces_dev=ctypes.c_void_p((1 << 20) + 4))
    assert rc == 2 and 'aligned' in msg
    rc, msg = _reduce([GOOD], ps=0)
    assert rc == 2 and 'bad argument' in msg
    rc, msg = _reduce([GOOD], ps=512, f=512, c=32)
    assert rc == 2 and 'too wide' in msg
