"""Reduced-resolution region reads (``CompressedSlide.downsampled``, ``cae_tiles_crop_reduce_u8``)
against the numpy reduction of what decompress_image writes: a 12 x 13-chunk slide at PS = 64 with
40 px and 24 px edge chunks, compared byte for byte at every factor from 1 to 64."""
import ctypes
import os
import shutil

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ARCH = dict(channels_org=3, channels_net=32, channels_bn=16, compression_level=3,
            act_layer_type='LeakyReLU')
PS = 64
FACTORS = [1, 2, 4, 8, 16, 32, 64]


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


@pytest.fixture(scope='module')
def store(tmp_path_factory):
    """(store path, checkpoint, decompress_image's reconstruction of the whole slide)."""
    from oracle import cae_oracle as O
    from cnn_autoencoder_b200 import compress, decompress
    chk = O.make_checkpoint(ARCH, seed=9)
    s = np.concatenate([np.concatenate([O.synth_tissue_tile(i, j, ps=PS, seed=2) for j in range(13)],
                                       axis=1) for i in range(12)], axis=0)
    slide = np.ascontiguousarray(s[:12 * PS - 24, :13 * PS - 40])
    path = str(tmp_path_factory.mktemp('region_reduce') / 'slide.zarr')
    compress.compress_image('CAE', chk, slide, path, patch_size=PS, batch_tiles=16, coder_tiles=96)
    canvas = torch.zeros(slide.shape, dtype=torch.uint8).pin_memory().numpy()
    decompress.decompress_image(path, canvas, checkpoint=chk, batch_tiles=16, coder_tiles=96)
    assert np.unique(canvas).size > 16
    return path, chk, canvas


@pytest.fixture(scope='module')
def reader(store):
    from cnn_autoencoder_b200.region import CompressedSlide
    path, chk, _ = store
    with CompressedSlide(path, chk, batch_tiles=16) as r:
        yield r


@pytest.fixture(scope='module')
def levels(store):
    _, _, canvas = store
    return {f: reduce_ref(canvas, f) for f in FACTORS}


def _touched(shape, f, boxes, h, w):
    """Level-0 chunks under the level-0 footprints of level boxes."""
    Y, X = shape[:2]
    return {(iy, ix) for y, x in boxes
            for iy in range(y * f // PS, (min((y + h) * f, Y) - 1) // PS + 1)
            for ix in range(x * f // PS, (min((x + w) * f, X) - 1) // PS + 1)}


@pytest.mark.parametrize('f', FACTORS)
def test_windows_equal_the_reduction(store, reader, levels, f):
    _, _, canvas = store
    want = levels[f]
    ly, lx, c = want.shape
    lc = PS // f
    view = reader.downsampled(f)
    assert view.shape == want.shape and view.chunks == (lc, lc, 3) and view.dtype == np.uint8
    assert view.downsample == f
    d, e = max(1, lc // 4), max(1, lc // 3)
    for y, x, h, w in [(lc + lc // 4, 2 * lc + lc // 4, max(1, lc // 2), max(1, lc // 2)),  # one chunk
                       (3 * lc - d, 5 * lc - e, 2 * d, 2 * e),                     # a 2 x 2 corner
                       (ly - min(ly, lc + 1), lx - min(lx, lc + 2), min(ly, lc + 1),
                        min(lx, lc + 2)),                                          # ragged edge
                       (0, 0, ly, lx)]:                                            # the whole level
        got = view.read_region(y, x, h, w)
        assert got.is_cuda and tuple(got.shape) == (h, w, c)
        assert np.array_equal(got.cpu().numpy(), want[y:y + h, x:x + w]), (f, y, x, h, w)
        assert reader.stats['decoded'] == reader.stats['chunks'] == \
            len(_touched(canvas.shape, f, [(y, x)], h, w))


@pytest.mark.parametrize('f', FACTORS)
def test_patch_batch_equals_the_reduction(store, reader, levels, f):
    _, _, canvas = store
    want = levels[f]
    ly, lx, _ = want.shape
    h, w = min(ly, 48 // f + 1), min(lx, 40 // f + 1)
    rng = np.random.default_rng(70 + f)
    boxes = [(int(rng.integers(0, ly - h + 1)), int(rng.integers(0, lx - w + 1))) for _ in range(200)]
    got = reader.downsampled(f).read_regions(boxes, h, w)
    assert tuple(got.shape) == (200, h, w, 3)
    assert np.array_equal(got.cpu().numpy(), np.stack([want[y:y + h, x:x + w] for y, x in boxes]))
    assert reader.stats['decoded'] == len(_touched(canvas.shape, f, boxes, h, w))


@pytest.mark.parametrize('f', [4, 16])
def test_getitem_follows_numpy_slicing(reader, levels, f):
    want = levels[f]
    view = reader.downsampled(f)
    keys = [(slice(3, 30), slice(5, 40)), (slice(-10, None), slice(-7, None)), (5, slice(2, 9)),
            (slice(2, 9), 5), (-1, -1), (slice(None), slice(None)), slice(4, 11), 3,
            (slice(20, 10), slice(None)), (slice(1, 4), slice(6, 9), slice(None)),
            (slice(-2000, 3), slice(None, -3)), (slice(0, 1000), -2)]
    for key in keys:
        got = view[key]
        assert isinstance(got, np.ndarray) and got.shape == want[key].shape, key
        assert np.array_equal(got, want[key]), key
    for bad in [(slice(0, 10, 2), slice(None)), (10 ** 6, 0), (slice(None), slice(None), 0), 1.5]:
        with pytest.raises(IndexError):
            view[bad]


def test_out_arguments(reader, levels):
    want = levels[8]
    view = reader.downsampled(8)
    y, x, h, w = 10, 13, 30, 41
    dev = torch.full((h, w, 3), 5, dtype=torch.uint8, device='cuda')
    assert view.read_region(y, x, h, w, out=dev) is dev
    assert np.array_equal(dev.cpu().numpy(), want[y:y + h, x:x + w])
    host = np.zeros((h, w, 3), dtype=np.uint8)
    assert view.read_region(y, x, h, w, out=host) is host
    assert np.array_equal(host, want[y:y + h, x:x + w])
    with pytest.raises(ValueError):
        view.read_region(y, x, h, w, out=torch.empty((h, w + 1, 3), dtype=torch.uint8, device='cuda'))
    with pytest.raises(ValueError):
        view.read_region(want.shape[0] - 3, 0, 4, 4)


def test_missing_chunk_reads_as_zeros(store, tmp_path):
    from cnn_autoencoder_b200.region import CompressedSlide
    path, chk, canvas = store
    i, j = 5, 6
    assert canvas[i * PS:(i + 1) * PS, j * PS:(j + 1) * PS].any()
    copy = str(tmp_path / 'holey.zarr')
    shutil.copytree(path, copy)
    os.remove(os.path.join(copy, '0/0', '%d.%d.0' % (i, j)))
    holey = canvas.copy()
    holey[i * PS:(i + 1) * PS, j * PS:(j + 1) * PS] = 0
    with CompressedSlide(copy, chk) as r:
        for f in (4, 64):
            assert np.array_equal(r.downsampled(f)[:, :], reduce_ref(holey, f)), f
            assert r.stats['missing'] == 1 and r.stats['decoded'] == 155
        lc = PS // 4                                       # a window across the hole's top edge
        y, x = i * lc - 3, j * lc + 2
        win = r.downsampled(4).read_region(y, x, 8, 10).cpu().numpy()
        assert r.stats['missing'] == 1 and r.stats['decoded'] == 1
        assert np.array_equal(win, reduce_ref(holey, 4)[y:y + 8, x:x + 10]) and not win[3:].any()


def test_device_and_host_coder_give_the_same_bytes(store, levels):
    from cnn_autoencoder_b200.region import CompressedSlide
    path, chk, _ = store
    rng = np.random.default_rng(13)
    with CompressedSlide(path, chk, batch_tiles=8) as r:
        got = {}
        for name, threshold in (('device', 1), ('host', 10 ** 9)):
            r.fact_ent.GPU_CODER_MIN_STREAMS = threshold       # instance override, this reader only
            got[name] = []
            for f in (2, 8, 32):
                ly, lx, _ = levels[f].shape
                boxes = [(int(rng.integers(0, ly - 3)), int(rng.integers(0, lx - 5))) for _ in range(40)]
                got[name].append((boxes, r.downsampled(f).read_regions(boxes, 3, 5).cpu().numpy(),
                                  r.downsampled(f)[:, :]))
                st = r.stats
                assert st['device_decoded'] == (st['decoded'] if name == 'device' else 0)
    for name in got:
        for f, (boxes, patches, whole) in zip((2, 8, 32), got[name]):
            assert np.array_equal(whole, levels[f]), (name, f)
            assert np.array_equal(patches, np.stack([levels[f][y:y + 3, x:x + 5] for y, x in boxes]))


def test_factor_one_is_the_level0_read(store, reader):
    _, _, canvas = store
    view = reader.downsampled(1)
    assert view.shape == canvas.shape and view.chunks == reader.chunks and view.downsample == 1
    y, x, h, w = 3 * PS - 20, 5 * PS - 30, 50, 70
    assert torch.equal(view.read_region(y, x, h, w), reader.read_region(y, x, h, w))
    boxes = [(0, 0), (100, 200), (canvas.shape[0] - 33, canvas.shape[1] - 21)]
    assert torch.equal(view.read_regions(boxes, 33, 21), reader.read_regions(boxes, 33, 21))
    assert np.array_equal(view[-40:, 100:140], reader[-40:, 100:140])


def test_views_are_read_only_and_refuse_bad_factors(reader):
    for f in (0, 3, 6, 128, -2, 2.0):
        with pytest.raises(ValueError):
            reader.downsampled(f)
    for f in (1, 4):
        view = reader.downsampled(f)
        with pytest.raises(TypeError, match='read-only'):
            view[0:4, 0:4] = 0


def test_reduced_reads_see_the_readers_writes(store, tmp_path):
    from cnn_autoencoder_b200.region import CompressedSlide
    path, chk, canvas = store
    copy = str(tmp_path / 'written.zarr')
    shutil.copytree(path, copy)
    with CompressedSlide(copy, chk, mode='r+') as r:
        before = r.downsampled(4)[:, :]
        # a partly covered window across four chunks, and a whole chunk
        r[2 * PS - 30:2 * PS + 50, 3 * PS - 20:3 * PS + 60] = 0
        r[6 * PS:7 * PS, 8 * PS:9 * PS] = np.full((PS, PS, 3), 230, dtype=np.uint8)
        full = r[:, :]
        for f in (4, 16):
            after = r.downsampled(f)[:, :]
            assert np.array_equal(after, reduce_ref(full, f)), f
        after = r.downsampled(4)[:, :]
        assert not np.array_equal(after, before)
        assert (after[(2 * PS - 28) // 4:(2 * PS + 48) // 4, (3 * PS - 16) // 4:(3 * PS + 60) // 4]
                != before[(2 * PS - 28) // 4:(2 * PS + 48) // 4,
                          (3 * PS - 16) // 4:(3 * PS + 60) // 4]).any()


def _reduce_case(c, f, rng):
    """Tiles (ps 64), pieces of the level grid of random tiles with random in-array extents,
    one fill piece, and the numpy result in 4 boxes of 20 x 24 (sentinel 77 outside the pieces)."""
    n_tiles, ps, n_boxes, bh, bw = 5, 64, 4, 20, 24
    lc = ps // f
    tiles = rng.integers(0, 256, size=(n_tiles, ps, ps, c), dtype=np.uint8)
    want = np.full((n_boxes, bh, bw, c), 77, dtype=np.uint8)
    pieces = []
    for b in range(n_boxes):
        for q in range(2):
            k = -1 if (b, q) == (2, 1) else int(rng.integers(0, n_tiles))
            vh, vw = int(rng.integers(1, ps + 1)), int(rng.integers(1, ps + 1))
            if q == 0:                          # a full-extent tile for every other piece
                vh, vw = (ps, ps) if b % 2 else (vh, vw)
            ly, lx = -(-vh // f), -(-vw // f)   # level rows / columns with in-array pixels
            h, w = int(rng.integers(1, min(ly, bh // 2) + 1)), int(rng.integers(1, min(lx, bw) + 1))
            sy, sx = int(rng.integers(0, ly - h + 1)), int(rng.integers(0, lx - w + 1))
            dy, dx = q * (bh // 2), int(rng.integers(0, bw - w + 1))
            pieces.append([k, b, sy, sx, dy, dx, h, w, vh, vw, 0, 0])
            want[b, dy:dy + h, dx:dx + w] = 0 if k < 0 else \
                reduce_ref(tiles[k, :vh, :vw], f)[sy:sy + h, sx:sx + w]
    return tiles, np.array(pieces, dtype=np.int32), want


@pytest.mark.parametrize('shift', [0, 4, 1])       # tile base off the 16- and 4-byte grids
@pytest.mark.parametrize('c', [1, 3])
@pytest.mark.parametrize('f', FACTORS)
def test_reduce_kernel_equals_numpy(f, c, shift):
    from cnn_autoencoder_b200 import _cabi as C
    rng = np.random.default_rng(1000 * f + 10 * c + shift)
    tiles, pieces, want = _reduce_case(c, f, rng)
    buf = torch.zeros(tiles.size + shift, dtype=torch.uint8, device='cuda')
    t = buf[shift:]
    t.copy_(torch.from_numpy(tiles.ravel()))
    out = torch.full(want.shape, 77, dtype=torch.uint8, device='cuda')
    pdev = torch.empty(pieces.size, dtype=torch.int32, device='cuda')
    C.check(C.lib().cae_tiles_crop_reduce_u8(
        t.data_ptr(), tiles.shape[0], tiles.shape[1], c, f, pieces.ctypes.data, len(pieces),
        pdev.data_ptr(), out.data_ptr(), want.shape[0], want.shape[1], want.shape[2],
        ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    assert np.array_equal(out.cpu().numpy(), want)
