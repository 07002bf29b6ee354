"""Region reads (``region.CompressedSlide``, ``cae_tiles_crop_u8``) against what decompress_image
writes for the same positions: a 12 x 13-chunk slide at PS = 64 with 40 px and 24 px edge chunks,
compared byte for byte."""
import ctypes
import json
import os
import shutil
import threading

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ARCH = dict(channels_org=3, channels_net=32, channels_bn=16, compression_level=3,
            act_layer_type='LeakyReLU')
PS = 64


def _slide(gy, gx, crop):
    from oracle import cae_oracle as O
    s = np.concatenate([np.concatenate([O.synth_tissue_tile(i, j, ps=PS, seed=2) for j in range(gx)],
                                       axis=1) for i in range(gy)], axis=0)
    return np.ascontiguousarray(s[:s.shape[0] - crop[0], :s.shape[1] - crop[1]])


def _pinned(shape):
    return torch.zeros(shape, dtype=torch.uint8).pin_memory().numpy()


@pytest.fixture(scope='module')
def store(tmp_path_factory):
    """(store path, checkpoint, decompress_image's reconstruction of the whole slide)."""
    from oracle import cae_oracle as O
    from cnn_autoencoder_b200 import compress, decompress
    chk = O.make_checkpoint(ARCH, seed=9)              # (seeds 31 and 5 reconstruct a constant 0)
    slide = _slide(12, 13, (24, 40))
    path = str(tmp_path_factory.mktemp('region') / 'slide.zarr')
    compress.compress_image('CAE', chk, slide, path, patch_size=PS, batch_tiles=16, coder_tiles=96)
    canvas = _pinned(slide.shape)
    ds = decompress.decompress_image(path, canvas, checkpoint=chk, batch_tiles=16, coder_tiles=96)
    assert ds['engine'] == 'slide'
    assert np.unique(canvas).size > 16                 # byte-for-byte comparisons of real content
    return path, chk, canvas


@pytest.fixture(scope='module')
def reader(store):
    from cnn_autoencoder_b200.region import CompressedSlide
    path, chk, _ = store
    with CompressedSlide(path, chk, batch_tiles=16) as r:
        yield r


def _touched(boxes, h, w):
    return {(iy, ix) for y, x in boxes for iy in range(y // PS, (y + h - 1) // PS + 1)
            for ix in range(x // PS, (x + w - 1) // PS + 1)}


def test_windows_equal_the_reconstruction(store, reader):
    _, _, canvas = store
    H, W, c = canvas.shape
    assert reader.shape == canvas.shape and reader.chunks == (PS, PS, 3) and reader.dtype == np.uint8
    for y, x, h, w in [(10, 5, 40, 50),                          # inside one chunk
                       (3 * PS - 20, 5 * PS - 30, 50, 70),       # across a 2 x 2 chunk corner
                       (H - 30, W - 50, 30, 50),                 # the ragged bottom-right edge
                       (0, 0, H, W)]:                            # the whole slide
        got = reader.read_region(y, x, h, w)
        assert got.is_cuda and tuple(got.shape) == (h, w, c)
        assert np.array_equal(got.cpu().numpy(), canvas[y:y + h, x:x + w]), (y, x, h, w)
        assert reader.stats['decoded'] == len(_touched([(y, x)], h, w))
    assert reader.stats['device_decoded'] == 156


def test_patch_batch_equals_the_reconstruction(store, reader):
    _, _, canvas = store
    H, W, _ = canvas.shape
    rng = np.random.default_rng(7)
    boxes = [(int(rng.integers(0, H - 48 + 1)), int(rng.integers(0, W - 40 + 1))) for _ in range(200)]
    got = reader.read_regions(boxes, 48, 40)
    want = np.stack([canvas[y:y + 48, x:x + 40] for y, x in boxes])
    assert np.array_equal(got.cpu().numpy(), want)
    assert reader.stats['decoded'] == reader.stats['chunks'] == len(_touched(boxes, 48, 40))


def test_device_and_host_coder_give_the_same_bytes(store):
    from cnn_autoencoder_b200.region import CompressedSlide
    path, chk, canvas = store
    H, W, _ = canvas.shape
    rng = np.random.default_rng(11)
    boxes = [(int(rng.integers(0, H - 33 + 1)), int(rng.integers(0, W - 57 + 1))) for _ in range(60)]
    want = np.stack([canvas[y:y + 33, x:x + 57] for y, x in boxes])
    with CompressedSlide(path, chk, batch_tiles=8) as r:
        got = {}
        for name, threshold in (('device', 1), ('host', 10 ** 9)):
            r.fact_ent.GPU_CODER_MIN_STREAMS = threshold       # instance override, this reader only
            got[name] = (r.read_regions(boxes, 33, 57).cpu().numpy(), r.read_region(0, 0, H, W).cpu().numpy())
            st = r.stats
            assert st['device_decoded'] == (st['decoded'] if name == 'device' else 0)
    for name in got:
        assert np.array_equal(got[name][0], want), name
        assert np.array_equal(got[name][1], canvas), name


def test_getitem_follows_numpy_slicing(store, reader):
    _, _, canvas = store
    keys = [(slice(10, 100), slice(20, 300)), (slice(-100, None), slice(-50, None)),
            (slice(700, 2000), slice(780, 900)), (5, slice(10, 20)), (slice(10, 20), 5), (-1, -1),
            (slice(None), slice(None)), slice(100, 140), 17, (slice(100, 50), slice(None)),
            (slice(3, 9), slice(60, 70), slice(None)), (slice(-2000, 3), slice(None, -700))]
    for key in keys:
        got = reader[key]
        want = canvas[key]
        assert isinstance(got, np.ndarray) and got.shape == want.shape, key
        assert np.array_equal(got, want), key
    for bad in [(slice(0, 10, 2), slice(None)), ([1, 2], slice(None)), (slice(None), slice(None), 0),
                (10 ** 6, 0), 1.5]:
        with pytest.raises(IndexError):
            reader[bad]


def test_out_arguments(store, reader):
    _, _, canvas = store
    y, x, h, w = 100, 130, 70, 90
    want = canvas[y:y + h, x:x + w]
    dev = torch.full((h, w, 3), 5, dtype=torch.uint8, device='cuda')
    assert reader.read_region(y, x, h, w, out=dev) is dev
    assert np.array_equal(dev.cpu().numpy(), want)
    for host in (_pinned((h, w, 3)), np.zeros((h, w, 3), dtype=np.uint8)):
        assert reader.read_region(y, x, h, w, out=host) is host
        assert np.array_equal(host, want)
    boxes = [(0, 0), (500, 700), (y, x)]
    many = torch.empty((3, h, w, 3), dtype=torch.uint8, device='cuda')
    assert reader.read_regions(boxes, h, w, out=many) is many
    assert np.array_equal(many.cpu().numpy(), np.stack([canvas[a:a + h, b:b + w] for a, b in boxes]))
    with pytest.raises(ValueError):
        reader.read_region(y, x, h, w, out=torch.empty((h, w + 1, 3), dtype=torch.uint8, device='cuda'))
    with pytest.raises(ValueError):
        reader.read_region(y, x, h, w, out=np.zeros((h, w, 3), dtype=np.float32))
    with pytest.raises(ValueError):
        reader.read_region(canvas.shape[0] - 10, 0, 20, 20)


def test_missing_chunk_reads_as_zeros(store, tmp_path):
    from cnn_autoencoder_b200.region import CompressedSlide
    path, chk, canvas = store
    # the interior chunk with the most non-zero pixels: its zeros are a visible change
    i, j = max(((i, j) for i in range(1, 11) for j in range(1, 12)),
               key=lambda t: np.count_nonzero(canvas[t[0] * PS:(t[0] + 1) * PS, t[1] * PS:(t[1] + 1) * PS]))
    assert canvas[i * PS:(i + 1) * PS, j * PS:(j + 1) * PS].any()
    copy = str(tmp_path / 'holey.zarr')
    shutil.copytree(path, copy)
    os.remove(os.path.join(copy, '0/0', '%d.%d.0' % (i, j)))
    want = canvas.copy()
    want[i * PS:(i + 1) * PS, j * PS:(j + 1) * PS] = 0
    with CompressedSlide(copy, chk) as r:
        assert np.array_equal(r[:, :], want)
        assert r.stats['missing'] == 1 and r.stats['decoded'] == 155
        y, x = i * PS - 5, j * PS + 10                  # 5 rows of chunk (i - 1, j), 15 of the hole
        win = r.read_region(y, x, 20, 30).cpu().numpy()
        assert r.stats['missing'] == 1 and r.stats['decoded'] == 1
        assert np.array_equal(win, want[y:y + 20, x:x + 30]) and not win[5:].any()


def test_refuses_latent_stores_and_odd_patch_sizes(tmp_path, store):
    from oracle import cae_oracle as O
    from cnn_autoencoder_b200 import compress
    from cnn_autoencoder_b200.region import CompressedSlide
    chk = O.make_checkpoint(ARCH, seed=17)
    slide = np.ascontiguousarray(_slide(4, 5, (0, 0))[:200, :304])
    out = str(tmp_path / 'lat.zarr')
    compress.compress_image('CAE', chk, slide, out, patch_size=128, save_as_bottleneck=True, batch_tiles=4)
    arr_dir = os.path.join(out, '0/0')
    for f in os.listdir(arr_dir):                 # refused on the metadata: no chunk is read
        if not f.startswith('.'):
            os.remove(os.path.join(arr_dir, f))
    with pytest.raises(ValueError, match='decompress_image'):
        CompressedSlide(out, chk)
    path, chk_s, _ = store
    odd = str(tmp_path / 'odd.zarr')
    shutil.copytree(path, odd)
    meta_file = os.path.join(odd, '0/0/.zarray')
    meta = json.load(open(meta_file))
    meta['chunks'] = [60, 60, 3]
    json.dump(meta, open(meta_file, 'w'))
    with pytest.raises(ValueError, match='multiple of 2'):
        CompressedSlide(odd, chk_s)


def _crop_case(c, mode, rng):
    """Tiles, pieces (quadrants of every box; one fill quadrant) and the numpy result."""
    n_tiles, ps, n_boxes = 5, 64, 4
    bh, bw, split_x = (48, 64, 32) if mode != 'unaligned' else (48, 61, 29)
    tiles = rng.integers(0, 256, size=(n_tiles, ps, ps, c), dtype=np.uint8)
    want = np.full((n_boxes, bh, bw, c), 77, dtype=np.uint8)
    pieces = []
    for b in range(n_boxes):
        for dy, h in ((0, 24), (24, bh - 24)):
            for dx, w in ((0, split_x), (split_x, bw - split_x)):
                k = -1 if (b, dy, dx) == (1, 24, 0) else int(rng.integers(0, n_tiles))
                if mode == 'unaligned':
                    sy, sx = int(rng.integers(0, ps - h + 1)), int(rng.integers(0, ps - w + 1))
                else:
                    sy, sx = int(rng.integers(0, ps - h + 1)), 16 * int(rng.integers(0, (ps - w) // 16 + 1))
                pieces.append([k, b, sy, sx, dy, dx, h, w])
                want[b, dy:dy + h, dx:dx + w] = 0 if k < 0 else tiles[k, sy:sy + h, sx:sx + w]
    return tiles, np.array(pieces, dtype=np.int32), want


@pytest.mark.parametrize('mode', ['aligned', 'unaligned', 'aligned_out_offset'])
@pytest.mark.parametrize('c', [1, 3, 4])
def test_crop_kernel_equals_numpy(c, mode):
    from cnn_autoencoder_b200 import _cabi as C
    rng = np.random.default_rng(c * 10 + len(mode))
    tiles, pieces, want = _crop_case(c, mode, rng)
    n_boxes, bh, bw = want.shape[:3]
    t = torch.from_numpy(tiles).cuda()
    shift = 4 if mode == 'aligned_out_offset' else 0         # a box base off the 16-byte grid
    buf = torch.full((want.size + shift,), 77, dtype=torch.uint8, device='cuda')
    out = buf[shift:]
    pdev = torch.empty(pieces.size, dtype=torch.int32, device='cuda')
    C.check(C.lib().cae_tiles_crop_u8(t.data_ptr(), tiles.shape[0], tiles.shape[1], c,
                                      pieces.ctypes.data, len(pieces), pdev.data_ptr(), out.data_ptr(),
                                      n_boxes, bh, bw,
                                      ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    assert np.array_equal(out.cpu().numpy().reshape(want.shape), want)
    assert (buf[:shift].cpu().numpy() == 77).all()


def test_reads_beside_decompress_image_on_another_thread(store, reader):
    """A reader and a decompress_image call of the same store and checkpoint on two threads:
    the reader has its own model and buffers, so both give the same bytes as alone."""
    from cnn_autoencoder_b200 import decompress
    path, chk, canvas = store
    H, W, _ = canvas.shape
    rng = np.random.default_rng(3)
    boxes = [(int(rng.integers(0, H - 64 + 1)), int(rng.integers(0, W - 64 + 1))) for _ in range(150)]
    want = np.stack([canvas[y:y + 64, x:x + 64] for y, x in boxes])
    other = _pinned(canvas.shape)
    got, errors = [], []

    def run_decompress():
        try:
            decompress.decompress_image(path, other, checkpoint=chk, batch_tiles=16, coder_tiles=96)
        except Exception as e:                       # re-raised on the main thread
            errors.append(e)
    t = threading.Thread(target=run_decompress)
    t.start()
    for _ in range(3):
        got.append(reader.read_regions(boxes, 64, 64).cpu().numpy())
        got.append(reader.read_region(0, 0, H, W).cpu().numpy())
    t.join()
    torch.cuda.synchronize()
    assert not errors, errors
    assert np.array_equal(other, canvas)
    for k in range(0, len(got), 2):
        assert np.array_equal(got[k], want) and np.array_equal(got[k + 1], canvas)
